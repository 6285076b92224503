// Grouped bf16 GEMM on the 5th-generation tensor cores (tcgen05.mma, TMEM accumulators, TMA operand staging).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <string.h>

#include "common.cuh"

namespace b200ppo {

enum TcEpilogue : int {
  TC_EPI_FWD = 0,    // h = act(acc + bias[n]) -> bf16 (and optionally fp32)
  TC_EPI_DGRAD = 1,  // dz = acc * act'(aux[m,n]) -> bf16
  TC_EPI_STORE = 2,  // fp32 store of a split-K partial; column `bias_col` is routed to bias_grad[m]
  // Output layers of the PPO update with the loss fused in (one accumulator row = one sample, all act_dim outputs of
  // the row live in one thread): nothing but the gradient seeds and per-CTA loss partials leaves the kernel.
  TC_EPI_PPO_ACTOR = 3,   // mean = [scale*tanh](acc + bias); log-prob, ratio, clipped surrogate; dz -> bf16; partial sums
  TC_EPI_PPO_CRITIC = 4,  // v = acc + bias; Huber; dv -> bf16; partial sum
};

// Extra operands of the fused PPO epilogues (src/entities/algorithms/ppo.py:113-132).
struct TcPpo {
  const float* logstd;     // [A]
  const float* action;     // [M, A]
  const float* old_logp;   // [M]
  const float* advantage;  // [M]
  const float* target;     // [M]
  __nv_bfloat16* dz_out;   // actor: [M, dz_pitch] ; critic: [M, dz_pitch] with dv in column 0
  float* partials;         // [gridDim.x][2 + A]: (sum surrogate, sum huber, sum d loss / d logstd_j) per CTA
  int dz_pitch, act_dim, final_tanh;
  float clip_eps, inv_global_batch;
};

// activation codes of TC_EPI_FWD beyond B200PPO_ACT_TANH / B200PPO_ACT_RELU
constexpr int TC_ACT_NONE = 2;        // out = acc + bias
constexpr int TC_ACT_TANH_SCALE = 3;  // out = out_scale * tanh(acc + bias)   (linear/actor.py:28)

// C[m,n] = sum_k A(m,k) * B(n,k), bf16 operands, fp32 accumulation in TMEM.
// K-major operand: global bf16 [rows = M or N][k], k contiguous.   MN-major operand: global bf16 [k][M or N].
struct TcProblem {
  CUtensorMap tmA, tmB;
  int M, N, K;
  int a_mn_major, b_mn_major;
  int tiles_m, tiles_n, split_k, k_tiles_per_split, tile_begin;
  int epilogue, act;
  const float* bias;
  __nv_bfloat16* out_bf16;
  int ld_bf16;
  float* out_f32;
  int ld_f32;
  int64_t split_stride;
  const __nv_bfloat16* aux;
  int ld_aux;
  float* bias_grad;
  int bias_col;  // -1: none
  float out_scale;
  int staged;  // epilogue goes through the shared-memory staging tile (set by tc_group_add)
  // fp32-tolerance mode (gemm_split.cu): both operands are stored as three bf16 terms per value (x = a + b + c to 2^-24,
  // the terms side by side along the contiguous dimension, `a_part` / `b_part` elements apart) and the K loop runs the six
  // products ac ca bb ab ba aa into the same fp32 accumulator — smallest first: the tensor core TRUNCATES the fp32
  // accumulator after every K = 16 step (measured, profiles/rz_probe.py: -0.47 ulp per step), so only the aa steps, which
  // come last, may happen at the accumulator's full magnitude.  0: plain bf16 operands.
  // parts == 2: two fp16 terms of the SCALED value (x 2^e, e from the tensor's largest magnitude, split_exponent below:
  // 11 + 11 significant bits), products ab' ba' aa' — half the tensor work and operand traffic of the three-term mode; the
  // epilogue multiplies the accumulator by 2^-(eA + eB), read from amax_a / amax_b.
  int parts, a_part, b_part;
  const float *amax_a, *amax_b;
  // three-term mode, forward / dgrad epilogues: the fp32 result is ALSO written as its three bf16 terms, [M][3 * split_cp] with
  // the zero padding (and the ones-column, split_ones) of gemm_split.cu's layout — the next GEMM's operand without a split pass
  __nv_bfloat16* out_split;
  int split_cp, split_ones;
  const float* aux_f32;  // TC_EPI_DGRAD: activation operand in fp32 (instead of `aux`)
  int precise;           // TC_EPI_FWD: tanhf instead of the MUFU approximation
  TcPpo ppo;
};

// the six (A term, B term) products of the fp32-tolerance mode, one nibble per product
constexpr uint32_t kSplitTermsA = 0x010120u, kSplitTermsB = 0x001102u;
constexpr int kSplitProducts = 6;
// two-term mode: ab', ba', aa'
constexpr uint32_t kSplit2TermsA = 0x010u, kSplit2TermsB = 0x001u;
constexpr int kSplit2Products = 3;
__host__ __device__ inline int split_products(int parts) { return parts == 2 ? kSplit2Products : kSplitProducts; }
__host__ __device__ inline uint32_t split_terms_a(int parts) { return parts == 2 ? kSplit2TermsA : kSplitTermsA; }
__host__ __device__ inline uint32_t split_terms_b(int parts) { return parts == 2 ? kSplit2TermsB : kSplitTermsB; }

// Two-term fp16 mode of the fp32-tolerance GEMMs (gemm_split.cu): a tensor whose largest magnitude is amax is scaled by
// 2^e with e = 14 - ceil(log2(amax)), so that its largest value lands in (2^13, 2^14] — inside fp16's range with the
// residual terms still normal numbers.  Exact integer arithmetic on the float's bits; amax = 0 -> e = 0.
__host__ __device__ inline int split_exponent(float amax) {
  if (!(amax > 0.f)) return 0;
#ifdef __CUDA_ARCH__
  const uint32_t bits = __float_as_uint(amax);
#else
  uint32_t bits;
  memcpy(&bits, &amax, 4);
#endif
  const int ex = int((bits >> 23) & 0xffu) - 127;          // floor(log2(amax)) for normal numbers
  const int ceil_log2 = (bits & 0x7fffffu) ? ex + 1 : ex;
  int e = 14 - ceil_log2;
  return e > 100 ? 100 : (e < -100 ? -100 : e);
}

// Fused PPO epilogue applies when a warp's action slab (32 x A floats) and bf16 seed slab (32 x pad8(A)) share its 4 KB
// staging tile, i.e. A <= 21 (Humanoid 17, Ant 8, HalfCheetah 6, Hopper 3).
inline bool tc_ppo_fits(int act_dim) { return act_dim >= 1 && act_dim * 128 + ((act_dim + 7) / 8 * 8) * 64 <= 4096; }

constexpr int kMaxTcProblems = 6;

struct TcGroup {
  TcProblem p[kMaxTcProblems];
  int count;
  int total_tiles;
  long long* trace;  // debug: clock64 phase marks of every 37th CTA, 8 slots each (nullptr in production)
};

// Operand description handed to tc_group_add (device pointers to bf16, pitches in elements).
struct TcOperand {
  const __nv_bfloat16* ptr;
  int64_t pitch;   // elements between consecutive rows of the global array
  int mn_major;    // 0: array is [MN][K] (K contiguous); 1: array is [K][MN] (MN contiguous)
};

// 2-D bf16 tensor map with 128-byte swizzle over a [outer][pitch] array whose first `inner` columns are addressable (cached).
int tc_make_map(CUtensorMap* out, const __nv_bfloat16* ptr, int64_t inner, int64_t outer, int64_t pitch, int box_inner, int box_outer);
int tc_init();  // resolves cuTensorMapEncodeTiled; returns B200PPO_OK or an error
// bn: N tile (64, 128 or 256).  Fills tensor maps (cached) and tile bookkeeping.
int tc_group_add(TcGroup& g, TcProblem p, const TcOperand& A, const TcOperand& B, int bn, int split_k);
// two_per_sm: the 192- / 256-wide tiles with a two-stage ring and two CTAs per SM (default: deep ring, one CTA)
int launch_tc_group(const TcGroup& g, int bn, cudaStream_t st, int* grid_out = nullptr, bool two_per_sm = false);
// Persistent instance (tc_persist.cu): one CTA per SM walks the tiles, accumulators double-buffered in TMEM; bn 192 or 256,
// plain epilogues (forward / dgrad / store).  Used by the fp32-tolerance GEMMs.
int launch_tc_persist(const TcGroup& g, int bn, cudaStream_t st);
int tc_pick_bn(int64_t rows_total_tiles_m, int N);
int tc_ctas_per_sm(int bn);
// Persistent weights-stationary variant (tc_ws.cu) for forward / dgrad groups with many row tiles.
bool tc_ws_applicable(int64_t total_tiles_m, int maxN, int maxK);
int tc_ws_bn(int maxN, int maxK);
// w_early: the weights were last written two or more kernels back in the stream (never true right after the optimizer)
int launch_tc_ws(const TcGroup& g, cudaStream_t st, int* grid_out = nullptr, bool w_early = false);  // resident CTAs per SM of the bn-wide kernel instance

// CTA-pair weight-gradient kernel (tc_wgrad.cu): every problem MN-major x MN-major with fp32 split-K partials; N is the
// layer's input width without a ones-column, the bias gradient comes from a second MMA against a tile of ones.
int launch_tc_wgrad2(const TcGroup& g, int max_split, cudaStream_t st, int* split_out);

}  // namespace b200ppo
