// Grouped bf16 GEMM on tcgen05 tensor cores — the throughput arithmetic of the actor/critic MLP (2e-2 variant).
//
// replaces: aten::addmm / aten::mm of NetworkBlock.forward (src/models/network_block_creator.py:74-86) and of the
//           autograd backward of ppo.py:121,134, for the hidden layers.
//
// Per CTA (320 threads, one 128 x BN output tile, BN in {64,128,256}):
//   warp 0  TMA producer : cp.async.bulk.tensor 2-D boxes (128-byte swizzle) of A and B into a 4-stage smem ring,
//                          completion on per-stage mbarriers; out-of-bounds rows/columns are zero-filled by TMA,
//                          so ragged M/N/K need no padding in global memory.
//   warp 1  MMA issuer   : one elected lane issues tcgen05.mma.cta_group::1.kind::f16 (M=128, N=BN, K=16) x 4 per
//                          stage into a TMEM accumulator (BN fp32 columns), tcgen05.commit frees the stage.
//   warps 2-9 epilogue   : tcgen05.ld 32x32b.x32 (one accumulator row per thread, two warps per TMEM lane quarter
//                          splitting the columns), fused bias + MUFU tanh / relu, or
//                          activation-derivative multiply (dgrad), or fp32 split-K partial store (wgrad) with
//                          the bias gradient read off an appended ones-column of the B operand.
// Operands may be K-major or MN-major (UMMA descriptor major bits), so forward (X W^T), dgrad (dZ W, W MN-major)
// and wgrad (dZ^T X, both operands MN-major) share the kernel with no transposes.
#include <map>
#include <mutex>
#include <tuple>

#include "tc_common.cuh"

namespace b200ppo {

// smem ring depth: K loops are 1-6 tiles for forward/dgrad, so for BN <= 128 two 32 KB stages + the 32 KB epilogue
// staging area let two CTAs share an SM (one CTA's epilogue overlaps the other's TMA/MMA main loop); the wide tiles
// used by the long-K weight-gradient GEMM run one CTA per SM with a deeper ring.
// OCC = 2 with a wide tile (the fp32-tolerance GEMMs, whose K loops are six times as long as their epilogue is wide): two
// stages and no staging area, 100 KB per CTA, so that here too one CTA's epilogue overlaps the other's main loop.
template <int BN, int OCC> struct TcCfg {
  static constexpr int STAGES = OCC == 2 ? 2 : (BN <= 192 ? 5 : 4);  // 200 / 192 KB of operands in flight per SM at one CTA
  static constexpr int CTAS_PER_SM = OCC;
  static constexpr int STAGE_AREA = BN <= 128 ? TC_EPI_WARPS * 4096 : 0;  // (TC_STAGE_BYTES per epilogue warp; BN > 128 never stages)
};
int tc_ctas_per_sm(int bn) { return bn <= 128 ? 2 : 1; }

template <int BN, int OCC>
__global__ void __launch_bounds__(TC_THREADS, OCC) tc_gemm_kernel(const __grid_constant__ TcGroup grp) {
  constexpr int TC_STAGES = TcCfg<BN, OCC>::STAGES;
  constexpr int B_BYTES = BN * TC_BK * 2;
  constexpr uint32_t TMEM_COLS = BN <= 32 ? 32 : (BN <= 64 ? 64 : (BN <= 128 ? 128 : 256));  // power of two
  extern __shared__ uint8_t smem_raw[];
  // pointer + offset (not an integer round trip): the compiler keeps the shared address space and emits LDS / STS
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sA = smem;
  uint8_t* sB = smem + TC_STAGES * TC_A_BYTES;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(sB + TC_STAGES * B_BYTES);
  uint64_t* empty_bar = full_bar + TC_STAGES;
  uint64_t* tmem_full_bar = empty_bar + TC_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);
  float* bias_s = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(full_bar) + 256);  // BN floats (<= 256)
  float* consts_s = bias_s + 256;                                                        // 96 floats (fused PPO epilogue)
  float* red_s = bias_s + 352;                                                           // 8 x 34 floats
  uint8_t* stage_area = reinterpret_cast<uint8_t*>(bias_s) + 3072;                        // TC_EPI_WARPS x 4 KB

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // debug timeline: 0 entry, 1 set-up done (after the PDL wait), 2 first operands landed, 3 last MMA issued, 4 accumulator
  // complete (seen by warp 2), 5 warp 2's epilogue done, 6 CTA end; %smid in slot 7
  long long* const trc = (grp.trace != nullptr && blockIdx.x % 37 == 0 && blockIdx.x / 37 < 64) ? grp.trace + (blockIdx.x / 37) * 8 : nullptr;
  if (trc != nullptr && threadIdx.x == 0) {
    trc[0] = clock64();
    uint32_t smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    trc[7] = smid;
  }

  const TcTile T = tc_tile<BN>(grp, int(blockIdx.x));
  const TcProblem& P = grp.p[T.pi];
  const int split = T.split, m0 = T.m0, n0 = T.n0, n_it = T.n_it;
  const bool has_k = n_it > 0;

  if (warp == 1 && lane == 0) {
    for (int s = 0; s < TC_STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(tmem_full_bar, 1);
    mbar_init_fence();
  } else if (warp == 2) {
    tmem_alloc<1, TMEM_COLS>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait_then_release();  // everything below reads what earlier kernels of the chain wrote
  if (trc != nullptr && threadIdx.x == 0) trc[1] = clock64();
  if (warp >= 2) {          // epilogue warps stage their constants (named barrier 1: the other two warps are already streaming)
    tc_stage_bias(P, n0, BN, bias_s, threadIdx.x - 64, TC_THREADS - 64);
    tc_ppo_stage_consts(P, consts_s, threadIdx.x - 64);
    asm volatile("bar.sync 1, %0;" ::"n"(TC_THREADS - 64) : "memory");
  }

  if (warp == 0) {
    if (lane == 0 && has_k) {  // ===== TMA producer =====
      for (int it = 0; it < n_it; ++it) {
        const int s = it % TC_STAGES;
        const uint32_t ph = (it / TC_STAGES) & 1;
        mbar_wait(&empty_bar[s], ph ^ 1);
        mbar_expect_tx(&full_bar[s], TC_A_BYTES + B_BYTES);
        tc_load_stage<BN>(P, T, it, sA + s * TC_A_BYTES, sB + s * B_BYTES, &full_bar[s]);
      }
    }
  } else if (warp == 1) {
    if (has_k) {  // ===== MMA issuer =====
      const TcMma mma = tc_mma_setup<BN>(P);
      for (int it = 0; it < n_it; ++it) {
        const int s = it % TC_STAGES;
        const uint32_t ph = (it / TC_STAGES) & 1;
        mbar_wait(&full_bar[s], ph);
        tc_fence_after();
        if (trc != nullptr && lane == 0 && it == 0) trc[2] = clock64();
        if (trc != nullptr && lane == 0 && it == n_it - 1) trc[3] = clock64();
        if (lane == 0) {
          tc_mma_stage(mma, tmem_base, smem_u32(sA + s * TC_A_BYTES), smem_u32(sB + s * B_BYTES), it > 0);
          umma_commit(&empty_bar[s]);
          if (it == n_it - 1) umma_commit(tmem_full_bar);
        }
        __syncwarp();
      }
    }
  } else {  // ===== epilogue warps 2..9 =====
    if constexpr (BN <= 128) {
      if (P.epilogue >= TC_EPI_PPO_ACTOR) {
        uint8_t* st = stage_area + (warp - 2) * TC_STAGE_BYTES;
        PpoAcc acc;
        acc.clear();
        const bool worker = ((warp - 2) >> 2) == 0;
        tc_ppo_issue(P, m0, warp, lane, st, worker);
        tc_epilogue_ppo<BN>(P, tmem_base, m0, warp, lane, tmem_full_bar, 0, st, bias_s, consts_s, 0, acc, worker);
        tc_ppo_finish(P, warp, lane, red_s, acc, false);
      } else if (P.staged) {
        uint8_t* st = stage_area + (warp - 2) * TC_STAGE_BYTES;
        tc_issue_aux<BN>(P, m0, n0, warp, lane, st, true);
        tc_epilogue_staged<BN>(P, split, tmem_base, has_k, m0, n0, warp, lane, tmem_full_bar, 0, st, bias_s, 0);
      } else {
        tc_epilogue<BN>(P, split, tmem_base, has_k, m0, n0, warp, lane, tmem_full_bar, 0, bias_s);
      }
    } else tc_epilogue<BN>(P, split, tmem_base, has_k, m0, n0, warp, lane, tmem_full_bar, 0, bias_s);
    tc_fence_before();
    if (trc != nullptr && warp == 2 && lane == 0) trc[5] = clock64();
  }
  __syncthreads();
  if (trc != nullptr && threadIdx.x == 0) trc[6] = clock64();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<1, TMEM_COLS>(tmem_base);
  }
}

// ---- host side ---------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;
static std::mutex g_map_mutex;
static std::map<std::tuple<const void*, int64_t, int64_t, int64_t, int, int>, CUtensorMap> g_map_cache;

int tc_init() {
  if (g_encode) return B200PPO_OK;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  B2_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
  if (fn == nullptr || qres != cudaDriverEntryPointSuccess) {
    set_error("cuTensorMapEncodeTiled is not available from this driver");
    return B200PPO_ECUDA;
  }
  g_encode = reinterpret_cast<EncodeTiledFn>(fn);
  return B200PPO_OK;
}

int tc_make_map(CUtensorMap* out, const __nv_bfloat16* ptr, int64_t inner, int64_t outer, int64_t pitch, int box_inner,
                    int box_outer) {
  B2_TRY(tc_init());
  auto key = std::make_tuple(static_cast<const void*>(ptr), inner, outer, pitch, box_inner, box_outer);
  std::lock_guard<std::mutex> lock(g_map_mutex);
  auto it = g_map_cache.find(key);
  if (it != g_map_cache.end()) {
    *out = it->second;
    return B200PPO_OK;
  }
  B2_CHECK_ARG(aligned16(ptr) && (pitch * 2) % 16 == 0 && inner > 0 && outer > 0, "tensor map: base/pitch must be 16-byte aligned");
  cuuint64_t gdim[2] = {cuuint64_t(inner), cuuint64_t(outer)};
  cuuint64_t gstride[1] = {cuuint64_t(pitch * 2)};
  cuuint32_t box[2] = {cuuint32_t(box_inner), cuuint32_t(box_outer)};
  cuuint32_t estr[2] = {1, 1};
  CUtensorMap m;
  const CUresult r = g_encode(&m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<__nv_bfloat16*>(ptr), gdim, gstride, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) for extents [%lld,%lld] pitch %lld box [%d,%d]", int(r), (long long)inner,
              (long long)outer, (long long)pitch, box_inner, box_outer);
    return B200PPO_ECUDA;
  }
  if (g_map_cache.size() > 65536) g_map_cache.clear();
  g_map_cache.emplace(key, m);
  *out = m;
  return B200PPO_OK;
}

int tc_group_add(TcGroup& g, TcProblem p, const TcOperand& A, const TcOperand& B, int bn, int split_k) {
  if (p.M <= 0 || p.N <= 0 || p.K <= 0) return B200PPO_OK;
  B2_CHECK_ARG(g.count < kMaxTcProblems, "too many problems in one tensor-core group");
  p.a_mn_major = A.mn_major;
  p.b_mn_major = B.mn_major;
  // fp32-tolerance mode: the whole row (three terms) is addressable, the producer adds the term's offset to the coordinate
  const int64_t a_inner = p.parts ? p.parts * int64_t(p.a_part) : (A.mn_major ? p.M : p.K);
  const int64_t b_inner = p.parts ? p.parts * int64_t(p.b_part) : (B.mn_major ? p.N : p.K);
  if (!A.mn_major) B2_TRY(tc_make_map(&p.tmA, A.ptr, a_inner, p.M, A.pitch, TC_BK, TC_BM));
  else B2_TRY(tc_make_map(&p.tmA, A.ptr, a_inner, p.K, A.pitch, 64, TC_BK));
  if (!B.mn_major) B2_TRY(tc_make_map(&p.tmB, B.ptr, b_inner, p.N, B.pitch, TC_BK, bn));
  else B2_TRY(tc_make_map(&p.tmB, B.ptr, b_inner, p.K, B.pitch, 64, TC_BK));
  const int total_kt = (p.K + TC_BK - 1) / TC_BK;
  if (split_k < 1) split_k = 1;
  if (split_k > total_kt && !p.parts) split_k = total_kt;  // (fp32-tolerance mode: the caller sums exactly split_k partials; empty ones store zeros)
  p.split_k = split_k;
  p.k_tiles_per_split = (total_kt + split_k - 1) / split_k;
  p.tiles_m = (p.M + TC_BM - 1) / TC_BM;
  p.tiles_n = (p.N + bn - 1) / bn;
  p.tile_begin = g.total_tiles;
  p.staged = tc_can_stage(p) ? 1 : 0;
  g.total_tiles += p.tiles_m * p.tiles_n * split_k;
  g.p[g.count++] = p;
  return B200PPO_OK;
}

template <int BN, int OCC>
static int launch_bn(const TcGroup& g, cudaStream_t st) {
  constexpr int smem = TcCfg<BN, OCC>::STAGES * (TC_A_BYTES + BN * TC_BK * 2) + 1024 + 256 + 3072 + TcCfg<BN, OCC>::STAGE_AREA;
  static bool configured = false;
  if (!configured) {
    B2_CUDA(cudaFuncSetAttribute(tc_gemm_kernel<BN, OCC>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    configured = true;
  }
  B2_CUDA(launch_pdl(tc_gemm_kernel<BN, OCC>, dim3(g.total_tiles), dim3(TC_THREADS), smem, st, g));
  B2_LAUNCH_CHECK();
  return B200PPO_OK;
}

int launch_tc_group(const TcGroup& g, int bn, cudaStream_t st, int* grid_out, bool two_per_sm) {
  if (grid_out) *grid_out = g.total_tiles;
  if (g.total_tiles == 0) return B200PPO_OK;
  switch (bn) {
    case 64: return launch_bn<64, 2>(g, st);
    case 128: return launch_bn<128, 2>(g, st);
    case 192: return two_per_sm ? launch_bn<192, 2>(g, st) : launch_bn<192, 1>(g, st);
    case 256: return two_per_sm ? launch_bn<256, 2>(g, st) : launch_bn<256, 1>(g, st);
  }
  set_error("unsupported tensor-core N tile %d", bn);
  return B200PPO_EINVAL;
}

int tc_pick_bn(int64_t tiles_m_total, int N) {
  // 128-wide tiles run two CTAs per SM (epilogue of one overlaps the main loop of the other); narrower only when
  // the problem is narrow or would leave SMs idle
  (void)tiles_m_total;
  return N > 64 ? 128 : 64;
}

// ---- debug entry point: C = A * B^T through the tensor-core kernel (used by the GPU tests) -------------------------
__global__ void cast_pad_bf16_kernel(const float* __restrict__ src, int64_t rows, int64_t cols, int64_t pitch,
                                     __nv_bfloat16* __restrict__ dst) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= rows * pitch) return;
  const int64_t r = i / pitch, c = i % pitch;
  dst[i] = __float2bfloat16_rn(c < cols ? src[r * cols + c] : 0.f);
}

__global__ void sum_splits_kernel(const float* __restrict__ part, int splits, int64_t stride, int64_t n, float* __restrict__ out) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float s = 0.f;
  for (int k = 0; k < splits; ++k) s += part[k * stride + i];
  out[i] = s;
}

__global__ void bf16_rows_to_f32_kernel(const __nv_bfloat16* __restrict__ src, int64_t rows, int64_t cols, int64_t pitch, float* __restrict__ dst) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= rows * cols) return;
  dst[i] = __bfloat162float(src[(i / cols) * pitch + i % cols]);
}

}  // namespace b200ppo

using namespace b200ppo;

extern "C" B2_EXPORT int b200ppo_debug_tc_gemm(const float* A, const float* B, float* C, int32_t M, int32_t N, int32_t K,
                                               int32_t a_mn_major, int32_t b_mn_major, int32_t bn, int32_t split_k,
                                               b200ppo_stream stream) {
  B2_CHECK_ARG(A && B && C && M > 0 && N > 0 && K > 0, "b200ppo_debug_tc_gemm: bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  auto pad8 = [](int64_t x) { return (x + 7) / 8 * 8; };
  // global arrays: K-major operand [MN][K]; MN-major operand [K][MN]
  const int64_t a_rows = a_mn_major ? K : M, a_cols = a_mn_major ? M : K;
  const int64_t b_rows = b_mn_major ? K : N, b_cols = b_mn_major ? N : K;
  const int64_t a_pitch = pad8(a_cols), b_pitch = pad8(b_cols);
  __nv_bfloat16 *Ab = nullptr, *Bb = nullptr;
  float* part = nullptr;
  if (split_k < 1) split_k = 1;
  B2_CUDA(cudaMalloc(&Ab, a_rows * a_pitch * 2));
  B2_CUDA(cudaMalloc(&Bb, b_rows * b_pitch * 2));
  const int64_t mn = int64_t(M) * N, stride = (mn + 3) / 4 * 4;
  B2_CUDA(cudaMalloc(&part, size_t(split_k) * stride * 4));
  cast_pad_bf16_kernel<<<unsigned((a_rows * a_pitch + 255) / 256), 256, 0, st>>>(A, a_rows, a_cols, a_pitch, Ab);
  B2_LAUNCH_CHECK();
  cast_pad_bf16_kernel<<<unsigned((b_rows * b_pitch + 255) / 256), 256, 0, st>>>(B, b_rows, b_cols, b_pitch, Bb);
  B2_LAUNCH_CHECK();
  TcGroup g{};
  TcProblem p{};
  p.M = M; p.N = N; p.K = K;
  p.epilogue = TC_EPI_STORE;
  p.out_f32 = part; p.ld_f32 = N; p.split_stride = stride; p.bias_col = -1;
  // bn = -1: the persistent weights-stationary kernel;
  // bn = -3: forward epilogue, C = float(tanh(A B^T) rounded to bf16) — the path the CTA-pair kernel takes for N > 128
  // bn = -4: dgrad epilogue, C on entry holds the activation operand h; C = float(bf16(A B^T * (1 - bf16(h)^2)))
  B2_CHECK_ARG(bn >= 0 || bn == -1 || bn == -3 || bn == -4, "b200ppo_debug_tc_gemm: bn must be >= 0, -1, -3 or -4");
  const bool ws = bn < 0;
  const bool fwd_check = bn == -3 || bn == -4;
  if (bn == -4) {
    p.epilogue = TC_EPI_DGRAD; p.act = B200PPO_ACT_TANH;
    p.out_f32 = nullptr;
    const int64_t ld = (N + 7) / 8 * 8;
    __nv_bfloat16* auxb = nullptr;
    B2_CUDA(cudaMalloc(&p.out_bf16, size_t(M) * ld * 2));
    B2_CUDA(cudaMalloc(&auxb, size_t(M) * ld * 2));
    cast_pad_bf16_kernel<<<unsigned((int64_t(M) * ld + 255) / 256), 256, 0, st>>>(C, M, N, ld, auxb);
    B2_LAUNCH_CHECK();
    p.ld_bf16 = int(ld); p.aux = auxb; p.ld_aux = int(ld);
  }
  if (bn == -3) {
    p.epilogue = TC_EPI_FWD; p.act = B200PPO_ACT_TANH;  // the production forward epilogue, bf16 output
    p.out_f32 = nullptr;
    B2_CUDA(cudaMalloc(&p.out_bf16, size_t(M) * ((N + 7) / 8 * 8) * 2));
    p.ld_bf16 = (N + 7) / 8 * 8;
  }
  if (ws) bn = tc_ws_bn(N, K);
  int rc = tc_group_add(g, p, TcOperand{Ab, a_pitch, a_mn_major}, TcOperand{Bb, b_pitch, b_mn_major}, bn, split_k);
  if (rc == B200PPO_OK) rc = ws ? launch_tc_ws(g, st) : launch_tc_group(g, bn, st);
  if (rc == B200PPO_OK && fwd_check) {
    bf16_rows_to_f32_kernel<<<unsigned((mn + 255) / 256), 256, 0, st>>>(p.out_bf16, M, N, p.ld_bf16, C);
    count_launch();
  } else if (rc == B200PPO_OK) {
    sum_splits_kernel<<<unsigned((mn + 255) / 256), 256, 0, st>>>(part, g.p[0].split_k, stride, mn, C);
    count_launch();
  }
  cudaStreamSynchronize(st);
  if (p.out_bf16 != nullptr) cudaFree(p.out_bf16);
  if (p.aux != nullptr) cudaFree(const_cast<__nv_bfloat16*>(p.aux));
  cudaFree(Ab); cudaFree(Bb); cudaFree(part);
  {
    std::lock_guard<std::mutex> lock(g_map_mutex);
    g_map_cache.clear();  // the temporaries above are gone
  }
  if (rc != B200PPO_OK) return rc;
  B2_CUDA(cudaGetLastError());
  return B200PPO_OK;
}
