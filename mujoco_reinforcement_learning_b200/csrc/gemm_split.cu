// fp32-tolerance variant of the actor/critic GEMMs on tcgen05 (north_star's 1e-5 variant on the tensor cores).
//
// replaces: the same aten::addmm / aten::mm calls as gemm.cu (src/models/network_block_creator.py:74-86 forward, autograd
//           of ppo.py:121,134 backward) — gemm.cu does them with FFMA, this file with six bf16 MMAs per product.
//
// A bf16 value carries 8 significant bits, an fp32 value 24: x = a + b + c with a = bf16(x), b = bf16(x - a),
// c = bf16(x - a - b) is exact to 2^-24 |x| (both subtractions are exact in fp32).  For a dot product
//   sum x y = sum (a + b + c)(a' + b' + c') = aa' + ab' + ba' + bb' + ac' + ca'  +  O(2^-24 |x||y|)
// — the three dropped products (bc', cb', cc') are below 2^-24 — and every bf16 x bf16 product is exact in the tensor
// core's fp32 accumulator.  Measured against fp64 on the bench shapes (profiles/README.md): max error / max |C| 3e-7, the
// same as an fp32 FFMA loop (8e-7); three products (aa' + ab' + ba') give 5e-6, too close to the 1e-5 tolerance.
//
// Data layout: a [rows][cols] fp32 operand becomes bf16 [rows][3 * cp], cp = pad64(cols + 1): the three terms of a row
// side by side, each padded with zeros to a whole number of 64-element k tiles.  The contiguous dimension is K for a
// K-major operand and M / N for an MN-major one; either way the tile kernel (tc_gemm.cu) reaches term t by adding t * cp
// to the box coordinate along that dimension, so ONE split of an activation serves the forward (K-major A operand) and the
// weight gradient (MN-major B operand).  Activations get a column of ones behind their last column (term a only): as the
// weight gradient's B operand that column makes the bias gradient fall out of the same MMAs (TcProblem.bias_col).
//
// Environment switches (read once per process; none needed in use):
//   B200PPO_FP32_TC=0              keep every fp32 GEMM on the FFMA kernels
//   B200PPO_SPLIT_TRACE=<n>        phase timeline of the n-th launch on stderr
#include "gemm_split.cuh"

#include <cuda_fp16.h>

#include <algorithm>

#include "tc_gemm.cuh"

namespace b200ppo {

static inline int pad64(int x) { return (x + 63) / 64 * 64; }
int64_t split_arena_elems(int64_t rows, int cols) { return (rows * 3 * pad64(cols + 1) + 511) / 512 * 512; }

int split_arena_reserve(SplitArena& a, int64_t elems) {
  if (a.amax == nullptr) B2_TRY(a.amax.alloc(SplitArena::kMaxEntries));
  return a.base.grow(elems);
}

// ---- the split pass ------------------------------------------------------------------------------------------------------
struct SplitJob {
  const float* src;
  __nv_bfloat16* dst;
  float* amax;                   // two-term mode: this operand's largest magnitude (filled by absmax_kernel, or from the bound)
  const float* bound_dev;        // a caller-supplied upper bound of it (device value; nullptr: `bound`; both empty: measure)
  float bound;
  int64_t rows, ld, unit_begin;  // first 8-column unit of this job in the launch
  int cols, cp, ones, vec, terms;
};
constexpr int kMaxSplitJobs = 2 * kMaxGemmProblems;
struct SplitJobs {
  SplitJob j[kMaxSplitJobs];
  int n;
  int64_t units;
};

__device__ __forceinline__ uint32_t pack2(__nv_bfloat16 lo, __nv_bfloat16 hi) {
  return uint32_t(__bfloat16_as_ushort(lo)) | (uint32_t(__bfloat16_as_ushort(hi)) << 16);
}

// one thread = 8 consecutive columns of one row
__device__ __forceinline__ void split_load8(const SplitJob& J, int64_t row, int c0, float (&x)[8], float one) {
  const float* sp = J.src + row * J.ld + c0;
  if (J.vec && c0 + 8 <= J.cols) {
    const float4 p = __ldg(reinterpret_cast<const float4*>(sp)), q = __ldg(reinterpret_cast<const float4*>(sp) + 1);
    x[0] = p.x; x[1] = p.y; x[2] = p.z; x[3] = p.w; x[4] = q.x; x[5] = q.y; x[6] = q.z; x[7] = q.w;
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j) x[j] = (c0 + j < J.cols) ? __ldg(sp + j) : ((c0 + j == J.cols && J.ones) ? one : 0.f);
  }
}

__device__ __forceinline__ bool J_ones_first(const SplitJob& J, int64_t u) { return J.ones != 0 && u == J.unit_begin; }

// Largest magnitude of every job's source (two-term mode), one atomicMax per warp on the float's bits; an operand that
// carries the ones-column counts a 1.0, so that the column's scaled value 2^e stays inside fp16.
__global__ void __launch_bounds__(256) absmax_kernel(const __grid_constant__ SplitJobs jobs) {
  const int64_t u = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  float m = 0.f;
  int ji = 0;
  if (u < jobs.units) {
#pragma unroll 1
    for (int i = 1; i < jobs.n; ++i)
      if (u >= jobs.j[i].unit_begin) ji = i;
    const SplitJob& J = jobs.j[ji];
    const int upr = J.cp >> 3;
    const int64_t local = u - J.unit_begin;
    const int64_t row = local / upr;
    const int c0 = int(local - row * upr) * 8;
    float x[8];
    split_load8(J, row, c0, x, 1.f);
#pragma unroll
    for (int j = 0; j < 8; ++j) m = fmaxf(m, fabsf(x[j]));
  }
  // warp -> block -> one atomic per (block, job), and none at all when the block cannot raise the current value
  __shared__ float wm[8];
  __shared__ int wj[8];
  const bool live = u < jobs.units;
  const int key = live ? ji : -1;
  const unsigned same = __match_any_sync(0xffffffffu, key);
  const int wid = threadIdx.x >> 5;
  if (same == 0xffffffffu) {
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) { wm[wid] = m; wj[wid] = key; }
  } else {  // a warp that straddles a job boundary (or the end of the launch): lane by lane
    if ((threadIdx.x & 31) == 0) { wm[wid] = 0.f; wj[wid] = -1; }
    if (live && m > 0.f) atomicMax(reinterpret_cast<unsigned*>(jobs.j[ji].amax), __float_as_uint(m));
  }
  if (live && J_ones_first(jobs.j[ji], u)) atomicMax(reinterpret_cast<unsigned*>(jobs.j[ji].amax), __float_as_uint(1.f));
  __syncthreads();
  if (threadIdx.x == 0) {
    int cur = -1;
    float best = 0.f;
    for (int w = 0; w <= 8; ++w) {
      const int j = w < 8 ? wj[w] : -2;
      if (j != cur) {
        if (cur >= 0 && best > 0.f) {
          unsigned* dst = reinterpret_cast<unsigned*>(jobs.j[cur].amax);
          if (__float_as_uint(best) > *reinterpret_cast<volatile unsigned*>(dst)) atomicMax(dst, __float_as_uint(best));
        }
        cur = j;
        best = 0.f;
      }
      if (w < 8) best = fmaxf(best, wm[w]);
    }
  }
}

// Bias gradients of the two-term mode: bias_grad[s][m] = sum over split s's rows k of A[k][m], fp32, fixed order (a thread
// walks its rows in order, the eight row groups of a block meet in shared memory in order): deterministic.
struct ColsumJob {
  const float* src;   // [rows][ld], `cols` columns used
  float* dst;         // [splits][split_stride], column m at dst[s * split_stride + m]
  int64_t rows, ld, split_stride;
  int cols, splits, block_begin;
};
struct ColsumJobs {
  ColsumJob j[kMaxGemmProblems];
  int n, blocks;
};

__global__ void __launch_bounds__(256) colsum_kernel(const __grid_constant__ ColsumJobs jobs) {
  int ji = 0;
#pragma unroll 1
  for (int i = 1; i < jobs.n; ++i)
    if (int(blockIdx.x) >= jobs.j[i].block_begin) ji = i;
  const ColsumJob& J = jobs.j[ji];
  const int local = int(blockIdx.x) - J.block_begin;
  const int strips = (J.cols + 31) / 32;
  const int s = local / strips, c = (local - s * strips) * 32 + int(threadIdx.x & 31);
  const int ty = threadIdx.x >> 5;
  const int64_t per = (J.rows + J.splits - 1) / J.splits;
  const int64_t r0 = int64_t(s) * per, r1 = min(r0 + per, J.rows);
  float acc = 0.f;
  if (c < J.cols) {
    const float* sp = J.src + c;
    int64_t r = r0 + ty;
    for (; r + 24 < r1; r += 32) {  // four independent loads in flight
      const float a0 = __ldg(sp + r * J.ld), a1 = __ldg(sp + (r + 8) * J.ld), a2 = __ldg(sp + (r + 16) * J.ld), a3 = __ldg(sp + (r + 24) * J.ld);
      acc += a0; acc += a1; acc += a2; acc += a3;
    }
    for (; r < r1; r += 8) acc += __ldg(sp + r * J.ld);
  }
  __shared__ float part[8][32];
  part[ty][threadIdx.x & 31] = acc;
  __syncthreads();
  if (ty == 0 && c < J.cols) {
    float t = part[0][threadIdx.x];
#pragma unroll
    for (int i = 1; i < 8; ++i) t += part[i][threadIdx.x];
    J.dst[int64_t(s) * J.split_stride + c] = t;
  }
}

__global__ void __launch_bounds__(256) split3_kernel(const __grid_constant__ SplitJobs jobs) {
  asm volatile("griddepcontrol.wait;" ::: "memory");
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const int64_t u = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (u >= jobs.units) return;
  int ji = 0;
#pragma unroll 1
  for (int i = 1; i < jobs.n; ++i)
    if (u >= jobs.j[i].unit_begin) ji = i;
  const SplitJob& J = jobs.j[ji];
  const int upr = J.cp >> 3;
  const int64_t local = u - J.unit_begin;
  const int64_t row = local / upr;
  const int c0 = int(local - row * upr) * 8;
  float x[8];
  split_load8(J, row, c0, x, 1.f);
  if (J.terms == 2) {  // two fp16 terms of x * 2^e
    float am;
    if (J.bound_dev != nullptr || J.bound > 0.f) {  // no measuring pass ran: publish the bound for the GEMM's epilogue
      am = J.bound_dev != nullptr ? __ldg(J.bound_dev) : J.bound;
      if (J.ones) am = fmaxf(am, 1.f);
      if (u == J.unit_begin) *J.amax = am;
    } else {
      am = __ldg(J.amax);
    }
    const float sc = exp2f(float(split_exponent(am)));
    uint32_t o[2][4];
#pragma unroll
    for (int j = 0; j < 8; j += 2) {
      __half t[2][2];
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        float r = x[j + k] * sc;  // exact: a power of two, no overflow by the choice of e
#pragma unroll
        for (int p = 0; p < 2; ++p) {
          t[p][k] = __float2half_rn(r);
          r -= __half2float(t[p][k]);  // exact
        }
      }
#pragma unroll
      for (int p = 0; p < 2; ++p) o[p][j >> 1] = uint32_t(__half_as_ushort(t[p][0])) | (uint32_t(__half_as_ushort(t[p][1])) << 16);
    }
    __nv_bfloat16* dp = J.dst + row * (2 * int64_t(J.cp)) + c0;
#pragma unroll
    for (int p = 0; p < 2; ++p) *reinterpret_cast<uint4*>(dp + int64_t(p) * J.cp) = make_uint4(o[p][0], o[p][1], o[p][2], o[p][3]);
    return;
  }
  uint32_t o[3][4];
#pragma unroll
  for (int j = 0; j < 8; j += 2) {
    __nv_bfloat16 t[3][2];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      float r = x[j + k];
#pragma unroll
      for (int p = 0; p < 3; ++p) {
        t[p][k] = __float2bfloat16_rn(r);
        r -= __bfloat162float(t[p][k]);  // exact: the term shares r's leading bits
      }
    }
#pragma unroll
    for (int p = 0; p < 3; ++p) o[p][j >> 1] = pack2(t[p][0], t[p][1]);
  }
  __nv_bfloat16* dp = J.dst + row * (3 * int64_t(J.cp)) + c0;
#pragma unroll
  for (int p = 0; p < 3; ++p) *reinterpret_cast<uint4*>(dp + int64_t(p) * J.cp) = make_uint4(o[p][0], o[p][1], o[p][2], o[p][3]);
}

// Finds the split of (src, rows, cols, ld) in the arena or queues the job that makes it.
static int get_split(SplitArena& arena, SplitJobs& jobs, const float* src, int64_t rows, int cols, int64_t ld, int ones, int terms,
                     float bound, const float* bound_dev, const __nv_bfloat16** out, int* cp_out, const float** amax_out) {
  for (int i = 0; i < arena.n; ++i) {
    const SplitArena::Entry& e = arena.e[i];
    if (e.src == src && e.rows == rows && e.cols == cols && e.ld == ld && e.ones >= ones && e.terms == terms) {
      *out = e.dst;
      *cp_out = e.cp;
      *amax_out = e.amax;
      return B200PPO_OK;
    }
  }
  const int cp = pad64(cols + 1);
  const int64_t elems = split_arena_elems(rows, cols);
  if (arena.n >= SplitArena::kMaxEntries || arena.used + elems > arena.base.cap() || jobs.n >= kMaxSplitJobs) {
    set_error("three-term operand arena exhausted (%d entries, %lld of %lld elements used, %lld more asked)", arena.n,
              (long long)arena.used, (long long)arena.base.cap(), (long long)elems);
    return B200PPO_EINVAL;
  }
  __nv_bfloat16* dst = arena.base + arena.used;
  arena.used += elems;
  float* am = arena.amax + arena.n;
  *amax_out = am;
  arena.e[arena.n++] = SplitArena::Entry{src, rows, ld, cols, ones, cp, terms, dst, am};
  SplitJob& J = jobs.j[jobs.n++];
  J.src = src; J.dst = dst; J.rows = rows; J.ld = ld; J.cols = cols; J.cp = cp; J.ones = ones;
  J.terms = terms; J.amax = am;
  J.bound = bound; J.bound_dev = bound_dev;
  J.vec = (aligned16(src) && ld % 4 == 0) ? 1 : 0;
  J.unit_begin = jobs.units;
  jobs.units += rows * (cp / 8);
  *out = dst;
  *cp_out = cp;
  return B200PPO_OK;
}

bool gemm_split_applicable(const GemmGroup& g) {
  static const bool on = []() {
    const char* e = getenv("B200PPO_FP32_TC");
    return !(e != nullptr && e[0] == '0');
  }();
  if (!on || g.count == 0 || g.count > kMaxTcProblems) return false;
  double macs = 0;
  for (int i = 0; i < g.count; ++i) {
    const GemmProblem& p = g.p[i];
    if (p.C_bf16 != nullptr) return false;
    if (p.M <= 0 || p.N <= 0 || p.K <= 0) return false;
    const bool a_k = p.a_sk == 1 && p.a_sm >= p.K, a_mn = p.a_sm == 1 && p.a_sk >= p.M;
    const bool b_k = p.b_sk == 1 && p.b_sn >= p.K, b_mn = p.b_sn == 1 && p.b_sk >= p.N;
    if (!(a_k || a_mn) || !(b_k || b_mn)) return false;
    if (p.bias_grad != nullptr && !((a_mn && !a_k) && (b_mn && !b_k))) return false;  // bias gradients only off the wgrad layout
    macs += double(p.M) * p.N * p.K;
  }
  return macs >= double(1ll << 27);
}

int launch_gemm_group_split(const GemmGroup& g, SplitArena& arena, cudaStream_t st) {
  if (g.total_tiles == 0 || g.count == 0) return B200PPO_OK;
  B2_TRY(tc_init());
  const int terms = arena.terms == 2 ? 2 : 3;
  SplitJobs jobs{};
  ColsumJobs colsums{};
  TcGroup tg{};
  // N tile: 256 when the outputs are wide (the A tile is fetched once per 256 columns), 192 for the weight gradients
  // (N = in + 1 = 377 or 257 columns: two 192-wide tiles instead of three 128-wide ones)
  int maxN = 0;
  bool any_wgrad = false;
  for (int i = 0; i < g.count; ++i) {
    maxN = std::max(maxN, g.p[i].N + ((g.p[i].bias_grad != nullptr && terms == 3) ? 1 : 0));
    any_wgrad |= g.p[i].bias_grad != nullptr;
  }
  const int BN = maxN <= 128 ? 128 : ((any_wgrad && terms == 3) ? 192 : 256);
  const bool use_persist = BN >= 192;  // one CTA per SM walks the tiles; the 128-wide tiles run one per CTA
  for (int i = 0; i < g.count; ++i) {
    const GemmProblem& p = g.p[i];
    const bool a_mn = !(p.a_sk == 1 && p.a_sm >= p.K), b_mn = !(p.b_sk == 1 && p.b_sn >= p.K);
    const bool wgrad = a_mn && b_mn, fwd = !a_mn && !b_mn;
    const __nv_bfloat16 *As = nullptr, *Bs = nullptr;
    const float *a_amax = nullptr, *b_amax = nullptr;
    int a_cp = 0, b_cp = 0;
    // the arrays as stored: K-major [M or N][K], MN-major [K][M or N]; one scale per tensor
    B2_TRY(get_split(arena, jobs, p.A, a_mn ? p.K : p.M, a_mn ? p.M : p.K, a_mn ? p.a_sk : p.a_sm, (fwd && terms == 3) ? 1 : 0, terms, p.a_bound,
                     p.a_bound_dev, &As, &a_cp, &a_amax));
    B2_TRY(get_split(arena, jobs, p.B, b_mn ? p.K : p.N, b_mn ? p.N : p.K, b_mn ? p.b_sk : p.b_sn, (wgrad && terms == 3) ? 1 : 0, terms, p.b_bound,
                     p.b_bound_dev, &Bs, &b_cp, &b_amax));
    TcProblem t{};
    t.M = p.M; t.N = p.N; t.K = p.K;
    t.parts = terms; t.a_part = a_cp; t.b_part = b_cp;
    t.amax_a = a_amax; t.amax_b = b_amax;
    t.out_f32 = p.C; t.ld_f32 = p.ldc; t.split_stride = p.c_split_stride;
    t.bias_col = -1;
    t.out_scale = p.out_scale;
    t.precise = 1;
    switch (p.epilogue) {
      case EPI_STORE:
        t.epilogue = TC_EPI_STORE;
        if (p.bias_grad != nullptr && terms == 3) {  // the ones-column behind the B operand's last column
          t.N = p.N + 1;
          t.bias_col = p.N;
          t.bias_grad = p.bias_grad;
        } else if (p.bias_grad != nullptr) {
          // Two fp16 terms carry 22 bits: enough for the products, not for a bias gradient that is the small difference of
          // large sums (measured: 2.4e-4 relative on a critic bias whose terms cancel 1000 : 1).  Those are plain fp32 column
          // sums (colsum_kernel), one partial per split like the weight gradient's.
          ColsumJob& cj = colsums.j[colsums.n++];
          cj.src = p.A; cj.rows = p.K; cj.cols = p.M; cj.ld = p.a_sk;
          cj.dst = p.bias_grad; cj.splits = p.split_k; cj.split_stride = p.c_split_stride;
          cj.block_begin = colsums.blocks;
          colsums.blocks += p.split_k * ((p.M + 31) / 32);
        }
        break;
      case EPI_BIAS: t.epilogue = TC_EPI_FWD; t.act = TC_ACT_NONE; t.bias = p.bias; break;
      case EPI_BIAS_TANH: t.epilogue = TC_EPI_FWD; t.act = B200PPO_ACT_TANH; t.bias = p.bias; break;
      case EPI_BIAS_RELU: t.epilogue = TC_EPI_FWD; t.act = B200PPO_ACT_RELU; t.bias = p.bias; break;
      case EPI_BIAS_TANH_SCALE: t.epilogue = TC_EPI_FWD; t.act = TC_ACT_TANH_SCALE; t.bias = p.bias; break;
      case EPI_DTANH: t.epilogue = TC_EPI_DGRAD; t.act = B200PPO_ACT_TANH; t.aux_f32 = p.aux; t.ld_aux = p.ld_aux; break;
      case EPI_DRELU: t.epilogue = TC_EPI_DGRAD; t.act = B200PPO_ACT_RELU; t.aux_f32 = p.aux; t.ld_aux = p.ld_aux; break;
      default: set_error("gemm_split: unknown epilogue %d", p.epilogue); return B200PPO_EINVAL;
    }
    // Three-term mode: a hidden activation (forward) or a dL/dz block (dgrad) is the next GEMMs' operand — the epilogue writes
    // its terms straight into the arena (the persistent kernel's epilogue hides behind the next tile's main loop), which
    // saves the split pass over it.  (Two-term mode cannot: the scale is only known once the whole tensor exists.)
    const bool producer = p.epilogue == EPI_BIAS_TANH || p.epilogue == EPI_BIAS_RELU || p.epilogue == EPI_DTANH || p.epilogue == EPI_DRELU;
    if (use_persist && terms == 3 && producer && p.N % 16 == 0 && arena.n < SplitArena::kMaxEntries) {
      const int ocp = pad64(p.N + 1);
      const int64_t oelems = split_arena_elems(p.M, p.N);
      const int ones = (p.epilogue == EPI_BIAS_TANH || p.epilogue == EPI_BIAS_RELU) ? 1 : 0;
      bool known = false;
      for (int e = 0; e < arena.n; ++e) known |= arena.e[e].src == p.C && arena.e[e].rows == p.M && arena.e[e].cols == p.N;
      if (!known && arena.used + oelems <= arena.base.cap()) {
        __nv_bfloat16* odst = arena.base + arena.used;
        arena.used += oelems;
        arena.e[arena.n++] = SplitArena::Entry{p.C, int64_t(p.M), int64_t(p.ldc), p.N, ones, ocp, 3, odst, arena.amax};
        t.out_split = odst; t.split_cp = ocp; t.split_ones = ones;
      }
    }
    B2_TRY(tc_group_add(tg, t, TcOperand{As, terms * int64_t(a_cp), a_mn ? 1 : 0}, TcOperand{Bs, terms * int64_t(b_cp), b_mn ? 1 : 0}, BN,
                        p.split_k));
  }
  if (jobs.n > 0) {
    const unsigned blocks = unsigned((jobs.units + 255) / 256);
    if (terms == 2) {
      if (!arena.amax_zeroed) {
        B2_CUDA(cudaMemsetAsync(arena.amax, 0, SplitArena::kMaxEntries * sizeof(float), st));
        arena.amax_zeroed = true;
      }
      SplitJobs measure{};  // the operands nobody gave a bound for
      for (int i = 0; i < jobs.n; ++i) {
        const SplitJob& J = jobs.j[i];
        if (J.bound_dev != nullptr || J.bound > 0.f) continue;
        SplitJob& Mj = measure.j[measure.n++];
        Mj = J;
        Mj.unit_begin = measure.units;
        measure.units += J.rows * (J.cp / 8);
      }
      if (measure.n > 0) {
        absmax_kernel<<<unsigned((measure.units + 255) / 256), 256, 0, st>>>(measure);
        B2_LAUNCH_CHECK();
      }
    }
    B2_CUDA(launch_pdl(split3_kernel, dim3(blocks), dim3(256), 0, st, jobs));
    B2_LAUNCH_CHECK();
  }
  // debug: B200PPO_SPLIT_TRACE=<n> prints phase marks (cycles) of every 37th CTA of the n-th launch
  static const char* trace_env = getenv("B200PPO_SPLIT_TRACE");
  static int calls = 0;
  DevBuf<long long> trace;  // declared before `dump`, so freed after it has printed
  if (trace_env != nullptr && ++calls == atoi(trace_env)) {
    B2_TRY(trace.alloc(64 * 8, true));
    tg.trace = trace;
  }
  struct TraceDump {
    long long* t; cudaStream_t st; int tiles; bool persistent = false;
    ~TraceDump() {
      if (t == nullptr) return;
      cudaStreamSynchronize(st);
      long long h[64 * 8];
      cudaMemcpy(h, t, sizeof(h), cudaMemcpyDeviceToHost);
      if (persistent) {  // tc_persist_kernel: the tiles of CTA 0 (slot 3 = epilogue enters, before it waits for the accumulator)
        const long long t0 = h[5];
        fprintf(stderr, "persistent split GEMM, %d tiles, CTA 0: tile | producer first, last load | issuer: accumulator, first operands, last MMA | epilogue: enters, done\n", tiles);
        for (int i = 0; i < 64 && h[i * 8 + 5] != 0; ++i)
          fprintf(stderr, "  %2d | %7lld %7lld | %7lld %7lld %7lld | %7lld %7lld\n", i, h[i * 8 + 5] - t0, h[i * 8 + 6] - t0, h[i * 8] - t0,
                  h[i * 8 + 1] - t0, h[i * 8 + 2] - t0, h[i * 8 + 3] - t0, h[i * 8 + 4] - t0);
        return;
      }
      long long t0 = h[0];
      for (int i = 0; i < 64; ++i) if (h[i * 8] != 0 && h[i * 8] < t0) t0 = h[i * 8];
      fprintf(stderr, "split GEMM launch, %d CTAs: cta | sm | entry, set-up done, first operands, last MMA issued, epilogue done (warp 2), end  (cycles since the first entry; clocks of different SMs are not aligned)\n", tiles);
      for (int i = 0; i < 64 && h[i * 8] != 0; ++i)
        fprintf(stderr, "  %4d | %3lld | %7lld %7lld %7lld %7lld %7lld %7lld   (own: set-up %lld, to first operands %lld, main loop %lld, epilogue %lld)\n", i * 37, h[i * 8 + 7],
                h[i * 8] - t0, h[i * 8 + 1] - t0, h[i * 8 + 2] - t0, h[i * 8 + 3] - t0, h[i * 8 + 5] - t0, h[i * 8 + 6] - t0,
                h[i * 8 + 1] - h[i * 8], h[i * 8 + 2] - h[i * 8 + 1], h[i * 8 + 3] - h[i * 8 + 2], h[i * 8 + 5] - h[i * 8 + 3]);
    }
  } dump{trace, st, tg.total_tiles};
  // forward / dgrad: two CTAs per SM (two-stage rings); weight gradients: one CTA with the deep ring — measured, profiles/README.md
  const bool two = !any_wgrad;
  if (colsums.n > 0) {
    colsum_kernel<<<unsigned(colsums.blocks), 256, 0, st>>>(colsums);
    B2_LAUNCH_CHECK();
  }
  if (use_persist) {
    dump.persistent = true;
    return launch_tc_persist(tg, BN, st);
  }
  return launch_tc_group(tg, BN, st, nullptr, two);
}

}  // namespace b200ppo

namespace b200ppo {
int launch_absmax(const float* src, int64_t rows, int cols, int64_t ld, float* out, cudaStream_t st) {
  if (rows <= 0 || cols <= 0) return B200PPO_OK;
  B2_CUDA(cudaMemsetAsync(out, 0, sizeof(float), st));
  SplitJobs jobs{};
  SplitJob& J = jobs.j[jobs.n++];
  J.src = src; J.rows = rows; J.ld = ld; J.cols = cols; J.cp = (cols + 1 + 63) / 64 * 64; J.ones = 0;
  J.vec = (aligned16(src) && ld % 4 == 0) ? 1 : 0;
  J.amax = out;
  jobs.units = rows * (J.cp / 8);
  absmax_kernel<<<unsigned((jobs.units + 255) / 256), 256, 0, st>>>(jobs);
  B2_LAUNCH_CHECK();
  return B200PPO_OK;
}
}  // namespace b200ppo

// ---- test hook --------------------------------------------------------------------------------------------------------------
using namespace b200ppo;

extern "C" B2_EXPORT int b200ppo_debug_gemm_split(const float* A, const float* B, float* C, float* bias_grad, int32_t M, int32_t N,
                                                  int32_t K, int32_t a_mn_major, int32_t b_mn_major, int32_t split_k,
                                                  b200ppo_stream stream) {
  B2_CHECK_ARG(A && B && C && M > 0 && N > 0 && K > 0 && split_k >= 1, "b200ppo_debug_gemm_split: bad argument");
  B2_CHECK_ARG(bias_grad == nullptr || (a_mn_major && b_mn_major), "b200ppo_debug_gemm_split: bias_grad needs both operands MN-major");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  SplitArena arena;
  if (const char* e = getenv("B200PPO_DEBUG_SPLIT_TERMS")) arena.terms = atoi(e) == 2 ? 2 : 3;  // read per call (tests switch it)
  const int64_t need = split_arena_elems(a_mn_major ? K : M, a_mn_major ? M : K) + split_arena_elems(b_mn_major ? K : N, b_mn_major ? N : K) +
                       4 * (int64_t(M) + K + 2048);
  B2_TRY(split_arena_reserve(arena, need));
  const int64_t mn = int64_t(M) * N, stride = (mn + M + 3) / 4 * 4;
  DevBuf<float> part;
  B2_TRY(part.alloc(int64_t(split_k) * stride));
  GemmGroup g{};
  GemmProblem p{};
  p.A = A; p.B = B; p.C = part; p.ldc = N;
  p.M = M; p.N = N; p.K = K;
  p.a_sm = a_mn_major ? 1 : K; p.a_sk = a_mn_major ? M : 1;
  p.b_sn = b_mn_major ? 1 : K; p.b_sk = b_mn_major ? N : 1;
  p.epilogue = EPI_STORE;
  p.c_split_stride = stride;
  if (bias_grad != nullptr) p.bias_grad = part + mn;
  gemm_group_add(g, p, 64, 64, split_k);
  int rc = launch_gemm_group_split(g, arena, st);
  if (rc == B200PPO_OK) {
    sum_splits_kernel<<<unsigned((mn + 255) / 256), 256, 0, st>>>(part, split_k, stride, mn, C);
    count_launch();
    if (bias_grad != nullptr) {
      sum_splits_kernel<<<unsigned((M + 255) / 256), 256, 0, st>>>(part + mn, split_k, stride, M, bias_grad);
      count_launch();
    }
  }
  cudaStreamSynchronize(st);
  if (rc != B200PPO_OK) return rc;
  B2_CUDA(cudaGetLastError());
  return B200PPO_OK;
}
