// K5 — fused Adam (one launch for every parameter of actor and critic).
//
// replaces: torch.optim.Adam.step(), single-tensor CPU path (`_single_tensor_adam`, no amsgrad, no weight
//           decay), called at src/entities/algorithms/ppo.py:122,135 for the optimisers built at
//           src/entities/agents/ppo_agent.py:15-18.
//
// The reduction of the split-K weight-gradient partials is fused into the optimiser: the kernel sums
// `n_partials` partial gradients in index order (deterministic), then applies the reference's update
//   m = m + (1-b1)(g - m);  v = v*b2 + (1-b2)*g*g;  p += -(lr/bc1) * m / (sqrt(v)/sqrt(bc2) + eps)
// with the scalar factors computed in double on the host exactly as the Python code does.
// Algorithmic bytes: 28 per parameter (read p,g,m,v; write p,m,v) when n_partials == 1.
#include <math.h>

#include "adam.cuh"

namespace b200ppo {

__device__ __forceinline__ void adam_update(float& p, float g, float& m, float& v, const AdamScalars& s) {
  m = __fadd_rn(m, __fmul_rn(s.one_minus_b1, __fsub_rn(g, m)));               // exp_avg.lerp_(grad, 1-beta1)
  v = __fadd_rn(__fmul_rn(v, s.b2), __fmul_rn(__fmul_rn(s.one_minus_b2, g), g));  // mul_(b2).addcmul_(g,g,1-b2)
  const float denom = __fadd_rn(__fdiv_rn(__fsqrt_rn(v), s.bc2_sqrt), s.eps);
  p = __fadd_rn(p, __fmul_rn(s.neg_step_size, __fdiv_rn(m, denom)));          // addcdiv_(m, denom, -step_size)
}

__global__ void __launch_bounds__(256)
adam_kernel(float* __restrict__ params, const float* __restrict__ grads, int n_partials, int64_t partial_stride,
            float* __restrict__ exp_avg, float* __restrict__ exp_avg_sq, int64_t n, int64_t seg_split,
            AdamScalars s0, AdamScalars s1, float* __restrict__ grad_out) {
  const int64_t tid = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t nthreads = int64_t(gridDim.x) * blockDim.x;
  const int64_t n4 = n >> 2;
  for (int64_t i = tid; i < n4; i += nthreads) {
    float4 g = *reinterpret_cast<const float4*>(grads + 4 * i);
    for (int k = 1; k < n_partials; ++k) {
      const float4 h = *reinterpret_cast<const float4*>(grads + k * partial_stride + 4 * i);
      g.x += h.x; g.y += h.y; g.z += h.z; g.w += h.w;
    }
    float4 p = *reinterpret_cast<float4*>(params + 4 * i);
    float4 m = *reinterpret_cast<float4*>(exp_avg + 4 * i);
    float4 v = *reinterpret_cast<float4*>(exp_avg_sq + 4 * i);
    const int64_t e = 4 * i;
    adam_update(p.x, g.x, m.x, v.x, e + 0 < seg_split ? s0 : s1);
    adam_update(p.y, g.y, m.y, v.y, e + 1 < seg_split ? s0 : s1);
    adam_update(p.z, g.z, m.z, v.z, e + 2 < seg_split ? s0 : s1);
    adam_update(p.w, g.w, m.w, v.w, e + 3 < seg_split ? s0 : s1);
    *reinterpret_cast<float4*>(params + 4 * i) = p;
    *reinterpret_cast<float4*>(exp_avg + 4 * i) = m;
    *reinterpret_cast<float4*>(exp_avg_sq + 4 * i) = v;
    if (grad_out != nullptr) *reinterpret_cast<float4*>(grad_out + 4 * i) = g;
  }
  for (int64_t e = 4 * n4 + tid; e < n; e += nthreads) {  // tail (n % 4)
    float g = grads[e];
    for (int k = 1; k < n_partials; ++k) g += grads[k * partial_stride + e];
    float p = params[e], m = exp_avg[e], v = exp_avg_sq[e];
    adam_update(p, g, m, v, e < seg_split ? s0 : s1);
    params[e] = p; exp_avg[e] = m; exp_avg_sq[e] = v;
    if (grad_out != nullptr) grad_out[e] = g;
  }
}

// g += grads[k][4i .. 4i+3] for k in [k0, n_partials), in index order (deterministic) — with the loads of up to eight
// partials ISSUED before the first add.  Written as load-add-load-add (the first version) the compiler kept that order,
// and the 9 split-K partials of the bench shape cost 9 dependent L2 round trips: 47 % of this kernel's stall samples sat
// on those adds (profiles/r02_ncu_chain_wgrad_B32768.csv, 14.7 us for 329 k parameters).
__device__ __forceinline__ void add_partials(float4& g, const float* __restrict__ grads, int k0, int n_partials, int64_t partial_stride, int64_t i) {
  constexpr int NB = 8;  // + the first partial read by the caller = the 9 of the bench shape in one round; 85 registers keep the grid in one wave
  for (; k0 < n_partials; k0 += NB) {
    float4 h[NB];
#pragma unroll
    for (int j = 0; j < NB; ++j)
      if (k0 + j < n_partials) h[j] = __ldg(reinterpret_cast<const float4*>(grads + int64_t(k0 + j) * partial_stride + 4 * i));
#pragma unroll
    for (int j = 0; j < NB; ++j)
      if (k0 + j < n_partials) { g.x += h[j].x; g.y += h[j].y; g.z += h[j].z; g.w += h[j].w; }
  }
}

struct CastTable {
  int64_t begin[2 * B200PPO_MAX_LAYERS], end[2 * B200PPO_MAX_LAYERS];  // element range of each matrix in the flat buffer
  __nv_bfloat16* dst[2 * B200PPO_MAX_LAYERS];
  int in[2 * B200PPO_MAX_LAYERS], pitch[2 * B200PPO_MAX_LAYERS];
  int count;
};

// Block-level finish of the fused-epilogue loss partials: s_lc[0] = sum surrogate, [1] = sum huber, [2+j] = logstd grads.
__device__ __forceinline__ void combine_losses(const LossCombine& lc, float* s_lc, float* s_scr) {
  const int tid = threadIdx.x;
  const float s = combine_partials<256>(lc.partials, unsigned(lc.n_cta), 2 + lc.act_dim, tid, s_scr);
  if (tid < 2 + lc.act_dim) s_lc[tid] = tid < 2 ? s : s - lc.ent_coef * lc.rank_share / float(lc.act_dim);
  if (tid == 0 && lc.losses_out != nullptr) {
    float ent = 0.f;  // mean over [B, A] of 0.5 + 0.5 log(2 pi) + log sigma_j
    for (int j = 0; j < lc.act_dim; ++j) ent += 0.5f + 0.91893853320467274178f + logf(expf(lc.logstd[j]));
    ent /= float(lc.act_dim);
    lc.losses_out[0] = -s * lc.inv_global_batch - lc.ent_coef * ent * lc.rank_share;
  }
  if (tid == 1 && lc.losses_out != nullptr) lc.losses_out[1] = s * lc.inv_global_batch;
  __syncthreads();
}

// Flag exchange of the peer-memory all-reduce: tell every peer that this rank's buffer of exchange `seq` is complete
// (the kernel that wrote it finished before this one started), then wait until every peer has said the same.
// Returns false (for the whole block) when a peer did not show up within ps.timeout_cycles: the caller must then NOT
// touch the parameters — whatever sits in that peer's exchange buffer is an older or half-written gradient — and the
// error flag tells the host (b200ppo_poll_error), which fails the call instead of letting the replicas drift apart.
__device__ __forceinline__ bool peer_exchange_barrier(const PeerSrc& ps) {
  const int q = threadIdx.x;
  int timed_out = 0;
  if (q < ps.world && q != ps.rank) {
    if (blockIdx.x == 0) {
      if (ps.local_out != nullptr) {  // fused reduce: this rank's buffer is complete once every block of this grid has said so
        const long long t0 = clock64();
        unsigned d;
        do {
          asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(d) : "l"(ps.done_counter) : "memory");
        } while (int(d - ps.done_target) < 0 && clock64() - t0 <= ps.timeout_cycles);
      }
      __threadfence_system();
      asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(ps.flags_peer[q] + ps.rank), "r"(ps.seq) : "memory");
    }
    const long long t0 = clock64();
    unsigned v;
    do {
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(ps.flags_local + q) : "memory");
      if (clock64() - t0 > ps.timeout_cycles) {  // a peer died or stalled: flag the error instead of hanging the GPU
        if (ps.err != nullptr) atomicMax(ps.err, B200PPO_ERRFLAG_PEER_TIMEOUT);
        timed_out = 1;
        break;
      }
    } while (int(v - ps.seq) < 0);
  }
  return __syncthreads_or(timed_out) == 0;
}

__device__ __forceinline__ float4 ld_peer4(const float* p) {  // peer memory: never through a stale L1 line
  float4 r;
  asm volatile("ld.volatile.global.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w) : "l"(p) : "memory");
  return r;
}

// PEERS: the gradient is the rank-ordered sum of every rank's exchange buffer (multi-GPU); kept out of the single-GPU
// instantiation, whose register count (64) sets its occupancy.
template <bool PEERS>
__global__ void __launch_bounds__(256, 3)
adam_cast_kernel(float* __restrict__ params, const float* __restrict__ grads, int n_partials, int64_t partial_stride,
                 float* __restrict__ exp_avg, float* __restrict__ exp_avg_sq, int64_t n, int64_t seg_split, AdamScalars s0,
                 AdamScalars s1, const __grid_constant__ CastTable ct, const __grid_constant__ LossCombine lc,
                 const __grid_constant__ PeerSrc ps) {
  __shared__ float s_lc[64];
  __shared__ float s_scr[256];
  pdl_wait_then_release();  // the gradient partials come from the kernel right before this one (common.cuh, PDL)
  const int64_t tid = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t nthreads = int64_t(gridDim.x) * blockDim.x;
  const int64_t n4 = n >> 2;  // the flat buffer is padded to a multiple of 32 elements
  // the block whose grid-stride chunks contain actor_logstd finishes the loss partials (before anything is updated)
  const bool lc_owner = lc.partials != nullptr && int64_t(blockIdx.x) == ((lc.logstd_off >> 2) / blockDim.x) % gridDim.x;
  if (lc_owner) combine_losses(lc, s_lc, s_scr);
  float4 g_local = make_float4(0.f, 0.f, 0.f, 0.f);
  bool fused = false;
  if constexpr (PEERS) {
    fused = ps.local_out != nullptr;
    if (fused) {
      // Fused reduce (one element per thread): this rank's split-K partials are summed HERE, in index order, into its
      // exchange buffer — the separate reduction launch in front of the exchange (11-13 us per minibatch) is gone.  Every
      // block counts itself done; block 0 raises this rank's flag at the peers only when all have (see the barrier).
      if (tid < n4) {
        g_local = __ldg(reinterpret_cast<const float4*>(grads + 4 * tid));
        add_partials(g_local, grads, 1, n_partials, partial_stride, tid);
        if (lc_owner && 4 * tid + 3 >= lc.logstd_off && 4 * tid < lc.logstd_off + lc.act_dim) {
          const int64_t r = 4 * tid - lc.logstd_off;
          if (r + 0 >= 0 && r + 0 < lc.act_dim) g_local.x = s_lc[2 + r + 0];
          if (r + 1 >= 0 && r + 1 < lc.act_dim) g_local.y = s_lc[2 + r + 1];
          if (r + 2 >= 0 && r + 2 < lc.act_dim) g_local.z = s_lc[2 + r + 2];
          if (r + 3 >= 0 && r + 3 < lc.act_dim) g_local.w = s_lc[2 + r + 3];
        }
        *reinterpret_cast<float4*>(ps.local_out + 4 * tid) = g_local;
      }
      __threadfence();
      __syncthreads();
      if (threadIdx.x == 0) atomicAdd(ps.done_counter, 1u);
    }
    if (!peer_exchange_barrier(ps)) return;  // no update from stale peer data; the host sees the flag
    if (blockIdx.x == 0 && threadIdx.x < 2 && ps.losses_out != nullptr) {
      float l = 0.f;
      for (int r = 0; r < ps.world; ++r) {
        float t;
        asm volatile("ld.volatile.global.f32 %0, [%1];" : "=f"(t) : "l"(ps.src[r] + n + threadIdx.x) : "memory");
        l += t;
      }
      ps.losses_out[threadIdx.x] = l;
    }
  }
  for (int64_t i = tid; i < n4; i += nthreads) {
    // every load of this element is issued before the first use: the kernel is one L2 round trip deep, not n_partials
    const float4 p0 = *reinterpret_cast<float4*>(params + 4 * i);
    const float4 m0 = *reinterpret_cast<float4*>(exp_avg + 4 * i);
    const float4 v0 = *reinterpret_cast<float4*>(exp_avg_sq + 4 * i);
    float4 g;
    if constexpr (PEERS) {  // every rank's buffer, all loads in flight, summed in rank order
      float4 h[kMaxPeers];
#pragma unroll
      for (int r = 0; r < kMaxPeers; ++r)
        if (r < ps.world) h[r] = (fused && r == ps.rank) ? g_local : ld_peer4(ps.src[r] + 4 * i);  // own sum: still in the register
      g = h[0];
#pragma unroll
      for (int r = 1; r < kMaxPeers; ++r)
        if (r < ps.world) { g.x += h[r].x; g.y += h[r].y; g.z += h[r].z; g.w += h[r].w; }
    } else {
      g = *reinterpret_cast<const float4*>(grads + 4 * i);
    }
    if constexpr (!PEERS) add_partials(g, grads, 1, n_partials, partial_stride, i);
    if (!PEERS && lc_owner && 4 * i + 3 >= lc.logstd_off && 4 * i < lc.logstd_off + lc.act_dim) {
      const int64_t r = 4 * i - lc.logstd_off;
      if (r + 0 >= 0 && r + 0 < lc.act_dim) g.x = s_lc[2 + r + 0];
      if (r + 1 >= 0 && r + 1 < lc.act_dim) g.y = s_lc[2 + r + 1];
      if (r + 2 >= 0 && r + 2 < lc.act_dim) g.z = s_lc[2 + r + 2];
      if (r + 3 >= 0 && r + 3 < lc.act_dim) g.w = s_lc[2 + r + 3];
    }
    float4 p = p0, m = m0, v = v0;
    const int64_t e = 4 * i;
    adam_update(p.x, g.x, m.x, v.x, e + 0 < seg_split ? s0 : s1);
    adam_update(p.y, g.y, m.y, v.y, e + 1 < seg_split ? s0 : s1);
    adam_update(p.z, g.z, m.z, v.z, e + 2 < seg_split ? s0 : s1);
    adam_update(p.w, g.w, m.w, v.w, e + 3 < seg_split ? s0 : s1);
    *reinterpret_cast<float4*>(params + 4 * i) = p;
    *reinterpret_cast<float4*>(exp_avg + 4 * i) = m;
    *reinterpret_cast<float4*>(exp_avg_sq + 4 * i) = v;
    // bf16 shadow copies of the matrix this float4 belongs to (tensors start on 32-element boundaries, so a float4
    // never straddles two tensors; it may straddle two rows when `in` is not a multiple of 4)
    int k = -1;
#pragma unroll 1
    for (int c = 0; c < ct.count; ++c)
      if (e >= ct.begin[c] && e < ct.end[c]) k = c;
    if (k >= 0 && (ct.in[k] & 3) == 0 && (ct.pitch[k] & 3) == 0 && e + 3 < ct.end[k]) {
      // whole float4 inside one row (rows are multiples of 4 wide): one 32-bit division, one 8-byte store
      const uint32_t in = uint32_t(ct.in[k]), rel = uint32_t(e - ct.begin[k]);
      const uint32_t o = rel / in, c2 = rel - o * in;
      const __nv_bfloat162 lo = __floats2bfloat162_rn(p.x, p.y), hi = __floats2bfloat162_rn(p.z, p.w);
      uint2 w;
      w.x = *reinterpret_cast<const uint32_t*>(&lo);
      w.y = *reinterpret_cast<const uint32_t*>(&hi);
      *reinterpret_cast<uint2*>(ct.dst[k] + int64_t(o) * ct.pitch[k] + c2) = w;
    } else if (k >= 0) {
      const float pv[4] = {p.x, p.y, p.z, p.w};
      const int in = ct.in[k];
      const int64_t rel = e - ct.begin[k];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (e + j >= ct.end[k]) break;
        const int o = int((rel + j) / in), c2 = int((rel + j) - int64_t(o) * in);
        ct.dst[k][int64_t(o) * ct.pitch[k] + c2] = __float2bfloat16_rn(pv[j]);
      }
    }
  }
}

// Sum partials only (used before the gradient exchange between ranks and by the grads-only entry point).
// float4 per thread, partials added in index order with four loads in flight (n is padded to a multiple of 4 by the
// callers that pass aligned buffers; the scalar loop covers everything else).
__global__ void __launch_bounds__(256)
reduce_partials_kernel(const float* __restrict__ grads, int n_partials, int64_t partial_stride, int64_t n,
                       float* __restrict__ out, const __grid_constant__ LossCombine lc, int vec4) {
  __shared__ float s_lc[64];
  __shared__ float s_scr[256];
  pdl_wait_then_release();
  const int64_t tid = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t nthreads = int64_t(gridDim.x) * blockDim.x;
  const int64_t n4 = vec4 ? (n >> 2) : 0;
  const bool lc_owner = lc.partials != nullptr && int64_t(blockIdx.x) == (vec4 ? ((lc.logstd_off >> 2) / blockDim.x) % gridDim.x
                                                                               : (lc.logstd_off / blockDim.x) % gridDim.x);
  if (lc_owner) combine_losses(lc, s_lc, s_scr);
  for (int64_t i = tid; i < n4; i += nthreads) {
    float4 g = *reinterpret_cast<const float4*>(grads + 4 * i);
    add_partials(g, grads, 1, n_partials, partial_stride, i);
    if (lc_owner && 4 * i + 3 >= lc.logstd_off && 4 * i < lc.logstd_off + lc.act_dim) {
      const int64_t r = 4 * i - lc.logstd_off;
      if (r + 0 >= 0 && r + 0 < lc.act_dim) g.x = s_lc[2 + r + 0];
      if (r + 1 >= 0 && r + 1 < lc.act_dim) g.y = s_lc[2 + r + 1];
      if (r + 2 >= 0 && r + 2 < lc.act_dim) g.z = s_lc[2 + r + 2];
      if (r + 3 >= 0 && r + 3 < lc.act_dim) g.w = s_lc[2 + r + 3];
    }
    *reinterpret_cast<float4*>(out + 4 * i) = g;
  }
  for (int64_t e = 4 * n4 + tid; e < n; e += nthreads) {
    float g = grads[e];
    for (int k = 1; k < n_partials; ++k) g += grads[k * partial_stride + e];
    if (lc_owner && e >= lc.logstd_off && e < lc.logstd_off + lc.act_dim) g = s_lc[2 + (e - lc.logstd_off)];
    out[e] = g;
  }
}

AdamScalars make_adam_scalars(double lr, double beta1, double beta2, double eps, int64_t step) {
  AdamScalars s;
  const double bc1 = 1.0 - pow(beta1, double(step));
  const double bc2 = 1.0 - pow(beta2, double(step));
  s.one_minus_b1 = float(1.0 - beta1);
  s.b2 = float(beta2);
  s.one_minus_b2 = float(1.0 - beta2);
  s.bc2_sqrt = float(sqrt(bc2));
  s.eps = float(eps);
  s.neg_step_size = float(-(lr / bc1));
  return s;
}

static inline unsigned ew_grid(int64_t work_items) {
  int64_t blocks = (work_items + 255) / 256;
  const int64_t cap = int64_t(num_sms()) * 8;
  if (blocks > cap) blocks = cap;
  return unsigned(blocks < 1 ? 1 : blocks);
}

int launch_adam(float* params, const float* grads, int n_partials, int64_t partial_stride, float* exp_avg,
                float* exp_avg_sq, int64_t n, int64_t seg_split, const AdamScalars& s0, const AdamScalars& s1,
                float* grad_out, cudaStream_t st) {
  if (n == 0) return B200PPO_OK;
  adam_kernel<<<ew_grid((n + 3) / 4), 256, 0, st>>>(params, grads, n_partials, partial_stride, exp_avg, exp_avg_sq, n,
                                                    seg_split, s0, s1, grad_out);
  B2_LAUNCH_CHECK();
  return B200PPO_OK;
}

int adam_cast_grid(int64_t n) { return int(ew_grid(n / 4)); }

int launch_adam_cast(float* params, const float* grads, int n_partials, int64_t partial_stride, float* exp_avg,
                     float* exp_avg_sq, int64_t n, int64_t seg_split, const AdamScalars& s0, const AdamScalars& s1,
                     const WeightCastGroup& casts, const LossCombine& lc, cudaStream_t st, const PeerSrc* peers) {
  if (n == 0) return B200PPO_OK;
  const PeerSrc no_peers{};
  B2_CHECK_ARG(lc.partials == nullptr || (lc.act_dim + 2 <= 64 && lc.logstd_off % 4 == 0), "loss combine: act_dim <= 62");
  B2_CHECK_ARG(n % 4 == 0, "fused Adam + cast expects the padded flat parameter buffer");
  CastTable ct{};
  ct.count = casts.count;
  for (int k = 0; k < casts.count; ++k) {
    const WeightCast& w = casts.w[k];
    ct.begin[k] = w.src - params;
    ct.end[k] = ct.begin[k] + int64_t(w.out) * w.in;
    B2_CHECK_ARG(ct.begin[k] >= 0 && ct.end[k] <= n, "weight cast source outside the parameter buffer");
    ct.dst[k] = w.dst;
    ct.in[k] = w.in; ct.pitch[k] = w.pitch;
  }
  B2_CHECK_ARG(peers == nullptr || peers->local_out == nullptr || int64_t(ew_grid(n / 4)) * 256 >= n / 4,
               "fused reduce + exchange: one element per thread");
  if (peers != nullptr && peers->world > 0)
    B2_CUDA(launch_pdl(adam_cast_kernel<true>, dim3(ew_grid(n / 4)), dim3(256), 0, st, params, grads, n_partials, partial_stride, exp_avg,
                       exp_avg_sq, n, seg_split, s0, s1, ct, lc, *peers));
  else
    B2_CUDA(launch_pdl(adam_cast_kernel<false>, dim3(ew_grid(n / 4)), dim3(256), 0, st, params, grads, n_partials, partial_stride, exp_avg,
                       exp_avg_sq, n, seg_split, s0, s1, ct, lc, no_peers));
  B2_LAUNCH_CHECK();
  return B200PPO_OK;
}

int launch_reduce_partials(const float* grads, int n_partials, int64_t partial_stride, int64_t n, float* out,
                           cudaStream_t st, const LossCombine* lc) {
  if (n == 0) return B200PPO_OK;
  const LossCombine none{};
  const int vec4 = (n % 4 == 0 && partial_stride % 4 == 0 && aligned16(grads) && aligned16(out) && (lc == nullptr || lc->logstd_off % 4 == 0)) ? 1 : 0;
  B2_CUDA(launch_pdl(reduce_partials_kernel, dim3(ew_grid(vec4 ? n / 4 : n)), dim3(256), 0, st, grads, n_partials, partial_stride, n, out,
                     lc ? *lc : none, vec4));
  B2_LAUNCH_CHECK();
  return B200PPO_OK;
}

// Polyak averaging of a flat parameter buffer: target = target * (1 - tau) + source * tau.
// replaces: soft_update (src/entities/algorithms/soft_actor_critic.py:12-14), one launch for every tensor of both
// Q networks.  The two products and the sum are rounded separately, like the three ATen ops of the reference.
// Algorithmic bytes: 12 per parameter.
__global__ void __launch_bounds__(256)
polyak_kernel(float* __restrict__ target, const float* __restrict__ source, int64_t n, float one_minus_tau, float tau) {
  const int64_t tid = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  const int64_t nthreads = int64_t(gridDim.x) * blockDim.x;
  const int64_t n4 = ((reinterpret_cast<uintptr_t>(target) | reinterpret_cast<uintptr_t>(source)) & 15u) == 0 ? (n >> 2) : 0;
  for (int64_t i = tid; i < n4; i += nthreads) {
    float4 t = ldg_stream4(target + 4 * i);
    const float4 s = ldg_stream4(source + 4 * i);
    t.x = __fadd_rn(__fmul_rn(t.x, one_minus_tau), __fmul_rn(s.x, tau));
    t.y = __fadd_rn(__fmul_rn(t.y, one_minus_tau), __fmul_rn(s.y, tau));
    t.z = __fadd_rn(__fmul_rn(t.z, one_minus_tau), __fmul_rn(s.z, tau));
    t.w = __fadd_rn(__fmul_rn(t.w, one_minus_tau), __fmul_rn(s.w, tau));
    stg_stream4(target + 4 * i, t);
  }
  for (int64_t e = 4 * n4 + tid; e < n; e += nthreads)
    target[e] = __fadd_rn(__fmul_rn(target[e], one_minus_tau), __fmul_rn(source[e], tau));
}

}  // namespace b200ppo

using namespace b200ppo;

extern "C" B2_EXPORT int b200ppo_polyak_update(float* target, const float* source, int64_t n, double tau, b200ppo_stream stream) {
  B2_CHECK_ARG(target && source && n >= 0, "b200ppo_polyak_update: bad argument");
  if (n == 0) return B200PPO_OK;
  polyak_kernel<<<ew_grid((n + 3) / 4), 256, 0, static_cast<cudaStream_t>(stream)>>>(target, source, n, float(1.0 - tau), float(tau));
  B2_LAUNCH_CHECK();
  return B200PPO_OK;
}

extern "C" B2_EXPORT int b200ppo_adam_step(float* params, const float* grads, int32_t n_partials, int64_t partial_stride,
                                 float* exp_avg, float* exp_avg_sq, int64_t n, double lr, double beta1, double beta2,
                                 double eps, int64_t step, b200ppo_stream stream) {
  B2_CHECK_ARG(params && grads && exp_avg && exp_avg_sq, "b200ppo_adam_step: null pointer");
  B2_CHECK_ARG(n >= 0 && n_partials >= 1 && step >= 1, "b200ppo_adam_step: bad n/n_partials/step");
  B2_CHECK_ARG(aligned16(params) && aligned16(grads) && aligned16(exp_avg) && aligned16(exp_avg_sq) &&
                   (n_partials == 1 || partial_stride % 4 == 0),
               "b200ppo_adam_step: buffers must be 16-byte aligned");
  const AdamScalars s = make_adam_scalars(lr, beta1, beta2, eps, step);
  return launch_adam(params, grads, n_partials, partial_stride, exp_avg, exp_avg_sq, n, n, s, s, nullptr,
                     static_cast<cudaStream_t>(stream));
}
