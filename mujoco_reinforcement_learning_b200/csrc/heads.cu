// Fused output layers + losses + first backward step of the actor-critic pair.
//
// replaces, in ONE kernel per minibatch:
//   * the last Linear of the actor (+ output_max_value * tanh) and of the critic
//     (src/models/linear/actor.py:25-30, src/models/critic.py:22-25),
//   * Normal.log_prob(...).sum(1), entropy, ratio / clamp / min surrogate and Huber loss with their autograd
//     seeds (src/entities/algorithms/ppo.py:113-132; the math: ppo_math.cuh),
//   * the dgrad of those last Linears through the hidden activation: dZ_hidden = (dZ_out W_out) * act'(H).
// The output layers are tall-skinny (N = act_dim <= 32 and N = 1): GEMV-shaped work that would leave a GEMM tile
// ~90% empty, so a warp owns a sample row instead: lanes split the hidden dimension (coalesced 128-bit loads of
// the row), W_out lives in shared memory, the act_dim dot products are butterfly-reduced, the loss terms are
// computed on lanes [0, act_dim) and dZ_hidden is written back row-coalesced.  Loss sums and the logstd gradient are
// reduced in a fixed order (deterministic).
#include <algorithm>

#include "heads.cuh"

namespace b200ppo {

constexpr int kHeadsWarps = 8;
constexpr int kHeadsThreads = kHeadsWarps * 32;
constexpr int kMaxChunk = 8;  // hidden width <= 32 lanes * 4 floats * kMaxChunk = 1024 (kernel is templated on the
                              // chunk count actually needed so a 256-wide layer keeps 16 registers of row data, not 64)

__device__ __forceinline__ float act_deriv(float h, int act) { return act == B200PPO_ACT_TANH ? 1.f - h * h : (h > 0.f ? 1.f : 0.f); }

template <int NCHUNK>
__global__ void __launch_bounds__(kHeadsThreads) heads_fused_kernel(const __grid_constant__ HeadsArgs a) {
  extern __shared__ __align__(16) float smem[];
  const int A = a.act_dim, Ha = a.hid_a, Hc = a.hid_c;
  float* s_w3a = smem;                 // [A][Ha]
  float* s_w3c = s_w3a + A * Ha;       // [Hc]
  float* s_red = s_w3c + Hc;           // [kHeadsWarps][2 + 32], reused (>= kHeadsThreads floats) by the final combine
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  {  // weights -> smem: 128-bit loads, unrolled so the L2 round trips overlap instead of serialising on the store
    const int n4 = (A * Ha) >> 2;
    const float4* src = reinterpret_cast<const float4*>(a.w3a);
    float4* dst = reinterpret_cast<float4*>(s_w3a);
#pragma unroll 6
    for (int i = tid; i < n4; i += kHeadsThreads) dst[i] = __ldg(src + i);
    for (int i = tid; i < (Hc >> 2); i += kHeadsThreads) reinterpret_cast<float4*>(s_w3c)[i] = __ldg(reinterpret_cast<const float4*>(a.w3c) + i);
  }
  __syncthreads();

  // per-lane constants of action dimension j = lane
  const bool jl = lane < A;
  float logsig = 0.f, inv_var = 0.f, two_var = 1.f, b3a = 0.f;
  if (jl) {
    const PpoSigma c = ppo_sigma(__ldg(a.logstd + lane));
    logsig = c.logsig; inv_var = c.inv_var; two_var = c.two_var;
    b3a = __ldg(a.b3a + lane);
  }
  const float b3c = __ldg(a.b3c);
  const int nca = (Ha + 127) / 128, ncc = (Hc + 127) / 128;

  float acc_surr = 0.f, acc_hub = 0.f, acc_dl = 0.f;  // acc_dl: lane j accumulates d loss / d logstd_j
  const int64_t row_stride = int64_t(gridDim.x) * kHeadsWarps;
  for (int64_t b = int64_t(blockIdx.x) * kHeadsWarps + warp; b < a.batch; b += row_stride) {
    // ---- actor output layer: z_j = h . W3a[j] + b3a[j] -----------------------------------------------------
    float4 h[NCHUNK], hc[NCHUNK];
#pragma unroll
    for (int c = 0; c < NCHUNK; ++c) {
      const int k = c * 128 + lane * 4;
      h[c] = (c < nca && k < Ha) ? __ldg(reinterpret_cast<const float4*>(a.h_a + b * Ha + k)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    // issue every load of this row up front (one memory round trip per row instead of four)
#pragma unroll
    for (int c = 0; c < NCHUNK; ++c) {
      const int k = c * 128 + lane * 4;
      hc[c] = (c < ncc && k < Hc) ? __ldg(reinterpret_cast<const float4*>(a.h_c + b * Hc + k)) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    const float act_in = jl ? __ldg(a.action + b * A + lane) : 0.f;
    const float adv = __ldg(a.advantage + b);
    const float old_lp = __ldg(a.old_logp + b);
    const float target = __ldg(a.target + b);
    float zmine = 0.f;  // lane j keeps z_j
    for (int j = 0; j < A; ++j) {
      float p = 0.f;
#pragma unroll
      for (int c = 0; c < NCHUNK; ++c) {
        const int k = c * 128 + lane * 4;
        if (c < nca && k < Ha) {
          const float4 w = *reinterpret_cast<const float4*>(s_w3a + j * Ha + k);
          p = fmaf(h[c].x, w.x, p); p = fmaf(h[c].y, w.y, p); p = fmaf(h[c].z, w.z, p); p = fmaf(h[c].w, w.w, p);
        }
      }
      p = warp_sum(p);
      if (lane == j) zmine = p;
    }
    float mean = 0.f, th = 0.f, d = 0.f, lp_term = 0.f;
    if (jl) {
      const float z = zmine + b3a;
      if (a.final_tanh) { th = tanhf(z); mean = a.out_scale * th; } else { mean = z; }
      d = act_in - mean;
      lp_term = ppo_logp_term(d, logsig, two_var);
    }
    const PpoSurrogate ps = ppo_surrogate(warp_sum(lp_term), old_lp, adv, a.clip_eps, a.inv_global_batch);
    float dz3 = 0.f;
    if (jl) {
      dz3 = ppo_mean_seed(ps.g_lp, d, inv_var, a.final_tanh, a.out_scale, [&] { return th; });
      acc_dl += ppo_logstd_term(ps.g_lp, d, inv_var);
      if (a.dz3_f32 != nullptr) a.dz3_f32[b * A + lane] = dz3;
    }
    if (lane == 0) acc_surr += ps.surr;
    // ---- actor dgrad through the hidden activation: dZ2a[k] = (sum_j dz3_j W3a[j,k]) * act'(h_k) --------------
    float4 g[NCHUNK];
#pragma unroll
    for (int c = 0; c < NCHUNK; ++c) g[c] = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int j = 0; j < A; ++j) {
      const float dj = __shfl_sync(0xffffffffu, dz3, j);
#pragma unroll
      for (int c = 0; c < NCHUNK; ++c) {
        const int k = c * 128 + lane * 4;
        if (c < nca && k < Ha) {
          const float4 w = *reinterpret_cast<const float4*>(s_w3a + j * Ha + k);
          g[c].x = fmaf(dj, w.x, g[c].x); g[c].y = fmaf(dj, w.y, g[c].y); g[c].z = fmaf(dj, w.z, g[c].z); g[c].w = fmaf(dj, w.w, g[c].w);
        }
      }
    }
#pragma unroll
    for (int c = 0; c < NCHUNK; ++c) {
      const int k = c * 128 + lane * 4;
      if (c < nca && k < Ha) {
        float4 o;
        o.x = g[c].x * act_deriv(h[c].x, a.act); o.y = g[c].y * act_deriv(h[c].y, a.act);
        o.z = g[c].z * act_deriv(h[c].z, a.act); o.w = g[c].w * act_deriv(h[c].w, a.act);
        if (a.dz_a_f32 != nullptr) *reinterpret_cast<float4*>(a.dz_a_f32 + b * Ha + k) = o;
      }
    }
    // ---- critic: v = h_c . w3c + b3c ; Huber ; dZ2c -----------------------------------------------------------
    float pv = 0.f;
#pragma unroll
    for (int c = 0; c < NCHUNK; ++c) {
      const int k = c * 128 + lane * 4;
      h[c] = hc[c];
      if (c < ncc && k < Hc) {
        const float4 w = *reinterpret_cast<const float4*>(s_w3c + k);
        pv = fmaf(h[c].x, w.x, pv); pv = fmaf(h[c].y, w.y, pv); pv = fmaf(h[c].z, w.z, pv); pv = fmaf(h[c].w, w.w, pv);
      }
    }
    const PpoHuber hub = ppo_huber(warp_sum(pv) + b3c, target, a.inv_global_batch);
    const float dv = hub.dv;
    if (lane == 0) {
      acc_hub += hub.loss;
      if (a.dv_f32 != nullptr) a.dv_f32[b] = dv;
    }
#pragma unroll
    for (int c = 0; c < NCHUNK; ++c) {
      const int k = c * 128 + lane * 4;
      if (c < ncc && k < Hc) {
        const float4 w = *reinterpret_cast<const float4*>(s_w3c + k);
        float4 o;
        o.x = dv * w.x * act_deriv(h[c].x, a.act_c); o.y = dv * w.y * act_deriv(h[c].y, a.act_c);
        o.z = dv * w.z * act_deriv(h[c].z, a.act_c); o.w = dv * w.w * act_deriv(h[c].w, a.act_c);
        if (a.dz_c_f32 != nullptr) *reinterpret_cast<float4*>(a.dz_c_f32 + b * Hc + k) = o;
      }
    }
  }

  // ---- CTA partials in a fixed order, last CTA combines (same scheme as ppo_loss.cu) ------------------------------
  float* red = s_red + warp * 34;
  if (lane == 0) { red[0] = acc_surr; red[1] = acc_hub; }
  red[2 + lane] = acc_dl;
  __syncthreads();
  float* part = a.partials + int64_t(blockIdx.x) * (2 + A);
  for (int c = tid; c < 2 + A; c += kHeadsThreads) {
    float s = 0.f;
    for (int w = 0; w < kHeadsWarps; ++w) s += s_red[w * 34 + c];
    part[c] = s;
  }
  ppo_last_cta_finish<kHeadsThreads>(a, a.ent_coef, a.rank_share, a.ticket, s_red,
                                     [&](int j) { return logf(expf(__ldg(a.logstd + j))); }, a.losses, a.logstd_grad, nullptr);
}

bool heads_supported(int act_dim, int hid_a, int hid_c) {
  return act_dim >= 1 && act_dim <= 32 && hid_a % 4 == 0 && hid_c % 4 == 0 && hid_a <= 128 * kMaxChunk &&
         hid_c <= 128 * kMaxChunk && (size_t(act_dim) * hid_a + hid_c + kHeadsThreads + 64) * 4 <= 200 * 1024;
}

int heads_grid(int64_t batch) {
  // one row per warp while that still fits a few resident waves: the kernel is latency-bound, so rows in flight win
  int64_t g = (batch + kHeadsWarps - 1) / kHeadsWarps;
  const int64_t cap = 8ll * num_sms();
  return int(g < 1 ? 1 : (g > cap ? cap : g));
}

int launch_heads(const HeadsArgs& a, cudaStream_t st) {
  if (a.batch == 0) return B200PPO_OK;
  const size_t smem = (size_t(a.act_dim) * a.hid_a + a.hid_c + kHeadsThreads + 64) * sizeof(float);
  const int need = (std::max(a.hid_a, a.hid_c) + 127) / 128;
  const int grid = heads_grid(a.batch);
#define HEADS_GO(NC)                                                                                                  \
  do {                                                                                                                \
    if (smem > 48 * 1024) {                                                                                           \
      static bool attr_set = false;                                                                                   \
      if (!attr_set) {                                                                                                \
        B2_CUDA(cudaFuncSetAttribute(heads_fused_kernel<NC>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024)); \
        attr_set = true;                                                                                              \
      }                                                                                                               \
    }                                                                                                                 \
    heads_fused_kernel<NC><<<grid, kHeadsThreads, smem, st>>>(a);                                                     \
  } while (0)
  if (need <= 1) HEADS_GO(1);
  else if (need <= 2) HEADS_GO(2);
  else if (need <= 4) HEADS_GO(4);
  else HEADS_GO(8);
#undef HEADS_GO
  B2_LAUNCH_CHECK();
  return B200PPO_OK;
}

}  // namespace b200ppo
