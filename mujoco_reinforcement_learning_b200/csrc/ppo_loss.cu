// Diagonal-Gaussian log-prob, entropy, clipped-ratio surrogate, Huber value loss and their gradient seeds (the math:
// ppo_math.cuh) as a kernel of its own, for the shapes no fused route takes, and Normal.sample / log_prob of the
// rollout (ppo.py:23-26).
//
// One thread per sample (rows are short: A floats).  Loss sums and the logstd gradient are reduced per CTA
// in a fixed order and combined by the last CTA to finish (atomic ticket), so results are deterministic.
#include "ppo_loss.cuh"

namespace b200ppo {

constexpr int kLossThreads = 128;

// One thread per sample row, but every global access is a block-wide contiguous slab copy: the 128 rows a CTA owns
// are adjacent in the row-major [B, A] arrays, so `mean`, `action` and the gradient seeds move through shared memory
// with fully coalesced 128-byte lines (rows of A = 17 floats would otherwise cost one line per thread).
// dynamic smem: 3 x [A] sigma constants | mean [T][A] | action [T][A] | dz fp32 [T][A] (also the logstd-gradient
// contributions after use) | dl [T][A] | dz bf16 [T][pitch]
__global__ void __launch_bounds__(kLossThreads)
ppo_loss_seed_kernel(LossArgs a) {
  extern __shared__ __align__(16) float smem[];
  const int A = a.act_dim;
  float* s_logsig = smem;
  float* s_inv_var = smem + A;
  float* s_two_var = smem + 2 * A;
  float* s_mean = smem + 3 * A;
  float* s_act = s_mean + kLossThreads * A;
  float* s_dz = s_act + kLossThreads * A;
  float* s_dl = s_dz + kLossThreads * A;
  __nv_bfloat16* s_dzb = reinterpret_cast<__nv_bfloat16*>(s_dl + kLossThreads * A);
  __shared__ float s_red[2][kLossThreads / 32];
  __shared__ float s_comb[kLossThreads];
  const int tid = threadIdx.x;
  const int64_t b0 = int64_t(blockIdx.x) * kLossThreads;
  const int64_t remaining = a.batch - b0;
  const int rows = remaining < kLossThreads ? int(remaining) : kLossThreads;
  for (int j = tid; j < A; j += kLossThreads) {
    const PpoSigma c = ppo_sigma(a.logstd[j]);
    s_logsig[j] = c.logsig;
    s_inv_var[j] = c.inv_var;
    s_two_var[j] = c.two_var;
  }
  for (int i = tid; i < rows * A; i += kLossThreads) {
    s_mean[i] = __ldg(a.mean + b0 * A + i);
    s_act[i] = __ldg(a.action + b0 * A + i);
  }
  __syncthreads();
  const int64_t b = b0 + tid;
  const bool active = tid < rows;
  const bool want_seed = a.dz_actor != nullptr || a.dz_actor_bf16 != nullptr;
  const int pitch = a.dz_actor_pitch;
  float surr = 0.f, hub = 0.f;
  if (active) {
    const float* mu = s_mean + tid * A;
    const float* ac = s_act + tid * A;
    float lp = 0.f;
    for (int j = 0; j < A; ++j) lp += ppo_logp_term(ac[j] - mu[j], s_logsig[j], s_two_var[j]);
    if (a.logp_out != nullptr) a.logp_out[b] = lp;
    if (want_seed) {
      const PpoSurrogate ps = ppo_surrogate(lp, a.old_logp[b], a.advantage[b], a.clip_eps, a.inv_global_batch);
      surr = ps.surr;
      for (int j = 0; j < A; ++j) {
        const float d = ac[j] - mu[j], inv_var = s_inv_var[j];
        const float dmu = ppo_mean_seed(ps.g_lp, d, inv_var, a.final_tanh, a.out_scale, [&] { return mu[j] / a.out_scale; });
        s_dz[tid * A + j] = dmu;
        if (a.dz_actor_bf16 != nullptr) s_dzb[tid * pitch + j] = __float2bfloat16_rn(dmu);
        s_dl[tid * A + j] = ppo_logstd_term(ps.g_lp, d, inv_var);
      }
      if (a.dz_actor_bf16 != nullptr)
        for (int j = A; j < pitch; ++j) s_dzb[tid * pitch + j] = __float2bfloat16_rn(0.f);
    }
    if (a.dv != nullptr || a.dv_bf16 != nullptr) {
      const PpoHuber h = ppo_huber(a.value[b], a.target[b], a.inv_global_batch);
      hub = h.loss;
      if (a.dv != nullptr) a.dv[b] = h.dv;
      if (a.dv_bf16 != nullptr) ppo_store_dv_bf16(a.dv_bf16, b, a.dv_pitch, h.dv);
    }
  } else if (want_seed) {
    for (int j = 0; j < A; ++j) s_dl[tid * A + j] = 0.f;
  }
  __syncthreads();
  if (want_seed) {  // coalesced slab stores of the seeds
    if (a.dz_actor != nullptr)
      for (int i = tid; i < rows * A; i += kLossThreads) a.dz_actor[b0 * A + i] = s_dz[i];
    if (a.dz_actor_bf16 != nullptr) {
      const uint32_t* src = reinterpret_cast<const uint32_t*>(s_dzb);  // pitch is even: whole 32-bit words
      uint32_t* dst = reinterpret_cast<uint32_t*>(a.dz_actor_bf16 + b0 * pitch);
      for (int i = tid; i < rows * pitch / 2; i += kLossThreads) dst[i] = src[i];
    }
  }
  if (a.partials == nullptr) return;

  // CTA reduction (fixed order) -> partials[cta][2 + A]
  const float ws = warp_sum(surr), wh = warp_sum(hub);
  if ((tid & 31) == 0) { s_red[0][tid >> 5] = ws; s_red[1][tid >> 5] = wh; }
  __syncthreads();
  float* part = a.partials + int64_t(blockIdx.x) * (2 + A);
  if (tid == 0) {
    float x = 0.f, y = 0.f;
    for (int w = 0; w < kLossThreads / 32; ++w) { x += s_red[0][w]; y += s_red[1][w]; }
    part[0] = x; part[1] = y;
  }
  if (want_seed) {
    for (int j = tid; j < A; j += kLossThreads) {
      float s = 0.f;
      for (int r = 0; r < kLossThreads; ++r) s += s_dl[r * A + j];
      part[2 + j] = s;
    }
  }
  ppo_last_cta_finish<kLossThreads>(a, a.ent_coef, a.rank_share, a.ticket, s_comb, [&](int j) { return s_logsig[j]; }, a.losses,
                                    a.logstd_grad, a.entropy_out);
}

__global__ void __launch_bounds__(128)
sample_logp_kernel(const float* __restrict__ mean, const float* __restrict__ logstd, const float* __restrict__ noise,
                   int64_t batch, int A, float* __restrict__ action, float* __restrict__ logp) {
  const int64_t b = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (b >= batch) return;
  float lp = 0.f;
  for (int j = 0; j < A; ++j) {
    const PpoSigma c = ppo_sigma(__ldg(logstd + j));
    const float mu = mean[b * A + j];
    const float act = noise != nullptr ? mu + c.sig * noise[b * A + j] : mu;  // torch.normal(mean, std) = mean + std*eps
    if (action != nullptr) action[b * A + j] = act;
    lp += ppo_logp_term(act - mu, c.logsig, c.two_var);
  }
  if (logp != nullptr) logp[b] = lp;
}

int launch_ppo_loss(const LossArgs& a, cudaStream_t st) {
  if (a.batch == 0) return B200PPO_OK;
  const int pitch = a.dz_actor_bf16 != nullptr ? a.dz_actor_pitch : 0;
  B2_CHECK_ARG(a.act_dim + 2 <= 64, "act_dim %d too large for the loss kernel (<= 62)", a.act_dim);
  B2_CHECK_ARG(pitch % 2 == 0, "bf16 seed pitch must be even");
  const size_t smem = sizeof(float) * (3 * size_t(a.act_dim) + 4 * size_t(kLossThreads) * a.act_dim) + size_t(kLossThreads) * pitch * 2 + 16;
  if (smem > 48 * 1024) {
    static bool attr_set = false;
    if (!attr_set) {
      B2_CUDA(cudaFuncSetAttribute(ppo_loss_seed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      attr_set = true;
    }
    B2_CHECK_ARG(smem <= 200 * 1024, "act_dim %d too large for the loss kernel", a.act_dim);
  }
  const unsigned grid = unsigned((a.batch + kLossThreads - 1) / kLossThreads);
  ppo_loss_seed_kernel<<<grid, kLossThreads, smem, st>>>(a);
  B2_LAUNCH_CHECK();
  return B200PPO_OK;
}

int loss_grid_size(int64_t batch) { return int((batch + kLossThreads - 1) / kLossThreads); }

int launch_sample_logp(const float* mean, const float* logstd, const float* noise, int64_t batch, int A, float* action,
                       float* logp, cudaStream_t st) {
  if (batch == 0) return B200PPO_OK;
  sample_logp_kernel<<<unsigned((batch + 127) / 128), 128, 0, st>>>(mean, logstd, noise, batch, A, action, logp);
  B2_LAUNCH_CHECK();
  return B200PPO_OK;
}

}  // namespace b200ppo
