// The PPO loss of one sample row and its gradient seeds, defined once for every kernel that computes them: the
// separate loss kernel (ppo_loss.cu), the fp32 heads kernel (heads.cu), the fused output-layer epilogues of the
// tcgen05 kernels (tc_common.cuh) and the chain kernel (tc_chain.cu).  The optimizer kernel finishes the fused
// routes' partials with the same column finish (adam.cu).
//
// replaces: Normal.log_prob(...).sum(1), Normal.entropy().mean(), ratio / clamp / min / mean and huber_loss
//           (src/entities/algorithms/ppo.py:113-132) together with what autograd derives from them
//           (SURVEY.md §8a row a10).
//
// Each piece is the exact expression, in the exact operand order, that every route computed before it was shared:
// the routes are compared bit for bit, so a change here is a change of every route's result.
#pragma once
#include <cuda_bf16.h>

#include "common.cuh"

namespace b200ppo {

// Per-row operands of the loss, shared by every route's argument struct (filled by ppo_operands, passes.cu).
struct PpoOperands {
  const float* logstd;     // [A]
  const float* action;     // [B, A]
  const float* old_logp;   // [B]
  const float* advantage;  // [B]
  const float* target;     // [B]
  float* partials;         // [CTAs][2 + A]: (sum surrogate, sum huber, sum d loss / d logstd_j) per CTA
  int act_dim, final_tanh;
  float clip_eps;
  float inv_global_batch;  // 1 / (global minibatch size): the divisor of both loss means
};

constexpr float kLogSqrt2Pi = 0.91893853320467274178f;  // math.log(math.sqrt(2*math.pi))

// sigma-derived constants of one action column
struct PpoSigma {
  float sig, logsig, inv_var, two_var;
};
__device__ __forceinline__ PpoSigma ppo_sigma(float logstd) {
  const float sig = expf(logstd);
  const float var = sig * sig;
  return {sig, logf(sig), 1.f / var, 2.f * var};
}

// One column's term of the Gaussian log-prob, -(a - mu)^2 / (2 var) - log sigma - log sqrt(2 pi), d = a - mu.  The fp32
// routes divide by 2 var, as torch does; the bf16 epilogues multiply by 0.5 / var, because a true division per column
// was what limited their launch and the bf16 route's 2e-2 tolerance does not need it.
__device__ __forceinline__ float ppo_logp_term(float d, float logsig, float two_var) {
  return -(d * d) / two_var - logsig - kLogSqrt2Pi;
}
__device__ __forceinline__ float ppo_logp_term_bf16(float d, float logsig, float inv_var) {
  return -(d * d) * (0.5f * inv_var) - logsig - kLogSqrt2Pi;
}

// Clipped surrogate min(r A, clamp(r, 1 - eps, 1 + eps) A) of one row, r = exp(lp - old_lp), and the seed
// g_lp = d loss_actor / d lp.  autograd: minimum() sends the gradient to the smaller argument (half each on ties);
// clamp passes it inside [lo, hi] inclusive.
struct PpoSurrogate {
  float surr, g_lp;
};
__device__ __forceinline__ PpoSurrogate ppo_surrogate(float lp, float old_lp, float adv, float clip_eps, float inv_global_batch) {
  const float ratio = expf(lp - old_lp);
  const float lo = 1.f - clip_eps, hi = 1.f + clip_eps;
  const float s1 = ratio * adv;
  const float s2 = fminf(fmaxf(ratio, lo), hi) * adv;
  const float w1 = s1 < s2 ? 1.f : (s1 > s2 ? 0.f : 0.5f);
  const float in_range = (ratio >= lo && ratio <= hi) ? 1.f : 0.f;
  return {fminf(s1, s2), -(w1 * adv + (1.f - w1) * adv * in_range) * inv_global_batch * ratio};
}

// Seeds of one action column, d = a - mu.  Mean seed: d loss / d z of the actor's output, through scale * tanh(z) when
// final_tanh (th() returns tanh(z) as the route has it).  Logstd term: this row's part of d loss / d logstd_j.
template <class Tanh>
__device__ __forceinline__ float ppo_mean_seed(float g_lp, float d, float inv_var, bool final_tanh, float scale, Tanh th) {
  float dmu = g_lp * (d * inv_var);
  if (final_tanh) {
    const float t = th();
    dmu *= scale * (1.f - t * t);
  }
  return dmu;
}
__device__ __forceinline__ float ppo_logstd_term(float g_lp, float d, float inv_var) { return g_lp * (d * (d * inv_var) - 1.f); }

// Huber loss (delta = 1) of one row's value and its seed dv = d loss_critic / d value
struct PpoHuber {
  float loss, dv;
};
__device__ __forceinline__ PpoHuber ppo_huber(float value, float target, float inv_global_batch) {
  const float e = value - target;
  const float ae = fabsf(e);
  return {ae < 1.f ? 0.5f * e * e : ae - 0.5f, fminf(fmaxf(e, -1.f), 1.f) * inv_global_batch};
}

// Row `row` of a [B, pitch] bf16 seed matrix with dv in column 0: 16 bytes per row when pitch == 8
__device__ __forceinline__ void ppo_store_dv_bf16(__nv_bfloat16* dst, int64_t row, int pitch, float dv) {
  __nv_bfloat16* o = dst + row * pitch;
  if (pitch == 8) {
    const __nv_bfloat162 v0 = __floats2bfloat162_rn(dv, 0.f);
    *reinterpret_cast<uint4*>(o) = make_uint4(*reinterpret_cast<const uint32_t*>(&v0), 0u, 0u, 0u);
  } else {
    for (int j = 0; j < pitch; ++j) o[j] = __float2bfloat16_rn(j == 0 ? dv : 0.f);
  }
}

// Column c of the partials summed over every CTA (s): 0 gives the entropy and the actor loss, 1 the critic loss,
// 2 + j the logstd gradient.  The entropy is the mean over [B, A] of 0.5 + log sqrt(2 pi) + log sigma_j (the row is
// constant in b); log_sigma(j) returns log sigma_j as the caller has it.  Outputs are nullable.
template <class LogSigma>
__device__ __forceinline__ void ppo_finish_column(const PpoOperands& op, float ent_coef, float rank_share, int c, float s,
                                                  LogSigma log_sigma, float* losses, float* logstd_grad, float* entropy_out) {
  const int A = op.act_dim;
  if (c == 0) {
    if (losses == nullptr && entropy_out == nullptr) return;
    float ent = 0.f;
    for (int j = 0; j < A; ++j) ent += 0.5f + kLogSqrt2Pi + log_sigma(j);
    ent /= float(A);
    if (entropy_out != nullptr) *entropy_out = ent;
    if (losses != nullptr) losses[0] = -s * op.inv_global_batch - ent_coef * ent * rank_share;
  } else if (c == 1) {
    if (losses != nullptr) losses[1] = s * op.inv_global_batch;
  } else if (logstd_grad != nullptr) {
    logstd_grad[c - 2] = s - ent_coef * rank_share / float(A);
  }
}

// Called by every thread of the CTA once its row of partials is written: the last CTA to get here (atomic ticket)
// sums all rows in a fixed order (deterministic), finishes every column and resets the ticket for the next launch on
// the stream.  s_scratch: THREADS floats of shared memory.
template <int THREADS, class LogSigma>
__device__ __forceinline__ void ppo_last_cta_finish(const PpoOperands& op, float ent_coef, float rank_share, unsigned* ticket,
                                                    float* s_scratch, LogSigma log_sigma, float* losses, float* logstd_grad,
                                                    float* entropy_out) {
  __shared__ bool s_last;
  const int tid = threadIdx.x;
  __threadfence();
  __syncthreads();
  if (tid == 0) s_last = (atomicAdd(ticket, 1u) == gridDim.x - 1);
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  const float s = combine_partials<THREADS>(op.partials, gridDim.x, 2 + op.act_dim, tid, s_scratch);
  if (tid < 2 + op.act_dim) ppo_finish_column(op, ent_coef, rank_share, tid, s, log_sigma, losses, logstd_grad, entropy_out);
  if (tid == 0) *ticket = 0u;
}

}  // namespace b200ppo
