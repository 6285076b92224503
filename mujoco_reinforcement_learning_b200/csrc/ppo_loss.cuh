// Internal interface of the loss / gradient-seed kernels (ppo_loss.cu).
#pragma once
#include "ppo_math.cuh"

namespace b200ppo {

struct LossArgs : PpoOperands {  // old_logp needed when dz_actor != null, target when dv != null
  // inputs
  const float* mean;       // [B, A] actor output (out_scale * tanh(z) when final_tanh)
  const float* value;      // [B]   critic output (needed when dv != null)
  int64_t batch;           // local rows
  float out_scale;
  float ent_coef;
  float rank_share;        // 1 / world_size: share of the batch-independent entropy term owned by this rank
  // outputs (all nullable)
  float* logp_out;      // [B] new log-prob
  float* dz_actor;      // [B, A] dL_actor / d z_last
  float* dv;            // [B]    dL_critic / d value
  __nv_bfloat16* dz_actor_bf16;  // [B, dz_actor_pitch] bf16 copy for the tensor-core dgrad / wgrad (padding zeroed)
  __nv_bfloat16* dv_bf16;        // [B, dv_pitch]
  int dz_actor_pitch, dv_pitch;
  unsigned* ticket;     // zero-initialised counter, self-resetting
  float* losses;        // [2] actor_loss, critic_loss
  float* logstd_grad;   // [A]
  float* entropy_out;   // [1]
};

int launch_ppo_loss(const LossArgs& a, cudaStream_t st);
int loss_grid_size(int64_t batch);
int launch_sample_logp(const float* mean, const float* logstd, const float* noise, int64_t batch, int A, float* action,
                       float* logp, cudaStream_t st);

}  // namespace b200ppo
