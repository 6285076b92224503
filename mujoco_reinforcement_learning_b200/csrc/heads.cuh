// Internal interface of the fused output-layer / loss / first-dgrad kernel (heads.cu).
#pragma once
#include "ppo_math.cuh"

namespace b200ppo {

struct HeadsArgs : PpoOperands {
  // inputs
  const float* h_a;  // [B, hid_a] last hidden activation of the actor (fp32)
  const float* h_c;  // [B, hid_c] last hidden activation of the critic
  const float *w3a, *b3a, *w3c, *b3c;
  int64_t batch;
  int hid_a, hid_c;
  int act, act_c;  // hidden activation codes of actor / critic
  float out_scale, ent_coef, rank_share;
  // outputs (nullable unless noted)
  float* dz3_f32;            // [B, A]      dL/dz of the actor's output layer
  float* dv_f32;             // [B]         dL/dv
  float* dz_a_f32;           // [B, hid_a]  dL/dz of the actor's last hidden layer
  float* dz_c_f32;           // [B, hid_c]
  unsigned* ticket;          // zero-initialised, self-resetting (required; partials too)
  float* losses;             // [2]
  float* logstd_grad;        // [A]
};

bool heads_supported(int act_dim, int hid_a, int hid_c);
int heads_grid(int64_t batch);
int launch_heads(const HeadsArgs& a, cudaStream_t st);

}  // namespace b200ppo
