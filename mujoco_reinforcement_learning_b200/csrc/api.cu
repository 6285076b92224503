// C-ABI entry points that each run one piece of the actor-critic on a caller's batch (see include/b200ppo.h).
//
// replaces: the per-call glue of Actor/Critic.forward (src/models/linear/actor.py:25-30, src/models/critic.py:22-25).
#include "context.cuh"

namespace b200ppo {

__global__ void tanh_scale_bwd_kernel(const float* __restrict__ grad_out, const float* __restrict__ out, float scale,
                                      int64_t n, float* __restrict__ dz) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) {
    const float th = out[i] / scale;
    dz[i] = grad_out[i] * scale * (1.f - th * th);
  }
}

// The bf16 variant's rollout inference: weights and observations to bf16, then ONE tensor-core launch (the forward half
// of the chain kernel) that leaves mean, sampled action, its log-probability and the value (B200PPO_CHAIN_INFER=0: the
// fp32 path instead).
static bool chain_infer_enabled(const b200ppo_ctx* ctx) {
  if (ctx->precision != B200PPO_PREC_BF16 || !chain_applicable(ctx)) return false;
  static const char* mode = getenv("B200PPO_CHAIN_INFER");
  return !(mode != nullptr && mode[0] == '0');
}

static int run_chain_infer(b200ppo_ctx* ctx, const float* params, const float* obs, int64_t n, const ChainInfer& inf,
                           cudaStream_t st) {
  B2_TRY(cast_weights(ctx, params, st));
  B2_TRY(launch_cast_rows_ones(obs, n, ctx->net[0].d.in_dim, ctx->bf.X, ctx->bf.pitchX, st));
  int grid = 0;
  return launch_chain(ctx, params, ctx->bf.X, n, nullptr, nullptr, nullptr, nullptr, nullptr, &grid, st, false, &inf);
}

}  // namespace b200ppo

using namespace b200ppo;

extern "C" B2_EXPORT int b200ppo_mlp_forward(b200ppo_ctx* ctx, int32_t net, const float* params, const float* x, int64_t batch,
                                   float* out, float* saved, b200ppo_stream stream) {
  B2_TRY(check_batch(ctx, batch, "b200ppo_mlp_forward"));
  B2_CHECK_ARG((net == 0 || net == 1) && params && x && out, "b200ppo_mlp_forward: bad argument");
  if (batch == 0) return B200PPO_OK;
  float* acts[2] = {ctx->ws_act[0], ctx->ws_act[1]};
  float* outs[2] = {nullptr, nullptr};
  if (saved) acts[net] = saved;
  outs[net] = out;
  return forward_nets(ctx, params, x, batch, 1 << net, acts, outs, static_cast<cudaStream_t>(stream), false, fresh_arena(ctx));
}

extern "C" B2_EXPORT int b200ppo_mlp_backward(b200ppo_ctx* ctx, int32_t net, const float* params, const float* x,
                                    const float* out, const float* saved, const float* grad_out, int64_t batch,
                                    float* grad_params, float* grad_x, b200ppo_stream stream) {
  B2_TRY(check_batch(ctx, batch, "b200ppo_mlp_backward"));
  B2_CHECK_ARG((net == 0 || net == 1) && params && x && out && saved && grad_out && grad_params,
               "b200ppo_mlp_backward: bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const Net& N = ctx->net[net];
  const int64_t n_seg = (net == 0 ? ctx->logstd_off : N.seg_end) - N.seg_begin;
  if (batch == 0) {
    B2_CUDA(cudaMemsetAsync(grad_params, 0, size_t(n_seg) * sizeof(float), st));
    return B200PPO_OK;
  }
  float* acts[2] = {nullptr, nullptr};
  float* dz[2] = {nullptr, nullptr};
  float* gx[2] = {nullptr, nullptr};
  acts[net] = const_cast<float*>(saved);
  dz[net] = ctx->ws_dz[net];
  gx[net] = grad_x;
  float* dz_last = dz[net] + N.dz_off(N.d.n_layers - 1, batch);
  const int64_t n_out = batch * N.out_dim();
  if (N.d.final_tanh) {
    tanh_scale_bwd_kernel<<<unsigned((n_out + 255) / 256), 256, 0, st>>>(grad_out, out, N.d.out_scale, n_out, dz_last);
    B2_LAUNCH_CHECK();
  } else {
    B2_CUDA(cudaMemcpyAsync(dz_last, grad_out, size_t(n_out) * sizeof(float), cudaMemcpyDeviceToDevice, st));
  }
  int split = 1;
  B2_TRY(backward_nets(ctx, params, x, batch, 1 << net, acts, dz, ctx->gpart, &split, gx, st, false, fresh_arena(ctx)));
  return launch_reduce_partials(ctx->gpart + N.seg_begin, split, ctx->n_params, n_seg, grad_params, st);
}

extern "C" B2_EXPORT int b200ppo_policy_infer(b200ppo_ctx* ctx, const float* params, const float* obs, int64_t batch,
                                    const float* noise, float* mean, float* value, float* action, float* logp,
                                    b200ppo_stream stream) {
  B2_TRY(check_batch(ctx, batch, "b200ppo_policy_infer"));
  B2_CHECK_ARG(params && obs, "b200ppo_policy_infer: null pointer");
  if (batch == 0) return B200PPO_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* acts[2] = {ctx->ws_act[0], ctx->ws_act[1]};
  float* outs[2] = {mean ? mean : ctx->ws_out[0], value ? value : ctx->ws_out[1]};
  const bool need_actor = mean || action || logp;
  const int nets = (need_actor ? 1 : 0) | (value ? 2 : 0);
  if (nets == 0) return B200PPO_OK;
  if (chain_infer_enabled(ctx)) {
    ChainInfer inf{};
    inf.noise = noise; inf.mean = mean; inf.value = value; inf.action = action; inf.logp = logp;
    return run_chain_infer(ctx, params, obs, batch, inf, st);
  }
  B2_TRY(forward_nets(ctx, params, obs, batch, nets, acts, outs, st, false, fresh_arena(ctx)));
  if (action || logp)
    B2_TRY(launch_sample_logp(outs[0], params + ctx->logstd_off, noise, batch, ctx->net[0].out_dim(), action, logp, st));
  return B200PPO_OK;
}

__global__ void rollout_scatter_kernel(const float* __restrict__ value, const float* __restrict__ action, const float* __restrict__ logp,
                                       int64_t n, int A, int64_t t, int64_t T, float* __restrict__ buf_value,
                                       float* __restrict__ buf_next_value, float* __restrict__ buf_action, float* __restrict__ buf_logp) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float v = value[i];
  if (buf_value != nullptr) buf_value[i * T + t] = v;
  if (buf_next_value != nullptr) buf_next_value[i * T + t - 1] = v;
  if (buf_action != nullptr)
    for (int j = 0; j < A; ++j) buf_action[(i * T + t) * A + j] = action[i * A + j];
  if (buf_logp != nullptr) buf_logp[i * T + t] = logp[i];
}

// One environment step of the rollout (ppo.py:20-49) written straight into the [N, T, ...] buffers: state s_t, V(s_t),
// the sampled action and its log-probability at time index t — and V(s_t) once more as next_state_value of step t - 1,
// which the reference computes with a second critic call on the very same tensor (ppo.py:27-29: next_state of step t - 1
// is cloned into current_state of step t).  t == T: only that last next_state_value (no action is sampled).
extern "C" B2_EXPORT int b200ppo_rollout_step(b200ppo_ctx* ctx, const float* params, const float* obs, int64_t n_envs,
                                              const float* noise, int64_t t, int64_t T, float* buf_state, float* buf_value,
                                              float* buf_next_value, float* buf_action, float* buf_logp, b200ppo_stream stream) {
  B2_TRY(check_batch(ctx, n_envs, "b200ppo_rollout_step"));
  B2_CHECK_ARG(params && obs && n_envs > 0 && T > 0 && t >= 0 && t <= T, "b200ppo_rollout_step: bad argument");
  B2_CHECK_ARG(t == T || (buf_value && buf_action && buf_logp), "b200ppo_rollout_step: null buffer");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int D = ctx->net[0].d.in_dim, A = ctx->net[0].out_dim();
  const bool last = t == T;
  if (!last && buf_state != nullptr)
    B2_CUDA(cudaMemcpy2DAsync(buf_state + t * D, size_t(T) * D * sizeof(float), obs, size_t(D) * sizeof(float), size_t(D) * sizeof(float),
                              size_t(n_envs), cudaMemcpyDeviceToDevice, st));
  float* nv = (t > 0 && buf_next_value != nullptr) ? buf_next_value + (t - 1) : nullptr;
  if (chain_infer_enabled(ctx)) {
    ChainInfer inf{};
    inf.noise = last ? nullptr : noise;
    inf.value = last ? nullptr : buf_value + t;
    inf.value2 = nv;
    inf.action = last ? nullptr : buf_action + t * A;
    inf.logp = last ? nullptr : buf_logp + t;
    inf.ld_action = T * A; inf.ld_value = T; inf.ld_logp = T;
    return run_chain_infer(ctx, params, obs, n_envs, inf, st);
  }
  // other contexts: the plain inference into scratch (value, actions, log-probs for max_batch rows), then one scatter into
  // the buffers
  B2_TRY(ctx->rollout_tmp.grow(ctx->max_batch * (A + 2)));
  float* tv = ctx->rollout_tmp;
  float* ta = tv + ctx->max_batch;
  float* tl = ta + ctx->max_batch * A;
  B2_TRY(b200ppo_policy_infer(ctx, params, obs, n_envs, last ? nullptr : noise, nullptr, tv, last ? nullptr : ta, last ? nullptr : tl, stream));
  rollout_scatter_kernel<<<unsigned((n_envs + 127) / 128), 128, 0, st>>>(tv, ta, tl, n_envs, A, t, T, last ? nullptr : buf_value,
                                                                         (t > 0) ? buf_next_value : nullptr, last ? nullptr : buf_action,
                                                                         last ? nullptr : buf_logp);
  B2_LAUNCH_CHECK();
  return B200PPO_OK;
}

extern "C" B2_EXPORT int b200ppo_evaluate(b200ppo_ctx* ctx, const float* params, const float* obs, const float* action,
                                int64_t batch, float* logp, float* value, float* entropy, b200ppo_stream stream) {
  B2_TRY(check_batch(ctx, batch, "b200ppo_evaluate"));
  B2_CHECK_ARG(params && obs && action && batch > 0, "b200ppo_evaluate: bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* acts[2] = {ctx->ws_act[0], ctx->ws_act[1]};
  float* outs[2] = {ctx->ws_out[0], value ? value : ctx->ws_out[1]};
  B2_TRY(forward_nets(ctx, params, obs, batch, 3, acts, outs, st, false, fresh_arena(ctx)));
  LossArgs la{ppo_operands(ctx, params, nullptr, batch, action, nullptr, nullptr, nullptr)};
  la.mean = outs[0]; la.batch = batch; la.out_scale = ctx->net[0].d.out_scale; la.rank_share = 1.f;
  la.logp_out = logp; la.entropy_out = entropy; la.ticket = ctx->ticket;
  return launch_ppo_loss(la, st);
}

extern "C" B2_EXPORT int b200ppo_minibatch_grads(b200ppo_ctx* ctx, const float* params, const float* obs, const float* action,
                                       const float* old_logp, const float* advantage, const float* target,
                                       int64_t batch, const b200ppo_hparams* hp, float* grads, float* losses,
                                       b200ppo_stream stream) {
  B2_TRY(check_batch(ctx, batch, "b200ppo_minibatch_grads"));
  B2_CHECK_ARG(params && obs && action && old_logp && advantage && target && hp && grads && batch > 0,
               "b200ppo_minibatch_grads: bad argument");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int split = 1;
  if (ctx->precision == B200PPO_PREC_BF16) {
    B2_TRY(cast_weights(ctx, params, st));
    B2_TRY(launch_cast_rows_ones(obs, batch, ctx->net[0].d.in_dim, ctx->bf.X, ctx->bf.pitchX, st));
  }
  int loss_ctas = 0;
  float* loss_dst = losses ? losses : ctx->scratch;
  B2_TRY(minibatch_fwd_bwd(ctx, params, obs, ctx->bf.X, action, old_logp, advantage, target, batch, hp, loss_dst, &split,
                           &loss_ctas, st));
  const LossCombine lc = make_loss_combine(ctx, params, loss_ctas, batch, hp, loss_dst);
  return launch_reduce_partials(ctx->gpart, split, ctx->n_params, ctx->n_params, grads, st, &lc);
}
