/*
 * b200ppo.h — C ABI of the B200-native PPO hot path (libb200ppo.so).
 *
 * Drop-in boundary for aminrezaee/mujoco_reinforcement_learning's PPO update path.  The reference has
 * no FFI of its own (it is pure Python over torch CPU operators), so every entry point below replaces
 * a Python call site of the reference; the citation after "replaces:" is that call site, relative to
 * the reference repository root.  Plain pointers and sizes only — no torch types.
 *
 * Conventions
 *  - All data pointers are DEVICE pointers on the current CUDA device unless the name ends in `_host`.
 *  - Tensors are dense, row-major, fp32 unless stated; bool tensors are one byte per element (torch.bool).
 *  - Rollout buffers use the reference layout: env-major, time-minor ([N_envs, T], flat index n*T + t;
 *    src/entities/algorithms/ppo.py:60,99).
 *  - `stream` is a cudaStream_t (NULL = legacy default stream).  Calls only enqueue work; they never
 *    synchronise the device unless documented (`*_host` entry points do).
 *  - Return value: 0 on success, a negative B200PPO_E* code otherwise; `b200ppo_last_error()` returns a
 *    thread-local message.  There is no CPU fallback: without a CUDA device every compute call fails.
 */
#ifndef B200PPO_H_
#define B200PPO_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200PPO_VERSION 100

#define B200PPO_OK 0
#define B200PPO_EINVAL (-1)  /* bad argument (shape, alignment, null pointer) */
#define B200PPO_ECUDA (-2)   /* CUDA runtime error, message in b200ppo_last_error() */
#define B200PPO_ENOMEM (-3)
#define B200PPO_ESTATE (-4)  /* call not valid for this context (e.g. batch larger than max_batch) */
#define B200PPO_ENCCL (-5)   /* collective / peer-exchange failure (NCCL error, a peer rank that did not arrive) */
#define B200PPO_EINDEX (-6)  /* an index handed to a gather lies outside the table (the reference raises IndexError) */

#define B200PPO_MAX_LAYERS 8

#define B200PPO_ACT_TANH 0
#define B200PPO_ACT_RELU 1

/* GEMM arithmetic of the actor/critic MLP. */
#define B200PPO_PREC_FP32 0 /* fp32 FFMA everywhere: 1e-5 parity with the reference */
#define B200PPO_PREC_BF16 1 /* bf16 operands on tcgen05 tensor cores, fp32 accumulate / master weights: 2e-2 */

typedef void* b200ppo_stream; /* cudaStream_t */
typedef struct b200ppo_ctx b200ppo_ctx;

/* One NetworkBlock: n_layers Linear layers, hidden activation after all but the last.
 * replaces: src/models/network_block_creator.py:24-86 (no batch-norm / skip / end-normalisation: those
 * branches are off on the PPO path). */
typedef struct b200ppo_mlp_desc {
  int32_t n_layers;                 /* Linear layers including the last one, 1..B200PPO_MAX_LAYERS */
  int32_t in_dim;                   /* input features (obs_dim * window_length, flattened) */
  int32_t dims[B200PPO_MAX_LAYERS]; /* output features of each Linear */
  int32_t activation;               /* B200PPO_ACT_* applied after every hidden Linear */
  int32_t final_tanh;               /* 1: out = out_scale * tanh(z_last) (linear/actor.py:28); 0: out = z_last */
  float out_scale;                  /* network_config.output_max_value */
} b200ppo_mlp_desc;

/* Hyper-parameters read by the update step (src/main.py:41-54, src/entities/algorithms/ppo.py:95-137). */
typedef struct b200ppo_hparams {
  double learning_rate_actor;
  double learning_rate_critic;
  double beta1, beta2, adam_eps; /* torch.optim.Adam defaults 0.9, 0.999, 1e-8 (ppo_agent.py:15-18) */
  double clip_epsilon;           /* ppo_config.clip_epsilon */
  double entropy_eps;            /* ppo_config.entropy_eps */
} b200ppo_hparams;

int b200ppo_version(void);
const char* b200ppo_last_error(void);

/* ---------------------------------------------------------------------------------------------
 * K1 — advantage pipeline.
 * replaces: PPO.calculate_advantages, src/entities/algorithms/ppo.py:62-91, and the torchrl call inside
 *           it (torchrl 0.6.0 generalized_advantage_estimate, call site ppo.py:76-80).
 *   reward        [N,T] fp32, or fp64 when reward_is_f64 (real rollouts: ppo.py:42-43)
 *   value, next_value [N,T] fp32
 *   terminated    [N,T] bool bytes
 *   done          [N,T] bool bytes, or NULL = "terminated with the last step forced to 1" (ppo.py:70-72)
 *   normalize_rewards / normalize_advantage: per-env over time, unbiased std, no epsilon, times
 *   advantage_scaler (ppo.py:66-69, 81-88); normalize_advantage normalises BOTH outputs.
 *   advantage, value_target [N,T] fp32 out.
 */
int b200ppo_gae(const void* reward, int reward_is_f64, const float* value, const float* next_value,
                const uint8_t* terminated, const uint8_t* done, int64_t n_envs, int64_t n_steps, double gamma,
                double lmbda, int normalize_rewards, int normalize_advantage, double advantage_scaler,
                float* advantage, float* value_target, b200ppo_stream stream);

/* ---------------------------------------------------------------------------------------------
 * K2 — minibatch permutation gather.
 * replaces: `shuffled_memory = memory[idx]` + the minibatch slice, ppo.py:103-106 (tensordict index).
 * Gathers `count` rows idx[0..count) of the five leaves the update reads.  Bit-exact copies.
 * idx is int64 (torch.randperm), values in [-n_rows, n_rows); out-of-range indices set *err_flag (device
 * int32, may be NULL) to 1 and copy nothing for that row.
 */
int b200ppo_gather_minibatch(const int64_t* idx, int64_t count, int64_t n_rows, const float* obs, int64_t obs_dim,
                             const float* action, int64_t act_dim, const float* logp, const float* advantage,
                             const float* target, float* obs_out, float* action_out, float* logp_out,
                             float* advantage_out, float* target_out, int32_t* err_flag, b200ppo_stream stream);

/* Generic leaf gather: dst[i, :] = src[idx[i], :] for rows of row_bytes bytes (any dtype). */
int b200ppo_gather_rows(const void* src, int64_t row_bytes, int64_t n_rows, const int64_t* idx, int64_t count,
                        void* dst, int32_t* err_flag, b200ppo_stream stream);

/* ---------------------------------------------------------------------------------------------
 * K5 — Adam.
 * replaces: torch.optim.Adam.step (single-tensor path) at ppo.py:122,135; built at ppo_agent.py:15-18.
 * One segment of n contiguous fp32 parameters.  `step` is the 1-based step count of THIS update.
 * grads may hold n_partials partial sums laid out [n_partials][partial_stride]; they are summed in
 * index order before the update (n_partials = 1 for a plain gradient).
 */
int b200ppo_adam_step(float* params, const float* grads, int32_t n_partials, int64_t partial_stride,
                      float* exp_avg, float* exp_avg_sq, int64_t n, double lr, double beta1, double beta2,
                      double eps, int64_t step, b200ppo_stream stream);

/* ---------------------------------------------------------------------------------------------
 * Actor-critic context: owns activations / gradient workspaces for batches up to max_batch.
 * Parameter layout (one flat fp32 buffer owned by the caller):
 *   actor:  for each layer l: W_l [dims[l], in_l] row-major (nn.Linear.weight), then b_l [dims[l]]
 *           then actor_logstd [act_dim]
 *   critic: same per-layer layout, appended after the actor segment.
 * b200ppo_param_count / b200ppo_param_offset describe it (offsets in elements).
 */
int b200ppo_create(const b200ppo_mlp_desc* actor, const b200ppo_mlp_desc* critic, int64_t max_batch,
                   int32_t precision, b200ppo_ctx** out);
void b200ppo_destroy(b200ppo_ctx* ctx);
int64_t b200ppo_param_count(const b200ppo_ctx* ctx);
int64_t b200ppo_actor_param_count(const b200ppo_ctx* ctx); /* includes logstd; critic segment starts here */
/* net: 0 actor, 1 critic; layer in [0,n_layers); what: 0 weight, 1 bias; (net 0, layer n_layers, what 0) = logstd */
int64_t b200ppo_param_offset(const b200ppo_ctx* ctx, int32_t net, int32_t layer, int32_t what);

/* K3 forward only.  replaces: Actor.forward (src/models/linear/actor.py:25-30) and Critic.forward
 * (src/models/critic.py:22-25).  net: 0 actor → out [B, act_dim] = mean; 1 critic → out [B,1].
 * saved (nullable) receives the hidden activations [sum(hidden dims)][B] needed by b200ppo_mlp_backward,
 * layer after layer, each [B, dims[l]] row-major; size b200ppo_saved_size(ctx, net, B) floats. */
int64_t b200ppo_saved_size(const b200ppo_ctx* ctx, int32_t net, int64_t batch);
int b200ppo_mlp_forward(b200ppo_ctx* ctx, int32_t net, const float* params, const float* x, int64_t batch,
                        float* out, float* saved, b200ppo_stream stream);
/* K4 for the autograd façade: given dL/dout [B, out_dim] returns dL/dparams for that net (same layout as
 * its parameter segment, logstd slot untouched) and optionally dL/dx (nullable). */
int b200ppo_mlp_backward(b200ppo_ctx* ctx, int32_t net, const float* params, const float* x, const float* out,
                         const float* saved, const float* grad_out, int64_t batch, float* grad_params,
                         float* grad_x, b200ppo_stream stream);

/* K6 — rollout inference.  replaces: ppo.py:22-26 (critic(s), actor(s), Normal.sample, log_prob.sum).
 * noise (nullable) is the standard-normal draw [B, act_dim]: action = mean + exp(logstd) * noise; NULL →
 * action = mean (test_phase, agent.py:36-38).  Any of mean/value/action/logp may be NULL. */
int b200ppo_policy_infer(b200ppo_ctx* ctx, const float* params, const float* obs, int64_t batch,
                         const float* noise, float* mean, float* value, float* action, float* logp,
                         b200ppo_stream stream);

/* "evaluate": ppo.py:109-115,125 — new log-prob [B], value [B], entropy (device scalar) for given actions. */
int b200ppo_evaluate(b200ppo_ctx* ctx, const float* params, const float* obs, const float* action, int64_t batch,
                     float* logp, float* value, float* entropy, b200ppo_stream stream);

/* K3+K4 — losses and gradients of one minibatch, no optimiser step.
 * replaces: ppo.py:109-134 minus the two optimizer.step() calls.
 * grads [param_count] receives dL_actor/dθ_actor and dL_critic/dθ_critic; losses[0] = actor loss,
 * losses[1] = critic loss (device). */
int b200ppo_minibatch_grads(b200ppo_ctx* ctx, const float* params, const float* obs, const float* action,
                            const float* old_logp, const float* advantage, const float* target, int64_t batch,
                            const b200ppo_hparams* hp, float* grads, float* losses, b200ppo_stream stream);

/* The trainer's update step.  replaces: PPO.train, ppo.py:93-154 (epochs × minibatches of
 * gather → forward → losses → backward → two Adam steps), with the permutations supplied
 * (`torch.randperm` stays the caller's, ppo.py:103, so indices are bit-exact).
 *   obs [M,obs_dim] action [M,act_dim] old_logp/advantage/target [M]   — the flattened rollout
 *   perms [epochs][M] int64
 *   batch = training_config.batch_size; minibatches per epoch = floor(M / batch), the tail is dropped
 *   (ppo.py:97-98,107-108); max_minibatches_per_epoch > 0 truncates an epoch (bounded benchmarking).
 *   adam_step_io (host): Adam step count before the call; updated to the count after it.
 *   losses_out (device, nullable) [epochs * minibatches][2] = (actor_loss, critic_loss) per minibatch.
 */
int b200ppo_train(b200ppo_ctx* ctx, float* params, float* exp_avg, float* exp_avg_sq, int64_t* adam_step_io,
                  const float* obs, const float* action, const float* old_logp, const float* advantage,
                  const float* target, int64_t n_samples, const int64_t* perms, int32_t epochs, int64_t batch,
                  int64_t max_minibatches_per_epoch, const b200ppo_hparams* hp, float* losses_out,
                  b200ppo_stream stream);

/* End-to-end entry point with HOST buffers (pinned or pageable): advantage pipeline + PPO.train for one
 * rollout.  Copies the rollout host→device, runs b200ppo_gae + b200ppo_train, copies the per-minibatch
 * losses back and synchronises `stream`.  Parameters and Adam state stay on the device.
 * replaces: PPO._iterate minus rollout, ppo.py:158-159. */
int b200ppo_update_host(b200ppo_ctx* ctx, float* params, float* exp_avg, float* exp_avg_sq, int64_t* adam_step_io,
                        const float* obs_host, const float* action_host, const float* old_logp_host,
                        const float* reward_host, const float* value_host, const float* next_value_host,
                        const uint8_t* terminated_host, int64_t n_envs, int64_t n_steps, double gamma, double lmbda,
                        int normalize_rewards, int normalize_advantage, double advantage_scaler,
                        const int64_t* perms_host, int32_t epochs, int64_t batch,
                        int64_t max_minibatches_per_epoch, const b200ppo_hparams* hp, float* losses_host,
                        b200ppo_stream stream);

/* The same in two halves, for a caller that can hand over rollout k + 1 while rollout k is still being trained on:
 * `_begin` only enqueues the host->device copies of one rollout on the library's copy stream into staging set `slot`
 * (0 or 1) and returns; `_end` makes `stream` wait for them (the advantage pass for the four small arrays only, so it
 * runs while the observations still stream in), runs b200ppo_gae + b200ppo_train, copies the losses back and
 * synchronises `stream`.  begin(k + 1, slot ^ 1) may be called before end(k, slot): the upload (875 MB at the bench
 * shape, PCIe-bound) then hides behind the update.  The host buffers of a slot must stay valid until its `_end` returns.
 * replaces: ppo.py:158-159 across consecutive iterations. */
int b200ppo_update_host_begin(b200ppo_ctx* ctx, const float* obs_host, const float* action_host, const float* old_logp_host,
                              const float* reward_host, const float* value_host, const float* next_value_host,
                              const uint8_t* terminated_host, int64_t n_envs, int64_t n_steps, const int64_t* perms_host,
                              int32_t epochs, int32_t slot);
int b200ppo_update_host_end(b200ppo_ctx* ctx, float* params, float* exp_avg, float* exp_avg_sq, int64_t* adam_step_io,
                            double gamma, double lmbda, int normalize_rewards, int normalize_advantage, double advantage_scaler,
                            int64_t batch, int64_t max_minibatches_per_epoch, const b200ppo_hparams* hp, float* losses_host,
                            int32_t slot, b200ppo_stream stream);

/* ---------------------------------------------------------------------------------------------
 * Observation normalisation feeding the policy (SURVEY.md §8f rank 3).
 * replaces: EnvironmentHelper.normalize_state/_normalize/get_state,
 *           src/environments/humanoid/running_gym_sequential_vectorized.py:61-92.
 *   obs        [N, obs_dim, window] fp32, or fp64 when obs_is_f64 (gym observations)
 *   seg_bounds device int32 [n_segments + 1]: each range [b_s, b_{s+1}) of the observation vector is centred and
 *              divided by its unbiased std (std == 0 -> 1) per env and per frame, in the input's precision;
 *              normalize = 0 skips that and only casts / permutes (run.normalize_observations = False)
 *   out        [N, window, obs_dim] fp32 (the permute(0, 2, 1) of get_state)
 */
int b200ppo_normalize_obs(const void* obs, int obs_is_f64, int64_t n_envs, int32_t obs_dim, int32_t window,
                          const int32_t* seg_bounds, int32_t n_segments, int normalize, float* out, b200ppo_stream stream);

/* ---------------------------------------------------------------------------------------------
 * Instrumentation (used by bench.py; no reference counterpart).
 * b200ppo_launch_count: CUDA kernels this library has launched in this process so far.
 * b200ppo_profile_begin/end: between the two calls every kernel group launched by b200ppo_train on this
 * context is bracketed by CUDA events on its stream; _end synchronises and returns, per class, the summed
 * device time in ms and the number of timed groups (a forward "group" is one launch per layer).
 */
#define B200PPO_PROF_GATHER 0
#define B200PPO_PROF_GEMM_FWD 1
#define B200PPO_PROF_LOSS 2
#define B200PPO_PROF_GEMM_DGRAD 3
#define B200PPO_PROF_GEMM_WGRAD 4
#define B200PPO_PROF_ADAM 5
#define B200PPO_PROF_ALLREDUCE 6
#define B200PPO_PROF_OTHER 7
#define B200PPO_PROF_CLASSES 8
/* Deferred device-side errors of the asynchronous entry points (b200ppo_train, the gathers inside it): synchronises
 * `stream`, reads and clears the context's error word.  B200PPO_EINDEX: a permutation entry was outside [0, n_samples)
 * (those rows were skipped; the reference raises IndexError at ppo.py:104).  B200PPO_ENCCL: the peer-memory gradient
 * exchange timed out on a rank (B200PPO_PEER_TIMEOUT_MS, default 30000) — the optimizer step of that minibatch was NOT
 * applied on this rank.  b200ppo_update_host polls by itself. */
int b200ppo_poll_error(b200ppo_ctx* ctx, b200ppo_stream stream);

int64_t b200ppo_launch_count(void);
int b200ppo_profile_begin(b200ppo_ctx* ctx);
int b200ppo_profile_end(b200ppo_ctx* ctx, double ms_out[B200PPO_PROF_CLASSES], int64_t launches_out[B200PPO_PROF_CLASSES]);
/* Test hook for the tcgen05 GEMM kernel: C[M,N] (fp32) = A * B^T with operands rounded to bf16.  A is [M,K]
 * (a_mn_major = 0) or [K,M] (a_mn_major = 1); B is [N,K] or [K,N]; bn in {64,128,192,256}, or -1 for the
 * persistent weights-stationary kernel (K-major A, N <= 256, split_k = 1); -3: its forward epilogue,
 * C = float(bf16(tanh(A B^T))); -4: its dgrad epilogue, C holds the activation operand h on entry and
 * float(bf16(A B^T (1 - bf16(h)^2))) on return; split_k >= 1.
 * Allocates temporaries and synchronises `stream`. */
int b200ppo_debug_tc_gemm(const float* A, const float* B, float* C, int32_t M, int32_t N, int32_t K, int32_t a_mn_major,
                          int32_t b_mn_major, int32_t bn, int32_t split_k, b200ppo_stream stream);

/* One environment step of the rollout written straight into the env-major [N, T, ...] buffers (replaces the per-step
 * get_state_value / act / log_prob calls and TensorDict appends of src/entities/algorithms/ppo.py:20-49): at time index t
 * buf_state[:, t] = obs, buf_value[:, t] = V(obs), buf_action[:, t] = mean(obs) + sigma * noise (noise NULL: the mean),
 * buf_logp[:, t] = log-prob of that action, and — for t > 0 — buf_next_value[:, t - 1] = V(obs): the reference's second critic
 * call per step evaluates the tensor that becomes the next step's current_state (ppo.py:21,27-29), so T + 1 critic
 * evaluations fill both value buffers instead of 2 T.  t == T: only buf_next_value[:, T - 1] (pass the final state).
 * bf16 contexts with 256-wide nets: one tensor-core launch behind the two bf16 casts.  buf_state / buf_next_value nullable. */
int b200ppo_rollout_step(b200ppo_ctx* ctx, const float* params, const float* obs, int64_t n_envs, const float* noise, int64_t t,
                         int64_t T, float* buf_state, float* buf_value, float* buf_next_value, float* buf_action, float* buf_logp,
                         b200ppo_stream stream);

/* fp32-precision contexts, GEMMs large enough for the tensor-core route (csrc/gemm_split.cu): how an fp32 operand value is
 * handed to tcgen05.  3 (default): three bf16 terms, six products per fp32 product — 24-bit operands, north_star's 1e-5
 * variant.  2: two fp16 terms of the value scaled by a power of two taken from the tensor's largest magnitude, three
 * products — 22-bit operands, about 1.3x faster; gradients stay within 1e-5 of their tensor's scale, sums that cancel
 * 1000 : 1 do not (DESIGN.md §3.3). */
int b200ppo_set_fp32_terms(b200ppo_ctx* ctx, int32_t terms);

/* Test hook for the fp32-tolerance tensor-core GEMM (csrc/gemm_split.cu: three bf16 terms per operand value, six products):
 * C[M,N] = A * B^T with the operand layouts of b200ppo_debug_tc_gemm, `split_k` split-K partials summed in order;
 * bias_grad (nullable; both operands MN-major): bias_grad[m] = sum_k A(m,k), read off the ones-column the split appends.
 * Allocates temporaries and synchronises `stream`. */
int b200ppo_debug_gemm_split(const float* A, const float* B, float* C, float* bias_grad, int32_t M, int32_t N, int32_t K,
                             int32_t a_mn_major, int32_t b_mn_major, int32_t split_k, b200ppo_stream stream);

/* Test hook: the bf16 intermediates the last bf16 minibatch left in the context, as fp32 [rows][dims[layer]].
 * kind 0: hidden activation H_layer (layer < n_layers - 1); kind 1: dL/dz of `layer` (the seeds for the output layer). */
int b200ppo_debug_activations(b200ppo_ctx* ctx, int32_t net, int32_t kind, int32_t layer, int64_t rows, float* out,
                              b200ppo_stream stream);

/* Polyak averaging, in place: target[i] = target[i] * (1 - tau) + source[i] * tau over flat fp32 buffers.
 * replaces: soft_update, src/entities/algorithms/soft_actor_critic.py:12-14 (SURVEY 8f rank 4: the SAC update step). */
int b200ppo_polyak_update(float* target, const float* source, int64_t n, double tau, b200ppo_stream stream);

/* ---------------------------------------------------------------------------------------------
 * Multi-GPU (one process per GPU).  The update is data-parallel over samples: every rank computes the
 * gradient of its slice of each minibatch, gradients are summed over ranks (NCCL all-reduce over
 * NVLink), every rank applies the same Adam step.  Loss means use the GLOBAL minibatch size.
 * unique_id: the 128-byte ncclUniqueId from b200ppo_comm_unique_id on rank 0, distributed by the caller.
 */
int b200ppo_comm_unique_id(uint8_t id_out[128]);
int b200ppo_comm_init(b200ppo_ctx* ctx, const uint8_t unique_id[128], int32_t rank, int32_t world_size);
int b200ppo_comm_world(const b200ppo_ctx* ctx, int32_t* rank, int32_t* world_size);
/* Layout of the `perms` argument of b200ppo_train on this rank.  0 (default): the global permutations,
 * [epochs][n_samples].  1: only the slots this rank consumes, [epochs][floor(n_samples / batch)][batch / world_size] —
 * slot (e, i, j) = global slot e * n_samples + i * batch + rank * (batch / world_size) + j (the rows of
 * `distributed.rank_rows`) — so that a rank uploads 1 / world_size of the index bytes.  The result is identical.
 * replaces: nothing in the reference (its `torch.randperm`, ppo.py:103, is consumed whole by one process). */
int b200ppo_set_perm_layout(b200ppo_ctx* ctx, int32_t rank_slices);
/* Optional, after b200ppo_comm_init, bf16 path, world_size <= 8 on one NVLink/NVSwitch node: replace the per-minibatch
 * ncclAllReduce by an exchange over peer-mapped memory fused into the optimizer kernel.  Every rank exports the
 * 64-byte cudaIpcMemHandle of its exchange buffer, the caller all-gathers the handles (rank order) and hands the
 * world_size x 64 bytes to every rank, then b200ppo_p2p_enable(ctx, 1) on every rank.  Same result on every rank; ranks
 * sum in rank order. */
int b200ppo_p2p_export(b200ppo_ctx* ctx, uint8_t handle_out[64]);
int b200ppo_p2p_import(b200ppo_ctx* ctx, const uint8_t* handles, int32_t world_size);
/* Switch the exchange on once EVERY rank has imported successfully (the caller agrees on that with a collective), or off. */
int b200ppo_p2p_enable(b200ppo_ctx* ctx, int32_t on);
/* Optional (same conditions): share the rollout's observations between ranks without an all-gather.  Every rank keeps
 * its own env slab as a bf16 table (rows of in_dim values + the ones-column) that its peers map over NVLink;
 * b200ppo_train(obs = NULL, n_samples = world_size * rows_local) then gathers the rows of the GLOBAL permutation
 * straight from the owners' tables with the copy engine, on a side stream behind the previous epoch's kernels.
 * replaces: nothing in the reference (single process); it stands in for gathering `memory['current_state']` of
 * src/entities/algorithms/ppo.py:104 when that tensor is spread over ranks.
 * export (re)allocates the table for rows_local rows and returns its cudaIpcMemHandle; import takes the handles of all
 * ranks (rank order); fill converts the rank's fp32 slab [rows_local, in_dim] on `stream`.  The caller orders fill
 * before every peer's train (e.g. the all-gather of the small leaves on the same stream) and the next fill after every
 * peer's train (any collective). */
int b200ppo_table_export(b200ppo_ctx* ctx, int64_t rows_local, uint8_t handle_out[64]);
int b200ppo_table_import(b200ppo_ctx* ctx, const uint8_t* handles, int32_t world_size, int64_t rows_local);
int b200ppo_table_fill(b200ppo_ctx* ctx, const float* obs_local, int64_t rows_local, b200ppo_stream stream);
/* Optional, after EVERY rank's b200ppo_table_fill has completed (e.g. behind a collective that follows the fill in stream
 * order on all ranks): copies the peers' tables into local memory once ((world - 1) x rows x pitch bf16 over NVLink), so
 * that the per-epoch gathers of b200ppo_train(obs = NULL, ...) read local HBM instead of pulling 1 - 1/world of every
 * epoch's rows from the peers.  The next b200ppo_table_fill invalidates the copy. */
int b200ppo_table_replicate(b200ppo_ctx* ctx, b200ppo_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* B200PPO_H_ */
