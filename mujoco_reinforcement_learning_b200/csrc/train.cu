// The PPO update: epochs of shuffled minibatches, each a forward / backward and an optimizer step, on one GPU or with
// the gradients exchanged across ranks; and the host-staged variant that uploads a rollout and runs GAE first.
//
// replaces: the Python control flow of PPO.train (src/entities/algorithms/ppo.py:93-154).
#include <algorithm>

#include "context.cuh"
#include "gather.cuh"

namespace b200ppo {

__global__ void copy2_kernel(const float* __restrict__ src, float* __restrict__ dst) {
  if (threadIdx.x < 2) dst[threadIdx.x] = src[threadIdx.x];
}

namespace {

struct ScopedFlag {  // clears the flag when the call returns, however it returns
  bool& f;
  ~ScopedFlag() { f = false; }
};

// Both buffer sets of the shuffled epochs, for `rows` rows each; the side stream and events of the epoch-ahead gather.
int ensure_shuffle_capacity(b200ppo_ctx* ctx, int64_t rows) {
  if (rows <= ctx->sh_cap) return B200PPO_OK;
  B2_CUDA(cudaDeviceSynchronize());
  for (auto* b : {&ctx->sh_obs, &ctx->sh_act, &ctx->sh_logp, &ctx->sh_adv, &ctx->sh_tgt}) b->reset();
  ctx->bf.sh_obs.reset();
  ctx->sh_cap = 0;
  const int D = ctx->net[0].d.in_dim, A = ctx->net[0].out_dim();
  if (ctx->precision == B200PPO_PREC_BF16) B2_TRY(ctx->bf.sh_obs.alloc(2 * rows * ctx->bf.pitchX));
  else B2_TRY(ctx->sh_obs.alloc(2 * rows * D));
  B2_TRY(ctx->sh_act.alloc(2 * rows * A));
  B2_TRY(ctx->sh_logp.alloc(2 * rows));
  B2_TRY(ctx->sh_adv.alloc(2 * rows));
  B2_TRY(ctx->sh_tgt.alloc(2 * rows));
  ctx->sh_cap = rows;
  if (ctx->gather_stream == nullptr) {
    B2_CUDA(cudaStreamCreateWithFlags(&ctx->gather_stream, cudaStreamNonBlocking));
    for (int i = 0; i < 2; ++i) {
      B2_CUDA(cudaEventCreateWithFlags(&ctx->ev_ready[i], cudaEventDisableTiming));
      B2_CUDA(cudaEventCreateWithFlags(&ctx->ev_free[i], cudaEventDisableTiming));
    }
    B2_CUDA(cudaEventCreateWithFlags(&ctx->ev_start, cudaEventDisableTiming));
  }
  return B200PPO_OK;
}

// Where an epoch's minibatch observations come from.
enum class ObsSource {
  kShared,   // every rank's bf16 table (b200ppo_table_*), or the local replica of it, pulled by the copy engine
  kTable,    // the rollout converted to bf16 once (ctx->bf.obs_table), rows gathered byte for byte
  kConvert,  // fp32 rollout rows converted to bf16 as they are gathered
  kFp32,     // fp32 rows (fp32 contexts)
};

// Every epoch gathers `rows` observation rows.  Converting on the fly reads 4D and writes 2*pitch bytes per row and
// epoch; converting the whole rollout ONCE and then gathering bf16 rows byte for byte (bulk-copy kernel) costs
// n_samples*(4D + 2*pitch) up front and 4*pitch per row and epoch.  Same bits either way.
ObsSource pick_obs_source(const b200ppo_ctx* ctx, bool shared, int64_t n_samples, int64_t rows, int epochs) {
  if (shared) return ObsSource::kShared;
  if (ctx->precision != B200PPO_PREC_BF16) return ObsSource::kFp32;
  const int D = ctx->net[0].d.in_dim, PX = ctx->bf.pitchX;
  if (PX % 8 == 0) {
    const double direct = double(epochs) * double(rows) * (4.0 * D + 2.0 * PX);
    const double pre = double(n_samples) * (4.0 * D + 2.0 * PX) + double(epochs) * double(rows) * 4.0 * PX;
    if (pre < 0.9 * direct && rows >= 4096) return ObsSource::kTable;
  }
  return ObsSource::kConvert;
}

// The gather every epoch repeats: `job` addresses epoch 0 and writes buffer set 0.
struct EpochGather {
  GatherJob job;
  int64_t perm_stride;  // entries of `perms` per epoch
  ObsSource source;
  const float* obs;     // the caller's fp32 observations (kConvert, kFp32)
};

int gather_epoch(b200ppo_ctx* ctx, const EpochGather& g, int e, int set, cudaStream_t st) {
  const int D = ctx->net[0].d.in_dim, A = ctx->net[0].out_dim(), PX = ctx->bf.pitchX;
  const int64_t o = int64_t(set) * ctx->sh_cap;
  GatherJob j = g.job;
  j.idx += int64_t(e) * g.perm_stride;
  j.act_o += o * A; j.logp_o += o; j.adv_o += o; j.tgt_o += o;
  switch (g.source) {
    case ObsSource::kShared: {  // rows pulled from every rank's table over NVLink by the copy engine
      const float* parts[kMaxPeers];
      for (int r = 0; r < ctx->world; ++r)
        parts[r] = reinterpret_cast<const float*>((ctx->replicated && r != ctx->rank) ? ctx->replica + int64_t(r) * ctx->shared_rows * PX
                                                                                        : ctx->peer_table[r]);
      return launch_gather_parts(j, parts, ctx->world, ctx->shared_rows, PX / 2, reinterpret_cast<float*>(ctx->bf.sh_obs + o * PX), st);
    }
    case ObsSource::kTable:  // bf16 rows moved as PX/2 "floats" by the bulk-copy gather: a byte copy
      return launch_gather_chunked(j, reinterpret_cast<const float*>(ctx->bf.obs_table.get()), PX / 2,
                                   reinterpret_cast<float*>(ctx->bf.sh_obs + o * PX), st);
    case ObsSource::kConvert:
      return launch_gather_chunked_bf16(j, g.obs, D, ctx->bf.sh_obs + o * PX, PX, st);
    case ObsSource::kFp32:
      return launch_gather_chunked(j, g.obs, D, ctx->sh_obs + o * D, st);
  }
  return B200PPO_OK;
}

// How the ranks combine their gradients before the optimizer step.
enum class Exchange { kSingle, kP2p, kNccl };

// The optimizer state of one b200ppo_train call and the Adam factors of the current step.
struct Step {
  float *params, *exp_avg, *exp_avg_sq;
  const b200ppo_hparams* hp;
  int64_t lb;  // rows of each minibatch on this rank
  AdamScalars sa, sc;
};

float* p2p_buffer(const b200ppo_ctx* ctx, unsigned seq) { return ctx->xbuf + int64_t(seq & 1) * ctx->xstride; }

PeerSrc peer_src(b200ppo_ctx* ctx, unsigned seq, float* loss_slot) {
  PeerSrc ps{};
  ps.world = ctx->world; ps.rank = ctx->rank; ps.seq = seq; ps.err = ctx->err_flag; ps.losses_out = loss_slot;
  static const long long timeout_ms = []() { const char* e = getenv("B200PPO_PEER_TIMEOUT_MS"); return e ? atoll(e) : 30000ll; }();
  ps.timeout_cycles = timeout_ms * 2000000ll;  // ~2 GHz SM clock
  ps.flags_local = reinterpret_cast<unsigned*>(ctx->xbuf + 2 * ctx->xstride);
  const int64_t xo = int64_t(seq & 1) * ctx->xstride;
  for (int r = 0; r < ctx->world; ++r) {
    ps.src[r] = ctx->peer_x[r] + xo;
    ps.flags_peer[r] = reinterpret_cast<unsigned*>(ctx->peer_x[r] + 2 * ctx->xstride);
  }
  return ps;
}

// Adam on the gradient partials `grads` (+ for bf16, in the same pass, the re-cast of the weights and the finish `lc` of
// the fused-epilogue loss partials).
int adam(b200ppo_ctx* ctx, const Step& s, const float* grads, int n_partials, const LossCombine& lc, cudaStream_t st,
         const PeerSrc* ps = nullptr) {
  if (ctx->precision == B200PPO_PREC_BF16)
    PROF(ctx, B200PPO_PROF_ADAM, st,
         launch_adam_cast(s.params, grads, n_partials, ctx->n_params, s.exp_avg, s.exp_avg_sq, ctx->n_params, ctx->n_actor, s.sa,
                          s.sc, cast_group(ctx, s.params), lc, st, ps));
  else
    PROF(ctx, B200PPO_PROF_ADAM, st,
         launch_adam(s.params, grads, n_partials, ctx->n_params, s.exp_avg, s.exp_avg_sq, ctx->n_params, ctx->n_actor, s.sa, s.sc,
                     nullptr, st));
  return B200PPO_OK;
}

// Peer-memory exchange fused into the optimizer kernel (bf16): reduce the split-K partials into this rank's exchange
// buffer, then Adam waits for the peers' flags and sums the G buffers in rank order (adam.cu).
int optimizer_p2p(b200ppo_ctx* ctx, const Step& s, int split, int loss_ctas, unsigned seq, float* loss_slot, cudaStream_t st) {
  float* xb = p2p_buffer(ctx, seq);
  const LossCombine lc = make_loss_combine(ctx, s.params, loss_ctas, s.lb, s.hp, xb + ctx->n_params);
  // the sum of this rank's split-K partials into its exchange buffer happens inside the optimizer kernel (one
  // element per thread); a small grid or no loss partials keep the separate launch in front of it
  const int agrid = adam_cast_grid(ctx->n_params);
  const bool fused = loss_ctas > 0 && int64_t(agrid) * 256 >= ctx->n_params / 4;
  PeerSrc ps = peer_src(ctx, seq, loss_slot);
  if (!fused) {
    PROF(ctx, B200PPO_PROF_OTHER, st, launch_reduce_partials(ctx->gpart, split, ctx->n_params, ctx->n_params, xb, st, &lc));
    return adam(ctx, s, xb, 1, LossCombine{}, st, &ps);
  }
  ps.local_out = xb;
  ps.done_counter = ctx->done_counter;
  ctx->done_total += unsigned(agrid);
  ps.done_target = ctx->done_total;
  return adam(ctx, s, ctx->gpart, split, lc, st, &ps);
}

// NCCL: the reduced gradient and the two loss sums (grad_flat) all-reduced, then Adam on the sum.
int optimizer_nccl(b200ppo_ctx* ctx, const Step& s, int split, int loss_ctas, float* loss_slot, cudaStream_t st) {
  float* red_losses = ctx->grad_flat + ctx->n_params;
  const LossCombine lc = make_loss_combine(ctx, s.params, loss_ctas, s.lb, s.hp, red_losses);
  PROF(ctx, B200PPO_PROF_OTHER, st, launch_reduce_partials(ctx->gpart, split, ctx->n_params, ctx->n_params, ctx->grad_flat, st, &lc));
  PROF(ctx, B200PPO_PROF_ALLREDUCE, st, nccl_all_reduce(ctx->grad_flat, ctx->n_params + 4, ctx->comm, st));
  B2_TRY(adam(ctx, s, ctx->grad_flat, 1, LossCombine{}, st));
  copy2_kernel<<<1, 32, 0, st>>>(red_losses, loss_slot);
  B2_LAUNCH_CHECK();
  return B200PPO_OK;
}

// Makes epoch e's rows ready on `st`: gathered there, or (overlap) gathered one epoch ahead on the side stream into the
// other buffer set.
int begin_epoch(b200ppo_ctx* ctx, const EpochGather& g, int e, int epochs, bool overlap, cudaStream_t st) {
  if (!overlap) {
    PROF(ctx, B200PPO_PROF_GATHER, st, gather_epoch(ctx, g, e, 0, st));
    return B200PPO_OK;
  }
  if (e == 0) {
    B2_CUDA(cudaEventRecord(ctx->ev_start, st));  // the rollout (and the bf16 table) are complete on the caller's stream
    B2_CUDA(cudaStreamWaitEvent(ctx->gather_stream, ctx->ev_start, 0));
    B2_TRY(gather_epoch(ctx, g, 0, 0, ctx->gather_stream));
    B2_CUDA(cudaEventRecord(ctx->ev_ready[0], ctx->gather_stream));
  }
  if (e + 1 < epochs) {
    if (e >= 1) B2_CUDA(cudaStreamWaitEvent(ctx->gather_stream, ctx->ev_free[(e + 1) & 1], 0));  // epoch e-1 is done with that set
    B2_TRY(gather_epoch(ctx, g, e + 1, (e + 1) & 1, ctx->gather_stream));
    B2_CUDA(cudaEventRecord(ctx->ev_ready[(e + 1) & 1], ctx->gather_stream));
  }
  B2_CUDA(cudaStreamWaitEvent(st, ctx->ev_ready[e & 1], 0));
  return B200PPO_OK;
}

}  // namespace
}  // namespace b200ppo

using namespace b200ppo;

extern "C" B2_EXPORT int b200ppo_train(b200ppo_ctx* ctx, float* params, float* exp_avg, float* exp_avg_sq,
                             int64_t* adam_step_io, const float* obs, const float* action, const float* old_logp,
                             const float* advantage, const float* target, int64_t n_samples, const int64_t* perms,
                             int32_t epochs, int64_t batch, int64_t max_minibatches_per_epoch,
                             const b200ppo_hparams* hp, float* losses_out, b200ppo_stream stream) {
  B2_CHECK_ARG(ctx && params && exp_avg && exp_avg_sq && adam_step_io && action && old_logp && advantage && target && perms && hp,
               "b200ppo_train: null pointer");
  const bool shared_obs = obs == nullptr;  // observations come from the ranks' shared bf16 tables (b200ppo_table_*)
  B2_CHECK_ARG(!shared_obs || (ctx->shared_rows > 0 && ctx->shared_filled && ctx->precision == B200PPO_PREC_BF16 &&
                               n_samples == ctx->shared_rows * ctx->world),
               "b200ppo_train: obs == NULL needs filled shared observation tables covering n_samples = world x rows");
  B2_CHECK_ARG(epochs >= 0 && batch > 0 && n_samples >= 0, "b200ppo_train: bad sizes");
  B2_CHECK_ARG(batch % ctx->world == 0, "b200ppo_train: batch %lld not divisible by world size %d", (long long)batch, ctx->world);
  const int64_t lb = batch / ctx->world;  // rows of each minibatch owned by this rank
  B2_TRY(check_batch(ctx, lb, "b200ppo_train"));
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int64_t nb = n_samples / batch;  // int(T*N / batch_size): the tail is dropped (ppo.py:97-98,107-108)
  if (max_minibatches_per_epoch > 0) nb = std::min(nb, max_minibatches_per_epoch);
  if (nb == 0 || epochs == 0) return B200PPO_OK;
  B2_TRY(ensure_shuffle_capacity(ctx, nb * lb));
  const int D = ctx->net[0].d.in_dim, A = ctx->net[0].out_dim(), PX = ctx->bf.pitchX;
  const bool tc = ctx->precision == B200PPO_PREC_BF16;
  if (tc) PROF(ctx, B200PPO_PROF_OTHER, st, cast_weights(ctx, params, st));
  // fp32-tolerance tensor-core GEMMs: the largest observation of the rollout bounds every minibatch's rows, so their fp16
  // scale needs no measuring pass per minibatch (gemm.cuh a_bound_dev)
  ScopedFlag bound_flag{ctx->obs_amax_ok};
  if (!tc && !shared_obs && ctx->arena_need > 0 && lb * int64_t(D) >= (1 << 20)) {
    PROF(ctx, B200PPO_PROF_OTHER, st, launch_absmax(obs, n_samples, D, D, ctx->obs_amax, st));
    ctx->obs_amax_ok = true;
  }
  EpochGather g{};
  g.source = pick_obs_source(ctx, shared_obs, n_samples, nb * lb, epochs);
  g.obs = obs;
  if (g.source == ObsSource::kTable) {
    B2_TRY(ctx->bf.obs_table.grow(n_samples * PX));
    PROF(ctx, B200PPO_PROF_GATHER, st, launch_cast_rows_ones(obs, n_samples, D, ctx->bf.obs_table, PX, st));
  }
  // shuffled_memory = memory[idx] restricted to the rows this rank will consume (ppo.py:103-106).  Global permutations:
  // rank r's rows of minibatch i sit at slots i * batch + r * lb ...; rank slices: at i * lb ...
  const bool sliced = ctx->perm_rank_slices;
  GatherJob& j = g.job;
  j.idx = perms; j.count = nb * lb; j.n_rows = n_samples;
  j.chunk = lb; j.chunk_stride = sliced ? lb : batch; j.chunk_offset = sliced ? 0 : int64_t(ctx->rank) * lb;
  j.act = action; j.act_dim = A; j.logp = old_logp; j.adv = advantage; j.tgt = target;
  j.act_o = ctx->sh_act; j.logp_o = ctx->sh_logp; j.adv_o = ctx->sh_adv; j.tgt_o = ctx->sh_tgt; j.err_flag = ctx->err_flag;
  g.perm_stride = sliced ? (n_samples / batch) * lb : n_samples;
  // The permutations are known up front, so the gather of epoch e + 1 runs on a side stream into the other buffer set
  // while epoch e trains: the update kernels are latency-bound and leave HBM idle, the copy engine work hides behind them.
  const bool overlap = epochs > 1 && !ctx->prof.on;
  const Exchange mode = ctx->world == 1 ? Exchange::kSingle : (ctx->p2p && tc) ? Exchange::kP2p : Exchange::kNccl;
  Step s{params, exp_avg, exp_avg_sq, hp, lb, {}, {}};
  int64_t step = *adam_step_io;
  ScopedFlag epoch_flag{ctx->in_epoch};
  for (int e = 0; e < epochs; ++e) {
    const int set = overlap ? (e & 1) : 0;
    B2_TRY(begin_epoch(ctx, g, e, epochs, overlap, st));
    for (int64_t i = 0; i < nb; ++i) {
      const int64_t r0 = int64_t(set) * ctx->sh_cap + i * lb;
      // from the second minibatch of an epoch on, the kernel in front of the chain kernel is this epoch's optimizer step
      // and the minibatch's rows were gathered before it: the chain kernel may prefetch them across the PDL boundary
      ctx->in_epoch = i > 0;
      float* loss_slot = losses_out ? losses_out + (int64_t(e) * nb + i) * 2 : ctx->scratch;
      ++step;
      s.sa = make_adam_scalars(hp->learning_rate_actor, hp->beta1, hp->beta2, hp->adam_eps, step);
      s.sc = make_adam_scalars(hp->learning_rate_critic, hp->beta1, hp->beta2, hp->adam_eps, step);
      const unsigned seq = mode == Exchange::kP2p ? ++ctx->p2p_seq : 0;
      float* loss_dst = mode == Exchange::kSingle ? loss_slot
                        : mode == Exchange::kP2p  ? p2p_buffer(ctx, seq) + ctx->n_params
                                                  : ctx->grad_flat + ctx->n_params;
      int split = 1, loss_ctas = 0;
      B2_TRY(minibatch_fwd_bwd(ctx, params, tc ? nullptr : ctx->sh_obs + r0 * D, tc ? ctx->bf.sh_obs + r0 * PX : nullptr,
                               ctx->sh_act + r0 * A, ctx->sh_logp + r0, ctx->sh_adv + r0, ctx->sh_tgt + r0, lb, hp, loss_dst,
                               &split, &loss_ctas, st));
      if (mode == Exchange::kSingle) B2_TRY(adam(ctx, s, ctx->gpart, split, make_loss_combine(ctx, params, loss_ctas, lb, hp, loss_slot), st));
      else if (mode == Exchange::kP2p) B2_TRY(optimizer_p2p(ctx, s, split, loss_ctas, seq, loss_slot, st));
      else B2_TRY(optimizer_nccl(ctx, s, split, loss_ctas, loss_slot, st));
    }
    if (overlap) B2_CUDA(cudaEventRecord(ctx->ev_free[set], st));
  }
  *adam_step_io = step;
  return B200PPO_OK;
}

extern "C" B2_EXPORT int b200ppo_update_host_begin(b200ppo_ctx* ctx, const float* obs_host, const float* action_host,
                                                   const float* old_logp_host, const float* reward_host, const float* value_host,
                                                   const float* next_value_host, const uint8_t* terminated_host, int64_t n_envs,
                                                   int64_t n_steps, const int64_t* perms_host, int32_t epochs, int32_t slot) {
  B2_CHECK_ARG(ctx == nullptr || !ctx->perm_rank_slices, "b200ppo_update_host: takes the global permutations (b200ppo_set_perm_layout(ctx, 0))");
  B2_CHECK_ARG(ctx && obs_host && action_host && old_logp_host && reward_host && value_host && next_value_host &&
                   terminated_host && perms_host,
               "b200ppo_update_host: null pointer");
  B2_CHECK_ARG(n_envs > 0 && n_steps > 0 && epochs > 0 && (slot == 0 || slot == 1), "b200ppo_update_host: bad sizes");
  const int64_t M = n_envs * n_steps;
  const int D = ctx->net[0].d.in_dim, A = ctx->net[0].out_dim();
  auto& h = ctx->host[slot];
  if (ctx->copy_stream == nullptr) B2_CUDA(cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking));
  if (h.ev_small == nullptr) {
    B2_CUDA(cudaEventCreateWithFlags(&h.ev_small, cudaEventDisableTiming));
    B2_CUDA(cudaEventCreateWithFlags(&h.ev_all, cudaEventDisableTiming));
  }
  if (h.rows < M) {
    B2_CUDA(cudaDeviceSynchronize());
    for (auto* b : {&h.obs, &h.act, &h.logp, &h.rew, &h.val, &h.nval, &h.adv, &h.tgt}) b->reset();
    h.term.reset();
    h.rows = 0;
    B2_TRY(h.obs.alloc(M * D)); B2_TRY(h.act.alloc(M * A)); B2_TRY(h.logp.alloc(M));
    B2_TRY(h.rew.alloc(M)); B2_TRY(h.val.alloc(M)); B2_TRY(h.nval.alloc(M));
    B2_TRY(h.adv.alloc(M)); B2_TRY(h.tgt.alloc(M)); B2_TRY(h.term.alloc(M));
    h.rows = M;
  }
  B2_TRY(h.perms.grow(int64_t(epochs) * M));
  h.n_envs = n_envs; h.n_steps = n_steps; h.epochs = epochs;
  cudaStream_t cs = ctx->copy_stream;
  const auto H2D = cudaMemcpyHostToDevice;
  // the advantage pass only needs the four small arrays: they go first, so that it runs while the observations stream in
  B2_CUDA(cudaMemcpyAsync(h.rew, reward_host, size_t(M) * 4, H2D, cs));
  B2_CUDA(cudaMemcpyAsync(h.val, value_host, size_t(M) * 4, H2D, cs));
  B2_CUDA(cudaMemcpyAsync(h.nval, next_value_host, size_t(M) * 4, H2D, cs));
  B2_CUDA(cudaMemcpyAsync(h.term, terminated_host, size_t(M), H2D, cs));
  B2_CUDA(cudaEventRecord(h.ev_small, cs));
  B2_CUDA(cudaMemcpyAsync(h.obs, obs_host, size_t(M) * D * 4, H2D, cs));
  B2_CUDA(cudaMemcpyAsync(h.act, action_host, size_t(M) * A * 4, H2D, cs));
  B2_CUDA(cudaMemcpyAsync(h.logp, old_logp_host, size_t(M) * 4, H2D, cs));
  B2_CUDA(cudaMemcpyAsync(h.perms, perms_host, size_t(epochs) * M * 8, H2D, cs));
  B2_CUDA(cudaEventRecord(h.ev_all, cs));
  return B200PPO_OK;
}

extern "C" B2_EXPORT int b200ppo_update_host_end(b200ppo_ctx* ctx, float* params, float* exp_avg, float* exp_avg_sq,
                                                 int64_t* adam_step_io, double gamma, double lmbda, int normalize_rewards,
                                                 int normalize_advantage, double advantage_scaler, int64_t batch,
                                                 int64_t max_minibatches_per_epoch, const b200ppo_hparams* hp, float* losses_host,
                                                 int32_t slot, b200ppo_stream stream) {
  B2_CHECK_ARG(ctx && params && exp_avg && exp_avg_sq && adam_step_io && hp && (slot == 0 || slot == 1), "b200ppo_update_host_end: bad argument");
  auto& h = ctx->host[slot];
  B2_CHECK_ARG(h.ev_all != nullptr && h.n_envs > 0 && batch > 0, "b200ppo_update_host_end: no upload was begun in slot %d", slot);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t M = h.n_envs * h.n_steps;
  int64_t nb = M / batch;
  if (max_minibatches_per_epoch > 0) nb = std::min(nb, max_minibatches_per_epoch);
  const int64_t n_loss = int64_t(h.epochs) * nb * 2;
  B2_TRY(h.losses.grow(n_loss));
  B2_CUDA(cudaStreamWaitEvent(st, h.ev_small, 0));
  B2_TRY(b200ppo_gae(h.rew, 0, h.val, h.nval, h.term, nullptr, h.n_envs, h.n_steps, gamma, lmbda, normalize_rewards,
                     normalize_advantage, advantage_scaler, h.adv, h.tgt, stream));
  B2_CUDA(cudaStreamWaitEvent(st, h.ev_all, 0));
  B2_TRY(b200ppo_train(ctx, params, exp_avg, exp_avg_sq, adam_step_io, h.obs, h.act, h.logp, h.adv, h.tgt, M, h.perms,
                       h.epochs, batch, max_minibatches_per_epoch, hp, h.losses, stream));
  if (losses_host && n_loss > 0)
    B2_CUDA(cudaMemcpyAsync(losses_host, h.losses, size_t(n_loss) * 4, cudaMemcpyDeviceToHost, st));
  h.n_envs = 0;  // consumed
  return b200ppo_poll_error(ctx, stream);  // synchronises the stream; bad permutation entries / peer time-outs fail the call
}

extern "C" B2_EXPORT int b200ppo_update_host(b200ppo_ctx* ctx, float* params, float* exp_avg, float* exp_avg_sq,
                                   int64_t* adam_step_io, const float* obs_host, const float* action_host,
                                   const float* old_logp_host, const float* reward_host, const float* value_host,
                                   const float* next_value_host, const uint8_t* terminated_host, int64_t n_envs,
                                   int64_t n_steps, double gamma, double lmbda, int normalize_rewards,
                                   int normalize_advantage, double advantage_scaler, const int64_t* perms_host,
                                   int32_t epochs, int64_t batch, int64_t max_minibatches_per_epoch,
                                   const b200ppo_hparams* hp, float* losses_host, b200ppo_stream stream) {
  B2_CHECK_ARG(hp && batch > 0, "b200ppo_update_host: bad argument");
  B2_TRY(b200ppo_update_host_begin(ctx, obs_host, action_host, old_logp_host, reward_host, value_host, next_value_host,
                                   terminated_host, n_envs, n_steps, perms_host, epochs, 0));
  return b200ppo_update_host_end(ctx, params, exp_avg, exp_avg_sq, adam_step_io, gamma, lmbda, normalize_rewards, normalize_advantage,
                                 advantage_scaler, batch, max_minibatches_per_epoch, hp, losses_host, 0, stream);
}

extern "C" B2_EXPORT int b200ppo_poll_error(b200ppo_ctx* ctx, b200ppo_stream stream) {
  B2_CHECK_ARG(ctx, "b200ppo_poll_error: null context");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  int32_t flag = 0;
  B2_CUDA(cudaMemcpyAsync(&flag, ctx->err_flag, sizeof(flag), cudaMemcpyDeviceToHost, st));
  B2_CUDA(cudaStreamSynchronize(st));
  if (ctx->gather_stream != nullptr) {  // an epoch gather may still be running on the side stream
    B2_CUDA(cudaStreamSynchronize(ctx->gather_stream));
    B2_CUDA(cudaMemcpy(&flag, ctx->err_flag, sizeof(flag), cudaMemcpyDeviceToHost));
  }
  if (flag == 0) return B200PPO_OK;
  B2_CUDA(cudaMemsetAsync(ctx->err_flag, 0, sizeof(flag), st));
  if (flag == B200PPO_ERRFLAG_PEER_TIMEOUT) {
    set_error("gradient exchange: a peer rank did not arrive within the timeout (B200PPO_PEER_TIMEOUT_MS); the update of that "
              "minibatch was skipped on this rank and the replicas are no longer in step");
    return B200PPO_ENCCL;
  }
  set_error("index out of range: a permutation entry lies outside [0, n_samples)");
  return B200PPO_EINDEX;
}
