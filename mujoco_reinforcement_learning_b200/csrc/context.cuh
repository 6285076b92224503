// The library context (b200ppo_ctx) and the passes that the C-ABI files share.
//
//   context.cu  create / destroy, parameter layout, profiling and debug accessors
//   passes.cu   forward / backward of both nets (fp32 and bf16), the fused chain kernel, one minibatch's gradients
//   api.cu      single-call entry points (forward, backward, inference, rollout step, evaluate, minibatch gradients)
//   train.cu    the epoch / minibatch loop and the host-staged update
//   comm.cu     multi-GPU: NCCL, the peer-memory gradient exchange and the shared observation tables
#pragma once
#include <vector>

#include "adam.cuh"
#include "cast.cuh"
#include "common.cuh"
#include "gemm.cuh"
#include "gemm_split.cuh"
#include "heads.cuh"
#include "ppo_loss.cuh"
#include "tc_chain.cuh"
#include "tc_gemm.cuh"

namespace b200ppo {

struct Net {
  b200ppo_mlp_desc d;
  int64_t w_off[B200PPO_MAX_LAYERS], b_off[B200PPO_MAX_LAYERS];
  int64_t seg_begin, seg_end;  // [begin, end) in the flat buffer (actor: includes logstd)
  int64_t hidden_sum;          // sum of hidden widths
  int in_dim(int l) const { return l == 0 ? d.in_dim : d.dims[l - 1]; }
  int out_dim() const { return d.dims[d.n_layers - 1]; }
  int64_t act_off(int l, int64_t B) const {  // hidden activation l (l < n_layers-1) inside an acts buffer
    int64_t s = 0;
    for (int i = 0; i < l; ++i) s += d.dims[i];
    return s * B;
  }
  int64_t dz_off(int l, int64_t B) const { return act_off(l, B); }  // dZ buffer also holds the last layer
};

// Optional per-kernel-class timing with CUDA events on the launching stream (bench.py's roofline numbers).
struct Profiler {
  bool on = false;
  struct Rec { int cls; cudaEvent_t a, b; };
  std::vector<Rec> recs;
  void begin(int cls, cudaStream_t st) {
    if (!on) return;
    Rec r{cls, nullptr, nullptr};
    cudaEventCreate(&r.a); cudaEventCreate(&r.b);
    cudaEventRecord(r.a, st);
    recs.push_back(r);
  }
  void end(cudaStream_t st) {
    if (!on) return;
    cudaEventRecord(recs.back().b, st);
  }
};

}  // namespace b200ppo

struct b200ppo_ctx {
  template <typename T>
  using DevBuf = b200ppo::DevBuf<T>;
  static constexpr int kMaxPeers = b200ppo::kMaxPeers;
  static constexpr int kMaxLayers = B200PPO_MAX_LAYERS;

  b200ppo::Profiler prof;
  b200ppo::Net net[2];
  int64_t logstd_off = 0, n_params = 0, n_actor = 0;
  int64_t max_batch = 0;
  int precision = 0;
  int max_split = 1;
  DevBuf<float> ws_act[2], ws_dz[2], ws_out[2];
  DevBuf<float> gpart;       // [max_split][n_params]
  DevBuf<float> grad_flat;   // [n_params + 4]: summed gradient + (actor_loss, critic_loss) for the all-reduce
  DevBuf<float> loss_partials;
  int64_t loss_partial_rows = 0;
  DevBuf<unsigned> ticket;
  DevBuf<unsigned> done_counter;  // fused reduce of the peer exchange: blocks of the optimizer grid that have written their slice (monotone)
  unsigned done_total = 0;        // what that counter reaches after the launches issued so far
  DevBuf<float> scratch;     // [8] losses / entropy scratch
  // three-term bf16 operands of the fp32-tolerance tensor-core GEMMs (gemm_split.cuh); allocated at first use
  mutable b200ppo::SplitArena arena;
  int64_t arena_need = 0;
  DevBuf<float> rollout_tmp;  // b200ppo_rollout_step, contexts without the one-launch path: value / action / log-prob of a step
  DevBuf<float> obs_amax;     // max |observation| of the rollout b200ppo_train is working on (a bound for every minibatch's rows)
  bool obs_amax_ok = false;   // valid: inside b200ppo_train's minibatch loop
  DevBuf<int32_t> err_flag;
  // shuffled-epoch buffers (train), all sized for sh_cap rows and grown together
  // two sets (rows [0, sh_cap) and [sh_cap, 2 sh_cap)): epoch e+1 is gathered on a side stream while epoch e trains
  DevBuf<float> sh_obs, sh_act, sh_logp, sh_adv, sh_tgt;
  int64_t sh_cap = 0;
  // peer-memory gradient exchange (multi-GPU, see adam.cuh PeerSrc): two buffers of xstride floats + a flag array, one
  // allocation so that one cudaIpc handle covers it
  DevBuf<float> xbuf;
  int64_t xstride = 0;
  float* peer_x[kMaxPeers] = {};  // mapped with cudaIpcOpenMemHandle (peer_x[rank] is xbuf)
  bool p2p = false;
  // rollout observations shared across ranks as bf16 tables (each rank converts its own slab; peers map it)
  __nv_bfloat16* peer_table[kMaxPeers] = {};  // mapped like peer_x (peer_table[rank] is bf.obs_table)
  int64_t shared_rows = 0;   // rows of every rank's table; 0 = tables not shared
  bool shared_filled = false;
  // b200ppo_table_replicate: the peers' tables copied once per rollout into local memory, so that the per-epoch gathers
  // read HBM and leave NVLink to the gradient exchange
  DevBuf<__nv_bfloat16> replica;
  bool replicated = false;
  bool perm_rank_slices = false;  // b200ppo_set_perm_layout: `perms` holds only this rank's slots
  bool in_epoch = false;          // inside b200ppo_train's minibatch loop: the minibatch operands predate the previous kernel
  unsigned p2p_seq = 0;
  cudaStream_t gather_stream = nullptr;
  cudaEvent_t ev_ready[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr}, ev_start = nullptr;
  // device staging of the host entry point
  // two sets: b200ppo_update_host_begin(slot) uploads rollout k + 1 on the copy stream while _end(other slot) trains on rollout k
  struct HostStage {
    DevBuf<float> obs, act, logp, rew, val, nval, adv, tgt;  // sized for `rows` rows and grown together, with term
    DevBuf<uint8_t> term;
    int64_t rows = 0;
    DevBuf<int64_t> perms;
    DevBuf<float> losses;
    int64_t n_envs = 0, n_steps = 0;
    int32_t epochs = 0;
    cudaEvent_t ev_small = nullptr, ev_all = nullptr;  // scalars of the advantage pass uploaded / everything uploaded
  } host[2];
  cudaStream_t copy_stream = nullptr;
  // bf16 operands of the tensor-core path (precision == B200PPO_PREC_BF16); hidden layers only
  struct {
    DevBuf<__nv_bfloat16> H[2][kMaxLayers];   // hidden activations [max_batch, pitchH], ones in column dims[l]
    DevBuf<__nv_bfloat16> dZ[2][kMaxLayers];  // dL/dz of every layer [max_batch, pitchZ]
    DevBuf<__nv_bfloat16> W[2][kMaxLayers];   // W_l   [dims[l], pitchW]
    int pitchH[2][kMaxLayers] = {}, pitchZ[2][kMaxLayers] = {}, pitchW[2][kMaxLayers] = {};
    DevBuf<__nv_bfloat16> X;          // [max_batch, pitchX] staged observations (grads-only entry point)
    DevBuf<__nv_bfloat16> sh_obs;     // [2 sh_cap, pitchX] shuffled observations of an epoch (one of the sh_* group)
    DevBuf<__nv_bfloat16> obs_table;  // [rows, pitchX] the whole rollout's observations as bf16 rows (+ ones-column)
    int pitchX = 0;
    b200ppo::WeightCastGroup casts{};
  } bf;
  void* comm = nullptr;
  int rank = 0, world = 1;
};

namespace b200ppo {

#define PROF(ctx, cls, st, expr)          \
  do {                                    \
    (ctx)->prof.begin(cls, st);           \
    int _pr = (expr);                     \
    (ctx)->prof.end(st);                  \
    if (_pr != B200PPO_OK) return _pr;    \
  } while (0)

int check_batch(const b200ppo_ctx* ctx, int64_t B, const char* who);

// ---- passes.cu -------------------------------------------------------------------------------------------------------
// The arena of three-term operands, emptied: call where a new set of sources starts (a minibatch, an entry point).
// nullptr when the context cannot use it — the callers then stay on the FFMA kernels.
SplitArena* fresh_arena(const b200ppo_ctx* ctx);
// nets: bit 0 actor, bit 1 critic.  acts[n]: hidden activations (dense for `B` rows); outs[n]: [B, out_dim].
// arena (nullable): where the fp32-tolerance tensor-core GEMMs keep their three-term operands; nullptr = FFMA only.
int forward_nets(const b200ppo_ctx* ctx, const float* params, const float* x, int64_t B, int nets, float* const acts[2],
                 float* const outs[2], cudaStream_t st, bool skip_last = false, SplitArena* arena = nullptr);
// dz[n] holds dL/dz of every layer; the last layer's block must be filled on entry.  Weight / bias gradients go
// to gpart as `*split_out` split-K partials laid out like the parameter buffer.  grad_x[n] (nullable): dL/dx.
int backward_nets(b200ppo_ctx* ctx, const float* params, const float* x, int64_t B, int nets, float* const acts[2],
                  float* const dz[2], float* gpart, int* split_out, float* const grad_x[2], cudaStream_t st,
                  bool skip_last_dgrad = false, SplitArena* arena = nullptr);
WeightCastGroup cast_group(const b200ppo_ctx* ctx, const float* params);
int cast_weights(b200ppo_ctx* ctx, const float* params, cudaStream_t st);
bool chain_applicable(const b200ppo_ctx* ctx);

// Outputs of the forward-only instance of the chain kernel (rollout inference); nullptr members are skipped.
struct ChainInfer {
  const float* noise;
  float *mean, *value, *action, *logp;
  int64_t ld_action = 0, ld_value = 1, ld_logp = 1;  // row strides (0: act_dim)
  float* value2 = nullptr;
};
int launch_chain(b200ppo_ctx* ctx, const float* params, const __nv_bfloat16* xb, int64_t B, const float* action,
                 const float* old_logp, const float* adv, const float* tgt, const b200ppo_hparams* hp, int* loss_ctas,
                 cudaStream_t st, bool x_early, const ChainInfer* inf = nullptr);

// forward + losses + backward of one minibatch; gradients left as split-K partials in ctx->gpart.
// obs: fp32 rows (fp32 path) — or obs_b: bf16 rows with the ones-column (tensor-core path).
// *loss_ctas_out > 0: the loss sums were left as that many rows of ctx->loss_partials (fused epilogues) and the kernel
// that consumes the gradients must finish them (LossCombine); 0: losses_dev and the logstd gradient are already final.
int minibatch_fwd_bwd(b200ppo_ctx* ctx, const float* params, const float* obs, const __nv_bfloat16* obs_b, const float* action,
                      const float* old_logp, const float* adv, const float* tgt, int64_t B, const b200ppo_hparams* hp,
                      float* losses_dev, int* split_out, int* loss_ctas_out, cudaStream_t st);
// the per-row loss operands of a B-row minibatch (hp may be null when no loss is computed)
PpoOperands ppo_operands(const b200ppo_ctx* ctx, const float* params, const b200ppo_hparams* hp, int64_t B, const float* action,
                         const float* old_logp, const float* adv, const float* tgt);
LossCombine make_loss_combine(const b200ppo_ctx* ctx, const float* params, int loss_ctas, int64_t B, const b200ppo_hparams* hp,
                              float* losses_out);

// ---- comm.cu ---------------------------------------------------------------------------------------------------------
int nccl_all_reduce(float* buf, int64_t count, void* comm, cudaStream_t st);  // in place, float sum
void nccl_comm_destroy(void* comm);
void close_peer_tables(b200ppo_ctx* ctx);  // unmaps the peers' observation tables (the device must be idle)

}  // namespace b200ppo
