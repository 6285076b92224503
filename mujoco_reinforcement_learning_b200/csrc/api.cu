// C-ABI entry points and host-side orchestration of the actor-critic update (see include/b200ppo.h).
//
// replaces: the Python control flow of PPO.train (src/entities/algorithms/ppo.py:93-154) and the
//           per-call glue of Actor/Critic.forward (src/models/linear/actor.py:25-30, src/models/critic.py:22-25).
#include <dlfcn.h>
#include <stdarg.h>
#include <string.h>

#include <algorithm>
#include <atomic>
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

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

static std::atomic<long long> g_launches{0};
void count_launch() { g_launches.fetch_add(1, std::memory_order_relaxed); }

constexpr int64_t kParamAlign = 32;  // every parameter tensor starts on a 128-byte boundary of the flat buffer
static inline int64_t align_up(int64_t x, int64_t a) { return (x + a - 1) / a * a; }

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

// NCCL is resolved at run time from the library torch already loaded (no link-time dependency).
struct NcclApi {
  struct Id128 { char b[128]; };  // ncclUniqueId, passed by value
  void* handle = nullptr;
  int (*GetUniqueId)(void*) = nullptr;
  int (*CommInitRank)(void**, int, Id128, int) = nullptr;
  int (*AllReduce)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*CommDestroy)(void*) = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
static NcclApi g_nccl;

static int load_nccl() {
  if (g_nccl.AllReduce) return B200PPO_OK;
  void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!h) {
    set_error("NCCL not found: %s", dlerror());
    return B200PPO_ENCCL;
  }
  g_nccl.handle = h;
  *(void**)(&g_nccl.GetUniqueId) = dlsym(h, "ncclGetUniqueId");
  *(void**)(&g_nccl.CommInitRank) = dlsym(h, "ncclCommInitRank");
  *(void**)(&g_nccl.AllReduce) = dlsym(h, "ncclAllReduce");
  *(void**)(&g_nccl.CommDestroy) = dlsym(h, "ncclCommDestroy");
  *(void**)(&g_nccl.GetErrorString) = dlsym(h, "ncclGetErrorString");
  if (!g_nccl.GetUniqueId || !g_nccl.CommInitRank || !g_nccl.AllReduce) {
    set_error("NCCL symbols missing");
    return B200PPO_ENCCL;
  }
  return B200PPO_OK;
}

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

using namespace b200ppo;

struct b200ppo_ctx {
  Profiler prof;
  Net net[2];
  int64_t logstd_off = 0, n_params = 0, n_actor = 0;
  int64_t max_batch = 0;
  int precision = 0;
  int max_split = 1;
  float* ws_act[2] = {nullptr, nullptr};
  float* ws_dz[2] = {nullptr, nullptr};
  float* ws_out[2] = {nullptr, nullptr};
  float* gpart = nullptr;       // [max_split][n_params]
  float* grad_flat = nullptr;   // [n_params + 4]: summed gradient + (actor_loss, critic_loss) for the all-reduce
  float* loss_partials = nullptr;
  int64_t loss_partial_rows = 0;
  unsigned* ticket = nullptr;
  unsigned* done_counter = nullptr;  // fused reduce of the peer exchange: blocks of the optimizer grid that have written their slice (monotone)
  unsigned done_total = 0;           // what that counter reaches after the launches issued so far
  float* scratch = nullptr;     // [8] losses / entropy scratch
  // three-term bf16 operands of the fp32-tolerance tensor-core GEMMs (gemm_split.cuh); allocated at first use
  mutable SplitArena arena;
  int64_t arena_need = 0;
  float* rollout_tmp = nullptr;  // b200ppo_rollout_step, contexts without the one-launch path: value / action / log-prob of a step
  int64_t rollout_tmp_rows = 0;
  float* obs_amax = nullptr;   // max |observation| of the rollout b200ppo_train is working on (a bound for every minibatch's rows)
  bool obs_amax_ok = false;    // valid: inside b200ppo_train's minibatch loop
  int32_t* err_flag = nullptr;
  // shuffled-epoch buffers (train)
  // two sets (rows [0, sh_cap) and [sh_cap, 2 sh_cap)): epoch e+1 is gathered on a side stream while epoch e trains
  float *sh_obs = nullptr, *sh_act = nullptr, *sh_logp = nullptr, *sh_adv = nullptr, *sh_tgt = nullptr;
  int64_t sh_cap = 0;
  // peer-memory gradient exchange (multi-GPU, see adam.cuh PeerSrc): two buffers of xstride floats + a flag array, one
  // allocation so that one cudaIpc handle covers it
  float* xbuf = nullptr;
  int64_t xstride = 0;
  float* peer_x[kMaxPeers] = {};
  bool p2p = false;
  // rollout observations shared across ranks as bf16 tables (each rank converts its own slab; peers map it)
  __nv_bfloat16* peer_table[kMaxPeers] = {};
  int64_t shared_rows = 0;   // rows of every rank's table; 0 = tables not shared
  bool shared_filled = false;
  // b200ppo_table_replicate: the peers' tables copied once per rollout into local memory, so that the per-epoch gathers
  // read HBM and leave NVLink to the gradient exchange
  __nv_bfloat16* replica = nullptr;
  int64_t replica_cap = 0;   // elements
  bool replicated = false;
  bool perm_rank_slices = false;  // b200ppo_set_perm_layout: `perms` holds only this rank's slots
  bool in_epoch = false;          // inside b200ppo_train's minibatch loop: the minibatch operands predate the previous kernel
  unsigned p2p_seq = 0;
  cudaStream_t gather_stream = nullptr;
  cudaEvent_t ev_ready[2] = {nullptr, nullptr}, ev_free[2] = {nullptr, nullptr}, ev_start = nullptr;
  // device staging of the host entry point
  // two sets: b200ppo_update_host_begin(slot) uploads rollout k + 1 on the copy stream while _end(other slot) trains on rollout k
  struct HostStage {
    float *obs = nullptr, *act = nullptr, *logp = nullptr, *rew = nullptr, *val = nullptr, *nval = nullptr;
    float *adv = nullptr, *tgt = nullptr, *losses = nullptr;
    uint8_t* term = nullptr;
    int64_t* perms = nullptr;
    int64_t rows = 0, perm_elems = 0, loss_elems = 0;
    int64_t n_envs = 0, n_steps = 0;
    int32_t epochs = 0;
    cudaEvent_t ev_small = nullptr, ev_all = nullptr;  // scalars of the advantage pass uploaded / everything uploaded
  } host[2];
  cudaStream_t copy_stream = nullptr;
  // bf16 operands of the tensor-core path (precision == B200PPO_PREC_BF16); hidden layers only
  struct {
    __nv_bfloat16* H[2][B200PPO_MAX_LAYERS] = {};   // hidden activations [max_batch, pitchH], ones in column dims[l]
    __nv_bfloat16* dZ[2][B200PPO_MAX_LAYERS] = {};  // dL/dz of every layer [max_batch, pitchZ]
    __nv_bfloat16* W[2][B200PPO_MAX_LAYERS] = {};   // W_l   [dims[l], pitchW]
    int pitchH[2][B200PPO_MAX_LAYERS] = {}, pitchZ[2][B200PPO_MAX_LAYERS] = {}, pitchW[2][B200PPO_MAX_LAYERS] = {};
    __nv_bfloat16* X = nullptr;      // [max_batch, pitchX] staged observations (grads-only entry point)
    __nv_bfloat16* sh_obs = nullptr; // [sh_cap, pitchX] shuffled observations of an epoch
    __nv_bfloat16* obs_table = nullptr;  // [table_cap, pitchX] the whole rollout's observations as bf16 rows (+ ones-column)
    int64_t table_cap = 0;
    int pitchX = 0;
    WeightCastGroup casts{};
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

static int layout_net(Net& n, const b200ppo_mlp_desc* d, int64_t& cursor) {
  B2_CHECK_ARG(d->n_layers >= 1 && d->n_layers <= B200PPO_MAX_LAYERS, "n_layers %d out of range", d->n_layers);
  B2_CHECK_ARG(d->in_dim > 0, "in_dim must be positive");
  B2_CHECK_ARG(d->activation == B200PPO_ACT_TANH || d->activation == B200PPO_ACT_RELU, "unknown activation %d", d->activation);
  n.d = *d;
  n.seg_begin = cursor;
  n.hidden_sum = 0;
  for (int l = 0; l < d->n_layers; ++l) {
    B2_CHECK_ARG(d->dims[l] > 0, "layer %d has non-positive width", l);
    n.w_off[l] = cursor;
    cursor = align_up(cursor + int64_t(d->dims[l]) * n.in_dim(l), kParamAlign);
    n.b_off[l] = cursor;
    cursor = align_up(cursor + d->dims[l], kParamAlign);
    if (l < d->n_layers - 1) n.hidden_sum += d->dims[l];
  }
  n.seg_end = cursor;
  return B200PPO_OK;
}

template <typename T>
static int dev_alloc(T** p, int64_t elems, bool zero = false) {
  *p = nullptr;
  if (elems <= 0) elems = 1;
  cudaError_t e = cudaMalloc(reinterpret_cast<void**>(p), size_t(elems) * sizeof(T));
  if (e != cudaSuccess) {
    set_error("cudaMalloc(%lld bytes) failed: %s", (long long)(elems * sizeof(T)), cudaGetErrorString(e));
    return e == cudaErrorMemoryAllocation ? B200PPO_ENOMEM : B200PPO_ECUDA;
  }
  if (zero) B2_CUDA(cudaMemset(*p, 0, size_t(elems) * sizeof(T)));
  return B200PPO_OK;
}

template <typename T>
static void dev_free(T*& p) {
  if (p) cudaFree(p);
  p = nullptr;
}

__global__ void tanh_scale_bwd_kernel(const float* __restrict__ grad_out, const float* __restrict__ out, float scale,
                                      int64_t n, float* __restrict__ dz) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < n) {
    const float th = out[i] / scale;
    dz[i] = grad_out[i] * scale * (1.f - th * th);
  }
}

__global__ void copy2_kernel(const float* __restrict__ src, float* __restrict__ dst) {
  if (threadIdx.x < 2) dst[threadIdx.x] = src[threadIdx.x];
}

// The arena of three-term operands, emptied: call where a new set of sources starts (a minibatch, an entry point).
// nullptr when the context cannot use it — the callers then stay on the FFMA kernels.
static SplitArena* fresh_arena(const b200ppo_ctx* ctx) {
  if (ctx->arena_need <= 0) return nullptr;
  if (ctx->arena.cap < ctx->arena_need && split_arena_reserve(ctx->arena, ctx->arena_need) != B200PPO_OK) return nullptr;
  split_arena_reset(ctx->arena);
  return &ctx->arena;
}

// ---- forward -----------------------------------------------------------------------------------------
// nets: bit 0 actor, bit 1 critic.  acts[n]: hidden activations (dense for `B` rows); outs[n]: [B, out_dim].
// arena (nullable): where the fp32-tolerance tensor-core GEMMs keep their three-term operands; nullptr = FFMA only.
static int forward_nets(const b200ppo_ctx* ctx, const float* params, const float* x, int64_t B, int nets,
                        float* const acts[2], float* const outs[2], cudaStream_t st, bool skip_last = false,
                        SplitArena* arena = nullptr) {
  int maxL = 0;
  for (int n = 0; n < 2; ++n)
    if (nets & (1 << n)) maxL = std::max(maxL, ctx->net[n].d.n_layers);
  for (int l = 0; l < maxL; ++l) {
    GemmGroup g{};
    int64_t large_tiles = 0;
    GemmProblem probs[2];
    int np = 0;
    for (int n = 0; n < 2; ++n) {
      const Net& N = ctx->net[n];
      if (!(nets & (1 << n)) || l >= N.d.n_layers) continue;
      const bool last = (l == N.d.n_layers - 1);
      if (last && skip_last) continue;
      GemmProblem p{};
      p.A = (l == 0) ? x : acts[n] + N.act_off(l - 1, B);
      p.a_sm = N.in_dim(l); p.a_sk = 1;
      if (l == 0) p.a_bound_dev = ctx->obs_amax_ok ? ctx->obs_amax : nullptr;
      else if (N.d.activation == B200PPO_ACT_TANH) p.a_bound = 1.f;  // |tanh| <= 1
      p.B = params + N.w_off[l];
      p.b_sn = N.in_dim(l); p.b_sk = 1;
      p.bias = params + N.b_off[l];
      p.C = last ? outs[n] : acts[n] + N.act_off(l, B);
      p.ldc = N.d.dims[l];
      p.M = int(B); p.N = N.d.dims[l]; p.K = N.in_dim(l);
      p.out_scale = N.d.out_scale;
      if (last) p.epilogue = N.d.final_tanh ? EPI_BIAS_TANH_SCALE : EPI_BIAS;
      else p.epilogue = N.d.activation == B200PPO_ACT_TANH ? EPI_BIAS_TANH : EPI_BIAS_RELU;
      large_tiles += int64_t((p.M + 127) / 128) * ((p.N + 127) / 128);
      if (p.N < 96) large_tiles = -(1ll << 40);
      probs[np++] = p;
    }
    if (np == 0) continue;
    const bool large = large_tiles >= (2 * num_sms()) / 3;
    for (int i = 0; i < np; ++i) gemm_group_add(g, probs[i], large ? 128 : 64, large ? 128 : 64, 1);
    if (arena != nullptr && gemm_split_applicable(g)) B2_TRY(launch_gemm_group_split(g, *arena, st));
    else B2_TRY(launch_gemm_group(g, large, st));
  }
  return B200PPO_OK;
}

static int pick_split(const b200ppo_ctx* ctx, int64_t tiles, int64_t K) {
  if (tiles <= 0) return 1;
  int64_t s = (4ll * num_sms() + tiles - 1) / tiles;
  s = std::min<int64_t>(s, std::max<int64_t>(1, K / 64));
  s = std::min<int64_t>(s, std::min(ctx->max_split, 32));
  return int(std::max<int64_t>(1, s));
}

// ---- backward ----------------------------------------------------------------------------------------
// dz[n] holds dL/dz of every layer; the last layer's block must be filled on entry.  Weight / bias gradients go
// to gpart as `*split_out` split-K partials laid out like the parameter buffer.  grad_x[n] (nullable): dL/dx.
static int backward_nets(b200ppo_ctx* ctx, const float* params, const float* x, int64_t B, int nets,
                         float* const acts[2], float* const dz[2], float* gpart, int* split_out,
                         float* const grad_x[2], cudaStream_t st, bool skip_last_dgrad = false, SplitArena* arena = nullptr) {
  int maxL = 0;
  for (int n = 0; n < 2; ++n)
    if (nets & (1 << n)) maxL = std::max(maxL, ctx->net[n].d.n_layers);
  // dgrad chain, grouped by distance from the output (s = 0: through the output layer — done by the fused heads
  // kernel when skip_last_dgrad)
  for (int s = skip_last_dgrad ? 1 : 0; s < maxL; ++s) {
    GemmProblem probs[2];
    int np = 0;
    int64_t large_tiles = 0;
    for (int n = 0; n < 2; ++n) {
      const Net& N = ctx->net[n];
      if (!(nets & (1 << n))) continue;
      const int l = N.d.n_layers - 1 - s;
      if (l < 0) continue;
      if (l == 0 && (grad_x == nullptr || grad_x[n] == nullptr)) continue;
      GemmProblem p{};
      p.A = dz[n] + N.dz_off(l, B);
      p.a_sm = N.d.dims[l]; p.a_sk = 1;
      p.B = params + N.w_off[l];
      p.b_sn = 1; p.b_sk = N.in_dim(l);
      p.M = int(B); p.N = N.in_dim(l); p.K = N.d.dims[l];
      p.ldc = N.in_dim(l);
      if (l == 0) {
        p.C = grad_x[n];
        p.epilogue = EPI_STORE;
      } else {
        p.C = dz[n] + N.dz_off(l - 1, B);
        p.aux = acts[n] + N.act_off(l - 1, B);
        p.ld_aux = N.d.dims[l - 1];
        p.epilogue = N.d.activation == B200PPO_ACT_TANH ? EPI_DTANH : EPI_DRELU;
      }
      large_tiles += int64_t((p.M + 127) / 128) * ((p.N + 127) / 128);
      if (p.N < 96) large_tiles = -(1ll << 40);
      probs[np++] = p;
    }
    if (np == 0) continue;
    const bool large = large_tiles >= (2 * num_sms()) / 3;
    GemmGroup g{};
    for (int i = 0; i < np; ++i) gemm_group_add(g, probs[i], large ? 128 : 64, large ? 128 : 64, 1);
    if (arena != nullptr && gemm_split_applicable(g)) PROF(ctx, B200PPO_PROF_GEMM_DGRAD, st, launch_gemm_group_split(g, *arena, st));
    else PROF(ctx, B200PPO_PROF_GEMM_DGRAD, st, launch_gemm_group(g, large, st));
  }
  // every weight / bias gradient in one grouped split-K launch
  if (gpart != nullptr) {
    GemmProblem probs[kMaxGemmProblems];
    int np = 0;
    int64_t tiles = 0;
    for (int n = 0; n < 2; ++n) {
      const Net& N = ctx->net[n];
      if (!(nets & (1 << n))) continue;
      for (int l = 0; l < N.d.n_layers; ++l) {
        GemmProblem p{};
        p.A = dz[n] + N.dz_off(l, B);
        p.a_sm = 1; p.a_sk = N.d.dims[l];
        p.B = (l == 0) ? x : acts[n] + N.act_off(l - 1, B);
        p.b_sn = 1; p.b_sk = N.in_dim(l);
        if (l == 0) p.b_bound_dev = ctx->obs_amax_ok ? ctx->obs_amax : nullptr;
        else if (N.d.activation == B200PPO_ACT_TANH) p.b_bound = 1.f;
        p.M = N.d.dims[l]; p.N = N.in_dim(l); p.K = int(B);
        p.C = gpart + N.w_off[l];
        p.ldc = N.in_dim(l);
        p.bias_grad = gpart + N.b_off[l];
        p.c_split_stride = ctx->n_params;
        p.epilogue = EPI_STORE;
        tiles += int64_t((p.M + 63) / 64) * ((p.N + 63) / 64);
        probs[np++] = p;
      }
    }
    int split = pick_split(ctx, tiles, B);
    GemmGroup g{};
    for (int i = 0; i < np; ++i) gemm_group_add(g, probs[i], 64, 64, split);
    if (arena != nullptr && gemm_split_applicable(g)) {
      // The tensor core truncates its fp32 accumulator after every K = 16 step (gemm_split.cu), so the number of samples one
      // accumulator sums is kept to kSplitChain: more split-K partials, which the optimizer kernel adds in fp32 (round to nearest).
      split = int(std::min<int64_t>(ctx->max_split, std::max<int64_t>(split, (B + kSplitChain - 1) / kSplitChain)));
      g = GemmGroup{};
      for (int i = 0; i < np; ++i) gemm_group_add(g, probs[i], 64, 64, split);
      PROF(ctx, B200PPO_PROF_GEMM_WGRAD, st, launch_gemm_group_split(g, *arena, st));
    } else {
      PROF(ctx, B200PPO_PROF_GEMM_WGRAD, st, launch_gemm_group(g, false, st));
    }
    if (split_out) *split_out = split;
  }
  return B200PPO_OK;
}


static inline int pad8(int x) { return (x + 7) / 8 * 8; }
static inline int pad16(int x) { return (x + 15) / 16 * 16; }  // rows that start on 32-byte sectors (256-bit loads / stores)

// bf16 operands of the tensor-core path.  Every Linear of both nets runs on tcgen05 (the 17- and 1-wide output
// layers too: a mostly-empty 128x64 tile costs less than a latency-bound SIMT pass).
static int alloc_bf16_workspaces(b200ppo_ctx* c) {
  B2_TRY(tc_init());
  auto& bf = c->bf;
  const int64_t Bm = c->max_batch;
  bf.pitchX = pad8(c->net[0].d.in_dim + 1);
  B2_TRY(dev_alloc(&bf.X, Bm * bf.pitchX));
  B2_TRY(launch_init_ones_column(bf.X, Bm, bf.pitchX, c->net[0].d.in_dim, nullptr));
  bf.casts.count = 0;
  bf.casts.max_elems = 0;
  for (int n = 0; n < 2; ++n) {
    const Net& N = c->net[n];
    B2_CHECK_ARG(N.d.n_layers >= 2, "the bf16 tensor-core path needs at least one hidden layer per network");
    for (int l = 0; l < N.d.n_layers; ++l) {
      const bool last = l == N.d.n_layers - 1;
      bf.pitchZ[n][l] = pad8(N.d.dims[l]);
      bf.pitchW[n][l] = pad8(N.in_dim(l));
      if (!last) {  // hidden activation with the ones-column the wgrad reads the bias gradient from
        bf.pitchH[n][l] = pad16(N.d.dims[l] + 1);
        B2_TRY(dev_alloc(&bf.H[n][l], Bm * bf.pitchH[n][l]));
        B2_TRY(launch_init_ones_column(bf.H[n][l], Bm, bf.pitchH[n][l], N.d.dims[l], nullptr));
      }
      B2_TRY(dev_alloc(&bf.dZ[n][l], Bm * bf.pitchZ[n][l], true));
      B2_TRY(dev_alloc(&bf.W[n][l], int64_t(N.d.dims[l]) * bf.pitchW[n][l], true));
      WeightCast& w = bf.casts.w[bf.casts.count++];
      w.src = nullptr;  // the parameter base is a per-call argument: filled in by cast_weights()
      w.dst = bf.W[n][l];
      w.out = N.d.dims[l]; w.in = N.in_dim(l); w.pitch = bf.pitchW[n][l];
      bf.casts.max_elems = std::max(bf.casts.max_elems, w.out * w.in);
    }
  }
  B2_CUDA(cudaDeviceSynchronize());
  return B200PPO_OK;
}

static WeightCastGroup cast_group(const b200ppo_ctx* ctx, const float* params) {
  WeightCastGroup g = ctx->bf.casts;
  int k = 0;
  for (int n = 0; n < 2; ++n)
    for (int l = 0; l < ctx->net[n].d.n_layers; ++l) g.w[k++].src = params + ctx->net[n].w_off[l];
  return g;
}

static int cast_weights(b200ppo_ctx* ctx, const float* params, cudaStream_t st) {
  return launch_cast_weights(cast_group(ctx, params), st);
}

// forward of both nets on the tensor cores; hidden activations in bf16 (+ ones column), outputs in fp32.
// The minibatch leaves the fused PPO epilogues of the output layers consume (nullptr = plain forward).
struct PpoFuse {
  const float *action, *old_logp, *advantage, *target;
  const b200ppo_hparams* hp;
  int loss_ctas;  // out: CTAs that wrote a row of loss partials
};

static int forward_nets_bf16(b200ppo_ctx* ctx, const float* params, const __nv_bfloat16* xb, int64_t B,
                             float* const outs[2], cudaStream_t st, PpoFuse* fuse = nullptr) {
  auto& bf = ctx->bf;
  int maxL = 0;
  for (int n = 0; n < 2; ++n) maxL = std::max(maxL, ctx->net[n].d.n_layers);
  for (int l = 0; l < maxL; ++l) {
    TcGroup g{};
    int maxN = 0, nets_here = 0;
    for (int n = 0; n < 2; ++n)
      if (l < ctx->net[n].d.n_layers) { maxN = std::max(maxN, ctx->net[n].d.dims[l]); ++nets_here; }
    int maxK = 0;
    for (int n = 0; n < 2; ++n)
      if (l < ctx->net[n].d.n_layers) maxK = std::max(maxK, ctx->net[n].in_dim(l));
    const bool ws = tc_ws_applicable(int64_t((B + 127) / 128) * nets_here, maxN, maxK);
    const int bn = ws ? tc_ws_bn(maxN, maxK) : tc_pick_bn(int64_t((B + 127) / 128) * nets_here, maxN);
    for (int n = 0; n < 2; ++n) {
      const Net& N = ctx->net[n];
      if (l >= N.d.n_layers) continue;
      const bool last = l == N.d.n_layers - 1;
      TcProblem p{};
      p.M = int(B); p.N = N.d.dims[l]; p.K = N.in_dim(l);
      p.epilogue = TC_EPI_FWD;
      p.bias = params + N.b_off[l];
      p.bias_col = -1;
      if (last && fuse != nullptr) {
        p.epilogue = n == 0 ? TC_EPI_PPO_ACTOR : TC_EPI_PPO_CRITIC;
        p.out_scale = N.d.out_scale;
        p.ppo.logstd = params + ctx->logstd_off;
        p.ppo.action = fuse->action; p.ppo.old_logp = fuse->old_logp; p.ppo.advantage = fuse->advantage;
        p.ppo.target = fuse->target;
        p.ppo.dz_out = bf.dZ[n][l]; p.ppo.dz_pitch = bf.pitchZ[n][l];
        p.ppo.partials = ctx->loss_partials;
        p.ppo.act_dim = ctx->net[0].out_dim();
        p.ppo.final_tanh = N.d.final_tanh;
        p.ppo.clip_eps = float(fuse->hp->clip_epsilon);
        p.ppo.inv_global_batch = 1.f / float(B * ctx->world);
      } else if (last) {
        p.act = N.d.final_tanh ? TC_ACT_TANH_SCALE : TC_ACT_NONE;
        p.out_scale = N.d.out_scale;
        p.out_f32 = outs[n]; p.ld_f32 = N.d.dims[l];
      } else {
        p.act = N.d.activation;
        p.out_bf16 = bf.H[n][l]; p.ld_bf16 = bf.pitchH[n][l];
      }
      TcOperand A{l == 0 ? xb : bf.H[n][l - 1], l == 0 ? bf.pitchX : bf.pitchH[n][l - 1], 0};
      TcOperand Bop{bf.W[n][l], bf.pitchW[n][l], 0};
      B2_TRY(tc_group_add(g, p, A, Bop, bn, 1));
    }
    int grid = 0;
    // layer 0 may directly follow the optimizer (its weights are then one kernel old): only deeper layers preload W
    PROF(ctx, B200PPO_PROF_GEMM_FWD, st, ws ? launch_tc_ws(g, st, &grid, l > 0) : launch_tc_group(g, bn, st, &grid));
    if (fuse != nullptr && l == maxL - 1) fuse->loss_ctas = grid;
  }
  return B200PPO_OK;
}

// backward of both nets on the tensor cores.  bf.dZ[n][L-1] (dL/dz of the output layers, bf16) is filled on entry.
static int backward_nets_bf16(b200ppo_ctx* ctx, const __nv_bfloat16* xb, int64_t B, float* gpart, int* split_out,
                              cudaStream_t st, bool skip_dgrad = false) {
  auto& bf = ctx->bf;
  int maxL = 0;
  for (int n = 0; n < 2; ++n) maxL = std::max(maxL, ctx->net[n].d.n_layers);
  // dgrads, deepest first: dZ_{l-1} = (dZ_l W_l) * act'(H_{l-1}),  B operand = the bf16 copy of W_l read MN-major
  // (skip_dgrad: the fused chain kernel already left every dZ_l in place)
  for (int s = 0; s < (skip_dgrad ? 0 : maxL); ++s) {
    TcGroup g{};
    int maxN = 0, nets_here = 0;
    for (int n = 0; n < 2; ++n) {
      const int l = ctx->net[n].d.n_layers - 1 - s;
      if (l >= 1) { maxN = std::max(maxN, ctx->net[n].in_dim(l)); ++nets_here; }
    }
    if (nets_here == 0) break;
    int maxK = 0;
    for (int n = 0; n < 2; ++n) {
      const int l = ctx->net[n].d.n_layers - 1 - s;
      if (l >= 1) maxK = std::max(maxK, ctx->net[n].d.dims[l]);
    }
    const bool ws = tc_ws_applicable(int64_t((B + 127) / 128) * nets_here, maxN, maxK);
    const int bn = ws ? tc_ws_bn(maxN, maxK) : tc_pick_bn(int64_t((B + 127) / 128) * nets_here, maxN);
    for (int n = 0; n < 2; ++n) {
      const Net& N = ctx->net[n];
      const int l = N.d.n_layers - 1 - s;
      if (l < 1) continue;
      TcProblem p{};
      p.M = int(B); p.N = N.in_dim(l); p.K = N.d.dims[l];
      p.epilogue = TC_EPI_DGRAD; p.act = N.d.activation;
      p.aux = bf.H[n][l - 1]; p.ld_aux = bf.pitchH[n][l - 1];
      p.out_bf16 = bf.dZ[n][l - 1]; p.ld_bf16 = bf.pitchZ[n][l - 1];
      p.bias_col = -1;
      TcOperand A{bf.dZ[n][l], bf.pitchZ[n][l], 0};
      TcOperand Bop{bf.W[n][l], bf.pitchW[n][l], 1};  // W_l is [out = K][in = N]: an MN-major operand, no transposed copy
      B2_TRY(tc_group_add(g, p, A, Bop, bn, 1));
    }
    PROF(ctx, B200PPO_PROF_GEMM_DGRAD, st, ws ? launch_tc_ws(g, st, nullptr, true) : launch_tc_group(g, bn, st));
  }
  // every weight / bias gradient: dW_l = dZ_l^T [H_{l-1} | 1], both operands MN-major, split-K over the batch.
  // N tile: the width that wastes the least padded MMA work over all problems (N = in+1 is 257 / 377 for 256 / 376
  // inputs: 192-wide tiles cover both in two tiles where 128-wide ones need three); split-K: as many splits as fill
  // ONE wave of resident CTAs — one CTA more than a wave would double the kernel's duration.
  const int n_problems = ctx->net[0].d.n_layers + ctx->net[1].d.n_layers;
  if (B >= 2048 && n_problems <= kMaxTcProblems) {
    // CTA pairs: 256 x 256 output blocks, bias gradient from a ones-tile MMA (tc_wgrad.cu)
    TcGroup g{};
    for (int n = 0; n < 2; ++n) {
      const Net& N = ctx->net[n];
      for (int l = 0; l < N.d.n_layers; ++l) {
        TcProblem p{};
        p.M = N.d.dims[l]; p.N = N.in_dim(l); p.K = int(B);
        p.epilogue = TC_EPI_STORE;
        p.out_f32 = gpart + N.w_off[l]; p.ld_f32 = N.in_dim(l); p.split_stride = ctx->n_params;
        p.bias_grad = gpart + N.b_off[l]; p.bias_col = -1;
        TcOperand A{bf.dZ[n][l], bf.pitchZ[n][l], 1};
        TcOperand Bop{l == 0 ? xb : bf.H[n][l - 1], l == 0 ? bf.pitchX : bf.pitchH[n][l - 1], 1};
        B2_TRY(tc_group_add(g, p, A, Bop, 128, 1));
      }
    }
    int split = 1;
    PROF(ctx, B200PPO_PROF_GEMM_WGRAD, st, launch_tc_wgrad2(g, ctx->max_split, st, &split));
    if (split_out) *split_out = split;
    return B200PPO_OK;
  }
  int bn = 64;
  {
    int maxN = 0;
    for (int n = 0; n < 2; ++n)
      for (int l = 0; l < ctx->net[n].d.n_layers; ++l) maxN = std::max(maxN, ctx->net[n].in_dim(l) + 1);
    if (maxN > 64) {
      int64_t best = -1;
      for (int cand : {128, 192, 256}) {
        int64_t work = 0;
        for (int n = 0; n < 2; ++n)
          for (int l = 0; l < ctx->net[n].d.n_layers; ++l)
            work += int64_t((ctx->net[n].d.dims[l] + 127) / 128) * ((ctx->net[n].in_dim(l) + 1 + cand - 1) / cand) * cand;
        if (best < 0 || work < best) { best = work; bn = cand; }
      }
    }
  }
  int64_t tiles = 0;
  for (int n = 0; n < 2; ++n)
    for (int l = 0; l < ctx->net[n].d.n_layers; ++l)
      tiles += int64_t((ctx->net[n].d.dims[l] + 127) / 128) * ((ctx->net[n].in_dim(l) + 1 + bn - 1) / bn);
  const int64_t slots = int64_t(num_sms()) * tc_ctas_per_sm(bn);
  int split = int(std::min<int64_t>(std::max<int64_t>(1, slots / std::max<int64_t>(tiles, 1)), ctx->max_split));
  split = int(std::min<int64_t>(split, (B + 63) / 64));
  if (split < 1) split = 1;
  TcGroup g{};
  for (int n = 0; n < 2; ++n) {
    const Net& N = ctx->net[n];
    for (int l = 0; l < N.d.n_layers; ++l) {
      TcProblem p{};
      p.M = N.d.dims[l]; p.N = N.in_dim(l) + 1; p.K = int(B);
      p.epilogue = TC_EPI_STORE;
      p.out_f32 = gpart + N.w_off[l]; p.ld_f32 = N.in_dim(l); p.split_stride = ctx->n_params;
      p.bias_grad = gpart + N.b_off[l]; p.bias_col = N.in_dim(l);
      TcOperand A{bf.dZ[n][l], bf.pitchZ[n][l], 1};
      TcOperand Bop{l == 0 ? xb : bf.H[n][l - 1], l == 0 ? bf.pitchX : bf.pitchH[n][l - 1], 1};
      if (g.count == kMaxTcProblems) {
        PROF(ctx, B200PPO_PROF_GEMM_WGRAD, st, launch_tc_group(g, bn, st));
        g = TcGroup{};
      }
      B2_TRY(tc_group_add(g, p, A, Bop, bn, split));
    }
  }
  PROF(ctx, B200PPO_PROF_GEMM_WGRAD, st, launch_tc_group(g, bn, st));
  if (split_out) *split_out = split;
  return B200PPO_OK;
}

static int check_batch(const b200ppo_ctx* ctx, int64_t B, const char* who) {
  if (ctx == nullptr) {
    set_error("%s: null context", who);
    return B200PPO_EINVAL;
  }
  if (B < 0 || B > ctx->max_batch) {
    set_error("%s: batch %lld exceeds the context's max_batch %lld", who, (long long)B, (long long)ctx->max_batch);
    return B200PPO_ESTATE;
  }
  return B200PPO_OK;
}

// The fused chain kernel (tc_chain.cu) takes the minibatch when both nets are in -> 256 -> 256 -> out with the same
// activation (the Humanoid / Ant shapes of BASELINE.json); other shapes keep the per-layer launches.
static bool chain_applicable(const b200ppo_ctx* ctx) {
  static const char* mode = getenv("B200PPO_CHAIN");  // profiling switch: "0" keeps the per-layer launches
  if (mode != nullptr && mode[0] == '0') return false;
  const Net& a = ctx->net[0];
  const Net& c = ctx->net[1];
  if (a.d.n_layers != 3 || c.d.n_layers != 3 || a.d.activation != c.d.activation || c.d.final_tanh) return false;
  if (!tc_chain_shape_ok(a.d.in_dim, a.d.dims[0], a.d.dims[1], a.out_dim())) return false;
  if (!tc_chain_shape_ok(c.d.in_dim, c.d.dims[0], c.d.dims[1], c.out_dim())) return false;
  const auto& bf = ctx->bf;
  for (int n = 0; n < 2; ++n) {
    for (int l = 0; l < 2; ++l)
      if (bf.pitchH[n][l] % 16 != 0 || bf.pitchZ[n][l] % 16 != 0) return false;
    if (bf.pitchZ[n][2] % 8 != 0 || bf.pitchZ[n][2] > 32) return false;
  }
  return int64_t(num_sms()) + 8 <= ctx->loss_partial_rows;
}

// Outputs of the forward-only instance (rollout inference); nullptr members are skipped.
struct ChainInfer {
  const float* noise;
  float *mean, *value, *action, *logp;
  int64_t ld_action = 0, ld_value = 1, ld_logp = 1;  // row strides (0: act_dim)
  float* value2 = nullptr;
};

static int launch_chain(b200ppo_ctx* ctx, const float* params, const __nv_bfloat16* xb, int64_t B, const float* action,
                        const float* old_logp, const float* adv, const float* tgt, const b200ppo_hparams* hp, int* loss_ctas,
                        cudaStream_t st, bool x_early, const ChainInfer* inf = nullptr) {
  auto& bf = ctx->bf;
  ChainArgs a{};
  const int D = ctx->net[0].d.in_dim;
  B2_TRY(tc_make_map(&a.x, xb, D, B, bf.pitchX, TC_CHAIN_BK, 128));
  for (int n = 0; n < 2; ++n) {
    const Net& N = ctx->net[n];
    ChainNet& c = a.net[n];
    const int out = N.out_dim();
    B2_TRY(tc_make_map(&c.w1, bf.W[n][0], D, kChainHidden, bf.pitchW[n][0], TC_CHAIN_BK, 128));
    B2_TRY(tc_make_map(&c.w2k, bf.W[n][1], kChainHidden, kChainHidden, bf.pitchW[n][1], TC_CHAIN_BK, 128));
    B2_TRY(tc_make_map(&c.w2m, bf.W[n][1], kChainHidden, kChainHidden, bf.pitchW[n][1], 64, TC_CHAIN_BK));
    B2_TRY(tc_make_map(&c.w3k, bf.W[n][2], kChainHidden, out, bf.pitchW[n][2], TC_CHAIN_BK, n ? 8 : 16));
    B2_TRY(tc_make_map(&c.w3m, bf.W[n][2], kChainHidden, out, bf.pitchW[n][2], 64, n ? 16 : 32));
    B2_TRY(tc_make_map(&c.sH1, bf.H[n][0], kChainHidden, B, bf.pitchH[n][0], 64, 32));
    B2_TRY(tc_make_map(&c.sH2, bf.H[n][1], kChainHidden, B, bf.pitchH[n][1], 64, 32));
    B2_TRY(tc_make_map(&c.sZ1, bf.dZ[n][0], kChainHidden, B, bf.pitchZ[n][0], 64, 32));
    B2_TRY(tc_make_map(&c.sZ2, bf.dZ[n][1], kChainHidden, B, bf.pitchZ[n][1], 64, 32));
    c.b1 = params + N.b_off[0]; c.b2 = params + N.b_off[1]; c.b3 = params + N.b_off[2];
    c.H1 = bf.H[n][0]; c.H2 = bf.H[n][1]; c.dZ1 = bf.dZ[n][0]; c.dZ2 = bf.dZ[n][1]; c.dZ3 = bf.dZ[n][2];
    c.pH1 = bf.pitchH[n][0]; c.pH2 = bf.pitchH[n][1]; c.pZ1 = bf.pitchZ[n][0]; c.pZ2 = bf.pitchZ[n][1]; c.pZ3 = bf.pitchZ[n][2];
  }
  a.ppo.logstd = params + ctx->logstd_off;
  a.ppo.action = action; a.ppo.old_logp = old_logp; a.ppo.advantage = adv; a.ppo.target = tgt;
  a.ppo.partials = ctx->loss_partials;
  a.ppo.act_dim = ctx->net[0].out_dim();
  a.ppo.final_tanh = ctx->net[0].d.final_tanh;
  a.ppo.clip_eps = hp != nullptr ? float(hp->clip_epsilon) : 0.f;
  a.ppo.inv_global_batch = 1.f / float(B * ctx->world);
  if (inf != nullptr) {
    a.inf_noise = inf->noise; a.inf_mean = inf->mean; a.inf_value = inf->value; a.inf_action = inf->action; a.inf_logp = inf->logp;
    a.inf_ld_action = inf->ld_action > 0 ? inf->ld_action : ctx->net[0].out_dim();
    a.inf_ld_value = inf->ld_value; a.inf_ld_logp = inf->ld_logp; a.inf_value2 = inf->value2;
  }
  a.out_scale = ctx->net[0].d.out_scale;
  a.M = int(B);
  a.KB1 = (D + TC_CHAIN_BK - 1) / TC_CHAIN_BK;
  a.act = ctx->net[0].d.activation;
  a.tiles2 = int((B + 255) / 256);
  a.x_early = x_early ? 1 : 0;
  a.trace = inf != nullptr ? nullptr : g_chain_trace;
  return launch_tc_chain(a, st, loss_ctas, inf != nullptr);
}

// forward + losses + backward of one minibatch; gradients left as split-K partials in ctx->gpart.
static void fill_loss_args(const b200ppo_ctx* ctx, LossArgs& la, const float* params, const float* mean, const float* value,
                           const float* action, const float* old_logp, const float* adv, const float* tgt, int64_t B,
                           const b200ppo_hparams* hp) {
  const Net& Na = ctx->net[0];
  la.mean = mean; la.logstd = params + ctx->logstd_off; la.action = action; la.old_logp = old_logp;
  la.advantage = adv; la.value = value; la.target = tgt; la.batch = B; la.act_dim = Na.out_dim();
  la.final_tanh = Na.d.final_tanh; la.out_scale = Na.d.out_scale;
  la.clip_eps = float(hp->clip_epsilon); la.ent_coef = float(hp->entropy_eps);
  la.inv_global_batch = 1.f / float(B * ctx->world);
  la.rank_share = 1.f / float(ctx->world);
}

// obs: fp32 rows (fp32 path) — or obs_b: bf16 rows with the ones-column (tensor-core path).
// *loss_ctas_out > 0: the loss sums were left as that many rows of ctx->loss_partials (fused epilogues) and the kernel
// that consumes the gradients must finish them (LossCombine); 0: losses_dev and the logstd gradient are already final.
static int minibatch_fwd_bwd(b200ppo_ctx* ctx, const float* params, const float* obs, const __nv_bfloat16* obs_b,
                             const float* action, const float* old_logp, const float* adv, const float* tgt, int64_t B,
                             const b200ppo_hparams* hp, float* losses_dev, int* split_out, int* loss_ctas_out,
                             cudaStream_t st) {
  *loss_ctas_out = 0;
  float* acts[2] = {ctx->ws_act[0], ctx->ws_act[1]};
  float* outs[2] = {ctx->ws_out[0], ctx->ws_out[1]};
  float* dz[2] = {ctx->ws_dz[0], ctx->ws_dz[1]};
  const Net& Na = ctx->net[0];
  const Net& Nc = ctx->net[1];
  const int La = Na.d.n_layers, Lc = Nc.d.n_layers;
  if (ctx->precision == B200PPO_PREC_BF16) {
    // tcgen05 everywhere: forward (L launches; PPO loss fused into the output layers' epilogue), dgrads (L-1), wgrads (1)
    if (chain_applicable(ctx)) {  // one launch: forward, losses, dgrads (tc_chain.cu); then the weight gradients
      int grid = 0;
      PROF(ctx, B200PPO_PROF_GEMM_FWD, st, launch_chain(ctx, params, obs_b, B, action, old_logp, adv, tgt, hp, &grid, st, ctx->in_epoch));
      *loss_ctas_out = grid;
      return backward_nets_bf16(ctx, obs_b, B, ctx->gpart, split_out, st, true);
    }
    const bool same_depth = La == Lc;  // both output layers in the same launch
    if (same_depth && tc_ppo_fits(Na.out_dim()) && Na.out_dim() <= 32 &&
        int64_t(2 * ((B + 127) / 128) + 8) <= ctx->loss_partial_rows) {
      PpoFuse fuse{action, old_logp, adv, tgt, hp, 0};
      B2_TRY(forward_nets_bf16(ctx, params, obs_b, B, outs, st, &fuse));
      *loss_ctas_out = fuse.loss_ctas;
      return backward_nets_bf16(ctx, obs_b, B, ctx->gpart, split_out, st);
    }
    B2_TRY(forward_nets_bf16(ctx, params, obs_b, B, outs, st));
    LossArgs la{};
    fill_loss_args(ctx, la, params, outs[0], outs[1], action, old_logp, adv, tgt, B, hp);
    la.dz_actor_bf16 = ctx->bf.dZ[0][La - 1]; la.dz_actor_pitch = ctx->bf.pitchZ[0][La - 1];
    la.dv_bf16 = ctx->bf.dZ[1][Lc - 1]; la.dv_pitch = ctx->bf.pitchZ[1][Lc - 1];
    la.partials = ctx->loss_partials; la.ticket = ctx->ticket;
    la.losses = losses_dev; la.logstd_grad = ctx->gpart + ctx->logstd_off;
    PROF(ctx, B200PPO_PROF_LOSS, st, launch_ppo_loss(la, st));
    return backward_nets_bf16(ctx, obs_b, B, ctx->gpart, split_out, st);
  }
  const bool heads = La >= 2 && Lc >= 2 && heads_supported(Na.out_dim(), Na.d.dims[La - 2], Nc.d.dims[Lc - 2]);
  SplitArena* arena = fresh_arena(ctx);
  PROF(ctx, B200PPO_PROF_GEMM_FWD, st, forward_nets(ctx, params, obs, B, 3, acts, outs, st, heads, arena));
  if (heads) {
    HeadsArgs h{};
    h.h_a = acts[0] + Na.act_off(La - 2, B); h.h_c = acts[1] + Nc.act_off(Lc - 2, B);
    h.w3a = params + Na.w_off[La - 1]; h.b3a = params + Na.b_off[La - 1];
    h.w3c = params + Nc.w_off[Lc - 1]; h.b3c = params + Nc.b_off[Lc - 1];
    h.logstd = params + ctx->logstd_off;
    h.action = action; h.old_logp = old_logp; h.advantage = adv; h.target = tgt;
    h.batch = B; h.act_dim = Na.out_dim(); h.hid_a = Na.d.dims[La - 2]; h.hid_c = Nc.d.dims[Lc - 2];
    h.act = Na.d.activation; h.act_c = Nc.d.activation;
    h.final_tanh = Na.d.final_tanh; h.out_scale = Na.d.out_scale;
    h.clip_eps = float(hp->clip_epsilon); h.ent_coef = float(hp->entropy_eps);
    h.inv_global_batch = 1.f / float(B * ctx->world); h.rank_share = 1.f / float(ctx->world);
    h.dz3_f32 = dz[0] + Na.dz_off(La - 1, B); h.dv_f32 = dz[1] + Nc.dz_off(Lc - 1, B);
    h.dz_a_f32 = dz[0] + Na.dz_off(La - 2, B); h.dz_c_f32 = dz[1] + Nc.dz_off(Lc - 2, B);
    h.partials = ctx->loss_partials; h.ticket = ctx->ticket;
    h.losses = losses_dev; h.logstd_grad = ctx->gpart + ctx->logstd_off;
    PROF(ctx, B200PPO_PROF_LOSS, st, launch_heads(h, st));
  } else {
    LossArgs la{};
    fill_loss_args(ctx, la, params, outs[0], outs[1], action, old_logp, adv, tgt, B, hp);
    la.dz_actor = dz[0] + Na.dz_off(La - 1, B);
    la.dv = dz[1] + Nc.dz_off(Lc - 1, B);
    la.partials = ctx->loss_partials; la.ticket = ctx->ticket;
    la.losses = losses_dev; la.logstd_grad = ctx->gpart + ctx->logstd_off;
    PROF(ctx, B200PPO_PROF_LOSS, st, launch_ppo_loss(la, st));
  }
  return backward_nets(ctx, params, obs, B, 3, acts, dz, ctx->gpart, split_out, nullptr, st, heads, arena);
}

static LossCombine make_loss_combine(const b200ppo_ctx* ctx, const float* params, int loss_ctas, int64_t B,
                                     const b200ppo_hparams* hp, float* losses_out) {
  LossCombine lc{};
  if (loss_ctas <= 0) return lc;
  lc.partials = ctx->loss_partials;
  lc.n_cta = loss_ctas;
  lc.act_dim = ctx->net[0].out_dim();
  lc.logstd_off = ctx->logstd_off;
  lc.logstd = params + ctx->logstd_off;
  lc.inv_global_batch = 1.f / float(B * ctx->world);
  lc.ent_coef = float(hp->entropy_eps);
  lc.rank_share = 1.f / float(ctx->world);
  lc.losses_out = losses_out;
  return lc;
}

static int ensure_shuffle_capacity(b200ppo_ctx* ctx, int64_t rows) {
  if (rows <= ctx->sh_cap) return B200PPO_OK;
  B2_CUDA(cudaDeviceSynchronize());
  dev_free(ctx->sh_obs); dev_free(ctx->sh_act); dev_free(ctx->sh_logp); dev_free(ctx->sh_adv); dev_free(ctx->sh_tgt);
  dev_free(ctx->bf.sh_obs);
  ctx->sh_cap = 0;
  const int D = ctx->net[0].d.in_dim, A = ctx->net[0].out_dim();
  if (ctx->precision == B200PPO_PREC_BF16) B2_TRY(dev_alloc(&ctx->bf.sh_obs, 2 * rows * ctx->bf.pitchX));
  else B2_TRY(dev_alloc(&ctx->sh_obs, 2 * rows * D));
  B2_TRY(dev_alloc(&ctx->sh_act, 2 * rows * A));
  B2_TRY(dev_alloc(&ctx->sh_logp, 2 * rows));
  B2_TRY(dev_alloc(&ctx->sh_adv, 2 * rows));
  B2_TRY(dev_alloc(&ctx->sh_tgt, 2 * rows));
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

int launch_gather_chunked(const int64_t* idx, int64_t count, int64_t n_rows, int64_t chunk, int64_t chunk_stride,
                          int64_t chunk_offset, const float* obs, int obs_dim, const float* act, int act_dim,
                          const float* logp, const float* adv, const float* tgt, float* obs_o, float* act_o,
                          float* logp_o, float* adv_o, float* tgt_o, int32_t* err_flag, cudaStream_t st);
int launch_gather_parts(const int64_t* idx, int64_t count, int64_t n_rows, int64_t chunk, int64_t chunk_stride, int64_t chunk_offset,
                        const float* const* obs_parts, int n_parts, int64_t rows_per_part, int row_floats, const float* act,
                        int act_dim, const float* logp, const float* adv, const float* tgt, float* obs_o, float* act_o,
                        float* logp_o, float* adv_o, float* tgt_o, int32_t* err_flag, cudaStream_t st);
int launch_gather_chunked_bf16(const int64_t* idx, int64_t count, int64_t n_rows, int64_t chunk, int64_t chunk_stride,
                               int64_t chunk_offset, const float* obs, int obs_dim, const float* act, int act_dim,
                               const float* logp, const float* adv, const float* tgt, __nv_bfloat16* obs_o, int pitch,
                               float* act_o, float* logp_o, float* adv_o, float* tgt_o, int32_t* err_flag, cudaStream_t st);

}  // namespace b200ppo

// =========================================================================================================
extern "C" B2_EXPORT int b200ppo_version(void) { return B200PPO_VERSION; }
extern "C" B2_EXPORT const char* b200ppo_last_error(void) { return g_err; }

extern "C" B2_EXPORT int b200ppo_create(const b200ppo_mlp_desc* actor, const b200ppo_mlp_desc* critic, int64_t max_batch,
                              int32_t precision, b200ppo_ctx** out) {
  B2_CHECK_ARG(actor && critic && out, "b200ppo_create: null pointer");
  B2_CHECK_ARG(max_batch > 0 && max_batch < (1ll << 30), "b200ppo_create: bad max_batch");
  B2_CHECK_ARG(precision == B200PPO_PREC_FP32 || precision == B200PPO_PREC_BF16, "b200ppo_create: bad precision");
  B2_CHECK_ARG(actor->in_dim == critic->in_dim, "actor and critic must read the same observation");
  B2_CHECK_ARG(critic->dims[critic->n_layers > 0 ? critic->n_layers - 1 : 0] == 1, "critic output width must be 1");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    set_error("b200ppo_create: no CUDA device (this library has no CPU fallback)");
    return B200PPO_ECUDA;
  }
  b200ppo_ctx* c = new b200ppo_ctx();
  int64_t cursor = 0;
  int r = layout_net(c->net[0], actor, cursor);
  if (r == B200PPO_OK) {
    c->logstd_off = cursor;
    cursor = align_up(cursor + c->net[0].out_dim(), kParamAlign);
    c->net[0].seg_end = cursor;
    c->n_actor = cursor;
    r = layout_net(c->net[1], critic, cursor);
  }
  if (r != B200PPO_OK) { delete c; return r; }
  c->n_params = cursor;
  c->max_batch = max_batch;
  c->precision = precision;
  c->max_split = precision == B200PPO_PREC_FP32 ? 64 : 32;
  const int64_t Bm = max_batch;
  for (int n = 0; n < 2 && r == B200PPO_OK; ++n) {
    const Net& N = c->net[n];
    r = dev_alloc(&c->ws_act[n], Bm * N.hidden_sum);
    if (r == B200PPO_OK) r = dev_alloc(&c->ws_dz[n], Bm * (N.hidden_sum + N.out_dim()));
    if (r == B200PPO_OK) r = dev_alloc(&c->ws_out[n], Bm * N.out_dim());
  }
  if (r == B200PPO_OK) r = dev_alloc(&c->gpart, int64_t(c->max_split) * c->n_params, true);
  if (r == B200PPO_OK) r = dev_alloc(&c->grad_flat, c->n_params + 4, true);
  c->loss_partial_rows = std::max<int64_t>(std::max(loss_grid_size(Bm), 8 * num_sms()), 2 * ((Bm + 127) / 128) + 8);
  if (r == B200PPO_OK) r = dev_alloc(&c->loss_partials, c->loss_partial_rows * (2 + c->net[0].out_dim()), true);
  if (r == B200PPO_OK) r = dev_alloc(&c->ticket, 1, true);
  if (r == B200PPO_OK) r = dev_alloc(&c->done_counter, 1, true);
  if (r == B200PPO_OK) r = dev_alloc(&c->scratch, 8, true);
  if (r == B200PPO_OK) r = dev_alloc(&c->err_flag, 1, true);
  if (r == B200PPO_OK) r = dev_alloc(&c->obs_amax, 1, true);
  if (r == B200PPO_OK && precision == B200PPO_PREC_BF16) r = alloc_bf16_workspaces(c);
  {
    // (the fp32 entry points of a bf16 context — rollout inference, evaluate — use it too)
    // what one minibatch can put into the arena of three-term operands: per net the observations, every hidden activation,
    // every dL/dz block and every weight matrix (reserved at first use: small problems never touch it)
    for (int n = 0; n < 2; ++n) {
      const Net& N = c->net[n];
      c->arena_need += split_arena_elems(Bm, N.d.in_dim) + 8 * (Bm + 4096);  // (+ the per-row / per-column scale vectors)
      for (int l = 0; l < N.d.n_layers; ++l)
        c->arena_need += 3 * split_arena_elems(Bm, N.d.dims[l]) + split_arena_elems(N.d.dims[l], N.in_dim(l)) +  // H_l, dL/dz_l by row and by column
                         split_arena_elems(N.in_dim(l), N.d.dims[l]);
    }
  }
  if (r != B200PPO_OK) { b200ppo_destroy(c); return r; }
  *out = c;
  return B200PPO_OK;
}

extern "C" B2_EXPORT void b200ppo_destroy(b200ppo_ctx* c) {
  if (!c) return;
  cudaDeviceSynchronize();
  for (int n = 0; n < 2; ++n) { dev_free(c->ws_act[n]); dev_free(c->ws_dz[n]); dev_free(c->ws_out[n]); }
  dev_free(c->gpart); dev_free(c->grad_flat); dev_free(c->loss_partials); dev_free(c->ticket); dev_free(c->done_counter); dev_free(c->scratch);
  dev_free(c->err_flag);
  dev_free(c->obs_amax);
  dev_free(c->rollout_tmp);
  split_arena_free(c->arena);
  for (int n = 0; n < 2; ++n)
    for (int l = 0; l < B200PPO_MAX_LAYERS; ++l) { dev_free(c->bf.H[n][l]); dev_free(c->bf.dZ[n][l]); dev_free(c->bf.W[n][l]); }
  dev_free(c->bf.X); dev_free(c->bf.sh_obs); dev_free(c->bf.obs_table); dev_free(c->replica);
  dev_free(c->sh_obs); dev_free(c->sh_act); dev_free(c->sh_logp); dev_free(c->sh_adv); dev_free(c->sh_tgt);
  for (auto& h : c->host) {
    dev_free(h.obs); dev_free(h.act); dev_free(h.logp); dev_free(h.rew); dev_free(h.val);
    dev_free(h.nval); dev_free(h.adv); dev_free(h.tgt); dev_free(h.losses); dev_free(h.term);
    dev_free(h.perms);
    if (h.ev_small) cudaEventDestroy(h.ev_small);
    if (h.ev_all) cudaEventDestroy(h.ev_all);
  }
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  for (int r = 0; r < kMaxPeers; ++r) {
    if (c->peer_x[r] != nullptr && c->peer_x[r] != c->xbuf) cudaIpcCloseMemHandle(c->peer_x[r]);
    if (c->peer_table[r] != nullptr && c->peer_table[r] != c->bf.obs_table) cudaIpcCloseMemHandle(c->peer_table[r]);
  }
  dev_free(c->xbuf);
  if (c->gather_stream) {
    cudaStreamDestroy(c->gather_stream);
    for (int i = 0; i < 2; ++i) { cudaEventDestroy(c->ev_ready[i]); cudaEventDestroy(c->ev_free[i]); }
    cudaEventDestroy(c->ev_start);
  }
  if (c->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(c->comm);
  delete c;
}

extern "C" B2_EXPORT int b200ppo_set_fp32_terms(b200ppo_ctx* ctx, int32_t terms) {
  B2_CHECK_ARG(ctx && (terms == 2 || terms == 3), "b200ppo_set_fp32_terms: terms must be 2 or 3");
  ctx->arena.terms = terms;
  return B200PPO_OK;
}

extern "C" B2_EXPORT int64_t b200ppo_param_count(const b200ppo_ctx* c) { return c ? c->n_params : 0; }
extern "C" B2_EXPORT int64_t b200ppo_actor_param_count(const b200ppo_ctx* c) { return c ? c->n_actor : 0; }

extern "C" B2_EXPORT int64_t b200ppo_param_offset(const b200ppo_ctx* c, int32_t net, int32_t layer, int32_t what) {
  if (!c || net < 0 || net > 1) return -1;
  const Net& N = c->net[net];
  if (net == 0 && layer == N.d.n_layers && what == 0) return c->logstd_off;
  if (layer < 0 || layer >= N.d.n_layers || what < 0 || what > 1) return -1;
  return what == 0 ? N.w_off[layer] : N.b_off[layer];
}

extern "C" B2_EXPORT int64_t b200ppo_saved_size(const b200ppo_ctx* c, int32_t net, int64_t batch) {
  if (!c || net < 0 || net > 1) return -1;
  return c->net[net].hidden_sum * batch;
}

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
  if (ctx->precision == B200PPO_PREC_BF16 && chain_applicable(ctx)) {
    // the bf16 variant's rollout step: weights and observations to bf16, then ONE tensor-core launch (the forward half of the
    // chain kernel) that leaves mean, sampled action, its log-probability and the value (B200PPO_CHAIN_INFER=0: fp32 path)
    static const char* mode = getenv("B200PPO_CHAIN_INFER");
    if (!(mode != nullptr && mode[0] == '0')) {
      B2_TRY(cast_weights(ctx, params, st));
      B2_TRY(launch_cast_rows_ones(obs, batch, ctx->net[0].d.in_dim, ctx->bf.X, ctx->bf.pitchX, st));
      ChainInfer inf{};
      inf.noise = noise; inf.mean = mean; inf.value = value; inf.action = action; inf.logp = logp;
      int grid = 0;
      return launch_chain(ctx, params, ctx->bf.X, batch, nullptr, nullptr, nullptr, nullptr, nullptr, &grid, st, false, &inf);
    }
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
  if (ctx->precision == B200PPO_PREC_BF16 && chain_applicable(ctx)) {
    static const char* mode = getenv("B200PPO_CHAIN_INFER");
    if (!(mode != nullptr && mode[0] == '0')) {
      B2_TRY(cast_weights(ctx, params, st));
      B2_TRY(launch_cast_rows_ones(obs, n_envs, D, ctx->bf.X, ctx->bf.pitchX, st));
      ChainInfer inf{};
      inf.noise = last ? nullptr : noise;
      inf.value = last ? nullptr : buf_value + t;
      inf.value2 = nv;
      inf.action = last ? nullptr : buf_action + t * A;
      inf.logp = last ? nullptr : buf_logp + t;
      inf.ld_action = T * A; inf.ld_value = T; inf.ld_logp = T;
      int grid = 0;
      return launch_chain(ctx, params, ctx->bf.X, n_envs, nullptr, nullptr, nullptr, nullptr, nullptr, &grid, st, false, &inf);
    }
  }
  // other contexts: the plain inference into scratch, then one scatter into the buffers
  if (ctx->rollout_tmp_rows < n_envs) {
    B2_CUDA(cudaDeviceSynchronize());
    dev_free(ctx->rollout_tmp);
    ctx->rollout_tmp_rows = 0;
    B2_TRY(dev_alloc(&ctx->rollout_tmp, ctx->max_batch * (A + 2)));
    ctx->rollout_tmp_rows = ctx->max_batch;
  }
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
  LossArgs la{};
  la.mean = outs[0]; la.logstd = params + ctx->logstd_off; la.action = action; la.batch = batch;
  la.act_dim = ctx->net[0].out_dim(); la.final_tanh = ctx->net[0].d.final_tanh; la.out_scale = ctx->net[0].d.out_scale;
  la.inv_global_batch = 1.f / float(batch); la.rank_share = 1.f;
  la.logp_out = logp; la.entropy_out = entropy;
  la.partials = ctx->loss_partials; la.ticket = ctx->ticket;
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
  const int D = ctx->net[0].d.in_dim, A = ctx->net[0].out_dim();
  int64_t step = *adam_step_io;
  const bool tc = ctx->precision == B200PPO_PREC_BF16;
  const int PX = ctx->bf.pitchX;
  if (tc) PROF(ctx, B200PPO_PROF_OTHER, st, cast_weights(ctx, params, st));
  // fp32-tolerance tensor-core GEMMs: the largest observation of the rollout bounds every minibatch's rows, so their fp16
  // scale needs no measuring pass per minibatch (gemm.cuh a_bound_dev)
  struct BoundFlag { bool& f; ~BoundFlag() { f = false; } } bound_flag{ctx->obs_amax_ok};
  if (!tc && !shared_obs && ctx->arena_need > 0 && lb * int64_t(D) >= (1 << 20)) {
    PROF(ctx, B200PPO_PROF_OTHER, st, launch_absmax(obs, n_samples, D, D, ctx->obs_amax, st));
    ctx->obs_amax_ok = true;
  }
  // Every epoch gathers nb*lb observation rows.  Converting on the fly reads 4D and writes 2*pitch bytes per row and
  // epoch; converting the whole rollout ONCE and then gathering bf16 rows byte for byte (bulk-copy kernel) costs
  // n_samples*(4D + 2*pitch) up front and 4*pitch per row and epoch.  Same bits either way.
  bool table = false;
  if (tc && PX % 8 == 0 && !shared_obs) {
    const double direct = double(epochs) * double(nb * lb) * (4.0 * D + 2.0 * PX);
    const double pre = double(n_samples) * (4.0 * D + 2.0 * PX) + double(epochs) * double(nb * lb) * 4.0 * PX;
    table = pre < 0.9 * direct && nb * lb >= 4096;
  }
  if (table) {
    if (n_samples > ctx->bf.table_cap) {
      B2_CUDA(cudaDeviceSynchronize());
      dev_free(ctx->bf.obs_table);
      ctx->bf.table_cap = 0;
      B2_TRY(dev_alloc(&ctx->bf.obs_table, n_samples * PX));
      ctx->bf.table_cap = n_samples;
    }
    PROF(ctx, B200PPO_PROF_GATHER, st, launch_cast_rows_ones(obs, n_samples, D, ctx->bf.obs_table, PX, st));
  }
  // shuffled_memory = memory[idx] restricted to the rows this rank will consume (ppo.py:103-106).  The permutations are
  // known up front, so the gather of epoch e + 1 runs on a side stream into the other buffer set while epoch e trains:
  // the update kernels are latency-bound and leave HBM idle, the copy engine work hides behind them.
  const bool overlap = epochs > 1 && !ctx->prof.on;
  const int64_t cap = ctx->sh_cap;
  auto gather_epoch = [&](int e, int set, cudaStream_t gs) -> int {
    const int64_t o = int64_t(set) * cap;
    // global permutations: rank r's rows of minibatch i sit at slots i * batch + r * lb ...; rank slices: at i * lb ...
    const bool sliced = ctx->perm_rank_slices;
    const int64_t* idx = perms + int64_t(e) * (sliced ? (n_samples / batch) * lb : n_samples);
    const int64_t cstride = sliced ? lb : batch, coff = sliced ? 0 : int64_t(ctx->rank) * lb;
    if (shared_obs) {  // rows pulled from every rank's table over NVLink by the copy engine
      const float* parts[kMaxPeers];
      for (int r = 0; r < ctx->world; ++r)
        parts[r] = reinterpret_cast<const float*>((ctx->replicated && r != ctx->rank) ? ctx->replica + int64_t(r) * ctx->shared_rows * PX
                                                                                        : ctx->peer_table[r]);
      return launch_gather_parts(idx, nb * lb, n_samples, lb, cstride, coff, parts, ctx->world, ctx->shared_rows, PX / 2,
                                 action, A, old_logp, advantage, target, reinterpret_cast<float*>(ctx->bf.sh_obs + o * PX),
                                 ctx->sh_act + o * A, ctx->sh_logp + o, ctx->sh_adv + o, ctx->sh_tgt + o, ctx->err_flag, gs);
    }
    if (table)  // bf16 rows moved as PX/2 "floats" by the bulk-copy gather: a byte copy
      return launch_gather_chunked(idx, nb * lb, n_samples, lb, cstride, coff,
                                   reinterpret_cast<const float*>(ctx->bf.obs_table), PX / 2, action, A, old_logp, advantage, target,
                                   reinterpret_cast<float*>(ctx->bf.sh_obs + o * PX), ctx->sh_act + o * A, ctx->sh_logp + o,
                                   ctx->sh_adv + o, ctx->sh_tgt + o, ctx->err_flag, gs);
    if (tc)
      return launch_gather_chunked_bf16(idx, nb * lb, n_samples, lb, cstride, coff, obs, D, action, A, old_logp,
                                        advantage, target, ctx->bf.sh_obs + o * PX, PX, ctx->sh_act + o * A, ctx->sh_logp + o,
                                        ctx->sh_adv + o, ctx->sh_tgt + o, ctx->err_flag, gs);
    return launch_gather_chunked(idx, nb * lb, n_samples, lb, cstride, coff, obs, D, action, A, old_logp, advantage,
                                 target, ctx->sh_obs + o * D, ctx->sh_act + o * A, ctx->sh_logp + o, ctx->sh_adv + o, ctx->sh_tgt + o,
                                 ctx->err_flag, gs);
  };
  if (overlap) {
    B2_CUDA(cudaEventRecord(ctx->ev_start, st));  // the rollout (and the bf16 table) are complete on the caller's stream
    B2_CUDA(cudaStreamWaitEvent(ctx->gather_stream, ctx->ev_start, 0));
    B2_TRY(gather_epoch(0, 0, ctx->gather_stream));
    B2_CUDA(cudaEventRecord(ctx->ev_ready[0], ctx->gather_stream));
  }
  for (int e = 0; e < epochs; ++e) {
    const int set = overlap ? (e & 1) : 0;
    if (overlap) {
      if (e + 1 < epochs) {
        if (e >= 1) B2_CUDA(cudaStreamWaitEvent(ctx->gather_stream, ctx->ev_free[(e + 1) & 1], 0));  // epoch e-1 is done with that set
        B2_TRY(gather_epoch(e + 1, (e + 1) & 1, ctx->gather_stream));
        B2_CUDA(cudaEventRecord(ctx->ev_ready[(e + 1) & 1], ctx->gather_stream));
      }
      B2_CUDA(cudaStreamWaitEvent(st, ctx->ev_ready[set], 0));
    } else {
      PROF(ctx, B200PPO_PROF_GATHER, st, gather_epoch(e, 0, st));
    }
    const int64_t so = int64_t(set) * cap;
    for (int64_t i = 0; i < nb; ++i) {
      const int64_t r0 = so + i * lb;
      // from the second minibatch of an epoch on, the kernel in front of the chain kernel is this epoch's optimizer step
      // and the minibatch's rows were gathered before it: the chain kernel may prefetch them across the PDL boundary
      struct EpochFlag { bool& f; ~EpochFlag() { f = false; } } epoch_flag{ctx->in_epoch};
      ctx->in_epoch = i > 0;
      float* loss_slot = losses_out ? losses_out + (int64_t(e) * nb + i) * 2 : ctx->scratch;
      int split = 1, loss_ctas = 0;
      ++step;
      const AdamScalars sa = make_adam_scalars(hp->learning_rate_actor, hp->beta1, hp->beta2, hp->adam_eps, step);
      const AdamScalars sc = make_adam_scalars(hp->learning_rate_critic, hp->beta1, hp->beta2, hp->adam_eps, step);
      if (ctx->world == 1) {
        B2_TRY(minibatch_fwd_bwd(ctx, params, tc ? nullptr : ctx->sh_obs + r0 * D, tc ? ctx->bf.sh_obs + r0 * PX : nullptr,
                                 ctx->sh_act + r0 * A, ctx->sh_logp + r0, ctx->sh_adv + r0, ctx->sh_tgt + r0, lb, hp,
                                 loss_slot, &split, &loss_ctas, st));
        if (tc)  // Adam + bf16 re-cast of the weights (+ the finish of the fused-epilogue loss partials) in one pass
          PROF(ctx, B200PPO_PROF_ADAM, st,
               launch_adam_cast(params, ctx->gpart, split, ctx->n_params, exp_avg, exp_avg_sq, ctx->n_params, ctx->n_actor,
                                sa, sc, cast_group(ctx, params), make_loss_combine(ctx, params, loss_ctas, lb, hp, loss_slot),
                                st));
        else
          PROF(ctx, B200PPO_PROF_ADAM, st,
               launch_adam(params, ctx->gpart, split, ctx->n_params, exp_avg, exp_avg_sq, ctx->n_params, ctx->n_actor, sa,
                           sc, nullptr, st));
      } else if (ctx->p2p && tc) {
        // peer-memory exchange fused into the optimizer kernel: reduce the split-K partials into this rank's exchange
        // buffer, then Adam waits for the peers' flags and sums the G buffers in rank order (adam.cu)
        const unsigned seq = ++ctx->p2p_seq;
        const int64_t xo = int64_t(seq & 1) * ctx->xstride;
        float* xb = ctx->xbuf + xo;
        float* red_losses = xb + ctx->n_params;
        B2_TRY(minibatch_fwd_bwd(ctx, params, nullptr, ctx->bf.sh_obs + r0 * PX, ctx->sh_act + r0 * A, ctx->sh_logp + r0,
                                 ctx->sh_adv + r0, ctx->sh_tgt + r0, lb, hp, red_losses, &split, &loss_ctas, st));
        const LossCombine lc = make_loss_combine(ctx, params, loss_ctas, lb, hp, red_losses);
        // the sum of this rank's split-K partials into its exchange buffer happens inside the optimizer kernel (one
        // element per thread); a small grid or no loss partials keep the separate launch in front of it
        const int agrid = adam_cast_grid(ctx->n_params);
        const bool fused = loss_ctas > 0 && int64_t(agrid) * 256 >= ctx->n_params / 4;
        if (!fused) PROF(ctx, B200PPO_PROF_OTHER, st, launch_reduce_partials(ctx->gpart, split, ctx->n_params, ctx->n_params, xb, st, &lc));
        PeerSrc ps{};
        ps.world = ctx->world; ps.rank = ctx->rank; ps.seq = seq; ps.err = ctx->err_flag; ps.losses_out = loss_slot;
        static const long long timeout_ms = []() { const char* e = getenv("B200PPO_PEER_TIMEOUT_MS"); return e ? atoll(e) : 30000ll; }();
        ps.timeout_cycles = timeout_ms * 2000000ll;  // ~2 GHz SM clock
        unsigned* flags0 = reinterpret_cast<unsigned*>(ctx->xbuf + 2 * ctx->xstride);
        ps.flags_local = flags0;
        for (int r = 0; r < ctx->world; ++r) {
          ps.src[r] = ctx->peer_x[r] + xo;
          ps.flags_peer[r] = reinterpret_cast<unsigned*>(ctx->peer_x[r] + 2 * ctx->xstride);
        }
        if (fused) {
          ps.local_out = xb;
          ps.done_counter = ctx->done_counter;
          ctx->done_total += unsigned(agrid);
          ps.done_target = ctx->done_total;
          PROF(ctx, B200PPO_PROF_ADAM, st,
               launch_adam_cast(params, ctx->gpart, split, ctx->n_params, exp_avg, exp_avg_sq, ctx->n_params, ctx->n_actor, sa, sc,
                                cast_group(ctx, params), lc, st, &ps));
        } else {
          PROF(ctx, B200PPO_PROF_ADAM, st,
               launch_adam_cast(params, xb, 1, ctx->n_params, exp_avg, exp_avg_sq, ctx->n_params, ctx->n_actor, sa, sc,
                                cast_group(ctx, params), LossCombine{}, st, &ps));
        }
      } else {
        float* red_losses = ctx->grad_flat + ctx->n_params;
        B2_TRY(minibatch_fwd_bwd(ctx, params, tc ? nullptr : ctx->sh_obs + r0 * D, tc ? ctx->bf.sh_obs + r0 * PX : nullptr,
                                 ctx->sh_act + r0 * A, ctx->sh_logp + r0, ctx->sh_adv + r0, ctx->sh_tgt + r0, lb, hp,
                                 red_losses, &split, &loss_ctas, st));
        const LossCombine lc = make_loss_combine(ctx, params, loss_ctas, lb, hp, red_losses);
        PROF(ctx, B200PPO_PROF_OTHER, st,
             launch_reduce_partials(ctx->gpart, split, ctx->n_params, ctx->n_params, ctx->grad_flat, st, &lc));
        ctx->prof.begin(B200PPO_PROF_ALLREDUCE, st);
        const int rc = g_nccl.AllReduce(ctx->grad_flat, ctx->grad_flat, size_t(ctx->n_params + 4), /*ncclFloat32*/ 7,
                                        /*ncclSum*/ 0, ctx->comm, st);
        ctx->prof.end(st);
        if (rc != 0) {
          set_error("ncclAllReduce failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?");
          return B200PPO_ENCCL;
        }
        if (tc)
          PROF(ctx, B200PPO_PROF_ADAM, st,
               launch_adam_cast(params, ctx->grad_flat, 1, ctx->n_params, exp_avg, exp_avg_sq, ctx->n_params, ctx->n_actor,
                                sa, sc, cast_group(ctx, params), LossCombine{}, st));
        else
          PROF(ctx, B200PPO_PROF_ADAM, st,
               launch_adam(params, ctx->grad_flat, 1, ctx->n_params, exp_avg, exp_avg_sq, ctx->n_params, ctx->n_actor, sa,
                           sc, nullptr, st));
        copy2_kernel<<<1, 32, 0, st>>>(red_losses, loss_slot);
        B2_LAUNCH_CHECK();
      }
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
    dev_free(h.obs); dev_free(h.act); dev_free(h.logp); dev_free(h.rew); dev_free(h.val); dev_free(h.nval);
    dev_free(h.adv); dev_free(h.tgt); dev_free(h.term);
    h.rows = 0;
    B2_TRY(dev_alloc(&h.obs, M * D)); B2_TRY(dev_alloc(&h.act, M * A)); B2_TRY(dev_alloc(&h.logp, M));
    B2_TRY(dev_alloc(&h.rew, M)); B2_TRY(dev_alloc(&h.val, M)); B2_TRY(dev_alloc(&h.nval, M));
    B2_TRY(dev_alloc(&h.adv, M)); B2_TRY(dev_alloc(&h.tgt, M)); B2_TRY(dev_alloc(&h.term, M));
    h.rows = M;
  }
  if (h.perm_elems < int64_t(epochs) * M) {
    B2_CUDA(cudaDeviceSynchronize());
    dev_free(h.perms);
    B2_TRY(dev_alloc(&h.perms, int64_t(epochs) * M));
    h.perm_elems = int64_t(epochs) * M;
  }
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
  if (h.loss_elems < n_loss) {
    B2_CUDA(cudaDeviceSynchronize());
    dev_free(h.losses);
    B2_TRY(dev_alloc(&h.losses, n_loss));
    h.loss_elems = n_loss;
  }
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

// ---- instrumentation -----------------------------------------------------------------------------------
extern "C" B2_EXPORT int64_t b200ppo_launch_count(void) { return g_launches.load(); }

namespace b200ppo {
__global__ void bf16_rows_to_f32(const __nv_bfloat16* __restrict__ src, int64_t rows, int cols, int pitch, float* __restrict__ dst) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i < rows * cols) dst[i] = __bfloat162float(src[(i / cols) * pitch + i % cols]);
}
}  // namespace b200ppo

extern "C" B2_EXPORT int b200ppo_debug_activations(b200ppo_ctx* ctx, int32_t net, int32_t kind, int32_t layer, int64_t rows,
                                                   float* out, b200ppo_stream stream) {
  B2_CHECK_ARG(ctx && out && (net == 0 || net == 1) && (kind == 0 || kind == 1), "b200ppo_debug_activations: bad argument");
  B2_CHECK_ARG(ctx->precision == B200PPO_PREC_BF16, "b200ppo_debug_activations: bf16 contexts only");
  const Net& N = ctx->net[net];
  B2_CHECK_ARG(layer >= 0 && layer < N.d.n_layers - (kind == 0 ? 1 : 0) && rows > 0 && rows <= ctx->max_batch,
               "b200ppo_debug_activations: layer / rows out of range");
  const __nv_bfloat16* src = kind == 0 ? ctx->bf.H[net][layer] : ctx->bf.dZ[net][layer];
  const int pitch = kind == 0 ? ctx->bf.pitchH[net][layer] : ctx->bf.pitchZ[net][layer];
  const int cols = N.d.dims[layer];
  bf16_rows_to_f32<<<unsigned((rows * cols + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(src, rows, cols, pitch, out);
  B2_LAUNCH_CHECK();
  return B200PPO_OK;
}

extern "C" B2_EXPORT int b200ppo_profile_begin(b200ppo_ctx* ctx) {
  B2_CHECK_ARG(ctx, "b200ppo_profile_begin: null context");
  for (auto& r : ctx->prof.recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
  ctx->prof.recs.clear();
  ctx->prof.on = true;
  return B200PPO_OK;
}

extern "C" B2_EXPORT int b200ppo_profile_end(b200ppo_ctx* ctx, double ms_out[B200PPO_PROF_CLASSES],
                                             int64_t launches_out[B200PPO_PROF_CLASSES]) {
  B2_CHECK_ARG(ctx && ms_out && launches_out, "b200ppo_profile_end: null pointer");
  ctx->prof.on = false;
  B2_CUDA(cudaDeviceSynchronize());
  for (int i = 0; i < B200PPO_PROF_CLASSES; ++i) { ms_out[i] = 0.0; launches_out[i] = 0; }
  for (auto& r : ctx->prof.recs) {
    float ms = 0.f;
    if (r.b != nullptr && cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) {
      ms_out[r.cls] += ms;
      launches_out[r.cls] += 1;
    }
    cudaEventDestroy(r.a); cudaEventDestroy(r.b);
  }
  ctx->prof.recs.clear();
  return B200PPO_OK;
}

// ---- multi-GPU ----------------------------------------------------------------------------------------
extern "C" B2_EXPORT int b200ppo_comm_unique_id(uint8_t id_out[128]) {
  B2_TRY(load_nccl());
  const int rc = g_nccl.GetUniqueId(id_out);
  if (rc != 0) { set_error("ncclGetUniqueId failed (%d)", rc); return B200PPO_ENCCL; }
  return B200PPO_OK;
}

extern "C" B2_EXPORT int b200ppo_comm_init(b200ppo_ctx* ctx, const uint8_t unique_id[128], int32_t rank, int32_t world_size) {
  B2_CHECK_ARG(ctx && unique_id && world_size >= 1 && rank >= 0 && rank < world_size, "b200ppo_comm_init: bad argument");
  if (world_size == 1) { ctx->rank = 0; ctx->world = 1; return B200PPO_OK; }
  B2_TRY(load_nccl());
  NcclApi::Id128 id;
  memcpy(id.b, unique_id, 128);
  void* comm = nullptr;
  const int rc = g_nccl.CommInitRank(&comm, world_size, id, rank);
  if (rc != 0) {
    set_error("ncclCommInitRank failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?");
    return B200PPO_ENCCL;
  }
  ctx->comm = comm; ctx->rank = rank; ctx->world = world_size;
  return B200PPO_OK;
}

extern "C" B2_EXPORT int b200ppo_p2p_export(b200ppo_ctx* ctx, uint8_t handle_out[64]) {
  B2_CHECK_ARG(ctx && handle_out, "b200ppo_p2p_export: null pointer");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  if (ctx->xbuf == nullptr) {
    ctx->xstride = (ctx->n_params + 4 + 31) / 32 * 32;
    B2_TRY(dev_alloc(&ctx->xbuf, 2 * ctx->xstride + 64, true));  // + the flag array (kMaxPeers words, padded)
    B2_CUDA(cudaDeviceSynchronize());
  }
  cudaIpcMemHandle_t h;
  B2_CUDA(cudaIpcGetMemHandle(&h, ctx->xbuf));
  memcpy(handle_out, &h, 64);
  return B200PPO_OK;
}

extern "C" B2_EXPORT int b200ppo_p2p_import(b200ppo_ctx* ctx, const uint8_t* handles, int32_t world_size) {
  B2_CHECK_ARG(ctx && handles, "b200ppo_p2p_import: null pointer");
  B2_CHECK_ARG(ctx->xbuf != nullptr, "b200ppo_p2p_import: call b200ppo_p2p_export first");
  B2_CHECK_ARG(world_size == ctx->world && world_size >= 2 && world_size <= kMaxPeers,
               "b200ppo_p2p_import: world size %d does not match the communicator (%d) or exceeds %d", world_size, ctx->world, kMaxPeers);
  for (int r = 0; r < world_size; ++r) {
    if (r == ctx->rank) {
      ctx->peer_x[r] = ctx->xbuf;
      continue;
    }
    cudaIpcMemHandle_t h;
    memcpy(&h, handles + 64 * r, 64);
    void* ptr = nullptr;
    B2_CUDA(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
    ctx->peer_x[r] = static_cast<float*>(ptr);
  }
  return B200PPO_OK;
}

extern "C" B2_EXPORT int b200ppo_set_perm_layout(b200ppo_ctx* ctx, int32_t rank_slices) {
  B2_CHECK_ARG(ctx, "b200ppo_set_perm_layout: null context");
  ctx->perm_rank_slices = rank_slices != 0;
  return B200PPO_OK;
}

extern "C" B2_EXPORT int b200ppo_p2p_enable(b200ppo_ctx* ctx, int32_t on) {
  B2_CHECK_ARG(ctx, "b200ppo_p2p_enable: null context");
  if (on) {
    B2_CHECK_ARG(ctx->xbuf != nullptr && ctx->world >= 2, "b200ppo_p2p_enable: export / import the exchange buffers first");
    for (int r = 0; r < ctx->world; ++r) B2_CHECK_ARG(ctx->peer_x[r] != nullptr, "b200ppo_p2p_enable: rank %d is not mapped", r);
  }
  ctx->p2p = on != 0;
  return B200PPO_OK;
}

extern "C" B2_EXPORT int b200ppo_table_export(b200ppo_ctx* ctx, int64_t rows_local, uint8_t handle_out[64]) {
  B2_CHECK_ARG(ctx && handle_out && rows_local > 0, "b200ppo_table_export: bad argument");
  B2_CHECK_ARG(ctx->precision == B200PPO_PREC_BF16 && ctx->bf.pitchX % 8 == 0, "b200ppo_table_export: bf16 contexts only");
  if (rows_local > ctx->bf.table_cap || ctx->shared_rows != rows_local) {
    B2_CUDA(cudaDeviceSynchronize());
    for (int r = 0; r < kMaxPeers; ++r) {
      if (ctx->peer_table[r] != nullptr && ctx->peer_table[r] != ctx->bf.obs_table) cudaIpcCloseMemHandle(ctx->peer_table[r]);
      ctx->peer_table[r] = nullptr;
    }
    if (rows_local > ctx->bf.table_cap) {
      dev_free(ctx->bf.obs_table);
      ctx->bf.table_cap = 0;
      B2_TRY(dev_alloc(&ctx->bf.obs_table, rows_local * ctx->bf.pitchX));
      ctx->bf.table_cap = rows_local;
    }
  }
  ctx->shared_rows = 0;  // until b200ppo_table_import
  ctx->shared_filled = false;
  cudaIpcMemHandle_t h;
  B2_CUDA(cudaIpcGetMemHandle(&h, ctx->bf.obs_table));
  memcpy(handle_out, &h, 64);
  return B200PPO_OK;
}

extern "C" B2_EXPORT int b200ppo_table_import(b200ppo_ctx* ctx, const uint8_t* handles, int32_t world_size, int64_t rows_local) {
  B2_CHECK_ARG(ctx && handles && rows_local > 0 && rows_local <= ctx->bf.table_cap, "b200ppo_table_import: bad argument");
  B2_CHECK_ARG(world_size == ctx->world && world_size >= 2 && world_size <= kMaxPeers, "b200ppo_table_import: world size mismatch");
  for (int r = 0; r < world_size; ++r) {
    if (r == ctx->rank) {
      ctx->peer_table[r] = ctx->bf.obs_table;
      continue;
    }
    cudaIpcMemHandle_t h;
    memcpy(&h, handles + 64 * r, 64);
    void* ptr = nullptr;
    B2_CUDA(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
    ctx->peer_table[r] = static_cast<__nv_bfloat16*>(ptr);
  }
  ctx->shared_rows = rows_local;
  return B200PPO_OK;
}

extern "C" B2_EXPORT int b200ppo_table_fill(b200ppo_ctx* ctx, const float* obs_local, int64_t rows_local, b200ppo_stream stream) {
  B2_CHECK_ARG(ctx && obs_local, "b200ppo_table_fill: null pointer");
  B2_CHECK_ARG(ctx->shared_rows > 0 && rows_local == ctx->shared_rows, "b200ppo_table_fill: tables are shared for %lld rows per rank",
               (long long)ctx->shared_rows);
  B2_TRY(launch_cast_rows_ones(obs_local, rows_local, ctx->net[0].d.in_dim, ctx->bf.obs_table, ctx->bf.pitchX,
                               static_cast<cudaStream_t>(stream)));
  ctx->shared_filled = true;
  ctx->replicated = false;
  return B200PPO_OK;
}

extern "C" B2_EXPORT int b200ppo_table_replicate(b200ppo_ctx* ctx, b200ppo_stream stream) {
  B2_CHECK_ARG(ctx, "b200ppo_table_replicate: null context");
  B2_CHECK_ARG(ctx->shared_rows > 0 && ctx->shared_filled, "b200ppo_table_replicate: fill the shared tables first");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int64_t slab = ctx->shared_rows * ctx->bf.pitchX;
  if (ctx->replica_cap < slab * ctx->world) {
    B2_CUDA(cudaDeviceSynchronize());
    dev_free(ctx->replica);
    ctx->replica_cap = 0;
    B2_TRY(dev_alloc(&ctx->replica, slab * ctx->world));
    ctx->replica_cap = slab * ctx->world;
  }
  // start with the next rank so that the eight ranks do not all pull from rank 0 first
  for (int k = 1; k < ctx->world; ++k) {
    const int r = (ctx->rank + k) % ctx->world;
    B2_CUDA(cudaMemcpyAsync(ctx->replica + int64_t(r) * slab, ctx->peer_table[r], size_t(slab) * sizeof(__nv_bfloat16),
                            cudaMemcpyDeviceToDevice, st));
  }
  ctx->replicated = true;
  return B200PPO_OK;
}

extern "C" B2_EXPORT int b200ppo_comm_world(const b200ppo_ctx* ctx, int32_t* rank, int32_t* world_size) {
  B2_CHECK_ARG(ctx, "b200ppo_comm_world: null context");
  if (rank) *rank = ctx->rank;
  if (world_size) *world_size = ctx->world;
  return B200PPO_OK;
}
