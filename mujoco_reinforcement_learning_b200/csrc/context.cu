// The context: error text, launch counter, parameter layout, create / destroy, profiling and debug accessors.
#include <stdarg.h>

#include <algorithm>
#include <atomic>

#include "context.cuh"

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

static inline int pad8(int x) { return (x + 7) / 8 * 8; }
static inline int pad16(int x) { return (x + 15) / 16 * 16; }  // rows that start on 32-byte sectors (256-bit loads / stores)

// bf16 operands of the tensor-core path.  Every Linear of both nets runs on tcgen05 (the 17- and 1-wide output
// layers too: a mostly-empty 128x64 tile costs less than a latency-bound SIMT pass).
static int alloc_bf16_workspaces(b200ppo_ctx* c) {
  B2_TRY(tc_init());
  auto& bf = c->bf;
  const int64_t Bm = c->max_batch;
  bf.pitchX = pad8(c->net[0].d.in_dim + 1);
  B2_TRY(bf.X.alloc(Bm * bf.pitchX));
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
        B2_TRY(bf.H[n][l].alloc(Bm * bf.pitchH[n][l]));
        B2_TRY(launch_init_ones_column(bf.H[n][l], Bm, bf.pitchH[n][l], N.d.dims[l], nullptr));
      }
      B2_TRY(bf.dZ[n][l].alloc(Bm * bf.pitchZ[n][l], true));
      B2_TRY(bf.W[n][l].alloc(int64_t(N.d.dims[l]) * bf.pitchW[n][l], true));
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

int check_batch(const b200ppo_ctx* ctx, int64_t B, const char* who) {
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

// Every buffer the context owns from the start; the ones that grow on demand are sized by their first use.
static int alloc_workspaces(b200ppo_ctx* c) {
  const int64_t Bm = c->max_batch;
  for (int n = 0; n < 2; ++n) {
    const Net& N = c->net[n];
    B2_TRY(c->ws_act[n].alloc(Bm * N.hidden_sum));
    B2_TRY(c->ws_dz[n].alloc(Bm * (N.hidden_sum + N.out_dim())));
    B2_TRY(c->ws_out[n].alloc(Bm * N.out_dim()));
  }
  B2_TRY(c->gpart.alloc(int64_t(c->max_split) * c->n_params, true));
  B2_TRY(c->grad_flat.alloc(c->n_params + 4, true));
  B2_TRY(c->loss_partials.alloc(c->loss_partial_rows * (2 + c->net[0].out_dim()), true));
  B2_TRY(c->ticket.alloc(1, true));
  B2_TRY(c->done_counter.alloc(1, true));
  B2_TRY(c->scratch.alloc(8, true));
  B2_TRY(c->err_flag.alloc(1, true));
  B2_TRY(c->obs_amax.alloc(1, true));
  if (c->precision == B200PPO_PREC_BF16) B2_TRY(alloc_bf16_workspaces(c));
  return B200PPO_OK;
}

}  // namespace b200ppo

using namespace b200ppo;

extern "C" B2_EXPORT int b200ppo_version(void) { return B200PPO_VERSION; }
extern "C" B2_EXPORT const char* b200ppo_last_error(void) { return g_err; }
extern "C" B2_EXPORT int64_t b200ppo_launch_count(void) { return g_launches.load(); }

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
  c->loss_partial_rows = std::max<int64_t>(std::max(loss_grid_size(Bm), 8 * num_sms()), 2 * ((Bm + 127) / 128) + 8);
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
  r = alloc_workspaces(c);
  if (r != B200PPO_OK) { b200ppo_destroy(c); return r; }
  *out = c;
  return B200PPO_OK;
}

extern "C" B2_EXPORT void b200ppo_destroy(b200ppo_ctx* c) {
  if (!c) return;
  cudaDeviceSynchronize();
  close_peer_tables(c);
  for (int r = 0; r < kMaxPeers; ++r)
    if (c->peer_x[r] != nullptr && c->peer_x[r] != c->xbuf) cudaIpcCloseMemHandle(c->peer_x[r]);
  for (auto& h : c->host) {
    if (h.ev_small) cudaEventDestroy(h.ev_small);
    if (h.ev_all) cudaEventDestroy(h.ev_all);
  }
  if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
  if (c->gather_stream) {
    cudaStreamDestroy(c->gather_stream);
    for (int i = 0; i < 2; ++i) { cudaEventDestroy(c->ev_ready[i]); cudaEventDestroy(c->ev_free[i]); }
    cudaEventDestroy(c->ev_start);
  }
  for (auto& r : c->prof.recs) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }  // profile_begin without _end
  if (c->comm) nccl_comm_destroy(c->comm);
  delete c;  // the device buffers free themselves
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
  bf16_rows_to_f32_kernel<<<unsigned((rows * cols + 255) / 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(src, rows, cols, pitch, out);
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
