// Multi-GPU: the NCCL communicator, the peer-memory gradient exchange and the observation tables shared across ranks.
#include <dlfcn.h>
#include <string.h>

#include "context.cuh"

namespace b200ppo {

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

int nccl_all_reduce(float* buf, int64_t count, void* comm, cudaStream_t st) {
  const int rc = g_nccl.AllReduce(buf, buf, size_t(count), /*ncclFloat32*/ 7, /*ncclSum*/ 0, comm, st);
  if (rc != 0) {
    set_error("ncclAllReduce failed: %s", g_nccl.GetErrorString ? g_nccl.GetErrorString(rc) : "?");
    return B200PPO_ENCCL;
  }
  return B200PPO_OK;
}

void nccl_comm_destroy(void* comm) {
  if (g_nccl.CommDestroy) g_nccl.CommDestroy(comm);
}

void close_peer_tables(b200ppo_ctx* ctx) {
  for (int r = 0; r < kMaxPeers; ++r) {
    if (ctx->peer_table[r] != nullptr && ctx->peer_table[r] != ctx->bf.obs_table) cudaIpcCloseMemHandle(ctx->peer_table[r]);
    ctx->peer_table[r] = nullptr;
  }
}

// Maps the buffer of every other rank from its 64-byte IPC handle; slot `rank` gets the local buffer.
template <typename T>
static int open_peers(const b200ppo_ctx* ctx, const uint8_t* handles, int world, T* local, T** out) {
  for (int r = 0; r < world; ++r) {
    if (r == ctx->rank) {
      out[r] = local;
      continue;
    }
    cudaIpcMemHandle_t h;
    memcpy(&h, handles + 64 * r, 64);
    void* ptr = nullptr;
    B2_CUDA(cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess));
    out[r] = static_cast<T*>(ptr);
  }
  return B200PPO_OK;
}

}  // namespace b200ppo

using namespace b200ppo;

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
    B2_TRY(ctx->xbuf.alloc(2 * ctx->xstride + 64, true));  // + the flag array (kMaxPeers words, padded)
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
  return open_peers(ctx, handles, world_size, ctx->xbuf.get(), ctx->peer_x);
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
  const int64_t elems = rows_local * ctx->bf.pitchX;
  if (elems > ctx->bf.obs_table.cap() || ctx->shared_rows != rows_local) {
    B2_CUDA(cudaDeviceSynchronize());
    close_peer_tables(ctx);
    if (elems > ctx->bf.obs_table.cap()) B2_TRY(ctx->bf.obs_table.alloc(elems));  // (the device is idle already)
  }
  ctx->shared_rows = 0;  // until b200ppo_table_import
  ctx->shared_filled = false;
  cudaIpcMemHandle_t h;
  B2_CUDA(cudaIpcGetMemHandle(&h, ctx->bf.obs_table));
  memcpy(handle_out, &h, 64);
  return B200PPO_OK;
}

extern "C" B2_EXPORT int b200ppo_table_import(b200ppo_ctx* ctx, const uint8_t* handles, int32_t world_size, int64_t rows_local) {
  B2_CHECK_ARG(ctx && handles && rows_local > 0 && ctx->bf.obs_table != nullptr &&
                   rows_local * ctx->bf.pitchX <= ctx->bf.obs_table.cap(),
               "b200ppo_table_import: bad argument");
  B2_CHECK_ARG(world_size == ctx->world && world_size >= 2 && world_size <= kMaxPeers, "b200ppo_table_import: world size mismatch");
  B2_TRY(open_peers(ctx, handles, world_size, ctx->bf.obs_table.get(), ctx->peer_table));
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
  B2_TRY(ctx->replica.grow(slab * ctx->world));
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
