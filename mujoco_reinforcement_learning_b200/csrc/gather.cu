// K2 — minibatch permutation gather (bit-exact row copies).
//
// replaces: `idx = torch.randperm(len(memory)); shuffled_memory = memory[idx]` and the minibatch slice,
//           src/entities/algorithms/ppo.py:103-106 (tensordict gathers every leaf by idx along dim 0).
//
// One warp per output row: the lane-parallel copy of the obs row is 128-bit vectorised when rows are
// 16-byte aligned (obs_dim % 4 == 0), otherwise 32-bit.  Reads are streamed (ld.global.nc, no L1
// allocation): each source row is touched exactly once per epoch.  The scalar leaves and the short action
// row ride along in the same warp so a minibatch costs one launch.
// Algorithmic bytes per sample: 2*(4*D + 4*A + 12) + 8  (SURVEY.md §8d).
#include <cuda_bf16.h>

#include <algorithm>

#include "common.cuh"
#include "gather.cuh"
#include "tc_ptx.cuh"

namespace b200ppo {

__device__ __forceinline__ int64_t resolve_index(const int64_t* __restrict__ idx, int64_t i, int64_t n_rows,
                                                 int32_t* err_flag) {
  int64_t s = __ldg(idx + i);
  if (s < 0) s += n_rows;  // torch index semantics
  if (s < 0 || s >= n_rows) {
    if (err_flag != nullptr) *err_flag = 1;
    return -1;
  }
  return s;
}

template <bool VEC4>
__global__ void __launch_bounds__(256)
gather_minibatch_kernel(const int64_t* __restrict__ idx, int64_t count, int64_t n_rows, int64_t chunk,
                        int64_t chunk_stride, int64_t chunk_offset, const float* __restrict__ obs, int obs_dim, const float* __restrict__ act, int act_dim,
                        const float* __restrict__ logp, const float* __restrict__ adv, const float* __restrict__ tgt,
                        float* __restrict__ obs_o, float* __restrict__ act_o, float* __restrict__ logp_o,
                        float* __restrict__ adv_o, float* __restrict__ tgt_o, int32_t* err_flag) {
  const int lane = threadIdx.x & 31;
  const int warps_per_block = blockDim.x >> 5;
  for (int64_t i = int64_t(blockIdx.x) * warps_per_block + (threadIdx.x >> 5); i < count;
       i += int64_t(gridDim.x) * warps_per_block) {
    // output row i reads permutation slot (i / chunk) * chunk_stride + chunk_offset + i % chunk: one chunk for a
    // plain gather; one chunk per minibatch when a rank takes its slice of every minibatch.
    const int64_t pos = (chunk == count) ? i + chunk_offset : (i / chunk) * chunk_stride + chunk_offset + i % chunk;
    const int64_t s = resolve_index(idx, pos, n_rows, err_flag);
    if (s < 0) continue;
    const float* src = obs + s * obs_dim;
    float* dst = obs_o + i * obs_dim;
    if constexpr (VEC4) {
      const int n4 = obs_dim >> 2;
      // issue every load of the row before the first store (up to 4 x 128-bit in flight per lane)
      int k = lane;
      for (; k + 96 < n4; k += 128) {
        float4 a = ldg_stream4(src + 4 * k), b = ldg_stream4(src + 4 * (k + 32));
        float4 c = ldg_stream4(src + 4 * (k + 64)), d = ldg_stream4(src + 4 * (k + 96));
        stg_stream4(dst + 4 * k, a); stg_stream4(dst + 4 * (k + 32), b);
        stg_stream4(dst + 4 * (k + 64), c); stg_stream4(dst + 4 * (k + 96), d);
      }
      float4 v[3];
      int m = 0;
#pragma unroll
      for (int u = 0; u < 3; ++u)
        if (k + 32 * u < n4) { v[u] = ldg_stream4(src + 4 * (k + 32 * u)); m = u + 1; }
#pragma unroll
      for (int u = 0; u < 3; ++u)
        if (u < m) stg_stream4(dst + 4 * (k + 32 * u), v[u]);
    } else {
      for (int k = lane; k < obs_dim; k += 32) dst[k] = __ldg(src + k);
    }
    if (act != nullptr)
      for (int k = lane; k < act_dim; k += 32) act_o[i * act_dim + k] = __ldg(act + s * act_dim + k);
    if (lane == 0 && logp != nullptr) logp_o[i] = __ldg(logp + s);
    if (lane == 1 && adv != nullptr) adv_o[i] = __ldg(adv + s);
    if (lane == 2 && tgt != nullptr) tgt_o[i] = __ldg(tgt + s);
  }
}


// The observation rows may live in several arrays of equal length (multi-GPU: every rank's slab of the rollout, its own
// and its peers' mapped over NVLink) — row s is row s % rows_per_part of part s / rows_per_part.
struct ObsParts {
  const float* part[8];
  int64_t rows_per_part;
  int count;  // 0: one array (`obs`)
};

// ---- TMA (bulk-copy) variant of the fp32 gather ----------------------------------------------------------------------
// When an observation row is a multiple of 16 bytes (376 floats = 1504 B), each LANE drives its own row through the
// copy engine: cp.async.bulk global -> its shared-memory slot (mbarrier completion), then cp.async.bulk slot -> global.
// No registers hold row data, 32 rows are in flight per warp (48 KB), and the short leaves (action row, three
// scalars) are copied by the same lane while its bulk load is in the air.  One warp per CTA, slots = 32 x row_bytes.
__global__ void __launch_bounds__(32)
gather_minibatch_tma_kernel(const int64_t* __restrict__ idx, int64_t count, int64_t n_rows, int64_t chunk, int64_t chunk_stride,
                            int64_t chunk_offset, const float* __restrict__ obs, int obs_dim, const float* __restrict__ act,
                            int act_dim, const float* __restrict__ logp, const float* __restrict__ adv,
                            const float* __restrict__ tgt, float* __restrict__ obs_o, float* __restrict__ act_o,
                            float* __restrict__ logp_o, float* __restrict__ adv_o, float* __restrict__ tgt_o, int32_t* err_flag,
                            const ObsParts parts) {
  extern __shared__ __align__(128) uint8_t slots[];
  __shared__ __align__(8) uint64_t bars[32];
  const int lane = threadIdx.x;
  const uint32_t row_bytes = uint32_t(obs_dim) * 4u;
  const uint32_t slot = smem_u32(slots) + lane * row_bytes;
  uint64_t* bar = &bars[lane];
  mbar_init(bar, 1);
  mbar_init_fence();
  __syncwarp();
  uint32_t phase = 0;
  for (int64_t i = int64_t(blockIdx.x) * 32 + lane; i < count; i += int64_t(gridDim.x) * 32) {
    const int64_t pos = (chunk == count) ? i + chunk_offset : (i / chunk) * chunk_stride + chunk_offset + i % chunk;
    const int64_t s = resolve_index(idx, pos, n_rows, err_flag);
    if (s < 0) continue;
    // the previous bulk store of this lane must have finished READING the slot before it is refilled
    bulk_wait_read<0>();
    mbar_expect_tx(bar, row_bytes);
    const float* src;
    if (parts.count > 0) {
      const int64_t pi = s / parts.rows_per_part;
      src = parts.part[pi] + (s - pi * parts.rows_per_part) * obs_dim;
    } else {
      src = obs + s * obs_dim;
    }
    bulk_load(slot, src, row_bytes, bar);
    // short leaves while the row is in flight
    if (act != nullptr)
      for (int k = 0; k < act_dim; ++k) act_o[i * act_dim + k] = __ldg(act + s * act_dim + k);
    if (logp != nullptr) logp_o[i] = __ldg(logp + s);
    if (adv != nullptr) adv_o[i] = __ldg(adv + s);
    if (tgt != nullptr) tgt_o[i] = __ldg(tgt + s);
    mbar_wait(bar, phase);
    phase ^= 1u;
    bulk_store(obs_o + i * obs_dim, slot, row_bytes);
    bulk_commit();
  }
  bulk_wait<0>();
}

// Same gather, observations emitted as bf16 rows of pitch `pitch` elements with a 1.0 in column obs_dim (the
// ones-column from which the tensor-core wgrad reads the bias gradient); the other leaves stay fp32.
__global__ void __launch_bounds__(256)
gather_minibatch_bf16_kernel(const int64_t* __restrict__ idx, int64_t count, int64_t n_rows, int64_t chunk,
                             int64_t chunk_stride, int64_t chunk_offset, const float* __restrict__ obs, int obs_dim,
                             const float* __restrict__ act, int act_dim, const float* __restrict__ logp,
                             const float* __restrict__ adv, const float* __restrict__ tgt,
                             __nv_bfloat16* __restrict__ obs_o, int pitch, float* __restrict__ act_o,
                             float* __restrict__ logp_o, float* __restrict__ adv_o, float* __restrict__ tgt_o,
                             int32_t* err_flag, int vec4) {
  const int lane = threadIdx.x & 31;
  const int warps_per_block = blockDim.x >> 5;
  for (int64_t i = int64_t(blockIdx.x) * warps_per_block + (threadIdx.x >> 5); i < count;
       i += int64_t(gridDim.x) * warps_per_block) {
    const int64_t pos = (chunk == count) ? i + chunk_offset : (i / chunk) * chunk_stride + chunk_offset + i % chunk;
    const int64_t s = resolve_index(idx, pos, n_rows, err_flag);
    if (s < 0) continue;
    const float* src = obs + s * obs_dim;
    __nv_bfloat16* dst = obs_o + i * pitch;
    if (vec4) {
      const int n4 = obs_dim >> 2;
      for (int k = lane; k < n4; k += 32) {
        const float4 v = ldg_stream4(src + 4 * k);
        const __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
        uint2 w;
        w.x = *reinterpret_cast<const uint32_t*>(&lo);
        w.y = *reinterpret_cast<const uint32_t*>(&hi);
        *reinterpret_cast<uint2*>(dst + 4 * k) = w;
      }
    } else {
      for (int k = lane; k < obs_dim; k += 32) dst[k] = __float2bfloat16_rn(__ldg(src + k));
    }
    for (int k = obs_dim + lane; k < pitch; k += 32) dst[k] = __float2bfloat16_rn(k == obs_dim ? 1.f : 0.f);
    if (act != nullptr)
      for (int k = lane; k < act_dim; k += 32) act_o[i * act_dim + k] = __ldg(act + s * act_dim + k);
    if (lane == 0 && logp != nullptr) logp_o[i] = __ldg(logp + s);
    if (lane == 1 && adv != nullptr) adv_o[i] = __ldg(adv + s);
    if (lane == 2 && tgt != nullptr) tgt_o[i] = __ldg(tgt + s);
  }
}

// Generic leaf gather on raw bytes (16-byte chunks when possible).
template <typename ChunkT>
__global__ void __launch_bounds__(256)
gather_rows_kernel(const ChunkT* __restrict__ src, int64_t chunks_per_row, int64_t n_rows,
                   const int64_t* __restrict__ idx, int64_t count, ChunkT* __restrict__ dst, int32_t* err_flag) {
  const int lane = threadIdx.x & 31;
  const int warps_per_block = blockDim.x >> 5;
  for (int64_t i = int64_t(blockIdx.x) * warps_per_block + (threadIdx.x >> 5); i < count;
       i += int64_t(gridDim.x) * warps_per_block) {
    const int64_t s = resolve_index(idx, i, n_rows, err_flag);
    if (s < 0) continue;
    for (int64_t k = lane; k < chunks_per_row; k += 32) dst[i * chunks_per_row + k] = __ldg(src + s * chunks_per_row + k);
  }
}

static inline unsigned gather_grid(int64_t count, int warps_per_block) {
  int64_t blocks = (count + warps_per_block - 1) / warps_per_block;
  int64_t cap = int64_t(num_sms()) * 8 * 16;  // grid-stride beyond 16 resident waves
  if (blocks > cap) blocks = (cap / num_sms()) * num_sms();
  return unsigned(blocks < 1 ? 1 : blocks);
}

int launch_gather_chunked(const GatherJob& j, const float* obs, int obs_dim, float* obs_o, cudaStream_t st) {
  if (j.count == 0) return B200PPO_OK;
  const bool vec = (obs_dim % 4 == 0) && aligned16(obs) && aligned16(obs_o);
  const size_t tma_smem = size_t(32) * obs_dim * 4;
  if (vec && tma_smem <= 56 * 1024 && j.count >= 4096) {  // bulk-copy engine path (rows are whole 16-byte multiples)
    static bool configured = false;
    if (!configured) {
      B2_CUDA(cudaFuncSetAttribute(gather_minibatch_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 56 * 1024));
      configured = true;
    }
    const int per_sm = int(std::max<size_t>(1, std::min<size_t>(16, (200 * 1024) / std::max<size_t>(tma_smem, 1))));
    int64_t blocks = std::min<int64_t>((j.count + 31) / 32, int64_t(num_sms()) * per_sm);
    gather_minibatch_tma_kernel<<<unsigned(blocks), 32, tma_smem, st>>>(j.idx, j.count, j.n_rows, j.chunk, j.chunk_stride,
                                                                        j.chunk_offset, obs, obs_dim, j.act, j.act_dim, j.logp,
                                                                        j.adv, j.tgt, obs_o, j.act_o, j.logp_o, j.adv_o, j.tgt_o,
                                                                        j.err_flag, ObsParts{});
    B2_LAUNCH_CHECK();
    return B200PPO_OK;
  }
  dim3 block(256), grid(gather_grid(j.count, 8));
  if (vec)
    gather_minibatch_kernel<true><<<grid, block, 0, st>>>(j.idx, j.count, j.n_rows, j.chunk, j.chunk_stride, j.chunk_offset, obs,
                                                          obs_dim, j.act, j.act_dim, j.logp, j.adv, j.tgt, obs_o, j.act_o,
                                                          j.logp_o, j.adv_o, j.tgt_o, j.err_flag);
  else
    gather_minibatch_kernel<false><<<grid, block, 0, st>>>(j.idx, j.count, j.n_rows, j.chunk, j.chunk_stride, j.chunk_offset, obs,
                                                           obs_dim, j.act, j.act_dim, j.logp, j.adv, j.tgt, obs_o, j.act_o,
                                                           j.logp_o, j.adv_o, j.tgt_o, j.err_flag);
  B2_LAUNCH_CHECK();
  return B200PPO_OK;
}

int launch_gather_parts(const GatherJob& j, const float* const* obs_parts, int n_parts, int64_t rows_per_part, int row_floats,
                        float* obs_o, cudaStream_t st) {
  if (j.count == 0) return B200PPO_OK;
  B2_CHECK_ARG(n_parts >= 1 && n_parts <= 8 && rows_per_part > 0 && j.n_rows <= rows_per_part * n_parts, "gather: bad parts");
  const size_t tma_smem = size_t(32) * row_floats * 4;
  B2_CHECK_ARG(row_floats % 4 == 0 && tma_smem <= 56 * 1024 && aligned16(obs_o), "gather from parts: rows must be 16-byte multiples <= 1792 bytes");
  ObsParts parts{};
  parts.count = n_parts;
  parts.rows_per_part = rows_per_part;
  for (int i = 0; i < n_parts; ++i) {
    B2_CHECK_ARG(obs_parts[i] != nullptr && aligned16(obs_parts[i]), "gather from parts: null or misaligned part");
    parts.part[i] = obs_parts[i];
  }
  static bool configured = false;
  if (!configured) {
    B2_CUDA(cudaFuncSetAttribute(gather_minibatch_tma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 56 * 1024));
    configured = true;
  }
  const int per_sm = int(std::max<size_t>(1, std::min<size_t>(16, (200 * 1024) / std::max<size_t>(tma_smem, 1))));
  int64_t blocks = std::min<int64_t>((j.count + 31) / 32, int64_t(num_sms()) * per_sm);
  gather_minibatch_tma_kernel<<<unsigned(blocks), 32, tma_smem, st>>>(j.idx, j.count, j.n_rows, j.chunk, j.chunk_stride,
                                                                      j.chunk_offset, nullptr, row_floats, j.act, j.act_dim, j.logp,
                                                                      j.adv, j.tgt, obs_o, j.act_o, j.logp_o, j.adv_o, j.tgt_o,
                                                                      j.err_flag, parts);
  B2_LAUNCH_CHECK();
  return B200PPO_OK;
}

int launch_gather_chunked_bf16(const GatherJob& j, const float* obs, int obs_dim, __nv_bfloat16* obs_o, int pitch, cudaStream_t st) {
  if (j.count == 0) return B200PPO_OK;
  const int vec = (obs_dim % 4 == 0) && aligned16(obs) && (pitch % 4 == 0) && ((uintptr_t)obs_o % 8 == 0);
  dim3 block(256), grid(gather_grid(j.count, 8));
  gather_minibatch_bf16_kernel<<<grid, block, 0, st>>>(j.idx, j.count, j.n_rows, j.chunk, j.chunk_stride, j.chunk_offset, obs,
                                                       obs_dim, j.act, j.act_dim, j.logp, j.adv, j.tgt, obs_o, pitch, j.act_o,
                                                       j.logp_o, j.adv_o, j.tgt_o, j.err_flag, vec);
  B2_LAUNCH_CHECK();
  return B200PPO_OK;
}

}  // namespace b200ppo

using namespace b200ppo;

extern "C" B2_EXPORT int b200ppo_gather_minibatch(const int64_t* idx, int64_t count, int64_t n_rows, const float* obs,
                                        int64_t obs_dim, const float* action, int64_t act_dim, const float* logp,
                                        const float* advantage, const float* target, float* obs_out,
                                        float* action_out, float* logp_out, float* advantage_out, float* target_out,
                                        int32_t* err_flag, b200ppo_stream stream) {
  B2_CHECK_ARG(idx && obs && obs_out, "b200ppo_gather_minibatch: null pointer");
  B2_CHECK_ARG((!action || action_out) && (!logp || logp_out) && (!advantage || advantage_out) && (!target || target_out),
               "b200ppo_gather_minibatch: missing output for a supplied leaf");
  B2_CHECK_ARG(count >= 0 && n_rows >= 0 && obs_dim > 0 && obs_dim < (1 << 30) && act_dim >= 0 && act_dim < (1 << 30),
               "b200ppo_gather_minibatch: bad sizes");
  GatherJob j{};
  j.idx = idx; j.count = count; j.n_rows = n_rows; j.chunk = count; j.chunk_stride = count; j.chunk_offset = 0;
  j.act = action; j.act_dim = int(act_dim); j.logp = logp; j.adv = advantage; j.tgt = target;
  j.act_o = action_out; j.logp_o = logp_out; j.adv_o = advantage_out; j.tgt_o = target_out; j.err_flag = err_flag;
  return launch_gather_chunked(j, obs, int(obs_dim), obs_out, static_cast<cudaStream_t>(stream));
}

extern "C" B2_EXPORT int b200ppo_gather_rows(const void* src, int64_t row_bytes, int64_t n_rows, const int64_t* idx,
                                   int64_t count, void* dst, int32_t* err_flag, b200ppo_stream stream) {
  B2_CHECK_ARG(src && idx && dst, "b200ppo_gather_rows: null pointer");
  B2_CHECK_ARG(row_bytes > 0 && count >= 0 && n_rows >= 0, "b200ppo_gather_rows: bad sizes");
  if (count == 0) return B200PPO_OK;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  dim3 block(256), grid(gather_grid(count, 8));
  if (row_bytes % 16 == 0 && aligned16(src) && aligned16(dst))
    gather_rows_kernel<uint4><<<grid, block, 0, st>>>(static_cast<const uint4*>(src), row_bytes / 16, n_rows, idx, count, static_cast<uint4*>(dst), err_flag);
  else if (row_bytes % 4 == 0 && (uintptr_t)src % 4 == 0 && (uintptr_t)dst % 4 == 0)
    gather_rows_kernel<uint32_t><<<grid, block, 0, st>>>(static_cast<const uint32_t*>(src), row_bytes / 4, n_rows, idx, count, static_cast<uint32_t*>(dst), err_flag);
  else
    gather_rows_kernel<uint8_t><<<grid, block, 0, st>>>(static_cast<const uint8_t*>(src), row_bytes, n_rows, idx, count, static_cast<uint8_t*>(dst), err_flag);
  B2_LAUNCH_CHECK();
  return B200PPO_OK;
}
