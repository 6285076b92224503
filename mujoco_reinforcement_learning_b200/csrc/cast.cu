// bf16 shadow copies of the fp32 master weights and bf16 staging of observations for the tcgen05 path.
// The optimiser keeps fp32 master parameters (b200ppo_adam_step); after every step the hidden-layer weights are
// re-emitted as bf16 (W as is: K-major for the forward GEMMs, MN-major for the dgrad).
#include <algorithm>

#include "cast.cuh"

namespace b200ppo {

__global__ void __launch_bounds__(256) cast_weights_kernel(const __grid_constant__ WeightCastGroup g) {
  const WeightCast& w = g.w[blockIdx.y];
  const int total = w.out * w.in;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < total; e += gridDim.x * blockDim.x) {
    const int o = e / w.in, i = e - o * w.in;
    w.dst[int64_t(o) * w.pitch + i] = __float2bfloat16_rn(__ldg(w.src + e));
  }
}

__global__ void __launch_bounds__(256)
cast_rows_ones_kernel(const float* __restrict__ src, int64_t rows, int cols, __nv_bfloat16* __restrict__ dst, int pitch) {
  const int64_t total = rows * pitch;
  for (int64_t e = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; e < total; e += int64_t(gridDim.x) * blockDim.x) {
    const int64_t r = e / pitch;
    const int c = int(e - r * pitch);
    dst[e] = __float2bfloat16_rn(c < cols ? __ldg(src + r * cols + c) : (c == cols ? 1.f : 0.f));
  }
}

// Vector path (cols and pitch multiples of 4, 16-byte aligned rows): one float4 in, four bf16 out per thread and step.
__global__ void __launch_bounds__(256)
cast_rows_ones_vec4_kernel(const float* __restrict__ src, int64_t rows, int cols, __nv_bfloat16* __restrict__ dst, int pitch) {
  const int upr = pitch >> 2;  // 4-element units per output row
  const int64_t total = rows * upr;
  for (int64_t u = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; u < total; u += int64_t(gridDim.x) * blockDim.x) {
    const int64_t r = u / upr;
    const int c = int(u - r * upr) << 2;
    float4 v;
    if (c < cols) v = ldg_stream4(src + r * cols + c);
    else v = make_float4(c == cols ? 1.f : 0.f, 0.f, 0.f, 0.f);
    const __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
    uint2 w;
    w.x = *reinterpret_cast<const uint32_t*>(&lo);
    w.y = *reinterpret_cast<const uint32_t*>(&hi);
    *reinterpret_cast<uint2*>(dst + r * pitch + c) = w;
  }
}

__global__ void __launch_bounds__(256) init_ones_column_kernel(__nv_bfloat16* __restrict__ dst, int64_t rows, int pitch, int col) {
  const int64_t total = rows * pitch;
  for (int64_t e = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; e < total; e += int64_t(gridDim.x) * blockDim.x)
    dst[e] = __float2bfloat16_rn((e % pitch) == col ? 1.f : 0.f);
}

int launch_cast_weights(const WeightCastGroup& g, cudaStream_t st) {
  if (g.count == 0) return B200PPO_OK;
  dim3 grid(unsigned(std::min<int64_t>((g.max_elems + 255) / 256, 4 * num_sms())), unsigned(g.count));
  if (grid.x == 0) grid.x = 1;
  cast_weights_kernel<<<grid, 256, 0, st>>>(g);
  B2_LAUNCH_CHECK();
  return B200PPO_OK;
}

int launch_cast_rows_ones(const float* src, int64_t rows, int cols, __nv_bfloat16* dst, int pitch, cudaStream_t st) {
  if (rows == 0) return B200PPO_OK;
  if (cols % 4 == 0 && pitch % 4 == 0 && aligned16(src) && aligned16(dst)) {
    const int64_t blocks = std::min<int64_t>((rows * (pitch / 4) + 255) / 256, 32 * num_sms());
    cast_rows_ones_vec4_kernel<<<unsigned(blocks), 256, 0, st>>>(src, rows, cols, dst, pitch);
    B2_LAUNCH_CHECK();
    return B200PPO_OK;
  }
  const int64_t blocks = std::min<int64_t>((rows * pitch + 255) / 256, 16 * num_sms());
  cast_rows_ones_kernel<<<unsigned(blocks), 256, 0, st>>>(src, rows, cols, dst, pitch);
  B2_LAUNCH_CHECK();
  return B200PPO_OK;
}

int launch_init_ones_column(__nv_bfloat16* dst, int64_t rows, int pitch, int col, cudaStream_t st) {
  if (rows == 0) return B200PPO_OK;
  const int64_t blocks = std::min<int64_t>((rows * pitch + 255) / 256, 16 * num_sms());
  init_ones_column_kernel<<<unsigned(blocks), 256, 0, st>>>(dst, rows, pitch, col);
  B2_LAUNCH_CHECK();
  return B200PPO_OK;
}

}  // namespace b200ppo
