// bf16 operand preparation for the tensor-core path (cast.cu).
#pragma once
#include <cuda_bf16.h>

#include "common.cuh"

namespace b200ppo {

struct WeightCast {
  const float* src;        // W [out, in] fp32 (nn.Linear.weight)
  __nv_bfloat16* dst;      // [out, pitch]      K-major operand of the forward GEMM, MN-major operand of the dgrad
  int out, in, pitch;
};

struct WeightCastGroup {
  WeightCast w[2 * B200PPO_MAX_LAYERS];
  int count;
  int max_elems;
};

int launch_cast_weights(const WeightCastGroup& g, cudaStream_t st);
// dst[r, 0:cols] = bf16(src[r, 0:cols]); dst[r, cols] = 1; dst[r, cols+1:pitch] = 0
int launch_cast_rows_ones(const float* src, int64_t rows, int cols, __nv_bfloat16* dst, int pitch, cudaStream_t st);
// zero a [rows, pitch] bf16 buffer and set column `col` to 1
int launch_init_ones_column(__nv_bfloat16* dst, int64_t rows, int pitch, int col, cudaStream_t st);

}  // namespace b200ppo
