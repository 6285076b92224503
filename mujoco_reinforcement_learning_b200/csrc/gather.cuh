// Launchers of the minibatch gathers (gather.cu).
#pragma once
#include <cuda_bf16.h>

#include "common.cuh"

namespace b200ppo {

// Rows of a shuffled minibatch: output row i takes source row idx[pos] of every leaf, with
// pos = (i / chunk) * chunk_stride + chunk_offset + i % chunk (one rank's slice of each minibatch of an epoch).
// A null leaf is skipped; an index outside [0, n_rows) raises *err_flag.
struct GatherJob {
  const int64_t* idx = nullptr;
  int64_t count = 0, n_rows = 0, chunk = 0, chunk_stride = 0, chunk_offset = 0;
  const float *act = nullptr, *logp = nullptr, *adv = nullptr, *tgt = nullptr;
  int act_dim = 0;
  float *act_o = nullptr, *logp_o = nullptr, *adv_o = nullptr, *tgt_o = nullptr;
  int32_t* err_flag = nullptr;
};

// fp32 observations [n_rows][obs_dim] -> obs_o [count][obs_dim]
int launch_gather_chunked(const GatherJob& j, const float* obs, int obs_dim, float* obs_o, cudaStream_t st);
// observation rows of row_floats floats (a multiple of 4) from n_parts arrays of rows_per_part rows each, every array
// 16-byte aligned, by the bulk-copy kernel
int launch_gather_parts(const GatherJob& j, const float* const* obs_parts, int n_parts, int64_t rows_per_part, int row_floats,
                        float* obs_o, cudaStream_t st);
// fp32 observations converted to bf16 rows [count][pitch] with the ones-column
int launch_gather_chunked_bf16(const GatherJob& j, const float* obs, int obs_dim, __nv_bfloat16* obs_o, int pitch, cudaStream_t st);

}  // namespace b200ppo
