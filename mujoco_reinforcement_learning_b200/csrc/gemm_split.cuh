// fp32-tolerance GEMMs on the tcgen05 tensor cores: every fp32 operand is written as three bf16 terms (x = a + b + c
// to 2^-24 relative) and the products aa, ab, ba, bb, ac, ca accumulate in one fp32 TMEM accumulator (gemm_split.cu).
#pragma once
#include "gemm.cuh"

namespace b200ppo {

// Device arena of the three-term operands of ONE minibatch.  An operand split once (the observations, a hidden
// activation, a weight matrix, a dL/dz block) is found again by source pointer and shape, so the forward's A operand is
// the weight gradient's B operand without a second pass.  Reset whenever the sources may have changed.
struct SplitArena {
  struct Entry {
    const float* src;
    int64_t rows, ld;
    int cols, ones, cp, terms;
    __nv_bfloat16* dst;
    float* amax;  // two-term mode: the largest magnitude of src, the source of its scale
  };
  static constexpr int kMaxEntries = 96;  // 2 nets x B200PPO_MAX_LAYERS x (activation, two dL/dz views, weights) and room to spare
  DevBuf<__nv_bfloat16> base;
  DevBuf<float> amax;         // [kMaxEntries] largest magnitude of every entry's source (two-term mode: the scale comes from it)
  bool amax_zeroed = false;   // since the last reset
  int64_t used = 0;           // elements of base
  Entry e[kMaxEntries];
  int n = 0;
  // 3: three bf16 terms per value, six products — 24-bit operands, the 1e-5 variant (default).  2: two fp16 terms of the
  // scaled value, three products — 22-bit operands: 1.3x faster, every gradient tensor still within 1e-5 of its scale, but a
  // sum that cancels 1000 : 1 (a zero-initialised bias after Adam) shows the two missing bits (b200ppo_set_fp32_terms).
  int terms = 3;
};

int split_arena_reserve(SplitArena& a, int64_t elems);  // grows base to `elems` (DevBuf::grow)
inline void split_arena_reset(SplitArena& a) { a.used = 0; a.n = 0; a.amax_zeroed = false; }
// samples one tensor-core accumulator of a weight gradient may sum (see backward_nets in passes.cu)
constexpr int kSplitChain = 512;
// elements one [rows][cols] operand occupies in the arena
int64_t split_arena_elems(int64_t rows, int cols);

// Every problem K- or MN-contiguous on both operands, no bf16 mirror output, and enough arithmetic to pay for the splits.
bool gemm_split_applicable(const GemmGroup& g);
// max |src[r][c]| over a [rows][cols] array with row pitch ld, into *out (device), on `st`
int launch_absmax(const float* src, int64_t rows, int cols, int64_t ld, float* out, cudaStream_t st);
// Same contract as launch_gemm_group (gemm.cuh): C, bias_grad and split-K partials land where the FFMA kernel puts them.
int launch_gemm_group_split(const GemmGroup& g, SplitArena& arena, cudaStream_t st);

}  // namespace b200ppo
