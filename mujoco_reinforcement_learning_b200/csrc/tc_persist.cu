// Persistent variant of the grouped tcgen05 tile kernel (tc_gemm.cu) for the fp32-tolerance GEMMs (gemm_split.cu).
//
// replaces: the same aten::addmm / aten::mm calls as tc_gemm.cu (src/models/network_block_creator.py:74-86, autograd of
//           ppo.py:121,134).
//
// Why: with six products per k range a 128 x 256 tile's main loop is 22-24 k cycles, its set-up + operand latency + epilogue
// another 15 k (profiles/README.md), and a launch of 512 tiles is 3.46 tiles per SM: one-tile CTAs pay the 15 k per tile and
// round 3.46 up to 4.  Here ONE CTA per SM walks the tile list; the accumulator is double-buffered in TMEM (2 x BN columns),
// so the producer and the MMA issuer run into tile i + 1 while the eight epilogue warps drain tile i, and the operand
// ring never empties between tiles.
//
//   warp 0   TMA producer: same boxes as tc_gemm_kernel (three-term coordinates included), ring state carried across tiles
//   warp 1   MMA issuer  : accumulator (tile count & 1); waits for the epilogue to have drained it two tiles ago
//   warps 2-9 epilogue   : tc_epilogue<BN> on the finished accumulator, bias of the tile staged per accumulator
// Tiles whose split has no k tiles (more splits than k tiles) take no accumulator: all three roles skip them alike.
#include "tc_common.cuh"

namespace b200ppo {

template <int BN> struct PersistCfg {
  static constexpr int STAGES = BN <= 192 ? 5 : 4;  // 200 / 192 KB of operands
};

template <int BN>
__global__ void __launch_bounds__(TC_THREADS, 1) tc_persist_kernel(const __grid_constant__ TcGroup grp) {
  constexpr int STAGES = PersistCfg<BN>::STAGES;
  constexpr int B_BYTES = BN * TC_BK * 2;
  constexpr uint32_t TMEM_COLS = 512;  // two accumulators of BN <= 256 columns
  constexpr uint32_t ACC_STRIDE = 256;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* sA = smem;
  uint8_t* sB = smem + STAGES * TC_A_BYTES;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(sB + STAGES * B_BYTES);
  uint64_t* empty_bar = full_bar + STAGES;
  uint64_t* acc_full = empty_bar + STAGES;   // [2]
  uint64_t* acc_empty = acc_full + 2;        // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
  float* bias_s = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(full_bar) + 256);  // [2][256]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int i = 0; i < 2; ++i) {
      mbar_init(&acc_full[i], 1);
      mbar_init(&acc_empty[i], TC_EPI_WARPS);
    }
    mbar_init_fence();
  } else if (warp == 2) {
    tmem_alloc<1, TMEM_COLS>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait_then_release();  // everything below reads what earlier kernels of the stream wrote

  const int n_tiles = grp.total_tiles;
  // debug timeline of CTA 0, eight slots per tile: 0 issuer has the accumulator, 1 first operands, 2 last MMA issued,
  // 3 epilogue (warp 2) sees the accumulator, 4 epilogue done, 5 producer issued the tile's first load, 6 its last load
  long long* const trc = (grp.trace != nullptr && blockIdx.x == 0) ? grp.trace : nullptr;
  if (warp == 0) {
    if (lane == 0) {  // ===== TMA producer =====
      uint32_t git = 0;  // ring iterations since the kernel began
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const TcTile T = tc_tile<BN>(grp, tile);
        const TcProblem& P = grp.p[T.pi];
        for (int it = 0; it < T.n_it; ++it, ++git) {
          const uint32_t s = git % STAGES, ph = (git / STAGES) & 1;
          mbar_wait(&empty_bar[s], ph ^ 1);
          if (trc != nullptr && tile / int(gridDim.x) < 64 && (it == 0 || it == T.n_it - 1)) trc[(tile / gridDim.x) * 8 + (it == 0 ? 5 : 6)] = clock64();
          mbar_expect_tx(&full_bar[s], TC_A_BYTES + B_BYTES);
          tc_load_stage<BN>(P, T, it, sA + s * TC_A_BYTES, sB + s * B_BYTES, &full_bar[s]);
        }
      }
    }
  } else if (warp == 1) {  // ===== MMA issuer =====
    uint32_t git = 0, use = 0;  // ring iterations; accumulators handed out so far
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      const TcTile T = tc_tile<BN>(grp, tile);
      if (T.n_it <= 0) continue;
      const TcProblem& P = grp.p[T.pi];
      const uint32_t acc = use & 1;
      mbar_wait(&acc_empty[acc], ((use >> 1) & 1) ^ 1);  // the epilogue drained this accumulator (two uses ago)
      tc_fence_after();
      if (trc != nullptr && lane == 0 && tile / int(gridDim.x) < 64) trc[(tile / gridDim.x) * 8 + 0] = clock64();
      const uint32_t d = tmem_base + acc * ACC_STRIDE;
      const TcMma mma = tc_mma_setup<BN>(P);
      for (int it = 0; it < T.n_it; ++it, ++git) {
        const uint32_t s = git % STAGES, ph = (git / STAGES) & 1;
        mbar_wait(&full_bar[s], ph);
        tc_fence_after();
        if (trc != nullptr && lane == 0 && tile / int(gridDim.x) < 64 && (it == 0 || it == T.n_it - 1)) trc[(tile / gridDim.x) * 8 + (it == 0 ? 1 : 2)] = clock64();
        if (lane == 0) {
          tc_mma_stage(mma, d, smem_u32(sA + s * TC_A_BYTES), smem_u32(sB + s * B_BYTES), it > 0);
          umma_commit(&empty_bar[s]);
          if (it == T.n_it - 1) umma_commit(&acc_full[acc]);
        }
        __syncwarp();
      }
      ++use;
    }
  } else {  // ===== epilogue warps 2..9 =====
    uint32_t use = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
      const TcTile T = tc_tile<BN>(grp, tile);
      const TcProblem& P = grp.p[T.pi];
      const bool has_k = T.n_it > 0;
      const uint32_t acc = use & 1;
      float* bs = bias_s + acc * 256;
      // the bias of this tile's columns: the warps that read bs for the tile two uses ago have all passed this barrier's
      // predecessor, and nobody reads it before the barrier below
      tc_stage_bias(P, T.n0, BN, bs, threadIdx.x - 64, TC_THREADS - 64);
      asm volatile("bar.sync 1, %0;" ::"n"(TC_THREADS - 64) : "memory");
      if (trc != nullptr && warp == 2 && lane == 0 && tile / int(gridDim.x) < 64) trc[(tile / gridDim.x) * 8 + 3] = clock64();
      tc_epilogue<BN, true>(P, T.split, tmem_base + acc * ACC_STRIDE, has_k, T.m0, T.n0, warp, lane, &acc_full[acc], (use >> 1) & 1, bs);
      if (trc != nullptr && warp == 2 && lane == 0 && tile / int(gridDim.x) < 64) trc[(tile / gridDim.x) * 8 + 4] = clock64();
      if (has_k) {
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_empty[acc]);
        ++use;
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<1, TMEM_COLS>(tmem_base);
  }
}

template <int BN>
static int launch_persist_bn(const TcGroup& g, cudaStream_t st) {
  constexpr int smem = PersistCfg<BN>::STAGES * (TC_A_BYTES + BN * TC_BK * 2) + 1024 + 256 + 2 * 256 * 4 + 64;
  static bool configured = false;
  if (!configured) {
    B2_CUDA(cudaFuncSetAttribute(tc_persist_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    configured = true;
  }
  const int grid = std::min(g.total_tiles, num_sms());
  B2_CUDA(launch_pdl(tc_persist_kernel<BN>, dim3(grid), dim3(TC_THREADS), smem, st, g));
  B2_LAUNCH_CHECK();
  return B200PPO_OK;
}

int launch_tc_persist(const TcGroup& g, int bn, cudaStream_t st) {
  if (g.total_tiles == 0) return B200PPO_OK;
  for (int i = 0; i < g.count; ++i)
    B2_CHECK_ARG(g.p[i].epilogue <= TC_EPI_STORE && !g.p[i].staged, "persistent tile kernel: plain epilogues only");
  switch (bn) {
    case 192: return launch_persist_bn<192>(g, st);
    case 256: return launch_persist_bn<256>(g, st);
  }
  set_error("persistent tile kernel: unsupported N tile %d", bn);
  return B200PPO_EINVAL;
}

}  // namespace b200ppo
