// One launch for the whole per-minibatch op chain of PPO.train up to the weight gradients: forward of both MLPs,
// log-prob / ratio / clipped surrogate / Huber losses with their gradient seeds, and the dgrad chain back to dZ1.
//
// replaces: ppo.py:110-134 as far as it is row-local — actor(obs), critic(obs) (network_block_creator.py:74-86,
//           linear/actor.py:25-30, critic.py:22-25), Normal.log_prob, the two losses (ppo.py:113-132) and the
//           activation-gradient half of their autograd backward.  Weight gradients (a reduction over rows) stay in
//           tc_wgrad.cu, the optimizer in adam.cu.
//
// Why: as separate launches (tc_ws.cu) every activation crossed HBM twice and every launch paid ~10 us of fill/drain
// for ~10 us of row tiles.  Here a CTA PAIR (cta_group::2) owns a 256-row tile (128 rows per CTA) and walks it through
// ten MMA steps; the epilogue of a step writes its bf16 result STRAIGHT INTO SHARED MEMORY in the K-major 128-byte
// swizzled layout the next step's tcgen05.mma reads as its A operand (and once to HBM for the weight-gradient kernel):
//
//   step  MMA (M = 256, accumulators ping-pong between two 256-column TMEM buffers)      epilogue (16 warps / CTA)
//   0 L1a  X   . W1a^T  K = in   N = 256   -> buf0     H1a = act(acc + b1a)      -> smem HA, global
//   1 L1c  X   . W1c^T                     -> buf1     H1c                       -> smem HC (aliases X), global
//   2 L2a  H1a . W2a^T  K = 256            -> buf0     H2a                       -> smem HA (over H1a), global
//   3 L2c  H1c . W2c^T                     -> buf1     H2c                       -> smem HC, global
//   4 L3a  H2a . W3a^T  N = 32             -> buf0     log-prob, ratio, surrogate, seeds dz3a -> smem, global
//   5 L3c  H2c . W3c^T  N = 16             -> buf1     Huber, seed dv            -> smem, global
//   6 D3a  dz3a . W3a   K = 32  N = 256    -> buf0     dZ2a = acc * act'(H2a)    in place in HA, global
//   7 D3c  dv   . W3c   K = 16             -> buf1     dZ2c                      in place in HC, global
//   8 D2a  dZ2a . W2a   K = 256            -> buf0     dZ1a = acc * act'(H1a from L2) -> global
//   9 D2c  dZ2c . W2c                      -> buf1     dZ1c                      -> global
//
// Actor and critic alternate, so while the epilogue warps finish step s the tensor pipe already runs step s + 1 of the
// other network; step s + 2 (same network) needs exactly what the epilogue of step s produces (its A operand and its
// drained accumulator), which is ONE mbarrier per TMEM buffer.  The weights (640 KB + 256 KB for the dgrads) do not fit
// next to the tiles, so they stream from L2 through a 4-stage ring of 16 KB per CTA (each CTA holds half of N; the pair
// halves the L2->SM weight traffic per row) in exactly the order the MMAs consume them.
//   warp 0 (both CTAs)  TMA producer: X k-blocks + the weight stream; bytes counted on the LEADER's mbarriers
//   warp 1 (leader)     MMA issuer: tcgen05.mma.cta_group::2; tcgen05.commit multicast frees ring stages / publishes accumulators
//   warps 2-17 (both)   epilogue: warp = (TMEM lane quarter, 64-column chunk = one k-block of the next A operand)
#include <algorithm>
#include <cstdlib>

#include "tc_chain.cuh"
#include "tc_common.cuh"

namespace b200ppo {

constexpr int CH_EPI_WARPS = 16;
constexpr int CH_THREADS = (2 + CH_EPI_WARPS) * 32;
constexpr int CH_SLOT = 16384;  // one k-block of a 128-row operand tile: 128 rows x 128 B
constexpr int CH_NSLOT = 14;
constexpr int CH_RING = 4;
// slot map: X k-blocks 0-5 | actor tile 6-9 | weight ring 10-13; the critic tile aliases X 2-5 (free once both first
// layers have read X), the output-layer seeds alias X 0-1.  The ring must hold ~64 KB in flight: one 16 KB stage feeds
// 512 tensor cycles and a refill (commit -> producer -> L2 -> shared memory) takes ~2 k cycles under load.
constexpr int CH_X0 = 0, CH_HA0 = 6, CH_RING0 = 10, CH_HC0 = 2, CH_DZ3A = 0, CH_DZ3C = 1;
// what is left of the 227 KB: barriers, the output layers' constants, running loss sums, bf16 hidden biases
constexpr int kChainMaxAct = 24;
constexpr int CH_RED_W = 2 + kChainMaxAct;
constexpr int CH_MISC_B3 = 192, CH_MISC_CONST = 296, CH_MISC_RED = 488, CH_MISC_BIAS = 1024;
constexpr int CH_MISC = 3072;
constexpr int CH_SMEM = CH_NSLOT * CH_SLOT + CH_MISC;  // = 227 KB, the dynamic shared memory starts 1024-byte aligned (checked)
static_assert(CH_SMEM <= 227 * 1024, "chain kernel shared memory");
static_assert(CH_MISC_B3 + 4 * (kChainMaxAct + 1) <= CH_MISC_CONST && CH_MISC_CONST + 8 * kChainMaxAct <= CH_MISC_RED &&
                  CH_MISC_RED + 16 * CH_RED_W <= CH_MISC_BIAS && CH_MISC_BIAS + 2048 <= CH_MISC,
              "chain kernel misc layout");

__device__ __forceinline__ void ch_bias16(const float* __restrict__ b, float (&o)[16]) {  // warp-uniform address: one L1 wavefront each
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(b) + u);
    o[4 * u] = t.x; o[4 * u + 1] = t.y; o[4 * u + 2] = t.z; o[4 * u + 3] = t.w;
  }
}
// 16 accumulator columns + bias -> activation -> 16 bf16 (8 words)
__device__ __forceinline__ void ch_act16(const uint32_t (&v)[16], const float (&b)[16], int act, uint32_t (&o)[8]) {
  if (act == B200PPO_ACT_TANH) {
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = tanh_bf16x2(pack_bf16(__uint_as_float(v[2 * j]) + b[2 * j], __uint_as_float(v[2 * j + 1]) + b[2 * j + 1]));
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j)
      o[j] = pack_bf16(fmaxf(__uint_as_float(v[2 * j]) + b[2 * j], 0.f), fmaxf(__uint_as_float(v[2 * j + 1]) + b[2 * j + 1], 0.f));
  }
}
__device__ __forceinline__ void ch_lds_bias16(uint32_t saddr, float (&b)[16]) {  // 16 bf16 biases; broadcast reads: every lane the same 32 bytes
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    uint32_t w[4];
    asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(w[0]), "=r"(w[1]), "=r"(w[2]), "=r"(w[3]) : "r"(saddr + 16u * u) : "memory");
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      b[8 * u + 2 * j] = __uint_as_float(w[j] << 16);
      b[8 * u + 2 * j + 1] = __uint_as_float(w[j] & 0xFFFF0000u);
    }
  }
}

// Hidden-layer forward epilogue of this warp's 32 rows x 64 columns: TMEM -> bias (shared memory) + activation -> bf16
// -> the next A operand in shared memory (the caller then bulk-stores the same 4 KB sub-tile to global memory).  TMEM
// loads run one 16-column slab ahead of the math.
__device__ __forceinline__ void ch_epi_forward(uint32_t tcol, uint32_t bias_s, int act, uint32_t srow, uint32_t sw) {
  uint32_t va[16], vb[16], o[8];
  float b[16];
  tmem_ld16_nowait(tcol, va);
  ch_lds_bias16(bias_s, b);
  tmem_ld_wait();
  tmem_ld16_nowait(tcol + 16, vb);
  ch_act16(va, b, act, o); sts_unit_pair(srow, sw, 0, o);
  ch_lds_bias16(bias_s + 32, b);
  tmem_ld_wait();
  tmem_ld16_nowait(tcol + 32, va);
  ch_act16(vb, b, act, o); sts_unit_pair(srow, sw, 1, o);
  ch_lds_bias16(bias_s + 64, b);
  tmem_ld_wait();
  tmem_ld16_nowait(tcol + 48, vb);
  ch_act16(va, b, act, o); sts_unit_pair(srow, sw, 2, o);
  ch_lds_bias16(bias_s + 96, b);
  tmem_ld_wait();
  ch_act16(vb, b, act, o); sts_unit_pair(srow, sw, 3, o);
}

// dgrad epilogue, activation in shared memory (the tile this thread wrote two steps earlier): dZ = acc * act'(h),
// written back IN PLACE — it is the next step's A operand and the source of the bulk store to global memory.
__device__ __forceinline__ void ch_epi_dgrad_smem(uint32_t tcol, int act, uint32_t srow, uint32_t sw) {
  uint32_t va[16], vb[16], h[8], o[8];
  tmem_ld16_nowait(tcol, va);
  lds_unit_pair(srow, sw, 0, h);
  tmem_ld_wait();
  tmem_ld16_nowait(tcol + 16, vb);
  act_grad16(va, h, act, o); sts_unit_pair(srow, sw, 0, o);
  lds_unit_pair(srow, sw, 1, h);
  tmem_ld_wait();
  tmem_ld16_nowait(tcol + 32, va);
  act_grad16(vb, h, act, o); sts_unit_pair(srow, sw, 1, o);
  lds_unit_pair(srow, sw, 2, h);
  tmem_ld_wait();
  tmem_ld16_nowait(tcol + 48, vb);
  act_grad16(va, h, act, o); sts_unit_pair(srow, sw, 2, o);
  lds_unit_pair(srow, sw, 3, h);
  tmem_ld_wait();
  act_grad16(vb, h, act, o); sts_unit_pair(srow, sw, 3, o);
}

// dgrad epilogue of the first hidden layer: its activation was overwritten in shared memory by the second layer's, so
// the row comes back from global memory (an L2 hit), requested by the caller BEFORE the accumulator is awaited.  The
// result is no A operand: it goes straight from registers to global memory, one 32-byte sector per access.
__device__ __forceinline__ void ch_epi_dgrad_glob(uint32_t tcol, int act, const uint32_t (&ax)[4][8], __nv_bfloat16* grow, bool row_ok) {
  uint32_t va[16], vb[16], o[8];
  tmem_ld16_nowait(tcol, va);
  tmem_ld_wait();
  tmem_ld16_nowait(tcol + 16, vb);
  act_grad16(va, ax[0], act, o);
  if (row_ok) stg256(grow, o);
  tmem_ld_wait();
  tmem_ld16_nowait(tcol + 32, va);
  act_grad16(vb, ax[1], act, o);
  if (row_ok) stg256(grow + 16, o);
  tmem_ld_wait();
  tmem_ld16_nowait(tcol + 48, vb);
  act_grad16(va, ax[2], act, o);
  if (row_ok) stg256(grow + 32, o);
  tmem_ld_wait();
  act_grad16(vb, ax[3], act, o);
  if (row_ok) stg256(grow + 48, o);
}

// ... the actor's variant: staged in its (idle) tile so that it leaves through the bulk store
__device__ __forceinline__ void ch_epi_dgrad_stage(uint32_t tcol, int act, const uint32_t (&ax)[4][8], uint32_t srow, uint32_t sw) {
  uint32_t va[16], vb[16], o[8];
  tmem_ld16_nowait(tcol, va);
  tmem_ld_wait();
  tmem_ld16_nowait(tcol + 16, vb);
  act_grad16(va, ax[0], act, o); sts_unit_pair(srow, sw, 0, o);
  tmem_ld_wait();
  tmem_ld16_nowait(tcol + 32, va);
  act_grad16(vb, ax[1], act, o); sts_unit_pair(srow, sw, 1, o);
  tmem_ld_wait();
  tmem_ld16_nowait(tcol + 48, vb);
  act_grad16(va, ax[2], act, o); sts_unit_pair(srow, sw, 2, o);
  tmem_ld_wait();
  act_grad16(vb, ax[3], act, o); sts_unit_pair(srow, sw, 3, o);
}

__device__ __forceinline__ float ldg_f32_now(const float* p) {  // volatile: issued where it is written, not sunk to its use
  float v;
  asm volatile("ld.global.nc.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}

// Sum over the warp's 32 rows of eight per-row values at once: three exchange stages halve the number of values a lane
// carries (8 -> 4 -> 2 -> 1), two plain stages finish; 9 shuffles instead of 40.  Returns the total of column
// ch_red8_col(lane) in every lane.
__device__ __forceinline__ int ch_red8_col(int lane) { return ((lane >> 4) & 1) * 4 + ((lane >> 3) & 1) * 2 + ((lane >> 2) & 1); }
__device__ __forceinline__ float ch_red8(const float (&v)[8], int lane) {
  float w[4], x[2];
  const bool h16 = (lane & 16) != 0, h8 = (lane & 8) != 0, h4 = (lane & 4) != 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float keep = h16 ? v[4 + i] : v[i], send = h16 ? v[i] : v[4 + i];
    w[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
  }
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const float keep = h8 ? w[2 + i] : w[i], send = h8 ? w[i] : w[2 + i];
    x[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
  }
  float y = (h4 ? x[1] : x[0]) + __shfl_xor_sync(0xffffffffu, h4 ? x[0] : x[1], 4);
  y += __shfl_xor_sync(0xffffffffu, y, 2);
  y += __shfl_xor_sync(0xffffffffu, y, 1);
  return y;
}

// ACT: the hidden activation as a compile-time constant, and the two networks of a step pair share ONE copy of every
// epilogue body (loops over the pair not unrolled): the first version carried ~100 KB of code — three times the
// instruction cache — and every step of every tile started with instruction fetches from L2.
//
// Order inside a step pair: actor first in the forward half (steps 0-5), CRITIC first in the backward half (6-9).  The
// critic's tile aliases X k-blocks 2-5: forward, its first epilogue may only write there once BOTH first-layer MMAs have
// read X (so it goes second); backward, the earlier its last MMA (step 8) retires, the earlier the next tile's
// observations can stream in behind the actor's step 9.  The one irregular dependency this creates: step 6 (critic)
// needs the seeds of step 5, not of step 4.
//
// INFER: the rollout's policy evaluation (K6: PPOAgent.act, src/entities/agents/ppo_agent.py:act) as the same pipeline cut
// after step 5 — no dgrad steps, no global copies of the hidden activations; step 4 turns the actor's output row into
// mean, sampled action and its log-probability, step 5 writes the value.
template <int ACT, bool INFER>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(CH_THREADS, 1) tc_chain_kernel(const __grid_constant__ ChainArgs a) {
  constexpr uint32_t TMEM_COLS = 512;
  constexpr int H = kChainHidden;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* misc = smem + CH_NSLOT * CH_SLOT;
  uint64_t* bars = reinterpret_cast<uint64_t*>(misc);
  uint64_t* ring_full = bars;        // [4]  leader: both CTAs' TMA bytes
  uint64_t* ring_empty = bars + 4;   // [4]  commit multicast
  uint64_t* x_full = bars + 8;       // [6]  leader
  uint64_t* x_free = bars + 14;      // [2]  slots 0-1 (after step 7), slots 2-5 (after step 8); commit multicast
  uint64_t* acc_full = bars + 16;    // [2]  commit multicast
  uint64_t* epi_done = bars + 18;    // [2]  leader: 2 x 16 epilogue warps
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 20);
  float* b3_s = reinterpret_cast<float*>(misc + CH_MISC_B3);        // [0,24) actor output bias, [24] critic output bias
  float* consts_s = reinterpret_cast<float*>(misc + CH_MISC_CONST); // [0,24) log sigma, [24,48) 1/var
  float* red_s = reinterpret_cast<float*>(misc + CH_MISC_RED);      // [4][26] running loss sums per TMEM lane quarter

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair_local = int(blockIdx.x) >> 1, pairs = int(gridDim.x) >> 1;
  const int KB1 = a.KB1, tiles2 = a.tiles2;
  const uint32_t smem_base = smem_u32(smem);
  if ((smem_base & 1023u) != 0) __trap();  // the 128-byte swizzle atoms need it; there is no slack left to realign

  if (warp == 0 && lane < 19) {  // the kernel walks nineteen tensor maps: fetch the descriptors before the first copy needs them
    const CUtensorMap* tm = lane == 0 ? &a.x : nullptr;
    if (lane >= 1 && lane < 11) {
      const ChainNet& Np = a.net[(lane - 1) / 5];
      const int w = (lane - 1) % 5;
      tm = w == 0 ? &Np.w1 : (w == 1 ? &Np.w2k : (w == 2 ? &Np.w2m : (w == 3 ? &Np.w3k : &Np.w3m)));
    } else if (lane >= 11) {
      const ChainNet& Np = a.net[(lane - 11) / 4];
      const int w = (lane - 11) % 4;
      tm = w == 0 ? &Np.sH1 : (w == 1 ? &Np.sH2 : (w == 2 ? &Np.sZ1 : &Np.sZ2));
    }
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tm)) : "memory");
  }
  if (warp == 1 && lane == 0) {
    for (int i = 0; i < 18; ++i) mbar_init(&bars[i], 1);
    mbar_init(&epi_done[0], 2 * CH_EPI_WARPS);
    mbar_init(&epi_done[1], 2 * CH_EPI_WARPS);
    mbar_init_fence();
  } else if (warp == 2) {
    tmem_alloc<2, TMEM_COLS>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // The observations of a minibatch were gathered before the epoch began — older than the previous kernel — so the
  // producer may request its first tile's X k-blocks while that kernel (the optimizer) is still draining; the weights it
  // has just re-cast are only touched after the wait (common.cuh, PDL rule 2).
  const bool x_early = a.x_early != 0 && pair_local < tiles2;
  if (warp == 0 && lane == 0 && x_early) {
    const int m0 = pair_local * 256 + int(rank) * 128;
    for (int kb = 0; kb < KB1; ++kb) {
      if (rank == 0) mbar_expect_tx(&x_full[kb], 2u * CH_SLOT);
      tma_load_2d_pair(smem + (CH_X0 + kb) * CH_SLOT, &a.x, mapa_u32(smem_u32(&x_full[kb]), 0), kb * TC_BK, m0);
    }
  }
  pdl_wait_then_release();  // the weights were re-cast by the optimizer kernel right before this one

  if (warp == 0) {
    if (lane == 0) {  // ===== TMA producer =====
      uint32_t rs = 0, rph = 0, cur_bar = 0;  // ring stage and its phase bit
#ifdef B200PPO_CHAIN_RING_TRACE  // per-stage timestamps of the weight ring (build with -DB200PPO_CHAIN_RING_TRACE; off in production:
      uint32_t rn = 0;             // the producer and issuer threads are the latency-critical ones)
#endif
      auto ring_acquire = [&](uint32_t bytes) -> uint8_t* {
        mbar_wait(&ring_empty[rs], rph ^ 1);
#ifdef B200PPO_CHAIN_RING_TRACE
        if (a.trace != nullptr && blockIdx.x == 0 && rn < 64) a.trace[480 + rn * 4 + 0] = clock64();
        ++rn;
#endif
        if (rank == 0) mbar_expect_tx(&ring_full[rs], 2u * bytes);
        cur_bar = mapa_u32(smem_u32(&ring_full[rs]), 0);
        uint8_t* dst = smem + (CH_RING0 + rs) * CH_SLOT;
        if (++rs == CH_RING) { rs = 0; rph ^= 1; }
        return dst;
      };
      int ti = 0;
      for (int tile = pair_local; tile < tiles2; tile += pairs, ++ti) {
        const int m0 = tile * 256 + int(rank) * 128;
        const uint32_t xph = uint32_t(ti & 1);
        for (int o = 0; o < 2; ++o)
          for (int kb = 0; kb < KB1; ++kb) {
            if (o == 0 && !(ti == 0 && x_early)) {
              if (kb == 0) mbar_wait(&x_free[0], xph ^ 1);
              if (kb == 2) mbar_wait(&x_free[1], xph ^ 1);
              if (rank == 0) mbar_expect_tx(&x_full[kb], 2u * CH_SLOT);
              tma_load_2d_pair(smem + (CH_X0 + kb) * CH_SLOT, &a.x, mapa_u32(smem_u32(&x_full[kb]), 0), kb * TC_BK, m0);
            }
            uint8_t* dst = ring_acquire(CH_SLOT);
            tma_load_2d_pair(dst, &a.net[o].w1, cur_bar, kb * TC_BK, int(rank) * 128);
          }
        for (int o = 0; o < 2; ++o)
          for (int kb = 0; kb < H / TC_BK; ++kb) {
            uint8_t* dst = ring_acquire(CH_SLOT);
            tma_load_2d_pair(dst, &a.net[o].w2k, cur_bar, kb * TC_BK, int(rank) * 128);
          }
        {  // output layers, K-major: 16 (actor) / 8 (critic) rows of W3 per CTA, all four k-blocks in one stage
          uint8_t* dst = ring_acquire(4 * 2048);
          for (int kb = 0; kb < 4; ++kb) tma_load_2d_pair(dst + kb * 2048, &a.net[0].w3k, cur_bar, kb * TC_BK, int(rank) * 16);
          dst = ring_acquire(4 * 1024);
          for (int kb = 0; kb < 4; ++kb) tma_load_2d_pair(dst + kb * 1024, &a.net[1].w3k, cur_bar, kb * TC_BK, int(rank) * 8);
        }
        if constexpr (INFER) continue;
        {  // dgrad through the output layers: W3 as [K = out][N = hidden], this CTA's 128 hidden columns as two 64-wide atoms
          uint8_t* dst = ring_acquire(2 * 2048);
          for (int j = 0; j < 2; ++j) tma_load_2d_pair(dst + j * 2048, &a.net[1].w3m, cur_bar, int(rank) * 128 + 64 * j, 0);
          dst = ring_acquire(2 * 4096);
          for (int j = 0; j < 2; ++j) tma_load_2d_pair(dst + j * 4096, &a.net[0].w3m, cur_bar, int(rank) * 128 + 64 * j, 0);
        }
        for (int o = 0; o < 2; ++o)
          for (int kb = 0; kb < H / TC_BK; ++kb) {
            uint8_t* dst = ring_acquire(CH_SLOT);
            for (int j = 0; j < 2; ++j) tma_load_2d_pair(dst + j * 8192, &a.net[1 - o].w2m, cur_bar, int(rank) * 128 + 64 * j, kb * TC_BK);
          }
      }
      // every commit the leader multicast to this CTA has landed before the CTA may exit
      for (int i = 0; i < CH_RING; ++i) {
        mbar_wait(&ring_empty[rs], rph ^ 1);
        if (++rs == CH_RING) { rs = 0; rph ^= 1; }
      }
      if (ti > 0) {
        mbar_wait(&x_free[0], uint32_t((ti - 1) & 1));
        mbar_wait(&x_free[1], uint32_t((ti - 1) & 1));
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && rank == 0) {  // ===== MMA issuer of the pair =====
      constexpr uint32_t ID_N256 = umma_idesc(256, 256, false, false), ID_N256_BMN = umma_idesc(256, 256, false, true);
      constexpr uint32_t ID_N32 = umma_idesc(256, 32, false, false), ID_N16 = umma_idesc(256, 16, false, false);
      uint32_t rs = 0, rph = 0, g = 0;
      auto step_begin = [&]() -> uint32_t {  // the epilogue of step g - 2 has drained this accumulator and written this step's A operand
        mbar_wait(&epi_done[g & 1], ((g >> 1) & 1) ^ 1);
        tc_fence_after();
        if (a.trace != nullptr && blockIdx.x == 0 && g < 60) a.trace[g * 8 + 0] = clock64();
        return tmem_base + (g & 1) * 256u;
      };
      auto step_end = [&]() {
        umma2_commit(&acc_full[g & 1]);
        if (a.trace != nullptr && blockIdx.x == 0 && g < 60) a.trace[g * 8 + 1] = clock64();
        ++g;
      };
#ifdef B200PPO_CHAIN_RING_TRACE
      uint32_t wn = 0;
#endif
      auto ring_wait = [&]() -> uint32_t {
        mbar_wait(&ring_full[rs], rph);
        tc_fence_after();
#ifdef B200PPO_CHAIN_RING_TRACE
        if (a.trace != nullptr && blockIdx.x == 0 && wn < 64) a.trace[480 + wn * 4 + 1] = clock64();
#endif
        return smem_base + (CH_RING0 + rs) * CH_SLOT;
      };
      auto ring_release = [&]() {
        umma2_commit(&ring_empty[rs]);
#ifdef B200PPO_CHAIN_RING_TRACE
        if (a.trace != nullptr && blockIdx.x == 0 && wn < 64) a.trace[480 + wn * 4 + 2] = clock64();
        ++wn;
#endif
        if (++rs == CH_RING) { rs = 0; rph ^= 1; }
      };
      int ti = 0;
      for (int tile = pair_local; tile < tiles2; tile += pairs, ++ti) {
        for (int o = 0; o < 2; ++o) {  // steps 0, 1: first hidden layer (actor, critic)
          const uint32_t d = step_begin();
          for (int kb = 0; kb < KB1; ++kb) {
            if (o == 0) {
              mbar_wait(&x_full[kb], uint32_t(ti & 1));
              tc_fence_after();
            }
            const uint32_t b = ring_wait(), aa = smem_base + (CH_X0 + kb) * CH_SLOT;
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma2_bf16(d, umma_desc(aa + k * 32, 0, 1024), umma_desc(b + k * 32, 0, 1024), ID_N256, (kb > 0 || k > 0) ? 1u : 0u);
            ring_release();
          }
          step_end();
        }
        for (int o = 0; o < 2; ++o) {  // steps 2, 3: second hidden layer
          const uint32_t d = step_begin();
          for (int kb = 0; kb < H / TC_BK; ++kb) {
            const uint32_t b = ring_wait(), aa = smem_base + ((o ? CH_HC0 : CH_HA0) + kb) * CH_SLOT;
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma2_bf16(d, umma_desc(aa + k * 32, 0, 1024), umma_desc(b + k * 32, 0, 1024), ID_N256, (kb > 0 || k > 0) ? 1u : 0u);
            ring_release();
          }
          step_end();
        }
        for (int o = 0; o < 2; ++o) {  // steps 4, 5: output layers (N = 32 actor / 16 critic)
          const uint32_t d = step_begin();
          const uint32_t b = ring_wait();
          for (int kb = 0; kb < H / TC_BK; ++kb) {
            const uint32_t aa = smem_base + ((o ? CH_HC0 : CH_HA0) + kb) * CH_SLOT, bb = b + kb * (o ? 1024 : 2048);
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma2_bf16(d, umma_desc(aa + k * 32, 0, 1024), umma_desc(bb + k * 32, 0, 1024), o ? ID_N16 : ID_N32, (kb > 0 || k > 0) ? 1u : 0u);
          }
          ring_release();
          if (INFER && o == 1) {  // nothing reads the observations or the critic tile after this step
            umma2_commit(&x_free[0]);
            umma2_commit(&x_free[1]);
          }
          step_end();
        }
        if constexpr (INFER) continue;
        for (int o = 0; o < 2; ++o) {  // steps 6, 7: dgrad through the output layers (K = 16 critic / 32 actor)
          const uint32_t d = step_begin();
          if (o == 0) {  // the critic's seeds come from step 5, the previous step (see the note on the order above)
            mbar_wait(&epi_done[1], ((g - 1) >> 1) & 1);
            tc_fence_after();
          }
          const uint32_t b = ring_wait(), aa = smem_base + (o ? CH_DZ3A : CH_DZ3C) * CH_SLOT;
          const int nk = o ? 2 : 1;
          for (int k = 0; k < nk; ++k)
            umma2_bf16(d, umma_desc(aa + k * 32, 0, 1024), umma_desc(b + k * 2048, o ? 4096 : 2048, 1024), ID_N256_BMN, k > 0 ? 1u : 0u);
          ring_release();
          if (o == 1) umma2_commit(&x_free[0]);  // both seed tiles (X slots 0-1) have been read
          step_end();
        }
        for (int o = 0; o < 2; ++o) {  // steps 8, 9: dgrad through the second hidden layer
          const uint32_t d = step_begin();
          for (int kb = 0; kb < H / TC_BK; ++kb) {
            const uint32_t b = ring_wait(), aa = smem_base + ((o ? CH_HA0 : CH_HC0) + kb) * CH_SLOT;
#pragma unroll
            for (int k = 0; k < 4; ++k)
              umma2_bf16(d, umma_desc(aa + k * 32, 0, 1024), umma_desc(b + k * 2048, 8192, 1024), ID_N256_BMN, (kb > 0 || k > 0) ? 1u : 0u);
            ring_release();
          }
          if (o == 0) umma2_commit(&x_free[1]);  // the critic tile (X slots 2-5) has been read: the next observations may land
          step_end();
        }
      }
    }
  } else {  // ===== epilogue warps =====
    const int q = warp & 3, chunk = (warp - 2) >> 2;
    const int r = q * 32 + lane;
    const uint32_t sw = uint32_t(lane & 7);
    constexpr int act = ACT;
    const int A = a.ppo.act_dim;
    {  // constants (written by the optimizer before this kernel: after the PDL wait)
      const int t = threadIdx.x - 64;
      if (t < kChainMaxAct) {
        b3_s[t] = t < A ? __ldg(a.net[0].b3 + t) : 0.f;
        float ls = 0.f, iv = 0.f;
        if (t < A) {
          const float sig = expf(__ldg(a.ppo.logstd + t));
          ls = logf(sig); iv = 1.f / (sig * sig);
        }
        consts_s[t] = ls; consts_s[kChainMaxAct + t] = iv;
      } else if (t == kChainMaxAct) {
        b3_s[kChainMaxAct] = __ldg(a.net[1].b3);
      }
      for (int i = t; i < 4 * CH_RED_W; i += CH_EPI_WARPS * 32) red_s[i] = 0.f;
      // hidden-layer biases as bf16 [net][layer][256]: the kernel leaves next to no L1, so a bias load from global memory
      // would be an L2 round trip in front of every accumulator slab; 2 KB is what is left of shared memory
      __nv_bfloat16* bias_dst = reinterpret_cast<__nv_bfloat16*>(misc + CH_MISC_BIAS);
      for (int i = t; i < 4 * H; i += CH_EPI_WARPS * 32) {
        const int nl = i / H, c = i - nl * H;
        const ChainNet& Nb = a.net[nl >> 1];
        bias_dst[i] = __float2bfloat16_rn(__ldg(((nl & 1) ? Nb.b2 : Nb.b1) + c));
      }
      asm volatile("bar.sync 1, %0;" ::"n"(CH_EPI_WARPS * 32) : "memory");
    }
    const uint32_t bias_chunk_s = smem_base + CH_NSLOT * CH_SLOT + CH_MISC_BIAS + uint32_t(chunk) * 128u;  // + (net * 2 + layer) * 512
    const uint32_t lead_done0 = mapa_u32(smem_u32(&epi_done[0]), 0), lead_done1 = mapa_u32(smem_u32(&epi_done[1]), 0);
    const uint32_t lane_base = tmem_base + (uint32_t(q * 32) << 16);
    // this warp's 32 x 64 sub-tile (4 KB) of the actor / critic tile, and this thread's row in it
    const uint32_t sub_a = smem_base + (CH_HA0 + chunk) * CH_SLOT + uint32_t(q) * 4096u;
    const uint32_t sub_c = smem_base + (CH_HC0 + chunk) * CH_SLOT + uint32_t(q) * 4096u;
    const uint32_t row_a = sub_a + uint32_t(lane) * 128u, row_c = sub_c + uint32_t(lane) * 128u;
    const uint32_t row_z3a = smem_base + CH_DZ3A * CH_SLOT + uint32_t(r) * 128u;
    const uint32_t row_z3c = smem_base + CH_DZ3C * CH_SLOT + uint32_t(r) * 128u;
    float* red_row = red_s + q * CH_RED_W;
    uint32_t g = 0;
    auto tr = [&](int slot) {
      if (a.trace != nullptr && blockIdx.x == 0 && warp == 2 && lane == 0 && g < 60) a.trace[g * 8 + slot] = clock64();
    };
    auto acc_wait = [&]() {
      mbar_wait(&acc_full[g & 1], (g >> 1) & 1);
      tc_fence_after();
      __syncwarp();
      tr(2);
    };
    // End of a step for this warp: its shared-memory writes become visible to the async proxy (the tensor core's
    // operand reads and the bulk store), the issuer learns that this warp has drained the accumulator and written its
    // part of the next A operand, and the sub-tile it wrote leaves for global memory through the copy engine (one
    // elected lane; rows past the batch are clipped by the tensor map).
    auto step_done = [&](const CUtensorMap* store_map, uint32_t sub, int grow0) {
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        // relaxed: a release here is MEMBAR.ALL.GPU in front of every arrive (19 % of the first version's stall samples);
        // the proxy fence above has already completed this warp's shared-memory writes, which is all the issuer's MMAs read
        mbar_arrive_cluster((g & 1) ? lead_done1 : lead_done0);
        if (store_map != nullptr) {
          tma_store_2d(store_map, sub, chunk * 64, grow0);
          bulk_commit();
        }
        if (a.trace != nullptr && blockIdx.x == 0 && g < 60)
          atomicMax(reinterpret_cast<unsigned long long*>(a.trace) + g * 8 + 3, (unsigned long long)clock64());
      }
      tr(6);
      ++g;
    };
    // Bulk stores of a warp, in order: H1a H1c H2a H2c (steps 0-3), dZ2c dZ2a (6, 7), dZ1a (9).  Before a sub-tile is
    // overwritten the store that last read it must have drained it: the youngest one in steps 0, 6 and 9, (at most) the
    // second youngest elsewhere.
    auto stores_drained = [&](bool youngest) {
      if (lane == 0) {
        if (youngest) bulk_wait_read<0>();
        else bulk_wait_read<1>();
      }
      __syncwarp();
    };
    // H1 of a network comes back from global memory for the last dgrad step: its bulk store (three / five groups back
    // where the critic's / the actor's rows are requested) must be complete, not merely read
    auto h1_visible = [&](bool critic) {
      if (lane == 0) {
        // (completion of a bulk group makes its writes visible to the waiting thread; __syncwarp orders the other lanes'
        // loads after it.  A fence.proxy.async.global here was measured at ~4 k cycles per use.)
        if (critic) bulk_wait<3>();
        else bulk_wait<5>();
      }
      __syncwarp();
    };
    uint32_t ax[4][8];  // this thread's 64 H1 values of the next dgrad step, requested one step ahead
    for (int tile = pair_local; tile < tiles2; tile += pairs) {
      const int grow0 = tile * 256 + int(rank) * 128 + q * 32;  // first global row of this warp's sub-tile
      const int64_t m = int64_t(grow0) + lane;
      const bool row_ok = m < a.M;
      const int64_t mm = row_ok ? m : 0;
      float av[8], old_lp = 0.f, adv = 0.f, tgt = 0.f;  // loss operands of this row, requested two steps ahead
#pragma unroll 1
      for (int layer = 0; layer < 2; ++layer) {
#pragma unroll 1
        for (int o = 0; o < 2; ++o) {  // steps 0-3: hidden layers forward (actor, critic)
          const ChainNet& N = a.net[o];
          if (INFER) {
            // (the noise row is read in step 4 by the one warp per lane quarter that finishes the actor's outputs)
          } else if (layer == 1) {  // the loss operands of this row: requested now (volatile: not to be sunk to their use), needed in steps 4 / 5
            if (o == 0) {
              const float* ap = a.ppo.action + mm * A + chunk * 8;
#pragma unroll
              for (int i = 0; i < 8; ++i) av[i] = (row_ok && chunk * 8 + i < A) ? ldg_f32_now(ap + i) : 0.f;
              if (row_ok) { old_lp = ldg_f32_now(a.ppo.old_logp + mm); adv = ldg_f32_now(a.ppo.advantage + mm); }
            } else if (chunk == 0 && row_ok) {
              tgt = ldg_f32_now(a.ppo.target + mm);
            }
          }
          acc_wait();
          stores_drained(layer == 0 && o == 0);
          tr(4);
          ch_epi_forward(lane_base + uint32_t(o) * 256u + uint32_t(chunk * 64), bias_chunk_s + uint32_t(o * 2 + layer) * 512u, act,
                         o ? row_c : row_a, sw);
          tr(5);
          step_done(INFER ? nullptr : (layer ? &N.sH2 : &N.sH1), o ? sub_c : sub_a, grow0);
        }
      }
      if constexpr (INFER) {
        {  // step 4: the actor's output row -> mean, action = mean + sigma * noise, log-prob of that action (one warp per lane quarter)
          acc_wait();
          if (chunk == 0) {
            const float scale = a.out_scale;
            const bool ft = a.ppo.final_tanh != 0;
            float lp = 0.f;
#pragma unroll 1
            for (int j0 = 0; j0 < A; j0 += 8) {
              uint32_t v[8];
              tmem_ld8(lane_base + uint32_t(j0), v);
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const int j = j0 + i;
                if (j < A && row_ok) {
                  const float pre = __uint_as_float(v[i]) + b3_s[j];
                  const float mean = ft ? scale * tanhf(pre) : pre;
                  const float nz = a.inf_noise != nullptr ? __ldg(a.inf_noise + mm * A + j) : 0.f;
                  if (a.inf_mean != nullptr) a.inf_mean[mm * A + j] = mean;
                  if (a.inf_action != nullptr) a.inf_action[mm * a.inf_ld_action + j] = mean + expf(consts_s[j]) * nz;
                  lp += -0.5f * nz * nz - consts_s[j] - kTcLogSqrt2Pi;
                }
              }
            }
            if (row_ok && a.inf_logp != nullptr) a.inf_logp[mm * a.inf_ld_logp] = lp;
          }
          step_done(nullptr, 0, 0);
        }
        {  // step 5: the critic's value
          acc_wait();
          if (chunk == 0) {
            uint32_t v[8];
            tmem_ld8(lane_base + 256u, v);
            if (row_ok) {
              const float val = __uint_as_float(v[0]) + b3_s[kChainMaxAct];
              if (a.inf_value != nullptr) a.inf_value[mm * a.inf_ld_value] = val;
              if (a.inf_value2 != nullptr) a.inf_value2[mm * a.inf_ld_value] = val;
            }
          }
          step_done(nullptr, 0, 0);
        }
        continue;
      }
      {  // step 4: actor output layer + loss.  A row's columns are split over the four warps of its TMEM lane quarter
        // (8 action columns each): partial log-probs meet in a 16-byte unit of the seed tile's row that the seeds do
        // not use, then every warp finishes its own columns' seeds — one 16-byte unit of the K-major seed tile each.
        const int j0 = chunk * 8;
        acc_wait();
        const float scale = a.out_scale;
        const bool ft = a.ppo.final_tanh != 0;
        float d[8], th[8];
        float lp = 0.f;
        if (j0 < A) {  // warp-uniform
          uint32_t v[8];
          tmem_ld8(lane_base + uint32_t(j0), v);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int j = j0 + i;
            d[i] = 0.f; th[i] = 0.f;
            if (j < A) {
              const float pre = __uint_as_float(v[i]) + b3_s[j];
              th[i] = ft ? tanh_fast(pre) : pre;
              const float mean = ft ? scale * th[i] : pre;
              d[i] = av[i] - mean;
              lp += -(d[i] * d[i]) * (0.5f * consts_s[kChainMaxAct + j]) - consts_s[j] - kTcLogSqrt2Pi;
            }
          }
        }
        const uint32_t lp_unit = row_z3a + ((4u ^ sw) << 4);
        tr(4);
        asm volatile("st.shared.f32 [%0], %1;" ::"r"(lp_unit + uint32_t(chunk) * 4u), "f"(lp) : "memory");
        asm volatile("bar.sync %0, 128;" ::"r"(2 + q) : "memory");  // the four warps of this lane quarter
        tr(5);
        float l0, l1, l2, l3;
        asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(l0), "=f"(l1), "=f"(l2), "=f"(l3) : "r"(lp_unit) : "memory");
        const float lp_row = ((l0 + l1) + l2) + l3;  // same order in all four warps
        float g_lp = 0.f, surr = 0.f;
        if (row_ok) {
          const float lo = 1.f - a.ppo.clip_eps, hi = 1.f + a.ppo.clip_eps;
          const float ratio = expf(lp_row - old_lp);
          const float s1 = ratio * adv, s2 = fminf(fmaxf(ratio, lo), hi) * adv;
          const float w1 = s1 < s2 ? 1.f : (s1 > s2 ? 0.f : 0.5f);
          const float in_range = (ratio >= lo && ratio <= hi) ? 1.f : 0.f;
          g_lp = -(w1 * adv + (1.f - w1) * adv * in_range) * a.ppo.inv_global_batch * ratio;
          surr = fminf(s1, s2);
        }
        uint32_t pk[4];
#pragma unroll
        for (int i = 0; i < 8; i += 2) {
          float dm[2];
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const int j = j0 + i + u;
            dm[u] = 0.f;
            if (j < A) {
              const float dn = d[i + u] * consts_s[kChainMaxAct + j];
              float dmu = g_lp * dn;
              if (ft) dmu *= scale * (1.f - th[i + u] * th[i + u]);
              dm[u] = dmu;                              // g_lp = 0 for rows past the batch
              d[i + u] = g_lp * (d[i + u] * dn - 1.f);  // this row's d loss / d logstd_j
            }
          }
          pk[i >> 1] = pack_bf16(dm[0], dm[1]);
        }
        asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(row_z3a + ((uint32_t(chunk) ^ sw) << 4)), "r"(pk[0]), "r"(pk[1]), "r"(pk[2]), "r"(pk[3]) : "memory");
        if (row_ok && j0 < a.net[0].pZ3)
          *reinterpret_cast<uint4*>(a.net[0].dZ3 + mm * a.net[0].pZ3 + j0) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        tr(7);
        if (j0 < A) {  // warp-uniform
          const float tot = ch_red8(d, lane);
          const int col = j0 + ch_red8_col(lane);
          if ((lane & 3) == 0 && col < A) red_row[2 + col] += tot;
        }
        if (chunk == 0) {
          const float ssum = warp_sum(surr);
          if (lane == 0) red_row[0] += ssum;
        }
        step_done(nullptr, 0, 0);
      }
      {  // step 5: critic output + Huber loss (one value per row: the chunk-0 warps; the others only keep step)
        acc_wait();
        if (chunk == 0) {
          uint32_t v[8];
          tmem_ld8(lane_base + 256u, v);
          float dv = 0.f, hub = 0.f;
          if (row_ok) {
            const float e = __uint_as_float(v[0]) + b3_s[kChainMaxAct] - tgt;
            const float ae = fabsf(e);
            hub = ae < 1.f ? 0.5f * e * e : ae - 0.5f;
            dv = fminf(fmaxf(e, -1.f), 1.f) * a.ppo.inv_global_batch;
          }
          const uint32_t w0 = pack_bf16(dv, 0.f);
          asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(row_z3c + ((0u ^ sw) << 4)), "r"(w0), "r"(0u), "r"(0u), "r"(0u) : "memory");
          asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(row_z3c + ((1u ^ sw) << 4)), "r"(0u), "r"(0u), "r"(0u), "r"(0u) : "memory");
          if (row_ok) {
            const int pitch = a.net[1].pZ3;
            uint4* gp = reinterpret_cast<uint4*>(a.net[1].dZ3 + mm * pitch);
            gp[0] = make_uint4(w0, 0u, 0u, 0u);
            for (int c = 1; 8 * c < pitch; ++c) gp[c] = make_uint4(0u, 0u, 0u, 0u);
          }
          const float hs = warp_sum(hub);
          if (lane == 0) red_row[1] += hs;
        }
        step_done(nullptr, 0, 0);
      }
#pragma unroll 1
      for (int o = 0; o < 2; ++o) {  // steps 6, 7: dgrad through the output layer, activation derivative from the tile in shared memory
        const ChainNet& N = a.net[1 - o];
        acc_wait();
        stores_drained(o == 0);
        tr(4);
        ch_epi_dgrad_smem(lane_base + uint32_t(o) * 256u + uint32_t(chunk * 64), act, o ? row_a : row_c, sw);
        tr(5);
        step_done(&N.sZ2, o ? sub_a : sub_c, grow0);
        if (o == 0) {  // the critic's H1 row for step 8: in flight behind the actor's step 7
          h1_visible(true);
          const __nv_bfloat16* hrow = a.net[1].H1 + mm * a.net[1].pH1 + chunk * 64;
#pragma unroll
          for (int s4 = 0; s4 < 4; ++s4) ldg256_na(hrow + s4 * 16, ax[s4]);
        }
      }
      {  // step 8: critic dgrad through the second hidden layer; the result only feeds the weight-gradient kernel and its
        // tile (X slots 2-5) is about to take the next observations: straight from registers to global memory
        acc_wait();
        tr(4);
        ch_epi_dgrad_glob(lane_base + uint32_t(chunk * 64), act, ax, a.net[1].dZ1 + mm * a.net[1].pZ1 + chunk * 64, row_ok);
        tr(5);
        step_done(nullptr, 0, 0);
        h1_visible(false);  // the actor's H1 row for step 9
        const __nv_bfloat16* hrow = a.net[0].H1 + mm * a.net[0].pH1 + chunk * 64;
#pragma unroll
        for (int s4 = 0; s4 < 4; ++s4) ldg256_na(hrow + s4 * 16, ax[s4]);
      }
      {  // step 9: actor dgrad through the second hidden layer, staged in the (now idle) actor tile for the bulk store
        acc_wait();
        stores_drained(true);
        tr(4);
        ch_epi_dgrad_stage(lane_base + 256u + uint32_t(chunk * 64), act, ax, row_a, sw);
        tr(5);
        step_done(&a.net[0].sZ1, sub_a, grow0);
      }
    }
    if (lane == 0) bulk_wait<0>();
    // this CTA's row of loss partials: (sum surrogate, sum huber, sum d loss / d logstd_j)
    asm volatile("bar.sync 1, %0;" ::"n"(CH_EPI_WARPS * 32) : "memory");
    const int t = threadIdx.x - 64;
    if (!INFER && t < 2 + A)
      a.ppo.partials[int64_t(blockIdx.x) * (2 + A) + t] = red_s[t] + red_s[CH_RED_W + t] + red_s[2 * CH_RED_W + t] + red_s[3 * CH_RED_W + t];
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // the peer may still be reading this CTA's operands / arriving on its barriers
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<2, TMEM_COLS>(tmem_base);
  }
}

long long* g_chain_trace = nullptr;

bool tc_chain_shape_ok(int in_dim, int h1, int h2, int out_dim) {
  return in_dim >= 1 && in_dim <= kChainMaxIn && h1 == kChainHidden && h2 == kChainHidden && out_dim >= 1 && out_dim <= kChainMaxAct;
}

int launch_tc_chain(const ChainArgs& a, cudaStream_t st, int* grid_out, bool infer) {
  B2_CHECK_ARG(a.M > 0 && a.KB1 >= 1 && a.KB1 <= 6 && a.tiles2 == (a.M + 255) / 256, "chain kernel: bad shape");
  static bool configured = false;
  if (!configured) {
    B2_CUDA(cudaFuncSetAttribute(tc_chain_kernel<B200PPO_ACT_TANH, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, CH_SMEM));
    B2_CUDA(cudaFuncSetAttribute(tc_chain_kernel<B200PPO_ACT_RELU, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, CH_SMEM));
    B2_CUDA(cudaFuncSetAttribute(tc_chain_kernel<B200PPO_ACT_TANH, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, CH_SMEM));
    B2_CUDA(cudaFuncSetAttribute(tc_chain_kernel<B200PPO_ACT_RELU, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, CH_SMEM));
    configured = true;
  }
  const int pairs = std::min(num_sms() / 2, a.tiles2);
  if (grid_out) *grid_out = 2 * pairs;
  void (*kernel)(ChainArgs);
  if (infer) kernel = a.act == B200PPO_ACT_TANH ? tc_chain_kernel<B200PPO_ACT_TANH, true> : tc_chain_kernel<B200PPO_ACT_RELU, true>;
  else kernel = a.act == B200PPO_ACT_TANH ? tc_chain_kernel<B200PPO_ACT_TANH, false> : tc_chain_kernel<B200PPO_ACT_RELU, false>;
  // profiling aid: B200PPO_CHAIN_TRACE=<n> prints the clock64 timeline of pair 0 of the n-th launch (cycles since its
  // first step): when the issuer got its operands, when it had issued the step, when the epilogue saw the accumulator
  // and when the slowest epilogue warp of the leader was done with it
  static const char* trace_env = getenv("B200PPO_CHAIN_TRACE");
  static int calls = 0;
  if (trace_env != nullptr && !infer && ++calls == atoi(trace_env)) {
    long long* tr = nullptr;
    B2_CUDA(cudaMalloc(&tr, (60 * 8 + 64 * 4) * sizeof(long long)));
    B2_CUDA(cudaMemset(tr, 0, (60 * 8 + 64 * 4) * sizeof(long long)));
    ChainArgs b = a;
    b.trace = tr;
    B2_CUDA(launch_pdl(kernel, dim3(2 * pairs), dim3(CH_THREADS), CH_SMEM, st, b));
    B2_LAUNCH_CHECK();
    B2_CUDA(cudaStreamSynchronize(st));
    long long h[60 * 8 + 64 * 4];
    B2_CUDA(cudaMemcpy(h, tr, sizeof(h), cudaMemcpyDeviceToHost));
    cudaFree(tr);
    static const char* names[10] = {"L1a", "L1c", "L2a", "L2c", "L3a", "L3c", "D3c", "D3a", "D2c", "D2a"};
    fprintf(stderr, "chain kernel, pair 0 (M = %d, %d pairs): step | operands ready, issued | accumulator seen, epilogue done\n", a.M, pairs);
    for (int g = 0; g < 60 && h[g * 8] != 0; ++g)
      fprintf(stderr, "  %2d %s | %7lld %7lld | %7lld %7lld | warp 2: body %lld..%lld end %lld (%lld)\n", g, names[g % 10], h[g * 8] - h[0],
              h[g * 8 + 1] - h[0], h[g * 8 + 2] - h[0], h[g * 8 + 3] - h[0], h[g * 8 + 4] ? h[g * 8 + 4] - h[0] : 0,
              h[g * 8 + 5] ? h[g * 8 + 5] - h[0] : 0, h[g * 8 + 6] ? h[g * 8 + 6] - h[0] : 0, h[g * 8 + 7] ? h[g * 8 + 7] - h[0] : 0);
#ifdef B200PPO_CHAIN_RING_TRACE
    fprintf(stderr, "weight ring of CTA 0, stage n: producer saw it empty | issuer saw it full, committed its MMAs  (-> refill = full[n] - empty[n]; turn-around = empty[n + %d] - committed[n])\n", CH_RING);
    for (int n = 0; n < 64 && h[480 + n * 4 + 1] != 0; ++n)
      fprintf(stderr, "  %2d | %7lld | %7lld %7lld | refill %5lld  turn-around %5lld\n", n, h[480 + n * 4] - h[0], h[480 + n * 4 + 1] - h[0],
              h[480 + n * 4 + 2] - h[0], h[480 + n * 4 + 1] - h[480 + n * 4],
              (n + CH_RING < 64 && h[480 + (n + CH_RING) * 4] != 0) ? h[480 + (n + CH_RING) * 4] - h[480 + n * 4 + 2] : 0);
#endif
    return B200PPO_OK;
  }
  B2_CUDA(launch_pdl(kernel, dim3(2 * pairs), dim3(CH_THREADS), CH_SMEM, st, a));
  B2_LAUNCH_CHECK();
  return B200PPO_OK;
}

}  // namespace b200ppo
