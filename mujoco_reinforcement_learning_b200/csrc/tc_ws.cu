// Persistent, weights-stationary tcgen05 GEMM for the forward and dgrad passes of the MLP (large minibatches).
//
// C[M, N] = A[M, K] * W[N, K]^T with M = minibatch rows (tens of thousands), N <= 256, K <= 384: the weight matrix
// is a few hundred KB at most, the activations are what streams.  The tile-per-CTA kernel (tc_gemm.cu) re-reads the
// weight tile for every 128 rows, which makes it L2->SM bandwidth bound (64 FLOP per byte staged).  Here a CTA
// loads its problem's whole W into shared memory ONCE (TMA, 128-byte swizzle, K-major), then walks over its share
// of the 128-row tiles: only A moves (4x the arithmetic intensity), the accumulator is double-buffered in TMEM
// (2 x BN columns) so the epilogue of tile t overlaps the MMAs of tile t+1.
//   warp 0      TMA producer: W once, then the A k-blocks of every tile through an n-stage mbarrier ring
//   warp 1      MMA issuer (one lane): tcgen05.mma M=128, N=BN, K=16, commit -> frees the A stage / publishes the tile
//   warps 2-9   epilogue (shared with tc_gemm.cu): tcgen05.ld, bias + MUFU tanh | act' multiply, bf16/fp32 stores
#include <algorithm>

#include "tc_common.cuh"

namespace b200ppo {

constexpr int kWsMaxSlots = 4;

// A slot = (problem, N tile): its CTAs keep that BN-wide slice of the problem's W in shared memory.
struct WsGroup {
  TcProblem p[2];
  int count;
  int n_slots;
  int slot_prob[kWsMaxSlots], slot_n0[kWsMaxSlots];
  int cta_begin[kWsMaxSlots + 1];  // CTAs [cta_begin[i], cta_begin[i+1]) serve slot i
  CUtensorMap tm_out[2];           // per problem: bf16 output as 64-column x 32-row swizzled boxes (bulk-store epilogue)
  int tma_out[2];                  // the problem's epilogue leaves through tm_out
  int stage_tiles;                 // 4 KB staging tiles per epilogue warp (2, or 3 when a dgrad's weights leave room)
  int w_early;                     // the stationary weights were written >= 2 kernels back: load them before the PDL wait
};

template <int BN>
__global__ void __launch_bounds__(TC_THREADS, 1) tc_ws_kernel(const __grid_constant__ WsGroup grp, int a_stages) {
  constexpr uint32_t TMEM_COLS = 2 * BN <= 32 ? 32 : (2 * BN <= 64 ? 64 : (2 * BN <= 128 ? 128 : (2 * BN <= 256 ? 256 : 512)));
  constexpr int W_KB_BYTES = BN * TC_BK * 2;  // one 64-wide k-block of W
  extern __shared__ uint8_t smem_raw[];
  // pointer + offset (not an integer round trip): the compiler keeps the shared address space and emits LDS / STS
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int slot = 0;
#pragma unroll 1
  for (int i = 1; i < grp.n_slots; ++i)
    if (int(blockIdx.x) >= grp.cta_begin[i]) slot = i;
  const TcProblem& P = grp.p[grp.slot_prob[slot]];
  const int n0 = grp.slot_n0[slot];
  const int cta_local = int(blockIdx.x) - grp.cta_begin[slot];
  const int ctas = grp.cta_begin[slot + 1] - grp.cta_begin[slot];
  const int KB = (P.K + TC_BK - 1) / TC_BK;
  const int tiles_m = P.tiles_m;

  uint8_t* sW = smem;
  uint8_t* sA = smem + size_t(KB) * W_KB_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sA + size_t(a_stages) * TC_A_BYTES);
  uint64_t* w_full = bars;
  uint64_t* a_full = bars + 1;
  uint64_t* a_empty = a_full + a_stages;
  uint64_t* acc_full = a_empty + a_stages;
  uint64_t* acc_empty = acc_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
  float* bias_s = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + 512);  // BN floats (<= 256)
  float* consts_s = bias_s + 256;                                                    // 96 floats (fused PPO epilogue)
  float* red_s = bias_s + 352;                                                       // 8 x 34 floats
  uint8_t* stage_area = reinterpret_cast<uint8_t*>(bars) + 4096;  // TC_EPI_WARPS x stage_tiles x 4 KB, 1024-byte aligned (swizzle atoms)

  if (warp == 1 && lane == 0) {
    mbar_init(w_full, 1);
    for (int s = 0; s < a_stages; ++s) { mbar_init(&a_full[s], 1); mbar_init(&a_empty[s], 1); }
    // fused PPO epilogue: the two warp groups alternate tiles, so only four warps release an accumulator
    const uint32_t releasers = P.epilogue >= TC_EPI_PPO_ACTOR ? TC_EPI_WARPS / 2 : TC_EPI_WARPS;
    for (int b = 0; b < 2; ++b) { mbar_init(&acc_full[b], 1); mbar_init(&acc_empty[b], releasers); }
    mbar_init_fence();
  } else if (warp == 2) {
    tmem_alloc<1, TMEM_COLS>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  auto load_w = [&]() {
    mbar_expect_tx(w_full, uint32_t(KB) * W_KB_BYTES);
    if (!P.b_mn_major) {
      for (int kb = 0; kb < KB; ++kb) tma_load_2d(sW + size_t(kb) * W_KB_BYTES, &P.tmB, w_full, kb * TC_BK, n0);
    } else {  // W given as [K][N] (the dgrad reads nn.Linear's [out, in] weight as is): 64-wide N atoms per k-block
      for (int kb = 0; kb < KB; ++kb)
#pragma unroll
        for (int j = 0; j < BN / 64; ++j)
          tma_load_2d(sW + size_t(kb) * W_KB_BYTES + j * 64 * TC_BK * 2, &P.tmB, w_full, n0 + 64 * j, kb * TC_BK);
    }
  };
  if (warp == 0 && lane == 0 && grp.w_early) load_w();  // overlaps the tail of the previous kernel (see common.cuh, PDL)
  pdl_wait_then_release();
  if (warp >= 2) {  // epilogue warps stage their constants (named barrier 1: the other two warps are already streaming)
    tc_stage_bias(P, n0, BN, bias_s, threadIdx.x - 64, TC_THREADS - 64);
    tc_ppo_stage_consts(P, consts_s, threadIdx.x - 64);
    asm volatile("bar.sync 1, %0;" ::"n"(TC_THREADS - 64) : "memory");
  }

  if (warp == 0) {
    if (lane == 0) {  // ===== TMA producer =====
      if (!grp.w_early) load_w();
      int it = 0;
      for (int tile = cta_local; tile < tiles_m; tile += ctas) {
        for (int kb = 0; kb < KB; ++kb, ++it) {
          const int s = it % a_stages;
          const uint32_t ph = (it / a_stages) & 1;
          mbar_wait(&a_empty[s], ph ^ 1);
          mbar_expect_tx(&a_full[s], TC_A_BYTES);
          tma_load_2d(sA + size_t(s) * TC_A_BYTES, &P.tmA, &a_full[s], kb * TC_BK, tile * TC_BM);
        }
      }
    }
  } else if (warp == 1) {  // ===== MMA issuer: ONE thread runs the whole loop (31 idle lanes would only add polling) =====
    if (lane == 0) {
      const uint32_t idesc = umma_idesc(TC_BM, BN, false, P.b_mn_major != 0);
      const uint32_t b_lbo = P.b_mn_major ? TC_BK * 128 : 0, b_kstep = P.b_mn_major ? 2048 : 32;
      mbar_wait(w_full, 0);
      int it = 0, t = 0;
      for (int tile = cta_local; tile < tiles_m; tile += ctas, ++t) {
        const int buf = t & 1;
        mbar_wait(&acc_empty[buf], ((t >> 1) & 1) ^ 1);  // epilogue has drained this accumulator
        tc_fence_after();
        for (int kb = 0; kb < KB; ++kb, ++it) {
          const int s = it % a_stages;
          const uint32_t ph = (it / a_stages) & 1;
          mbar_wait(&a_full[s], ph);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(sA + size_t(s) * TC_A_BYTES), b_addr = smem_u32(sW + size_t(kb) * W_KB_BYTES);
#pragma unroll
          for (int k = 0; k < TC_BK / 16; ++k)
            umma_bf16(tmem_base + uint32_t(buf * BN), umma_desc(a_addr + k * 32, 0, 1024), umma_desc(b_addr + k * b_kstep, b_lbo, 1024),
                      idesc, (kb > 0 || k > 0) ? 1u : 0u);
          umma_commit(&a_empty[s]);
          if (kb == KB - 1) umma_commit(&acc_full[buf]);
        }
      }
    }
  } else {  // ===== epilogue warps =====
    int t = 0;
    if constexpr (BN <= 128) {
      // two staging tiles per warp: while tile t is finished and stored from one, the dgrad's activation slab of tile
      // t + ctas is already streaming into the other (cp.async), i.e. behind the MMAs of the next tile
      uint8_t* st[2] = {stage_area + (warp - 2) * grp.stage_tiles * TC_STAGE_BYTES, stage_area + (warp - 2) * grp.stage_tiles * TC_STAGE_BYTES + TC_STAGE_BYTES};
      if (P.epilogue >= TC_EPI_PPO_ACTOR) {  // output layers with the PPO loss fused in
        // warp group g (warps 2-5 / 6-9) takes the tiles t with t % 2 == g: tile t lives in TMEM buffer t % 2, so each
        // group always drains the same accumulator while the other group works on the next tile.
        PpoAcc acc;
        acc.clear();
        const int grp_id = (warp - 2) >> 2;
        const int step = 2 * ctas;
        int tile = cta_local + grp_id * ctas, u = 0;  // u counts this group's tiles
        tc_ppo_issue(P, tile * TC_BM, warp, lane, st[0], tile < tiles_m);
        for (; tile < tiles_m; tile += step, ++u) {
          const int next = tile + step;
          tc_ppo_issue(P, next * TC_BM, warp, lane, st[(u & 1) ^ 1], next < tiles_m);
          tc_epilogue_ppo<BN>(P, tmem_base + uint32_t(grp_id * BN), tile * TC_BM, warp, lane, &acc_full[grp_id], uint32_t(u & 1),
                              st[u & 1], bias_s, consts_s, 1, acc, true);
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&acc_empty[grp_id]);
        }
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        tc_ppo_finish(P, warp, lane, red_s, acc, true);
      } else {
      const int pidx = grp.slot_prob[slot];
      const bool tma_out = BN == 128 && grp.tma_out[pidx] != 0;
      const CUtensorMap* tm_out = &grp.tm_out[pidx];
      const int ntiles = grp.stage_tiles;
      uint8_t* st_base = stage_area + (warp - 2) * ntiles * TC_STAGE_BYTES;
      if (P.staged) tc_issue_aux<BN>(P, cta_local * TC_BM, n0, warp, lane, st_base, cta_local < tiles_m);
      int cur_i = 0;  // t % ntiles
      for (int tile = cta_local; tile < tiles_m; tile += ctas, ++t) {
        const int buf = t & 1;
        if (P.staged) {
          const int next = tile + ctas;
          const int nxt_i = cur_i + 1 == ntiles ? 0 : cur_i + 1;
          uint8_t* cur = st_base + cur_i * TC_STAGE_BYTES;
          uint8_t* nxt = st_base + nxt_i * TC_STAGE_BYTES;
          if (tma_out) {
            // tile `cur` was last read by the bulk store of row tile t - ntiles, `nxt` by that of t + 1 - ntiles
            if (lane == 0) {
              if (ntiles == 1 || (ntiles == 2 && P.epilogue == TC_EPI_DGRAD)) bulk_wait_read<0>();
              else bulk_wait_read<1>();
            }
            __syncwarp();
          }
          tc_issue_aux<BN>(P, next * TC_BM, n0, warp, lane, nxt, next < tiles_m);
          if (tma_out)
            tc_epilogue_staged<BN, BN == 128>(P, 0, tmem_base + uint32_t(buf * BN), true, tile * TC_BM, n0, warp, lane, &acc_full[buf],
                                              uint32_t((t >> 1) & 1), cur, bias_s, 1, tm_out);
          else
            tc_epilogue_staged<BN>(P, 0, tmem_base + uint32_t(buf * BN), true, tile * TC_BM, n0, warp, lane, &acc_full[buf],
                                   uint32_t((t >> 1) & 1), cur, bias_s, 1);
          cur_i = nxt_i;
        } else {
          tc_epilogue<BN>(P, 0, tmem_base + uint32_t(buf * BN), true, tile * TC_BM, n0, warp, lane, &acc_full[buf], uint32_t((t >> 1) & 1), bias_s);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_empty[buf]);
      }
      if (tma_out && lane == 0) bulk_wait<0>();
      asm volatile("cp.async.wait_group 0;" ::: "memory");
      }
    } else {
      for (int tile = cta_local; tile < tiles_m; tile += ctas, ++t) {
        const int buf = t & 1;
        tc_epilogue<BN>(P, 0, tmem_base + uint32_t(buf * BN), true, tile * TC_BM, n0, warp, lane, &acc_full[buf], uint32_t((t >> 1) & 1), bias_s);
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(&acc_empty[buf]);
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

// ---- CTA-pair variant (cta_group::2) for wide forward layers ------------------------------------------------------------
// Measured with profiles/mma_probe.cu: a cta_group::1 MMA with N = 128 re-reads 8 KB of shared memory per 64 tensor
// cycles and tops out at 60% of the pipe before any epilogue or TMA traffic; N = 256 reaches 96-99%.  A 256-wide slice
// of W (K = 384: 192 KB) does not fit one SM next to the A ring, so two CTAs of a cluster pair up: each keeps HALF of
// the slice (128 rows, the same shared-memory layout as the single-CTA kernel) and its own 128 activation rows; the
// leader issues tcgen05.mma.cta_group::2 with M = 256, N = 256 and every CTA ends up with a 128 x 256 accumulator
// in its own TMEM (2 x 256 columns, double-buffered).  Per CTA and k-step that is 4 KB of A + 4 KB of B for 128
// tensor cycles: half the shared-memory traffic per FLOP, and the activation tile is read once per 256 output columns.
//   warp 0 (both CTAs)  TMA: own half of W once, own A rows per k-block; completion goes to the LEADER's mbarriers
//   warp 1 (leader)     MMA issuer; tcgen05.commit multicast frees the stage in both CTAs / publishes the accumulator
//   warps 2-9 (both)    epilogue on the CTA's own 128 rows: two 64-column chunks per warp, bulk-stored from staging
constexpr int WS2_EPI_WARPS = 16;  // four per TMEM lane quarter, one 64-column chunk each: MUFU.TANH (16/clk/SM) is the epilogue's
                                   // floor, and two lock-stepped warps per scheduler left it half idle
constexpr int WS2_THREADS = (2 + WS2_EPI_WARPS) * 32;
constexpr int WS2_MAX_KB = 8;

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(WS2_THREADS, 1) tc_ws2_kernel(const __grid_constant__ WsGroup grp, int a_stages) {
  constexpr int BN = 256, BNL = 128;
  constexpr uint32_t TMEM_COLS = 512;
  constexpr int W_KB_BYTES = BNL * TC_BK * 2;
  extern __shared__ uint8_t smem_raw[];
  // pointer + offset (not an integer round trip): the compiler keeps the shared address space and emits LDS / STS
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  int slot = 0;
#pragma unroll 1
  for (int i = 1; i < grp.n_slots; ++i)
    if (int(blockIdx.x) >= grp.cta_begin[i]) slot = i;
  const int pidx = grp.slot_prob[slot];
  const TcProblem& P = grp.p[pidx];
  const int n0 = grp.slot_n0[slot];
  const int pair_local = (int(blockIdx.x) - grp.cta_begin[slot]) >> 1;
  const int pairs = (grp.cta_begin[slot + 1] - grp.cta_begin[slot]) >> 1;
  const int KB = (P.K + TC_BK - 1) / TC_BK;
  const int tiles2 = (P.M + 2 * TC_BM - 1) / (2 * TC_BM);  // 256-row tiles of the pair

  uint8_t* sW = smem;
  uint8_t* sA = smem + size_t(KB) * W_KB_BYTES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sA + size_t(a_stages) * TC_A_BYTES);
  uint64_t* w_full = bars;  // one per k-block of W: the first MMAs start as soon as the first 2 x 16 KB have landed
  uint64_t* a_full = bars + WS2_MAX_KB;
  uint64_t* a_empty = a_full + a_stages;
  uint64_t* acc_full = a_empty + a_stages;
  uint64_t* acc_empty = acc_full + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(acc_empty + 2);
  float* bias_s = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(bars) + 512);  // 256 floats
  uint8_t* stage_area = reinterpret_cast<uint8_t*>(bars) + 4096;

  if (warp == 1 && lane == 0) {
    for (int kb = 0; kb < KB; ++kb) mbar_init(&w_full[kb], 1);
    for (int s = 0; s < a_stages; ++s) { mbar_init(&a_full[s], 1); mbar_init(&a_empty[s], 1); }
    for (int b = 0; b < 2; ++b) { mbar_init(&acc_full[b], 1); mbar_init(&acc_empty[b], 2 * WS2_EPI_WARPS); }
    mbar_init_fence();
  } else if (warp == 2) {
    tmem_alloc<2, TMEM_COLS>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // both CTAs' barriers exist before any remote arrive / TMA completion targets them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const bool w_early = grp.w_early != 0;
  if (!(warp == 0 && lane == 0 && w_early)) pdl_wait_then_release();  // the producer lane first requests W (below)
  if (warp >= 2) {  // epilogue warps stage the bias (named barrier 1)
    tc_stage_bias(P, n0, BN, bias_s, threadIdx.x - 64, WS2_THREADS - 64);
    asm volatile("bar.sync 1, %0;" ::"n"(WS2_THREADS - 64) : "memory");
  }

  if (warp == 0) {
    if (lane == 0) {  // ===== TMA producer (each CTA loads its own halves; bytes are counted on the leader's barriers) =====
      const int nw = n0 + int(rank) * BNL;
      auto load_w = [&](int kb) {
        const uint32_t leader_w = mapa_u32(smem_u32(&w_full[kb]), 0);
        if (rank == 0) mbar_expect_tx(&w_full[kb], 2u * W_KB_BYTES);
        if (!P.b_mn_major) {
          tma_load_2d_pair(sW + size_t(kb) * W_KB_BYTES, &P.tmB, leader_w, kb * TC_BK, nw);
        } else {
#pragma unroll
          for (int j = 0; j < BNL / 64; ++j)
            tma_load_2d_pair(sW + size_t(kb) * W_KB_BYTES + j * 64 * TC_BK * 2, &P.tmB, leader_w, nw + 64 * j, kb * TC_BK);
        }
      };
      if (w_early) {  // the whole slice is requested while the previous kernel drains; the activations only after it completed
        for (int kb = 0; kb < KB; ++kb) load_w(kb);
        pdl_wait_then_release();
      }
      int it = 0, tt = 0;
      for (int tile = pair_local; tile < tiles2; tile += pairs, ++tt) {
        const int m0 = tile * 2 * TC_BM + int(rank) * TC_BM;
        for (int kb = 0; kb < KB; ++kb, ++it) {
          const int s = it % a_stages;
          const uint32_t ph = (it / a_stages) & 1;
          mbar_wait(&a_empty[s], ph ^ 1);
          if (tt == 0 && !w_early) load_w(kb);  // W k-block and the first tile's A k-block interleaved: the MMA needs them in this order
          if (rank == 0) mbar_expect_tx(&a_full[s], 2u * TC_A_BYTES);
          tma_load_2d_pair(sA + size_t(s) * TC_A_BYTES, &P.tmA, mapa_u32(smem_u32(&a_full[s]), 0), kb * TC_BK, m0);
        }
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && rank == 0) {  // ===== MMA issuer of the pair =====
      const uint32_t idesc = umma_idesc(2 * TC_BM, BN, false, P.b_mn_major != 0);
      const uint32_t b_lbo = P.b_mn_major ? TC_BK * 128 : 0, b_kstep = P.b_mn_major ? 2048 : 32;
      int it = 0, t = 0;
      for (int tile = pair_local; tile < tiles2; tile += pairs, ++t) {
        const int buf = t & 1;
        mbar_wait(&acc_empty[buf], ((t >> 1) & 1) ^ 1);
        tc_fence_after();
        for (int kb = 0; kb < KB; ++kb, ++it) {
          const int s = it % a_stages;
          const uint32_t ph = (it / a_stages) & 1;
          if (t == 0) mbar_wait(&w_full[kb], 0);
          mbar_wait(&a_full[s], ph);
          tc_fence_after();
          const uint32_t a_addr = smem_u32(sA + size_t(s) * TC_A_BYTES), b_addr = smem_u32(sW + size_t(kb) * W_KB_BYTES);
#pragma unroll
          for (int k = 0; k < TC_BK / 16; ++k)
            umma2_bf16(tmem_base + uint32_t(buf * BN), umma_desc(a_addr + k * 32, 0, 1024), umma_desc(b_addr + k * b_kstep, b_lbo, 1024),
                       idesc, (kb > 0 || k > 0) ? 1u : 0u);
          umma2_commit(&a_empty[s]);
          if (kb == KB - 1) umma2_commit(&acc_full[buf]);
        }
      }
    }
  } else {  // ===== epilogue: this CTA's 128 rows x 256 columns; warp = (TMEM lane quarter q, 64-column chunk) =====
    const int q = warp & 3, chunk = (warp - 2) >> 2;
    const int ntiles = grp.stage_tiles;
    uint8_t* st_base = stage_area + (warp - 2) * ntiles * TC_STAGE_BYTES;
    const CUtensorMap* tm_out = &grp.tm_out[pidx];
    const int act = P.act;
    // two scalars and a select, not an array indexed by `buf`: the array lived in local memory (an LDL in front of every arrive)
    const uint32_t leader_empty0 = mapa_u32(smem_u32(&acc_empty[0]), 0), leader_empty1 = mapa_u32(smem_u32(&acc_empty[1]), 0);
    const int sw = lane & 7;
    const int col0 = chunk * 64;
    const float* bs = bias_s + col0;
    int t = 0, tile_i = 0;
    // dgrad straight from registers, no staging tile: shared memory is left to the operands (W half + a deep A ring), and
    // the epilogue does not compete with the MMAs for shared-memory bandwidth
    if (P.epilogue == TC_EPI_DGRAD) {  // direct: activation row in, result row out, 32 bytes per access (rows are 32-byte aligned)
      const bool cols_ok = n0 + col0 + 64 <= P.N;
      for (int tile = pair_local; tile < tiles2; tile += pairs, ++t) {
        const int buf = t & 1;
        const int m = tile * 2 * TC_BM + int(rank) * TC_BM + q * 32 + lane;
        const bool row_ok = m < P.M;
        const __nv_bfloat16* arow = P.aux + int64_t(row_ok ? m : 0) * P.ld_aux + n0 + col0;
        __nv_bfloat16* orow = P.out_bf16 + int64_t(row_ok ? m : 0) * P.ld_bf16 + n0 + col0;
        uint32_t ax[4][8];
        if (cols_ok) {  // requested before the accumulator is awaited: the latency hides behind the MMAs
#pragma unroll
          for (int sidx = 0; sidx < 4; ++sidx) ldg256(arow + sidx * 16, ax[sidx]);
        } else {
#pragma unroll
          for (int sidx = 0; sidx < 4; ++sidx)
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int c = n0 + col0 + sidx * 16 + 2 * j;
              const uint32_t lo = c < P.N ? uint32_t(__bfloat16_as_ushort(arow[sidx * 16 + 2 * j])) : 0u;
              const uint32_t hi = c + 1 < P.N ? uint32_t(__bfloat16_as_ushort(arow[sidx * 16 + 2 * j + 1])) : 0u;
              ax[sidx][j] = lo | (hi << 16);
            }
        }
        const uint32_t tcol = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(buf * BN + col0);
        mbar_wait(&acc_full[buf], uint32_t((t >> 1) & 1));
        tc_fence_after();
        __syncwarp();
        uint32_t va[16], vb[16], o[8];
        auto emit = [&](int sidx) {
          if (!row_ok) return;
          if (cols_ok) {
            stg256(orow + sidx * 16, o);
          } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const int c = n0 + col0 + sidx * 16 + 2 * j;
              if (c < P.N) orow[sidx * 16 + 2 * j] = __ushort_as_bfloat16(uint16_t(o[j] & 0xFFFFu));
              if (c + 1 < P.N) orow[sidx * 16 + 2 * j + 1] = __ushort_as_bfloat16(uint16_t(o[j] >> 16));
            }
          }
        };
        tmem_ld16_nowait(tcol, va);
        tmem_ld_wait();
        tmem_ld16_nowait(tcol + 16, vb);
        act_grad16(va, ax[0], act, o); emit(0);
        tmem_ld_wait();
        tmem_ld16_nowait(tcol + 32, va);
        act_grad16(vb, ax[1], act, o); emit(1);
        tmem_ld_wait();
        tmem_ld16_nowait(tcol + 48, vb);
        act_grad16(va, ax[2], act, o); emit(2);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(buf ? leader_empty1 : leader_empty0);
        act_grad16(vb, ax[3], act, o); emit(3);
      }
    } else if (grp.tma_out[pidx] == 0) {  // forward, direct: 32-byte row segments from registers (rows 32-byte aligned, whole chunk < N)
      for (int tile = pair_local; tile < tiles2; tile += pairs, ++t) {
        const int buf = t & 1;
        const int m = tile * 2 * TC_BM + int(rank) * TC_BM + q * 32 + lane;
        const bool row_ok = m < P.M;
        __nv_bfloat16* orow = P.out_bf16 + int64_t(row_ok ? m : 0) * P.ld_bf16 + n0 + col0;
        const uint32_t tcol = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(buf * BN + col0);
        mbar_wait(&acc_full[buf], uint32_t((t >> 1) & 1));
        tc_fence_after();
        __syncwarp();
        uint32_t va[16], vb[16], o[8];
        tmem_ld16_nowait(tcol, va);
        tmem_ld_wait();
        tmem_ld16_nowait(tcol + 16, vb);
        bias_act16(va, bs, act, o);
        if (row_ok) stg256(orow, o);
        tmem_ld_wait();
        tmem_ld16_nowait(tcol + 32, va);
        bias_act16(vb, bs + 16, act, o);
        if (row_ok) stg256(orow + 16, o);
        tmem_ld_wait();
        tmem_ld16_nowait(tcol + 48, vb);
        bias_act16(va, bs + 32, act, o);
        if (row_ok) stg256(orow + 32, o);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(buf ? leader_empty1 : leader_empty0);
        bias_act16(vb, bs + 48, act, o);
        if (row_ok) stg256(orow + 48, o);
      }
    } else
    for (int tile = pair_local; tile < tiles2; tile += pairs, ++t) {
      const int buf = t & 1;
      const int mq = tile * 2 * TC_BM + int(rank) * TC_BM + q * 32;
      uint8_t* st = st_base + tile_i * TC_STAGE_BYTES;
      tile_i = tile_i + 1 == ntiles ? 0 : tile_i + 1;
      const uint32_t sbase = smem_u32(st), my_row = sbase + uint32_t(lane) * 128u;
      const uint32_t tcol = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(buf * BN + col0);
      // the bulk store that last read this staging tile (ntiles row tiles ago) must have drained it
      if (lane == 0) {
        if (ntiles == 1) bulk_wait_read<0>();
        else bulk_wait_read<1>();
      }
      mbar_wait(&acc_full[buf], uint32_t((t >> 1) & 1));
      tc_fence_after();
      __syncwarp();
      uint32_t va[16], vb[16];
      tmem_ld16_nowait(tcol, va);
      tmem_ld_wait();
      tmem_ld16_nowait(tcol + 16, vb);
      ws2_finish16(va, bs, act, my_row, sw, 0);
      tmem_ld_wait();
      tmem_ld16_nowait(tcol + 32, va);
      ws2_finish16(vb, bs + 16, act, my_row, sw, 1);
      tmem_ld_wait();
      tmem_ld16_nowait(tcol + 48, vb);
      ws2_finish16(va, bs + 32, act, my_row, sw, 2);
      tmem_ld_wait();
      // every accumulator column of this warp has been read: release the TMEM buffer to the leader's MMA before the
      // last quarter of the math
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(buf ? leader_empty1 : leader_empty0);
      ws2_finish16(vb, bs + 48, act, my_row, sw, 3);
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        if (mq < P.M) {  // rows >= M and columns >= N inside the box are clipped by the tensor map
          tma_store_2d(tm_out, sbase, n0 + col0, mq);
        }
        bulk_commit();
      }
    }
    if (lane == 0) bulk_wait<0>();
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();  // the peer may still be reading this CTA's operands / arriving on its barriers
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<2, TMEM_COLS>(tmem_base);
  }
}

constexpr int kWsMaxSmem = 227 * 1024;
// alignment slack + (barriers, bias, PPO constants, reduction scratch) + epilogue staging tiles
static int ws_fixed_smem(int stage_tiles) { return 1024 + 4096 + stage_tiles * TC_EPI_WARPS * TC_STAGE_BYTES; }
static int ws2_fixed_smem(int stage_tiles) { return 1024 + 4096 + stage_tiles * WS2_EPI_WARPS * TC_STAGE_BYTES; }

// N tile, A-ring depth and staging tiles per warp for a group, or bn = 0 when the weights-stationary kernel does not apply.
// N tile <= 128: each epilogue warp then owns 64 columns = ONE 128-byte staging row, so the dgrad's whole activation
// tile is requested in a single burst before the accumulator is awaited (and W slices of <= 96 KB leave a deep A ring).
// A dgrad takes a third staging tile when the ring keeps >= 3 stages: tile t is stored by the copy engine while t + 1's
// activation slab streams in and t + 2's... is not yet needed, so no wait sits between a store and the next request.
// kind: 0 bulk-stored forward, 1 dgrad, 2 anything else.  force_bn > 0: only that N tile (the operands' tensor maps were
// built for tc_ws_bn(), which plans with kind 2).
static void ws_plan(int maxN, int maxK, int kind, int* bn_out, int* stages_out, int* stage_tiles_out, int force_bn = 0) {
  *bn_out = 0;
  *stages_out = 0;
  *stage_tiles_out = 2;
  const int kb = (maxK + TC_BK - 1) / TC_BK;
  for (int bn : {128, 64}) {
    if (force_bn > 0 && bn != force_bn) continue;
    if (bn > 64 && maxN <= bn / 2) continue;  // a narrower tile covers N
    const int64_t w_bytes = int64_t(kb) * bn * TC_BK * 2;
    if ((maxN + bn - 1) / bn * 2 > kWsMaxSlots) continue;
    for (int tiles : {3, 2, 1}) {
      // forward through the bulk store: one tile (its store has drained long before the next accumulator is ready) and
      // a deeper A ring instead — the K = 384 layer is bound by operand bytes in flight
      if (tiles == 3 && !(kind == 1 && bn == 128)) continue;
      if (tiles == 2 && kind == 0 && bn == 128) continue;
      if (tiles == 1 && !(kind == 0 && bn == 128)) continue;
      const int64_t avail = kWsMaxSmem - ws_fixed_smem(tiles) - w_bytes;
      const int stages = int(avail / TC_A_BYTES);
      if (stages < 3) continue;
      *bn_out = bn;
      *stages_out = stages > 8 ? 8 : stages;
      *stage_tiles_out = tiles;
      return;
    }
  }
}

bool tc_ws_applicable(int64_t total_tiles_m, int maxN, int maxK) {
  int bn, st, tl;
  ws_plan(maxN, maxK, 2, &bn, &st, &tl);
  // persistence pays once every CTA owns at least ~two row tiles; below that the one-tile kernel has more CTAs
  return bn != 0 && total_tiles_m >= 2ll * num_sms();
}

int tc_ws_bn(int maxN, int maxK) {
  int bn, st, tl;
  ws_plan(maxN, maxK, 2, &bn, &st, &tl);
  return bn;
}

template <int BN>
static int launch_ws_bn(const WsGroup& g, int stages, int kb_max, int grid, cudaStream_t st) {
  const int smem = kb_max * BN * TC_BK * 2 + stages * TC_A_BYTES + ws_fixed_smem(g.stage_tiles);
  static int configured = 0;
  if (configured < smem) {
    B2_CUDA(cudaFuncSetAttribute(tc_ws_kernel<BN>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    configured = smem;
  }
  B2_CUDA(launch_pdl(tc_ws_kernel<BN>, dim3(grid), dim3(TC_THREADS), smem, st, g, stages));
  B2_LAUNCH_CHECK();
  return B200PPO_OK;
}

// g: one or two forward / dgrad problems built with tc_group_add(..., bn = tc_ws_bn(maxN, maxK), split 1), K-major.
int launch_tc_ws(const TcGroup& g, cudaStream_t st, int* grid_out, bool w_early) {
  B2_CHECK_ARG(g.count >= 1 && g.count <= 2, "weights-stationary launch takes one or two problems");
  int maxN = 0, maxK = 0;
  for (int i = 0; i < g.count; ++i) {
    B2_CHECK_ARG(!g.p[i].a_mn_major && g.p[i].split_k == 1, "weights-stationary kernel: K-major A, no split-K");
    maxN = std::max(maxN, g.p[i].N);
    maxK = std::max(maxK, g.p[i].K);
  }
  int kind = 0;  // all problems staged forward -> 0; any dgrad -> 1; anything else -> 2
  for (int i = 0; i < g.count; ++i) {
    if (g.p[i].epilogue == TC_EPI_DGRAD) kind = std::max(kind, 1);
    else if (!(g.p[i].epilogue == TC_EPI_FWD && g.p[i].staged)) kind = 2;
  }
  int bn, stages, stage_tiles;
  ws_plan(maxN, maxK, kind, &bn, &stages, &stage_tiles, tc_ws_bn(maxN, maxK));
  // CTA pairs with 256-wide MMAs for wide forward layers (every problem N > 128, operands built for 128-row boxes)
  bool pair = (kind == 0 || kind == 1) && bn == 128;
  for (int i = 0; i < g.count; ++i) {
    const TcProblem& q = g.p[i];
    pair = pair && q.N > 128 && q.tiles_m >= 2;
    if (kind == 1)  // every problem a dgrad whose rows start on 32-byte sectors (direct 256-bit epilogue)
      pair = pair && q.epilogue == TC_EPI_DGRAD && q.out_bf16 != nullptr && q.aux != nullptr && q.ld_bf16 % 16 == 0 && q.ld_aux % 16 == 0 &&
             (reinterpret_cast<uintptr_t>(q.out_bf16) & 31u) == 0 && (reinterpret_cast<uintptr_t>(q.aux) & 31u) == 0;
  }
  const int pair_kb = (maxK + TC_BK - 1) / TC_BK;
  int pair_stages = 0;
  // forward epilogue: 256-bit stores straight from registers when every row segment is a whole, aligned 32-byte sector
  // (measured 3% faster than staging + bulk store, and the staging tiles' shared memory goes to the A ring instead)
  bool fwd_direct = kind == 0;
  for (int i = 0; i < g.count; ++i)
    fwd_direct = fwd_direct && g.p[i].N % 64 == 0 && g.p[i].ld_bf16 % 16 == 0 && (reinterpret_cast<uintptr_t>(g.p[i].out_bf16) & 31u) == 0;
  const int pair_tiles = (kind == 1 || fwd_direct) ? 0 : 1;  // staged forward: one tile per epilogue warp (a whole row tile to drain)
  if (pair) {
    const int64_t avail = kWsMaxSmem - ws2_fixed_smem(pair_tiles) - int64_t(pair_kb) * 128 * TC_BK * 2;
    pair_stages = int(std::min<int64_t>(8, avail / TC_A_BYTES));
    int slots = 0;
    for (int i = 0; i < g.count; ++i) slots += (g.p[i].N + 255) / 256;
    if (pair_stages < 3 || slots > kWsMaxSlots || pair_kb > WS2_MAX_KB) pair = false;
  }
  if (pair) {
    WsGroup w{};
    w.count = g.count;
    w.stage_tiles = pair_tiles;
    w.w_early = w_early ? 1 : 0;
    int64_t work = 0;
    for (int i = 0; i < g.count; ++i) {
      const TcProblem& q = g.p[i];
      w.p[i] = q;
      if (kind == 0) {
        if (!fwd_direct) B2_TRY(tc_make_map(&w.tm_out[i], q.out_bf16, q.N, q.M, q.ld_bf16, 64, 32));
        w.tma_out[i] = fwd_direct ? 0 : 1;
      }
      for (int n0 = 0; n0 < q.N; n0 += 256) {
        w.slot_prob[w.n_slots] = i;
        w.slot_n0[w.n_slots] = n0;
        ++w.n_slots;
        work += (q.M + 255) / 256;
      }
    }
    const int pairs_total = int(std::min<int64_t>(num_sms() / 2, work));
    int begin = 0;
    for (int sidx = 0; sidx < w.n_slots; ++sidx) {
      w.cta_begin[sidx] = 2 * begin;
      const int64_t tiles = (g.p[w.slot_prob[sidx]].M + 255) / 256;
      int share = (sidx == w.n_slots - 1) ? pairs_total - begin : int((int64_t(pairs_total) * tiles + work / 2) / work);
      if (share < 1) share = 1;
      begin += share;
    }
    const int total_pairs = std::max(begin, pairs_total);
    w.cta_begin[w.n_slots] = 2 * total_pairs;
    const int smem = pair_kb * 128 * TC_BK * 2 + pair_stages * TC_A_BYTES + ws2_fixed_smem(pair_tiles);
    static int configured = 0;
    if (configured < smem) {
      B2_CUDA(cudaFuncSetAttribute(tc_ws2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
      configured = smem;
    }
    if (grid_out) *grid_out = 2 * total_pairs;
    B2_CUDA(launch_pdl(tc_ws2_kernel, dim3(2 * total_pairs), dim3(WS2_THREADS), smem, st, w, pair_stages));
    B2_LAUNCH_CHECK();
    return B200PPO_OK;
  }
  B2_CHECK_ARG(bn != 0, "weights do not fit in shared memory");
  WsGroup w{};
  w.count = g.count;
  w.stage_tiles = stage_tiles;
  w.w_early = w_early ? 1 : 0;
  for (int i = 0; i < g.count; ++i) {
    const TcProblem& q = g.p[i];
    w.tma_out[i] = 0;
    if (bn == 128 && q.staged) {
      B2_TRY(tc_make_map(&w.tm_out[i], q.out_bf16, q.N, q.M, q.ld_bf16, 64, 32));
      w.tma_out[i] = 1;
    }
  }
  int64_t work = 0;  // row tiles summed over slots
  for (int i = 0; i < g.count; ++i) {
    w.p[i] = g.p[i];
    for (int n0 = 0; n0 < g.p[i].N; n0 += bn) {
      w.slot_prob[w.n_slots] = i;
      w.slot_n0[w.n_slots] = n0;
      ++w.n_slots;
      work += g.p[i].tiles_m;
    }
  }
  const int grid = int(std::min<int64_t>(num_sms(), work));
  int begin = 0;
  for (int sidx = 0; sidx < w.n_slots; ++sidx) {
    w.cta_begin[sidx] = begin;
    const int64_t tiles = g.p[w.slot_prob[sidx]].tiles_m;
    int share = (sidx == w.n_slots - 1) ? grid - begin : int((int64_t(grid) * tiles + work / 2) / work);
    if (share < 1) share = 1;
    begin += share;
  }
  w.cta_begin[w.n_slots] = std::max(begin, grid);
  const int kb_max = (maxK + TC_BK - 1) / TC_BK;
  const int total = w.cta_begin[w.n_slots];
  if (grid_out) *grid_out = total;
  switch (bn) {
    case 64: return launch_ws_bn<64>(w, stages, kb_max, total, st);
    case 128: return launch_ws_bn<128>(w, stages, kb_max, total, st);
  }
  set_error("weights-stationary kernel: unsupported N tile %d", bn);
  return B200PPO_EINVAL;
}

}  // namespace b200ppo
