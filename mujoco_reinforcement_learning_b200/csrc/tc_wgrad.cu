// Weight / bias gradients of the MLP on CTA pairs:  dW_l = dZ_l^T H_{l-1},  db_l = dZ_l^T 1   (split-K over the batch).
//
// replaces: the autograd backward of aten::addmm in NetworkBlock.forward (src/models/network_block_creator.py:74-86),
//           reached from ppo.py:121,134 (loss.backward()).
//
// Why a second kernel: the one-tile kernel (tc_gemm.cu) gives every 128 x 128 output tile its own CTA, so dZ is
// streamed once per N tile and H once per M tile — at the bench shape 408 MB of L2 reads per minibatch at ~10 TB/s,
// i.e. the weight gradient was bound by L2 -> SM bandwidth, and the bias gradient (a ones-column appended to H) cost
// a third N tile for ONE useful column (N = 257).  Here a cluster of two CTAs owns a 256 x 256 output block:
//   * tcgen05.mma.cta_group::2, M = 256 (each CTA stages its own 128 rows of dZ^T), N = 256 or 128 (each CTA stages
//     half of the H columns): every operand byte is read from L2 once per 256 x 256 block — 2.2x less traffic;
//   * the bias gradient is a second, 32-column MMA per k-step against a constant tile of ones that never leaves
//     shared memory (+12% tensor work, no memory traffic), into its own TMEM columns;
//   * both operands are MN-major views of row-major [batch][features] activations (no transposes), K tails and
//     ragged M / N are zero-filled by TMA.
//   warp 0 (both CTAs)  TMA producer, bytes counted on the leader's mbarriers      warp 1 (leader)  MMA issuer
//   warps 2-9 (both)    fp32 split-K partial store of the CTA's own 128 rows (summed deterministically inside Adam)
#include <algorithm>

#include "tc_common.cuh"

namespace b200ppo {

constexpr int kWg2MaxTiles = 24;
constexpr int WG2_STAGES = 6;
constexpr int WG2_STAGE_BYTES = TC_A_BYTES + 128 * TC_BK * 2;  // own 128 rows of dZ^T + own <= 128 columns of H
constexpr int WG2_ONES_BYTES = 4096;

struct Wg2Tile {
  int prob, m0, n0, nw, bias;  // nw: MMA N of this block (128 or 256); bias: this block also produces db
  // split-K of THIS block: the blocks stream different byte counts per k-tile (a 256 x 256 block 64 KB per pair, a
  // 256 x 128 one 48 KB, the 17-row output-layer block 33 KB), and the kernel is bound by that stream, so the batch is
  // cut into more pieces for the heavier blocks; pairs [pair_begin, pair_begin + splits) work on this block
  int pair_begin, splits, k_tiles_per_split;
};

struct Wg2Group {
  TcProblem p[kMaxTcProblems];
  Wg2Tile tile[kWg2MaxTiles];
  int count, n_tiles, max_splits;  // max_splits: partial slots the consumer sums; blocks with fewer splits zero-fill the rest
};

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(TC_THREADS, 1) tc_wgrad2_kernel(const __grid_constant__ Wg2Group grp) {
  constexpr uint32_t TMEM_COLS = 512;
  constexpr uint32_t BIAS_COL = 256;  // TMEM column of the 32-wide bias accumulator
  extern __shared__ uint8_t smem_raw[];
  // pointer + offset (not an integer round trip): the compiler keeps the shared address space and emits LDS / STS
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  uint8_t* ring = smem;
  uint8_t* ones = smem + WG2_STAGES * WG2_STAGE_BYTES;
  uint64_t* full_bar = reinterpret_cast<uint64_t*>(ones + WG2_ONES_BYTES);
  uint64_t* empty_bar = full_bar + WG2_STAGES;
  uint64_t* done_bar = empty_bar + WG2_STAGES;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(done_bar + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t rank = cluster_ctarank();
  const int pair = int(blockIdx.x) >> 1;
  int ti = 0;
#pragma unroll 1
  for (int i = 1; i < grp.n_tiles; ++i)
    if (pair >= grp.tile[i].pair_begin) ti = i;
  const Wg2Tile T = grp.tile[ti];
  const int split = pair - T.pair_begin;
  const TcProblem& P = grp.p[T.prob];
  const int total_kt = (P.K + TC_BK - 1) / TC_BK;
  const int kt_begin = split * T.k_tiles_per_split;
  const int kt_end = min(total_kt, kt_begin + T.k_tiles_per_split);
  const bool has_k = kt_end > kt_begin;
  const int nw_half = T.nw >> 1;  // H columns staged by each CTA
  const uint32_t stage_tx = 2u * uint32_t(TC_A_BYTES + nw_half * TC_BK * 2);

  // constant B operand of the bias MMA: bf16 ones (any layout of ones is a tile of ones)
  for (int i = threadIdx.x; i < WG2_ONES_BYTES / 4; i += TC_THREADS) reinterpret_cast<uint32_t*>(ones)[i] = 0x3F803F80u;
  fence_proxy_async_smem();
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < WG2_STAGES; ++s) { mbar_init(&full_bar[s], 1); mbar_init(&empty_bar[s], 1); }
    mbar_init(done_bar, 1);
    mbar_init_fence();
  } else if (warp == 2) {
    tmem_alloc<2, TMEM_COLS>(tmem_slot);
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait_then_release();  // dZ and H come from the kernels before this one

  if (warp == 0) {
    if (lane == 0 && has_k) {  // ===== TMA producer: own 128 rows of dZ^T (two 64-wide MN atoms) + own half of the H columns =====
      const int ma = T.m0 + int(rank) * TC_BM;
      const int nb = T.n0 + int(rank) * nw_half;
      for (int kt = kt_begin, it = 0; kt < kt_end; ++kt, ++it) {
        const int s = it % WG2_STAGES;
        const uint32_t ph = (it / WG2_STAGES) & 1;
        mbar_wait(&empty_bar[s], ph ^ 1);
        if (rank == 0) mbar_expect_tx(&full_bar[s], stage_tx);
        const uint32_t leader_full = mapa_u32(smem_u32(&full_bar[s]), 0);
        uint8_t* a = ring + s * WG2_STAGE_BYTES;
        uint8_t* b = a + TC_A_BYTES;
        tma_load_2d_pair(a, &P.tmA, leader_full, ma, kt * TC_BK);
        tma_load_2d_pair(a + 64 * TC_BK * 2, &P.tmA, leader_full, ma + 64, kt * TC_BK);
        tma_load_2d_pair(b, &P.tmB, leader_full, nb, kt * TC_BK);
        if (nw_half > 64) tma_load_2d_pair(b + 64 * TC_BK * 2, &P.tmB, leader_full, nb + 64, kt * TC_BK);
      }
    }
  } else if (warp == 1) {
    if (lane == 0 && rank == 0 && has_k) {  // ===== MMA issuer of the pair =====
      // D fp32, A/B bf16, both MN-major, N = nw, M = 256 | bias: B K-major (ones), N = 32
      const uint32_t idesc = umma_idesc(2 * TC_BM, T.nw, true, true);
      constexpr uint32_t idesc_bias = umma_idesc(2 * TC_BM, 32, true, false);
      const uint32_t lbo = TC_BK * 128;  // 64-wide MN atoms are 8 KB apart; a K = 16 step is 16 rows of 128 B
      const uint32_t ones_addr = smem_u32(ones);
      for (int kt = kt_begin, it = 0; kt < kt_end; ++kt, ++it) {
        const int s = it % WG2_STAGES;
        const uint32_t ph = (it / WG2_STAGES) & 1;
        mbar_wait(&full_bar[s], ph);
        tc_fence_after();
        const uint32_t a_addr = smem_u32(ring + s * WG2_STAGE_BYTES), b_addr = a_addr + TC_A_BYTES;
#pragma unroll
        for (int k = 0; k < TC_BK / 16; ++k) {
          const uint64_t ad = umma_desc(a_addr + k * 2048, lbo, 1024);
          const uint32_t acc = (it > 0 || k > 0) ? 1u : 0u;
          umma2_bf16(tmem_base, ad, umma_desc(b_addr + k * 2048, lbo, 1024), idesc, acc);
          if (T.bias) umma2_bf16(tmem_base + BIAS_COL, ad, umma_desc(ones_addr + k * 32, 0, 1024), idesc_bias, acc);
        }
        umma2_commit(&empty_bar[s]);
      }
      umma2_commit(done_bar);
    }
  } else {  // ===== epilogue: fp32 partials of this CTA's 128 rows =====
    const int q = warp & 3, half = (warp - 2) >> 2;
    const int m = T.m0 + int(rank) * TC_BM + q * 32 + lane;
    const bool row_ok = m < P.M;
    if (has_k) {
      mbar_wait(done_bar, 0);
      tc_fence_after();
    }
    float* outp = P.out_f32 + int64_t(split) * P.split_stride + int64_t(m) * P.ld_f32;
    const bool vec = (P.ld_f32 % 4 == 0) && (P.split_stride % 4 == 0) && ((reinterpret_cast<uintptr_t>(P.out_f32) & 15u) == 0);
    const int c_begin = half * nw_half, c_end = c_begin + nw_half;
    for (int c = c_begin; c < c_end; c += 16) {
      uint32_t v[16];
      if (has_k) {
        tmem_ld16(tmem_base + (uint32_t(q * 32) << 16) + uint32_t(c), v);
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) v[j] = 0u;
      }
      const int n = T.n0 + c;
      if (!row_ok || n >= P.N) continue;
      if (vec && n + 16 <= P.N) {
#pragma unroll
        for (int u = 0; u < 4; ++u)
          reinterpret_cast<float4*>(outp + n)[u] = make_float4(__uint_as_float(v[4 * u]), __uint_as_float(v[4 * u + 1]),
                                                                __uint_as_float(v[4 * u + 2]), __uint_as_float(v[4 * u + 3]));
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j)
          if (n + j < P.N) outp[n + j] = __uint_as_float(v[j]);
      }
    }
    if (T.bias && half == 0 && P.bias_grad != nullptr) {
      uint32_t v[16];
      if (has_k) {
        tmem_ld16(tmem_base + (uint32_t(q * 32) << 16) + BIAS_COL, v);
      } else {
        v[0] = 0u;
      }
      if (row_ok) P.bias_grad[int64_t(split) * P.split_stride + m] = __uint_as_float(v[0]);
    }
    // the consumer sums grp.max_splits partial slots: the ones this block has no split for are zero-filled by its pairs
    for (int z = split + T.splits; z < grp.max_splits; z += T.splits) {
      if (!row_ok) break;
      float* zp = P.out_f32 + int64_t(z) * P.split_stride + int64_t(m) * P.ld_f32;
      for (int c = c_begin; c < c_end; c += 4) {
        const int n = T.n0 + c;
        if (n >= P.N) break;
        if (vec && n + 4 <= P.N) *reinterpret_cast<float4*>(zp + n) = make_float4(0.f, 0.f, 0.f, 0.f);
        else
          for (int j = 0; j < 4; ++j)
            if (n + j < P.N) zp[n + j] = 0.f;
      }
      if (T.bias && half == 0 && P.bias_grad != nullptr) P.bias_grad[int64_t(z) * P.split_stride + m] = 0.f;
    }
    tc_fence_before();
  }
  __syncthreads();
  cluster_sync_all();  // the peer's MMAs read this CTA's operands until the last commit
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc<2, TMEM_COLS>(tmem_base);
  }
}

// Every problem of `g` was added with tc_group_add(..., both operands MN-major): C[M, N] fp32 partials at out_f32
// (+ split * split_stride), row sums of A^T (the bias gradient) at bias_grad.  N is the layer's input width WITHOUT a
// ones-column.  *split_out: partials written per output element.
int launch_tc_wgrad2(const TcGroup& g, int max_split, cudaStream_t st, int* split_out) {
  Wg2Group w{};
  w.count = g.count;
  int64_t K = 0;
  for (int i = 0; i < g.count; ++i) {
    const TcProblem& p = g.p[i];
    B2_CHECK_ARG(p.a_mn_major && p.b_mn_major && p.out_f32 != nullptr, "pair weight-gradient kernel: MN-major operands, fp32 output");
    B2_CHECK_ARG(i == 0 || p.K == K, "pair weight-gradient kernel: all problems share the batch dimension");
    K = p.K;
    w.p[i] = p;
    for (int m0 = 0; m0 < p.M; m0 += 2 * TC_BM)
      for (int n0 = 0; n0 < p.N; n0 += 256) {
        B2_CHECK_ARG(w.n_tiles < kWg2MaxTiles, "pair weight-gradient kernel: too many output blocks");
        const int rem = p.N - n0;
        w.tile[w.n_tiles++] = Wg2Tile{i, m0, n0, rem > 128 ? 256 : 128, n0 == 0 ? 1 : 0};
      }
  }
  if (w.n_tiles == 0) return B200PPO_OK;
  const int total_kt = int((K + TC_BK - 1) / TC_BK);
  const int pairs = num_sms() / 2;
  // The same split for every block: all blocks then walk the batch in step, so the operands two blocks share (dZ1 of the
  // two dW1 blocks, every k-tile of X / H) meet in L2.  Measured (profiles/README.md, round 2): splits in proportion to
  // the bytes a block streams were slower (8.28 vs 7.07 ms per 160 launches).
  int max_sp = 1;
  for (int t = 0; t < w.n_tiles; ++t) w.tile[t].splits = std::max(1, std::min({pairs / w.n_tiles, max_split, total_kt}));
  int begin = 0;
  for (int t = 0; t < w.n_tiles; ++t) {
    Wg2Tile& T = w.tile[t];
    T.k_tiles_per_split = (total_kt + T.splits - 1) / T.splits;
    T.splits = (total_kt + T.k_tiles_per_split - 1) / T.k_tiles_per_split;  // no empty trailing splits
    T.pair_begin = begin;
    begin += T.splits;
    max_sp = std::max(max_sp, T.splits);
  }
  w.max_splits = max_sp;
  const int total_pairs = begin;
  constexpr int smem = 1024 + WG2_STAGES * WG2_STAGE_BYTES + WG2_ONES_BYTES + 256;
  static bool configured = false;
  if (!configured) {
    B2_CUDA(cudaFuncSetAttribute(tc_wgrad2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    configured = true;
  }
  B2_CUDA(launch_pdl(tc_wgrad2_kernel, dim3(2 * total_pairs), dim3(TC_THREADS), smem, st, w));
  B2_LAUNCH_CHECK();
  if (split_out) *split_out = max_sp;
  return B200PPO_OK;
}

}  // namespace b200ppo
