// Device-side building blocks shared by the tcgen05 kernels (tc_gemm.cu, tc_persist.cu, tc_ws.cu, tc_wgrad.cu, tc_chain.cu):
// the one-tile / persistent tile pipeline and the epilogues.  The PTX primitives they are built from live in tc_ptx.cuh.
#pragma once
#include <string.h>

#include "tc_gemm.cuh"
#include "tc_ptx.cuh"

namespace b200ppo {

constexpr int TC_BM = 128;
constexpr int TC_BK = 64;  // bf16 elements: 128 bytes = one swizzle row
constexpr int TC_EPI_WARPS = 8;                        // two per TMEM lane quarter, each takes half of the columns
constexpr int TC_THREADS = (2 + TC_EPI_WARPS) * 32;    // + TMA producer warp + MMA issuer warp
constexpr int TC_A_BYTES = TC_BM * TC_BK * 2;

// MUFU.TANH: one instruction, max relative error ~2^-11 — below bf16's 2^-8 resolution of the stored activation
__device__ __forceinline__ float tanh_fast(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  __nv_bfloat162 h = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h);
}

__device__ __forceinline__ float split_unscale(float amax_a, float amax_b) {
  return exp2f(float(-(split_exponent(amax_a) + split_exponent(amax_b))));
}

// ---- tile pipeline of the one-tile (tc_gemm.cu) and persistent (tc_persist.cu) kernels ------------------------------
// Output tile `tile` of a group: its problem, split-K slice, corner and k range.  n_it ring iterations: in the
// fp32-tolerance mode the products of the terms run one after the other over the split's k range, smallest terms first.
struct TcTile {
  int pi, split, m0, n0, kt_begin, kt_len, n_it;
};

template <int BN>
__device__ __forceinline__ TcTile tc_tile(const TcGroup& grp, int tile) {
  TcTile t;
  t.pi = 0;
#pragma unroll 1
  for (int i = 1; i < grp.count; ++i)
    if (tile >= grp.p[i].tile_begin) t.pi = i;
  const TcProblem& P = grp.p[t.pi];
  int local = tile - P.tile_begin;
  const int tiles_mn = P.tiles_m * P.tiles_n;
  t.split = local / tiles_mn;
  local -= t.split * tiles_mn;
  t.m0 = (local / P.tiles_n) * TC_BM;
  t.n0 = (local % P.tiles_n) * BN;
  const int total_kt = (P.K + TC_BK - 1) / TC_BK;
  t.kt_begin = t.split * P.k_tiles_per_split;
  const int kt_end = min(total_kt, t.kt_begin + P.k_tiles_per_split);
  t.kt_len = max(kt_end - t.kt_begin, 0);
  t.n_it = P.parts ? split_products(P.parts) * t.kt_len : t.kt_len;
  return t;
}

// Producer: the A and B boxes of ring iteration `it` of tile T into one stage, completing on `bar`.
template <int BN>
__device__ __forceinline__ void tc_load_stage(const TcProblem& P, const TcTile& T, int it, uint8_t* a, uint8_t* b, uint64_t* bar) {
  int kb = T.kt_begin + it, ao = 0, bo = 0;  // k tile, offsets of the product's terms along the contiguous dimension
  if (P.parts) {
    const int c = it / T.kt_len;
    kb = T.kt_begin + (it - c * T.kt_len);
    ao = int((split_terms_a(P.parts) >> (4 * c)) & 3u) * P.a_part;
    bo = int((split_terms_b(P.parts) >> (4 * c)) & 3u) * P.b_part;
  }
  if (!P.a_mn_major) {
    tma_load_2d(a, &P.tmA, bar, ao + kb * TC_BK, T.m0);
  } else {
    tma_load_2d(a, &P.tmA, bar, ao + T.m0, kb * TC_BK);
    tma_load_2d(a + 64 * TC_BK * 2, &P.tmA, bar, ao + T.m0 + 64, kb * TC_BK);
  }
  if (!P.b_mn_major) {
    tma_load_2d(b, &P.tmB, bar, bo + kb * TC_BK, T.n0);
  } else {
#pragma unroll
    for (int j = 0; j < BN / 64; ++j) tma_load_2d(b + j * 64 * TC_BK * 2, &P.tmB, bar, bo + T.n0 + 64 * j, kb * TC_BK);
  }
}

// MMA issuer: a problem's instruction descriptor and operand descriptor steps ...
struct TcMma {
  uint32_t idesc, a_lbo, b_lbo, a_kstep, b_kstep;
};

template <int BN>
__device__ __forceinline__ TcMma tc_mma_setup(const TcProblem& P) {
  // K-major SW128: 8-row groups 1024 B apart; one K=16 step = +32 B inside the swizzle row.
  // MN-major SW128: K atoms (8 k-rows x 128 B) 1024 B apart (SBO), 64-wide MN atoms BK*128 B apart (LBO);
  //                 one K=16 step = +2048 B.
  TcMma m;
  const bool f16 = P.parts == 2;  // operand format: fp16 in the two-term mode, bf16 otherwise
  m.idesc = umma_idesc(TC_BM, BN, P.a_mn_major != 0, P.b_mn_major != 0, f16);
  m.a_lbo = P.a_mn_major ? TC_BK * 128 : 0;
  m.b_lbo = P.b_mn_major ? TC_BK * 128 : 0;
  m.a_kstep = P.a_mn_major ? 2048 : 32;
  m.b_kstep = P.b_mn_major ? 2048 : 32;
  return m;
}

// ... and the four K = 16 MMAs of one ring stage into the accumulator at TMEM address d
__device__ __forceinline__ void tc_mma_stage(const TcMma& m, uint32_t d, uint32_t a_addr, uint32_t b_addr, bool accumulate) {
#pragma unroll
  for (int k = 0; k < TC_BK / 16; ++k)
    umma_bf16(d, umma_desc(a_addr + k * m.a_kstep, m.a_lbo, 1024), umma_desc(b_addr + k * m.b_kstep, m.b_lbo, 1024), m.idesc,
              (accumulate || k > 0) ? 1u : 0u);
}

// Epilogue of one 128 x BN accumulator tile, executed by the 8 epilogue warps (warp index 2..9 of the CTA).
// X32: the fp32-tolerance problems' extras, compiled only into the kernels those problems use (the two-CTAs-per-SM
// instances keep their register budget): the fp32 activation operand of a dgrad is requested one chunk ahead, and full
// chunks of an fp32 output leave as 32-byte pieces (st.global.v8: whole sectors, half as many store instructions).
template <int BN, bool X32 = false>
__device__ __forceinline__ void tc_epilogue(const TcProblem& P, int split, uint32_t tmem_acc, bool has_k, int m0, int n0, int warp,
                                            int lane, uint64_t* tmem_full_bar, uint32_t full_parity, const float* bias_s) {
    // Problem fields into registers once (the indexed constant-bank loads of `P.` inside the column loop showed up
    // as long-scoreboard stalls), and everything the epilogue reads from global memory — the activation operand of
    // the dgrad, the bias of the forward — is requested BEFORE waiting for the accumulator, so that latency hides
    // behind the TMA/MMA main loop.
    const int epi = P.epilogue, act = P.act, Mrows = P.M, Ncols = P.N;
    __nv_bfloat16* __restrict__ outb = P.out_bf16;
    float* __restrict__ outf = P.out_f32 != nullptr ? P.out_f32 + int64_t(split) * P.split_stride : nullptr;
    float* __restrict__ bgrad = P.bias_grad != nullptr ? P.bias_grad + int64_t(split) * P.split_stride : nullptr;
    const __nv_bfloat16* __restrict__ auxp = P.aux;
    const float* __restrict__ auxf = P.aux_f32;
    const bool precise = P.precise != 0;
    const int ld_bf16 = P.ld_bf16, ld_f32 = P.ld_f32, ld_aux = P.ld_aux, bias_col = P.bias_col;
    const bool f32_vec = (P.ld_f32 % 4 == 0) && (P.split_stride % 4 == 0);
    const float out_scale = P.out_scale;
    const int q = warp & 3;  // TMEM lane quarter this warp may read
    const int m = m0 + q * 32 + lane;
    const bool row_ok = m < Mrows;
    // 16 accumulator columns per step (keeps the epilogue under the 102-register budget of two CTAs per SM)
    constexpr int CW = 16;
    constexpr int CHUNKS = BN / CW;
    constexpr int CH_PER_WARP = (CHUNKS + 1) / 2;
    const int c_begin = ((warp - 2) >> 2) * CH_PER_WARP;
    const int c_end = min(CHUNKS, c_begin + CH_PER_WARP);
    const bool aux_vec = (ld_aux % 8 == 0);
    // two-term fp16 mode: the operands were scaled by 2^eA and 2^eB
    const bool rescale = P.parts == 2;
    const float acc_scale = rescale ? split_unscale(__ldg(P.amax_a), __ldg(P.amax_b)) : 1.f;

    uint4 pre[2];  // prefetched 32 bytes of the dgrad's activation row for the NEXT step
    float4 pref[CW / 4];  // the same for an fp32 activation operand (64 bytes)
    const bool auxf_vec = X32 && auxf != nullptr && (ld_aux % 4 == 0);
    __nv_bfloat16* __restrict__ osplit = X32 ? P.out_split : nullptr;
    const int split_cp = P.split_cp;
    const bool f32_v8 = X32 && f32_vec && (P.ld_f32 % 8 == 0) && (P.split_stride % 8 == 0) && outf != nullptr &&
                        ((reinterpret_cast<uintptr_t>(outf) & 31u) == 0);
    auto prefetch_aux = [&](int c) {
      const int nb = n0 + c * CW;
      if (epi == TC_EPI_DGRAD && auxf == nullptr && row_ok && c < c_end && nb + CW <= Ncols && aux_vec) {
        const uint4* ap = reinterpret_cast<const uint4*>(auxp + int64_t(m) * ld_aux + nb);
        pre[0] = __ldg(ap);
        pre[1] = __ldg(ap + 1);
      }
      if (X32 && epi == TC_EPI_DGRAD && auxf_vec && row_ok && c < c_end && nb + CW <= Ncols) {
        const float4* ap = reinterpret_cast<const float4*>(auxf + int64_t(m) * ld_aux + nb);
#pragma unroll
        for (int u = 0; u < CW / 4; ++u) pref[u] = __ldg(ap + u);
      }
    };
    prefetch_aux(c_begin);
    if (has_k) {
      mbar_wait(tmem_full_bar, full_parity);
      tc_fence_after();
    }
#pragma unroll 1
    for (int c = c_begin; c < c_end; ++c) {
      uint32_t v[CW];
      if (has_k) {
        tmem_ld16(tmem_acc + (uint32_t(q * 32) << 16) + uint32_t(c * CW), v);
      } else {
#pragma unroll
        for (int j = 0; j < CW; ++j) v[j] = 0u;
      }
      if (rescale) {
#pragma unroll
        for (int j = 0; j < CW; ++j) v[j] = __float_as_uint(__uint_as_float(v[j]) * acc_scale);
      }
      const int nb = n0 + c * CW;
      const bool live = row_ok && nb < Ncols;
      const bool full = nb + CW <= Ncols;
      float h[CW];
      if (epi == TC_EPI_FWD) {
        if (live) {
          // bias of this CTA's columns was staged in shared memory once (broadcast reads, no global latency here)
#pragma unroll
          for (int u = 0; u < CW / 4; ++u) {
            const float4 t = *reinterpret_cast<const float4*>(bias_s + (nb - n0) + u * 4);
            h[u * 4] = t.x; h[u * 4 + 1] = t.y; h[u * 4 + 2] = t.z; h[u * 4 + 3] = t.w;
          }
          if (precise && (act == B200PPO_ACT_TANH || act == TC_ACT_TANH_SCALE)) {
            const float sc = act == TC_ACT_TANH_SCALE ? out_scale : 1.f;
#pragma unroll
            for (int j = 0; j < CW; ++j) h[j] = sc * tanhf(__uint_as_float(v[j]) + h[j]);
          } else if (act == B200PPO_ACT_TANH) {
#pragma unroll
            for (int j = 0; j < CW; ++j) h[j] = tanh_fast(__uint_as_float(v[j]) + h[j]);
          } else if (act == B200PPO_ACT_RELU) {
#pragma unroll
            for (int j = 0; j < CW; ++j) h[j] = fmaxf(__uint_as_float(v[j]) + h[j], 0.f);
          } else if (act == TC_ACT_TANH_SCALE) {
#pragma unroll
            for (int j = 0; j < CW; ++j) h[j] = out_scale * tanh_fast(__uint_as_float(v[j]) + h[j]);
          } else {
#pragma unroll
            for (int j = 0; j < CW; ++j) h[j] = __uint_as_float(v[j]) + h[j];
          }
        }
      } else if (epi == TC_EPI_DGRAD) {
        if (auxf != nullptr) {
          if (live) {
            const float* ap = auxf + int64_t(m) * ld_aux + nb;
            if (X32 && full && auxf_vec) {
#pragma unroll
              for (int u = 0; u < CW / 4; ++u) {
                const float4 t = pref[u];
                h[u * 4] = t.x; h[u * 4 + 1] = t.y; h[u * 4 + 2] = t.z; h[u * 4 + 3] = t.w;
              }
            } else if (full && (ld_aux % 4 == 0)) {
#pragma unroll
              for (int u = 0; u < CW / 4; ++u) {
                const float4 t = __ldg(reinterpret_cast<const float4*>(ap) + u);
                h[u * 4] = t.x; h[u * 4 + 1] = t.y; h[u * 4 + 2] = t.z; h[u * 4 + 3] = t.w;
              }
            } else {
#pragma unroll
              for (int j = 0; j < CW; ++j) h[j] = (nb + j < Ncols) ? __ldg(ap + j) : 0.f;
            }
          }
        } else if (live && full && aux_vec) {
#pragma unroll
          for (int u = 0; u < 2; ++u) {
            const uint32_t ww[4] = {pre[u].x, pre[u].y, pre[u].z, pre[u].w};
#pragma unroll
            for (int t = 0; t < 4; ++t) {
              const __nv_bfloat162 b2 = *reinterpret_cast<const __nv_bfloat162*>(&ww[t]);
              h[u * 8 + t * 2] = __low2float(b2);
              h[u * 8 + t * 2 + 1] = __high2float(b2);
            }
          }
        } else if (live) {
          const __nv_bfloat16* ap = auxp + int64_t(m) * ld_aux + nb;
#pragma unroll
          for (int j = 0; j < CW; ++j) h[j] = (nb + j < Ncols) ? __bfloat162float(ap[j]) : 0.f;
        }
        prefetch_aux(c + 1);  // next step's activation row in flight while this one is finished and stored
        if (live) {
#pragma unroll
          for (int j = 0; j < CW; ++j) {
            const float g = __uint_as_float(v[j]);
            h[j] = act == B200PPO_ACT_TANH ? g * (1.f - h[j] * h[j]) : (h[j] > 0.f ? g : 0.f);
          }
        }
      } else {
#pragma unroll
        for (int j = 0; j < CW; ++j) h[j] = __uint_as_float(v[j]);
      }
      if (!live) continue;
      if (X32 && osplit != nullptr && full) {  // (the launcher only asks for this when N is a multiple of 16)
        uint32_t w[3][CW / 2];
#pragma unroll
        for (int j = 0; j < CW; j += 2) {
          __nv_bfloat16 t[3][2];
#pragma unroll
          for (int k = 0; k < 2; ++k) {
            float r = h[j + k];
#pragma unroll
            for (int p = 0; p < 3; ++p) {
              t[p][k] = __float2bfloat16_rn(r);
              r -= __bfloat162float(t[p][k]);
            }
          }
#pragma unroll
          for (int p = 0; p < 3; ++p) w[p][j >> 1] = uint32_t(__bfloat16_as_ushort(t[p][0])) | (uint32_t(__bfloat16_as_ushort(t[p][1])) << 16);
        }
        __nv_bfloat16* sp = osplit + int64_t(m) * (3 * int64_t(split_cp)) + nb;
#pragma unroll
        for (int p = 0; p < 3; ++p)
          asm volatile("st.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(sp + int64_t(p) * split_cp), "r"(w[p][0]), "r"(w[p][1]),
                       "r"(w[p][2]), "r"(w[p][3]), "r"(w[p][4]), "r"(w[p][5]), "r"(w[p][6]), "r"(w[p][7])
                       : "memory");
      }
      if (outb != nullptr) {
        __nv_bfloat16* op = outb + int64_t(m) * ld_bf16 + nb;
        if (full && (ld_bf16 % 8 == 0)) {
#pragma unroll
          for (int u = 0; u < CW / 8; ++u)
            reinterpret_cast<uint4*>(op)[u] = make_uint4(pack_bf16(h[u * 8], h[u * 8 + 1]), pack_bf16(h[u * 8 + 2], h[u * 8 + 3]),
                                                         pack_bf16(h[u * 8 + 4], h[u * 8 + 5]), pack_bf16(h[u * 8 + 6], h[u * 8 + 7]));
        } else {
#pragma unroll
          for (int j = 0; j < CW; ++j)
            if (nb + j < Ncols) op[j] = __float2bfloat16_rn(h[j]);
        }
      }
      if (outf != nullptr) {
        const int ncols = bias_col >= 0 ? bias_col : Ncols;  // columns that belong to the matrix proper
        float* op = outf + int64_t(m) * ld_f32 + nb;
        if (X32 && nb + CW <= ncols && f32_v8) {
#pragma unroll
          for (int u = 0; u < CW / 8; ++u)
            asm volatile("st.global.v8.f32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"l"(op + u * 8), "f"(h[u * 8]), "f"(h[u * 8 + 1]),
                         "f"(h[u * 8 + 2]), "f"(h[u * 8 + 3]), "f"(h[u * 8 + 4]), "f"(h[u * 8 + 5]), "f"(h[u * 8 + 6]), "f"(h[u * 8 + 7])
                         : "memory");
        } else if (nb + CW <= ncols && f32_vec) {
#pragma unroll
          for (int u = 0; u < CW / 4; ++u) reinterpret_cast<float4*>(op)[u] = make_float4(h[u * 4], h[u * 4 + 1], h[u * 4 + 2], h[u * 4 + 3]);
        } else {
#pragma unroll
          for (int j = 0; j < CW; ++j)
            if (nb + j < ncols) op[j] = h[j];
        }
        if (bias_col >= nb && bias_col < nb + CW && bgrad != nullptr) {
          float bg = 0.f;
#pragma unroll
          for (int j = 0; j < CW; ++j)
            if (nb + j == bias_col) bg = h[j];
          bgrad[m] = bg;
        }
      }
    }
    // the terms' padding behind the last column: zeros, and the ones-column in the leading term (last N tile, the warps of
    // the upper column half, one row per thread)
    if (X32 && osplit != nullptr && row_ok && n0 + BN >= Ncols && c_end == CHUNKS) {
      __nv_bfloat16* sp = osplit + int64_t(m) * (3 * int64_t(split_cp));
      for (int pc = Ncols; pc < split_cp; pc += 16) {
#pragma unroll
        for (int p = 0; p < 3; ++p) {
          const uint32_t first = (p == 0 && pc == Ncols && P.split_ones) ? 0x00003f80u : 0u;  // bf16 1.0 in the low half
          asm volatile("st.global.v8.b32 [%0], {%1,%2,%2,%2,%2,%2,%2,%2};" ::"l"(sp + int64_t(p) * split_cp + pc), "r"(first), "r"(0u) : "memory");
        }
      }
    }
}


// Stage the bias of columns [n0, n0 + bn) into shared memory (zeros beyond N or when the problem has no bias).
__device__ __forceinline__ void tc_stage_bias(const TcProblem& P, int n0, int bn, float* bias_s, int tid, int nthreads) {
  for (int j = tid; j < bn; j += nthreads)
    bias_s[j] = (P.bias != nullptr && P.epilogue != TC_EPI_DGRAD && P.epilogue != TC_EPI_STORE && n0 + j < P.N) ? __ldg(P.bias + n0 + j) : 0.f;
}

// ---- shared-memory staged epilogue ---------------------------------------------------------------------------------
// tcgen05.ld hands every thread one accumulator ROW, so storing straight from registers makes each warp-wide store
// touch 32 different 128-byte lines (32 L1 wavefronts per instruction) — measured as THE bottleneck of the forward and
// dgrad kernels.  Instead each epilogue warp owns a 4 KB staging tile (32 rows x 128 B, 16-byte units XOR-swizzled by
// row & 7 so both the row-per-thread phase and the line-per-8-threads phase are bank-conflict free): results go
// registers -> staging -> global with every instruction writing four full 128-byte lines; the dgrad's activation
// operand comes in through the same tile the same way.
constexpr int TC_STAGE_BYTES = 4096;  // per epilogue warp

__device__ __forceinline__ uint32_t stage_off(int row, int unit) { return uint32_t(row * 128 + ((unit ^ (row & 7)) << 4)); }

// dgrad: request this warp's 32 x (BN/2) slab of the activation operand into its staging tile with cp.async (16 bytes
// per lane, 8 lanes per 128-byte line) and commit the group; nothing waits here, so the request overlaps the MMAs.
// Only for BN <= 128 (the slab is then a single 128-byte-row group).  Always commits (possibly empty) so that the
// caller's group counting stays uniform.
template <int BN>
__device__ __forceinline__ void tc_issue_aux(const TcProblem& P, int m0, int n0, int warp, int lane, uint8_t* stage, bool valid) {
  static_assert(BN <= 128, "staged dgrad needs BN <= 128");
  if (valid && P.epilogue == TC_EPI_DGRAD) {
    constexpr int WCOLS = BN / 2;
    const int q = warp & 3;
    const int mq = m0 + q * 32;
    const int nbg = n0 + ((warp - 2) >> 2) * WCOLS;
    constexpr int upr = WCOLS >> 3;
    const uint32_t sbase = smem_u32(stage);
    const __nv_bfloat16* auxp = P.aux;
    const int ld_aux = P.ld_aux;
#pragma unroll
    for (int idx = lane; idx < 32 * upr; idx += 32) {
      const int row = idx / upr, unit = idx - row * upr;
      const bool ok = mq + row < P.M && nbg + unit * 8 < P.N;
      const __nv_bfloat16* src = auxp + int64_t(ok ? mq + row : 0) * ld_aux + (ok ? nbg + unit * 8 : 0);
      const uint32_t bytes = ok ? 16u : 0u;  // src-size 0: zero fill
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(sbase + stage_off(row, unit)), "l"(src), "r"(bytes) : "memory");
    }
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
}

__device__ __forceinline__ uint32_t tanh_bf16x2(uint32_t x) {  // packed MUFU tanh on two bf16 values
  uint32_t y;
  asm("tanh.approx.bf16x2 %0, %1;" : "=r"(y) : "r"(x));
  return y;
}

// bf16-output epilogue (hidden-layer forward and dgrad) through the warp's staging tile.  BN <= 128: the warp's
// BN/2 columns are one group of <= 64 columns = one 128-byte staging row per accumulator row, and every index
// computation below is a compile-time constant or hoisted out of the loops (the first version spent ~900 warp
// instructions per tile here and was the limiter of the persistent kernel).
// TMA_OUT: the finished tile leaves through the copy engine (one cp.async.bulk.tensor store of the swizzled 32 x 64
// tile per warp, tile 1024-byte aligned) instead of 8 LDS + 8 STG per lane; the caller guards the tile's reuse with
// cp.async.bulk.wait_group.read.  Measured with profiles/mma_probe.cu: the LSU store path (32 B/clk/SM) serialises
// behind the warps that issue it, the bulk store drains in the background.
template <int BN, bool TMA_OUT = false>
__device__ __forceinline__ void tc_epilogue_staged(const TcProblem& P, int split, uint32_t tmem_acc, bool has_k, int m0, int n0,
                                                   int warp, int lane, uint64_t* tmem_full_bar, uint32_t full_parity,
                                                   uint8_t* stage, const float* bias_s, int aux_groups_in_flight,
                                                   const CUtensorMap* tm_out = nullptr) {
  static_assert(BN == 64 || BN == 128, "staged epilogue: BN <= 128");
  constexpr int WCOLS = BN / 2, STEPS = WCOLS / 16, UPR = WCOLS / 8, RSTEP = 32 / UPR;
  (void)split;
  const int epi = P.epilogue, act = P.act;
  const int q = warp & 3;
  const int mq = m0 + q * 32;
  const int col0 = ((warp - 2) >> 2) * WCOLS;
  const uint32_t sbase = smem_u32(stage);
  const uint32_t my_row = sbase + uint32_t(lane) * 128u;
  const int sw = lane & 7;
  if (epi == TC_EPI_DGRAD) {  // this tile's activation slab was requested with cp.async by tc_issue_aux
    if (aux_groups_in_flight > 0) asm volatile("cp.async.wait_group 1;" ::: "memory");
    else asm volatile("cp.async.wait_group 0;" ::: "memory");
  }
  if (has_k) {
    mbar_wait(tmem_full_bar, full_parity);
    tc_fence_after();
  }
  __syncwarp();
  const float* bs = bias_s + col0;
  // (loading the whole 64-column slab with one tcgen05.ld.x64 and a single wait was measured: no gain, +70 registers)
#pragma unroll
  for (int s = 0; s < STEPS; ++s) {
    uint32_t v[16];
    if (has_k) {
      tmem_ld16(tmem_acc + (uint32_t(q * 32) << 16) + uint32_t(col0 + s * 16), v);
    } else {
#pragma unroll
      for (int j = 0; j < 16; ++j) v[j] = 0u;
    }
    uint32_t o[8];
    if (epi == TC_EPI_FWD) {
      float z[16];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float4 t = *reinterpret_cast<const float4*>(bs + s * 16 + u * 4);
        z[u * 4] = __uint_as_float(v[u * 4]) + t.x; z[u * 4 + 1] = __uint_as_float(v[u * 4 + 1]) + t.y;
        z[u * 4 + 2] = __uint_as_float(v[u * 4 + 2]) + t.z; z[u * 4 + 3] = __uint_as_float(v[u * 4 + 3]) + t.w;
      }
      if (act == B200PPO_ACT_TANH) {
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = tanh_bf16x2(pack_bf16(z[2 * j], z[2 * j + 1]));
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j) o[j] = pack_bf16(fmaxf(z[2 * j], 0.f), fmaxf(z[2 * j + 1], 0.f));
      }
    } else {  // TC_EPI_DGRAD: dz = acc * act'(h), h from the staged activation slab (this thread's row)
      uint32_t w[8];
      lds_unit_pair(my_row, sw, s, w);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const __nv_bfloat162 b2 = *reinterpret_cast<const __nv_bfloat162*>(&w[j]);
        const float h0 = __low2float(b2), h1 = __high2float(b2);
        const float g0 = __uint_as_float(v[2 * j]), g1 = __uint_as_float(v[2 * j + 1]);
        if (act == B200PPO_ACT_TANH) o[j] = pack_bf16(g0 * (1.f - h0 * h0), g1 * (1.f - h1 * h1));
        else o[j] = pack_bf16(h0 > 0.f ? g0 : 0.f, h1 > 0.f ? g1 : 0.f);
      }
    }
    sts_unit_pair(my_row, sw, s, o);
  }
  if constexpr (TMA_OUT) {
    fence_proxy_async_smem();  // generic-proxy st.shared -> visible to the copy engine
    __syncwarp();
    if (lane == 0) {  // rows >= M and columns >= N are clipped by the tensor map
      tma_store_2d(tm_out, sbase, n0 + col0, mq);
      bulk_commit();
    }
    return;
  }
  __syncwarp();
  // staging -> global: UPR consecutive lanes write one row's 16-byte units (a full 128-byte line when UPR == 8)
  {
    const int unit = lane % UPR, row0 = lane / UPR;
    const int col = n0 + col0 + unit * 8;
    const bool col_ok = col < P.N;
    __nv_bfloat16* gp = P.out_bf16 + int64_t(mq + row0) * P.ld_bf16 + col;
    const int64_t gstep = int64_t(RSTEP) * P.ld_bf16;
    const int rows_left = P.M - mq - row0;  // this lane's rows are row0 + i*RSTEP
#pragma unroll
    for (int i = 0; i < UPR; ++i) {
      const int row = row0 + i * RSTEP;
      if (col_ok && i * RSTEP < rows_left) {
        uint32_t w0, w1, w2, w3;
        asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(w0), "=r"(w1), "=r"(w2), "=r"(w3)
                     : "r"(sbase + uint32_t(row * 128) + uint32_t((unit ^ (row & 7)) << 4)) : "memory");
        *reinterpret_cast<uint4*>(gp) = make_uint4(w0, w1, w2, w3);
      }
      gp += gstep;
    }
  }
  __syncwarp();
}

// Host-evaluated: may this problem use the staged epilogue (16-byte aligned rows and whole units inside the matrix)?
inline bool tc_can_stage(const TcProblem& p) {
  if (p.epilogue == TC_EPI_STORE) return false;  // measured: staging the fp32 split-K partials does not pay (58 vs 50 us)
  const bool out_ok = p.out_bf16 != nullptr && p.out_f32 == nullptr && p.ld_bf16 % 8 == 0 && p.N % 8 == 0 && aligned16(p.out_bf16);
  if (p.epilogue == TC_EPI_DGRAD) return out_ok && p.aux != nullptr && p.ld_aux % 8 == 0 && aligned16(p.aux);
  if (p.epilogue == TC_EPI_FWD) return out_ok && (p.act == B200PPO_ACT_TANH || p.act == B200PPO_ACT_RELU);
  return false;
}

// ---- fused PPO-loss epilogues of the output layers ---------------------------------------------------------------------
constexpr float kTcLogSqrt2Pi = 0.91893853320467274178f;

struct PpoAcc {  // per-thread running sums over the tiles a CTA processes
  float surr, hub;
  float dl[32];
  __device__ __forceinline__ void clear() {
    surr = 0.f; hub = 0.f;
#pragma unroll
    for (int j = 0; j < 32; ++j) dl[j] = 0.f;
  }
};


// sigma-derived constants of the diagonal Gaussian into shared memory: [0,32) log sigma, [32,64) 1/var, [64,96) 2 var
__device__ __forceinline__ void tc_ppo_stage_consts(const TcProblem& P, float* consts_s, int tid) {
  if (P.epilogue == TC_EPI_PPO_ACTOR && tid < 32) {
    float ls = 0.f, iv = 0.f, tv = 1.f;
    if (tid < P.ppo.act_dim) {
      const float sig = expf(__ldg(P.ppo.logstd + tid));
      const float var = sig * sig;
      ls = logf(sig); iv = 1.f / var; tv = 2.f * var;
    }
    consts_s[tid] = ls; consts_s[32 + tid] = iv; consts_s[64 + tid] = tv;
  }
}

// Request the 32 x A action slab of this warp's rows (cp.async, zero-filled past the batch) and commit the group.
__device__ __forceinline__ void tc_ppo_issue(const TcProblem& P, int m0, int warp, int lane, uint8_t* stage, bool valid) {
  if (valid && P.epilogue == TC_EPI_PPO_ACTOR) {
    const int A = P.ppo.act_dim;
    const int mq = m0 + (warp & 3) * 32;
    const int rows = min(32, P.M - mq);
    if (rows > 0) {
      const int bytes = rows * A * 4;
      const uint8_t* src = reinterpret_cast<const uint8_t*>(P.ppo.action + int64_t(mq) * A);
      const uint32_t sbase = smem_u32(stage);
      if ((reinterpret_cast<uintptr_t>(src) & 15) == 0) {
        for (int c = lane; c * 16 < bytes; c += 32) {
          const uint32_t nb = uint32_t(min(16, bytes - c * 16));
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(sbase + c * 16), "l"(src + c * 16), "r"(nb) : "memory");
        }
      } else {  // unaligned minibatch slice: plain loads
        float* dst = reinterpret_cast<float*>(stage);
        for (int i = lane; i < rows * A; i += 32) dst[i] = __ldg(P.ppo.action + int64_t(mq) * A + i);
      }
    }
  }
  asm volatile("cp.async.commit_group;" ::: "memory");
}

// One row of the actor's fused loss epilogue: log-prob of the stored action, ratio, clipped surrogate, gradient seeds
// (ppo.py:113-120 and its autograd), NC = act_dim rounded up to a multiple of 8 (columns >= act_dim are masked).
template <int NC>
__device__ __forceinline__ void tc_ppo_actor_row(const TcProblem& P, uint32_t tmem_acc, int q, bool row_ok, float old_lp, float adv,
                                                 const float* act_s, __nv_bfloat16* dz_s, const float* bias_s, const float* consts_s,
                                                 PpoAcc& acc) {
  const int A = P.ppo.act_dim, pitch = P.ppo.dz_pitch;
  float z[NC];
  {
    uint32_t v[16];
    tmem_ld16(tmem_acc + (uint32_t(q * 32) << 16), v);
#pragma unroll
    for (int j = 0; j < 16; ++j)
      if (j < NC) z[j] = __uint_as_float(v[j]);
    if constexpr (NC > 16) {
      tmem_ld16(tmem_acc + (uint32_t(q * 32) << 16) + 16u, v);
#pragma unroll
      for (int j = 0; j < NC - 16; ++j) z[16 + j] = __uint_as_float(v[j]);
    }
  }
  const float scale = P.out_scale, inv_scale = 1.f / P.out_scale;
  const bool ft = P.ppo.final_tanh != 0;
  float lp = 0.f;
#pragma unroll
  for (int j = 0; j < NC; ++j) {
    if (j < A) {
      const float pre = z[j] + bias_s[j];
      const float th = ft ? tanh_fast(pre) : pre;
      const float mean = ft ? scale * th : pre;
      const float d = act_s[j] - mean;
      lp += -(d * d) * (0.5f * consts_s[32 + j]) - consts_s[j] - kTcLogSqrt2Pi;  // -(a-mu)^2 / (2 var) - log sigma - log sqrt(2 pi)
      z[j] = d;  // keep (a - mean); tanh is recovered below as (a - d) / scale
    }
  }
  float g_lp = 0.f;
  if (row_ok) {
    const float lo = 1.f - P.ppo.clip_eps, hi = 1.f + P.ppo.clip_eps;
    const float ratio = expf(lp - old_lp);
    const float s1 = ratio * adv, s2 = fminf(fmaxf(ratio, lo), hi) * adv;
    const float w1 = s1 < s2 ? 1.f : (s1 > s2 ? 0.f : 0.5f);
    const float in_range = (ratio >= lo && ratio <= hi) ? 1.f : 0.f;
    g_lp = -(w1 * adv + (1.f - w1) * adv * in_range) * P.ppo.inv_global_batch * ratio;
    acc.surr += fminf(s1, s2);
  }
  uint32_t packed[NC / 2];
#pragma unroll
  for (int j = 0; j < NC; j += 2) {
    float dm[2];
#pragma unroll
    for (int u = 0; u < 2; ++u) {
      const int jj = j + u;
      dm[u] = 0.f;
      if (jj < A) {
        const float d = z[jj];
        const float dn = d * consts_s[32 + jj];
        float dmu = g_lp * dn;
        if (ft) {
          const float th = (act_s[jj] - d) * inv_scale;  // mean / scale
          dmu *= scale * (1.f - th * th);
        }
        dm[u] = row_ok ? dmu : 0.f;
        if (row_ok) acc.dl[jj] += g_lp * (d * dn - 1.f);
      }
    }
    packed[j >> 1] = pack_bf16(dm[0], dm[1]);
  }
  // this row's seeds: pitch % 8 == 0 bf16 values, zero beyond act_dim
  uint32_t* dzw = reinterpret_cast<uint32_t*>(dz_s);
#pragma unroll
  for (int w = 0; w < NC / 2; ++w)
    if (2 * w < pitch) dzw[w] = packed[w];
  for (int w = NC / 2; 2 * w < pitch; ++w) dzw[w] = 0u;
}

template <int BN>
__device__ __forceinline__ void tc_epilogue_ppo(const TcProblem& P, uint32_t tmem_acc, int m0, int warp, int lane,
                                                uint64_t* tmem_full_bar, uint32_t full_parity, uint8_t* stage,
                                                const float* bias_s, const float* consts_s, int groups_in_flight, PpoAcc& acc,
                                                bool worker) {
  // worker: this warp processes the tile's rows of its TMEM lane quarter (the <= 32 output columns all sit in one
  // thread).  Two warps share a lane quarter: the one-tile kernel lets the first work; the persistent kernel
  // alternates tiles between the two warp groups.
  const int q = warp & 3;
  const int mq = m0 + q * 32, m = mq + lane;
  const bool row_ok = m < P.M;
  if (groups_in_flight > 0) asm volatile("cp.async.wait_group 1;" ::: "memory");
  else asm volatile("cp.async.wait_group 0;" ::: "memory");
  // per-row scalars requested before the accumulator is awaited
  float old_lp = 0.f, adv = 0.f, tgt = 0.f;
  if (worker && row_ok) {
    if (P.epilogue == TC_EPI_PPO_ACTOR) { old_lp = __ldg(P.ppo.old_logp + m); adv = __ldg(P.ppo.advantage + m); }
    else tgt = __ldg(P.ppo.target + m);
  }
  mbar_wait(tmem_full_bar, full_parity);
  tc_fence_after();
  __syncwarp();
  if (!worker) return;
  if (P.epilogue == TC_EPI_PPO_CRITIC) {
    uint32_t v[16];
    tmem_ld16(tmem_acc + (uint32_t(q * 32) << 16), v);
    if (row_ok) {
      const float val = __uint_as_float(v[0]) + bias_s[0];
      const float e = val - tgt;
      const float ae = fabsf(e);
      acc.hub += ae < 1.f ? 0.5f * e * e : ae - 0.5f;
      const float dv = fminf(fmaxf(e, -1.f), 1.f) * P.ppo.inv_global_batch;
      const int pitch = P.ppo.dz_pitch;
      __nv_bfloat16* o = P.ppo.dz_out + int64_t(m) * pitch;
      if (pitch == 8) {
        const __nv_bfloat162 v0 = __floats2bfloat162_rn(dv, 0.f);
        *reinterpret_cast<uint4*>(o) = make_uint4(*reinterpret_cast<const uint32_t*>(&v0), 0u, 0u, 0u);
      } else {
        for (int j = 0; j < pitch; ++j) o[j] = __float2bfloat16_rn(j == 0 ? dv : 0.f);
      }
    }
    return;
  }
  // ---- actor ----
  // The per-row math below ran ~3500 instructions per row (clock64 timeline: 10-12 k cycles per tile, THE limiter of
  // this launch): all 32 possible action columns were unrolled with predicates and every column paid two IEEE divisions.
  // Now the column loop is unrolled to the next multiple of 8 of act_dim and the divisions are multiplications by the
  // reciprocals staged in shared memory (the bf16 path's 2e-2 tolerance; the fp32 path keeps true divisions).
  const int A = P.ppo.act_dim, pitch = P.ppo.dz_pitch;
  const float* act_s = reinterpret_cast<const float*>(stage) + lane * A;                         // this row's action
  __nv_bfloat16* dz_s = reinterpret_cast<__nv_bfloat16*>(stage + 32 * A * 4) + lane * pitch;   // this row's seeds
  const int nch = (A + 7) >> 3;
  if (nch <= 1) tc_ppo_actor_row<8>(P, tmem_acc, q, row_ok, old_lp, adv, act_s, dz_s, bias_s, consts_s, acc);
  else if (nch == 2) tc_ppo_actor_row<16>(P, tmem_acc, q, row_ok, old_lp, adv, act_s, dz_s, bias_s, consts_s, acc);
  else if (nch == 3) tc_ppo_actor_row<24>(P, tmem_acc, q, row_ok, old_lp, adv, act_s, dz_s, bias_s, consts_s, acc);
  else tc_ppo_actor_row<32>(P, tmem_acc, q, row_ok, old_lp, adv, act_s, dz_s, bias_s, consts_s, acc);
  __syncwarp();
  // coalesced store of the 32 x pitch bf16 seed slab (rows are adjacent in global memory)
  const int rows = min(32, P.M - mq);
  if (rows > 0) {
    const int bytes = rows * pitch * 2;  // pitch % 8 == 0: whole 16-byte chunks
    const uint32_t sbase = smem_u32(stage + 32 * A * 4);
    uint8_t* dst = reinterpret_cast<uint8_t*>(P.ppo.dz_out + int64_t(mq) * pitch);
    for (int c = lane; c * 16 < bytes; c += 32) {
      uint32_t w0, w1, w2, w3;
      asm volatile("ld.shared.v4.b32 {%0,%1,%2,%3}, [%4];" : "=r"(w0), "=r"(w1), "=r"(w2), "=r"(w3) : "r"(sbase + c * 16) : "memory");
      *reinterpret_cast<uint4*>(dst + c * 16) = make_uint4(w0, w1, w2, w3);
    }
  }
  __syncwarp();
}

// After the last tile: reduce the per-thread sums over the CTA (fixed order) and write this CTA's row of partials.
// red_s: TC_EPI_WARPS x 34 floats of shared memory.  Called by all epilogue warps.
__device__ __forceinline__ void tc_ppo_finish(const TcProblem& P, int warp, int lane, float* red_s, const PpoAcc& acc,
                                              bool all_warps_worked) {
  const int A = P.ppo.act_dim;
  const bool worker = all_warps_worked || ((warp - 2) >> 2) == 0;
  const int w = all_warps_worked ? warp - 2 : (warp & 3);
  const int n_rows = all_warps_worked ? TC_EPI_WARPS : 4;
  if (worker) {
    const float s = warp_sum(acc.surr), h = warp_sum(acc.hub);
    if (lane == 0) { red_s[w * 34] = s; red_s[w * 34 + 1] = h; }
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float d = warp_sum(j < A ? acc.dl[j] : 0.f);
      if (lane == 0) red_s[w * 34 + 2 + j] = d;
    }
  }
  asm volatile("bar.sync 1, %0;" ::"n"(TC_EPI_WARPS * 32) : "memory");  // epilogue warps only
  const int t = (warp - 2) * 32 + lane;
  if (t < 2 + A) {
    float s = 0.f;
    for (int k = 0; k < n_rows; ++k) s += red_s[k * 34 + t];
    if (P.epilogue == TC_EPI_PPO_CRITIC && t != 1) s = 0.f;
    if (P.epilogue == TC_EPI_PPO_ACTOR && t == 1) s = 0.f;
    P.ppo.partials[int64_t(blockIdx.x) * (2 + A) + t] = s;
  }
}

// 16 accumulator columns of this thread's row -> bias + activation -> 16 bf16 (8 words)
__device__ __forceinline__ void bias_act16(const uint32_t (&v)[16], const float* bs, int act, uint32_t (&o)[8]) {
  float z[16];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const float4 t = *reinterpret_cast<const float4*>(bs + u * 4);
    z[u * 4] = __uint_as_float(v[u * 4]) + t.x; z[u * 4 + 1] = __uint_as_float(v[u * 4 + 1]) + t.y;
    z[u * 4 + 2] = __uint_as_float(v[u * 4 + 2]) + t.z; z[u * 4 + 3] = __uint_as_float(v[u * 4 + 3]) + t.w;
  }
  if (act == B200PPO_ACT_TANH) {
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = tanh_bf16x2(pack_bf16(z[2 * j], z[2 * j + 1]));
  } else {
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = pack_bf16(fmaxf(z[2 * j], 0.f), fmaxf(z[2 * j + 1], 0.f));
  }
}
// ... into two swizzled 16-byte units of the row's staging line
__device__ __forceinline__ void ws2_finish16(const uint32_t (&v)[16], const float* bs, int act, uint32_t my_row, int sw, int s) {
  uint32_t o[8];
  bias_act16(v, bs, act, o);
  sts_unit_pair(my_row, sw, s, o);
}

// dz = acc * act'(h) for 16 columns of this thread's row; h: 16 bf16 activations (8 words)
__device__ __forceinline__ void act_grad16(const uint32_t (&v)[16], const uint32_t (&h)[8], int act, uint32_t (&o)[8]) {
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float h0 = __uint_as_float(h[j] << 16), h1 = __uint_as_float(h[j] & 0xFFFF0000u);
    const float g0 = __uint_as_float(v[2 * j]), g1 = __uint_as_float(v[2 * j + 1]);
    if (act == B200PPO_ACT_TANH) o[j] = pack_bf16(g0 * (1.f - h0 * h0), g1 * (1.f - h1 * h1));
    else o[j] = pack_bf16(h0 > 0.f ? g0 : 0.f, h1 > 0.f ? g1 : 0.f);
  }
}

}  // namespace b200ppo
