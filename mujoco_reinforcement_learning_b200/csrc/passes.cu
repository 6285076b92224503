// Forward / backward passes of both nets and the gradients of one minibatch, on the FFMA / three-term kernels (fp32)
// or on tcgen05 (bf16).
#include <algorithm>

#include "context.cuh"

namespace b200ppo {

// deepest of the selected nets (bit 0 actor, bit 1 critic)
static int max_layers(const b200ppo_ctx* ctx, int nets) {
  int maxL = 0;
  for (int n = 0; n < 2; ++n)
    if (nets & (1 << n)) maxL = std::max(maxL, ctx->net[n].d.n_layers);
  return maxL;
}

SplitArena* fresh_arena(const b200ppo_ctx* ctx) {
  if (ctx->arena_need <= 0) return nullptr;
  if (split_arena_reserve(ctx->arena, ctx->arena_need) != B200PPO_OK) return nullptr;
  split_arena_reset(ctx->arena);
  return &ctx->arena;
}

// ---- forward -----------------------------------------------------------------------------------------
int forward_nets(const b200ppo_ctx* ctx, const float* params, const float* x, int64_t B, int nets, float* const acts[2],
                 float* const outs[2], cudaStream_t st, bool skip_last, SplitArena* arena) {
  const int maxL = max_layers(ctx, nets);
  for (int l = 0; l < maxL; ++l) {
    GemmGroup g{};
    int64_t large_tiles = 0;
    GemmProblem probs[2];
    int np = 0;
    for (int n = 0; n < 2; ++n) {
      const Net& N = ctx->net[n];
      if (!(nets & (1 << n)) || l >= N.d.n_layers) continue;
      const bool last = (l == N.d.n_layers - 1);
      if (last && skip_last) continue;
      GemmProblem p{};
      p.A = (l == 0) ? x : acts[n] + N.act_off(l - 1, B);
      p.a_sm = N.in_dim(l); p.a_sk = 1;
      if (l == 0) p.a_bound_dev = ctx->obs_amax_ok ? ctx->obs_amax.get() : nullptr;
      else if (N.d.activation == B200PPO_ACT_TANH) p.a_bound = 1.f;  // |tanh| <= 1
      p.B = params + N.w_off[l];
      p.b_sn = N.in_dim(l); p.b_sk = 1;
      p.bias = params + N.b_off[l];
      p.C = last ? outs[n] : acts[n] + N.act_off(l, B);
      p.ldc = N.d.dims[l];
      p.M = int(B); p.N = N.d.dims[l]; p.K = N.in_dim(l);
      p.out_scale = N.d.out_scale;
      if (last) p.epilogue = N.d.final_tanh ? EPI_BIAS_TANH_SCALE : EPI_BIAS;
      else p.epilogue = N.d.activation == B200PPO_ACT_TANH ? EPI_BIAS_TANH : EPI_BIAS_RELU;
      large_tiles += int64_t((p.M + 127) / 128) * ((p.N + 127) / 128);
      if (p.N < 96) large_tiles = -(1ll << 40);
      probs[np++] = p;
    }
    if (np == 0) continue;
    const bool large = large_tiles >= (2 * num_sms()) / 3;
    for (int i = 0; i < np; ++i) gemm_group_add(g, probs[i], large ? 128 : 64, large ? 128 : 64, 1);
    if (arena != nullptr && gemm_split_applicable(g)) B2_TRY(launch_gemm_group_split(g, *arena, st));
    else B2_TRY(launch_gemm_group(g, large, st));
  }
  return B200PPO_OK;
}

static int pick_split(const b200ppo_ctx* ctx, int64_t tiles, int64_t K) {
  if (tiles <= 0) return 1;
  int64_t s = (4ll * num_sms() + tiles - 1) / tiles;
  s = std::min<int64_t>(s, std::max<int64_t>(1, K / 64));
  s = std::min<int64_t>(s, std::min(ctx->max_split, 32));
  return int(std::max<int64_t>(1, s));
}

// ---- backward ----------------------------------------------------------------------------------------
int backward_nets(b200ppo_ctx* ctx, const float* params, const float* x, int64_t B, int nets, float* const acts[2],
                  float* const dz[2], float* gpart, int* split_out, float* const grad_x[2], cudaStream_t st,
                  bool skip_last_dgrad, SplitArena* arena) {
  const int maxL = max_layers(ctx, nets);
  // dgrad chain, grouped by distance from the output (s = 0: through the output layer — done by the fused heads
  // kernel when skip_last_dgrad)
  for (int s = skip_last_dgrad ? 1 : 0; s < maxL; ++s) {
    GemmProblem probs[2];
    int np = 0;
    int64_t large_tiles = 0;
    for (int n = 0; n < 2; ++n) {
      const Net& N = ctx->net[n];
      if (!(nets & (1 << n))) continue;
      const int l = N.d.n_layers - 1 - s;
      if (l < 0) continue;
      if (l == 0 && (grad_x == nullptr || grad_x[n] == nullptr)) continue;
      GemmProblem p{};
      p.A = dz[n] + N.dz_off(l, B);
      p.a_sm = N.d.dims[l]; p.a_sk = 1;
      p.B = params + N.w_off[l];
      p.b_sn = 1; p.b_sk = N.in_dim(l);
      p.M = int(B); p.N = N.in_dim(l); p.K = N.d.dims[l];
      p.ldc = N.in_dim(l);
      if (l == 0) {
        p.C = grad_x[n];
        p.epilogue = EPI_STORE;
      } else {
        p.C = dz[n] + N.dz_off(l - 1, B);
        p.aux = acts[n] + N.act_off(l - 1, B);
        p.ld_aux = N.d.dims[l - 1];
        p.epilogue = N.d.activation == B200PPO_ACT_TANH ? EPI_DTANH : EPI_DRELU;
      }
      large_tiles += int64_t((p.M + 127) / 128) * ((p.N + 127) / 128);
      if (p.N < 96) large_tiles = -(1ll << 40);
      probs[np++] = p;
    }
    if (np == 0) continue;
    const bool large = large_tiles >= (2 * num_sms()) / 3;
    GemmGroup g{};
    for (int i = 0; i < np; ++i) gemm_group_add(g, probs[i], large ? 128 : 64, large ? 128 : 64, 1);
    if (arena != nullptr && gemm_split_applicable(g)) PROF(ctx, B200PPO_PROF_GEMM_DGRAD, st, launch_gemm_group_split(g, *arena, st));
    else PROF(ctx, B200PPO_PROF_GEMM_DGRAD, st, launch_gemm_group(g, large, st));
  }
  // every weight / bias gradient in one grouped split-K launch
  if (gpart != nullptr) {
    GemmProblem probs[kMaxGemmProblems];
    int np = 0;
    int64_t tiles = 0;
    for (int n = 0; n < 2; ++n) {
      const Net& N = ctx->net[n];
      if (!(nets & (1 << n))) continue;
      for (int l = 0; l < N.d.n_layers; ++l) {
        GemmProblem p{};
        p.A = dz[n] + N.dz_off(l, B);
        p.a_sm = 1; p.a_sk = N.d.dims[l];
        p.B = (l == 0) ? x : acts[n] + N.act_off(l - 1, B);
        p.b_sn = 1; p.b_sk = N.in_dim(l);
        if (l == 0) p.b_bound_dev = ctx->obs_amax_ok ? ctx->obs_amax.get() : nullptr;
        else if (N.d.activation == B200PPO_ACT_TANH) p.b_bound = 1.f;
        p.M = N.d.dims[l]; p.N = N.in_dim(l); p.K = int(B);
        p.C = gpart + N.w_off[l];
        p.ldc = N.in_dim(l);
        p.bias_grad = gpart + N.b_off[l];
        p.c_split_stride = ctx->n_params;
        p.epilogue = EPI_STORE;
        tiles += int64_t((p.M + 63) / 64) * ((p.N + 63) / 64);
        probs[np++] = p;
      }
    }
    int split = pick_split(ctx, tiles, B);
    GemmGroup g{};
    for (int i = 0; i < np; ++i) gemm_group_add(g, probs[i], 64, 64, split);
    if (arena != nullptr && gemm_split_applicable(g)) {
      // The tensor core truncates its fp32 accumulator after every K = 16 step (gemm_split.cu), so the number of samples one
      // accumulator sums is kept to kSplitChain: more split-K partials, which the optimizer kernel adds in fp32 (round to nearest).
      split = int(std::min<int64_t>(ctx->max_split, std::max<int64_t>(split, (B + kSplitChain - 1) / kSplitChain)));
      g = GemmGroup{};
      for (int i = 0; i < np; ++i) gemm_group_add(g, probs[i], 64, 64, split);
      PROF(ctx, B200PPO_PROF_GEMM_WGRAD, st, launch_gemm_group_split(g, *arena, st));
    } else {
      PROF(ctx, B200PPO_PROF_GEMM_WGRAD, st, launch_gemm_group(g, false, st));
    }
    if (split_out) *split_out = split;
  }
  return B200PPO_OK;
}


WeightCastGroup cast_group(const b200ppo_ctx* ctx, const float* params) {
  WeightCastGroup g = ctx->bf.casts;
  int k = 0;
  for (int n = 0; n < 2; ++n)
    for (int l = 0; l < ctx->net[n].d.n_layers; ++l) g.w[k++].src = params + ctx->net[n].w_off[l];
  return g;
}

int cast_weights(b200ppo_ctx* ctx, const float* params, cudaStream_t st) {
  return launch_cast_weights(cast_group(ctx, params), st);
}

PpoOperands ppo_operands(const b200ppo_ctx* ctx, const float* params, const b200ppo_hparams* hp, int64_t B, const float* action,
                         const float* old_logp, const float* adv, const float* tgt) {
  PpoOperands op{};
  op.logstd = params + ctx->logstd_off;
  op.action = action; op.old_logp = old_logp; op.advantage = adv; op.target = tgt;
  op.partials = ctx->loss_partials;
  op.act_dim = ctx->net[0].out_dim();
  op.final_tanh = ctx->net[0].d.final_tanh;
  op.clip_eps = hp != nullptr ? float(hp->clip_epsilon) : 0.f;
  op.inv_global_batch = 1.f / float(B * ctx->world);
  return op;
}

// forward of both nets on the tensor cores; hidden activations in bf16 (+ ones column), outputs in fp32.
// loss: the operands of the PPO loss fused into the output layers' epilogues (nullptr = plain forward); *loss_ctas is
// then set to the number of CTAs that wrote a row of loss partials.
static int forward_nets_bf16(b200ppo_ctx* ctx, const float* params, const __nv_bfloat16* xb, int64_t B,
                             float* const outs[2], cudaStream_t st, const PpoOperands* loss = nullptr, int* loss_ctas = nullptr) {
  auto& bf = ctx->bf;
  const int maxL = max_layers(ctx, 3);
  for (int l = 0; l < maxL; ++l) {
    TcGroup g{};
    int maxN = 0, maxK = 0, nets_here = 0;
    for (int n = 0; n < 2; ++n)
      if (l < ctx->net[n].d.n_layers) {
        maxN = std::max(maxN, ctx->net[n].d.dims[l]); maxK = std::max(maxK, ctx->net[n].in_dim(l)); ++nets_here;
      }
    const bool ws = tc_ws_applicable(int64_t((B + 127) / 128) * nets_here, maxN, maxK);
    const int bn = ws ? tc_ws_bn(maxN, maxK) : tc_pick_bn(int64_t((B + 127) / 128) * nets_here, maxN);
    for (int n = 0; n < 2; ++n) {
      const Net& N = ctx->net[n];
      if (l >= N.d.n_layers) continue;
      const bool last = l == N.d.n_layers - 1;
      TcProblem p{};
      p.M = int(B); p.N = N.d.dims[l]; p.K = N.in_dim(l);
      p.epilogue = TC_EPI_FWD;
      p.bias = params + N.b_off[l];
      p.bias_col = -1;
      if (last && loss != nullptr) {
        p.epilogue = n == 0 ? TC_EPI_PPO_ACTOR : TC_EPI_PPO_CRITIC;
        p.out_scale = N.d.out_scale;
        p.ppo = TcPpo{*loss, bf.dZ[n][l], bf.pitchZ[n][l]};
      } else if (last) {
        p.act = N.d.final_tanh ? TC_ACT_TANH_SCALE : TC_ACT_NONE;
        p.out_scale = N.d.out_scale;
        p.out_f32 = outs[n]; p.ld_f32 = N.d.dims[l];
      } else {
        p.act = N.d.activation;
        p.out_bf16 = bf.H[n][l]; p.ld_bf16 = bf.pitchH[n][l];
      }
      TcOperand A{l == 0 ? xb : bf.H[n][l - 1], l == 0 ? bf.pitchX : bf.pitchH[n][l - 1], 0};
      TcOperand Bop{bf.W[n][l], bf.pitchW[n][l], 0};
      B2_TRY(tc_group_add(g, p, A, Bop, bn, 1));
    }
    int grid = 0;
    // layer 0 may directly follow the optimizer (its weights are then one kernel old): only deeper layers preload W
    PROF(ctx, B200PPO_PROF_GEMM_FWD, st, ws ? launch_tc_ws(g, st, &grid, l > 0) : launch_tc_group(g, bn, st, &grid));
    if (loss != nullptr && l == maxL - 1) *loss_ctas = grid;
  }
  return B200PPO_OK;
}

// backward of both nets on the tensor cores.  bf.dZ[n][L-1] (dL/dz of the output layers, bf16) is filled on entry.
static int backward_nets_bf16(b200ppo_ctx* ctx, const __nv_bfloat16* xb, int64_t B, float* gpart, int* split_out,
                              cudaStream_t st, bool skip_dgrad = false) {
  auto& bf = ctx->bf;
  const int maxL = max_layers(ctx, 3);
  // dgrads, deepest first: dZ_{l-1} = (dZ_l W_l) * act'(H_{l-1}),  B operand = the bf16 copy of W_l read MN-major
  // (skip_dgrad: the fused chain kernel already left every dZ_l in place)
  for (int s = 0; s < (skip_dgrad ? 0 : maxL); ++s) {
    TcGroup g{};
    int maxN = 0, maxK = 0, nets_here = 0;
    for (int n = 0; n < 2; ++n) {
      const int l = ctx->net[n].d.n_layers - 1 - s;
      if (l >= 1) { maxN = std::max(maxN, ctx->net[n].in_dim(l)); maxK = std::max(maxK, ctx->net[n].d.dims[l]); ++nets_here; }
    }
    if (nets_here == 0) break;
    const bool ws = tc_ws_applicable(int64_t((B + 127) / 128) * nets_here, maxN, maxK);
    const int bn = ws ? tc_ws_bn(maxN, maxK) : tc_pick_bn(int64_t((B + 127) / 128) * nets_here, maxN);
    for (int n = 0; n < 2; ++n) {
      const Net& N = ctx->net[n];
      const int l = N.d.n_layers - 1 - s;
      if (l < 1) continue;
      TcProblem p{};
      p.M = int(B); p.N = N.in_dim(l); p.K = N.d.dims[l];
      p.epilogue = TC_EPI_DGRAD; p.act = N.d.activation;
      p.aux = bf.H[n][l - 1]; p.ld_aux = bf.pitchH[n][l - 1];
      p.out_bf16 = bf.dZ[n][l - 1]; p.ld_bf16 = bf.pitchZ[n][l - 1];
      p.bias_col = -1;
      TcOperand A{bf.dZ[n][l], bf.pitchZ[n][l], 0};
      TcOperand Bop{bf.W[n][l], bf.pitchW[n][l], 1};  // W_l is [out = K][in = N]: an MN-major operand, no transposed copy
      B2_TRY(tc_group_add(g, p, A, Bop, bn, 1));
    }
    PROF(ctx, B200PPO_PROF_GEMM_DGRAD, st, ws ? launch_tc_ws(g, st, nullptr, true) : launch_tc_group(g, bn, st));
  }
  // every weight / bias gradient: dW_l = dZ_l^T [H_{l-1} | 1], both operands MN-major, split-K over the batch.
  // N tile: the width that wastes the least padded MMA work over all problems (N = in+1 is 257 / 377 for 256 / 376
  // inputs: 192-wide tiles cover both in two tiles where 128-wide ones need three); split-K: as many splits as fill
  // ONE wave of resident CTAs — one CTA more than a wave would double the kernel's duration.
  const int n_problems = ctx->net[0].d.n_layers + ctx->net[1].d.n_layers;
  if (B >= 2048 && n_problems <= kMaxTcProblems) {
    // CTA pairs: 256 x 256 output blocks, bias gradient from a ones-tile MMA (tc_wgrad.cu)
    TcGroup g{};
    for (int n = 0; n < 2; ++n) {
      const Net& N = ctx->net[n];
      for (int l = 0; l < N.d.n_layers; ++l) {
        TcProblem p{};
        p.M = N.d.dims[l]; p.N = N.in_dim(l); p.K = int(B);
        p.epilogue = TC_EPI_STORE;
        p.out_f32 = gpart + N.w_off[l]; p.ld_f32 = N.in_dim(l); p.split_stride = ctx->n_params;
        p.bias_grad = gpart + N.b_off[l]; p.bias_col = -1;
        TcOperand A{bf.dZ[n][l], bf.pitchZ[n][l], 1};
        TcOperand Bop{l == 0 ? xb : bf.H[n][l - 1], l == 0 ? bf.pitchX : bf.pitchH[n][l - 1], 1};
        B2_TRY(tc_group_add(g, p, A, Bop, 128, 1));
      }
    }
    int split = 1;
    PROF(ctx, B200PPO_PROF_GEMM_WGRAD, st, launch_tc_wgrad2(g, ctx->max_split, st, &split));
    if (split_out) *split_out = split;
    return B200PPO_OK;
  }
  int bn = 64;
  {
    int maxN = 0;
    for (int n = 0; n < 2; ++n)
      for (int l = 0; l < ctx->net[n].d.n_layers; ++l) maxN = std::max(maxN, ctx->net[n].in_dim(l) + 1);
    if (maxN > 64) {
      int64_t best = -1;
      for (int cand : {128, 192, 256}) {
        int64_t work = 0;
        for (int n = 0; n < 2; ++n)
          for (int l = 0; l < ctx->net[n].d.n_layers; ++l)
            work += int64_t((ctx->net[n].d.dims[l] + 127) / 128) * ((ctx->net[n].in_dim(l) + 1 + cand - 1) / cand) * cand;
        if (best < 0 || work < best) { best = work; bn = cand; }
      }
    }
  }
  int64_t tiles = 0;
  for (int n = 0; n < 2; ++n)
    for (int l = 0; l < ctx->net[n].d.n_layers; ++l)
      tiles += int64_t((ctx->net[n].d.dims[l] + 127) / 128) * ((ctx->net[n].in_dim(l) + 1 + bn - 1) / bn);
  const int64_t slots = int64_t(num_sms()) * tc_ctas_per_sm(bn);
  int split = int(std::min<int64_t>(std::max<int64_t>(1, slots / std::max<int64_t>(tiles, 1)), ctx->max_split));
  split = int(std::min<int64_t>(split, (B + 63) / 64));
  if (split < 1) split = 1;
  TcGroup g{};
  for (int n = 0; n < 2; ++n) {
    const Net& N = ctx->net[n];
    for (int l = 0; l < N.d.n_layers; ++l) {
      TcProblem p{};
      p.M = N.d.dims[l]; p.N = N.in_dim(l) + 1; p.K = int(B);
      p.epilogue = TC_EPI_STORE;
      p.out_f32 = gpart + N.w_off[l]; p.ld_f32 = N.in_dim(l); p.split_stride = ctx->n_params;
      p.bias_grad = gpart + N.b_off[l]; p.bias_col = N.in_dim(l);
      TcOperand A{bf.dZ[n][l], bf.pitchZ[n][l], 1};
      TcOperand Bop{l == 0 ? xb : bf.H[n][l - 1], l == 0 ? bf.pitchX : bf.pitchH[n][l - 1], 1};
      if (g.count == kMaxTcProblems) {
        PROF(ctx, B200PPO_PROF_GEMM_WGRAD, st, launch_tc_group(g, bn, st));
        g = TcGroup{};
      }
      B2_TRY(tc_group_add(g, p, A, Bop, bn, split));
    }
  }
  PROF(ctx, B200PPO_PROF_GEMM_WGRAD, st, launch_tc_group(g, bn, st));
  if (split_out) *split_out = split;
  return B200PPO_OK;
}

// The fused chain kernel (tc_chain.cu) takes the minibatch when both nets are in -> 256 -> 256 -> out with the same
// activation (the Humanoid / Ant shapes of BASELINE.json); other shapes keep the per-layer launches.
bool chain_applicable(const b200ppo_ctx* ctx) {
  static const char* mode = getenv("B200PPO_CHAIN");  // profiling switch: "0" keeps the per-layer launches
  if (mode != nullptr && mode[0] == '0') return false;
  const Net& a = ctx->net[0];
  const Net& c = ctx->net[1];
  if (a.d.n_layers != 3 || c.d.n_layers != 3 || a.d.activation != c.d.activation || c.d.final_tanh) return false;
  if (!tc_chain_shape_ok(a.d.in_dim, a.d.dims[0], a.d.dims[1], a.out_dim())) return false;
  if (!tc_chain_shape_ok(c.d.in_dim, c.d.dims[0], c.d.dims[1], c.out_dim())) return false;
  const auto& bf = ctx->bf;
  for (int n = 0; n < 2; ++n) {
    for (int l = 0; l < 2; ++l)
      if (bf.pitchH[n][l] % 16 != 0 || bf.pitchZ[n][l] % 16 != 0) return false;
    if (bf.pitchZ[n][2] % 8 != 0 || bf.pitchZ[n][2] > 32) return false;
  }
  return int64_t(num_sms()) + 8 <= ctx->loss_partial_rows;
}

int launch_chain(b200ppo_ctx* ctx, const float* params, const __nv_bfloat16* xb, int64_t B, const float* action,
                 const float* old_logp, const float* adv, const float* tgt, const b200ppo_hparams* hp, int* loss_ctas,
                 cudaStream_t st, bool x_early, const ChainInfer* inf) {
  auto& bf = ctx->bf;
  ChainArgs a{};
  const int D = ctx->net[0].d.in_dim;
  B2_TRY(tc_make_map(&a.x, xb, D, B, bf.pitchX, TC_CHAIN_BK, 128));
  for (int n = 0; n < 2; ++n) {
    const Net& N = ctx->net[n];
    ChainNet& c = a.net[n];
    const int out = N.out_dim();
    B2_TRY(tc_make_map(&c.w1, bf.W[n][0], D, kChainHidden, bf.pitchW[n][0], TC_CHAIN_BK, 128));
    B2_TRY(tc_make_map(&c.w2k, bf.W[n][1], kChainHidden, kChainHidden, bf.pitchW[n][1], TC_CHAIN_BK, 128));
    B2_TRY(tc_make_map(&c.w2m, bf.W[n][1], kChainHidden, kChainHidden, bf.pitchW[n][1], 64, TC_CHAIN_BK));
    B2_TRY(tc_make_map(&c.w3k, bf.W[n][2], kChainHidden, out, bf.pitchW[n][2], TC_CHAIN_BK, n ? 8 : 16));
    B2_TRY(tc_make_map(&c.w3m, bf.W[n][2], kChainHidden, out, bf.pitchW[n][2], 64, n ? 16 : 32));
    B2_TRY(tc_make_map(&c.sH1, bf.H[n][0], kChainHidden, B, bf.pitchH[n][0], 64, 32));
    B2_TRY(tc_make_map(&c.sH2, bf.H[n][1], kChainHidden, B, bf.pitchH[n][1], 64, 32));
    B2_TRY(tc_make_map(&c.sZ1, bf.dZ[n][0], kChainHidden, B, bf.pitchZ[n][0], 64, 32));
    B2_TRY(tc_make_map(&c.sZ2, bf.dZ[n][1], kChainHidden, B, bf.pitchZ[n][1], 64, 32));
    c.b1 = params + N.b_off[0]; c.b2 = params + N.b_off[1]; c.b3 = params + N.b_off[2];
    c.H1 = bf.H[n][0]; c.H2 = bf.H[n][1]; c.dZ1 = bf.dZ[n][0]; c.dZ2 = bf.dZ[n][1]; c.dZ3 = bf.dZ[n][2];
    c.pH1 = bf.pitchH[n][0]; c.pH2 = bf.pitchH[n][1]; c.pZ1 = bf.pitchZ[n][0]; c.pZ2 = bf.pitchZ[n][1]; c.pZ3 = bf.pitchZ[n][2];
  }
  a.ppo = TcPpo{ppo_operands(ctx, params, hp, B, action, old_logp, adv, tgt)};
  if (inf != nullptr) {
    a.inf_noise = inf->noise; a.inf_mean = inf->mean; a.inf_value = inf->value; a.inf_action = inf->action; a.inf_logp = inf->logp;
    a.inf_ld_action = inf->ld_action > 0 ? inf->ld_action : ctx->net[0].out_dim();
    a.inf_ld_value = inf->ld_value; a.inf_ld_logp = inf->ld_logp; a.inf_value2 = inf->value2;
  }
  a.out_scale = ctx->net[0].d.out_scale;
  a.M = int(B);
  a.KB1 = (D + TC_CHAIN_BK - 1) / TC_CHAIN_BK;
  a.act = ctx->net[0].d.activation;
  a.tiles2 = int((B + 255) / 256);
  a.x_early = x_early ? 1 : 0;
  a.trace = inf != nullptr ? nullptr : g_chain_trace;
  return launch_tc_chain(a, st, loss_ctas, inf != nullptr);
}

// the separate loss kernel's arguments: losses and the logstd gradient final, dL/dz of the output layers still to be set
static LossArgs loss_args(const b200ppo_ctx* ctx, const PpoOperands& op, float* const outs[2], int64_t B, const b200ppo_hparams* hp,
                          float* losses_dev) {
  LossArgs la{op};
  la.mean = outs[0]; la.value = outs[1]; la.batch = B; la.out_scale = ctx->net[0].d.out_scale;
  la.ent_coef = float(hp->entropy_eps); la.rank_share = 1.f / float(ctx->world);
  la.ticket = ctx->ticket; la.losses = losses_dev; la.logstd_grad = ctx->gpart + ctx->logstd_off;
  return la;
}

int minibatch_fwd_bwd(b200ppo_ctx* ctx, const float* params, const float* obs, const __nv_bfloat16* obs_b, const float* action,
                      const float* old_logp, const float* adv, const float* tgt, int64_t B, const b200ppo_hparams* hp,
                      float* losses_dev, int* split_out, int* loss_ctas_out, cudaStream_t st) {
  *loss_ctas_out = 0;
  float* acts[2] = {ctx->ws_act[0], ctx->ws_act[1]};
  float* outs[2] = {ctx->ws_out[0], ctx->ws_out[1]};
  float* dz[2] = {ctx->ws_dz[0], ctx->ws_dz[1]};
  const Net& Na = ctx->net[0];
  const Net& Nc = ctx->net[1];
  const int La = Na.d.n_layers, Lc = Nc.d.n_layers;
  const PpoOperands op = ppo_operands(ctx, params, hp, B, action, old_logp, adv, tgt);
  if (ctx->precision == B200PPO_PREC_BF16) {
    // tcgen05 everywhere: forward (L launches; PPO loss fused into the output layers' epilogue), dgrads (L-1), wgrads (1)
    if (chain_applicable(ctx)) {  // one launch: forward, losses, dgrads (tc_chain.cu); then the weight gradients
      int grid = 0;
      PROF(ctx, B200PPO_PROF_GEMM_FWD, st, launch_chain(ctx, params, obs_b, B, action, old_logp, adv, tgt, hp, &grid, st, ctx->in_epoch));
      *loss_ctas_out = grid;
      return backward_nets_bf16(ctx, obs_b, B, ctx->gpart, split_out, st, true);
    }
    const bool same_depth = La == Lc;  // both output layers in the same launch
    if (same_depth && tc_ppo_fits(Na.out_dim()) && Na.out_dim() <= 32 &&
        int64_t(2 * ((B + 127) / 128) + 8) <= ctx->loss_partial_rows) {
      B2_TRY(forward_nets_bf16(ctx, params, obs_b, B, outs, st, &op, loss_ctas_out));
      return backward_nets_bf16(ctx, obs_b, B, ctx->gpart, split_out, st);
    }
    B2_TRY(forward_nets_bf16(ctx, params, obs_b, B, outs, st));
    LossArgs la = loss_args(ctx, op, outs, B, hp, losses_dev);
    la.dz_actor_bf16 = ctx->bf.dZ[0][La - 1]; la.dz_actor_pitch = ctx->bf.pitchZ[0][La - 1];
    la.dv_bf16 = ctx->bf.dZ[1][Lc - 1]; la.dv_pitch = ctx->bf.pitchZ[1][Lc - 1];
    PROF(ctx, B200PPO_PROF_LOSS, st, launch_ppo_loss(la, st));
    return backward_nets_bf16(ctx, obs_b, B, ctx->gpart, split_out, st);
  }
  const bool heads = La >= 2 && Lc >= 2 && heads_supported(Na.out_dim(), Na.d.dims[La - 2], Nc.d.dims[Lc - 2]);
  SplitArena* arena = fresh_arena(ctx);
  PROF(ctx, B200PPO_PROF_GEMM_FWD, st, forward_nets(ctx, params, obs, B, 3, acts, outs, st, heads, arena));
  if (heads) {
    HeadsArgs h{op};
    h.h_a = acts[0] + Na.act_off(La - 2, B); h.h_c = acts[1] + Nc.act_off(Lc - 2, B);
    h.w3a = params + Na.w_off[La - 1]; h.b3a = params + Na.b_off[La - 1];
    h.w3c = params + Nc.w_off[Lc - 1]; h.b3c = params + Nc.b_off[Lc - 1];
    h.batch = B; h.hid_a = Na.d.dims[La - 2]; h.hid_c = Nc.d.dims[Lc - 2];
    h.act = Na.d.activation; h.act_c = Nc.d.activation;
    h.out_scale = Na.d.out_scale; h.ent_coef = float(hp->entropy_eps); h.rank_share = 1.f / float(ctx->world);
    h.dz3_f32 = dz[0] + Na.dz_off(La - 1, B); h.dv_f32 = dz[1] + Nc.dz_off(Lc - 1, B);
    h.dz_a_f32 = dz[0] + Na.dz_off(La - 2, B); h.dz_c_f32 = dz[1] + Nc.dz_off(Lc - 2, B);
    h.ticket = ctx->ticket;
    h.losses = losses_dev; h.logstd_grad = ctx->gpart + ctx->logstd_off;
    PROF(ctx, B200PPO_PROF_LOSS, st, launch_heads(h, st));
  } else {
    LossArgs la = loss_args(ctx, op, outs, B, hp, losses_dev);
    la.dz_actor = dz[0] + Na.dz_off(La - 1, B);
    la.dv = dz[1] + Nc.dz_off(Lc - 1, B);
    PROF(ctx, B200PPO_PROF_LOSS, st, launch_ppo_loss(la, st));
  }
  return backward_nets(ctx, params, obs, B, 3, acts, dz, ctx->gpart, split_out, nullptr, st, heads, arena);
}

LossCombine make_loss_combine(const b200ppo_ctx* ctx, const float* params, int loss_ctas, int64_t B, const b200ppo_hparams* hp,
                              float* losses_out) {
  if (loss_ctas <= 0) return LossCombine{};
  LossCombine lc{ppo_operands(ctx, params, hp, B, nullptr, nullptr, nullptr, nullptr)};
  lc.n_cta = loss_ctas;
  lc.logstd_off = ctx->logstd_off;
  lc.ent_coef = float(hp->entropy_eps);
  lc.rank_share = 1.f / float(ctx->world);
  lc.losses_out = losses_out;
  return lc;
}

}  // namespace b200ppo
