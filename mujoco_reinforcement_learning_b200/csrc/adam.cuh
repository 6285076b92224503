// Internal interface of the fused Adam kernel (adam.cu).
#pragma once
#include "cast.cuh"
#include "common.cuh"
#include "ppo_math.cuh"

namespace b200ppo {

// Scalar factors of one Adam step, computed in double on the host like torch's Python code, then rounded
// to fp32 where ATen applies them to fp32 tensors.
struct AdamScalars {
  float one_minus_b1, b2, one_minus_b2, bc2_sqrt, eps, neg_step_size;
};

AdamScalars make_adam_scalars(double lr, double beta1, double beta2, double eps, int64_t step);

// Parameters [0, seg_split) use s0 (actor optimiser), [seg_split, n) use s1 (critic optimiser).
// grad_out (nullable) receives the summed gradient.
int launch_adam(float* params, const float* grads, int n_partials, int64_t partial_stride, float* exp_avg,
                float* exp_avg_sq, int64_t n, int64_t seg_split, const AdamScalars& s0, const AdamScalars& s1,
                float* grad_out, cudaStream_t st);

// When the loss sums come out of the fused PPO epilogues as per-CTA partials (tc_common.cuh), the kernel that consumes
// the gradients also finishes them: fixed-order sum over the CTAs, the two loss values, and d loss / d logstd.
// The operands used: partials ([n_cta][2 + act_dim]; nullptr = nothing to combine), act_dim, logstd (current actor_logstd,
// for the entropy term) and inv_global_batch.
struct LossCombine : PpoOperands {
  int n_cta = 0;
  int64_t logstd_off = 0;           // element offset of actor_logstd in the flat buffers
  float ent_coef = 0.f, rank_share = 1.f;
  float* losses_out = nullptr;      // [2]
};

// Multi-GPU without a library collective: every rank leaves its reduced gradient (+ trailing loss sums) in a buffer
// that its peers have mapped (cudaIpc over NVLink / NVSwitch), raises a flag in every peer's flag array, and the
// optimizer kernel itself waits for the G flags and sums the G buffers in rank order (identical bits on every rank)
// while applying Adam — the all-reduce, its launch and the separate reduction pass disappear from the critical path.
constexpr int kMaxPeers = 8;
constexpr int B200PPO_ERRFLAG_INDEX = 1;         // a gather met an index outside [0, n_rows)
constexpr int B200PPO_ERRFLAG_PEER_TIMEOUT = 3;  // the peer-memory gradient exchange gave up on a peer
struct PeerSrc {
  const float* src[kMaxPeers] = {};      // rank-ordered; src[rank] is the local buffer
  unsigned* flags_peer[kMaxPeers] = {};  // every rank's flag array [kMaxPeers] (slot q is written by rank q)
  unsigned* flags_local = nullptr;
  int world = 0, rank = 0;
  unsigned seq = 0;                      // value the flags must reach for this exchange
  int32_t* err = nullptr;                // raised to B200PPO_ERRFLAG_PEER_TIMEOUT when a peer does not show up in time
  long long timeout_cycles = 0;          // SM clocks to wait for a peer's flag (b200ppo_train: B200PPO_PEER_TIMEOUT_MS, default 30 s)
  float* losses_out = nullptr;           // [2] = sum over ranks of src[p][n + {0, 1}]
  // fused reduce (local_out != nullptr): the kernel's `grads` are this rank's split-K partials; it sums them into
  // local_out (= src[rank]) itself, and block 0 raises the flag once done_counter has reached done_target (every block
  // of the grid adds 1 per launch: the host passes launches * grid)
  float* local_out = nullptr;
  unsigned* done_counter = nullptr;
  unsigned done_target = 0;
};

// Same update, and in the same pass the bf16 shadow copies of the hidden/output weight matrices that the tensor-core
// GEMMs read (W and W^T, see cast.cuh) are re-emitted from the freshly updated fp32 master values: no separate cast
// launch, no second read of the parameters.  `casts.w[k].src` must point into `params`.
int launch_adam_cast(float* params, const float* grads, int n_partials, int64_t partial_stride, float* exp_avg,
                     float* exp_avg_sq, int64_t n, int64_t seg_split, const AdamScalars& s0, const AdamScalars& s1,
                     const WeightCastGroup& casts, const LossCombine& lc, cudaStream_t st, const PeerSrc* peers = nullptr);

int adam_cast_grid(int64_t n);  // blocks launch_adam_cast uses for n parameters

int launch_reduce_partials(const float* grads, int n_partials, int64_t partial_stride, int64_t n, float* out,
                           cudaStream_t st, const LossCombine* lc = nullptr);

}  // namespace b200ppo
