"""The update after the forward / dgrad kernels, pinned exactly: weight gradients, one optimizer step, whole epochs.

The oracle comparisons (2e-2 relative L2 for the bf16 variant) cannot see a bug that moves a tensor by less than that —
a skipped or stale bf16 weight copy costs one Adam step (~1e-3 of the tensor at lr 1e-4), one dropped minibatch row of
4097 about 1.6e-2.  The three parts here chain together and each has an exact or near-exact reference instead:

1. weight / bias gradients of a bf16 minibatch against float64 of the very operands the weight-gradient kernel read
   (the bf16 observations, and the bf16 H_l / dL/dz_l the chain or per-layer kernels left behind);
2. one optimizer step of `train` (Adam + bf16 re-cast + loss finish) against float64 Adam from the saved state and the
   gradient `minibatch_grads` returns for the same rows — the same kernels, so the same bits;
3. a multi-epoch `train` call (bf16 observation table, epoch-ahead gather on the side stream, bf16 weight copies
   re-emitted by the optimizer) bit for bit equal to the same minibatches run as single-step `train` calls, none of
   which takes the table or the overlap and each of which casts fresh weights.
"""
import numpy as np
import pytest
import torch

from mujoco_reinforcement_learning_b200 import _lib
from tests.test_update_gpu import make_pair

pytestmark = pytest.mark.gpu
DEV = "cuda"
HUMANOID = dict(D=376, A=17, H=[256, 256], C=[256, 256])


def _rows(oracle, M, seed):
    """M synthetic minibatch rows on the GPU; old log-probs within a few percent of the policy's (ratios near 1, so the
    surrogate's gradient is not clipped away)."""
    D, A = oracle.cfg.obs_dim, oracle.cfg.act_dim
    g = torch.Generator().manual_seed(seed)
    obs = torch.randn(M, D, generator=g)
    action = torch.randn(M, A, generator=g).clamp_(-3, 3)
    adv = torch.randn(M, generator=g)
    tgt = torch.randn(M, generator=g)
    with torch.no_grad():
        mean, std = oracle.networks["actor"](obs)
        logp = torch.distributions.Normal(mean, std).log_prob(action).sum(1) + 0.05 * torch.randn(M, generator=g)
    return [t.to(DEV) for t in (obs, action, logp, adv, tgt)]


def _slot_mask(eng):
    """True on the flat-buffer elements that belong to a parameter tensor, False on the padding between tensors."""
    mask = torch.zeros(eng.n_params, dtype=torch.bool)
    for p, off in eng.slots:
        mask[off:off + p.numel()] = True
    return mask


# ---- part 1: weight gradients against float64 of their own operands --------------------------------------------------
#
# Both weight-gradient kernels multiply the same bf16 operands float64 multiplies here; what differs is the tensor core's
# fp32 accumulator, which truncates, and the fp32 sum of the split-K partials.  `test_tc_gemm_gpu.py` holds 2e-5 of
# max |C| for random operands at K = 4096 rows per partial, and the largest partial here is ~3700 rows (B = 33000 cut
# in 9): the weights get that 2e-5 of max |ref|.  A bias entry is a row sum of dZ, its truncation error grows with the
# partial sums it passes through, ~sqrt(K) / 16 steps of 2^-23 of sum |dZ| (~5e-7 at K = 4096): 2e-6 of sum |dZ|.
# Measured on a B200 (1000 W): at most 4.6e-6 (weights, B = 33000) and 7.6e-8 (biases).  A lost row costs about
# 1 / sqrt(B) of a weight tensor and 1 / B of a bias entry's magnitude sum (2.4e-4 at B = 4097).
W_TOL, B_TOL = 2e-5, 2e-6


def _wgrad_refs(agent, obs, B):
    """{name: (kind, float64 reference, scale)} for every weight and bias of both nets, from the operands the weight-
    gradient launch of the last bf16 minibatch read: dW_l = dZ_l^T A_{l-1}, db_l = sum over rows of dZ_l."""
    eng = agent.engine
    name_of = {id(p): k for k, p in agent.networks.named_parameters()}
    refs = {}
    for net, block in ((0, agent.networks["actor"].actor), (1, agent.networks["critic"].network)):
        a_prev = obs.bfloat16().double()  # what the observation cast (round to nearest) hands the kernels
        for l, lin in enumerate(block.linears()):
            dz = eng.debug_activations(net, 1, l, B).double()
            ref_w = dz.T @ a_prev
            refs[name_of[id(lin.weight)]] = ("w", ref_w, ref_w.abs().max())
            refs[name_of[id(lin.bias)]] = ("b", dz.sum(0), dz.abs().sum(0).clamp_min(1e-30))
            if l + 1 < len(block.dims):
                a_prev = eng.debug_activations(net, 0, l, B).double()
    return refs


def _check_wgrad(agent, data, B, tag):
    eng = agent.engine
    hp = eng.hparams(1e-4, 1e-4, 0.1, 1e-4)
    obs, action, logp, adv, tgt = (t[:B] for t in data)
    _, grads = eng.minibatch_grads(obs, action, logp, adv, tgt, hp)
    torch.cuda.synchronize()
    assert torch.isfinite(grads).all(), tag
    by_name = eng.grads_by_name(grads, agent.networks.named_parameters())
    bad = []
    print()
    for name, (kind, ref, scale) in _wgrad_refs(agent, obs, B).items():
        e = ((by_name[name].double() - ref).abs() / scale).max().item()
        tol = W_TOL if kind == "w" else B_TOL
        print(f"  {tag:16s} {name:42s} {'max err / max |ref|' if kind == 'w' else 'max err / sum |dZ|'} {e:.2e}")
        if not e <= tol:
            bad.append((tag, name, e))
    return bad


def test_wgrad_humanoid_every_path_and_ragged_batch():
    """One context, minibatches from the bench size down: 33000 / 32768 rows (bench minibatch, ragged at that scale), 4097
    and 2500 (the CTA-pair kernel's last k-tile holds 1 / 196 rows: TMA's zero fill along the batch), 2048 (first size on
    the CTA-pair kernel), 1000 (one-tile kernel, bias from the ones-column).  Going down means the activation buffers
    still hold the previous, larger minibatch's rows past B: a kernel that reads past its batch meets nonzero rows."""
    sizes = (33000, 32768, 4097, 2500, 2048, 1000)
    s = HUMANOID
    oracle, agent, _ = make_pair(s["D"], s["A"], s["H"], s["C"], "tanh", batch=max(sizes), max_batch=max(sizes),
                                 precision="bf16", seed=11)
    bad = []
    for B in sizes:
        bad += _check_wgrad(agent, _rows(oracle, B, seed=B), B, f"humanoid B{B}")
    assert not bad, bad


WGRAD_SHAPES = [
    dict(D=27, A=8, H=[256, 256], C=[256, 256], B=2500),        # Ant: odd observation width, ones-column at 27
    dict(D=376, A=24, H=[256, 256], C=[256, 256], B=2500),      # widest action row the chain kernel takes
    dict(D=376, A=1, H=[256, 256], C=[256, 256], B=2500),       # narrowest
    dict(D=11, A=3, H=[64, 64], C=[64, 64], B=4097),            # per-layer launches with the fused PPO epilogue
    dict(D=376, A=17, H=[256, 192, 128], C=[128, 64], B=2500),  # 7 layer problems: one-tile kernel in two launches
]


@pytest.mark.parametrize("shape", WGRAD_SHAPES, ids=lambda s: "-".join(f"{k}{v}" for k, v in s.items() if k != "C") + f"-C{s['C']}")
def test_wgrad_matches_float64_of_its_operands(shape):
    B = shape["B"]
    oracle, agent, _ = make_pair(shape["D"], shape["A"], shape["H"], shape["C"], "tanh", batch=B, max_batch=B,
                                 precision="bf16", seed=12)
    bad = _check_wgrad(agent, _rows(oracle, B, seed=7), B, "B" + str(B))
    assert not bad, bad


# ---- part 2: one optimizer step against float64 Adam -------------------------------------------------------------------
def _ulp32(x):
    """Spacing of the float32 grid at |x| (x float64 on the CPU)."""
    return torch.from_numpy(np.spacing(np.abs(x.float().numpy()))).double()


@pytest.mark.parametrize("start", ["trained", "step1000"])
@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_one_train_step_is_float64_adam_of_minibatch_grads(precision, start):
    """`train` over one minibatch whose rows `minibatch_grads` already differentiated: the gradient is the same bits
    (same kernels, same split, the partials summed in index order by both), so the new moments and parameters are Adam
    of that gradient — checked per element against float64 from a state that is not the first step (after three trained
    minibatches, or at step 1000), with random moments and different actor / critic learning rates, so that the split
    at the actor's last tensor (actor_logstd, right before the critic's first weight) is checked too.  bf16: the fused
    Adam + re-cast + loss-finish kernel; fp32: the plain Adam kernel of the trainer."""
    s, B = HUMANOID, 2048
    M = 3 * B + 1000
    oracle, agent, _ = make_pair(s["D"], s["A"], s["H"], s["C"], "tanh", batch=B, max_batch=B, precision=precision, seed=13)
    eng = agent.engine
    data = _rows(oracle, M, seed=31)
    gen = torch.Generator().manual_seed(32)
    if start == "trained":
        eng.train(*data, torch.randperm(M, generator=gen)[None].to(DEV), batch=B, hp=eng.hparams(1e-3, 1e-3, 0.1, 1e-4))
        assert eng.adam_step == 3
    else:
        eng.adam_step = 1000
    lr_a, lr_c = 1e-3, 3e-3
    hp = eng.hparams(lr_a, lr_c, 0.1, 1e-4)
    perm = torch.randperm(M, generator=gen)
    rows = perm[:B].to(DEV)
    losses_g, g = eng.minibatch_grads(*(t[rows] for t in data), hp)
    torch.cuda.synchronize()
    mask = _slot_mask(eng)
    g = g.cpu()
    assert torch.isfinite(g[mask]).all()
    with torch.no_grad():  # moments of the scale of each tensor's gradient; the padding between tensors stays 0
        m0, v0 = torch.zeros(eng.n_params), torch.zeros(eng.n_params)
        for p, off in eng.slots:
            n = p.numel()
            rms = g[off:off + n].square().mean().sqrt().clamp_min(1e-12)
            m0[off:off + n] = rms * torch.randn(n, generator=gen)
            v0[off:off + n] = (rms * torch.randn(n, generator=gen)).square()
        eng.exp_avg.copy_(m0)
        eng.exp_avg_sq.copy_(v0)
    theta0, t0 = eng.flat.cpu(), eng.adam_step
    assert theta0[~mask].eq(0).all()
    losses_t = eng.train(*data, perm[None].to(DEV), batch=B, hp=hp, max_minibatches_per_epoch=1)
    assert eng.adam_step == t0 + 1
    assert losses_t.shape == (1, 2) and torch.equal(losses_t[0], losses_g), (losses_t, losses_g)
    theta1, m1, v1 = eng.flat.cpu(), eng.exp_avg.cpu(), eng.exp_avg_sq.cpu()
    # nothing but zeros in the padding (a 0 / (0 + eps) there would be fine, a NaN from an unwritten gradient not)
    for name, t in (("param", theta1), ("exp_avg", m1), ("exp_avg_sq", v1)):
        assert t[~mask].eq(0).all(), f"{name}: padding between tensors changed"
    b1, b2, eps, t = 0.9, 0.999, 1e-8, t0 + 1
    g64, m64, v64, th64 = g.double(), m0.double(), v0.double(), theta0.double()
    # adam.cu adam_update: m' = m + (1 - b1)(g - m);  v' = b2 v + (1 - b2) g g;  p' = p - lr/bc1 * m' / (sqrt(v')/sqrt(bc2) + eps)
    m_ref = m64 + (1 - b1) * (g64 - m64)
    v_ref = b2 * v64 + (1 - b2) * g64 * g64
    # fp32 roundings: m' three (the last scales with |m'|, the subtraction, the product and fp32(1 - b1) with (1 - b1)|g - m|,
    # which exceeds |m'| where g - m and m cancel); v' four of non-negative terms plus the fp32 constants — about one ulp
    # of m' and two of v'
    bound_m = 2.0 ** -23 * (m_ref.abs() + 2 * (1 - b1) * (g64 - m64).abs()) * 1.01 + 1e-45
    bound_v = 2.0 ** -22 * v_ref * 1.01 + 1e-45
    # the parameter from the kernel's own fp32 moments (just checked): the step's chain of roundings (sqrt, two divides,
    # + eps, * step size, the fp32 scalars) stays within 1e-6 of it, and the final add rounds to one ulp of p'
    lr = torch.where(torch.arange(eng.n_params) < eng.n_actor, lr_a, lr_c).double()
    step = lr / (1 - b1 ** t) * m1.double() / (v1.double().sqrt() / (1 - b2 ** t) ** 0.5 + eps)
    th_ref = th64 - step
    bound_th = _ulp32(th_ref) + 1e-6 * step.abs()
    report = []
    for name, got, ref, bound in (("exp_avg", m1, m_ref, bound_m), ("exp_avg_sq", v1, v_ref, bound_v),
                                  ("param", theta1, th_ref, bound_th)):
        err = (got.double() - ref).abs()
        over = (err > bound) & mask
        worst = (err / bound)[mask].max().item()
        print(f"  {precision} {start} {name:10s} max err / bound {worst:.2f}")
        if over.any():
            i = int(over.nonzero()[0])
            report.append((name, int(over.sum()), i, got[i].item(), ref[i].item()))
    assert not report, report
    # the step moved every tensor (a learning rate of 0 or a skipped segment would pass the checks above only if ref = p)
    for p, off in eng.slots:
        assert not torch.equal(theta1[off:off + p.numel()], theta0[off:off + p.numel()])


# ---- part 3: a multi-epoch call is its single-minibatch steps, bit for bit ---------------------------------------------
COMPOSE_CASES = [
    # Humanoid, 6 epochs of 4 x 4096: the bf16 observation table + byte-copy gather (b200ppo_train converts the whole
    # rollout once when that moves fewer bytes — five or more epochs at this shape), epoch-ahead gather on the side stream
    dict(D=376, A=17, H=[256, 256], B=4096, nb=4, E=6, precision="bf16", table=True),
    # Ant: W1 is 27 wide, so the optimizer re-emits its bf16 copy element by element (no table at 3 epochs)
    dict(D=27, A=8, H=[256, 256], B=4096, nb=3, E=3, precision="bf16", table=False),
    # Hopper widths: per-layer launches with the fused PPO epilogue, one-tile weight gradient
    dict(D=11, A=3, H=[64, 64], B=1024, nb=3, E=3, precision="bf16", table=False),
    # fp32 context: the plain Adam kernel and the fp32 epoch-ahead gather
    dict(D=376, A=17, H=[256, 256], B=4096, nb=4, E=3, precision="fp32", table=None),
]


@pytest.mark.parametrize("case", COMPOSE_CASES, ids=lambda c: f"D{c['D']}-A{c['A']}-H{c['H'][0]}-B{c['B']}-E{c['E']}-{c['precision']}")
def test_multi_epoch_train_equals_single_minibatch_calls(case):
    """One `train` call over E epochs of nb minibatches against E * nb calls with one minibatch each, whose permutation
    starts with that minibatch's rows (lr 1e-3: a step large enough to change many bf16 weight copies).  The single calls
    gather straight from the fp32 observations on the caller's stream and cast every weight afresh, so equal losses,
    parameters, moments and step count show that the long call's observation table gives the direct gather's bits, that
    its side-stream gather into two buffer sets is race-free, that the bf16 copies the optimizer re-emits are a fresh
    cast, and that the chain kernel's early observation prefetch within an epoch changes nothing.  The first differing
    loss tells where to look: minibatch 0 of epoch 0 the table / gather, minibatch 0 of a later epoch the buffer sets and
    their events, a later minibatch the re-emitted weights or the early prefetch."""
    D, A, H, B, nb, E, precision = (case[k] for k in ("D", "A", "H", "B", "nb", "E", "precision"))
    M = nb * B + 1000  # the tail is dropped every epoch
    agents = []
    for _ in range(3 if case["table"] else 2):
        oracle, agent, _ = make_pair(D, A, H, H, "tanh", batch=B, max_batch=B, precision=precision, seed=17)
        agents.append(agent)
    data = _rows(oracle, M, seed=41)
    gen = torch.Generator().manual_seed(42)
    perms = torch.stack([torch.randperm(M, generator=gen) for _ in range(E)])
    lib = _lib.load()
    hp = agents[0].engine.hparams(1e-3, 1e-3, 0.1, 1e-4)
    long_eng, short_eng = agents[0].engine, agents[1].engine

    n0 = lib.b200ppo_launch_count()
    long_losses = long_eng.train(*data, perms.to(DEV), batch=B, hp=hp)
    torch.cuda.synchronize()
    long_launches = lib.b200ppo_launch_count() - n0
    assert long_eng.adam_step == E * nb

    short_losses, short_launches = [], []
    for e in range(E):
        for i in range(nb):
            head = perms[e, i * B:(i + 1) * B]
            perm = torch.cat([head, perms[e, :i * B], perms[e, (i + 1) * B:]])
            n0 = lib.b200ppo_launch_count()
            short_losses.append(short_eng.train(*data, perm[None].to(DEV), batch=B, hp=hp, max_minibatches_per_epoch=1))
            torch.cuda.synchronize()
            short_launches.append(lib.b200ppo_launch_count() - n0)
    short_losses = torch.cat(short_losses)

    diff = (long_losses != short_losses).any(1).nonzero()
    first = None if len(diff) == 0 else divmod(int(diff[0]), nb)
    assert first is None, f"losses differ first at (epoch, minibatch) {first}: {long_losses[diff[0]]} vs {short_losses[diff[0]]}"
    assert long_eng.adam_step == short_eng.adam_step == E * nb
    for name in ("flat", "exp_avg", "exp_avg_sq"):
        a, b = getattr(long_eng, name), getattr(short_eng, name)
        assert torch.equal(a, b), f"{name}: {int((a != b).sum())} elements differ"

    if case["table"] is not None:
        # launches: a single call is (weight cast, gather, k per minibatch); the long call one weight cast, E gathers,
        # E * nb minibatches — and the conversion of the rollout into the bf16 table when it takes that path
        assert len(set(short_launches)) == 1, short_launches
        k = short_launches[0] - 2
        table_launches = long_launches - (1 + E + E * nb * k)
        assert table_launches == (1 if case["table"] else 0), (long_launches, short_launches[0])

    if case["table"]:
        # one GPU: the rank-sliced permutation layout ([E, nb, B], only the slots this rank consumes) gives the same bits
        sliced_eng = agents[2].engine
        sliced = perms[:, :nb * B].reshape(E, nb, B)
        sliced_losses = sliced_eng.train(*data, sliced.to(DEV), batch=B, hp=hp, rank_sliced_perms=True)
        assert torch.equal(sliced_losses, long_losses)
        for name in ("flat", "exp_avg", "exp_avg_sq"):
            assert torch.equal(getattr(sliced_eng, name), getattr(long_eng, name)), name
