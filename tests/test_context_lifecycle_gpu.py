"""Context buffers that grow on demand behave like freshly allocated ones, bit for bit.

A context allocates its per-call device buffers lazily and grows them when a later call needs more rows: the shuffled
epoch buffers and the bf16 observation table of `b200ppo_train`, the host stage of `b200ppo_update_host` (both slots),
and the inference scratch of `b200ppo_rollout_step`.  Each case runs a small call first, then a larger one on the same
context, and compares the larger call with a fresh context that ran only that call from the same starting state.  The
last case creates and destroys contexts repeatedly: every call succeeds and computes the same gradients each time.
"""
import ctypes as C

import numpy as np
import pytest
import torch

from mujoco_reinforcement_learning_b200 import _lib

pytestmark = pytest.mark.gpu
DEV = "cuda"
HP = _lib.HParams(3e-4, 1e-3, 0.9, 0.999, 1e-8, 0.2, 1e-3)


def _desc(D, dims, final_tanh):
    d = _lib.MlpDesc()
    d.n_layers, d.in_dim = len(dims), D
    for i, w in enumerate(dims):
        d.dims[i] = w
    d.activation, d.final_tanh, d.out_scale = _lib.ACT_TANH, int(final_tanh), 1.0
    return d


class Ctx:
    def __init__(self, D, A, H, max_batch, precision):
        self.lib = _lib.load()
        self.D, self.A = D, A
        self.h = C.c_void_p()
        actor, critic = _desc(D, H + [A], True), _desc(D, H + [1], False)
        _lib.check(self.lib.b200ppo_create(C.byref(actor), C.byref(critic), max_batch, precision, C.byref(self.h)), "create")
        self.n_params = self.lib.b200ppo_param_count(self.h)

    def close(self):
        self.lib.b200ppo_destroy(self.h)


def _state(n_params, seed):
    g = torch.Generator().manual_seed(seed)
    params = (0.05 * torch.randn(n_params, generator=g)).to(DEV)
    m = (1e-3 * torch.randn(n_params, generator=g)).to(DEV)
    v = (1e-6 * torch.rand(n_params, generator=g)).to(DEV)
    return params, m, v, 7


def _rollout(n, D, A, seed, device=DEV):
    g = torch.Generator().manual_seed(seed)
    t = dict(obs=torch.randn(n, D, generator=g), act=torch.randn(n, A, generator=g).clamp_(-2, 2),
             logp=-float(A) + 0.1 * torch.randn(n, generator=g), adv=torch.randn(n, generator=g),
             tgt=torch.randn(n, generator=g), rew=torch.randn(n, generator=g), val=torch.randn(n, generator=g),
             nval=torch.randn(n, generator=g), term=(torch.rand(n, generator=g) < 0.05).to(torch.uint8))
    return {k: v.to(device) for k, v in t.items()}


def _perms(epochs, n, seed):
    g = torch.Generator().manual_seed(seed)
    return torch.stack([torch.randperm(n, generator=g) for _ in range(epochs)])


def _train(ctx, state, roll, perms, epochs, batch):
    params, m, v, step = (s.clone() if torch.is_tensor(s) else s for s in state)
    step_io = C.c_int64(step)
    n = roll["obs"].shape[0]
    losses = torch.zeros(epochs * (n // batch) * 2, device=DEV)
    p = _lib.ptr
    _lib.check(ctx.lib.b200ppo_train(ctx.h, p(params), p(m), p(v), C.byref(step_io), p(roll["obs"]), p(roll["act"]),
                                     p(roll["logp"]), p(roll["adv"]), p(roll["tgt"]), n, p(perms.to(DEV)), epochs, batch, 0,
                                     C.byref(HP), p(losses), _lib.stream_ptr()), "train")
    torch.cuda.synchronize()
    return params, m, v, step_io.value, losses


def _host_update(ctx, state, roll, perms, epochs, batch, n_envs, n_steps, slot):
    params, m, v, step = (s.clone() if torch.is_tensor(s) else s for s in state)
    step_io = C.c_int64(step)
    h = {k: np.ascontiguousarray(t.numpy()) for k, t in roll.items()}
    perms_h = np.ascontiguousarray(perms.numpy())
    n_loss = epochs * (n_envs * n_steps // batch) * 2
    losses = np.zeros(n_loss, dtype=np.float32)
    a = lambda x: x.ctypes.data_as(C.c_void_p)
    p = _lib.ptr
    _lib.check(ctx.lib.b200ppo_update_host_begin(ctx.h, a(h["obs"]), a(h["act"]), a(h["logp"]), a(h["rew"]), a(h["val"]),
                                                 a(h["nval"]), a(h["term"]), n_envs, n_steps, a(perms_h), epochs, slot),
               "update_host_begin")
    _lib.check(ctx.lib.b200ppo_update_host_end(ctx.h, p(params), p(m), p(v), C.byref(step_io), 0.99, 0.95, 0, 1, 1.0, batch,
                                               0, C.byref(HP), a(losses), slot, _lib.stream_ptr()), "update_host_end")
    torch.cuda.synchronize()
    return params, m, v, step_io.value, torch.from_numpy(losses)


def _assert_same(got, ref, what):
    names = ("params", "exp_avg", "exp_avg_sq", "step", "losses")
    for name, g, r in zip(names, got, ref):
        if torch.is_tensor(g):
            assert torch.equal(g, r), f"{what}: {name} differs from a fresh context"
        else:
            assert g == r, f"{what}: {name} {g} != {r}"


def test_train_grown_buffers_equal_fresh():
    """bf16: the large update needs bigger shuffle buffers and a bigger bf16 observation table (6 epochs of 4096-row
    minibatches take the table) than the small one left behind."""
    D, A, H, lb, epochs = 376, 17, [256, 256], 4096, 6
    grown, fresh = Ctx(D, A, H, lb, _lib.PREC_BF16), Ctx(D, A, H, lb, _lib.PREC_BF16)
    try:
        state = _state(grown.n_params, 0)
        small, large = _rollout(lb, D, A, 1), _rollout(3 * lb, D, A, 2)
        _train(grown, state, small, _perms(epochs, lb, 3), epochs, lb)  # throwaway copies of the state
        perms = _perms(epochs, 3 * lb, 4)
        _assert_same(_train(grown, state, large, perms, epochs, lb), _train(fresh, state, large, perms, epochs, lb),
                     "train after a smaller train")
    finally:
        grown.close()
        fresh.close()


def test_host_stage_grown_equals_fresh():
    """Both host-stage slots grow from 4 x 32 to 8 x 64 rows (and their permutation and loss buffers with them)."""
    D, A, H, batch, epochs = 24, 5, [64, 64], 64, 2
    grown, fresh = Ctx(D, A, H, 256, _lib.PREC_BF16), Ctx(D, A, H, 256, _lib.PREC_BF16)
    try:
        state = _state(grown.n_params, 10)
        for slot in (0, 1):
            small = _rollout(4 * 32, D, A, 11 + slot, "cpu")
            _host_update(grown, state, small, _perms(epochs, 4 * 32, 13), epochs, batch, 4, 32, slot)
        for slot in (0, 1):
            large = _rollout(8 * 64, D, A, 20 + slot, "cpu")
            perms = _perms(epochs, 8 * 64, 22 + slot)
            _assert_same(_host_update(grown, state, large, perms, epochs, batch, 8, 64, slot),
                         _host_update(fresh, state, large, perms, epochs, batch, 8, 64, slot), f"host update, slot {slot}")
    finally:
        grown.close()
        fresh.close()


def _rollout_step(ctx, params, obs, noise, t, T):
    n = obs.shape[0]
    bufs = [torch.full(s, float("nan"), device=DEV) for s in ((n, T, ctx.D), (n, T), (n, T), (n, T, ctx.A), (n, T))]
    p = _lib.ptr
    _lib.check(ctx.lib.b200ppo_rollout_step(ctx.h, p(params), p(obs), n, p(noise), t, T, *(p(b) for b in bufs),
                                            _lib.stream_ptr()), "rollout_step")
    torch.cuda.synchronize()
    return bufs


def test_rollout_step_grown_equals_fresh():
    """fp32: the inference scratch of the rollout step is sized on first use; more environments later reuse it."""
    D, A, H, T = 24, 5, [64, 64], 4
    grown, fresh = Ctx(D, A, H, 512, _lib.PREC_FP32), Ctx(D, A, H, 512, _lib.PREC_FP32)
    try:
        params = _state(grown.n_params, 30)[0]
        r = _rollout(512, D, A, 31)
        noise = torch.randn(512, A, generator=torch.Generator().manual_seed(32)).to(DEV)
        _rollout_step(grown, params, r["obs"][:16].contiguous(), noise[:16].contiguous(), 1, T)
        for n in (100, 512):
            obs, nz = r["obs"][:n].contiguous(), noise[:n].contiguous()
            for t in (1, T):
                got, ref = _rollout_step(grown, params, obs, nz, t, T), _rollout_step(fresh, params, obs, nz, t, T)
                for g, f in zip(got, ref):
                    assert torch.equal(g.nan_to_num(7.0), f.nan_to_num(7.0)), f"rollout step n_envs={n} t={t}"
    finally:
        grown.close()
        fresh.close()


@pytest.mark.parametrize("precision", [_lib.PREC_BF16, _lib.PREC_FP32])
def test_create_destroy_repeatedly(precision):
    D, A, H, B = 24, 5, [64, 64], 256
    r = _rollout(B, D, A, 40)
    first = None
    for _ in range(20):
        ctx = Ctx(D, A, H, B, precision)
        try:
            params = _state(ctx.n_params, 41)[0]
            grads = torch.zeros(ctx.n_params, device=DEV)
            losses = torch.zeros(2, device=DEV)
            p = _lib.ptr
            rc = ctx.lib.b200ppo_minibatch_grads(ctx.h, p(params), p(r["obs"]), p(r["act"]), p(r["logp"]), p(r["adv"]),
                                                 p(r["tgt"]), B, C.byref(HP), p(grads), p(losses), _lib.stream_ptr())
            _lib.check(rc, "minibatch_grads")
            torch.cuda.synchronize()
        finally:
            ctx.close()
        if first is None:
            first = (grads, losses)
        else:
            assert torch.equal(grads, first[0]) and torch.equal(losses, first[1])
