"""K3/K4/K6 + trainer parity through the C ABI: forward, evaluate, inference, losses, gradients,
post-Adam parameters — against the reference's own outputs (tests/golden) and the oracle."""
import numpy as np
import pytest
import torch

import mujoco_reinforcement_learning_b200 as pkg
from oracle import ppo_oracle as O
import copy

from tests._util import (RTOL_BF16, RTOL_FP32, assert_close, assert_close_l2, assert_params_close, load_golden,
                         rel_l2, sub)

pytestmark = pytest.mark.gpu
DEV = "cuda"
TRAIN_CASES = ["train_tanh64", "train_relu3", "train_tanh96"]
ACT = {"tanh": torch.nn.Tanh, "relu": torch.nn.ReLU}


def make_pair(obs_dim, act_dim, hidden, critic_hidden, activation, out_max=1.0, batch=64, epochs=1, lr=1e-4, clip=0.1,
              ent=1e-4, n_envs=1, steps=1, init=None, seed=0, max_batch=None, precision="fp32"):
    """(oracle agent on CPU, CUDA agent) holding identical parameters."""
    cfg = O.OracleConfig(obs_dim=obs_dim, act_dim=act_dim, actor_hidden=list(hidden), critic_hidden=list(critic_hidden),
                         activation=activation, output_max_value=out_max, learning_rate=lr, batch_size=batch,
                         epochs=epochs, clip_epsilon=clip, entropy_eps=ent)
    torch.manual_seed(seed)
    oracle = O.OracleAgent(cfg)
    if init is not None:
        oracle.networks.load_state_dict({k: torch.from_numpy(v) for k, v in init.items()})
    run = pkg.Run(training_config=pkg.TrainingConfig(learning_rate=lr, batch_size=batch, epochs_per_iteration=epochs),
                  ppo_config=pkg.PPOConfig(clip_epsilon=clip, entropy_eps=ent),
                  environment_config=pkg.EnvironmentConfig(maximum_timesteps=steps, num_envs=n_envs, window_length=1),
                  network_config=pkg.NetworkConfig(input_shape=obs_dim, output_shape=act_dim, output_max_value=out_max,
                                                   activation_class=ACT[activation], num_linear_layers=len(hidden),
                                                   linear_hidden_shapes=list(hidden),
                                                   critic_hidden_shapes=list(critic_hidden)),
                  gemm_precision=precision)
    agent = pkg.PPOAgent(run, max_batch=max_batch or max(batch, 1024))
    agent.networks.load_state_dict(oracle.networks.state_dict())
    assert agent.engine.params_are_bound()
    return oracle, agent, run


def from_golden(name, precision="fp32"):
    g = load_golden(name)
    B, epochs, lr, clip, ent, out_max = g["cfg"]
    init, mem = sub(g, "init/"), sub(g, "mem/")
    n_envs, steps = mem["action_log_prob"].shape
    D = init["actor.actor.first_layers.0.weight"].shape[1]
    A = init["actor.actor_logstd"].shape[0]
    oracle, agent, run = make_pair(D, A, [int(h) for h in g["hidden"]], [128, 128], str(g["activation"]), float(out_max),
                                   int(B), int(epochs), float(lr), float(clip), float(ent), n_envs, steps, init,
                                   precision=precision)
    return g, mem, oracle, agent, run


def oracle_in_float64(oracle, fm, perms, max_minibatches=None):
    """The same algorithm run in float64 from the same initial parameters: the yardstick for fp32 noise."""
    o64 = O.OracleAgent(oracle.cfg)
    o64.networks.load_state_dict(oracle.networks.state_dict())
    o64.networks.double()
    o64.optimizers = {n: torch.optim.Adam(o64.networks[n].parameters(), lr=oracle.cfg.learning_rate, foreach=False)
                      for n in ("actor", "critic")}
    O.ppo_train(o64, {k: v.double() for k, v in fm.items()}, perms, max_minibatches=max_minibatches)
    return {k: v.detach() for k, v in o64.networks.state_dict().items()}


def flat_mem(mem):
    M = mem["action_log_prob"].size
    t = lambda k, *s: torch.from_numpy(mem[k]).reshape(M, *s)
    return {"current_state": t("current_state", -1), "action": t("action", -1), "action_log_prob": t("action_log_prob"),
            "advantage": t("advantage", 1), "current_state_value_target": t("current_state_value_target", 1)}


@pytest.mark.parametrize("name", TRAIN_CASES)
def test_forward_evaluate_infer_vs_oracle(name):
    g, mem, oracle, agent, run = from_golden(name)
    fm = flat_mem(mem)
    obs, act = fm["current_state"], fm["action"]
    with torch.no_grad():
        mean_ref, std_ref = oracle.networks["actor"](obs)
        v_ref = oracle.networks["critic"](obs)
        dist = torch.distributions.Normal(mean_ref, std_ref)
        mean, std = agent.networks["actor"](obs.to(DEV))
        v = agent.get_state_value(obs.to(DEV))
    assert mean.shape == mean_ref.shape and std.shape == std_ref.shape and v.shape == v_ref.shape
    assert_close(mean, mean_ref, RTOL_FP32, "mean")
    assert_close(std, std_ref, RTOL_FP32, "std")
    assert_close(v, v_ref, RTOL_FP32, "value")
    logp, ent, val = agent.evaluate(obs.to(DEV), act.to(DEV))
    assert_close(logp, dist.log_prob(act).sum(1), RTOL_FP32, "logp")
    assert_close(ent, dist.entropy().mean(), RTOL_FP32, "entropy")
    assert_close(val, v_ref, RTOL_FP32, "value(evaluate)")
    noise = torch.randn(obs.shape[0], act.shape[1], generator=torch.Generator().manual_seed(3))
    a, lp, vv = agent.act_fused(obs.to(DEV), noise.to(DEV))
    a_ref = mean_ref + std_ref * noise
    assert_close(a, a_ref, RTOL_FP32, "sampled action")
    assert_close(lp, dist.log_prob(a_ref).sum(1), 1e-4, "rollout logp")  # (a-mean) cancellation: a few ulp of |a|
    assert_close(vv, v_ref, RTOL_FP32, "rollout value")
    a_test, _, _ = agent.act_fused(obs.to(DEV), test_phase=True)
    assert_close(a_test, mean_ref, RTOL_FP32, "test-phase action")
    act_sample, d2 = agent.act(obs.to(DEV), return_dist=True)
    assert act_sample.shape == mean_ref.shape
    assert_close(d2.log_prob(act.to(DEV)).sum(1), dist.log_prob(act).sum(1), RTOL_FP32, "dist.log_prob")


@pytest.mark.parametrize("name", TRAIN_CASES)
def test_minibatch_losses_and_gradients_vs_oracle(name):
    g, mem, oracle, agent, run = from_golden(name)
    fm = flat_mem(mem)
    idx = torch.from_numpy(g["perms"][0])[:oracle.cfg.batch_size]
    b = {k: v[idx] for k, v in fm.items()}
    al, cl, grads_ref, _, _ = O.minibatch_grads(oracle, b["current_state"], b["action"], b["action_log_prob"],
                                                b["advantage"], b["current_state_value_target"])
    eng = agent.engine
    hp = eng.hparams(1e-4, 1e-4, oracle.cfg.clip_epsilon, oracle.cfg.entropy_eps)
    losses, grads = eng.minibatch_grads(*(b[k].to(DEV) for k in ("current_state", "action", "action_log_prob", "advantage",
                                                                  "current_state_value_target")), hp)
    assert abs(losses[0].item() - al) <= RTOL_FP32 * max(1.0, abs(al))
    assert abs(losses[1].item() - cl) <= RTOL_FP32 * max(1.0, abs(cl))
    by_name = eng.grads_by_name(grads, agent.networks.named_parameters())
    assert sorted(by_name) == sorted(grads_ref)
    for k, ref in grads_ref.items():
        assert_close(by_name[k], ref, RTOL_FP32, f"grad {k}")


@pytest.mark.parametrize("name", TRAIN_CASES)
def test_autograd_facade_matches_oracle_autograd(name):
    g, mem, oracle, agent, run = from_golden(name)
    fm = flat_mem(mem)
    obs, act = fm["current_state"][:50], fm["action"][:50]
    w = torch.randn(50, act.shape[1], generator=torch.Generator().manual_seed(9))
    mean_ref, _ = oracle.networks["actor"](obs)
    v_ref = oracle.networks["critic"](obs)
    ((mean_ref * w).sum() + (v_ref ** 2).sum()).backward()
    x = obs.to(DEV).requires_grad_(True)
    mean, std = agent.networks["actor"](x)
    v = agent.get_state_value(x)
    ((mean * w.to(DEV)).sum() + (v ** 2).sum() + std.sum()).backward()
    ref = dict(oracle.networks.named_parameters())
    for n, p in agent.networks.named_parameters():
        if n == "actor.actor_logstd":
            assert_close(p.grad, 50 * p.detach().exp(), RTOL_FP32, n)
            continue
        assert_close(p.grad, ref[n].grad, RTOL_FP32, f"autograd {n}")
    assert x.grad is not None and x.grad.shape == x.shape


@pytest.mark.parametrize("name", TRAIN_CASES)
def test_train_matches_reference_outputs(name):
    """PPO.train on the CUDA path vs the REFERENCE'S OWN final state (same inputs, same permutations)."""
    g, mem, oracle, agent, run = from_golden(name)
    n_envs, steps = mem["action_log_prob"].shape
    memory = pkg.RolloutMemory({k: torch.from_numpy(v).to(DEV) for k, v in mem.items() if v.dtype != np.float64
                                or k == "reward"}, (n_envs, steps))
    algo = pkg.PPO(type("H", (), {"run": run})(), agent)
    al, cl = algo.train(memory, perms=torch.from_numpy(g["perms"]))
    final = sub(g, "final/")
    ref64 = oracle_in_float64(oracle, flat_mem(mem), [torch.from_numpy(p) for p in g["perms"]])
    for k, v in agent.networks.state_dict().items():
        assert_params_close(v, final[k], ref64[k], f"param {k}")
    for oname, opt in agent.optimizers.items():
        sd = opt.state_dict()
        assert abs(sd["param_groups"][0]["lr"] - float(g[f"opt/{oname}/lr"])) < 1e-12  # scheduler stepped once
        for pid, st in sd["state"].items():
            assert_close(st["exp_avg"], g[f"opt/{oname}/{pid}/exp_avg"], RTOL_FP32, f"{oname}/{pid}/exp_avg")
            assert_close(st["exp_avg_sq"], g[f"opt/{oname}/{pid}/exp_avg_sq"], RTOL_FP32, f"{oname}/{pid}/exp_avg_sq")
            assert float(st["step"]) == float(g[f"opt/{oname}/{pid}/step"])
    np.testing.assert_allclose([al, cl], g["logged_losses"], rtol=1e-5, atol=1e-7)


@pytest.mark.parametrize("shape", [dict(D=376, A=17, H=[256, 256], N=16, T=64, B=500),    # Humanoid dims, reference B
                                   dict(D=27, A=8, H=[256, 256], N=32, T=32, B=256),      # Ant dims
                                   dict(D=376, A=17, H=[256, 256], N=64, T=128, B=4096),  # fp32-tolerance GEMMs on the tensor cores
                                   dict(D=11, A=3, H=[64, 64], N=16, T=256, B=4096),      # Hopper config, one big batch
                                   dict(D=17, A=6, H=[64, 64], N=1, T=2048, B=500),       # HalfCheetah config
                                   # last hidden width not a multiple of 4: the separate loss kernel's fp32 seeds
                                   dict(D=11, A=3, H=[30, 18], N=16, T=64, B=512)])
def test_train_vs_oracle_on_baseline_shapes(shape):
    _train_vs_oracle(shape, terms=3)


def test_train_two_term_fp16_mode_and_its_documented_bound():
    """The opt-in two-term mode of the fp32-tolerance GEMMs (22-bit operands): losses and every weight tensor as in the
    default mode; the zero-initialised biases, whose gradients are 1000 : 1 cancelling sums, within 1e-4 of their scale
    instead of max(1e-5, 2 x the fp32 oracle's own distance to float64) — measured 5.4e-5 (DESIGN.md §3.3)."""
    _train_vs_oracle(dict(D=376, A=17, H=[256, 256], N=64, T=128, B=4096), terms=2)


def _train_vs_oracle(shape, terms):
    D, A, H, N, T, B = (shape[k] for k in "DAHNTB")
    oracle, agent, run = make_pair(D, A, H, H, "tanh", batch=B, epochs=1, n_envs=N, steps=T, seed=4, max_batch=B)
    agent.engine.set_fp32_terms(terms)
    roll = O.synthetic_rollout(N, T, D, A, seed=77)
    adv, tgt = O.calculate_advantages(roll["reward"], roll["current_state_value"], roll["next_state_value"],
                                      roll["terminated"], 0.99, 0.98)
    M = N * T
    fm = {"current_state": roll["current_state"].reshape(M, D), "action": roll["action"].reshape(M, A),
          "advantage": adv.reshape(M, 1), "current_state_value_target": tgt.reshape(M, 1)}
    with torch.no_grad():
        mean, std = oracle.networks["actor"](fm["current_state"])
        fm["action_log_prob"] = torch.distributions.Normal(mean, std).log_prob(fm["action"]).sum(1) + 0.02 * torch.randn(M)
    perms = [torch.randperm(M, generator=torch.Generator().manual_seed(8))]
    max_mb = 3
    ref64 = oracle_in_float64(oracle, fm, perms, max_mb)
    ref_losses = O.ppo_train(oracle, fm, perms, max_minibatches=max_mb)
    memory = pkg.RolloutMemory({"current_state": roll["current_state"].to(DEV), "action": roll["action"].to(DEV),
                                "action_log_prob": fm["action_log_prob"].reshape(N, T).to(DEV),
                                "advantage": adv.to(DEV), "current_state_value_target": tgt.to(DEV)}, (N, T))
    algo = pkg.PPO(type("H", (), {"run": run})(), agent)
    algo.train(memory, perms=torch.stack(perms), max_minibatches_per_epoch=max_mb)
    got = algo.last_losses.cpu().numpy()
    np.testing.assert_allclose(got, np.array(ref_losses), rtol=1e-5, atol=1e-6)
    ref_sd = oracle.networks.state_dict()
    from tests._util import rel_err
    for k, v in agent.networks.state_dict().items():
        if terms == 2 and k.endswith("bias"):
            e = rel_err(v, ref_sd[k])
            assert e <= 1e-4, f"param {k} (two-term mode): scaled max error {e:.3e}"
        else:
            assert_params_close(v, ref_sd[k], ref64[k], f"param {k}")


def test_checkpoint_round_trip_and_reference_key_names(tmp_path):
    oracle, agent, run = make_pair(12, 4, [32, 32], [32, 32], "tanh")
    run.experiment_path = str(tmp_path)
    keys = list(agent.networks.state_dict().keys())
    assert keys[0] == "actor.actor_logstd" or "actor.actor.first_layers.0.weight" in keys
    assert "critic.network.last_layer.bias" in keys and "actor.actor_logstd" in keys
    before = {k: v.clone() for k, v in agent.networks.state_dict().items()}
    agent.engine.exp_avg.normal_()
    agent.engine.adam_step = 17
    agent.save()
    opt_sd = torch.load(f"{tmp_path}/networks/0/optimizer_actor.pth")
    assert set(opt_sd) == {"state", "param_groups"} and float(opt_sd["state"][0]["step"]) == 17.0
    # the reference's stock torch.optim.Adam can load it
    ref_opt = torch.optim.Adam(oracle.networks["actor"].parameters(), lr=1e-4)
    ref_opt.load_state_dict(opt_sd)
    saved_m = [agent.engine.exp_avg[off:off + p.numel()].clone() for p, off in agent.engine.slots]
    with torch.no_grad():
        agent.engine.flat.zero_()
        agent.engine.exp_avg.zero_()
    agent.engine.adam_step = 0
    agent.load()
    for k, v in agent.networks.state_dict().items():
        assert torch.equal(v, before[k])
    assert agent.engine.params_are_bound() and agent.engine.adam_step == 17
    for (p, off), m in zip(agent.engine.slots, saved_m):
        assert torch.equal(agent.engine.exp_avg[off:off + p.numel()], m)


def test_batch_larger_than_engine_capacity_is_an_error():
    _, agent, _ = make_pair(8, 2, [16, 16], [16, 16], "tanh", max_batch=32)
    with pytest.raises(RuntimeError, match="max_batch"):
        agent.get_state_value(torch.zeros(33, 8, device=DEV))


# ---- bf16 tensor-core variant (tcgen05 GEMMs for the hidden layers): north_star tolerance 2e-2 ---------------------
@pytest.mark.parametrize("name", TRAIN_CASES)
def test_bf16_minibatch_losses_and_gradients_vs_oracle(name):
    g, mem, oracle, agent, run = from_golden(name, precision="bf16")
    fm = flat_mem(mem)
    idx = torch.from_numpy(g["perms"][0])[:oracle.cfg.batch_size]
    b = {k: v[idx] for k, v in fm.items()}
    al, cl, grads_ref, _, _ = O.minibatch_grads(oracle, b["current_state"], b["action"], b["action_log_prob"],
                                                b["advantage"], b["current_state_value_target"])
    eng = agent.engine
    hp = eng.hparams(1e-4, 1e-4, oracle.cfg.clip_epsilon, oracle.cfg.entropy_eps)
    losses, grads = eng.minibatch_grads(*(b[k].to(DEV) for k in ("current_state", "action", "action_log_prob", "advantage",
                                                                  "current_state_value_target")), hp)
    assert abs(losses[0].item() - al) <= RTOL_BF16 * max(1.0, abs(al))
    assert abs(losses[1].item() - cl) <= RTOL_BF16 * max(1.0, abs(cl))
    by_name = eng.grads_by_name(grads, agent.networks.named_parameters())
    # train_relu3 is a 32-24-16 ReLU net on a 32-row minibatch: a single ReLU gate flipped by bf16 rounding moves a
    # gradient tensor by ~1/32 of its norm, so that case gets 5e-2; the full-width ReLU case below holds 2e-2.
    tol = 5e-2 if name == "train_relu3" else RTOL_BF16
    for k, ref in grads_ref.items():
        assert_close_l2(by_name[k], ref, tol, f"bf16 grad {k}")


@pytest.mark.parametrize("shape", [dict(D=376, A=17, H=[256, 256], N=64, T=64, B=4096),
                                   dict(D=376, A=17, H=[256, 256], N=64, T=64, B=4096, act="relu"),
                                   dict(D=376, A=17, H=[256, 256], N=16, T=64, B=500),
                                   dict(D=27, A=8, H=[256, 256], N=32, T=32, B=256),
                                   dict(D=11, A=3, H=[64, 64], N=16, T=256, B=1024),
                                   # enough row tiles for the persistent kernel: the PPO loss in tc_ws_kernel's epilogue
                                   dict(D=11, A=3, H=[64, 64], N=64, T=640, B=20480),
                                   # the bench minibatch: CTA-pair forward / dgrad / wgrad kernels, fused-loss output layer
                                   dict(D=376, A=17, H=[256, 256], N=256, T=128, B=32768)])
def test_bf16_train_vs_oracle(shape):
    D, A, H, N, T, B = (shape[k] for k in "DAHNTB")
    oracle, agent, run = make_pair(D, A, H, H, shape.get("act", "tanh"), batch=B, epochs=1, n_envs=N, steps=T, seed=4,
                                   max_batch=B, precision="bf16")
    roll = O.synthetic_rollout(N, T, D, A, seed=77)
    adv, tgt = O.calculate_advantages(roll["reward"], roll["current_state_value"], roll["next_state_value"],
                                      roll["terminated"], 0.99, 0.98)
    M = N * T
    fm = {"current_state": roll["current_state"].reshape(M, D), "action": roll["action"].reshape(M, A),
          "advantage": adv.reshape(M, 1), "current_state_value_target": tgt.reshape(M, 1)}
    with torch.no_grad():
        mean, std = oracle.networks["actor"](fm["current_state"])
        fm["action_log_prob"] = torch.distributions.Normal(mean, std).log_prob(fm["action"]).sum(1) + 0.02 * torch.randn(M)
    perms = [torch.randperm(M, generator=torch.Generator().manual_seed(8))]
    max_mb = 2
    ref_losses = O.ppo_train(oracle, fm, perms, max_minibatches=max_mb)
    memory = pkg.RolloutMemory({"current_state": roll["current_state"].to(DEV), "action": roll["action"].to(DEV),
                                "action_log_prob": fm["action_log_prob"].reshape(N, T).to(DEV),
                                "advantage": adv.to(DEV), "current_state_value_target": tgt.to(DEV)}, (N, T))
    algo = pkg.PPO(type("H", (), {"run": run})(), agent)
    algo.train(memory, perms=torch.stack(perms), max_minibatches_per_epoch=max_mb)
    got = algo.last_losses.cpu().numpy()
    np.testing.assert_allclose(got, np.array(ref_losses), rtol=RTOL_BF16, atol=2e-3)
    ref_sd = oracle.networks.state_dict()
    lr, steps = oracle.cfg.learning_rate, max_mb
    print()
    for k, v in agent.networks.state_dict().items():
        e = rel_l2(v, ref_sd[k])
        print(f"  bf16 param {k:48s} rel L2 err {e:.3e}  (max |ref| {ref_sd[k].abs().max().item():.2e})")
        if ref_sd[k].abs().max().item() > 4 * lr * steps:
            assert e <= RTOL_BF16, f"bf16 param {k}: relative L2 error {e:.3e} > {RTOL_BF16:.1e}"
        else:
            # A tensor that was zero-initialised (hidden biases, network_block_creator.py:51-52) consists, after two steps,
            # of nothing but Adam's own first steps, and the first step of Adam is -lr * sign(g) whatever |g| is: every
            # entry whose gradient is smaller than the bf16 GEMMs' rounding noise has an arbitrary sign in BOTH
            # implementations.  With a fraction f of such entries the tensor's relative L2 error is ~2 sqrt(f) (measured
            # 0.05-0.3 here, f ~ 0.1-2 %) — not an arithmetic error, and bounded by the step size per entry:
            assert (v.cpu() - ref_sd[k]).abs().max().item() <= 2.0 * lr * steps * 1.001, k
    # the gradients themselves (first moments after two steps) hold north_star's 2e-2 on every tensor.  ReLU: units whose
    # pre-activation is within bf16 rounding of zero flip their gate, which switches that unit's whole per-sample gradient
    # on or off (measured 4-6e-2 on the first-layer tensors, tests/test_chain_gpu.py): 1e-1 there.
    mom_tol = 1e-1 if shape.get("act") == "relu" else RTOL_BF16
    for oname, opt in agent.optimizers.items():
        ref_state = oracle.optimizers[oname].state_dict()["state"]
        for pid, st in opt.state_dict()["state"].items():
            e = rel_l2(st["exp_avg"], ref_state[pid]["exp_avg"])
            print(f"  bf16 {oname}/{pid}/exp_avg rel L2 err {e:.3e}")
            assert e <= mom_tol, f"bf16 {oname}/{pid}/exp_avg: relative L2 error {e:.3e} > {mom_tol:.1e}"
            assert float(st["step"]) == float(ref_state[pid]["step"])


def test_checkpoint_files_move_between_implementations(tmp_path):
    """`Agent.save` / `load` (agent.py:47-72): the files written by the CUDA agent load into stock torch modules and
    `torch.optim.Adam` (the reference's side), and back into a fresh CUDA agent, without loss."""
    oracle, agent, run = make_pair(11, 3, [32, 24], [32, 24], "tanh", batch=64, epochs=1, n_envs=4, steps=32, seed=3, max_batch=128)
    run.experiment_path = str(tmp_path)
    roll = O.synthetic_rollout(4, 32, 11, 3, seed=5)
    adv, tgt = O.calculate_advantages(roll["reward"], roll["current_state_value"], roll["next_state_value"], roll["terminated"], 0.99, 0.98)
    memory = pkg.RolloutMemory({"current_state": roll["current_state"].to(DEV), "action": roll["action"].to(DEV),
                                "action_log_prob": (torch.randn(4, 32) * 0.1 - 4).to(DEV), "advantage": adv.to(DEV),
                                "current_state_value_target": tgt.to(DEV)}, (4, 32))
    pkg.PPO(type("H", (), {"run": run})(), agent).train(memory, perms=torch.randperm(128)[None])
    agent.save()
    d = tmp_path / "networks" / "0"
    assert sorted(p.name for p in d.iterdir()) == ["networks.pth", "optimizer_actor.pth", "optimizer_critic.pth"]
    # reference side: same key names, same Adam state layout
    sd = torch.load(d / "networks.pth", map_location="cpu")
    assert list(sd.keys()) == list(oracle.networks.state_dict().keys())
    oracle.networks.load_state_dict(sd)
    for name in ("actor", "critic"):
        osd = torch.load(d / f"optimizer_{name}.pth", map_location="cpu")
        oracle.optimizers[name].load_state_dict(osd)
        assert all(float(st["step"]) == 2.0 for st in oracle.optimizers[name].state_dict()["state"].values())
    # back into a fresh CUDA agent
    _, agent2, run2 = make_pair(11, 3, [32, 24], [32, 24], "tanh", batch=64, epochs=1, n_envs=4, steps=32, seed=99, max_batch=128)
    run2.experiment_path = str(tmp_path)
    agent2.load()
    assert torch.equal(agent2.engine.flat, agent.engine.flat)
    assert torch.equal(agent2.engine.exp_avg, agent.engine.exp_avg) and torch.equal(agent2.engine.exp_avg_sq, agent.engine.exp_avg_sq)
    assert agent2.engine.adam_step == agent.engine.adam_step == 2
    assert agent2.engine.params_are_bound()


def test_adam_step_count_is_shared_by_both_update_paths(tmp_path):
    """ADVICE r1: `FusedAdam.step()` (user-driven loss.backward(); opt.step()), `state_dict()`, `load_state_dict()` and the
    fused trainer must agree on ONE step count per optimiser — checked against stock `torch.optim.Adam` on the same
    gradients (bias correction restarts at t = 1 if a path loses the count)."""
    oracle, agent, run = make_pair(11, 3, [32, 24], [32, 24], "tanh", batch=64, epochs=1, n_envs=4, steps=32, seed=5, max_batch=128)
    ref_opt = {n: torch.optim.Adam(oracle.networks[n].parameters(), lr=1e-3, foreach=False) for n in ("actor", "critic")}
    for opt in agent.optimizers.values():
        opt.param_groups[0]["lr"] = 1e-3
    g = torch.Generator().manual_seed(3)
    for it in range(3):  # three manual steps of both optimisers with the same synthetic gradients
        for (_, p_ref), (_, p) in zip(oracle.networks.named_parameters(), agent.networks.named_parameters()):
            grad = torch.randn(p_ref.shape, generator=g)
            p_ref.grad = grad.clone()
            p.grad = grad.to(DEV)
        for n in ("actor", "critic"):
            ref_opt[n].step()
            agent.optimizers[n].step()
        sd = agent.optimizers["actor"].state_dict()
        assert all(float(st["step"]) == it + 1 for st in sd["state"].values())  # state_dict keeps the manual count
    assert agent.engine.adam_steps == [3, 3] and agent.engine.adam_step == 3
    for (k, p_ref), (_, p) in zip(oracle.networks.named_parameters(), agent.networks.named_parameters()):
        assert_close(p, p_ref.detach(), 1e-5, f"param {k} after manual steps")
    # one optimiser ahead of the other: the fused trainer refuses to guess
    agent.optimizers["critic"].step()
    with pytest.raises(RuntimeError, match="different Adam steps"):
        _ = agent.engine.adam_step
    ref_opt["critic"].step()
    agent.optimizers["actor"].step()
    ref_opt["actor"].step()
    # checkpoint round trip keeps the count, and the fused trainer continues from it
    sd = {n: copy.deepcopy(agent.optimizers[n].state_dict()) for n in ("actor", "critic")}
    agent.engine.adam_step = 0
    for n in ("actor", "critic"):
        agent.optimizers[n].load_state_dict(sd[n])
    assert agent.engine.adam_steps == [4, 4]
    roll = O.synthetic_rollout(4, 32, 11, 3, seed=5)
    adv, tgt = O.calculate_advantages(roll["reward"], roll["current_state_value"], roll["next_state_value"], roll["terminated"], 0.99, 0.98)
    memory = pkg.RolloutMemory({"current_state": roll["current_state"].to(DEV), "action": roll["action"].to(DEV),
                                "action_log_prob": (torch.randn(4, 32) * 0.1 - 4).to(DEV), "advantage": adv.to(DEV),
                                "current_state_value_target": tgt.to(DEV)}, (4, 32))
    pkg.PPO(type("H", (), {"run": run})(), agent).train(memory, perms=torch.randperm(128)[None])
    assert agent.engine.adam_steps == [6, 6]
    assert all(float(st["step"]) == 6.0 for st in agent.optimizers["critic"].state_dict()["state"].values())


def test_out_of_range_permutation_raises_index_error():
    """ADVICE r1: the reference's `memory[idx]` raises IndexError on a bad index (ppo.py:104); the asynchronous CUDA path
    must not train on stale shuffle-buffer rows and return OK."""
    oracle, agent, run = make_pair(11, 3, [32, 24], [32, 24], "tanh", batch=64, epochs=1, n_envs=4, steps=32, seed=7, max_batch=128)
    roll = O.synthetic_rollout(4, 32, 11, 3, seed=5)
    adv, tgt = O.calculate_advantages(roll["reward"], roll["current_state_value"], roll["next_state_value"], roll["terminated"], 0.99, 0.98)
    memory = pkg.RolloutMemory({"current_state": roll["current_state"].to(DEV), "action": roll["action"].to(DEV),
                                "action_log_prob": (torch.randn(4, 32) * 0.1 - 4).to(DEV), "advantage": adv.to(DEV),
                                "current_state_value_target": tgt.to(DEV)}, (4, 32))
    perm = torch.randperm(128)[None].clone()
    perm[0, 5] = 128  # one past the end
    algo = pkg.PPO(type("H", (), {"run": run})(), agent)
    with pytest.raises(IndexError):
        algo.train(memory, perms=perm)
    algo.train(memory, perms=torch.randperm(128)[None])  # the error word was cleared: a good call goes through


def test_default_critic_loads_a_reference_checkpoint():
    """ADVICE r1: with `critic_hidden_shapes` left at its default the critic is the reference's hard-coded 128x128 MLP
    (models/critic.py:13-14), so a state_dict written by the reference's own agent loads without a shape mismatch."""
    g = load_golden("train_tanh64")
    init = sub(g, "init/")
    D = init["actor.actor.first_layers.0.weight"].shape[1]
    A = init["actor.actor_logstd"].shape[0]
    run = pkg.Run(environment_config=pkg.EnvironmentConfig(maximum_timesteps=8, num_envs=2, window_length=1),
                  network_config=pkg.NetworkConfig(input_shape=D, output_shape=A, activation_class=torch.nn.Tanh, num_linear_layers=2,
                                                   linear_hidden_shapes=[int(h) for h in g["hidden"]]))
    agent = pkg.PPOAgent(run, max_batch=64)
    agent.networks.load_state_dict({k: torch.from_numpy(v) for k, v in init.items()})  # strict
    assert tuple(agent.networks["critic"].network.dims) == (128, 128, 1)


def _host_update(agent, roll, logp, perms, B, E, pipelined):
    """One rollout through the host-buffer entry points of the C ABI; returns the losses [E * nb, 2]."""
    import ctypes as C
    from mujoco_reinforcement_learning_b200 import _lib
    eng = agent.engine
    lib = _lib.load()
    N, T = roll["reward"].shape[0], roll["reward"].shape[1]
    host = {k: roll[k].contiguous() for k in ("current_state", "action", "reward", "current_state_value", "next_state_value")}
    term = roll["terminated"].to(torch.uint8).contiguous()
    logp, perms = logp.contiguous(), perms.contiguous()
    nb = (N * T) // B
    losses = torch.empty(E * nb, 2)
    hp = eng.hparams(1e-4, 1e-4, 0.1, 1e-4)
    step = C.c_int64(eng.adam_step)
    p = lambda t: C.c_void_p(t.data_ptr())
    if pipelined:
        _lib.check(lib.b200ppo_update_host_begin(eng._ctx, p(host["current_state"]), p(host["action"]), p(logp), p(host["reward"]),
                                                 p(host["current_state_value"]), p(host["next_state_value"]), p(term), N, T, p(perms), E, 1),
                   "b200ppo_update_host_begin")
        _lib.check(lib.b200ppo_update_host_end(eng._ctx, _lib.ptr(eng.flat), _lib.ptr(eng.exp_avg), _lib.ptr(eng.exp_avg_sq), C.byref(step),
                                               0.99, 0.98, 0, 0, 1.0, B, 0, C.byref(hp), p(losses), 1, _lib.stream_ptr()),
                   "b200ppo_update_host_end")
    else:
        _lib.check(lib.b200ppo_update_host(eng._ctx, _lib.ptr(eng.flat), _lib.ptr(eng.exp_avg), _lib.ptr(eng.exp_avg_sq), C.byref(step),
                                           p(host["current_state"]), p(host["action"]), p(logp), p(host["reward"]),
                                           p(host["current_state_value"]), p(host["next_state_value"]), p(term), N, T, 0.99, 0.98, 0, 0,
                                           1.0, p(perms), E, B, 0, C.byref(hp), p(losses), _lib.stream_ptr()), "b200ppo_update_host")
    eng.adam_step = int(step.value)
    return losses


def test_host_entry_points_match_the_oracle_and_each_other():
    """`b200ppo_update_host` and its two-call form (`_begin` / `_end`, staging set 1) from HOST buffers: same losses and
    parameters as the oracle's calculate_advantages + ppo_train (fp32, 1e-5), and bit-identical to each other."""
    N, T, D, A, B, E = 8, 32, 11, 3, 64, 2
    roll = O.synthetic_rollout(N, T, D, A, seed=21)
    g = torch.Generator().manual_seed(4)
    perms = torch.stack([torch.randperm(N * T, generator=g) for _ in range(E)])
    results = []
    for pipelined in (False, True):
        oracle, agent, run = make_pair(D, A, [32, 24], [32, 24], "tanh", batch=B, epochs=E, n_envs=N, steps=T, seed=9, max_batch=128)
        with torch.no_grad():
            mean, std = oracle.networks["actor"](roll["current_state"].reshape(N * T, D))
            logp = torch.distributions.Normal(mean, std).log_prob(roll["action"].reshape(N * T, A)).sum(1)
        losses = _host_update(agent, roll, logp, perms, B, E, pipelined)
        results.append((losses, agent.engine.flat.clone()))
        adv, tgt = O.calculate_advantages(roll["reward"], roll["current_state_value"], roll["next_state_value"], roll["terminated"], 0.99, 0.98)
        fm = {"current_state": roll["current_state"].reshape(N * T, D), "action": roll["action"].reshape(N * T, A), "action_log_prob": logp,
              "advantage": adv.reshape(-1, 1), "current_state_value_target": tgt.reshape(-1, 1)}
        ref_losses = np.array(O.ppo_train(oracle, fm, list(perms)))
        np.testing.assert_allclose(losses.numpy(), ref_losses, rtol=1e-5, atol=1e-6)
        for k, v in agent.networks.state_dict().items():
            ref = oracle.networks.state_dict()[k]
            assert (v.cpu() - ref).abs().max().item() <= 1e-5 * max(ref.abs().max().item(), 1e-3) + 2e-6, k
    assert torch.equal(results[0][0], results[1][0]) and torch.equal(results[0][1], results[1][1])
