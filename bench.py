#!/usr/bin/env python
"""PPO-update benchmark on the Humanoid shape (BASELINE.json metric/config), one JSON line on stdout.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A *step* is one PPO iteration's update over one synthetic rollout: the advantage pipeline
(`PPO.calculate_advantages`) followed by `epochs` epochs of permutation-gather + minibatch
forward/loss/backward/Adam (`PPO.train`).  `value` = samples pushed through the update per second with the
rollout already resident in HBM; `e2e` = the same through the C-ABI host-buffer entry point
(`b200ppo_update_host`: pinned host rollout -> device, update, losses -> host).  With N GPUs every rank owns a
slab of `envs` environments (weak scaling): the slabs are all-gathered after the GAE scan, every rank takes its
1/N slice of every global minibatch (global permutation, as the reference indexes), gradients are summed by an
NCCL all-reduce per minibatch.

`--impl reference` times the reference's OWN `PPO.calculate_advantages` + `PPO.train` (staged verbatim under
`oracle/_ref` by `oracle/build_ref.py`, run behind `oracle/shims.py`) on the host cores, on a bounded sample of the same
workload with the GPU arm's step definition; without `oracle/_ref` it falls back to the oracle port
(`oracle/ppo_oracle.py`, `kind: "port"`).  `--scaling strong` keeps the TOTAL problem at `--envs` environments and
`--minibatch` rows (each of N ranks owns 1/N of both) instead of the default weak scaling.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries exactly ONE JSON line.  Libraries write there too (NCCL prints its version banner on stdout when the
# environment says NCCL_DEBUG=VERSION, which is left as the launcher set it): file descriptor 1 is pointed at stderr for
# the run and the JSON line goes to the saved original.
_JSON_FD = os.dup(1)
os.dup2(2, 1)


def emit(line: dict):
    os.write(_JSON_FD, (json.dumps(line) + "\n").encode())


OBS_DIM, ACT_DIM, HIDDEN = 376, 17, [256, 256]
TRAFFIC_BF16_B32768 = 294.4e6  # 123.4 MB (tc_chain_kernel) + 171.0 MB (tc_wgrad2_kernel), profiles/r02_ncu_chain_wgrad_B32768.csv


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return {"hbm": d["hbm_gbs"], "tensor_burst": d["bf16_tflops"], "tensor_sustained": d["bf16_tflops_sustained"],
                "source": "measured"}
    return {"hbm": 6650.0, "tensor_burst": 1590.0, "tensor_sustained": 1400.0, "source": "fallback"}


class ClockSampler:
    """nvidia-smi sampling of SM clocks and throttle reasons during the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        if len(self.rows) < 3:  # very short timed region: make sure a few samples land while the GPU is still warm
            time.sleep(0.35)
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for n, v in zip(names, r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_rollout(n_envs, steps, seed):
    from oracle.ppo_oracle import synthetic_rollout  # synthetic-input generator only (shared with the tests)
    return synthetic_rollout(n_envs, steps, OBS_DIM, ACT_DIM, seed=seed)


def flops_per_sample():
    macs = 0
    for out in (ACT_DIM, 1):
        dims = [OBS_DIM] + HIDDEN + [out]
        macs += sum(a * b for a, b in zip(dims[:-1], dims[1:]))
    first = 2 * OBS_DIM * HIDDEN[0]  # no dgrad into the observations (two nets)
    return {"fwd": 2 * macs, "dgrad": 2 * macs - 2 * first, "wgrad": 2 * macs, "total": 6 * macs - 2 * first}


# ------------------------------------------------------------------------------------------------------
class CpuArm:
    """The reference's CPU path on the host cores with the GPU arm's step definition: ONE advantage pass per step,
    amortised over E epochs, and epochs of (randperm + gather of every leaf + all minibatches).  Runs the reference's
    OWN code from `oracle/_ref` (kind "reference") or, where that is not staged, the oracle port (kind "port").
    The reference's `train` (ppo.py:93-154) only runs whole epochs, so `n_ep` full epochs are timed per step and the
    advantage pass is charged pro rata:  samples/s = n_ep * nb * B / (t_train + t_gae * n_ep / E)."""

    def __init__(self, envs, T, B, E):
        from oracle import build_ref
        self.envs, self.T, self.B, self.E = envs, T, B, E
        self.M, self.nb = envs * T, envs * T // B
        self.cores = os.cpu_count() or 1
        torch.set_num_threads(self.cores)
        roll = dict(make_rollout(envs, T, 1234 + 3))
        roll["current_state"] = roll["current_state"].reshape(envs, T, OBS_DIM)
        roll["action_log_prob"] = torch.zeros(envs, T)
        self.roll = roll
        if build_ref.available():
            from oracle.ref_runner import ReferencePPO
            self.ref = ReferencePPO(OBS_DIM, ACT_DIM, HIDDEN, B, 1, envs, T)
            self.kind = "reference"
            self.what = ("the reference's own PPO.calculate_advantages + PPO.train from oracle/_ref (verbatim sources behind "
                         "oracle/shims.py; its Critic hard-codes 128x128 hidden layers, models/critic.py:13-14, so this arm does "
                         "LESS arithmetic than the 256x256 GPU arm)")
        else:
            from oracle import ppo_oracle as O
            torch.manual_seed(0)
            self.O = O
            self.agent = O.OracleAgent(O.OracleConfig(obs_dim=OBS_DIM, act_dim=ACT_DIM, actor_hidden=HIDDEN, critic_hidden=HIDDEN,
                                                      batch_size=B, epochs=1))
            self.kind = "port"
            self.what = "oracle port of the reference path (oracle/ppo_oracle.py: the reference's torch CPU operators; oracle/_ref is not staged here)"

    def gae(self):
        r = self.roll
        if self.kind == "reference":
            mem = self.ref.memory(r)
            self.ref.calculate_advantages(mem)
            return mem
        adv, tgt = self.O.calculate_advantages(r["reward"], r["current_state_value"], r["next_state_value"], r["terminated"], 0.99, 0.98)
        return {"advantage": adv, "current_state_value_target": tgt}

    def train(self, mem, epochs, n_envs=None, batch=None):
        n_envs, batch = n_envs or self.envs, batch or self.B
        T, r = self.T, self.roll
        if self.kind == "reference":
            if n_envs != self.envs:
                mem = self.ref.TensorDict({k: mem[k][:n_envs] for k in mem.keys()}, batch_size=(n_envs, T))
            self.ref.run.environment_config.num_envs = n_envs
            self.ref.run.training_config.batch_size = batch
            self.ref.train(mem, epochs=epochs)
            return
        m = n_envs * T
        fm = {"current_state": r["current_state"].reshape(self.M, OBS_DIM)[:m], "action": r["action"].reshape(self.M, ACT_DIM)[:m],
              "action_log_prob": r["action_log_prob"].reshape(self.M)[:m], "advantage": mem["advantage"].reshape(self.M, 1)[:m],
              "current_state_value_target": mem["current_state_value_target"].reshape(self.M, 1)[:m]}
        self.agent.cfg.batch_size = batch
        self.O.ppo_train(self.agent, fm, [torch.randperm(m) for _ in range(epochs)])

    def warm_up(self):
        n = max(1, min(self.envs, (2 * self.B + self.T - 1) // self.T))  # two minibatches of one epoch
        self.train(self.gae(), 1, n)

    def timed_step(self, n_ep):
        t0 = time.perf_counter()
        mem = self.gae()
        t_gae = time.perf_counter() - t0
        t0 = time.perf_counter()
        self.train(mem, n_ep)
        t_train = time.perf_counter() - t0
        return t_gae, t_train, mem

    def describe(self, t_gae, t_train, n_ep):
        return (f"{self.what}; {self.cores} threads; per step: one advantage pass over {self.envs}x{self.T} ({t_gae * 1e3:.0f} ms, "
                f"charged {n_ep}/{self.E}) + {n_ep} full epoch(s) of randperm + gather of every leaf + all {self.nb} minibatches "
                f"of {self.B} ({t_train / n_ep * 1e3:.0f} ms per epoch)")

    def b500(self, mem):
        """The same code at the reference's default batch_size = 500 (main.py:44): 64 minibatches of one epoch."""
        n = max(1, min(self.envs, 64 * 500 // self.T))
        self.train(mem, 1, n, 500)  # warm-up of the small shapes
        t0 = time.perf_counter()
        self.train(mem, 1, n, 500)
        dt = time.perf_counter() - t0
        return (n * self.T // 500) * 500 / dt, f"{n * self.T // 500} minibatches of 500 (one epoch over {n} environments), same code"


def run_reference(args, config):
    """CPU arm (rank 0 only).  Every timed step is the bounded sample CpuArm.timed_step describes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    arm = CpuArm(args.envs, args.rollout_steps, args.minibatch, args.epochs)
    arm.warm_up()
    t_gae, t_train, mem = arm.timed_step(1)  # also sizes the sample: epochs per step within the budget
    n_ep = max(1, min(args.epochs, args.ref_epochs, int(args.ref_budget / max(t_train, 1e-3))))
    vals = []
    for k in range(args.steps):
        t_gae, t_train, mem = arm.timed_step(n_ep)
        vals.append(n_ep * arm.nb * arm.B / (t_train + t_gae * n_ep / arm.E))
    value = sum(vals) / len(vals)
    cb = {"value": value, "unit": "samples/s", "cores": arm.cores, "kind": arm.kind, "sample": arm.describe(t_gae, t_train, n_ep),
          "gae_GBps": 21 * arm.M / 1e9 / t_gae}
    if arm.B != 500:
        cb["value_B500"], cb["sample_B500"] = arm.b500(mem)
    samples_per_step = arm.E * arm.nb * arm.B
    line = {"impl": "reference", "metric": "ppo_update_samples_per_sec", "value": value, "unit": "samples/s", "n_gpus": args.gpus,
            "steps": len(vals), "warmup": args.warmup, "ms_per_step": samples_per_step / value * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config, "cpu_baseline": cb,
            "e2e": {"value": value, "unit": "samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "per_step_values": vals, "ms_per_step_note": "time of a full step (1 advantage pass + all epochs) at the measured rate"}
    emit(line)


# ------------------------------------------------------------------------------------------------------
def cuda_time(fn, iters, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(iters):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(); fn(); b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return statistics.median(ts), min(ts)


GAE_BYTES = 21  # read r, V, V' (12) + terminated (1), write advantage + target (8); `done` is implied (SURVEY §8d: 22 with it)


def c5_sweep(pk, world=1, rank=0):
    """BASELINE.json configs[4]: GAE / gather bandwidth over 256-65536 envs x 64-1024 steps.  With N ranks every rank owns
    1/N of the environments (env-slab sharding, no communication): time = max over ranks, bytes = all ranks'."""
    import mujoco_reinforcement_learning_b200 as pkg
    import torch.distributed as dist
    dev = torch.device("cuda", torch.cuda.current_device())
    pts = []
    for n, t in ((256, 64), (1024, 128), (4096, 128), (16384, 256), (65536, 256), (65536, 1024)):
        nl = max(1, n // world)
        r, v, vn = (torch.randn(nl, t, 1, device=dev) for _ in range(3))
        term = torch.rand(nl, t, device=dev) < 0.01
        med, _ = cuda_time(lambda: pkg.calculate_advantages(r, v, vn, term, 0.99, 0.98), 10)
        del r, v, vn, term
        m = min(nl * t, 4 * 1024 * 1024)  # the gather's tables are 1.5 KB per row: at most 4 M rows (13 GB in + out) per rank
        obs, act, s1 = torch.randn(m, OBS_DIM, device=dev), torch.randn(m, ACT_DIM, device=dev), torch.randn(m, device=dev)
        idx = torch.randperm(m, device=dev)
        medg, _ = cuda_time(lambda: pkg.gather_minibatch(idx, obs, act, s1, s1, s1, check=False), 5 if m > 2e6 else 10)
        if world > 1:
            tt = torch.tensor([med, medg], device=dev)
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            med, medg = float(tt[0]), float(tt[1])
        gby = GAE_BYTES * nl * t * world
        gaby = (2 * (4 * OBS_DIM + 4 * ACT_DIM + 12) + 8) * m * world
        l2 = (gby / world) < 100e6
        pts.append({"envs": n, "steps": t, "n_gpus": world, "gae_ms": med, "gae_GBps": gby / 1e9 / (med * 1e-3),
                    "gae_frac_hbm": gby / 1e9 / (med * 1e-3) / (pk["hbm"] * world),
                    "gather_rows_per_gpu": m, "gather_ms": medg, "gather_GBps": gaby / 1e9 / (medg * 1e-3),
                    "gather_frac_hbm": gaby / 1e9 / (medg * 1e-3) / (pk["hbm"] * world),
                    "note": "GAE working set fits L2" if l2 else ""})
        del obs, act, s1, idx
        torch.cuda.empty_cache()
    return pts


def k6_latency(agent, n_envs):
    """Rollout inference (ppo.py:20-29: V(s), pi(s) sample, log-prob) for one environment step of `n_envs` environments."""
    dev = torch.device("cuda", torch.cuda.current_device())
    obs = torch.randn(n_envs, OBS_DIM, device=dev)
    noise = torch.randn(n_envs, ACT_DIM, device=dev)
    med, best = cuda_time(lambda: agent.act_fused(obs, noise=noise), 50, warm=5)
    # the same C-ABI call with preallocated outputs, 100 calls back to back between two events: what the GPU needs per
    # environment step once the Python wrapper (four allocations per call) is out of the way
    from mujoco_reinforcement_learning_b200 import _lib
    eng = agent.engine
    lib = _lib.load()
    mean = torch.empty(n_envs, ACT_DIM, device=dev)
    action, logp, value = torch.empty_like(mean), torch.empty(n_envs, device=dev), torch.empty(n_envs, 1, device=dev)
    args = (eng._ctx, _lib.ptr(eng.flat), _lib.ptr(obs), n_envs, _lib.ptr(noise), _lib.ptr(mean), _lib.ptr(value), _lib.ptr(action),
            _lib.ptr(logp), _lib.stream_ptr())
    launches0 = lib.b200ppo_launch_count()
    _lib.check(lib.b200ppo_policy_infer(*args), "b200ppo_policy_infer")
    launches = lib.b200ppo_launch_count() - launches0
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(100):
        lib.b200ppo_policy_infer(*args)
    e1.record()
    torch.cuda.synchronize()
    us_infer = e0.elapsed_time(e1) * 10.0
    # the rollout's own entry point: the same step written straight into the [N, T, ...] buffers (state copy included), V(s') of
    # step t - 1 taken from step t's critic evaluation — what replaces ppo.py:20-49's three MLP calls per environment step
    Tb = 16
    buf = {"current_state": torch.empty(n_envs, Tb, OBS_DIM, device=dev), "current_state_value": torch.empty(n_envs, Tb, 1, device=dev),
           "next_state_value": torch.empty(n_envs, Tb, 1, device=dev), "action": torch.empty(n_envs, Tb, ACT_DIM, device=dev),
           "action_log_prob": torch.empty(n_envs, Tb, device=dev)}
    for t in range(Tb):
        eng.rollout_step(obs, noise, t, buf)
    torch.cuda.synchronize()
    launches0 = lib.b200ppo_launch_count()
    e0.record()
    for rep in range(8):
        for t in range(Tb):
            eng.rollout_step(obs, noise, t, buf)
    e1.record()
    torch.cuda.synchronize()
    us_step = e0.elapsed_time(e1) * 1e3 / (8 * Tb)
    step_launches = (lib.b200ppo_launch_count() - launches0) / (8 * Tb)
    return {"envs": n_envs, "us_per_env_step_batch": med * 1e3, "best_us": best * 1e3,
            "us_c_abi_back_to_back": us_infer, "launches_per_call": int(launches),
            "rollout_step": {"us": us_step, "launches": step_launches,
                             "api": "ActorCriticEngine.rollout_step -> b200ppo_rollout_step: s_t, V(s_t), a_t, log pi(a_t) into slice [:, t] of "
                                    "the rollout buffers and V(s_t) as next_state_value[:, t - 1]"},
            "api": "PPOAgent.act_fused -> b200ppo_policy_infer (actor + critic forward, sample, log-prob); bf16 context: weights and "
                   "observations to bf16 + the forward-only instance of tc_chain_kernel"}


def hbm_kernel_lines(pk):
    """Roofline of the HBM-bound kernels at sizes that do not fit the 126 MB L2 (SURVEY.md §8d cache caveat)."""
    import mujoco_reinforcement_learning_b200 as pkg
    out = {}
    dev = "cuda"
    # K1 at the sweep's large end: 65536 envs x 1024 steps = 1.48 GB algorithmic
    n, t = 65536, 1024
    r, v, vn = (torch.randn(n, t, 1, device=dev) for _ in range(3))
    term = torch.rand(n, t, device=dev) < 0.01
    med, best = cuda_time(lambda: pkg.calculate_advantages(r, v, vn, term, 0.99, 0.98), 10)
    # 21 B per (env, step): PPO.calculate_advantages derives `done` from `terminated` (ppo.py:70-72), the kernel reads no done array
    gb = GAE_BYTES * n * t / 1e9
    out["gae_65536x1024"] = {"bytes": GAE_BYTES * n * t, "ms": med, "GBps": gb / (med * 1e-3), "frac": gb / (med * 1e-3) / pk["hbm"]}
    medn, _ = cuda_time(lambda: pkg.calculate_advantages(r, v, vn, term, 0.99, 0.98, normalize_advantage=True), 5)
    out["gae_65536x1024_normalized"] = {"bytes": GAE_BYTES * n * t, "ms": medn, "GBps": gb / (medn * 1e-3), "frac": gb / (medn * 1e-3) / pk["hbm"]}
    del r, v, vn, term
    out["c5_sweep"] = c5_sweep(pk)
    # K1 at the Humanoid shape (11.5 MB: L2 resident, reported as time)
    n, t = 4096, 128
    r, v, vn = (torch.randn(n, t, 1, device=dev) for _ in range(3))
    term = torch.rand(n, t, device=dev) < 0.01
    med, best = cuda_time(lambda: pkg.calculate_advantages(r, v, vn, term, 0.99, 0.98), 20)
    out["gae_4096x128"] = {"bytes": GAE_BYTES * n * t, "ms": med, "GBps": GAE_BYTES * n * t / 1e9 / (med * 1e-3), "note": "L2-resident (11 MB)"}
    del r, v, vn, term
    # K2: one epoch's gather at the Humanoid shape, 1.665 GB algorithmic
    m = 4096 * 128
    obs, act = torch.randn(m, OBS_DIM, device=dev), torch.randn(m, ACT_DIM, device=dev)
    s = torch.randn(m, device=dev)
    idx = torch.randperm(m, device=dev)
    med, best = cuda_time(lambda: pkg.gather_minibatch(idx, obs, act, s, s, s, check=False), 10)
    by = (2 * (4 * OBS_DIM + 4 * ACT_DIM + 12) + 8) * m
    out["gather_epoch_524288"] = {"bytes": by, "ms": med, "GBps": by / 1e9 / (med * 1e-3), "frac": by / 1e9 / (med * 1e-3) / pk["hbm"]}
    ident = torch.arange(m, device=dev)
    med2, _ = cuda_time(lambda: pkg.gather_minibatch(ident, obs, act, s, s, s, check=False), 10)
    out["gather_epoch_524288_identity_idx"] = {"bytes": by, "ms": med2, "GBps": by / 1e9 / (med2 * 1e-3), "frac": by / 1e9 / (med2 * 1e-3) / pk["hbm"],
                                               "note": "same kernel, idx = arange: isolates the cost of the random 1504-byte row reads"}
    del obs, act, s, idx, ident
    # K5 on a 64M-parameter vector (1.79 GB) and on the real 329k-parameter set
    for n_par, key in ((64 * 1024 * 1024, "adam_64M"), (329251, "adam_329k")):
        p, g, mm, vv = (torch.randn(n_par, device=dev) for _ in range(4))
        vv.abs_()
        med, best = cuda_time(lambda: pkg.adam_step_(p, g, mm, vv, 10, 1e-4), 10)
        by = 28 * n_par
        out[key] = {"bytes": by, "ms": med, "GBps": by / 1e9 / (med * 1e-3)}
        if n_par > 10 ** 7:
            out[key]["frac"] = out[key]["GBps"] / pk["hbm"]
        else:
            out[key]["note"] = "L2-resident (9.2 MB): launch/latency bound"
        del p, g, mm, vv
    # SURVEY 8f rank 4 (SAC update step): the Polyak average as an HBM kernel (12 B/param) and one SoftActorCritic.train call
    n_par = 64 * 1024 * 1024
    tgt, src = torch.randn(n_par, device=dev), torch.randn(n_par, device=dev)
    med, best = cuda_time(lambda: pkg.polyak_update_(tgt, src, 0.005), 10)
    out["polyak_64M"] = {"bytes": 12 * n_par, "ms": med, "GBps": 12 * n_par / 1e9 / (med * 1e-3), "frac": 12 * n_par / 1e9 / (med * 1e-3) / pk["hbm"]}
    del tgt, src
    prev_run = pkg.Run.instance()
    sac_B, sac_obs = 4096, 188  # two-frame window of 188 features = the 376 inputs of the PPO bench; 256x256 tanh MLPs
    run_sac = pkg.Run(training_config=pkg.TrainingConfig(learning_rate=1e-4, batch_size=sac_B), environment_config=pkg.EnvironmentConfig(window_length=2),
                      network_config=pkg.NetworkConfig(input_shape=sac_obs, output_shape=ACT_DIM, linear_hidden_shapes=HIDDEN), device=str(dev))
    torch.manual_seed(0)
    sac_agent = pkg.SoftActorCriticAgent(run_sac)
    sac = pkg.SoftActorCritic(type("H", (), {"run": run_sac})(), sac_agent)
    n_env, n_t = 256, 256
    replay = {"current_state": torch.randn(n_env, n_t, 2, sac_obs, device=dev), "next_state": torch.randn(n_env, n_t, 2, sac_obs, device=dev),
              "action": torch.randn(n_env, n_t, ACT_DIM, device=dev), "reward": torch.randn(n_env, n_t, 1, device=dev),
              "is_alive": torch.rand(n_env, n_t, 1, device=dev) > 0.05}
    idx_host = torch.randperm(n_env * n_t)
    counter = [0]

    def sac_step():
        sac.train(replay, counter[0], idx=idx_host)
        counter[0] += 1
    med, best = cuda_time(sac_step, 10)
    out["sac_update_B4096"] = {"ms": med, "samples_per_s": sac_B / (med * 1e-3), "replay_rows": n_env * n_t,
                               "note": "one SoftActorCritic.train call (fp32 kernels): gather, TD target, twin-Q step, policy step through dQ/da, Polyak"}
    # the same call through the CPU oracle port (reference's torch CPU ops), all host threads, three calls
    from oracle import sac_oracle as SO
    torch.set_num_threads(os.cpu_count() or 1)
    ocfg = SO.SacConfig(state_dim=2 * sac_obs, act_dim=ACT_DIM, hidden=HIDDEN, batch_size=sac_B)
    oagent = SO.OracleSacAgent(ocfg)
    oflat = {k: v.reshape(n_env * n_t, *v.shape[2:]).cpu() for k, v in replay.items()}
    eps_host = torch.randn(2, sac_B, ACT_DIM)
    SO.sac_train_step(oagent, oflat, idx_host, eps_host[0], eps_host[1], 0)
    t0 = time.perf_counter()
    for c in range(3):
        SO.sac_train_step(oagent, oflat, idx_host, eps_host[0], eps_host[1], c + 1)
    cpu_ms = (time.perf_counter() - t0) / 3 * 1e3
    out["sac_update_B4096"]["cpu_port_ms"] = cpu_ms
    out["sac_update_B4096"]["cpu_cores"] = os.cpu_count() or 1
    del replay, sac, sac_agent, oagent, oflat
    pkg.Run._instance = prev_run
    torch.cuda.empty_cache()
    return out


def cpu_baseline(args):
    """Bounded CPU sample of the same workload (rank 0, N=1 only): CpuArm, one timed step of <= 2 epochs."""
    arm = CpuArm(args.envs, args.rollout_steps, args.minibatch, args.epochs)
    arm.warm_up()
    n_ep = 2 if arm.B >= 4096 else 1
    t_gae, t_train, mem = arm.timed_step(n_ep)
    out = {"value": n_ep * arm.nb * arm.B / (t_train + t_gae * n_ep / arm.E), "unit": "samples/s", "cores": arm.cores, "kind": arm.kind,
           "sample": arm.describe(t_gae, t_train, n_ep), "gae_GBps": 21 * arm.M / 1e9 / t_gae}
    if arm.B != 500:
        out["value_B500"], out["sample_B500"] = arm.b500(mem)
    return out


DUMP_MAX_ELEMENTS = 4 << 20  # per dumped array (16 MB in float32): the files of one dump stay under 64 MB in all


def dump_outputs(out_dir, agent, mem, losses):
    """`--dump-outputs`: what the last timed step hands a caller of `PPO.calculate_advantages` + `PPO.train`, as float32
    `out_dir/<name>.npy` — the advantages and value targets written into the rollout, the per-minibatch (actor, critic)
    losses, and the updated parameters and Adam moments under their `state_dict` names.  An array of more than
    DUMP_MAX_ELEMENTS values keeps a seeded sample of its rows (environments, minibatches): the same rows for the same
    arguments, so that dumps of two builds compare file for file."""
    import numpy as np
    eng = agent.engine
    named = list(agent.networks.named_parameters())
    out = {"advantage": mem["advantage"], "current_state_value_target": mem["current_state_value_target"], "losses": losses}
    for prefix, flat in (("param", eng.flat), ("adam_exp_avg", eng.exp_avg), ("adam_exp_avg_sq", eng.exp_avg_sq)):
        out.update({f"{prefix}.{name}": t for name, t in eng.grads_by_name(flat, named).items()})
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, t in out.items():
        if t.numel() > DUMP_MAX_ELEMENTS:
            rows = max(1, DUMP_MAX_ELEMENTS // (t.numel() // t.shape[0]))
            keep = torch.randperm(t.shape[0], generator=torch.Generator().manual_seed(0))[:rows].sort().values
            t = t[keep.to(t.device)]
        a = t.detach().to("cpu", torch.float32).numpy()
        total += a.nbytes
        np.save(os.path.join(out_dir, f"{name}.npy"), a)
    assert total <= 64 << 20, f"--dump-outputs wrote {total} bytes"


def run_b200(args, config):
    import torch.distributed as dist

    import mujoco_reinforcement_learning_b200 as pkg
    from mujoco_reinforcement_learning_b200 import _lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("launch with torch.distributed.run --nproc-per-node N for --gpus N")
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # one rank per GPU on a multi-socket host: run (and pin host buffers) on the CPUs local to this rank's GPU
        from mujoco_reinforcement_learning_b200.distributed import bind_host_to_gpu
        config["host_affinity"] = "gpu-local cpus" if bind_host_to_gpu(dev) else "unchanged"
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    pk = peaks()
    lib = _lib.load()

    n_envs, T, B, E = args.envs, args.rollout_steps, args.minibatch, args.epochs
    if args.scaling == "strong":  # the named problem (4096 envs x 128 steps, 32768-row minibatches) split over the ranks
        assert n_envs % world == 0 and B % world == 0, "--scaling strong: envs and minibatch must divide by the world size"
        n_envs, B = n_envs // world, B // world
    M_local, M = n_envs * T, n_envs * T * world
    GB = B * world
    run = pkg.Run(training_config=pkg.TrainingConfig(learning_rate=1e-4, batch_size=GB, epochs_per_iteration=E),
                  ppo_config=pkg.PPOConfig(), environment_config=pkg.EnvironmentConfig(maximum_timesteps=T, num_envs=n_envs * world),
                  network_config=pkg.NetworkConfig(input_shape=OBS_DIM, output_shape=ACT_DIM, linear_hidden_shapes=HIDDEN, critic_hidden_shapes=HIDDEN),
                  device=str(dev), gemm_precision=args.precision)
    torch.manual_seed(0)  # identical initial parameters on every rank
    agent = pkg.PPOAgent(run, max_batch=max(B, 4096))
    eng = agent.engine
    if world > 1:
        from mujoco_reinforcement_learning_b200 import distributed as D
        D.init_engine_comm(eng)
    algo = pkg.PPO(type("Helper", (), {"run": run})(), agent)

    roll = make_rollout(n_envs, T, 1234 + 3 + rank)
    host = {k: roll[k].contiguous() for k in ("current_state", "action", "reward", "current_state_value", "next_state_value", "terminated")}
    d = {k: v.to(dev) for k, v in host.items()}
    obs_flat = d["current_state"].reshape(M_local, OBS_DIM)
    logp = torch.empty(M_local, device=dev)
    for s in range(0, M_local, eng.max_batch):  # old log-prob under the initial policy (SURVEY §8d)
        lp, _, _ = eng.evaluate(obs_flat[s:s + eng.max_batch], d["action"].reshape(M_local, ACT_DIM)[s:s + eng.max_batch])
        logp[s:s + eng.max_batch] = lp
    d["action_log_prob"] = logp.reshape(n_envs, T)
    host["action_log_prob"] = d["action_log_prob"].cpu()
    n_total_steps = args.warmup + args.steps + 1
    gperm = torch.Generator().manual_seed(99)
    perms_host = [torch.stack([torch.randperm(M, generator=gperm) for _ in range(E)]) for _ in range(n_total_steps)]
    perms_dev = [p.to(dev) for p in perms_host]
    hp = eng.hparams(1e-4, 1e-4, 0.1, 1e-4)
    nb = M // GB
    samples_per_step = E * nb * GB

    def step_device(i):
        """One step; returns its losses and the rollout memory it wrote the advantages and value targets into."""
        mem = pkg.RolloutMemory(dict(d), (n_envs, T))
        algo.calculate_advantages(mem)
        fields = {"current_state": mem["current_state"].reshape(M_local, OBS_DIM), "action": mem["action"].reshape(M_local, ACT_DIM),
                  "action_log_prob": mem["action_log_prob"].reshape(M_local), "advantage": mem["advantage"].reshape(M_local),
                  "current_state_value_target": mem["current_state_value_target"].reshape(M_local)}
        if world > 1:
            fields = D.share_rollout(eng, fields)
        losses = eng.train(fields["current_state"], fields["action"], fields["action_log_prob"], fields["advantage"],
                           fields["current_state_value_target"], perms_dev[i], GB, hp)
        return losses, mem

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for i in range(args.warmup):
        step_device(i)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    launches0 = lib.b200ppo_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for k in range(args.steps):
        losses, last_mem = step_device(args.warmup + k)
    ev1.record()
    barrier()
    launches = lib.b200ppo_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    ms = ev0.elapsed_time(ev1)
    if world > 1:
        tmax = torch.tensor([ms], device=dev)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        ms = float(tmax.item())
    value = args.steps * samples_per_step / (ms * 1e-3)
    final_losses = losses[-1].tolist()
    if args.dump_outputs and rank == 0:  # before the measurements below move the parameters on
        dump_outputs(args.dump_outputs, agent, last_mem, losses)

    # ---- e2e through the C ABI with host buffers (single GPU: the host entry point is per-rank) --------------
    e2e = None
    if args.no_e2e:
        pass
    elif world == 1:
        pin = {k: v.pin_memory() for k, v in host.items()}
        pin_perms = [p.pin_memory() for p in perms_host]
        loss_host = torch.empty((E * nb, 2), dtype=torch.float32).pin_memory()

        def time_e2e(engine, steps, pipelined=True):
            """`steps` updates from pinned HOST buffers to losses on the host, wall clock around them; every step's
            host->device copies and its device->host loss read are inside the timed region.  pipelined: the two-call form
            (b200ppo_update_host_begin / _end): the upload of step k + 1 is enqueued before step k's update is waited for."""
            step_io = C.c_int64(engine.adam_step)
            if pipelined:
                def begin(i, slot):
                    _lib.check(lib.b200ppo_update_host_begin(engine._ctx, C.c_void_p(pin["current_state"].data_ptr()),
                                                             C.c_void_p(pin["action"].data_ptr()), C.c_void_p(pin["action_log_prob"].data_ptr()),
                                                             C.c_void_p(pin["reward"].data_ptr()), C.c_void_p(pin["current_state_value"].data_ptr()),
                                                             C.c_void_p(pin["next_state_value"].data_ptr()), C.c_void_p(pin["terminated"].data_ptr()),
                                                             n_envs, T, C.c_void_p(pin_perms[i % len(pin_perms)].data_ptr()), E, slot),
                               "b200ppo_update_host_begin")

                def end(slot):
                    _lib.check(lib.b200ppo_update_host_end(engine._ctx, _lib.ptr(engine.flat), _lib.ptr(engine.exp_avg), _lib.ptr(engine.exp_avg_sq),
                                                           C.byref(step_io), 0.99, 0.98, 0, 0, 1.0, B, 0, C.byref(hp),
                                                           C.c_void_p(loss_host.data_ptr()), slot, _lib.stream_ptr()), "b200ppo_update_host_end")

                begin(0, 0); end(0)  # warm-up: both staging sets get allocated outside the timed region
                begin(1, 1); end(1)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                begin(args.warmup, 0)
                marks = []
                for k in range(steps):
                    if k + 1 < steps:
                        begin(args.warmup + k + 1, (k + 1) & 1)
                    end(k & 1)  # returns with step k's losses on the host
                    marks.append(time.perf_counter())
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                engine.adam_step = int(step_io.value)
                # the first step's upload has nothing to hide behind; from the second step on every upload overlaps an update
                time_e2e.steady = (marks[-1] - marks[0]) / (steps - 1) if steps > 1 else None
                return dt / steps

            def step_host(i):
                _lib.check(lib.b200ppo_update_host(engine._ctx, _lib.ptr(engine.flat), _lib.ptr(engine.exp_avg), _lib.ptr(engine.exp_avg_sq),
                                                   C.byref(step_io), C.c_void_p(pin["current_state"].data_ptr()),
                                                   C.c_void_p(pin["action"].data_ptr()), C.c_void_p(pin["action_log_prob"].data_ptr()),
                                                   C.c_void_p(pin["reward"].data_ptr()), C.c_void_p(pin["current_state_value"].data_ptr()),
                                                   C.c_void_p(pin["next_state_value"].data_ptr()),
                                                   C.c_void_p(pin["terminated"].data_ptr()), n_envs, T, 0.99, 0.98, 0, 0, 1.0,
                                                   C.c_void_p(pin_perms[i % len(pin_perms)].data_ptr()), E, B, 0, C.byref(hp),
                                                   C.c_void_p(loss_host.data_ptr()), _lib.stream_ptr()), "b200ppo_update_host")

            for i in range(max(1, min(args.warmup, 2))):
                step_host(i)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for k in range(steps):
                step_host(args.warmup + k)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            engine.adam_step = int(step_io.value)
            return dt / steps

        dt_step = time_e2e(eng, args.steps)
        steady = getattr(time_e2e, "steady", None)
        dt_single = time_e2e(eng, max(2, args.steps // 2), pipelined=False)
        h2d = sum(v.numel() * v.element_size() for v in host.values()) + perms_host[0].numel() * 8
        e2e = {"value": samples_per_step / dt_step, "unit": "samples/s", "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": loss_host.numel() * 4, "ms_per_step": dt_step * 1e3,
               "api": "b200ppo_update_host_begin / _end (C ABI, pinned host buffers; the upload of step k + 1 is enqueued before step k's "
                      "update is waited for, all copies inside the timed region)",
               "gemm": args.precision,
               # steps 2..K only: the first step's upload (h2d_bytes_per_step over PCIe, ~15 ms) has no update to hide behind
               # and is charged to `value` in full; a trainer that keeps running sees this figure
               "steady_state": ({"value": samples_per_step / steady, "ms_per_step": steady * 1e3} if steady else None),
               "single_call": {"value": samples_per_step / dt_single, "ms_per_step": dt_single * 1e3,
                               "api": "b200ppo_update_host (one blocking call per step: upload, then update)"}}

    else:
        # N > 1: the public Python API per rank — pinned host slab -> device, GAE, slab all-gather (NCCL), global-permutation
        # update with the per-minibatch all-reduce, losses back on the host; barrier + max over ranks like `value`
        pin = {k: v.pin_memory() for k, v in host.items()}
        pin_perms = [p.pin_memory() for p in perms_host]

        copy_stream = torch.cuda.Stream(dev)

        def upload(i):
            """Step i's host slab and this rank's permutation slots onto the device, on a side stream (what a trainer does with
            the rollout it has just collected while the previous update is still running)."""
            with torch.cuda.stream(copy_stream):
                dd = {k: v.to(dev, non_blocking=True) for k, v in pin.items()}
                # every rank holds the same global permutations on its host and uploads only the slots it consumes
                my_perms = D.slice_perms_for_rank(pin_perms[i % len(pin_perms)], GB, world, rank, dev)
                ev = torch.cuda.Event()
                ev.record(copy_stream)
            return dd, my_perms, ev

        def step_host(staged):
            dd, my_perms, ev = staged
            cur = torch.cuda.current_stream()
            cur.wait_event(ev)
            for t in list(dd.values()) + [my_perms]:
                t.record_stream(cur)
            mem = pkg.RolloutMemory(dd, (n_envs, T))
            algo.calculate_advantages(mem)
            fields = D.share_rollout(eng, {
                "current_state": mem["current_state"].reshape(M_local, OBS_DIM), "action": mem["action"].reshape(M_local, ACT_DIM),
                "action_log_prob": mem["action_log_prob"].reshape(M_local), "advantage": mem["advantage"].reshape(M_local),
                "current_state_value_target": mem["current_state_value_target"].reshape(M_local)})
            out = eng.train(fields["current_state"], fields["action"], fields["action_log_prob"], fields["advantage"],
                            fields["current_state_value_target"], my_perms, GB, hp, rank_sliced_perms=True)
            return out.cpu()

        step_host(upload(0))
        barrier()
        t0 = time.perf_counter()
        staged = upload(args.warmup)  # inside the timed region, like every other upload; only this one has nothing to hide behind
        for k in range(args.steps):
            nxt = upload(args.warmup + k + 1) if k + 1 < args.steps else None
            loss_host = step_host(staged)
            staged = nxt
        barrier()
        dt = torch.tensor([time.perf_counter() - t0], device=dev)
        dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        dt = float(dt.item())
        h2d = sum(v.numel() * v.element_size() for v in host.values()) + perms_host[0].numel() * 8 // world
        e2e = {"value": args.steps * samples_per_step / dt, "unit": "samples/s", "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": loss_host.numel() * 4, "ms_per_step": dt / args.steps * 1e3,
               "api": "PPO.calculate_advantages + distributed.share_rollout + ActorCriticEngine.train per rank, pinned host slabs "
                      "uploaded on a side stream one step ahead, rank-sliced permutations (bytes are per rank)"}

    # ---- per-kernel-class device time of one step (CUDA events on the launching stream) ----------------------
    _lib.check(lib.b200ppo_profile_begin(eng._ctx))
    ga, gb_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    mem = pkg.RolloutMemory(dict(d), (n_envs, T))
    ga.record(); algo.calculate_advantages(mem); gb_.record()
    step_device(args.warmup + args.steps)
    ms_c = (C.c_double * 8)()
    n_c = (C.c_int64 * 8)()
    _lib.check(lib.b200ppo_profile_end(eng._ctx, ms_c, n_c))
    prof = {name: {"ms": ms_c[i], "groups": int(n_c[i])} for i, name in enumerate(_lib.PROF_CLASSES) if n_c[i]}
    prof["gae"] = {"ms": ga.elapsed_time(gb_), "groups": 1}
    fl = flops_per_sample()
    lb_rows = E * nb * B  # rows this rank pushed through the GEMMs in the profiled step
    gemm_ms = sum(prof[k]["ms"] for k in ("gemm_fwd", "gemm_dgrad", "gemm_wgrad") if k in prof)
    gemm_flops = fl["total"] * lb_rows
    achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    total_prof_ms = sum(v["ms"] for v in prof.values())
    for k, v in prof.items():
        v["share"] = v["ms"] / total_prof_ms if total_prof_ms else 0.0
    for k, key in (("gemm_fwd", "fwd"), ("gemm_dgrad", "dgrad"), ("gemm_wgrad", "wgrad")):
        if k in prof and prof[k]["ms"] > 0:
            prof[k]["TFLOPs"] = fl[key] * lb_rows / (prof[k]["ms"] * 1e-3) / 1e12
    if "gather" in prof and prof["gather"]["ms"] > 0:
        if args.precision == "bf16":
            # one fp32 -> bf16 conversion of the whole rollout (rows of PX = 384 bf16), then per epoch a byte gather of bf16
            # rows plus the fp32 leaves and the int64 index
            PX = (OBS_DIM + 1 + 7) // 8 * 8
            by = M_local * (4 * OBS_DIM + 2 * PX) + (2 * (2 * PX + 4 * ACT_DIM + 12) + 8) * (E * nb * B)
        else:
            by = (2 * (4 * OBS_DIM + 4 * ACT_DIM + 12) + 8) * (E * nb * B)
        prof["gather"]["GBps"] = by / 1e9 / (prof["gather"]["ms"] * 1e-3)
        prof["gather"]["frac_hbm"] = prof["gather"]["GBps"] / pk["hbm"]
    roofline = {"kernel": "fp32-tolerance GEMMs on tcgen05: split3_kernel + tc_gemm_kernel in three-term mode, six bf16 products per "
                          "fp32 product (gemm_split.cu); achieved counts the fp32 products once" if args.precision == "fp32"
                else "tcgen05 bf16 GEMMs: tc_chain_kernel (forward + losses + dgrads) and tc_wgrad2_kernel (weight gradients)",
                "bound": "tensor", "achieved": achieved, "peak": pk["tensor_sustained"], "unit": "TFLOP/s",
                "frac": achieved / pk["tensor_sustained"],
                # DRAM bytes of the six GEMM launches of ONE 32768-row minibatch (sum of dram__bytes_read+write over
                # profiles/r01_ncu_tc_kernels_B32768.csv); the HBM floor of the update is 1584 B/sample = 52 MB: the
                # excess is activations crossing HBM between the per-layer kernels
                "traffic": TRAFFIC_BF16_B32768 if (args.precision == "bf16" and B == 32768) else None,
                "traffic_note": "dram__bytes_read + write per 32768-row minibatch over its two GEMM launches, chain + weight gradients "
                                "(ncu --set full, profiles/r02_ncu_chain_wgrad_B32768.csv); round 1: 389.6 MB over six launches",
                "peak_source": pk["source"] + " bf16 sustained",
                "share_of_step": gemm_ms / total_prof_ms if total_prof_ms else None,
                "flops_per_sample": fl["total"], "launch_groups": sum(prof[k]["groups"] for k in ("gemm_fwd", "gemm_dgrad", "gemm_wgrad") if k in prof)}

    # ---- other settings of the same workload, measured the same way (reported, not the headline) -------------------
    variants = []
    if world == 1 and not args.no_variants:
        others = [(p, b) for p in ("bf16", "fp32") for b in (32768, 4096, 500) if not (p == args.precision and b == B)]
        others.append(("fp32x2", 32768))  # fp32 context with two scaled fp16 terms per operand value (22-bit operands)
        for prec, vb in others:
            vrun = pkg.Run(training_config=pkg.TrainingConfig(learning_rate=1e-4, batch_size=vb, epochs_per_iteration=E),
                           ppo_config=pkg.PPOConfig(), environment_config=pkg.EnvironmentConfig(maximum_timesteps=T, num_envs=n_envs),
                           network_config=pkg.NetworkConfig(input_shape=OBS_DIM, output_shape=ACT_DIM, linear_hidden_shapes=HIDDEN, critic_hidden_shapes=HIDDEN),
                           device=str(dev), gemm_precision="fp32" if prec == "fp32x2" else prec)
            torch.manual_seed(0)
            vagent = pkg.PPOAgent(vrun, max_batch=max(vb, 4096))
            veng = vagent.engine
            if prec == "fp32x2":
                veng.set_fp32_terms(2)
            vnb = M // vb
            vE = E if vb >= 4096 else 2  # 1048 minibatches/epoch at the reference's batch_size=500: two epochs suffice
            vperm = perms_dev[0][:vE]
            mem = pkg.RolloutMemory(dict(d), (n_envs, T))
            algo.calculate_advantages(mem)
            f = [mem["current_state"].reshape(M_local, OBS_DIM), mem["action"].reshape(M_local, ACT_DIM),
                 mem["action_log_prob"].reshape(M_local), mem["advantage"].reshape(M_local),
                 mem["current_state_value_target"].reshape(M_local)]
            for _ in range(2):
                veng.train(*f, vperm, vb, hp)
            torch.cuda.synchronize()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(2):
                veng.train(*f, vperm, vb, hp)
            a1.record()
            torch.cuda.synchronize()
            vms = a0.elapsed_time(a1) / 2
            variants.append({"gemm": prec, "minibatch": vb, "epochs_timed": vE, "ms_per_epoch": vms / vE,
                             "value": vE * vnb * vb / (vms * 1e-3), "unit": "samples/s (train() only, rollout resident)"})
            if vb == B and e2e is not None and not args.no_e2e:  # the other precision end to end, same entry point, same bytes
                dt_v = time_e2e(veng, 2)
                variants[-1]["e2e"] = {"value": samples_per_step / dt_v, "unit": "samples/s", "ms_per_step": dt_v * 1e3,
                                       "h2d_bytes_per_step": e2e["h2d_bytes_per_step"], "api": e2e["api"], "gemm": prec}
            del vagent, veng

    # replicas must hold bit-identical parameters after the timed steps (outside the timed region)
    replicas_identical = None
    if world > 1:
        bits = eng.flat.view(torch.int32).to(torch.int64)
        digest = torch.stack([bits.sum(), (bits * torch.arange(1, bits.numel() + 1, device=dev)).sum()])
        every = [torch.zeros_like(digest) for _ in range(world)]
        dist.all_gather(every, digest)
        replicas_identical = all(bool(torch.equal(every[0], e)) for e in every)
        assert replicas_identical, "data-parallel replicas diverged"
    k6 = k6_latency(agent, n_envs)
    sweep_multi = c5_sweep(pk, world, rank) if (world > 1 and not args.no_kernels) else None

    line = {"metric": "ppo_update_samples_per_sec", "value": value, "unit": "samples/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": args.scaling,
            "replicas_identical": replicas_identical, "rollout_inference": k6,
            "vs_baseline": None, "dtype": "f32" if args.precision == "fp32" else "bf16", "data": "synthetic", "config": config,
            "gpu_launches": int(launches), "clocks": clocks, "e2e": e2e, "roofline": roofline, "kernel_classes": prof,
            "final_losses": final_losses, "samples_per_step": samples_per_step, "variants": variants}
    if rank == 0:
        if world == 1 and not args.no_kernels:  # per-kernel roofline lines belong to the N=1 run (the other ranks would only wait)
            line["hbm_kernels"] = hbm_kernel_lines(pk)
        if world == 1 and not args.no_cpu:
            line["cpu_baseline"] = cpu_baseline(args)
        if sweep_multi is not None:
            line["hbm_kernels"] = {"c5_sweep": sweep_multi}
        # the two precisions side by side: bf16 GEMMs are the 2e-2 variant, fp32 the reference's own precision
        by_prec = {args.precision: {"value": value, "e2e": e2e["value"] if e2e else None}}
        for v in variants:
            if v["minibatch"] == B:
                by_prec[v["gemm"]] = {"value": v["value"], "e2e": v.get("e2e", {}).get("value")}
        line["headline_by_precision"] = by_prec
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs", type=int, default=4096, help="environments per GPU")
    ap.add_argument("--rollout-steps", type=int, default=128)
    ap.add_argument("--minibatch", type=int, default=32768, help="minibatch rows per GPU (global = N x this)")
    ap.add_argument("--epochs", type=int, default=10, help="epochs_per_iteration (reference default, main.py:45)")
    ap.add_argument("--precision", default="bf16", choices=["fp32", "bf16"],
                    help="GEMM arithmetic: bf16 tcgen05 (2e-2 parity, default) or fp32 tolerance (1e-5 parity: six bf16 tcgen05 "
                         "products per fp32 product at large minibatches, FFMA below)")
    ap.add_argument("--ref-epochs", type=int, default=4, help="reference arm: at most this many full epochs per timed step")
    ap.add_argument("--ref-budget", type=float, default=20.0, help="reference arm: seconds of epochs per timed step")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: --envs / --minibatch are per GPU; strong: they are the TOTAL problem, split over the N ranks")
    ap.add_argument("--no-kernels", action="store_true", help="skip the HBM-kernel roofline mini-benchmarks")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline sample")
    ap.add_argument("--no-variants", action="store_true", help="skip the secondary (precision, minibatch) settings")
    ap.add_argument("--no-e2e", action="store_true", help="profiling runs only: skip the host-buffer end-to-end measurement")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (advantages, value targets, losses, updated parameters and Adam "
                         "moments) as float32 DIR/<name>.npy; the inputs are seeded, so two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of --impl b200")
    if args.warmup < 3 and args.impl == "b200":
        args.warmup = 3  # timing rule: at least 3 warm-up steps
    world = int(os.environ.get("WORLD_SIZE", "1"))
    config = {"workload": "Humanoid-v4 shape PPO update (BASELINE.json configs[3]): GAE + epochs x (permutation gather + "
                          "minibatch actor-critic forward/loss/backward/Adam)",
              "envs_per_gpu": args.envs, "rollout_steps": args.rollout_steps, "obs_dim": OBS_DIM, "act_dim": ACT_DIM,
              "hidden": HIDDEN, "activation": "tanh", "gemm": args.precision, "minibatch_per_gpu": args.minibatch, "epochs_per_step": args.epochs,
              "parallelism": f"dp{max(world, 1)} (env-slab sharding, grad all-reduce)" if world > 1 else "single GPU",
              "scaling": args.scaling,
              "cache": "inputs larger than L2 (788 MB observation buffer re-gathered every epoch); no explicit flush"}
    if args.impl == "reference":
        run_reference(args, config)
    else:
        run_b200(args, config)


if __name__ == "__main__":
    main()
