#!/usr/bin/env python
"""bench.py -- learner transitions/sec per ICRL iteration (BASELINE.json's metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload halfcheetah|antwall|lapgrid|pointcircle]
    python bench.py --impl reference ...      # the reference's CPU algorithm (oracle port) on the host cores

One "step" = one full ICRL learner iteration on synthetic buffers of the named env's shape:
    R rollouts x (K1 cost relabel + K3 dual GAE + K4 PPO-Lagrangian update + dual step)  +  one K2 constraint-net train.
`value`  : whole-job transitions/s with all inputs resident in HBM (icrl_b200.learner.DeviceLearner, C-ABI device entry points).
`e2e`    : the same iteration through the reference-shaped Python API with HOST (numpy) buffers: ConstraintNet.cost_function,
           RolloutBufferWithCost.compute_returns_and_advantage, PPOLagrangian.train, ConstraintNet.train -- H2D / D2H inside.
`roofline`: the dominant kernel (K4 persistent PPO kernel): algorithmic bytes AND flops / measured launch duration against the
           measured HBM and 3xTF32 tensor peaks, the binding one named.
`workloads`: short runs of the other BASELINE configs (AntWall, LapGrid, PointCircle; N>1: AntWall), same value / e2e / roofline.
`sweep`   : the Ant-shaped 64K-16M transition sweep (BASELINE config 5), K1-K4 per size against their rooflines.
`dp_parity`: N>1 only -- the data-parallel K4 / K2 paths checked against the oracle before anything is timed.
`cpu_baseline`: the UNMODIFIED reference (baseline/_ref) on a bounded sample of the same iteration, extrapolated linearly
           (the oracle port only if that copy is absent).
Fixed work: KL early stops (ppo target_kl, cn target_kl_*) are disabled so every epoch / backward iteration runs.
`--dump-outputs DIR`: what the last timed step computed, as DIR/<name>.npy (see dump_outputs).  The inputs depend only on
the arguments, so two builds run with the same arguments can be compared array by array.  Inside the tree, use
`bench_outputs/` (git-ignored).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch as th  # noqa: E402

METRIC = "learner transitions/sec per ICRL iteration at 1/2/4/8 B200 vs host CPU"     # BASELINE.json's metric, verbatim
try:
    with open(os.path.join(ROOT, "BASELINE.json")) as _f:
        METRIC = json.load(_f).get("metric", METRIC)
except (OSError, ValueError):
    pass
UNIT = "transitions/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="halfcheetah")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--cpu-steps", type=int, default=1600, help="K4 optimiser steps in the CPU sample (one full HalfCheetah rollout)")
    ap.add_argument("--replicas", action="store_true", help="N>1: independent learners instead of data-parallel all-reduce")
    ap.add_argument("--ref-budget", type=float, default=150.0, help="--impl reference: seconds of CPU work for all samples")
    ap.add_argument("--no-workloads", action="store_true", help="skip the short AntWall / LapGrid / PointCircle runs")
    ap.add_argument("--aux-steps", type=int, default=2, help="timed iterations of each secondary workload")
    ap.add_argument("--no-sweep", action="store_true", help="skip the Ant-shaped 64K-16M transition sweep")
    ap.add_argument("--sweep-sizes", default="65536,262144,1048576,4194304,16777216", help="transitions per GPU")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step of the main workload computed as DIR/<name>.npy (rank 0); "
                         "bench_outputs/ in the repository root is git-ignored for this")
    return ap.parse_args()


# --------------------------------------------------------------------------------------------- helpers
def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f).get("hbm_gbs", 6650.0), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed region runs (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.proc, self.lines, self.gpu = None, [], gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.gpu)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True).start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dist_setup(n_gpus):
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    if world > 1:
        import torch.distributed as dist
        th.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=th.device("cuda", local))
    return rank, world, local


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    th.cuda.synchronize()


def max_over_ranks(x, world):
    if world > 1:
        import torch.distributed as dist
        t = th.tensor([x], dtype=th.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())
    return x


# --------------------------------------------------------------------------------------------- CPU baseline (oracle port)
def cpu_iteration_estimate(w, k4_steps, seed=0):
    """Times the oracle on a bounded sample of one ICRL iteration of workload `w` and extrapolates linearly.
    K1 in the reference's per-env-step form (VecCostWrapper.step_wait: one [n_envs, .] call per step), K3 one full
    rollout, K4 `k4_steps` optimiser steps of one rollout, K2 the full `backward_iters` (per-step IS via the O(N)
    identity, i.e. *cheaper* than the reference's N x N broadcast)."""
    from icrl_b200.learner import synth_demos, synth_rollouts
    from oracle import cn as ocn, costnorm, gae as ogae, ppo as oppo
    th.manual_seed(seed)
    T, E, n = w.n_steps, w.n_envs, w.n_steps * w.n_envs
    small = type(w)(**{**w.__dict__, "rollouts": 1})
    host = synth_rollouts(small, seed)
    low = high = None
    if not w.is_discrete:
        low, high = -np.ones(w.act_dim, np.float32), np.ones(w.act_dim, np.float32)
    spec = ocn.CNSpec(w.obs_dim, w.act_dim, w.cn_hidden, w.is_discrete, clip_obs=w.clip_obs, action_low=low, action_high=high,
                      regularizer_coeff=w.cn_reg, per_step_importance_sampling=w.per_step_is)
    dims = [spec.input_dims, *w.cn_hidden, 1]
    cn_params = []
    for i in range(len(dims) - 1):
        lin = th.nn.Linear(dims[i], dims[i + 1])
        cn_params += [lin.weight.detach().clone(), lin.bias.detach().clone()]
    t = {}
    # K1, per env step
    calls = min(T, 512)
    oo, aa = host["orig_obs"][0].astype(np.float64), host["actions"][0]
    t0 = time.perf_counter()
    costs = np.zeros((T, E), np.float32)
    news = np.concatenate([host["dones"][0][1:], host["last_dones"][0][None].astype(np.float32)]) != 0
    cstate = costnorm.reset(costnorm.initial_state(E))
    for s in range(calls):
        costs[s] = ocn.cost_function(cn_params, spec, oo[s], aa[s])
        if w.normalize_cost:      # VecNormalizeWithCost.step_wait, per env step as the reference runs it
            costs[s] = costnorm.normalize_rollout(costs[s:s + 1], news[s:s + 1], cstate)[0]
    t["k1"] = (time.perf_counter() - t0) / calls * T
    costs = np.tile(costs[:calls], (T // calls + 1, 1))[:T].copy()
    # K3
    P = oppo.init_policy(w.obs_dim, w.act_dim, w.is_discrete)
    obs_flat = th.tensor(host["obs"][0].reshape(n, w.obs_dim))
    acts_flat = th.tensor(host["actions"][0].reshape(n, -1))
    with th.no_grad():
        v, cv, lp, _ = oppo.evaluate_actions(P, obs_flat, acts_flat.flatten() if w.is_discrete else acts_flat, w.is_discrete)
    rv, cvv, lpp = (x.numpy().reshape(T, E) for x in (v, cv, lp))
    t0 = time.perf_counter()
    g = ogae.dual_gae(host["rewards"][0], rv, costs, cvv, host["dones"][0], rv[-1], cvv[-1], host["last_dones"][0], 0.99,
                      w.reward_gae_lambda, 0.99, w.cost_gae_lambda)
    t["k3"] = time.perf_counter() - t0
    # K4
    flat = {"observations": ogae.env_major(host["obs"][0]), "actions": ogae.env_major(host["actions"][0]),
            "old_log_prob": ogae.env_major(lpp), "old_reward_values": ogae.env_major(rv),
            "reward_advantages": ogae.env_major(g["reward_advantages"]), "reward_returns": ogae.env_major(g["reward_returns"]),
            "old_cost_values": ogae.env_major(cvv), "cost_advantages": ogae.env_major(g["cost_advantages"]),
            "cost_returns": ogae.env_major(g["cost_returns"])}
    rs = np.random.RandomState(seed)
    perms = [rs.permutation(n) for _ in range(w.n_epochs)]
    adam = ocn.adam_init(list(P.values()))
    steps_full = w.n_epochs * ((n + w.batch_size - 1) // w.batch_size)
    k4_steps = min(k4_steps, steps_full)
    t0 = time.perf_counter()
    out = oppo.train(P, adam, flat, perms, is_discrete=w.is_discrete, batch_size=w.batch_size, n_epochs=w.n_epochs,
                     lr=w.learning_rate, clip_range=w.clip_range, nu=w.penalty_initial_value, max_steps=k4_steps)
    t["k4"] = (time.perf_counter() - t0) / out["steps"] * steps_full
    # K2
    t["k2"] = 0.0
    if w.backward_iters > 0 and w.nominal_rows > 0:
        eo, ea, no, na, lengths = synth_demos(w, seed)
        t0 = time.perf_counter()
        ocn.train(cn_params, ocn.adam_init(cn_params), spec, w.backward_iters, no, na, lengths, eo, ea, lr=w.cn_lr)
        t["k2"] = time.perf_counter() - t0
    est = w.rollouts * (t["k1"] + t["k3"] + t["k4"]) + t["k2"]
    sample = (f"K1 {calls} of {T} per-step calls, K3 1 rollout, K4 {out['steps']} of {steps_full} optimiser steps of 1 rollout, "
              f"K2 full ({w.backward_iters} iters); x{w.rollouts} rollouts, linear extrapolation")
    return est, t, sample


def pick_cpu_threads(w):
    """The oracle's tensors are tiny (64-128 rows x 64 units): torch's intra-op threading can cost more than it gives.
    Time a few K4 optimiser steps with every host core and with one thread, keep the faster setting -- the CPU arm gets
    whatever thread count serves it best on this box."""
    cores = os.cpu_count() or 1
    best, best_t = cores, None
    for n in sorted({cores, max(1, cores // 4), 1}, reverse=True):
        th.set_num_threads(n)
        cpu_iteration_estimate(w, 8)                       # warm the thread pool / autograd
        t0 = time.perf_counter()
        _, parts, _ = cpu_iteration_estimate(w, 24)
        t = parts["k4"]
        if best_t is None or t < best_t:
            best, best_t = n, t
    th.set_num_threads(best)
    return best


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_model():
    try:
        with open("/proc/cpuinfo") as f:
            for line in f:
                if line.startswith("model name"):
                    return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


def reference_samples(w, n_samples, n_warm, budget_s):
    """The UNMODIFIED reference (baseline/_ref, see baseline/reference_arm.py) on the host cores: thread count calibrated
    on one-epoch train() calls (all cores vs one), then `n_warm` + `n_samples` bounded samples sized to `budget_s` seconds
    in total.  Returns a dict for the `cpu_baseline` key (value = best of the timed samples, BASELINE.md 3)."""
    from baseline import reference_arm as ra
    it = ra.ReferenceIteration(w)
    cores = host_cores()
    ra.k4_seconds_per_epoch(it, cores)                        # warm the thread pool / autograd
    per_epoch = {n: ra.k4_seconds_per_epoch(it, n) for n in sorted({cores, 1}, reverse=True)}
    threads = min(per_epoch, key=per_epoch.get)
    th.set_num_threads(threads)
    per_sample = max(1.5, budget_s / max(n_samples + n_warm, 1))
    # one K2 iteration is the other big piece (the N x N broadcast of per-step IS): time it once
    t0 = time.perf_counter()
    _, parts0, _ = it.sample(32, 1, 1)
    k2_iter = parts0["k2"] / max(w.backward_iters, 1)
    k4_epochs = int(max(1, min(w.n_epochs, (per_sample - k2_iter - 0.2) / max(per_epoch[threads], 1e-3))))
    ests, parts, desc = [], None, ""
    by_threads = {}
    t_wall = time.perf_counter()
    for i in range(n_warm + n_samples):
        if i < n_warm and i < len(per_epoch):                 # the first warm-up samples double as the all-cores / 1-core report
            n = sorted(per_epoch, reverse=True)[i]
            th.set_num_threads(n)
            est, _, _ = it.sample(128, k4_epochs, 1)
            by_threads[n] = w.transitions_per_iteration / est
            th.set_num_threads(threads)
            continue
        est, parts, desc = it.sample(128, k4_epochs, 1)
        if i >= n_warm:
            ests.append(est)
    best = min(ests)
    return {"value": w.transitions_per_iteration / best, "unit": UNIT, "cores": threads, "kind": "reference",
            "sample": desc, "host_cores": cores, "cpu_model": cpu_model(),
            "value_by_threads": {f"{n}": v for n, v in by_threads.items()},
            "k4_seconds_per_epoch_by_threads": {f"{n}": round(v, 4) for n, v in per_epoch.items()},
            "seconds_per_iteration_est": round(best, 2), "seconds_per_iteration_all_samples": [round(e, 2) for e in ests],
            "seconds_per_part": {k: round(v, 4) for k, v in parts.items()},
            "sample_wall_s": round(time.perf_counter() - t_wall, 2), "statistic": f"best of {len(ests)}"}


def port_samples(w, args, n_samples, n_warm):
    """Fallback when baseline/_ref is absent: the oracle port (kind "port")."""
    cores = pick_cpu_threads(w)
    for _ in range(max(n_warm, 1) - 1):
        cpu_iteration_estimate(w, max(20, args.cpu_steps // 10))
    ests, parts, sample = [], None, ""
    t_wall = time.perf_counter()
    for _ in range(max(n_samples, 1)):
        est, parts, sample = cpu_iteration_estimate(w, args.cpu_steps)
        ests.append(est)
    best = min(ests)
    return {"value": w.transitions_per_iteration / best, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
            "host_cores": host_cores(), "cpu_model": cpu_model(), "seconds_per_iteration_est": round(best, 2),
            "seconds_per_part": {k: round(v, 4) for k, v in parts.items()},
            "sample_wall_s": round(time.perf_counter() - t_wall, 2), "statistic": f"best of {len(ests)}"}


def run_reference(args, w):
    """--impl reference: the reference's own CPU implementation of the path on this box's host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    from baseline import reference_arm as ra
    if ra.available():
        cpu = reference_samples(w, max(args.steps, 1), max(args.warmup, 2), budget_s=float(args.ref_budget))
    else:
        cpu = port_samples(w, args, args.steps, args.warmup)
    val = cpu["value"]
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": cpu["seconds_per_iteration_est"] * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(w, 1, "host CPU only (the reference has no GPU or distributed path); each step is a bounded "
                                        "sample of one ICRL iteration, extrapolated linearly (see cpu_baseline.sample)"),
        "cpu_baseline": cpu,
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


def workload_config(w, world, parallelism):
    """The `config` object both arms print (same keys, so the driver can compare them)."""
    return {"workload": w.name, "transitions_per_step_per_gpu": w.transitions_per_iteration, "rollouts": w.rollouts,
            "n_steps": w.n_steps, "n_envs_per_gpu": w.n_envs, "batch_size": w.batch_size, "n_epochs": w.n_epochs,
            "backward_iters": w.backward_iters, "early_stop": "disabled (fixed work)",
            "l2": "flushed between timed steps (256 MB write, outside the timed region)", "parallelism": parallelism}


# --------------------------------------------------------------------------------------------- e2e through the public API
class _Env:
    def __init__(self, w, n_envs):
        from icrl_b200.learner import spaces_of
        self.observation_space, self.action_space = spaces_of(w)
        self.num_envs = n_envs


class HostLearner:
    """The same iteration through ConstraintNet / RolloutBufferWithCost / PPOLagrangian with numpy buffers."""

    def __init__(self, w, dev_learner, rank=0):
        from icrl_b200.buffers import RolloutBufferWithCost
        from icrl_b200.ppo_lag import PPOLagrangian
        self.w, self.cn = w, dev_learner.cn        # (in data-parallel mode the constraint net is already sharded: cn.comm)
        E = dev_learner.E
        self.algo = PPOLagrangian("TwoCriticsMlpPolicy", _Env(w, E), n_steps=w.n_steps, batch_size=w.batch_size,
                                  n_epochs=w.n_epochs, learning_rate=w.learning_rate, clip_range=w.clip_range,
                                  reward_gae_lambda=w.reward_gae_lambda, cost_gae_lambda=w.cost_gae_lambda, target_kl=None,
                                  penalty_initial_value=w.penalty_initial_value, penalty_learning_rate=w.penalty_learning_rate,
                                  seed=0, device=dev_learner.dev)
        if dev_learner.comm is not None and dev_learner.comm.world > 1:
            self.algo.policy.load_state_dict(dev_learner.policy.state_dict())      # replicated start on every rank
            self.algo.enable_data_parallel(dev_learner.comm)
        host = dev_learner.host
        self.bufs, self.pristine = [], []
        for r in range(w.rollouts):
            b = RolloutBufferWithCost(w.n_steps, self.algo.observation_space, self.algo.action_space, dev_learner.dev,
                                      reward_gamma=0.99, reward_gae_lambda=w.reward_gae_lambda, cost_gamma=0.99,
                                      cost_gae_lambda=w.cost_gae_lambda, n_envs=E)
            b.observations[:], b.orig_observations[:], b.actions[:] = host["obs"][r], host["orig_obs"][r], host["actions"][r]
            b.rewards[:], b.dones[:] = host["rewards"][r], host["dones"][r]
            b.reward_values[:] = dev_learner.reward_values[r].cpu().numpy()
            b.cost_values[:] = dev_learner.cost_values[r].cpu().numpy()
            b.log_probs[:] = dev_learner.log_probs[r].cpu().numpy()
            b.full, b.pos = True, w.n_steps
            self.bufs.append(b)
            self.pristine.append({k: getattr(b, k) for k in ("observations", "orig_observations", "actions", "log_probs",
                                                              "reward_values", "cost_values")})
        self.last_dones = host["last_dones"]
        # the cost statistics a VecNormalizeWithCost would carry (state after reset())
        import types
        from icrl_b200.vec_env import RunningMeanStd
        rms = RunningMeanStd(shape=())
        rms.update(np.zeros(E))
        self.vn = types.SimpleNamespace(cost_rms=rms, cost_ret=np.zeros(E), cost_gamma=0.99, epsilon=1e-8, clip_cost=10.0,
                                        norm_cost=True, training=True, old_cost=None)
        if w.nominal_rows:
            from icrl_b200.learner import synth_demos
            _, _, self.no, self.na, self.lengths = synth_demos(w, rank)
        self.h2d = self.d2h = 0

    def run(self):
        w, n = self.w, self.w.n_steps * self.bufs[0].n_envs
        h2d = d2h = 0
        for r, b in enumerate(self.bufs):
            for k, arr in self.pristine[r].items():   # "freshly collected" time-major arrays (train() rebinds env-major copies)
                setattr(b, k, arr)
            b.generator_ready = False
            if w.normalize_cost:                                                               # K1 + K5
                b.relabel_costs(self.cn, self.vn, self.last_dones[r])
                h2d += b.orig_observations.nbytes + b.actions.nbytes + b.dones.nbytes + b.n_envs + (3 + b.n_envs) * 8
                d2h += 2 * b.costs.nbytes + (3 + b.n_envs) * 8
            else:
                costs = self.cn.cost_function(b.orig_observations, b.actions)                  # K1
                b.costs[:], b.orig_costs[:] = costs, costs
                h2d += b.orig_observations.nbytes + b.actions.nbytes; d2h += costs.nbytes
            b.compute_returns_and_advantage(b.reward_values[-1], b.cost_values[-1], self.last_dones[r])   # K3
            h2d += 5 * n * 4 + 2 * b.n_envs * 4 + b.n_envs; d2h += 4 * n * 4
            self.algo.rollout_buffer = b
            self.algo.train()                                                                  # K4 + dual step
            h2d += (b.observations.nbytes + b.actions.nbytes + 7 * n * 4) + w.n_epochs * n * 4 + 4
            d2h += self.algo.last_train_stats.nbytes + 16 + 8
        if w.backward_iters > 0 and w.nominal_rows > 0:
            self.cn.train(w.backward_iters, self.no, self.na, self.lengths)                    # K2
            h2d += self.no.nbytes + self.na.nbytes + (len(self.lengths) + 1) * 4; d2h += 18 * 4
        self.h2d, self.d2h = h2d, d2h


# --------------------------------------------------------------------------------------------- main (B200 arm)
def time_steps(fn, steps, world, flush):
    """Device time of exactly `steps` calls of fn, L2 flushed between calls (flush excluded), max over ranks."""
    evs = [(th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)) for _ in range(steps)]
    barrier(world)
    for s, e in evs:
        flush.add_(1.0)                 # > L2 (126 MB) write: evicts the previous step's lines
        s.record()
        fn()
        e.record()
    barrier(world)
    return max_over_ranks(sum(s.elapsed_time(e) for s, e in evs) * 1e-3, world)


# dram__bytes_read.sum + dram__bytes_write.sum of ONE full single-cluster K4 launch: an OFFLINE constant from the
# `ncu --set full` captures summarised under profiles/ (not measured in this run: ncu replays kernels and bench numbers may not
# be taken under a profiler); keyed by Workload.name
K4_NCU_TRAFFIC_BYTES = {
    "HalfCheetah HCWithPos-v0 ICRL (cl 20, ft 2e5, bi 10)": 21652480,
    "AntWall-v0 ICRL (cl 40 40, ft 2e5, bi 5, batch 128, n_epochs 20)": 122238720 + 3342848,
}


def k4_flops_per_sample_pass(w):
    """2 * MACs of the three trunks + heads, forward + backward ~ 3x forward (SURVEY 8(d))."""
    a_out = w.act_dim
    fwd = 2 * (3 * (w.obs_dim * 64 + 64 * 64) + 64 * (a_out + 2))
    return 3 * fwd


def k4_bytes_per_sample_pass(w):
    return (w.obs_dim + (1 if w.is_discrete else w.act_dim) + 7) * 4


def kernel_roofline(learner, peaks):
    """Dominant kernel = the persistent K4 launch: CUDA events around each of R launches on the launching stream.
    Both rooflines are evaluated; `bound` names the binding one (the lower attainable throughput), as SURVEY 8(d) asks."""
    import ctypes as C
    from icrl_b200 import _lib
    w = learner.w
    cfg, pol = learner.ppo_cfg(), learner.policy
    times = []
    for r in range(w.rollouts):
        data = _lib.PpoData()
        data.observations, data.actions = learner.data["obs"][r].data_ptr(), learner.data["actions"][r].data_ptr()
        data.old_log_prob = learner.log_probs[r].data_ptr()
        data.old_reward_values, data.old_cost_values = learner.reward_values[r].data_ptr(), learner.cost_values[r].data_ptr()
        data.reward_advantages, data.reward_returns = learner.adv_r[r].data_ptr(), learner.ret_r[r].data_ptr()
        data.cost_advantages, data.cost_returns = learner.adv_c[r].data_ptr(), learner.ret_c[r].data_ptr()
        data.perm, data.nu_device = learner.perm[r].data_ptr(), learner.dual.nu.state[4:5].data_ptr()
        s, e = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
        s.record()
        _lib.check(_lib.lib().icrl_ppo_train(C.byref(cfg), C.byref(data), _lib.ptr(pol._params), _lib.ptr(pol._adam_m),
                                             _lib.ptr(pol._adam_v), pol.optimizer.step_count, _lib.ptr(learner.stats[r]),
                                             _lib.ptr(learner.result[r]), _lib.current_stream()))
        e.record()
        pol.optimizer.step_count += learner.steps_taken_per_rollout()
        th.cuda.synchronize()
        times.append(s.elapsed_time(e) * 1e-3)
    dur = float(np.mean(times))
    steps = w.n_epochs * learner.steps_per_epoch
    passes = learner.n * w.n_epochs
    alg_bytes = k4_bytes_per_sample_pass(w) * passes
    alg_flops = k4_flops_per_sample_pass(w) * passes
    gbs, tfs = alg_bytes / dur / 1e9, alg_flops / dur / 1e12
    tc_peak = peaks["tf32_mma_tflops"] / 3.0          # one fp32-class product = three TF32 MMAs (hi*hi + hi*lo + lo*hi)
    t_hbm, t_tc = alg_bytes / (peaks["hbm_gbs"] * 1e9), alg_flops / (tc_peak * 1e12)
    binding = "tensor" if t_tc >= t_hbm else "hbm"
    out = {"bound": binding, "kernel": "ppo_train_kernel (K4, persistent 6-CTA cluster: a CTA pair per trunk)",
           "achieved": tfs if binding == "tensor" else gbs, "peak": tc_peak if binding == "tensor" else peaks["hbm_gbs"],
           "unit": "TFLOP/s" if binding == "tensor" else "GB/s",
           "frac": (tfs / tc_peak) if binding == "tensor" else gbs / peaks["hbm_gbs"],
           "traffic": K4_NCU_TRAFFIC_BYTES.get(learner.w.name),
           "traffic_source": "offline constant: dram__bytes_read.sum + dram__bytes_write.sum of one launch from the ncu --set full "
                             "capture summarised under profiles/ (not measured in this run)",
           "peak_source": peaks["source"],
           "hbm": {"achieved": gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": gbs / peaks["hbm_gbs"]},
           "tensor": {"achieved": tfs, "peak": tc_peak, "unit": "TFLOP/s", "frac": tfs / tc_peak,
                      "what": "fp32-class 3xTF32 products on mma.sync.m16n8k8: measured TF32 mma.sync rate / 3",
                      "frac_of_fp32_ffma_peak": tfs / peaks["fp32_tflops"],
                      "frac_of_bf16_cublas_peak": tfs / peaks["bf16_tflops"] if peaks.get("bf16_tflops") else None},
           "launch_ms": dur * 1e3, "optimiser_steps_per_launch": steps, "us_per_optimiser_step": dur / steps * 1e6,
           "algorithmic_bytes_per_launch": alg_bytes, "algorithmic_flops_per_launch": alg_flops,
           "note": f"{steps} DEPENDENT optimiser steps on {w.batch_size} rows each: neither roofline is approachable at the "
                   "reference's batch size (SURVEY 7: step latency); us_per_optimiser_step is the figure of merit here and the "
                   "batch-scaled sweep (`sweep`) is where the kernels are held against their rooflines"}
    return out


def family_rooflines(learner, peaks):
    """Per-family achieved HBM GB/s for the streaming kernels (K1 relabel, K3 GAE, K5) at the workload's rollout size."""
    import ctypes as C
    from icrl_b200 import _lib
    w, L = learner.w, _lib.lib()
    peak = peaks["hbm_gbs"]
    out = {}

    desc = learner.cn._get_desc()
    k1_bytes_row = (learner.cn.input_dims + 1) * 4
    T, E = w.n_steps, learner.E
    n = T * E
    obs = th.randn(n, w.obs_dim, device=learner.dev)
    acs = (th.randint(0, w.act_dim, (n,), device=learner.dev).float() if w.is_discrete
           else th.randn(n, w.act_dim, device=learner.dev))
    cost = th.empty(n, device=learner.dev)
    d = timeit(lambda: _lib.check(L.icrl_cn_forward(C.byref(desc), _lib.ptr(obs), 0, _lib.ptr(acs), n, _lib.ptr(cost), 0,
                                                    _lib.current_stream())))
    out["k1_rollout"] = {"rows": n, "us": d * 1e6, "GB/s": k1_bytes_row * n / d / 1e9, "frac_hbm": k1_bytes_row * n / d / 1e9 / peak}
    arrs = [th.randn(T, E, device=learner.dev) for _ in range(4)] + [(th.rand(T, E, device=learner.dev) < 0.002).float()]
    lv = [th.randn(E, device=learner.dev) for _ in range(2)] + [th.zeros(E, dtype=th.uint8, device=learner.dev)]
    outs = [th.empty(T, E, device=learner.dev) for _ in range(4)]
    d = timeit(lambda: _lib.check(L.icrl_dual_gae(*[_lib.ptr(x) for x in arrs + lv], T, E, 0.99, 0.95, 0.99, 0.95,
                                                  *[_lib.ptr(o) for o in outs], _lib.current_stream())))
    out["k3_rollout"] = {"rows": n, "us": d * 1e6, "GB/s": 36 * n / d / 1e9, "frac_hbm": 36 * n / d / 1e9 / peak}
    # K5: T-serial float64 statistics chain (bit-exact with numpy) -- latency-bound, not a bandwidth kernel
    state = th.tensor([0.0, 1.0, 1e-4] + [0.0] * E, dtype=th.float64, device=learner.dev)
    d = timeit(lambda: _lib.check(L.icrl_cost_normalize(_lib.ptr(arrs[0]), _lib.ptr(arrs[4]), _lib.ptr(lv[2]), T, E,
                                                        0.99, 1e-8, 10.0, 1, 1, _lib.ptr(state), _lib.ptr(outs[0]),
                                                        _lib.current_stream())))
    out["k5_rollout"] = {"rows": n, "us": d * 1e6, "GB/s": 13 * n / d / 1e9, "frac_hbm": 13 * n / d / 1e9 / peak}
    # the reference's DEFAULT cost path: one ConstraintNet.cost_function([n_envs, obs], [n_envs, act]) host call per environment
    # step (VecCostWrapper.step_wait, vec_cost_wrapper.py:62) -- H2D + K1 + D2H + sync every call; wall clock, host buffers
    ho = np.random.default_rng(0).standard_normal((E, w.obs_dim))
    ha = (np.random.default_rng(1).integers(0, w.act_dim, size=(E,)).astype(np.float32) if w.is_discrete
          else np.random.default_rng(1).standard_normal((E, w.act_dim)).astype(np.float32))
    for _ in range(20):
        learner.cn.cost_function(ho, ha)
    t0 = time.perf_counter()
    for _ in range(300):
        learner.cn.cost_function(ho, ha)
    per_call = (time.perf_counter() - t0) / 300
    out["k1_per_env_step_call"] = {"rows": E, "us_per_call_wall": per_call * 1e6,
                                   "us_per_rollout_wall": per_call * 1e6 * T,
                                   "note": "per-step mode (the drivers' default); the whole-buffer relabel (K1 + K5 once per "
                                           "rollout, ICRL_WHOLE_BUFFER_RELABEL=1) is what `value` / `e2e` time"}
    return out


def timeit(fn, reps=5):
    fn(); th.cuda.synchronize()
    ts = []
    for _ in range(reps):
        s, e = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
        s.record(); fn(); e.record(); th.cuda.synchronize()
        ts.append(s.elapsed_time(e) * 1e-3)
    return float(np.median(ts))


def ant_sweep(rank, world, dev, ppo_comm, peaks, sizes):
    """BASELINE config 5: synthetic Ant-shaped buffers of N transitions PER GPU (weak scaling), N in `sizes`; every kernel
    family on device-resident data, max over ranks.  K1 rows, K3 env columns shard with no collective; K2 (sharded by episodes,
    2 backward iterations, per-step IS) and K4 (batch = N/80 rows per rank -> the many-cluster kernel, 2 epochs = 160 optimiser
    steps, gradients all-reduced inside the kernel) exchange over NVLink peer memory.  Each entry carries achieved GB/s and
    TFLOP/s against the measured HBM, FP32-FFMA and 3xTF32 peaks and names the binding roofline."""
    import ctypes as C
    from icrl_b200 import _lib
    from icrl_b200.constraint_net import ConstraintNet
    from icrl_b200.learner import WORKLOADS, spaces_of
    from icrl_b200.policies import ActorTwoCriticsPolicy
    L = _lib.lib()
    w = WORKLOADS["antwall"]
    D, A = w.obs_dim, w.act_dim
    hbm, fp32, tc = peaks["hbm_gbs"], peaks["fp32_tflops"], peaks["tf32_mma_tflops"] / 3.0
    th.manual_seed(0)
    low, high = -np.ones(A, np.float32), np.ones(A, np.float32)
    obs_space, act_space = spaces_of(w)
    rows_out = []

    def entry(rows, dur, bytes_per, flops_per, compute_peak, compute_name):
        dur = max_over_ranks(dur, world)
        gbs, tfs = bytes_per * rows / dur / 1e9, flops_per * rows / dur / 1e12
        f_h, f_c = gbs / hbm, tfs / compute_peak
        t_h, t_c = bytes_per / (hbm * 1e9), flops_per / (compute_peak * 1e12)
        return {"rows_per_gpu": rows, "ms": dur * 1e3, "rows_per_s_all_gpus": rows * world / dur, "GB/s_per_gpu": gbs,
                "frac_hbm": f_h, "TFLOP/s_per_gpu": tfs, f"frac_{compute_name}": f_c, "bound": "hbm" if t_h >= t_c else compute_name,
                "frac_of_binding_roofline": f_h if t_h >= t_c else f_c}

    for N in sizes:
        T = 2048
        E = N // T
        n = T * E
        ent = {"transitions_per_gpu": n}
        obs = th.randn(n, D, device=dev) * 3.0
        acs = th.randn(n, A, device=dev)
        # ---- K1
        cn = ConstraintNet(D, A, w.cn_hidden, None, lambda _: w.cn_lr, obs[:8].cpu().numpy(), acs[:8].cpu().numpy(), False,
                           w.cn_reg, per_step_importance_sampling=True, clip_obs=20., action_low=low, action_high=high,
                           target_kl_old_new=-1, target_kl_new_old=-1, device=dev)
        desc = cn._get_desc()
        cost = th.empty(n, device=dev)
        barrier(world)
        d = timeit(lambda: _lib.check(L.icrl_cn_forward(C.byref(desc), _lib.ptr(obs), 0, _lib.ptr(acs), n, _lib.ptr(cost), 0,
                                                        _lib.current_stream())), reps=3)
        ent["k1"] = entry(n, d, (cn.input_dims + 1) * 4, 2 * (121 * 40 + 40 * 40 + 40), fp32, "fp32")
        # ---- K3
        arrs = [th.randn(T, E, device=dev) for _ in range(4)] + [(th.rand(T, E, device=dev) < 0.002).float()]
        lv = [th.randn(E, device=dev) for _ in range(2)] + [th.zeros(E, dtype=th.uint8, device=dev)]
        outs = [th.empty(T, E, device=dev) for _ in range(4)]
        barrier(world)
        d = timeit(lambda: _lib.check(L.icrl_dual_gae(*[_lib.ptr(x) for x in arrs + lv], T, E, 0.99, 0.9, 0.99, 0.9,
                                                      *[_lib.ptr(o) for o in outs], _lib.current_stream())), reps=3)
        ent["k3"] = entry(n, d, 36, 14, fp32, "fp32")
        # ---- K2: nominal n rows in 500-step episodes, expert n rows, 2 backward iterations
        iters = 2
        n_ep = n // 500
        off = th.arange(0, n_ep + 1, dtype=th.int32, device=dev) * 500
        n2 = n_ep * 500
        cfg2 = _lib.CnTrainCfg(iterations=iters, importance_sampling=1, per_step_is=1, train_gail_lambda=0, eps=1e-5,
                               regularizer_coeff=float(w.cn_reg), target_kl_old_new=-1.0, target_kl_new_old=-1.0,
                               lr=float(w.cn_lr), adam_beta1=0.9, adam_beta2=0.999, adam_eps=1e-5, batch_size=0, perm=None)
        metrics = _lib.CnTrainMetrics()
        dp = world > 1 and ppo_comm is not None
        if dp:
            cn.enable_data_parallel(max_episodes=2 * n_ep * world)

        def k2():
            step = C.c_int64(cn.optimizer.step_count)
            args = (C.byref(desc), C.byref(cfg2), _lib.ptr(obs), 0, _lib.ptr(acs), n2, _lib.ptr(off), n_ep, _lib.ptr(obs), 0,
                    _lib.ptr(acs), n, _lib.ptr(cn._adam_m), _lib.ptr(cn._adam_v), C.byref(step), C.byref(metrics))
            if dp:
                dd = cn.comm.descriptor(n2 * world, n * world, n_ep * world, n_ep * rank)
                _lib.check(L.icrl_cn_train_dist(*args, C.byref(dd), _lib.current_stream()))
                cn.comm.advance(iters)
            else:
                _lib.check(L.icrl_cn_train(*args, _lib.current_stream()))
        barrier(world)
        d = timeit(k2, reps=2)
        # per backward iteration: IS forward over the nominal rows + forward/backward over nominal and expert rows
        cn_fwd = 2 * (121 * 40 + 40 * 40 + 40)
        ent["k2"] = entry(n2 * iters, d, 121 * 4 * 3 + 12, cn_fwd + 3 * cn_fwd * 2, fp32, "fp32")
        ent["k2"]["backward_iterations"] = iters
        if dp:
            cn.comm.close()
        # ---- K4: batch = n / 80 rows per rank (80 optimiser steps per epoch like the reference's 10 240 / 128), 2 epochs
        n_epochs, B = 2, max(2048, n // 80)
        pol = ActorTwoCriticsPolicy(obs_space, act_space, lambda _: w.learning_rate, device=dev)
        spe = -(-n // B)
        cfg4 = pol.make_cfg(T=T, E=E, batch_size=B, n_epochs=n_epochs, has_target_kl=0, target_kl=0.0, clip_range=w.clip_range,
                            ent_coef=0.0, reward_vf_coef=0.5, cost_vf_coef=0.5, max_grad_norm=0.5, nu=0.1, max_steps=0)
        sc = [th.randn(T, E, device=dev) for _ in range(6)]
        logp = th.randn(T, E, device=dev) * 0.1 - 11.3
        perm = th.stack([th.randperm(n, device=dev) for _ in range(n_epochs)]).to(th.int32)
        data = _lib.PpoData()
        data.observations, data.actions, data.old_log_prob = obs.data_ptr(), acs.data_ptr(), logp.data_ptr()
        data.old_reward_values, data.reward_advantages, data.reward_returns = (x.data_ptr() for x in sc[:3])
        data.old_cost_values, data.cost_advantages, data.cost_returns = (x.data_ptr() for x in sc[3:])
        data.perm = perm.data_ptr()
        stats = th.zeros(n_epochs * spe, 8, device=dev)
        result = th.zeros(4, dtype=th.int32, device=dev)
        advsums = th.zeros(n_epochs * spe, 4, dtype=th.float64, device=dev)

        def k4():
            if dp:
                _lib.check(L.icrl_ppo_local_advsums(C.byref(cfg4), C.byref(data), _lib.ptr(advsums), _lib.current_stream()))
                ppo_comm.all_reduce_sum(advsums)
                dd = ppo_comm.descriptor(advsums)
                _lib.check(L.icrl_ppo_train_dist(C.byref(cfg4), C.byref(data), _lib.ptr(pol._params), _lib.ptr(pol._adam_m),
                                                 _lib.ptr(pol._adam_v), pol.optimizer.step_count, _lib.ptr(stats),
                                                 _lib.ptr(result), C.byref(dd), _lib.current_stream()))
                ppo_comm.advance(n_epochs * spe)
            else:
                _lib.check(L.icrl_ppo_train(C.byref(cfg4), C.byref(data), _lib.ptr(pol._params), _lib.ptr(pol._adam_m),
                                            _lib.ptr(pol._adam_v), pol.optimizer.step_count, _lib.ptr(stats), _lib.ptr(result),
                                            _lib.current_stream()))
            pol.optimizer.step_count += n_epochs * spe
        barrier(world)
        d = timeit(k4, reps=2)
        res = result.cpu().numpy()
        ent["k4"] = entry(n * n_epochs, d, k4_bytes_per_sample_pass(w), k4_flops_per_sample_pass(w), tc, "tensor_3xtf32")
        ent["k4"].update(batch_size_per_gpu=B, global_batch=B * (world if dp else 1), optimiser_steps=int(res[1]), peer_timeout=bool(res[2]),
                         us_per_optimiser_step=max_over_ranks(d, world) / max(int(res[1]), 1) * 1e6)
        rows_out.append(ent)
        del obs, acs, cost, arrs, outs, sc, logp, perm, stats, advsums, pol, cn
        th.cuda.empty_cache()
    return rows_out


DUMP_LIMIT_BYTES = 64 * 1024 * 1024


def dump_outputs(learner, out_dir):
    """What the last DeviceLearner.run() computed, as out_dir/<name>.npy: per rollout the K1 costs (and their K5
    normalisation), K3 advantages and returns and K4 per-optimiser-step statistics; the policy, constraint net, Adam
    moments, dual variable and cost statistics the iteration leaves behind; the K2 metrics.  float32, or float64 where the
    path keeps float64.  Must run before anything else touches the learner: the e2e leg trains the same constraint net and
    the roofline relaunches K4."""
    w, pol, cn = learner.w, learner.policy, learner.cn
    arrays = {"costs": learner.costs, "reward_advantages": learner.adv_r, "reward_returns": learner.ret_r,
              "cost_advantages": learner.adv_c, "cost_returns": learner.ret_c, "ppo_step_stats": learner.stats,
              "policy_params": pol._params, "policy_adam_m": pol._adam_m, "policy_adam_v": pol._adam_v,
              "dual_state": learner.dual.nu.state, "cn_params": cn._params, "cn_adam_m": cn._adam_m, "cn_adam_v": cn._adam_v}
    if w.normalize_cost:
        arrays.update(normalized_costs=learner.costs_norm, cost_norm_state=learner.cost_state)
    arrays = {k: v.cpu().numpy() for k, v in arrays.items()}
    if w.backward_iters > 0 and w.nominal_rows > 0:
        m = learner.last_cn_metrics
        arrays["cn_train_metrics"] = np.array([getattr(m, f) for f, _ in m._fields_], np.float64)
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_LIMIT_BYTES, f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit"
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (k, a.dtype)
        np.save(os.path.join(out_dir, k + ".npy"), a)


def run_workload(name, args, rank, world, local, ppo_comm, peaks, flush, steps, warmup, want_e2e, want_family, dump_dir=None):
    """value (device-resident DeviceLearner), e2e (host-buffer public API) and the K4 launch roofline of one named workload;
    with `dump_dir`, rank 0 also writes what the last timed step computed (dump_outputs)."""
    from icrl_b200 import _lib
    from icrl_b200.learner import WORKLOADS, DeviceLearner
    w = WORKLOADS[name]
    dev = th.device("cuda", local)
    # data parallel: every rank owns n_envs environments (its own rollouts, seed = rank); networks replicated
    learner = DeviceLearner(w, seed=rank, device=dev, comm=ppo_comm, param_seed=0)
    for _ in range(warmup):
        learner.run()
    th.cuda.synchronize()
    learner.check()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    launches0 = _lib.lib().icrl_launch_count()
    t_dev = time_steps(learner.run, steps, world, flush)
    launches = _lib.lib().icrl_launch_count() - launches0
    clocks = sampler.stop() if rank == 0 else None
    learner.check()                                   # raises on an exchange time-out (result[2]) in any K4 launch
    if dump_dir is not None and rank == 0:
        dump_outputs(learner, dump_dir)
    per_step = t_dev / steps
    total_tr = w.transitions_per_iteration * world
    out = {"workload": w.name, "value": total_tr / per_step, "unit": UNIT, "ms_per_step": per_step * 1e3, "steps": steps,
           "warmup": warmup, "gpu_launches": int(launches), "clocks": clocks}
    dp = world > 1 and ppo_comm is not None
    par = "1 GPU" if world == 1 else (
        f"{world} independent learner replicas" if not dp else
        f"dp{world}: env-sharded rollouts (K1/K5/K3 local), K4 gradients all-reduced inside the persistent kernel over NVLink "
        f"peer memory every optimiser step (global batch {w.batch_size * world}), K2 sharded by episodes with in-kernel "
        f"exchanges")
    out["parallelism"] = par
    if want_e2e:
        hl = HostLearner(w, learner, rank)
        for _ in range(2):
            hl.run()
        th.cuda.synchronize()
        barrier(world)
        t0 = time.perf_counter()
        for _ in range(steps):
            hl.run()
        th.cuda.synchronize()
        t_e2e = max_over_ranks(time.perf_counter() - t0, world) / steps
        out["e2e"] = {"value": total_tr / t_e2e, "unit": UNIT,
                      "parallelism": "1 GPU" if world == 1 else (f"dp{world} through PPOLagrangian.train / ConstraintNet.train "
                                                                 "(enable_data_parallel)" if dp else f"{world} independent replicas"),
                      "h2d_bytes_per_step": int(hl.h2d), "d2h_bytes_per_step": int(hl.d2h), "ms_per_step": t_e2e * 1e3,
                      "path": "RolloutBufferWithCost.relabel_costs (or ConstraintNet.cost_function) / compute_returns_and_advantage"
                              " / PPOLagrangian.train / ConstraintNet.train with numpy buffers (pinned staging + async H2D, "
                              "D2H of costs, advantages, per-step stats, metrics)"}
    if dp:
        # soak evidence for the fence-less, self-validating NVLink exchange: after every warm-up + timed step of BOTH legs the
        # replicated parameters and Adam moments (policy and constraint net) must still be bit-identical on all ranks
        per_iter = w.rollouts * learner.steps_taken_per_rollout()
        tensors = [learner.policy._params, learner.policy._adam_m, learner.policy._adam_v, learner.cn._params,
                   learner.cn._adam_m, learner.cn._adam_v]
        n_exchanged = (warmup + steps) * per_iter
        if want_e2e:
            pol = hl.algo.policy
            tensors += [pol._params, pol._adam_m, pol._adam_v]
            n_exchanged += (2 + steps) * per_iter
        same = replicas_identical(tensors, world)
        out["replicas"] = {"bit_identical_after_run": same, "k4_exchange_steps": int(n_exchanged),
                           "k2_exchange_iterations": int((warmup + steps + (2 + steps if want_e2e else 0)) * w.backward_iters)}
        if not same:
            raise SystemExit(f"data-parallel replicas DIVERGED during the {name} run: {out['replicas']}")
    if rank == 0:
        out["roofline"] = kernel_roofline(learner, peaks)
        if want_family:
            out["kernels"] = family_rooflines(learner, peaks)
    return out, learner


def replicas_identical(tensors, world):
    """Data parallel: every rank must hold bit-identical copies of `tensors` (two order-sensitive 64-bit digests, all-gathered)."""
    import torch.distributed as dist
    flat = th.cat([t.detach().reshape(-1).view(th.int32).to(th.int64) for t in tensors])
    weights = th.arange(flat.numel(), device=flat.device, dtype=th.int64) % 65521 + 1
    h = th.stack([flat.sum(), (flat * weights).sum()])
    got = [th.zeros_like(h) for _ in range(world)]
    dist.all_gather(got, h)
    return all(bool((g == got[0]).all()) for g in got)


def all_peaks():
    """HBM (and bf16) from the driver-written MEASURED_PEAKS.json, FP32-FFMA and TF32 mma.sync measured here."""
    import ctypes as C
    from icrl_b200 import _lib
    hbm, src = measured_peaks()
    bf16 = None
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            bf16 = json.load(f).get("bf16_tflops")
    two = (C.c_double * 2)()
    _lib.check(_lib.lib().icrl_measure_peaks(two, _lib.current_stream()))
    return {"hbm_gbs": hbm, "bf16_tflops": bf16, "fp32_tflops": float(two[0]), "tf32_mma_tflops": float(two[1]),
            "source": f"HBM: {src}; FP32 FFMA {two[0]:.1f} TFLOP/s and mma.sync TF32 {two[1]:.1f} TFLOP/s measured in this run "
                      "(icrl_measure_peaks: the instructions the kernels issue, every SM busy)"}


def main():
    args = parse()
    from icrl_b200.learner import WORKLOADS
    w = WORKLOADS[args.workload]
    if args.impl == "reference":
        return run_reference(args, w)
    assert args.warmup >= 3, "timing rules: at least 3 warm-up steps"
    rank, world, local = dist_setup(args.gpus)
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world} (launch with torch.distributed.run)"
    th.cuda.set_device(local)
    dev = th.device("cuda", local)
    peaks = all_peaks()
    ppo_comm, dp_parity = None, None
    if world > 1 and not args.replicas:
        from icrl_b200.distributed import PpoComm
        ppo_comm = PpoComm()
        # data-parallel parity before anything is timed: rank-0 oracle check + bit-identical replicas across ranks
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import dp_worker
        dp_parity = [dp_worker.ppo_parity(rank, world, dev, "hc", comm=ppo_comm),
                     dp_worker.ppo_parity(rank, world, dev, "ant", comm=ppo_comm),
                     dp_worker.ppo_parity(rank, world, dev, "ant", wide=True, comm=ppo_comm),
                     dp_worker.cn_parity(rank, world, dev, "hc", per_step=True),
                     dp_worker.cn_parity(rank, world, dev, "ant", per_step=False)]
        if not all(p["ok"] for p in dp_parity):
            raise SystemExit(f"data-parallel parity FAILED, nothing timed: {dp_parity}")
    flush = th.zeros(64 * 1024 * 1024, device="cuda")      # 256 MB
    main_out, learner = run_workload(args.workload, args, rank, world, local, ppo_comm, peaks, flush, args.steps, args.warmup,
                                     not args.no_e2e, True, dump_dir=args.dump_outputs)
    del learner
    th.cuda.empty_cache()
    # the other BASELINE configs, short runs (N>1: AntWall only -- BASELINE config 3 is "AntWall on 1/2/4/8 B200")
    others = {}
    if not args.no_workloads:
        names = [n for n in (("antwall", "lapgrid", "pointcircle") if world == 1 else ("antwall",)) if n != args.workload]
        for n in names:
            o, lrn = run_workload(n, args, rank, world, local, ppo_comm, peaks, flush, args.aux_steps, 3, not args.no_e2e, False)
            others[n] = o
            del lrn
            th.cuda.empty_cache()
    sweep = None
    if not args.no_sweep:
        sizes = [int(x) for x in args.sweep_sizes.split(",")]
        sweep = ant_sweep(rank, world, dev, ppo_comm, peaks, sizes)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        from baseline import reference_arm as ra
        if ra.available():
            cpu = reference_samples(w, 1, 2, budget_s=24.0)
        else:
            cpu = port_samples(w, args, 1, 1)
    barrier(world)
    if rank == 0:
        print(json.dumps({
            "metric": METRIC, "value": main_out["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": main_out["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(w, world, main_out["parallelism"]),
            "clocks": main_out["clocks"], "e2e": main_out.get("e2e"), "gpu_launches": main_out["gpu_launches"],
            "roofline": main_out.get("roofline"), "kernels": main_out.get("kernels"), "peaks": peaks,
            "dp_parity": None if dp_parity is None else {"ok": True, "checks": dp_parity,
                                                          "max_param_err": max(p["max_param_err"] for p in dp_parity),
                                                          "replicas_after_timed_runs": {
                                                              **{args.workload: main_out.get("replicas")},
                                                              **{k: v.get("replicas") for k, v in others.items()}}},
            "workloads": others, "sweep": sweep, "cpu_baseline": cpu}))
    if ppo_comm is not None:
        ppo_comm.close()
    if world > 1:
        import torch.distributed as dist
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
