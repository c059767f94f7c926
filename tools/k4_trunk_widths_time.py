"""K4 optimiser-step time per library build, alternating the builds, for policies with uniform 64-64 trunks, with
per-trunk widths and with shared trunk layers.

Shapes (one K4 launch each; us per optimiser step from CUDA events over `--launches` launches after one warm-up):
  hc            HalfCheetah: obs 18, 6 actions, batch 64, 10 epochs, one 10 240-row rollout (single cluster)
  antwall       AntWall: obs 113, 8 actions, batch 128, 20 epochs, one 10 240-row rollout (single cluster)
  ant_wide      Ant-shaped many-cluster launch: obs 113, 8 actions, 262 144 rows, batch 4 096, 2 epochs
  hc_mixed      the hc shape with pi (64, 64), vf (32, 32), cvf (16, 48); its 64-64 embedding is `hc`
  ant_mixed     the antwall shape with pi (64, 64), vf (64, 32), cvf (48, 64)
  hc_sl1        the hc shape with net_arch [64, dict(pi=[64], vf=[32], cvf=[16])] (-sl 64); hc_sl1_sep: the same widths
                as separate trunks, pi (64, 64), vf (64, 32), cvf (64, 16)
  ant_sl1       the antwall shape (two chunks per step) with [64, dict(pi=[64], vf=[64], cvf=[48])]; ant_sl1_sep
  hc_sl2        the hc shape with one trunk under all three heads, [64, 64]; its separate-trunk net is `hc`
  ant_wide_sl1  the ant_wide shape (many clusters) with [64, dict(pi=[64], vf=[64], cvf=[64])]; its separate net is
                `ant_wide`
The *_mixed, *_sep and *_sl* shapes run only on builds that take per-trunk widths and shared layers (`name=path+`).

Usage: python tools/k4_trunk_widths_time.py [--reps 5] [--launches 5] name=path/to/libicrl_b200.so[+] ...
  e.g. branch=icrl_b200/libicrl_b200.so+ parent=tools/_variants/parent.so
Each (repeat, build) pair runs in its own process; the builds alternate, in reversed order on odd repeats.  Prints the
card name and power limit, every run's numbers and, per shape and build, the median and the spread (min..max)."""
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = {   # obs_dim, actions, rows (T x E), batch, epochs, trunks
    "hc": (18, 6, (2048, 5), 64, 10, ((64, 64),) * 3),
    "antwall": (113, 8, (2048, 5), 128, 20, ((64, 64),) * 3),
    "ant_wide": (113, 8, (2048, 128), 4096, 2, ((64, 64),) * 3),
    "hc_mixed": (18, 6, (2048, 5), 64, 10, ((64, 64), (32, 32), (16, 48))),
    "ant_mixed": (113, 8, (2048, 5), 128, 20, ((64, 64), (64, 32), (48, 64))),
    "hc_sl1": (18, 6, (2048, 5), 64, 10, [64, dict(pi=[64], vf=[32], cvf=[16])]),   # a list: net_arch itself
    "hc_sl1_sep": (18, 6, (2048, 5), 64, 10, ((64, 64), (64, 32), (64, 16))),
    "ant_sl1": (113, 8, (2048, 5), 128, 20, [64, dict(pi=[64], vf=[64], cvf=[48])]),
    "ant_sl1_sep": (113, 8, (2048, 5), 128, 20, ((64, 64), (64, 64), (64, 48))),
    "hc_sl2": (18, 6, (2048, 5), 64, 10, [64, 64]),
    "ant_wide_sl1": (113, 8, (2048, 128), 4096, 2, [64, dict(pi=[64], vf=[64], cvf=[64])]),
}


def child(lib_path, mixed, launches):
    sys.path.insert(0, ROOT)
    import torch as th
    from icrl_b200 import _lib
    _lib.LIB_PATH = os.path.abspath(lib_path)
    from icrl_b200.policies import ActorTwoCriticsPolicy
    from icrl_b200.spaces import Box
    explicit = ActorTwoCriticsPolicy.make_cfg

    def make_cfg(self, **kw):      # also fill hidden[], which is all a build without per-trunk widths reads
        cfg = explicit(self, **kw)
        cfg.hidden[0], cfg.hidden[1] = self.trunk_hidden[0]
        return cfg
    ActorTwoCriticsPolicy.make_cfg = make_cfg
    L = _lib.lib()
    dev = th.device("cuda")
    out = {}
    for name, (D, A, (T, E), B, n_epochs, trunks) in SHAPES.items():
        uniform = isinstance(trunks, tuple) and len(set(trunks)) == 1
        if not uniform and not mixed:
            continue
        th.manual_seed(0)
        net_arch = trunks if isinstance(trunks, list) else [dict(zip(("pi", "vf", "cvf"), (list(t) for t in trunks)))]
        pol = ActorTwoCriticsPolicy(Box(-1e9, 1e9, (D,)), Box(-1, 1, (A,)), lambda _: 3e-4, device=dev,
                                    net_arch=net_arch)
        n = T * E
        obs = th.randn(n, D, device=dev)
        acs = th.randn(n, A, device=dev)
        sc = [th.randn(T, E, device=dev) for _ in range(6)]
        logp = th.randn(T, E, device=dev) * 0.1 - 11.3
        perm = th.stack([th.randperm(n, device=dev) for _ in range(n_epochs)]).to(th.int32)
        spe = -(-n // B)
        cfg = pol.make_cfg(T=T, E=E, batch_size=B, n_epochs=n_epochs, has_target_kl=0, target_kl=0.0, clip_range=0.2,
                           ent_coef=0.0, reward_vf_coef=0.5, cost_vf_coef=0.5, max_grad_norm=0.5, nu=0.1, max_steps=0)
        data = _lib.PpoData()
        data.observations, data.actions, data.old_log_prob = obs.data_ptr(), acs.data_ptr(), logp.data_ptr()
        data.old_reward_values, data.reward_advantages, data.reward_returns = (x.data_ptr() for x in sc[:3])
        data.old_cost_values, data.cost_advantages, data.cost_returns = (x.data_ptr() for x in sc[3:])
        data.perm = perm.data_ptr()
        stats = th.zeros(n_epochs * spe, 8, device=dev)
        result = th.zeros(4, dtype=th.int32, device=dev)
        times = []
        for rep in range(launches + 1):
            s, e = th.cuda.Event(enable_timing=True), th.cuda.Event(enable_timing=True)
            s.record()
            _lib.check(L.icrl_ppo_train(C.byref(cfg), C.byref(data), _lib.ptr(pol._params), _lib.ptr(pol._adam_m),
                                        _lib.ptr(pol._adam_v), pol.optimizer.step_count, _lib.ptr(stats),
                                        _lib.ptr(result), _lib.current_stream()))
            e.record()
            th.cuda.synchronize()
            assert int(result[1]) == n_epochs * spe, result
            pol.optimizer.step_count += n_epochs * spe
            if rep:
                times.append(s.elapsed_time(e) * 1e3 / (n_epochs * spe))
        out[name] = sorted(times)[len(times) // 2]
    print("RESULT " + json.dumps(out), flush=True)


def main(argv):
    reps, launches, builds = 5, 5, []
    it = iter(argv)
    for a in it:
        if a == "--reps":
            reps = int(next(it))
        elif a == "--launches":
            launches = int(next(it))
        else:
            name, path = a.split("=", 1)
            builds.append((name, path.rstrip("+"), path.endswith("+")))
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip().splitlines()
    print(f"card: {card[0] if card else 'unknown'}")
    runs = {b[0]: [] for b in builds}
    for rep in range(reps):
        for name, path, mixed in (builds if rep % 2 == 0 else builds[::-1]):
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--child", path, str(int(mixed)),
                                str(launches)], capture_output=True, text=True, cwd=ROOT)
            line = [x for x in r.stdout.splitlines() if x.startswith("RESULT ")]
            if r.returncode != 0 or not line:
                raise SystemExit(f"{name} failed:\n{r.stdout[-2000:]}\n{r.stderr[-2000:]}")
            res = json.loads(line[0][7:])
            runs[name].append(res)
            print(f"rep {rep} {name:8s} " + "  ".join(f"{k} {v:.2f}" for k, v in res.items()), flush=True)
    print("us per optimiser step: median (min..max) over the repeats")
    for shape in SHAPES:
        cells = []
        for name, _, _ in builds:
            v = sorted(r[shape] for r in runs[name] if shape in r)
            if v:
                cells.append(f"{name} {v[len(v) // 2]:.2f} ({v[0]:.2f}..{v[-1]:.2f})")
        print(f"  {shape:12s} " + "   ".join(cells))


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "--child":
        child(sys.argv[2], sys.argv[3] == "1", int(sys.argv[4]))
    else:
        main(sys.argv[1:])
