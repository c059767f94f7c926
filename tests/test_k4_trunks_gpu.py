"""GPU: policies whose pi, vf and cvf trunks have different widths (net_arch=[dict(pi=[a, b], vf=[c, d], cvf=[e, f])],
the reference's -pl / -rvl / -cvl flags) through K4 training, the policy forward, checkpoints and the drivers.

Checks per case:
* embedding, oracle-free and bit exact: the mixed net's weights placed into a uniform 64-64 net with zeros in the extra
  rows and columns.  The padded units then have zero weights and bias, tanh(0) = 0, and every gradient into them is a
  product with an exact zero, so two train() calls of the mixed net give the same bits as the embedded net (parameters,
  both Adam moments, every stats column, the early-stop epoch), and the embedded net's padding stays exactly 0;
* trajectory against oracle.ppo.train, chain-free gradient against float64 and determinism, with the routines and
  tolerances of tests/test_k4_sweep_gpu.py;
* policy forward and evaluate_actions against float64;
plus zero vs explicit trunk_hidden, refusals, checkpoints and the run_me.py drivers.
"""
import glob
import io
import json
import os
import subprocess
import sys
import zipfile
from collections import OrderedDict
from dataclasses import replace

import numpy as np
import pytest
import torch as th

import test_k4_sweep_gpu as sweep
from helpers import FakeVecEnv
from k4_trunks_helpers import embed, init_policy_trunks
from oracle import ppo as oppo
from test_k4_sweep_gpu import NP_SEED, TRAJ_LR, Case, check_gradient, check_trajectory, time_major

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")

# Case.hidden holds one (h0, h1) pair per trunk: (pi, vf, cvf)
CASES = {
    # ---- single cluster, continuous
    "hc_d18_c6": Case(18, ((64, 64), (32, 32), (16, 48)), A=6, B=64),
    "ant_d113_c8_b128": Case(113, ((64, 64), (64, 32), (48, 64)), A=8, B=128),     # NT1 = 8, two chunks per step
    "d30_c12_pi_narrow": Case(30, ((7, 33), (48, 48), (64, 40)), A=12, T=50, B=100, ent=0.01),  # both head lanes
    # ---- single cluster, discrete
    "lgw_d1_d2": Case(1, ((20, 20), (64, 64), (1, 64)), A=2, disc=True, T=50, B=40, ent=0.02),
    # ---- every trunk's widths differ from the other two's and are swapped between trunks
    "permuted_d30_c4": Case(30, ((33, 7), (7, 33), (64, 1)), A=4, T=48, B=64),
    # ---- value clipping on each head, heads of different widths
    "vfclip_d20_c5": Case(20, ((64, 64), (24, 40), (40, 24)), A=5, cvf_r=0.2, cvf_c=0.3),
    # ---- many clusters: natural (batch_size >= 2048) and forced with a few clusters
    "wide_d18_b2048": Case(18, ((64, 64), (32, 32), (16, 48)), A=6, T=1050, B=2048, many=True),
    "forced_d40_cl4": Case(40, ((20, 20), (48, 24), (64, 16)), A=6, T=160, B=256, wide=4, many=True, ent=0.01),
}


_SWEEP_MAKE_DATA = sweep.make_data


class _SweepOracle:
    """oracle.ppo as tests/test_k4_sweep_gpu.py sees it, with init_policy taking one (h0, h1) pair per trunk."""

    def __getattr__(self, name):
        return getattr(oppo, name)

    @staticmethod
    def init_policy(obs_dim, act_dim, is_discrete, hidden, generator=None):
        return init_policy_trunks(obs_dim, act_dim, is_discrete, hidden, generator=generator)


def make_data(c: Case):
    """tests/test_k4_sweep_gpu.py::make_data for a per-trunk Case.hidden (the sweep's seeded rollout generator, with the
    starting policy drawn by init_policy_trunks)."""
    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(sweep, "oppo", _SweepOracle())
        return _SWEEP_MAKE_DATA(c)


def arch(c: Case):
    return dict(zip(("pi", "vf", "cvf"), (list(t) for t in c.hidden)))


def build_algo(c: Case, d, lr):
    """tests/test_k4_sweep_gpu.py::build_algo with per-trunk net_arch."""
    from icrl_b200.ppo_lag import PPOLagrangian
    algo = PPOLagrangian("TwoCriticsMlpPolicy", FakeVecEnv(c.D, c.A, c.disc, c.E), n_steps=c.T, batch_size=c.B,
                         n_epochs=c.epochs, learning_rate=lr, clip_range=c.clip, target_kl=c.target_kl, ent_coef=c.ent,
                         max_grad_norm=c.mgn, penalty_initial_value=c.nu, penalty_learning_rate=sweep.PENALTY_LR,
                         clip_range_reward_vf=c.cvf_r, clip_range_cost_vf=c.cvf_c,
                         policy_kwargs=dict(net_arch=[arch(c)]), seed=3, device="cuda")
    assert algo.policy.parameter_names() == oppo.param_names(c.disc)
    assert algo.policy.trunk_hidden == c.hidden
    algo.policy.load_state_dict({n: p.clone() for n, p in d["P"].items()})
    buf = algo.rollout_buffer
    for k, src in sweep.BUF_FIELDS.items():
        getattr(buf, k)[:] = time_major(c, d["flat"][src]).reshape(getattr(buf, k).shape)
    buf.orig_costs[:] = time_major(c, d["orig_costs"])
    buf.full, buf.pos = True, c.T
    return algo


@pytest.fixture
def mixed(monkeypatch):
    """The sweep's routines, building the per-trunk policy; the case's cluster regime in the environment."""
    monkeypatch.setattr(sweep, "build_algo", build_algo)
    monkeypatch.setattr(sweep, "make_data", make_data)

    def setup(name):
        c = CASES[name]
        sweep._env(c, monkeypatch)
        return c
    return setup


def named(pol, flat):
    return OrderedDict((n, flat[off:off + int(np.prod(shape))].reshape(shape).cpu())
                       for n, (off, shape) in zip(pol.parameter_names(), pol._slices))


def train_twice(algo):
    from icrl_b200 import logger
    logger.configure()
    np.random.seed(NP_SEED)
    out = []
    for _ in range(2):
        algo.train()
        pol = algo.policy
        out.append(dict(params=named(pol, pol._params), m=named(pol, pol._adam_m), v=named(pol, pol._adam_v),
                        stats=algo.last_train_stats.copy(), steps=pol.optimizer.step_count,
                        early=int(logger.Logger.CURRENT.name_to_value["train/early_stop_epoch"])))
    return out


def check_embedding(c: Case):
    d = make_data(c)
    c64 = replace(c, hidden=((64, 64),) * 3)
    d64 = dict(d, P=embed(d["P"], c.D, c.A, c.disc))
    got, want = train_twice(build_algo(c, d, TRAJ_LR)), train_twice(build_algo(c64, d64, TRAJ_LR))
    for call, (g, w) in enumerate(zip(got, want), 1):
        assert g["steps"] == w["steps"] and g["early"] == w["early"], call
        assert np.array_equal(g["stats"], w["stats"]), f"call {call}: stats differ"
        for key in ("params", "m", "v"):
            for n, t in g[key].items():
                big = w[key][n]
                inner = tuple(slice(0, s) for s in t.shape)
                assert th.equal(t, big[inner]), f"call {call}: {key} {n} differs from the embedded net's"
                pad = big.clone()
                pad[inner] = 0.0
                assert th.equal(pad, th.zeros_like(pad)), f"call {call}: {key} {n}: padding of the 64-64 net moved"


@pytest.mark.parametrize("name", list(CASES))
def test_embedding_in_64x64_is_bit_exact(name, mixed):
    check_embedding(mixed(name))


@pytest.mark.parametrize("name", list(CASES))
def test_trajectory_vs_oracle(name, mixed):
    check_trajectory(mixed(name))


@pytest.mark.parametrize("name", list(CASES))
def test_gradient_vs_float64(name, mixed):
    check_gradient(mixed(name))          # includes the clip-edge guard and a bit-identical repeat


FWD_ROWS = (1, 64, 65, 100_003)


@pytest.mark.parametrize("name", list(CASES))
def test_policy_forward_vs_float64(name):
    c = CASES[name]
    d = make_data(c)
    pol = build_algo(c, d, TRAJ_LR).policy
    P64 = {k: v.double() for k, v in d["P"].items()}
    rng = np.random.default_rng(5)
    worst = 0.0
    for n in FWD_ROWS:
        obs = (rng.standard_normal((n, c.D)) * 1.5).astype(np.float32)
        acts = (rng.integers(0, c.A, (n, 1)) if c.disc else rng.standard_normal((n, c.A))).astype(np.float32)
        head, v, cv = (x.cpu().numpy() for x in pol.forward_heads(th.tensor(obs)))
        ev, ecv, lp, ent = (x.cpu().numpy() for x in pol.evaluate_actions(th.tensor(obs).cuda(), th.tensor(acts).cuda()))
        rows = np.arange(n) if n < 10_000 else np.unique(np.concatenate(
            [np.arange(2048), np.arange(n - 2048, n), rng.integers(0, n, 4096)]))
        o64, a64 = th.tensor(obs[rows], dtype=th.float64), th.tensor(acts[rows], dtype=th.float64)
        with th.no_grad():
            wh, wv, wcv = oppo.policy_forward_mean(P64, o64, c.disc)
            _, _, wlp, went = oppo.evaluate_actions(P64, o64, a64.long().flatten() if c.disc else a64, c.disc)
        for got, want, what in ((head[rows], wh, "head"), (v[rows], wv.ravel(), "value"),
                                (cv[rows], wcv.ravel(), "cost value"), (ev[rows].ravel(), wv.ravel(), "evaluate value"),
                                (ecv[rows].ravel(), wcv.ravel(), "evaluate cost value"), (lp[rows], wlp, "log-prob"),
                                (ent[rows], went, "entropy")):
            want = want.numpy()
            worst = max(worst, float(np.max(np.abs(got - want) / (1e-6 + 1e-5 * np.abs(want)))))
            np.testing.assert_allclose(got, want, rtol=1e-5, atol=1e-6, err_msg=f"{what}, {n} rows")
    print(f"\n  forward: worst error {worst:.2f} x the tolerance", end="")


# ------------------------------------------------------------------------------------------------ zero vs explicit
@pytest.mark.parametrize("regime", ["single", "forced_wide"])
def test_zero_trunk_hidden_equals_explicit_uniform_widths(regime, monkeypatch):
    """trunk_hidden all zero (hidden[] for every trunk, what zero-initialising C callers pass) and trunk_hidden set to the
    same widths train and evaluate to the same bits."""
    c = Case(18, ((48, 24),) * 3, A=6, B=64) if regime == "single" else \
        Case(18, ((48, 24),) * 3, A=6, T=160, B=256, wide=4, many=True)
    sweep._env(c, monkeypatch)
    d = make_data(c)
    obs = th.tensor(np.random.default_rng(9).standard_normal((1000, c.D)), dtype=th.float32)
    runs = []
    for zero in (False, True):
        algo = build_algo(c, d, TRAJ_LR)
        pol = algo.policy
        if zero:
            explicit = pol.make_cfg

            def make_cfg(**kw):
                cfg = explicit(**kw)
                cfg.hidden[0], cfg.hidden[1] = 48, 24
                for t in range(3):
                    cfg.trunk_hidden[t][0] = cfg.trunk_hidden[t][1] = 0
                return cfg
            pol.make_cfg = make_cfg
        out = train_twice(algo)
        runs.append((out, [x.cpu() for x in pol.forward_heads(obs)]))
    (a, fa), (b, fb) = runs
    for g, w in zip(a, b):
        assert np.array_equal(g["stats"], w["stats"]) and g["early"] == w["early"]
        for key in ("params", "m", "v"):
            assert all(th.equal(g[key][n], w[key][n]) for n in g[key]), key
    assert all(th.equal(x, y) for x, y in zip(fa, fb))


# ------------------------------------------------------------------------------------------------ refusals
@pytest.mark.parametrize("net_arch,trunk", [
    (dict(pi=[64, 64], vf=[64, 65], cvf=[64, 64]), "vf"),
    (dict(pi=[64, 64], vf=[32], cvf=[64, 64]), "vf"),
    (dict(pi=[64, 64], vf=[64, 64], cvf=[16, 16, 16]), "cvf"),
    (dict(pi=[64, 64], vf=[64, 64]), "cvf"),
    (dict(pi=[0, 64], vf=[64, 64], cvf=[64, 64]), "pi"),
])
def test_unsupported_trunks_are_refused_at_construction(net_arch, trunk):
    from icrl_b200.ppo_lag import PPOLagrangian
    with pytest.raises(NotImplementedError, match=f"the {trunk} trunk"):
        PPOLagrangian("TwoCriticsMlpPolicy", FakeVecEnv(8, 4, False, 4), n_steps=8, batch_size=32,
                      policy_kwargs=dict(net_arch=[net_arch]), device="cuda")


def test_refused_train_leaves_the_state_alone():
    from icrl_b200 import _lib
    c = CASES["hc_d18_c6"]
    algo = build_algo(c, make_data(c), TRAJ_LR)
    pol = algo.policy
    pol._adam_m.fill_(0.25)
    pol._adam_v.fill_(0.5)
    before = [t.clone() for t in (pol._params, pol._adam_m, pol._adam_v)]
    pol.trunk_hidden = ((64, 64), (64, 65), (16, 48))
    with pytest.raises(_lib.IcrlError, match=r"trunk_hidden\[1\] \(vf\)"):
        algo.train()
    for a, b in zip(before, (pol._params, pol._adam_m, pol._adam_v)):
        assert th.equal(a, b)
    assert pol.optimizer.step_count == 0


# ------------------------------------------------------------------------------------------------ checkpoints
def test_save_load_round_trip_keeps_mixed_widths(tmp_path):
    from icrl_b200.ppo_lag import PPOLagrangian
    c = CASES["permuted_d30_c4"]
    algo = build_algo(c, make_data(c), TRAJ_LR)
    np.random.seed(NP_SEED)
    algo.train()
    algo.dual.update_parameter(0.3)
    path = str(tmp_path / "mixed")
    algo.save(path)
    again = PPOLagrangian.load(path)
    assert again.policy.trunk_hidden == c.hidden
    assert th.equal(again.policy.parameters_flat(), algo.policy.parameters_flat())
    assert th.equal(again.policy._adam_m, algo.policy._adam_m) and th.equal(again.policy._adam_v, algo.policy._adam_v)
    assert th.equal(again.dual.nu.state, algo.dual.nu.state) and again.dual.steps == algo.dual.steps
    assert again.policy.optimizer.step_count == algo.policy.optimizer.step_count


REF_TRUNKS = ((64, 48), (32, 64), (16, 8))


def _cut(t, name, trunks):
    """The reference 64-64 tensor `name` cut down to the per-trunk widths (leading rows / columns)."""
    if name == "log_std":
        return t.clone()
    if name.startswith("mlp_extractor."):
        _, trunk, layer, kind = name.split(".")
        h0, h1 = trunks[oppo.TRUNKS.index(trunk)]
        out_f, in_f = (h0, None) if layer == "0" else (h1, h0)
    else:
        out_f, in_f = None, trunks[("action_net", "value_net", "cost_value_net").index(name.split(".")[0])][1]
    return (t[:out_f, :in_f] if t.dim() == 2 else t[:out_f]).clone()


def test_reference_layout_zip_with_mixed_widths_loads_and_evaluates(tmp_path):
    """tests/golden/ref_hc_best_model.zip rewritten to mixed trunk widths (policy.pth, the optimiser moments and
    data["policy_kwargs"]["net_arch"]) loads, keeps its moments, and evaluates like the float64 oracle."""
    from icrl_b200.ppo_lag import PPOLagrangian
    src = os.path.join(GOLD, "ref_hc_best_model.zip")
    path = str(tmp_path / "ref_mixed.zip")
    with zipfile.ZipFile(src) as zin, zipfile.ZipFile(path, "w") as zout:
        for item in zin.namelist():
            raw = zin.read(item)
            if item == "data":
                data = json.loads(raw)
                data["policy_kwargs"]["net_arch"] = [dict(zip(("pi", "vf", "cvf"), (list(t) for t in REF_TRUNKS)))]
                raw = json.dumps(data).encode()
            elif item == "policy.pth":
                sd = th.load(io.BytesIO(raw), map_location="cpu", weights_only=False)
                sd = OrderedDict((n, _cut(t, n, REF_TRUNKS)) for n, t in sd.items())
                buf = io.BytesIO()
                th.save(sd, buf)
                raw = buf.getvalue()
            elif item == "policy.optimizer.pth":
                osd = th.load(io.BytesIO(raw), map_location="cpu", weights_only=False)
                g = osd["param_groups"][0]
                keys = [k for k in g.get("params", []) if k in osd["state"]] or sorted(osd["state"].keys())
                names = oppo.param_names(False)
                assert len(keys) == len(names)
                for k, n in zip(keys, names):
                    for m in ("exp_avg", "exp_avg_sq"):
                        osd["state"][k][m] = _cut(osd["state"][k][m], n, REF_TRUNKS)
                moments = [(osd["state"][k]["exp_avg"], osd["state"][k]["exp_avg_sq"]) for k in keys]
                buf = io.BytesIO()
                th.save(osd, buf)
                raw = buf.getvalue()
            zout.writestr(item, raw)
    model = PPOLagrangian.load(path)
    pol = model.policy
    assert pol.trunk_hidden == REF_TRUNKS
    P = OrderedDict((n, t.float()) for n, t in sd.items())
    got = named(pol, pol._params)
    assert list(got) == list(P) and all(th.equal(got[n], P[n]) for n in P)
    m, v = named(pol, pol._adam_m), named(pol, pol._adam_v)
    for n, (em, ev) in zip(P, moments):
        assert th.equal(m[n], em.float()) and th.equal(v[n], ev.float()), n
    rng = np.random.default_rng(11)
    obs = (rng.standard_normal((1000, 18)) * 1.5).astype(np.float32)
    acts = rng.standard_normal((1000, 6)).astype(np.float32)
    ev_, ecv, lp, ent = (x.cpu().numpy() for x in pol.evaluate_actions(th.tensor(obs).cuda(), th.tensor(acts).cuda()))
    P64 = {k: t.double() for k, t in P.items()}
    with th.no_grad():
        wv, wcv, wlp, went = oppo.evaluate_actions(P64, th.tensor(obs, dtype=th.float64),
                                                   th.tensor(acts, dtype=th.float64), False)
    for got, want in ((ev_, wv), (ecv, wcv), (lp, wlp), (ent, went)):
        np.testing.assert_allclose(got.ravel(), want.numpy().ravel(), rtol=1e-5, atol=1e-6)


# ------------------------------------------------------------------------------------------------ drivers
def _run(args, env):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "run_me.py")] + args, cwd=ROOT, env=env, capture_output=True,
                       text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    return r.stdout


def _zip_arch(path):
    with zipfile.ZipFile(path) as zf:
        net_arch = json.loads(zf.read("data"))["policy_kwargs"]["net_arch"]
        sd = th.load(io.BytesIO(zf.read("policy.pth")), map_location="cpu", weights_only=False)
    shapes = tuple((sd[f"mlp_extractor.{t}.0.weight"].shape[0], sd[f"mlp_extractor.{t}.2.weight"].shape[0])
                   for t in oppo.TRUNKS)
    return net_arch, shapes


def test_run_me_cpg_and_icrl_with_per_trunk_widths(tmp_path):
    """`cpg -pl 64 64 -rl 32 32 -cl 16 48`, then `icrl -rvl 32 32 -cvl 48 16` on the synthetic environment at the scaled-down
    sizes of tests/test_drivers_gpu.py::test_run_me_cpg_run_policy_icrl; the saved zips hold those shapes and reload."""
    from icrl_b200.ppo_lag import PPOLagrangian
    env = dict(os.environ, ICRL_SAVE_ROOT=str(tmp_path / "runs"))
    common = ["-tei", "SynthHCWithPos-v0", "-eei", "SynthHCWithPosTest-v0", "-ns", "256", "-nt", "4", "-s", "1"]
    _run(["cpg"] + common + ["-t", "4096", "-ee", "256", "-se", "512", "-tk", "0.01", "-pl", "64", "64", "-rl", "32", "32",
                             "-cl", "16", "48"], env)
    run_dir = os.path.dirname(glob.glob(str(tmp_path / "runs" / "*" / "files"))[0])
    best = os.path.join(run_dir, "files", "best_model.zip")
    net_arch, shapes = _zip_arch(best)
    assert net_arch == [dict(pi=[64, 64], vf=[32, 32], cvf=[16, 48])] and shapes == ((64, 64), (32, 32), (16, 48))
    assert PPOLagrangian.load(best).policy.trunk_hidden == ((64, 64), (32, 32), (16, 48))
    _run(["run_policy", "-l", run_dir, "-s", "EXPERT", "-nr", "3"], env)
    _run(["icrl"] + common + ["-ep", run_dir, "-er", "3", "-ft", "2048", "-ni", "2", "-bi", "3", "-cl", "20", "-clr",
                              "0.05", "-crc", "0.5", "-aclr", "0.9", "-psis", "-ctkno", "2.5", "-tk", "0.01",
                              "-rvl", "32", "32", "-cvl", "48", "16"], env)
    icrl_dir = [d for d in glob.glob(str(tmp_path / "runs" / "*" / "files")) if os.path.dirname(d) != run_dir][0]
    rows = [json.loads(line) for line in open(os.path.join(icrl_dir, "metrics.jsonl"))]
    assert len(rows) == 2 and all(np.isfinite(r["forward/policy_gradient_loss"]) for r in rows)
    nominal = os.path.join(icrl_dir, "models", "icrl_1_itrs", "nominal_agent.zip")
    net_arch, shapes = _zip_arch(nominal)
    assert net_arch == [dict(pi=[64, 64], vf=[32, 32], cvf=[48, 16])] and shapes == ((64, 64), (32, 32), (48, 16))
    assert PPOLagrangian.load(nominal).policy.trunk_hidden == ((64, 64), (32, 32), (48, 16))


# ------------------------------------------------------------------------------------------------ data parallel
@pytest.mark.parametrize("wide", [False, True])
def test_data_parallel_embedding_is_bit_exact(wide):
    """2 ranks: the mixed net and its 64-64 embedding through the in-kernel all-reduce give the same bits."""
    if th.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
           "127.0.0.1", "--master-port", "29573", os.path.join(ROOT, "tests", "k4_trunks_dp_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, ICRL_DP_TRUNKS_WIDE="1" if wide else "0"))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert "dp trunks ok" in r.stdout
