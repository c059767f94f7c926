"""GPU: policies whose trunks share layers (MlpExtractor.shared_net, the reference's -sl): one shared obs -> s layer
under private layers (net_arch [s, dict(pi=[p], vf=[v], cvf=[c])]) or one trunk under all three heads ([s0, s1]),
through K4 training, the policy forward, checkpoints and the drivers.

Checks per case:
* trajectory against oracle.ppo.train, chain-free gradient against float64 and determinism, with the routines and
  tolerances of tests/test_k4_sweep_gpu.py and the oracle's trunk applying the shared layers (k4_shared_helpers.trunk);
  the launch count there tells which kernel ran;
* sum rule, oracle-free: one optimiser step at clip coefficient 1 against the separate-trunk net that holds three copies
  of the shared layers (the already verified kernel).  The shared tensors' first moment is the sum of the three copies',
  every private tensor's and head's first moment is bit-identical (same forward, same head gradients);
* policy forward and evaluate_actions against float64;
plus refusals, checkpoints, a state_dict of an independently built SB3-structured module, and the run_me.py drivers.
"""
import glob
import io
import json
import os
import re
import subprocess
import sys
import zipfile
from collections import OrderedDict
from dataclasses import replace

import numpy as np
import pytest
import torch as th

import k4_shared_helpers as sh
import test_k4_sweep_gpu as sweep
from helpers import FakeVecEnv
from oracle import ppo as oppo
from test_k4_sweep_gpu import NP_SEED, TRAJ_LR, Case, check_gradient, check_trajectory, time_major
from test_k4_trunks_gpu import build_algo as build_separate

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# Case.hidden holds the architecture: (shared widths, private widths of pi, vf, cvf), see k4_shared_helpers
CASES = {
    # ---- one shared layer, single cluster
    "hc_d18_sl64_c6": Case(18, ((64,), (64, 32, 16)), A=6, B=64),
    "ant_d113_sl64_c8_b128": Case(113, ((64,), (64, 64, 48)), A=8, B=128, seed=1),   # NT1 = 8, two chunks per step
    "d30_sl7_c12": Case(30, ((7,), (33, 48, 64)), A=12, T=50, B=100, ent=0.01),  # narrow shared layer, both head lanes
    "vfclip_d20_sl48_c5": Case(20, ((48,), (24, 40, 64)), A=5, cvf_r=0.2, cvf_c=0.3),
    # oracle epoch-0 / epoch-1 mean approx_kl -1.1e-3 / 5.95e-3, 1.5 x target_kl = 3e-3: stops after epoch 1
    "tkl_d113_sl64_c8": Case(113, ((64,), (64, 64, 64)), A=8, T=64, B=128, epochs=3, target_kl=2e-3, seed=2),
    # ---- one trunk under all three heads
    "hc_d18_sl64x64_c6": Case(18, ((64, 64), ()), A=6, B=64),
    "lgw_d1_sl20x20_d2": Case(1, ((20, 20), ()), A=2, disc=True, T=50, B=40, ent=0.02),   # entropy bonus
    # ---- many clusters: natural (batch_size >= 2048) and forced, the 128-row minibatch leaves two clusters without rows
    "wide_d18_sl64_b2048": Case(18, ((64,), (64, 32, 16)), A=6, T=1050, B=2048, many=True),
    "forced_d40_sl48x24_cl4": Case(40, ((48, 24), ()), A=6, T=160, B=256, wide=4, many=True, ent=0.01),
}


class _SharedOracle:
    """oracle.ppo as tests/test_k4_sweep_gpu.py sees it, with init_policy taking a shared architecture."""

    def __getattr__(self, name):
        return getattr(oppo, name)

    @staticmethod
    def init_policy(obs_dim, act_dim, is_discrete, arch, generator=None):
        return sh.init_policy(obs_dim, act_dim, is_discrete, arch, generator=generator)


def build_algo(c: Case, d, lr):
    """tests/test_k4_sweep_gpu.py::build_algo with a shared net_arch."""
    from icrl_b200.ppo_lag import PPOLagrangian
    algo = PPOLagrangian("TwoCriticsMlpPolicy", FakeVecEnv(c.D, c.A, c.disc, c.E), n_steps=c.T, batch_size=c.B,
                         n_epochs=c.epochs, learning_rate=lr, clip_range=c.clip, target_kl=c.target_kl, ent_coef=c.ent,
                         max_grad_norm=c.mgn, penalty_initial_value=c.nu, penalty_learning_rate=sweep.PENALTY_LR,
                         clip_range_reward_vf=c.cvf_r, clip_range_cost_vf=c.cvf_c,
                         policy_kwargs=dict(net_arch=sh.net_arch(c.hidden)), seed=3, device="cuda")
    pol = algo.policy
    assert pol.parameter_names() == sh.param_names(c.disc, c.hidden)
    assert pol.trunk_hidden == sh.trunk_hidden(c.hidden) and pol.n_shared == len(c.hidden[0])
    pol.load_state_dict({n: p.clone() for n, p in d["P"].items()})
    buf = algo.rollout_buffer
    for k, src in sweep.BUF_FIELDS.items():
        getattr(buf, k)[:] = time_major(c, d["flat"][src]).reshape(getattr(buf, k).shape)
    buf.orig_costs[:] = time_major(c, d["orig_costs"])
    buf.full, buf.pos = True, c.T
    return algo


@pytest.fixture
def shared(monkeypatch):
    """The sweep's routines on the shared architecture; the case's cluster regime in the environment."""
    monkeypatch.setattr(oppo, "_trunk", sh.trunk)
    monkeypatch.setattr(sweep, "oppo", _SharedOracle())
    monkeypatch.setattr(sweep, "names_of", lambda c: sh.param_names(c.disc, c.hidden))
    monkeypatch.setattr(sweep, "build_algo", build_algo)

    def setup(name):
        c = CASES[name]
        sweep._env(c, monkeypatch)
        return c
    return setup


def named(pol, flat):
    return OrderedDict((n, flat[off:off + int(np.prod(shape))].reshape(shape).cpu())
                       for n, (off, shape) in zip(pol.parameter_names(), pol._slices))


@pytest.mark.parametrize("name", list(CASES))
def test_trajectory_vs_oracle(name, shared):
    c = shared(name)
    outs = check_trajectory(c)          # includes which kernel ran (launch count)
    if c.target_kl is not None:
        assert outs[0]["early_stop_epoch"] == 1


@pytest.mark.parametrize("name", list(CASES))
def test_gradient_vs_float64(name, shared):
    check_gradient(shared(name))        # includes the pre-clip norm, the clip-edge guard and a bit-identical repeat


SUM_RTOL = 1e-6


def one_step_moments(algo):
    np.random.seed(NP_SEED)
    algo._max_steps = 1
    algo.train()
    assert algo.last_train_stats.shape[0] == 1
    return named(algo.policy, algo.policy._adam_m)


@pytest.mark.parametrize("name", list(CASES))
def test_sum_rule_against_separate_trunks(name, shared):
    """One optimiser step with clip coefficient 1: Adam's first moment is (1 - beta1) g.  The shared layers' gradient is
    the sum over the three trunks of what the separate-trunk net gives each copy (to SUM_RTOL of the largest entry of
    the three copies' summed magnitudes: the two sides add the same products in a different order), and every other
    tensor's moment is bit-identical, as its arithmetic is the same."""
    c = replace(shared(name), mgn=1e9)
    d = sweep.make_data(c)
    m_sh = one_step_moments(build_algo(c, d, TRAJ_LR))
    cs = replace(c, hidden=sh.trunk_hidden(c.hidden))
    m_sep = one_step_moments(build_separate(cs, dict(d, P=sh.separate(d["P"], c.disc, c.hidden)), TRAJ_LR))
    worst = 0.0
    for n, m in m_sh.items():
        if n.startswith("mlp_extractor.shared_net."):
            layer, kind = n.split(".")[2:]
            copies = [m_sep[f"mlp_extractor.{t}.{layer}.{kind}"].double() for t in oppo.TRUNKS]
            scale = float(sum(x.abs() for x in copies).max())
            err = float((m.double() - sum(copies)).abs().max())
            worst = max(worst, err / scale)
            assert err <= SUM_RTOL * scale, f"{n}: {err:.3e} > {SUM_RTOL} x {scale:.3e}"
        else:
            src = n.replace(".0.", ".2.") if n.startswith("mlp_extractor.") else n   # private layer = layer 2 of a trunk
            assert th.equal(m, m_sep[src]), f"{n} differs from {src} of the separate-trunk net"
    print(f"\n  sum rule: worst {worst:.2e} of the copies' summed magnitude", end="")


FWD_ROWS = (1, 64, 65, 100_003)


@pytest.mark.parametrize("name", list(CASES))
def test_policy_forward_vs_float64(name, shared):
    c = shared(name)
    d = sweep.make_data(c)
    pol = build_algo(c, d, TRAJ_LR).policy
    P64 = {k: v.double() for k, v in d["P"].items()}
    rng = np.random.default_rng(5)
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
            np.testing.assert_allclose(got, want.numpy(), rtol=1e-5, atol=1e-6, err_msg=f"{what}, {n} rows")


# ------------------------------------------------------------------------------------------------ refusals
@pytest.mark.parametrize("net_arch,what", [
    ([64, dict(pi=[64, 64], vf=[64, 64], cvf=[64, 64])], "the pi trunk"),     # -sl 64 with the default -pl 64 64
    ([64], "the pi trunk"),                                                    # depth 1
    ([64, dict(pi=[64], vf=[32], cvf=[16, 16])], "the cvf trunk"),            # mixed private depths
    ([64, 64, dict(pi=[], vf=[8], cvf=[])], "the vf trunk"),
    ([64, dict(pi=[64], vf=[65], cvf=[64])], "the vf trunk"),
    ([65, dict(pi=[64], vf=[64], cvf=[64])], "the shared layers [65]"),
    ([0, 64], "the shared layers [0, 64]"),
    ([64, 64, 64], "the shared layers [64, 64, 64]"),
])
def test_unsupported_shapes_are_refused_at_construction(net_arch, what):
    from icrl_b200.ppo_lag import PPOLagrangian
    with pytest.raises(NotImplementedError, match=re.escape(what)):
        PPOLagrangian("TwoCriticsMlpPolicy", FakeVecEnv(8, 4, False, 4), n_steps=8, batch_size=32,
                      policy_kwargs=dict(net_arch=net_arch), device="cuda")


def test_data_parallel_is_refused():
    c = CASES["hc_d18_sl64_c6"]
    algo = build_algo(c, _data(c), TRAJ_LR)
    with pytest.raises(NotImplementedError, match="data-parallel training of shared policy layers"):
        algo.enable_data_parallel(comm=object())
    assert algo.comm is None


def _data(c):
    with pytest.MonkeyPatch.context() as mp:
        mp.setattr(oppo, "_trunk", sh.trunk)
        mp.setattr(sweep, "oppo", _SharedOracle())
        return sweep.make_data(c)


def test_refused_train_leaves_the_state_alone():
    from icrl_b200 import _lib
    c = CASES["hc_d18_sl64_c6"]
    algo = build_algo(c, _data(c), TRAJ_LR)
    pol = algo.policy
    pol._adam_m.fill_(0.25)
    pol._adam_v.fill_(0.5)
    before = [t.clone() for t in (pol._params, pol._adam_m, pol._adam_v)]
    pol.trunk_hidden = ((64, 64), (32, 32), (64, 16))
    with pytest.raises(_lib.IcrlError, match=r"equal h0 in every trunk \(pi 64, vf 32, cvf 64\)"):
        algo.train()
    for a, b in zip(before, (pol._params, pol._adam_m, pol._adam_v)):
        assert th.equal(a, b)
    assert pol.optimizer.step_count == 0


# ------------------------------------------------------------------------------------------------ checkpoints
@pytest.mark.parametrize("name", ["hc_d18_sl64_c6", "lgw_d1_sl20x20_d2"])
def test_save_load_round_trip_keeps_shared_layers(name, shared, tmp_path):
    from icrl_b200.ppo_lag import PPOLagrangian
    c = shared(name)
    algo = build_algo(c, sweep.make_data(c), TRAJ_LR)
    np.random.seed(NP_SEED)
    algo.train()
    algo.dual.update_parameter(0.3)
    path = str(tmp_path / "shared")
    algo.save(path)
    again = PPOLagrangian.load(path)
    assert again.policy.trunk_hidden == algo.policy.trunk_hidden and again.policy.n_shared == len(c.hidden[0])
    assert again.policy.parameter_names() == sh.param_names(c.disc, c.hidden)
    assert th.equal(again.policy.parameters_flat(), algo.policy.parameters_flat())
    assert th.equal(again.policy._adam_m, algo.policy._adam_m) and th.equal(again.policy._adam_v, algo.policy._adam_v)
    assert th.equal(again.dual.nu.state, algo.dual.nu.state) and again.dual.steps == algo.dual.steps
    assert again.policy.optimizer.step_count == algo.policy.optimizer.step_count


@pytest.mark.parametrize("arch", [((64,), (64, 32, 16)), ((20, 20), ())])
def test_sb3_structured_state_dict_loads_and_evaluates(arch, shared):
    """A state_dict of k4_shared_helpers.SB3Policy (MlpExtractor's structure, built without icrl_b200) loads into the
    policy under the same names and evaluates like the float64 oracle on those tensors."""
    from icrl_b200.policies import ActorTwoCriticsPolicy
    from icrl_b200.spaces import Box
    D, A = 18, 6
    th.manual_seed(11)
    ref = sh.SB3Policy(D, A, False, sh.net_arch(arch))
    with th.no_grad():
        for p in ref.parameters():
            p.add_(0.1 * th.randn_like(p))      # non-zero biases and log_std, heads away from the 0.01 gain
    sd = ref.state_dict()
    pol = ActorTwoCriticsPolicy(Box(-np.inf, np.inf, (D,)), Box(-1, 1, (A,)), lambda _: 3e-4,
                                net_arch=sh.net_arch(arch), device="cuda")
    pol.load_state_dict(sd)
    assert pol.parameter_names() == list(sd)
    rng = np.random.default_rng(3)
    obs = (rng.standard_normal((1000, D)) * 1.5).astype(np.float32)
    acts = rng.standard_normal((1000, A)).astype(np.float32)
    got = [x.cpu().numpy().ravel() for x in pol.evaluate_actions(th.tensor(obs).cuda(), th.tensor(acts).cuda())]
    P64 = OrderedDict((n, t.double()) for n, t in sd.items())
    with th.no_grad():
        want = oppo.evaluate_actions(P64, th.tensor(obs, dtype=th.float64), th.tensor(acts, dtype=th.float64), False)
        # the oracle's trunk and the module's own layers agree
        o64 = th.tensor(obs, dtype=th.float64)
        ref64 = ref.double()
        latent = ref64.mlp_extractor.shared_net(o64)
        np.testing.assert_allclose(ref64.value_net(ref64.mlp_extractor.value_net(latent)).numpy(), want[0].numpy(),
                                   rtol=1e-12, atol=1e-12)
    for g, w in zip(got, want):
        np.testing.assert_allclose(g, w.numpy().ravel(), rtol=1e-5, atol=1e-6)


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
    return net_arch, OrderedDict((n, tuple(t.shape)) for n, t in sd.items() if n.startswith("mlp_extractor."))


def test_run_me_cpg_and_icrl_with_shared_layers(tmp_path):
    """`cpg -sl 64 64 -pl -rl -cl`, then `icrl -sl 64 -pl 64 -rvl 32 -cvl 16` on the synthetic environment at the
    scaled-down sizes of tests/test_drivers_gpu.py; the saved zips hold those shapes and reload."""
    from icrl_b200.ppo_lag import PPOLagrangian
    env = dict(os.environ, ICRL_SAVE_ROOT=str(tmp_path / "runs"))
    common = ["-tei", "SynthHCWithPos-v0", "-eei", "SynthHCWithPosTest-v0", "-ns", "256", "-nt", "4", "-s", "1"]
    _run(["cpg"] + common + ["-t", "4096", "-ee", "256", "-se", "512", "-tk", "0.01", "-sl", "64", "64", "-pl", "-rl",
                             "-cl"], env)
    run_dir = os.path.dirname(glob.glob(str(tmp_path / "runs" / "*" / "files"))[0])
    best = os.path.join(run_dir, "files", "best_model.zip")
    net_arch, shapes = _zip_arch(best)
    assert net_arch == [64, 64, dict(pi=[], vf=[], cvf=[])]
    assert list(shapes) == ["mlp_extractor.shared_net.0.weight", "mlp_extractor.shared_net.0.bias",
                            "mlp_extractor.shared_net.2.weight", "mlp_extractor.shared_net.2.bias"]
    assert shapes["mlp_extractor.shared_net.0.weight"][0] == 64 and shapes["mlp_extractor.shared_net.2.weight"] == (64, 64)
    pol = PPOLagrangian.load(best).policy
    assert pol.n_shared == 2 and pol.trunk_hidden == ((64, 64),) * 3
    _run(["run_policy", "-l", run_dir, "-s", "EXPERT", "-nr", "3"], env)
    _run(["icrl"] + common + ["-ep", run_dir, "-er", "3", "-ft", "2048", "-ni", "2", "-bi", "3", "-cl", "20", "-clr",
                              "0.05", "-crc", "0.5", "-aclr", "0.9", "-psis", "-ctkno", "2.5", "-tk", "0.01",
                              "-sl", "64", "-pl", "64", "-rvl", "32", "-cvl", "16"], env)
    icrl_dir = [d for d in glob.glob(str(tmp_path / "runs" / "*" / "files")) if os.path.dirname(d) != run_dir][0]
    rows = [json.loads(line) for line in open(os.path.join(icrl_dir, "metrics.jsonl"))]
    assert len(rows) == 2 and all(np.isfinite(r["forward/policy_gradient_loss"]) for r in rows)
    nominal = os.path.join(icrl_dir, "models", "icrl_1_itrs", "nominal_agent.zip")
    net_arch, shapes = _zip_arch(nominal)
    assert net_arch == [64, dict(pi=[64], vf=[32], cvf=[16])]
    assert [(n, s[0]) for n, s in shapes.items() if n.endswith(".weight")] == [
        ("mlp_extractor.shared_net.0.weight", 64), ("mlp_extractor.policy_net.0.weight", 64),
        ("mlp_extractor.value_net.0.weight", 32), ("mlp_extractor.cost_value_net.0.weight", 16)]
    pol = PPOLagrangian.load(nominal).policy
    assert pol.n_shared == 1 and pol.trunk_hidden == ((64, 64), (64, 32), (64, 16))
