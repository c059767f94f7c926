"""GPU parity: K4 (PPO-Lagrangian update + dual step) through PPOLagrangian.train() against goldens produced by the
unmodified reference's PPOLagrangian.train() on identical buffers, parameters and numpy seed."""
import glob
import os

import numpy as np
import pytest
import torch as th

from conftest import GOLDEN, load_golden
from helpers import PARAM_RTOL, FakeVecEnv, max_param_err

pytestmark = pytest.mark.gpu
K4_CASES = sorted(os.path.basename(p)[3:-4] for p in glob.glob(os.path.join(GOLDEN, "k4_*.npz")))


def build_algo(d):
    from icrl_b200.ppo_lag import PPOLagrangian
    hp = {k[3:]: float(v) for k, v in d.items() if k.startswith("hp.")}
    names = [str(n) for n in d["param_order"]]
    discrete = "log_std" not in names
    T, E = int(hp["T"]), int(hp["E"])
    obs_dim = d["buf.observations"].shape[-1]
    act_dim = d["p0.action_net.weight"].shape[0]
    opt = lambda k: None if hp[k] < 0 else hp[k]
    algo = PPOLagrangian("TwoCriticsMlpPolicy", FakeVecEnv(obs_dim, act_dim, discrete, E), n_steps=T,
                         batch_size=None if hp["batch_size"] < 0 else int(hp["batch_size"]), n_epochs=int(hp["n_epochs"]),
                         learning_rate=hp["learning_rate"], clip_range=hp["clip_range"], target_kl=opt("target_kl"),
                         ent_coef=hp["ent_coef"], penalty_initial_value=hp["penalty_initial_value"],
                         penalty_learning_rate=hp["penalty_learning_rate"], clip_range_reward_vf=opt("clip_range_reward_vf"),
                         clip_range_cost_vf=opt("clip_range_cost_vf"), seed=3, device="cuda")
    assert algo.policy.parameter_names() == names
    algo.policy.load_state_dict({n: th.tensor(d["p0." + n]) for n in names})
    buf = algo.rollout_buffer
    for k in ("observations", "actions", "log_probs", "reward_values", "reward_advantages", "reward_returns",
              "cost_values", "cost_advantages", "cost_returns", "orig_costs"):
        getattr(buf, k)[:] = d["buf." + k].reshape(getattr(buf, k).shape)
    buf.full, buf.pos = True, T
    return algo, hp, names


def params_of(algo, names):
    sd = algo.policy.state_dict()
    return [sd[n].numpy() for n in names]


@pytest.mark.parametrize("case", K4_CASES)
def test_train_matches_reference(case):
    from icrl_b200 import logger
    d = load_golden(f"k4_{case}")
    algo, hp, names = build_algo(d)
    assert np.allclose(algo.dual.nu.log_nu.cpu().numpy(), d["log_nu0"], rtol=1e-6)
    logger.configure()
    np.random.seed(int(hp["numpy_seed"]))
    algo.train()
    err = max_param_err(params_of(algo, names), [d["p1." + n] for n in names])
    assert err <= PARAM_RTOL, f"params after train(): {err}"
    log = {k[4:]: float(v) for k, v in d.items() if k.startswith("log.")}
    got = logger.Logger.CURRENT.name_to_value
    assert int(got["train/early_stop_epoch"]) == int(log["train/early_stop_epoch"])
    for k in ("train/entropy_loss", "train/policy_gradient_loss", "train/reward_value_loss", "train/cost_value_loss",
              "train/clip_fraction", "train/loss", "train/approx_kl", "train/nu", "train/nu_loss", "train/average_cost",
              "train/std", "train/n_updates"):
        if k in log:
            assert abs(float(got[k]) - log[k]) <= 2e-4 * max(abs(log[k]), 1e-2), (k, float(got[k]), log[k])
    assert np.allclose(algo.dual.nu.log_nu.cpu().numpy(), d["log_nu1"], rtol=1e-5)
    # second train() on the same buffer: Adam moments, step count, nu and the numpy RNG stream carry over
    algo.train()
    err = max_param_err(params_of(algo, names), [d["p2." + n] for n in names])
    assert err <= 3 * PARAM_RTOL, f"params after second train(): {err}"
    assert np.allclose(algo.dual.nu.log_nu.cpu().numpy(), d["log_nu2"], rtol=1e-5)


K4X_CASES = sorted(os.path.basename(p)[4:-4] for p in glob.glob(os.path.join(GOLDEN, "k4x_*.npz")))
# parameters vs the reference after every train() of the round-2 fixtures.  hc_full is the drift test: 1 600 DEPENDENT
# optimiser steps (a whole HalfCheetah rollout: 2048 x 5, batch 64, 10 epochs) with 3xTF32 products, sqrt.approx and a fast
# division in Adam; the bound is what a chain of that length allows, the measured figure is in DESIGN.md section 2.
K4X_TOL = {"hc_full": 2e-3}


@pytest.mark.parametrize("case", K4X_CASES)
def test_full_size_and_large_batch_match_reference(case):
    """Round-2 fixtures: the full-size launch and the large-batch regime (batch >= 2048 selects the many-cluster kernel;
    ragged last minibatch, discrete actions, value clipping, full batch, KL early stop across launches)."""
    from icrl_b200 import logger
    from helpers import load_k4x
    d = load_k4x(case)
    algo, hp, names = build_algo(d)
    logger.configure()
    np.random.seed(int(hp["numpy_seed"]))
    tol = K4X_TOL.get(case, PARAM_RTOL)
    for call in range(1, int(hp["trains"]) + 1):
        algo.train()
        err = max_param_err(params_of(algo, names), [d[f"p{call}." + n] for n in names])
        print(f"k4x {case}: train() #{call}: {algo.policy.optimizer.step_count} optimiser steps, max param err {err:.3e}")
        assert err <= tol * (1 if call == 1 else 3), f"params after train() #{call}: {err}"
        assert np.allclose(algo.dual.nu.log_nu.cpu().numpy(), d[f"log_nu{call}"], rtol=1e-5)
        if call == 1:
            log = {k[4:]: float(v) for k, v in d.items() if k.startswith("log.")}
            got = logger.Logger.CURRENT.name_to_value
            assert int(got["train/early_stop_epoch"]) == int(log["train/early_stop_epoch"])
            for k in ("train/entropy_loss", "train/policy_gradient_loss", "train/reward_value_loss", "train/cost_value_loss",
                      "train/clip_fraction", "train/loss", "train/approx_kl"):
                assert abs(float(got[k]) - log[k]) <= 5e-4 * max(abs(log[k]), 1e-2), (k, float(got[k]), log[k])


@pytest.mark.parametrize("case,clusters", [("hc", 5), ("ant", 6), ("lgw", 5), ("hc_klstop", 8), ("hc_vfclip", 7), ("point", 24),
                                           ("hc_fullbatch", 3)])
def test_wide_kernel_on_small_fixtures(case, clusters, monkeypatch):
    """The many-cluster kernel forced onto the small fixtures (ICRL_PPO_WIDE=1): most clusters get no rows at all, so the
    zero-row paths of every exchange, the per-epoch launches and the device-side KL stop across launches are exercised
    against the same reference outputs."""
    from icrl_b200 import logger
    monkeypatch.setenv("ICRL_PPO_WIDE", "1")
    monkeypatch.setenv("ICRL_PPO_WIDE_CLUSTERS", str(clusters))
    d = load_golden(f"k4_{case}")
    algo, hp, names = build_algo(d)
    logger.configure()
    np.random.seed(int(hp["numpy_seed"]))
    algo.train()
    err = max_param_err(params_of(algo, names), [d["p1." + n] for n in names])
    assert err <= PARAM_RTOL, f"params after train(): {err}"
    log = {k[4:]: float(v) for k, v in d.items() if k.startswith("log.")}
    got = logger.Logger.CURRENT.name_to_value
    assert int(got["train/early_stop_epoch"]) == int(log["train/early_stop_epoch"])
    for k in ("train/policy_gradient_loss", "train/reward_value_loss", "train/cost_value_loss", "train/approx_kl", "train/loss"):
        assert abs(float(got[k]) - log[k]) <= 2e-4 * max(abs(log[k]), 1e-2), (k, float(got[k]), log[k])
    algo.train()
    err = max_param_err(params_of(algo, names), [d["p2." + n] for n in names])
    assert err <= 3 * PARAM_RTOL, f"params after second train(): {err}"


def test_one_update_and_adam_state():
    """The north-star gate: parameters after ONE optimiser step <= 1e-4, plus the Adam moments themselves."""
    d = load_golden("k4_hc_fullbatch")
    algo, hp, names = build_algo(d)
    np.random.seed(int(hp["numpy_seed"]))
    algo.train()
    assert algo.policy.optimizer.step_count == 1
    assert max_param_err(params_of(algo, names), [d["p1." + n] for n in names]) <= PARAM_RTOL
    st = algo.policy.optimizer.state_dict()["state"]
    m = [st[i]["exp_avg"].numpy() for i in range(len(names))]
    v = [st[i]["exp_avg_sq"].numpy() for i in range(len(names))]
    assert max_param_err(m, [d[f"adam.{i}.exp_avg"] for i in range(len(names))]) <= 1e-4
    assert max_param_err(v, [d[f"adam.{i}.exp_avg_sq"] for i in range(len(names))]) <= 2e-4


def test_first_minibatch_known_answers():
    """SURVEY §4: with log_probs produced by the current policy, the first minibatch has ratio == 1, clip_fraction == 0,
    approx_kl == 0."""
    d = load_golden("k4_hc")
    algo, hp, names = build_algo(d)
    buf = algo.rollout_buffer
    T, E = buf.buffer_size, buf.n_envs
    obs = th.tensor(buf.observations.reshape(T * E, -1))
    acts = th.tensor(buf.actions.reshape(T * E, -1))
    _, _, lp, _ = algo.policy.evaluate_actions(obs, acts)
    buf.log_probs[:] = lp.cpu().numpy().reshape(T, E)
    np.random.seed(0)
    algo.train()
    st = algo.last_train_stats
    assert st[0, 1] == 0.0 and abs(st[0, 5]) < 1e-6


def test_policy_forward_vs_oracle():
    from oracle import ppo as oppo
    from helpers import policy_params
    for case in ("hc", "ant", "lgw"):
        d = load_golden(f"k4_{case}")
        algo, hp, names = build_algo(d)
        P = policy_params(d, "p0.")
        obs = th.tensor(d["buf.observations"].reshape(-1, d["buf.observations"].shape[-1]))
        head, v, cv = algo.policy.forward_heads(obs)
        wh, wv, wcv = oppo.policy_forward_mean(P, obs, algo.policy.is_discrete)
        np.testing.assert_allclose(head.cpu().numpy(), wh.numpy(), rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(v.cpu().numpy(), wv.numpy().ravel(), rtol=1e-5, atol=1e-6)
        np.testing.assert_allclose(cv.cpu().numpy(), wcv.numpy().ravel(), rtol=1e-5, atol=1e-6)


def test_rollout_time_forward_zero_copy_path_equals_staged_path():
    """ActorTwoCriticsPolicy.forward on a handful of host rows (the per-environment-step call of collect_rollouts) reads them
    from, and writes heads / values to, a host-mapped pinned block with cached log_std terms; a CUDA input takes the staged
    path with blocking downloads.  Same torch seed -> identical actions, values and log-probs (also after a parameter change)."""
    for case in ("hc", "lgw"):
        d = load_golden(f"k4_{case}")
        algo, hp, names = build_algo(d)
        pol = algo.policy
        obs = th.tensor(d["buf.observations"].reshape(-1, d["buf.observations"].shape[-1])[:5].copy())
        for rep in range(2):
            th.manual_seed(11 + rep)
            small = pol.forward(obs)
            th.manual_seed(11 + rep)
            staged = pol.forward(obs.cuda())
            for a, b in zip(small, staged):
                assert a.device.type == "cpu" and b.device.type == "cpu"
                assert th.equal(a, b), case
            det = pol.forward(obs, deterministic=True)
            assert th.equal(det[0], pol.forward(obs.cuda(), deterministic=True)[0])
            if not pol.is_discrete:           # move log_std: the cached terms must follow
                pol._params[:pol.act_out] += 0.25
