"""K5 (whole-rollout cost normalisation, SURVEY §8 f1) against the oracle restatement of VecNormalizeWithCost's online
arithmetic -- bit-exact, float64 statistics included -- and the whole-buffer relabel mode of collect_rollouts against
the reference's per-step mode."""
import os
import sys

import numpy as np
import pytest
import torch as th

from conftest import load_golden
from icrl_b200 import _lib

pytestmark = pytest.mark.gpu
sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))


def _run_k5(orig, news, state, gamma=0.99, eps=1e-8, clip=10.0, norm=True, training=True):
    T, E = orig.shape
    dones = np.zeros((T, E), np.float32)
    dones[1:] = news[:-1]
    d = "cuda"
    st = th.from_numpy(np.concatenate([[state["mean"], state["var"], state["count"]], state["cost_ret"]])).to(d)
    o, dn = th.from_numpy(orig.astype(np.float32)).to(d), th.from_numpy(dones).to(d)
    last = th.from_numpy(news[-1].astype(np.uint8)).to(d)
    out = th.empty(T, E, device=d)
    _lib.check(_lib.lib().icrl_cost_normalize(_lib.ptr(o), _lib.ptr(dn), _lib.ptr(last), T, E, gamma, eps, clip, int(norm),
                                              int(training), _lib.ptr(st), _lib.ptr(out), _lib.current_stream()))
    st = st.cpu().numpy()
    return out.cpu().numpy(), dict(mean=st[0], var=st[1], count=st[2], cost_ret=st[3:])


@pytest.mark.parametrize("name,norm", [("all", True), ("nocost", False)])
def test_matches_reference_wrapper_fixture(name, norm):
    from oracle import costnorm
    g = load_golden(f"venv_{name}")
    E = g["orig_cost"].shape[1]
    out, st = _run_k5(g["orig_cost"], g["done"], costnorm.reset(costnorm.initial_state(E)), gamma=0.97, norm=norm)
    np.testing.assert_array_equal(out, g["cost"].astype(np.float32))
    assert st["mean"] == g["cost_rms_mean"] and st["var"] == g["cost_rms_var"] and st["count"] == float(g["cost_rms_count"])


def _data(kind, T, E, rng):
    """(orig_costs, news, starting state, clip_cost) of one test case."""
    from oracle import costnorm
    if kind == "signed":
        orig = rng.standard_normal((T, E)).astype(np.float32)
        orig[rng.random((T, E)) < 0.2] = 0.0
    elif kind == "clip":
        orig = (0.01 * rng.standard_normal((T, E))).astype(np.float32)
    else:
        orig = rng.uniform(0, 1, (T, E)).astype(np.float32) ** 3
    news = rng.random((T, E)) < 0.05
    if kind == "clip":          # after a long run of near-constant costs: sqrt(var + eps) ~ 1e-4, so costs reach the clip
        return orig, news, dict(mean=np.float64(0.0), var=np.float64(1e-12), count=np.float64(5e8),
                                cost_ret=np.zeros(E)), 0.5
    if kind == "bigcount":      # as after a long run or a loaded VecNormalize
        return orig, news, dict(mean=np.float64(0.31), var=np.float64(0.07), count=np.float64(1234567890.25),
                                cost_ret=rng.uniform(0, 2, E)), 10.0
    s0 = costnorm.reset(costnorm.initial_state(E))
    # a used state: two earlier rollouts' worth of statistics
    costnorm.normalize_rollout(rng.uniform(0, 1, (11, E)).astype(np.float32), rng.random((11, E)) < 0.1, s0)
    return orig, news, s0, 10.0


def _check_vs_oracle(orig, news, s0, clip=10.0, norm=True, training=True):
    from oracle import costnorm
    s_ref = {k: np.copy(v) for k, v in s0.items()}
    ref = costnorm.normalize_rollout(orig, news, s_ref, clip_cost=clip, norm_cost=norm, training=training)
    out, st = _run_k5(orig, news, s0, clip=clip, norm=norm, training=training)
    np.testing.assert_array_equal(out, ref)
    for k in ("mean", "var", "count"):
        assert st[k] == s_ref[k], (k, st[k], s_ref[k])
    np.testing.assert_array_equal(st["cost_ret"], s_ref["cost_ret"])
    return ref


# training with E <= 64 runs the fused single-CTA kernel in tiles of TT steps (TT = 110 at E = 64: T = 2048 is 19 tiles,
# the last one ragged); E > 64, or no training, runs cost_ret / cost_rms / cost_apply, whose cost_rms_kernel strides its
# 1024 threads over T.  Data: "cube" costs in [0, 1) from a used state, "signed" costs with negatives and zeros,
# "clip" costs that hit +-clip_cost, "bigcount" a state with count ~ 1e9.
K5_CASES = [(1, 1, "cube"), (7, 3, "cube"), (64, 5, "cube"), (2048, 5, "cube"), (33, 8, "cube"), (50, 13, "cube"),
            (40, 40, "cube"), (20, 128, "cube"), (9, 130, "cube"), (5, 300, "cube"), (3, 1000, "cube"),
            (300, 1, "signed"), (97, 7, "clip"), (12, 8, "bigcount"), (2048, 64, "cube"), (2048, 64, "signed"),
            (111, 64, "clip"), (111, 65, "bigcount"), (1025, 65, "cube"), (64, 127, "clip"), (40, 128, "bigcount"),
            (2048, 129, "signed"), (1025, 257, "clip"), (30, 1000, "bigcount")]


@pytest.mark.parametrize("T,E,data", K5_CASES)
@pytest.mark.parametrize("training", [True, False])
@pytest.mark.parametrize("norm", [True, False])
def test_bit_exact_vs_oracle(T, E, data, training, norm):
    rng = np.random.default_rng(T * 1000 + E)
    orig, news, s0, clip = _data(data, T, E, rng)
    ref = _check_vs_oracle(orig, news, s0, clip, norm, training)
    if data == "clip" and norm:
        assert (ref == clip).any() and (ref == -clip).any()


def test_fused_division_fallback_at_all_ones_significand():
    """The fused kernel divides by tot = count + E with Markstein's shortcut from a precomputed reciprocal, except where
    tot's significand is all ones.  count = 1 - 2^-52 with E = 1 makes the first tot 2 - 2^-52: the first block of
    four steps mixes the generic division (step 0) with the shortcut (steps 1-3)."""
    T, E = 300, 1
    count = 1.0 - 2.0 ** -52
    tots, c = [], count
    for _ in range(4):
        tots.append(c + E)
        c = E + c
    all_ones = [(int(np.float64(x).view(np.int64)) & (2 ** 52 - 1)) == 2 ** 52 - 1 for x in tots]
    assert all_ones == [True, False, False, False], [x.hex() for x in tots]
    rng = np.random.default_rng(7)
    orig = rng.uniform(0, 1, (T, E)).astype(np.float32)
    news = rng.random((T, E)) < 0.05
    s0 = dict(mean=np.float64(0.2), var=np.float64(0.5), count=np.float64(count), cost_ret=np.full(E, 0.3))
    _check_vs_oracle(orig, news, s0)


@pytest.mark.parametrize("E", [491529, 524288])
def test_largest_env_counts_vs_oracle(E):
    """numpy's pairwise sum splits n = 16k + r into 8k and 8k + r, so the batch moments of E >= 491 529 environments
    recurse 13 levels deep; 524 288 is the largest E icrl_cost_normalize accepts."""
    rng = np.random.default_rng(E)
    orig, news, s0, _ = _data("cube", 3, E, rng)
    _check_vs_oracle(orig, news, s0)


def _collect(whole_buffer):
    from scripted_env import ScriptedEnv
    from icrl_b200 import vec_env
    from icrl_b200.constraint_net import ConstraintNet
    from icrl_b200.ppo_lag import PPOLagrangian
    th.manual_seed(0)
    np.random.seed(0)
    rng = np.random.default_rng(0)
    cn = ConstraintNet(5, 2, (20,), None, lambda _: 1e-3, rng.standard_normal((50, 5)), rng.standard_normal((50, 2)),
                       False, 0.5, clip_obs=20, action_low=-np.ones(2, np.float32), action_high=np.ones(2, np.float32))
    env = vec_env.DummyVecEnv([(lambda i=i: ScriptedEnv(100 + i)) for i in range(4)])
    env = vec_env.VecCostWrapper(env)
    env = vec_env.VecNormalizeWithCost(env, training=True, cost_info_str="cost", reward_gamma=0.99, cost_gamma=0.99)
    env.set_cost_function(None if whole_buffer else cn.cost_function)
    model = PPOLagrangian("TwoCriticsMlpPolicy", env, n_steps=96, batch_size=64, n_epochs=1, seed=4)
    for _ in range(2):   # two rollouts: the statistics carry over
        model.learn(total_timesteps=96 * 4, cost_function=cn if whole_buffer else "cost", reset_num_timesteps=False)
    b = model.rollout_buffer
    return {k: b.time_major(k).copy() for k in ("costs", "orig_costs", "cost_advantages", "actions")}, env


def test_whole_buffer_relabel_equals_per_step_mode():
    a, env_a = _collect(False)
    b, env_b = _collect(True)
    np.testing.assert_array_equal(a["actions"], b["actions"])
    np.testing.assert_array_equal(a["orig_costs"], b["orig_costs"])
    np.testing.assert_array_equal(a["costs"], b["costs"])
    np.testing.assert_array_equal(a["cost_advantages"], b["cost_advantages"])
    assert env_a.cost_rms.var == env_b.cost_rms.var and env_a.cost_rms.mean == env_b.cost_rms.mean
    assert env_a.cost_rms.count == env_b.cost_rms.count
    np.testing.assert_array_equal(env_a.cost_ret, env_b.cost_ret)
