"""Shared helpers for the parity tests: rebuild oracle-side objects from golden fixtures."""
import numpy as np
import torch as th

from oracle import cn as ocn
from oracle import ppo as oppo

SHAPES = {
    "lgw": dict(obs_dim=1, acs_dim=2, is_discrete=True, hidden=(20,)),
    "hc": dict(obs_dim=18, acs_dim=6, is_discrete=False, hidden=(20,)),
    "ant": dict(obs_dim=113, acs_dim=8, is_discrete=False, hidden=(40, 40)),
    "point": dict(obs_dim=6, acs_dim=2, is_discrete=False, hidden=(40, 40)),
}

# tolerances (BASELINE.json north_star): costs / advantages rel <= 1e-5, params after one update <= 1e-4.
# `1 - sigmoid` in the reference is itself only resolved to 1 ulp(1.0) = 6e-8 absolute, hence the atol.
COST_RTOL, COST_ATOL = 1e-5, 2e-7
PARAM_RTOL = 1e-4


def cn_params(d, prefix="p."):
    """[W0, b0, W1, b1, ...] float32 tensors from a golden dict holding `<prefix>{0,2,4}.{weight,bias}`."""
    out, i = [], 0
    while f"{prefix}{i}.weight" in d:
        out += [th.tensor(d[f"{prefix}{i}.weight"]), th.tensor(d[f"{prefix}{i}.bias"])]
        i += 2
    return out


def cn_spec(shape, d, **kw):
    s = SHAPES[shape]
    low = high = None
    if not s["is_discrete"]:
        low, high = -np.ones(s["acs_dim"], np.float32), np.ones(s["acs_dim"], np.float32)
    base = dict(obs_dim=s["obs_dim"], acs_dim=s["acs_dim"], hidden_sizes=s["hidden"], is_discrete=s["is_discrete"],
                clip_obs=20., obs_mean=d.get("obs_mean"), obs_var=d.get("obs_var"), action_low=low, action_high=high)
    base.update(kw)
    return ocn.CNSpec(**base)


def policy_params(d, prefix="p0."):
    names = [str(n) for n in d["param_order"]]
    from collections import OrderedDict
    return OrderedDict((n, th.tensor(d[prefix + n])) for n in names)


def rel_err(a, b, floor=0.0):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.max(np.abs(a - b) / np.maximum(np.abs(b), floor + 1e-300)))


def max_param_err(pa, pb):
    """max over tensors of ||a-b||_inf / max(||b||_inf, 1e-3)  (per-tensor scale, so zero-init biases don't divide by 0)."""
    worst = 0.0
    for a, b in zip(pa, pb):
        a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
        worst = max(worst, float(np.max(np.abs(a - b)) / max(float(np.max(np.abs(b))), 1e-3)))
    return worst


def cn_grad64(params, spec, nominal_obs, nominal_acs, episode_lengths, expert_obs, expert_acs, start_params=None):
    """The float64 gradient of the K2 loss (ocn.loss_terms, full batch) at `params`, as a list of float64 arrays in the
    order of `params`.  The inputs are prepared in float32 as the reference prepares them, then widened; with importance
    sampling the weights come from float64 predictions at `start_params` (default: `params`, i.e. iteration 0) and at
    `params`."""
    p64 = [th.as_tensor(np.asarray(p), dtype=th.float64).clone().requires_grad_(True) for p in params]
    xn = th.tensor(ocn.prepare_data(spec, nominal_obs, nominal_acs), dtype=th.float64)
    xe = th.tensor(ocn.prepare_data(spec, expert_obs, expert_acs), dtype=th.float64)
    if spec.importance_sampling:
        s64 = p64 if start_params is None else [th.as_tensor(np.asarray(p), dtype=th.float64) for p in start_params]
        with th.no_grad():
            old, new = ocn.forward(s64, xn), ocn.forward(p64, xn)
        w, _, _ = ocn.compute_is_weights(old, new, episode_lengths, spec.eps, spec.per_step_importance_sampling)
        w = w.to(th.float64)
    else:
        w = th.ones(xn.shape[0], dtype=th.float64)
    loss = ocn.loss_terms(spec, ocn.forward(p64, xn), ocn.forward(p64, xe), w[..., None])[0]
    return [g.numpy() for g in th.autograd.grad(loss, p64)]


def max_grad_err(got, want):
    """max over tensors of ||got-want||_inf / ||want||_inf (a tensor whose reference gradient is all zero must be zero)."""
    worst = 0.0
    for a, b in zip(got, want):
        a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
        worst = max(worst, float(np.max(np.abs(a - b)) / max(float(np.max(np.abs(b))), 1e-30)))
    return worst


class FakeVecEnv:
    """Just enough of a VecEnv to build a PPOLagrangian whose rollout buffer the test fills by hand."""

    def __init__(self, obs_dim, act_dim, discrete, n_envs):
        from icrl_b200.spaces import Box, Discrete
        self.observation_space = Box(-np.inf, np.inf, (obs_dim,), np.float32)
        self.action_space = Discrete(act_dim) if discrete else Box(-1, 1, (act_dim,), np.float32)
        self.num_envs = n_envs

    def reset(self):
        return np.zeros((self.num_envs,) + self.observation_space.shape, np.float32)

    def step(self, actions):
        n = self.num_envs
        return self.reset(), np.zeros(n, np.float32), np.zeros(n, bool), [{} for _ in range(n)]


def k4x_inputs(seed, T, E, obs_dim, acs_dim, is_discrete):
    """The seeded inputs of the round-2 K4 fixtures (tests/golden/make_golden.py::k4x_inputs, same generator calls in the
    same order): only torch-dependent arrays and outputs are stored in the .npz files."""
    rng = np.random.default_rng(seed)
    n = T * E
    scale = rng.uniform(0.5, 8.0, size=obs_dim)
    obs = np.clip((rng.standard_normal((n, obs_dim)) * scale).astype(np.float32) / 4.0, -10, 10).astype(np.float32)
    acs = (rng.integers(0, acs_dim, size=(n, 1)).astype(np.float32) if is_discrete
           else rng.standard_normal((n, acs_dim)).astype(np.float32))
    rewards = np.abs(rng.standard_normal((T, E))).astype(np.float32)
    costs = (np.abs(rng.standard_normal((T, E))) * 0.2).astype(np.float32)
    dones = (rng.random((T, E)) < 0.02).astype(np.float32)
    lp_noise = (0.05 * rng.standard_normal((T, E))).astype(np.float32)
    last_dones = rng.random(E) < 0.3
    return obs, acs, rewards, costs, dones, lp_noise, last_dones


def load_k4x(name):
    """A k4x_* fixture completed with its regenerated inputs, in the key layout of the k4_* fixtures."""
    import os
    from conftest import GOLDEN
    d = dict(np.load(os.path.join(GOLDEN, f"k4x_{name}.npz"), allow_pickle=False))
    s = SHAPES[name.split("_")[0]]
    T, E = int(d["hp.T"]), int(d["hp.E"])
    obs, acs, _, costs, _, _, _ = k4x_inputs(int(d["input_seed"]), T, E, s["obs_dim"], s["acs_dim"], s["is_discrete"])
    assert float(obs.astype(np.float64).sum()) == float(d["obs_sum"]) and \
        float(acs.astype(np.float64).sum()) == float(d["acs_sum"]), "numpy Generator stream changed: regenerate k4x fixtures"
    d["buf.observations"] = obs.reshape(T, E, -1)
    d["buf.actions"] = acs.reshape(T, E, -1)
    d["buf.orig_costs"] = costs
    return d
