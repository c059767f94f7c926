"""GPU: K4 (PPO-Lagrangian training, csrc/k4_ppo_lag.cu) swept over every obs-width instantiation (NT1 = 1, 2, 4, 8 and
both ends of each), hidden sizes below 64 and h0 != h1, 1-16 continuous or discrete actions (both sides of the 8-lane
head split), single-cluster batches from 20 to 2047 rows with ragged last minibatches, and the many-cluster kernel
(natural batches >= 2048 and forced cluster counts) -- on seeded synthetic rollouts.  Plus the dual step
(csrc/k4_dual.cu) and the policy forward (csrc/k4_policy_forward.cu) at the same shapes.

The data make every term count: action head at gain 1 (not the reference's 0.01), non-zero biases, per-dimension
log_std, old log-probs = the float64 log-prob at the start + N(0, 0.15) (ratios on both sides of both clip edges),
advantages of both signs, old values spread around the start's values so value clipping binds on about half the rows.

Checks per case:
* trajectory: parameters after each of two PPOLagrangian.train() calls against oracle.ppo.train (fp32) on the same
  env-major data and permutations, every column of last_train_stats per step, early_stop_epoch, the Adam step count, the
  numpy RNG position, log_nu after the dual step, and which kernel ran (icrl_launch_count: the many-cluster path launches
  gather, stats and train once per epoch, the single-cluster path once per train());
* chain-free gradient: Adam's first moment is m_{k+1} = beta1 m_k + (1 - beta1) g_k, so runs of k and k + 1 optimiser
  steps from the same start give the clipped gradient of step k, compared with the float64 gradient of
  oracle.ppo.minibatch_loss at the GPU's own parameters on that step's minibatch, clipped the torch way (stats column 7
  against the float64 pre-clip norm).  The gradient runs use a small learning rate so the rows kept away from the clip
  edges at the start stay away; a guard asserts it at every checked step;
* determinism: a repeat of the longest gradient run gives the same bits (parameters, both moments, stats).
"""
from dataclasses import dataclass
from typing import Optional, Tuple

import numpy as np
import pytest
import torch as th

from helpers import PARAM_RTOL, FakeVecEnv, max_grad_err, max_param_err
from oracle import cn as ocn
from oracle import ppo as oppo

pytestmark = pytest.mark.gpu

BETA1 = 0.9
NP_SEED = 1234            # global numpy seed before the first train(): the permutations of both sides come from it
TRAJ_LR = 3e-4
GRAD_LR = 2e-5            # the gradient runs' learning rate: ratios and value deltas move < 1e-3 over the checked steps
PENALTY_LR = 0.05
# tolerances, each with the worst value measured over this file's cases on a B200 (1000 W power limit)
TRAJ_TOL = (PARAM_RTOL, 3 * PARAM_RTOL)   # params after call 1 / call 2, per-tensor inf-norm relative: 2.7e-6 / 2.7e-6
METRIC_RTOL = 2e-4                        # stats columns, relative with a 1e-2 floor (as tests/test_k4_gpu.py): 6.7e-5
GRAD_TOL = 1e-4                           # recovered clipped gradient vs float64 (see grad_err): 5.6e-5
NORM_RTOL = 2e-5                          # stats column 7 vs the float64 pre-clip norm: 7.3e-6
EDGE = 1e-2               # data: no row's float64 ratio (value delta) at the start within this of a clip edge
GUARD = 1e-4              # asserted at every checked step, at the GPU's parameters


@dataclass(frozen=True)
class Case:
    D: int                              # obs_dim
    hidden: Tuple[int, int] = (64, 64)
    A: int = 6                          # action dims (continuous) or actions (discrete)
    disc: bool = False
    T: int = 64
    E: int = 4
    B: Optional[int] = 64               # batch_size; None: the whole buffer
    epochs: int = 2
    nu: float = 1.0                     # penalty_initial_value (nu = softplus(log_nu) starts there)
    clip: float = 0.2
    cvf_r: Optional[float] = None
    cvf_c: Optional[float] = None
    ent: float = 0.0
    mgn: float = 0.5
    target_kl: Optional[float] = None
    wide: int = 0                       # > 0: ICRL_PPO_WIDE=1 with this many clusters
    many: bool = False                  # the many-cluster kernel is expected to run
    seed: int = 0

    @property
    def N(self):
        return self.T * self.E


CASES = {
    # ---- single cluster.  NT1 = 1 (obs_dim 1..16)
    "d1_c1_b20": Case(1, A=1, T=25, B=20),                                      # 20 rows: one CTA of each pair has 0
    "d16_h7x33_c8_b100": Case(16, (7, 33), A=8, T=90, E=5, B=100, clip=0.05, ent=0.01),  # 450 = 4 x 100 + 50
    # NT1 = 2 (17..32)
    "d17_h48x16_c9_vfr": Case(17, (48, 16), A=9, B=64, nu=0.0, cvf_r=0.2),      # 9 actions: head lanes u = 1
    "d32_h33x64_d3_full": Case(32, (33, 64), A=3, disc=True, T=75, B=None, ent=0.02, cvf_c=0.3),  # 300 rows, 5 chunks
    # NT1 = 4 (33..64)
    "d33_h64x8_c16_b1000": Case(33, (64, 8), A=16, T=1001, E=2, B=1000, nu=21.0),  # 1000 x 2 + 2-row tail, 16 chunks
    "d64_h1x1_d1": Case(64, (1, 1), A=1, disc=True, T=32, B=64, clip=10.0),
    # NT1 = 8 (65..128)
    "d65_d9_mgn1e3": Case(65, A=9, disc=True, T=50, B=64, mgn=1e3, ent=0.01),  # 3 x 64 + 8; clip coefficient clamps to 1
    "d128_d16_b2047": Case(128, A=16, disc=True, T=2047, E=2, B=2047),        # the largest single-cluster batch
    # target_kl between the oracle's epoch-0 and epoch-1 mean approx_kl (-3.1e-3 and 1.33e-2): stops after epoch 1
    "d113_c8_tkl": Case(113, A=8, T=64, B=128, epochs=3, target_kl=3.3e-3, seed=2),
    # ---- many clusters, natural (batch_size >= 2048)
    "wide_d18_b2048": Case(18, A=6, T=1050, B=2048, many=True),             # 2048, 2048, 104
    "wide_d40_h48x24_c12": Case(40, (48, 24), A=12, T=1500, B=3000, cvf_r=0.2, cvf_c=0.3, many=True),
    "wide_d100_h32x64_d10": Case(100, (32, 64), A=10, disc=True, T=1250, B=2500, ent=0.01, many=True),
    # epoch-0 / epoch-1 mean approx_kl 8.6e-4 / 1.13e-2, 1.5 x target_kl = 3.2e-3: stops after epoch 1
    "wide_d18_tkl": Case(18, A=6, T=1050, B=2048, epochs=3, target_kl=2.1e-3, many=True, seed=1),
    # ---- many clusters, forced (ICRL_PPO_WIDE=1): most clusters get few or no rows
    "forced_d1_d2_cl3": Case(1, A=2, disc=True, T=150, B=300, wide=3, many=True),
    "forced_d1_c4_cl7": Case(1, (20, 20), A=4, T=100, B=150, wide=7, many=True, ent=0.01),
    "forced_d40_h20_c6_cl4": Case(40, (20, 20), A=6, T=160, B=256, wide=4, many=True),
    "forced_d64_c16_cl9": Case(64, A=16, T=130, B=512, wide=9, many=True, cvf_c=0.3),
    # NT1 = 8 needs 5 clusters to spread the reduction (2 x clusters x 6 >= 58 floats): 3 falls back to one cluster
    "forced_d128_cl3_fallback": Case(128, A=6, T=64, B=128, wide=3, many=False),
}


# ------------------------------------------------------------------------------------------------ data
def names_of(c: Case):
    return oppo.param_names(c.disc)


def make_data(c: Case):
    """Seeded rollout (time-major [T, E, ...] float32 arrays, as the buffer holds them) and starting parameters."""
    rng = np.random.default_rng(1000 + 7 * c.seed + c.D)
    P = oppo.init_policy(c.D, c.A, c.disc, c.hidden, generator=th.Generator().manual_seed(c.seed))
    P["action_net.weight"] = P["action_net.weight"] * 100.0          # orthogonal at gain 1 instead of 0.01
    for n in P:
        if n.endswith(".bias"):
            P[n] = th.tensor(rng.normal(0.0, 0.3, tuple(P[n].shape)), dtype=th.float32)
    if not c.disc:
        P["log_std"] = th.tensor(rng.uniform(-1.5, 0.5, c.A), dtype=th.float32)
    N = c.N
    scale = rng.uniform(0.3, 2.0, c.D)
    obs = (rng.standard_normal((N, c.D)) * scale).astype(np.float32)           # env-major rows
    P64 = {k: v.double() for k, v in P.items()}
    o64 = th.tensor(obs, dtype=th.float64)
    with th.no_grad():
        head, v, cv = oppo.policy_forward_mean(P64, o64, c.disc)
        head = head.numpy()
        if c.disc:
            p = np.exp(head - head.max(1, keepdims=True))
            p /= p.sum(1, keepdims=True)
            u = rng.random((N, 1))
            acts = np.minimum((p.cumsum(1) < u).sum(1, keepdims=True), c.A - 1).astype(np.float32)
        else:
            acts = (head + np.exp(P["log_std"].double().numpy()) * rng.standard_normal((N, c.A))).astype(np.float32)
        _, _, lp, _ = oppo.evaluate_actions(P64, o64, th.tensor(acts, dtype=th.float64), c.disc)
    lp, v, cv = lp.numpy(), v.numpy().ravel(), cv.numpy().ravel()

    def noise_away_from(base, sd, edges, ratio):
        """base + N(0, sd), redrawn on rows whose ratio (or delta) at the start lies within EDGE of an edge."""
        x = rng.normal(0.0, sd, N)
        for _ in range(100):
            val = np.exp(-x) if ratio else -x
            bad = np.zeros(N, bool)
            for e in edges:
                bad |= np.abs(val - e) < EDGE
            if not bad.any():
                return base + x
            x[bad] = rng.normal(0.0, sd, int(bad.sum()))
        raise AssertionError("could not place the rows away from the clip edges")
    old_lp = noise_away_from(lp, 0.15, (1 - c.clip, 1 + c.clip), True)          # ratio = exp(lp - old_lp)
    old_v = noise_away_from(v, 0.3, (-c.cvf_r, c.cvf_r) if c.cvf_r else (), False)  # delta = v - old_v
    old_cv = noise_away_from(cv, 0.3, (-c.cvf_c, c.cvf_c) if c.cvf_c else (), False)
    flat = {
        "observations": obs, "actions": acts, "old_log_prob": old_lp.astype(np.float32),
        "old_reward_values": old_v.astype(np.float32),
        "reward_advantages": (rng.standard_normal(N) * 1.5 + 0.3).astype(np.float32),
        "reward_returns": (old_v + rng.standard_normal(N)).astype(np.float32),
        "old_cost_values": old_cv.astype(np.float32),
        "cost_advantages": (rng.standard_normal(N) * 0.7 - 0.1).astype(np.float32),
        "cost_returns": (old_cv + 0.5 * rng.standard_normal(N)).astype(np.float32),
    }
    orig_costs = np.abs(rng.standard_normal(N) * 0.3).astype(np.float32)
    return dict(P=P, flat=flat, orig_costs=orig_costs)


def time_major(c: Case, x):
    """env-major [E*T, ...] (row = e*T + t, what the reference's get() reads) -> the buffer's [T, E, ...]."""
    return np.ascontiguousarray(x.reshape(c.E, c.T, *x.shape[1:]).swapaxes(0, 1))


BUF_FIELDS = {"observations": "observations", "actions": "actions", "log_probs": "old_log_prob",
              "reward_values": "old_reward_values", "reward_advantages": "reward_advantages",
              "reward_returns": "reward_returns", "cost_values": "old_cost_values",
              "cost_advantages": "cost_advantages", "cost_returns": "cost_returns"}


def build_algo(c: Case, d, lr):
    from icrl_b200.ppo_lag import PPOLagrangian
    h = list(c.hidden)
    algo = PPOLagrangian("TwoCriticsMlpPolicy", FakeVecEnv(c.D, c.A, c.disc, c.E), n_steps=c.T, batch_size=c.B,
                         n_epochs=c.epochs, learning_rate=lr, clip_range=c.clip, target_kl=c.target_kl, ent_coef=c.ent,
                         max_grad_norm=c.mgn, penalty_initial_value=c.nu, penalty_learning_rate=PENALTY_LR,
                         clip_range_reward_vf=c.cvf_r, clip_range_cost_vf=c.cvf_c,
                         policy_kwargs=dict(net_arch=[dict(pi=h, vf=h, cvf=h)]), seed=3, device="cuda")
    assert algo.policy.parameter_names() == names_of(c)
    algo.policy.load_state_dict({n: p.clone() for n, p in d["P"].items()})
    buf = algo.rollout_buffer
    for k, src in BUF_FIELDS.items():
        getattr(buf, k)[:] = time_major(c, d["flat"][src]).reshape(getattr(buf, k).shape)
    buf.orig_costs[:] = time_major(c, d["orig_costs"])
    buf.full, buf.pos = True, c.T
    return algo


def draw_perms(c: Case):
    """What PPOLagrangian._draw_permutations draws from the current global numpy state, with the state after each."""
    perms, states = [], []
    for _ in range(c.epochs):
        perms.append(np.random.permutation(c.N))
        states.append(np.random.get_state())
    return perms, states


def oracle_kwargs(c: Case, lr, nu):
    return dict(is_discrete=c.disc, batch_size=c.B, n_epochs=c.epochs, lr=lr, clip_range=c.clip, nu=nu,
                ent_coef=c.ent, max_grad_norm=c.mgn, target_kl=c.target_kl, clip_range_reward_vf=c.cvf_r,
                clip_range_cost_vf=c.cvf_c)


def minibatch(c: Case, d, perms, k):
    """Rows of optimiser step k (epoch k // steps_per_epoch) as float64 tensors."""
    bs = c.B or c.N
    spe = -(-c.N // bs)
    e, j = divmod(k, spe)
    idx = perms[e][j * bs:(j + 1) * bs]
    mb = {f: th.tensor(d["flat"][f][idx], dtype=th.float64) for f in oppo.FLAT_FIELDS}
    for f in oppo.FLAT_FIELDS[2:]:
        mb[f] = mb[f].flatten()
    return mb


def grad64(c: Case, P64, mb, nu):
    """float64 clipped gradient (list, in parameter order), pre-clip norm, and the guard distances of the minibatch."""
    P = {n: p.clone().requires_grad_(True) for n, p in P64.items()}
    loss, _ = oppo.minibatch_loss(P, mb, c.disc, c.clip, nu, c.ent, 0.5, 0.5, c.cvf_r, c.cvf_c)
    g = th.autograd.grad(loss, list(P.values()), allow_unused=True)
    g = [th.zeros_like(p) if x is None else x for p, x in zip(P.values(), g)]
    clipped, total = oppo.clip_grad_norm(g, c.mgn)
    with th.no_grad():
        v, cv, lp, _ = oppo.evaluate_actions(P64, mb["observations"], mb["actions"].long().flatten() if c.disc
                                             else mb["actions"], c.disc)
        ratio = th.exp(lp - mb["old_log_prob"])
        dist = [float(th.min(th.abs(ratio - (1 - c.clip)))), float(th.min(th.abs(ratio - (1 + c.clip))))]
        for cr, val, old in ((c.cvf_r, v, mb["old_reward_values"]), (c.cvf_c, cv, mb["old_cost_values"])):
            if cr is not None:
                dv = val.flatten() - old
                dist += [float(th.min(th.abs(dv - cr))), float(th.min(th.abs(dv + cr)))]
    return [x.numpy() for x in clipped], float(total), min(dist)


# ------------------------------------------------------------------------------------------------ checks
def launches():
    from icrl_b200 import _lib
    return int(_lib.lib().icrl_launch_count())


def check_trajectory(c: Case):
    from icrl_b200 import logger
    d = make_data(c)
    algo = build_algo(c, d, TRAJ_LR)
    names = names_of(c)
    P = {n: p.clone() for n, p in d["P"].items()}
    adam = ocn.adam_init(list(P.values()))
    dual = oppo.dual_init(c.nu)
    logger.configure()
    np.random.seed(NP_SEED)
    bs = c.B or c.N
    worst = [0.0, 0.0]
    outs = []
    for call in (1, 2):
        nu = float(algo.dual.nu.state[4])            # the multiplier the kernel reads
        assert abs(nu - oppo.dual_nu(dual).item()) <= 1e-6 * max(1.0, nu)
        st0 = np.random.get_state()
        n0 = launches()
        algo.train()
        n_launch = launches() - n0
        rng_gpu = np.random.get_state()
        st = algo.last_train_stats
        early = int(logger.Logger.CURRENT.name_to_value["train/early_stop_epoch"])
        sd = algo.policy.state_dict()
        got = [sd[n].numpy().copy() for n in names]
        # the oracle on the same permutations
        np.random.set_state(st0)
        perms, states = draw_perms(c)
        out = oppo.train(P, adam, d["flat"], perms, **oracle_kwargs(c, TRAJ_LR, nu))
        outs.append(out)
        oppo.dual_step(dual, np.mean(time_major(c, d["orig_costs"])), 0.0, PENALTY_LR)
        np.random.set_state(rng_gpu)
        # which kernel ran: gather + stats + train per epoch (many clusters) or per call, plus the dual step
        assert n_launch == (3 * c.epochs if c.many else 3) + 1, (n_launch, c.many)
        err = max_param_err(got, [P[n].numpy() for n in names])
        worst[0] = max(worst[0], err)
        print(f"\n  trajectory call {call}: params {err:.2e}", end="")
        assert err <= TRAJ_TOL[call - 1], f"call {call}: params {err}"
        assert early == out["early_stop_epoch"], (early, out["early_stop_epoch"])
        assert algo.policy.optimizer.step_count == adam["step"] and st.shape[0] == out["steps"]
        want_rng = states[min(c.epochs, early + 1) - 1]
        assert rng_gpu[2] == want_rng[2] and np.array_equal(rng_gpu[1], want_rng[1]), f"call {call}: numpy RNG position"
        ps = out["per_step"]
        spe = -(-c.N // bs)
        for i in range(st.shape[0]):
            e, j = divmod(i, spe)
            bn = min(bs, c.N - j * bs)
            # approx_kl is a mean of differences of log-probs, each rounded to fp32 at its own magnitude: its floor
            # scales with the minibatch's mean |old log-prob| (up to ~20 with 16 action dims)
            lp_scale = float(np.mean(np.abs(d["flat"]["old_log_prob"][perms[e][j * bs:(j + 1) * bs]])))
            for col, key in ((0, "pg_loss"), (2, "reward_value_loss"), (3, "cost_value_loss"), (4, "entropy_loss"),
                             (5, "approx_kl"), (7, "grad_norm")):
                v, r = float(st[i, col]), ps[key][i]
                floor = max(1e-2, 1e-2 * lp_scale) if key == "approx_kl" else 1e-2
                worst[1] = max(worst[1], abs(v - r) / max(abs(r), floor))
                assert abs(v - r) <= METRIC_RTOL * max(abs(r), floor), (call, i, key, v, r)
            # clip_fraction: a ratio within an fp32 rounding of the edge may be counted on the other side
            assert abs(float(st[i, 1]) - ps["clip_fraction"][i]) <= 1.0 / bn + 1e-6, (call, i, st[i, 1])
            assert st[i, 6] == 0.0          # the total loss is assembled on the host from the parts
        np.testing.assert_allclose(algo.dual.nu.log_nu.cpu().numpy(), dual["log_nu"].numpy(), rtol=1e-6, atol=1e-6)
    print(f" (worst stat {worst[1]:.2e})", end="")
    return outs


def grad_err(got, want):
    """max over tensors of ||got - want||_inf / max(||want||_inf, ||g||_inf / 10), g the whole gradient: a tensor whose
    gradient cancels to a small sum of large per-row terms (a 1-wide layer, a bias of a saturated unit) carries the
    rounding of those terms, not of its sum (the fp32 oracle itself is 1.7e-5 off float64 there, relative to the
    tensor).  A tensor whose largest entry is at least a tenth of the largest overall is held to GRAD_TOL of its own
    size; a smaller one to GRAD_TOL of a tenth of the largest entry."""
    top = max(float(np.max(np.abs(np.asarray(b, np.float64)))) for b in want)
    return max_grad_err(got, want) if top == 0 else max(
        float(np.max(np.abs(np.asarray(a, np.float64) - b))) / max(float(np.max(np.abs(b))), top / 10, 1e-30)
        for a, b in zip(got, want))


def check_gradient(c: Case):
    d = make_data(c)
    bs = c.B or c.N
    spe = -(-c.N // bs)
    ks = sorted({0, 1, spe - 1, spe})           # first two steps, epoch 0's (ragged) last step, epoch 1's first step
    runs = {}

    def run(n):
        if n not in runs:
            algo = build_algo(c, d, GRAD_LR)
            np.random.seed(NP_SEED)
            nu = float(algo.dual.nu.state[4])
            stats = None
            if n:
                algo._max_steps = n
                algo.train()
                stats = algo.last_train_stats.copy()
                assert stats.shape[0] == n
            pol = algo.policy
            runs[n] = (pol.parameters_flat().double().cpu().clone(), pol._adam_m.double().cpu().clone(),
                       pol._adam_v.cpu().clone(), stats, nu, pol._slices)
        return runs[n]

    np.random.seed(NP_SEED)
    perms, _ = draw_perms(c)
    names = names_of(c)
    worst = 0.0
    for k in ks:
        theta, m_k, _, _, nu, slices = run(k)
        _, m_k1, _, stats, _, _ = run(k + 1)
        g = ((m_k1 - BETA1 * m_k) / (1 - BETA1)).numpy()
        P64 = {n: theta[off:off + int(np.prod(shape))].reshape(shape) for n, (off, shape) in zip(names, slices)}
        g64, norm64, dist = grad64(c, P64, minibatch(c, d, perms, k), nu)
        assert dist > GUARD, f"k={k}: a row sits {dist:.1e} from a clip edge (choose another seed)"
        assert abs(norm64 / c.mgn - 1) > 1e-3, f"k={k}: gradient norm {norm64} at max_grad_norm"
        got = [g[off:off + int(np.prod(shape))].reshape(shape) for off, shape in slices]
        err = grad_err(got, g64)
        nerr = abs(float(stats[k, 7]) - norm64) / norm64
        worst = max(worst, err)
        print(f"\n  gradient k={k}: {err:.2e}, norm {nerr:.2e}", end="")
        assert err <= GRAD_TOL, f"k={k}: gradient {err}"
        assert nerr <= NORM_RTOL, f"k={k}: pre-clip norm {stats[k, 7]} vs {norm64}"
    # deterministic: a repeat of the longest run gives the same bits
    n = max(ks) + 1
    first = runs.pop(n)
    again = run(n)
    for a, b in zip(first[:4], again[:4]):
        assert np.array_equal(np.asarray(a), np.asarray(b))
    return worst


def _env(c: Case, monkeypatch):
    if c.wide:
        monkeypatch.setenv("ICRL_PPO_WIDE", "1")
        monkeypatch.setenv("ICRL_PPO_WIDE_CLUSTERS", str(c.wide))
    else:
        monkeypatch.delenv("ICRL_PPO_WIDE", raising=False)
        monkeypatch.delenv("ICRL_PPO_WIDE_CLUSTERS", raising=False)


@pytest.mark.parametrize("name", list(CASES))
def test_trajectory_vs_oracle(name, monkeypatch):
    c = CASES[name]
    _env(c, monkeypatch)
    outs = check_trajectory(c)
    if c.target_kl is not None:          # the case means something: the first call stops after epoch 1
        assert outs[0]["early_stop_epoch"] == 1


@pytest.mark.parametrize("name", list(CASES))
def test_gradient_vs_float64(name, monkeypatch):
    c = CASES[name]
    _env(c, monkeypatch)
    check_gradient(c)


# ------------------------------------------------------------------------------------------------ policy forward
FWD_ROWS = (1, 63, 64, 65, 100_003)


@pytest.mark.parametrize("name", list(CASES))
def test_policy_forward_vs_float64(name):
    """forward_heads and evaluate_actions at every sweep shape against float64 oracle.ppo (tolerances of
    tests/test_k4_gpu.py::test_policy_forward_vs_oracle).  For 100 003 rows (a grid that strides) the oracle checks the
    first and last 2 048 rows and 4 096 drawn at random."""
    c = CASES[name]
    d = make_data(c)
    algo = build_algo(c, d, TRAJ_LR)
    pol = algo.policy
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


# ------------------------------------------------------------------------------------------------ refusals
def test_obs_dim_129_is_refused_and_leaves_the_state_alone():
    from icrl_b200 import _lib
    c = Case(129, A=4, T=32, B=64)
    d = make_data(c)
    algo = build_algo(c, d, TRAJ_LR)
    pol = algo.policy
    pol._adam_m.fill_(0.25)
    pol._adam_v.fill_(0.5)
    before = [t.clone() for t in (pol._params, pol._adam_m, pol._adam_v)]
    with pytest.raises(_lib.IcrlError, match="obs_dim 129"):
        algo.train()
    for a, b in zip(before, (pol._params, pol._adam_m, pol._adam_v)):
        assert th.equal(a, b)
    assert pol.optimizer.step_count == 0


@pytest.mark.parametrize("hidden,A", [((65, 65), 4), ((64, 64), 17)])
def test_unsupported_shapes_are_refused_at_construction(hidden, A):
    c = Case(8, hidden, A=A, T=8, B=32)
    from icrl_b200.ppo_lag import PPOLagrangian
    with pytest.raises(NotImplementedError):
        PPOLagrangian("TwoCriticsMlpPolicy", FakeVecEnv(c.D, c.A, False, c.E), n_steps=c.T, batch_size=c.B,
                      policy_kwargs=dict(net_arch=[dict(pi=list(hidden), vf=list(hidden), cvf=list(hidden))]),
                      device="cuda")


# ------------------------------------------------------------------------------------------------ dual step
# The kernel sums the costs in float64 and rounds the mean once to float32; numpy's float32 mean (what the reference
# feeds the dual step) sums pairwise in float32, within ceil(log2 n) float32 roundings of the exact mean.  The oracle is
# fed the float64 mean rounded to float32, so what remains is the scalar float32 arithmetic of one Adam step.
DUAL_CASES = {   # penalty_init, clamp_at, alpha, lr, cost means (one per step), n
    "above_and_below_alpha": (1.0, None, 0.5, 0.05, (0.9, 0.8, 0.2, 0.1, 0.7), 10_240),
    "clamp_binds": (1.0, None, 0.5, 1.0, (0.1, 0.05, 0.1, 0.2), 10_240),
    "softplus_threshold": (25.0, None, 0.2, 0.5, (0.1, 0.6, 0.3), 1_000_003),
    "one_cost": (2.0, 0.5, 0.1, 0.5, (0.3, -0.2, 0.5, 0.0), 1),
}


@pytest.mark.parametrize("name", list(DUAL_CASES))
def test_dual_step_vs_oracle(name):
    from icrl_b200.dual_variable import DualVariable
    p0, clamp_at, alpha, lr, means, n = DUAL_CASES[name]
    dv = DualVariable(alpha, lr, p0, clamp_at, device="cuda")
    ref = oppo.dual_init(p0, clamp_at=dv.nu.clamp_at)
    assert float(dv.nu.state[0]) == float(ref["log_nu"][0])
    rng = np.random.default_rng(len(name))
    clamped = above = below = 0
    for i, mean in enumerate(means):
        costs = (mean + rng.standard_normal(n) * (0.5 if n > 1 else 0.0)).astype(np.float32)
        exact = float(np.mean(costs, dtype=np.float64))
        dv.update_parameter(th.tensor(costs, device="cuda"))
        st = dv.nu.state.cpu().numpy()
        assert st[5] == np.float32(exact) or abs(float(st[5]) - exact) <= 1.2e-7 * abs(exact), (i, st[5], exact)
        bound = np.ceil(np.log2(max(n, 2))) * np.finfo(np.float32).eps * float(np.mean(np.abs(costs), dtype=np.float64))
        assert abs(float(st[5]) - float(np.mean(costs))) <= bound + 1e-12
        loss = oppo.dual_step(ref, np.float32(exact), alpha, lr)
        above += exact > alpha
        below += exact < alpha
        clamped += bool(ref["log_nu"][0] == np.float32(np.log(max(np.exp(ref["clamp_at"]) - 1, 1e-8))))
        want = float(ref["log_nu"][0])
        print(f"\n  step {i}: log_nu {float(st[0]):.7g} vs {want:.7g}, mean cost {float(st[5]):.7g} vs numpy "
              f"{float(np.mean(costs)):.7g}", end="")
        assert abs(float(st[0]) - want) <= 2e-6 * max(1.0, abs(want)), (i, float(st[0]), want)
        assert abs(float(st[4]) - float(oppo.dual_nu(ref)[0])) <= 2e-6 * max(1.0, abs(want)), (i, st[4])
        assert abs(float(st[3]) - float(loss[0])) <= 2e-6 * max(1.0, abs(float(loss[0]))), (i, st[3], loss)
        assert np.allclose(st[1:3], [float(ref["adam"]["exp_avg"][0][0]), float(ref["adam"]["exp_avg_sq"][0][0])],
                           rtol=1e-5, atol=1e-12)
    assert dv.steps == len(means) and ref["adam"]["step"] == len(means)
    if name == "above_and_below_alpha":
        assert above and below
    if name == "clamp_binds":
        assert clamped
    if name == "softplus_threshold":
        assert float(dv.nu.state[0]) > 20.0
