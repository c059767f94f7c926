"""CPU: the oracle (oracle/*.py) against the fixtures produced by the unmodified reference (tests/golden)."""
import glob
import os

import numpy as np
import pytest
import torch as th

from conftest import GOLDEN, load_golden
from helpers import COST_ATOL, COST_RTOL, SHAPES, cn_params, cn_spec, max_param_err, policy_params
from oracle import cn as ocn
from oracle import gae as ogae
from oracle import ppo as oppo

th.set_num_threads(1)


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("variant", ["raw", "norm"])
@pytest.mark.parametrize("tag", ["f64", "f32"])
def test_k1_cost_matches_reference(shape, variant, tag):
    d = load_golden(f"k1_{shape}_{variant}_{tag}")
    spec = cn_spec(shape, d)
    x = ocn.prepare_data(spec, d["obs"], d["acs"])
    assert x.dtype == np.float32 and np.array_equal(x, d["x"])          # input prep is bit exact
    cost = ocn.cost_function(cn_params(d), spec, d["obs"], d["acs"])
    assert cost.dtype == np.float32 and cost.shape == d["cost"].shape
    np.testing.assert_array_equal(cost, d["cost"])                       # same library, same arithmetic


def test_k1_3d_input():
    d = load_golden("k1_hc_3d")
    cost = ocn.cost_function(cn_params(d), cn_spec("hc", d), d["obs"], d["acs"])
    assert cost.shape == (6, 5)
    np.testing.assert_array_equal(cost, d["cost"])


def test_k1_real_checkpoints():
    d = load_golden("k1_point_ckpt")
    assert bool(d["loaded_clip_obs_is_none"]) and bool(d["loaded_action_high_is_none"])  # load() quirk a18
    # after ConstraintNet.load: no obs clipping, no action clipping, raw inputs, select [0,1]
    spec = ocn.CNSpec(6, 2, tuple(d["hidden_sizes"]), False, obs_select_dim=[0, 1], acs_select_dim=[-1], clip_obs=None)
    assert spec.select_dim == list(d["select_dim"])
    np.testing.assert_array_equal(ocn.cost_function(cn_params(d), spec, d["obs"], d["acs"]), d["cost"])
    d = load_golden("k1_antbroken_ckpt")
    spec = ocn.CNSpec(113, 8, tuple(d["hidden_sizes"]), False, clip_obs=None)
    np.testing.assert_array_equal(ocn.cost_function(cn_params(d), spec, d["obs"], d["acs"]), d["cost"])
    d = load_golden("k1_ant_expert_slice")
    np.testing.assert_array_equal(ocn.cost_function(cn_params(d), cn_spec("ant", d), d["obs"], d["acs"]), d["cost"])


K2_CASES = sorted(os.path.basename(p)[3:-4] for p in glob.glob(os.path.join(GOLDEN, "k2_*.npz")))


@pytest.mark.parametrize("case", K2_CASES)
def test_k2_train_matches_reference(case):
    d = load_golden(f"k2_{case}")
    shape = case.split("_")[0]
    spec = cn_spec(shape, d, regularizer_coeff=float(d["reg"]), importance_sampling=not bool(d["no_is"]),
                   per_step_importance_sampling=bool(d["per_step"]), target_kl_old_new=float(d["tkon"]),
                   target_kl_new_old=float(d["tkno"]), train_gail_lambda=bool(d.get("gail", False)))
    params = cn_params(d, "p0.")
    adam = ocn.adam_init(params)
    batch_size = int(d["batch_size"]) if int(d.get("batch_size", 0)) > 0 else None    # -cbs minibatch fixtures (round 2)
    if "numpy_seed" in d:
        np.random.seed(int(d["numpy_seed"]))
    for call in (1, 2):
        if f"p{call}.0.weight" not in d:
            break
        m = ocn.train(params, adam, spec, int(d["iters"]), d["nominal_obs"], d["nominal_acs"], d["lengths"],
                      d["expert_obs"], d["expert_acs"], lr=float(d["lr"]), materialize_broadcast=True,
                      batch_size=batch_size)
        if f"rng_pos{call}" in d:       # the global numpy RNG stands where the reference left it
            st = np.random.get_state()
            assert st[2] == int(d[f"rng_pos{call}"]) and (st[1][:4].astype(np.int64) == d[f"rng_probe{call}"]).all()
        ref = cn_params(d, f"p{call}.")
        assert max_param_err([p.numpy() for p in params], [p.numpy() for p in ref]) <= 1e-6
        for k, v in m.items():
            r = float(d[f"m{call}.{k}"])
            if np.isnan(r) or np.isinf(r):
                assert (np.isnan(v) and np.isnan(r)) or v == r, k
            else:
                assert abs(v - r) <= 1e-5 * max(abs(r), 1e-2), (k, v, r)
        nstep = float(d[f"c{call}.adam.0.step"])
        assert adam["step"] == nstep


@pytest.mark.parametrize("case", [c for c in K2_CASES if c.startswith("hc_") or "gail" in c])
def test_k2_float64_gradient_matches_first_adam_moment(case):
    """Adam's first moment after one step is exactly (1 - beta1) * g, so the fp32 oracle's exp_avg after one full-batch
    iteration reads back its gradient: the float64 gradient of ocn.loss_terms (the GPU suite's chain-free reference) must
    equal it to fp32 rounding.  Measured worst, relative to the tensor's largest entry: 7.9e-6 on the output bias (whose
    gradient is a difference of the nominal and the expert sums), <= 1.3e-6 on every other tensor."""
    from helpers import cn_grad64, max_grad_err
    d = load_golden(f"k2_{case}")
    spec = cn_spec(case.split("_")[0], d, regularizer_coeff=float(d["reg"]), importance_sampling=not bool(d["no_is"]),
                   per_step_importance_sampling=bool(d["per_step"]), train_gail_lambda=bool(d.get("gail", False)))
    params = cn_params(d, "p0.")
    g64 = cn_grad64(params, spec, d["nominal_obs"], d["nominal_acs"], d["lengths"], d["expert_obs"], d["expert_acs"])
    adam = ocn.adam_init(params)
    ocn.train(params, adam, spec, 1, d["nominal_obs"], d["nominal_acs"], d["lengths"], d["expert_obs"], d["expert_acs"],
              lr=float(d["lr"]))
    assert adam["step"] == 1
    err = max_grad_err([m.numpy() for m in adam["exp_avg"]], [0.1 * g for g in g64])
    assert err <= 2e-5, err


@pytest.mark.parametrize("case", ["hc_perstep_mild", "ant_perstep"])
def test_k2_quirk_a_identity(case):
    """mean over the reference's [N,N,1] broadcast == mean(w) * mean(log p): the O(N) form the product uses."""
    d = load_golden(f"k2_{case}")
    spec = cn_spec(case.split("_")[0], d, regularizer_coeff=float(d["reg"]), per_step_importance_sampling=True,
                   target_kl_old_new=float(d["tkon"]), target_kl_new_old=float(d["tkno"]))
    params = cn_params(d, "p0.")
    ocn.train(params, ocn.adam_init(params), spec, int(d["iters"]), d["nominal_obs"], d["nominal_acs"], d["lengths"],
              d["expert_obs"], d["expert_acs"], lr=float(d["lr"]), materialize_broadcast=False)
    ref = cn_params(d, "p1.")
    assert max_param_err([p.numpy() for p in params], [p.numpy() for p in ref]) <= 1e-4


K3_CASES = sorted(os.path.basename(p)[3:-4] for p in glob.glob(os.path.join(GOLDEN, "k3_*.npz")))


@pytest.mark.parametrize("case", K3_CASES)
def test_k3_gae_bit_exact(case):
    d = load_golden(f"k3_{case}")
    g = d["gammas"]
    out = ogae.dual_gae(d["rewards"], d["reward_values"], d["costs"], d["cost_values"], d["dones"],
                        d["reward_last_value"], d["cost_last_value"], d["last_dones"], g[0], g[1], g[2], g[3])
    for k, v in out.items():
        assert v.dtype == np.float32
        np.testing.assert_array_equal(v, d[k])


K4_CASES = sorted(os.path.basename(p)[3:-4] for p in glob.glob(os.path.join(GOLDEN, "k4_*.npz")))


def k4_inputs(d):
    flat = {
        "observations": ogae.env_major(d["buf.observations"]), "actions": ogae.env_major(d["buf.actions"]),
        "old_log_prob": ogae.env_major(d["buf.log_probs"]), "old_reward_values": ogae.env_major(d["buf.reward_values"]),
        "reward_advantages": ogae.env_major(d["buf.reward_advantages"]),
        "reward_returns": ogae.env_major(d["buf.reward_returns"]),
        "old_cost_values": ogae.env_major(d["buf.cost_values"]),
        "cost_advantages": ogae.env_major(d["buf.cost_advantages"]),
        "cost_returns": ogae.env_major(d["buf.cost_returns"]),
    }
    hp = {k[3:]: float(v) for k, v in d.items() if k.startswith("hp.")}
    return flat, hp


def k4_kwargs(hp, is_discrete, nu):
    opt = lambda k: None if hp[k] < 0 else hp[k]
    return dict(is_discrete=is_discrete, batch_size=None if hp["batch_size"] < 0 else int(hp["batch_size"]),
                n_epochs=int(hp["n_epochs"]), lr=hp["learning_rate"], clip_range=hp["clip_range"], nu=nu,
                ent_coef=hp["ent_coef"], target_kl=opt("target_kl"), clip_range_reward_vf=opt("clip_range_reward_vf"),
                clip_range_cost_vf=opt("clip_range_cost_vf"))


K4X_CASES = sorted(os.path.basename(p)[4:-4] for p in glob.glob(os.path.join(GOLDEN, "k4x_*.npz")))


@pytest.mark.parametrize("case", K4_CASES + ["x:" + c for c in K4X_CASES])
def test_k4_train_matches_reference(case):
    """k4_*: small fixtures; x:* (round 2): the full-size HalfCheetah train() (1 600 dependent optimiser steps) and the
    large-batch regime (batch >= 2048), inputs regenerated from their seed."""
    if case.startswith("x:"):
        from helpers import load_k4x
        d = load_k4x(case[2:])
    else:
        d = load_golden(f"k4_{case}")
    is_discrete = "log_std" not in [str(n) for n in d["param_order"]]
    flat, hp = k4_inputs(d)
    P = policy_params(d, "p0.")
    adam = ocn.adam_init(list(P.values()))
    dual = oppo.dual_init(hp["penalty_initial_value"])
    assert np.allclose(dual["log_nu"].numpy(), d["log_nu0"], rtol=0, atol=0)
    n = flat["observations"].shape[0]
    for call in range(1, int(hp.get("trains", 2)) + 1):
        if call == 1:
            np.random.seed(int(hp["numpy_seed"]))
        nu = oppo.dual_nu(dual).item()
        # the reference draws one permutation per epoch it actually runs (buffers.py:596)
        perms = []

        class LazyPerms:
            def __getitem__(self, e):
                while len(perms) <= e:
                    perms.append(np.random.permutation(n))
                return perms[e]
        out = oppo.train(P, adam, flat, LazyPerms(), **k4_kwargs(hp, is_discrete, nu))
        oppo.dual_step(dual, np.mean(d["buf.orig_costs"]), 0.0, hp["penalty_learning_rate"])
        ref = policy_params(d, f"p{call}.")
        err = max_param_err([p.numpy() for p in P.values()], [p.numpy() for p in ref.values()])
        # 1 600 dependent steps amplify last-bit differences between the oracle's explicit-weight autograd graph and the
        # reference's modules (hc_full: measured 6e-5)
        assert err <= (1e-4 if case == "x:hc_full" else 2e-5), err
        assert np.allclose(dual["log_nu"].numpy(), d[f"log_nu{call}"], rtol=1e-6)
        if call == 1:
            log = {k[4:]: float(v) for k, v in d.items() if k.startswith("log.")}
            ps = out["per_step"]
            chk = {"train/entropy_loss": np.mean(ps["entropy_loss"]), "train/policy_gradient_loss": np.mean(ps["pg_loss"]),
                   "train/reward_value_loss": np.mean(ps["reward_value_loss"]),
                   "train/cost_value_loss": np.mean(ps["cost_value_loss"]),
                   "train/clip_fraction": np.mean(ps["clip_fraction"]), "train/loss": ps["loss"][-1],
                   "train/approx_kl": out["last_epoch_approx_kl"], "train/early_stop_epoch": out["early_stop_epoch"]}
            for k, v in chk.items():
                assert abs(v - log[k]) <= 1e-5 * max(abs(log[k]), 1e-2), (k, v, log[k])


def test_k4_float64_gradient_matches_reference_first_adam_moment():
    """k4_hc_fullbatch takes one full-batch optimiser step, after which the reference's exp_avg is exactly
    (1 - beta1) * (clipped gradient): the float64 gradient of oracle.ppo.minibatch_loss at p0, clipped the torch way (the
    GPU sweep's chain-free reference, tests/test_k4_sweep_gpu.py), must equal it to fp32 rounding.  Measured worst,
    per tensor relative to its largest entry: 1.1e-6."""
    from helpers import max_grad_err
    d = load_golden("k4_hc_fullbatch")
    flat, hp = k4_inputs(d)
    names = [str(n) for n in d["param_order"]]
    P = {n: th.tensor(d["p0." + n], dtype=th.float64, requires_grad=True) for n in names}
    mb = {k: th.tensor(v, dtype=th.float64) for k, v in flat.items()}
    for k in oppo.FLAT_FIELDS[2:]:
        mb[k] = mb[k].flatten()
    nu = float(oppo.dual_nu(oppo.dual_init(hp["penalty_initial_value"])))
    opt = lambda k: None if hp[k] < 0 else hp[k]
    loss, _ = oppo.minibatch_loss(P, mb, "log_std" not in names, hp["clip_range"], nu, hp["ent_coef"], 0.5, 0.5,
                                  opt("clip_range_reward_vf"), opt("clip_range_cost_vf"))
    g, _ = oppo.clip_grad_norm(th.autograd.grad(loss, list(P.values())), hp.get("max_grad_norm", 0.5))
    want = [d[f"adam.{i}.exp_avg"].astype(np.float64) / (1 - 0.9) for i in range(len(names))]
    assert hp["batch_size"] < 0 or int(hp["batch_size"]) >= flat["observations"].shape[0]
    err = max_grad_err([x.numpy() for x in g], want)
    assert err <= 1e-5, err


# ------------------------------------------------------------------------------------------- cost normalisation (f1)
@pytest.mark.parametrize("name,norm", [("all", True), ("nocost", False)])
def test_costnorm_oracle_matches_reference_wrappers(name, norm):
    from oracle import costnorm
    g = load_golden(f"venv_{name}")
    T, E = g["orig_cost"].shape
    state = costnorm.reset(costnorm.initial_state(E))
    out = costnorm.normalize_rollout(g["orig_cost"], g["done"], state, cost_gamma=0.97, norm_cost=norm)
    np.testing.assert_array_equal(out, g["cost"].astype(np.float32))
    assert state["mean"] == g["cost_rms_mean"] and state["var"] == g["cost_rms_var"]
    assert state["count"] == float(g["cost_rms_count"])


# ------------------------------------------------------------------------------------------- GAIL discriminator cost (f4)
@pytest.mark.parametrize("name", ["antbroken", "point"])
def test_gail_discriminator_oracle_matches_reference(name):
    """GailDiscriminator.reward_function = select dims -> MLP -> sigmoid with nothing else applied to nominal data
    (gail_utils.py:233-250): the K1 oracle with clipping / normalisation switched off reproduces it bit for bit."""
    import os
    g = load_golden(f"gail_{name}")
    sd = th.load(os.path.join(os.path.dirname(__file__), "golden", f"ref_gail_{name}.pt"), weights_only=False)
    params = [sd["network"][k] for k in sd["network"]]
    sel = ocn.define_select_dim(sd["obs_dim"], sd["acs_dim"], sd["obs_select_dim"], sd["acs_select_dim"])
    spec = ocn.CNSpec(sd["obs_dim"], sd["acs_dim"], tuple(sd["hidden_sizes"]), False, obs_select_dim=sd["obs_select_dim"],
                      acs_select_dim=sd["acs_select_dim"], clip_obs=None)
    assert len(sel) == params[0].shape[1]
    pred = 1.0 - ocn.cost_function(params, spec, g["obs"], g["acs"])
    np.testing.assert_allclose(pred, g["d"], rtol=0, atol=6e-8)
