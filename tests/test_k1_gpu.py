"""GPU parity: K1 (constraint-net forward / cost relabel) through the reference-shaped API and the C-ABI,
against reference-generated goldens and the CPU oracle."""
import numpy as np
import pytest
import torch as th

from conftest import load_golden
from helpers import COST_ATOL, COST_RTOL, SHAPES, cn_params, cn_spec
from oracle import cn as ocn

pytestmark = pytest.mark.gpu


def make_cn(shape, d, hidden=None, **kw):
    from icrl_b200.constraint_net import ConstraintNet
    s = dict(SHAPES[shape], **({"hidden": hidden} if hidden else {}))
    low = high = None
    if not s["is_discrete"]:
        low, high = -np.ones(s["acs_dim"], np.float32), np.ones(s["acs_dim"], np.float32)
    base = dict(clip_obs=20., initial_obs_mean=d.get("obs_mean"), initial_obs_var=d.get("obs_var"), action_low=low,
                action_high=high)
    base.update(kw)
    cn = ConstraintNet(s["obs_dim"], s["acs_dim"], s["hidden"], None, lambda x: 1e-3, None, None, s["is_discrete"], **base)
    cn.load_network_state_dict({k[2:]: th.tensor(v) for k, v in d.items() if k.startswith("p.")})
    return cn


def assert_cost_close(got, want):
    assert got.dtype == np.float32 and got.shape == want.shape
    np.testing.assert_allclose(got, want, rtol=COST_RTOL, atol=COST_ATOL)


@pytest.mark.parametrize("shape", list(SHAPES))
@pytest.mark.parametrize("variant", ["raw", "norm"])
@pytest.mark.parametrize("tag", ["f64", "f32"])
def test_cost_function_vs_reference_golden(shape, variant, tag):
    d = load_golden(f"k1_{shape}_{variant}_{tag}")
    cn = make_cn(shape, d)
    assert_cost_close(cn.cost_function(d["obs"], d["acs"]), d["cost"])


def test_3d_input_and_expert_slice():
    d = load_golden("k1_hc_3d")
    got = make_cn("hc", d).cost_function(d["obs"], d["acs"])
    assert got.shape == (6, 5)
    assert_cost_close(got, d["cost"])
    d = load_golden("k1_ant_expert_slice")
    assert_cost_close(make_cn("ant", d).cost_function(d["obs"], d["acs"]), d["cost"])


@pytest.mark.parametrize("name,kw", [("k1_point_ckpt", dict(obs_dim=6, acs_dim=2, is_discrete=False, obs_select_dim=[0, 1],
                                                             acs_select_dim=[-1], clip_obs=None, obs_mean=None, obs_var=None,
                                                             action_low=-0.25 * np.ones(2, np.float32),
                                                             action_high=0.25 * np.ones(2, np.float32))),
                                     ("k1_antbroken_ckpt", dict(obs_dim=113, acs_dim=8, is_discrete=False))])
def test_load_frozen_checkpoint(tmp_path, name, kw):
    """cpg path (icrl/cpg.py:89-102): a reference-format best_cn_model.pt must load and give the reference's costs,
    including load()'s argument shift (no obs clipping, no action clipping)."""
    from icrl_b200.constraint_net import ConstraintNet
    d = load_golden(name)
    sel = name == "k1_point_ckpt"
    ckpt = dict(cn_network={k[2:]: th.tensor(v) for k, v in d.items() if k.startswith("p.")}, cn_optimizer={},
                obs_dim=113, acs_dim=8, is_discrete=False, obs_select_dim=[0, 1] if sel else None,
                acs_select_dim=[-1] if sel else None, clip_obs=20, obs_mean=None, obs_var=None,
                action_low=-np.ones(8, np.float32), action_high=np.ones(8, np.float32), device="cpu",
                hidden_sizes=[int(h) for h in d["hidden_sizes"]])
    path = str(tmp_path / "best_cn_model.pt")
    th.save(ckpt, path)
    cn = ConstraintNet.load(path, **kw)
    assert cn.clip_obs is None and cn.action_high is None and cn.optimizer is None
    assert cn.select_dim == [int(s) for s in d["select_dim"]]
    assert_cost_close(cn.cost_function(d["obs"], d["acs"]), d["cost"])


# synthetic nets "<inputs>_<hidden widths>_<observation dtype>": every padded width the kernels are built for (8 16 24 32
# 40 48 64), one to three hidden layers, a narrower layer after a wider one, float32 and float64 observations
SYNTH_NETS = ["hc_5_f64", "hc_16x16x16_f32", "ant_32x32_f64", "ant_48x7_f32", "hc_20_f64", "ant_40x40_f64",
              "hc_64x64_f32", "lgw_64x64_f64", "ant_64x64_f32", "ant_64x64_f64", "hc_64x64x64_f32", "hc_64x64x64_f64"]


def synthetic_net(name):
    """A golden-shaped dict for a synthetic net: weights uniform in +-1/sqrt(fan_in) (nn.Linear's default range) under a
    fixed seed, observation normalisation to unit scale for the `* 6` observations of the ragged test."""
    shape, widths, tag = name.split("_")
    hidden = tuple(int(w) for w in widths.split("x"))
    s = dict(SHAPES[shape], hidden=hidden)
    g = th.Generator().manual_seed(len(hidden) * 100 + sum(hidden))
    dims = [s["obs_dim"] + s["acs_dim"]] + list(hidden) + [1]
    d = {"obs_mean": np.zeros(s["obs_dim"]), "obs_var": np.full(s["obs_dim"], 36.0)}
    for i in range(len(dims) - 1):
        bound = 1.0 / np.sqrt(dims[i])
        d[f"p.{2 * i}.weight"] = ((th.rand(dims[i + 1], dims[i], generator=g) * 2 - 1) * bound).numpy()
        d[f"p.{2 * i}.bias"] = ((th.rand(dims[i + 1], generator=g) * 2 - 1) * bound).numpy()
    return shape, s, d, np.float64 if tag == "f64" else np.float32


@pytest.mark.parametrize("n", [1, 5, 31, 127, 128, 129, 1000, 4096 + 17, 16, 17, 18_949, 100_003])
@pytest.mark.parametrize("shape", ["lgw", "ant"] + SYNTH_NETS)
def test_ragged_sizes_vs_oracle(shape, n):
    """Row counts around the tile and warp sizes, and past 128 x 148 (18 949: the packed kernel is the default there for
    nets up to 32 wide), on the golden nets and on synthetic nets of every width."""
    if shape in SHAPES:
        s, d, dtype = SHAPES[shape], load_golden(f"k1_{shape}_norm_f32"), np.float32
        cn = make_cn(shape, d)
    else:
        shape, s, d, dtype = synthetic_net(shape)
        cn = make_cn(shape, d, hidden=s["hidden"])
    rng = np.random.default_rng(n)
    obs = (rng.standard_normal((n, s["obs_dim"])) * 6).astype(dtype)
    acs = (rng.integers(0, s["acs_dim"], (n, 1)).astype(np.float32) if s["is_discrete"]
           else rng.standard_normal((n, s["acs_dim"])).astype(np.float32) * 1.5)
    want = ocn.cost_function(cn_params(d), cn_spec(shape, d, hidden_sizes=s["hidden"]), obs, acs)
    assert_cost_close(cn.cost_function(obs, acs), want)


def test_empty_batch():
    d = load_golden("k1_hc_raw_f32")
    out = make_cn("hc", d).cost_function(np.zeros((0, 18), np.float32), np.zeros((0, 6), np.float32))
    assert out.shape == (0,)


def test_device_resident_relabel_large():
    """Whole-buffer relabel on device-resident [T,E,.] tensors at a size well past L2-resident tiles (1M rows, HC shape)
    vs the oracle on a strided sample + exact agreement with the host-buffer entry point."""
    d = load_golden("k1_hc_raw_f32")
    cn = make_cn("hc", d)
    g = th.Generator(device="cuda").manual_seed(0)
    T, E = 2048, 512
    obs = th.randn(T, E, 18, device="cuda", generator=g) * 5
    acs = th.randn(T, E, 6, device="cuda", generator=g)
    cost = cn.cost_function_device(obs, acs)
    th.cuda.synchronize()
    assert cost.shape == (T, E)
    idx = th.arange(0, T * E, 997, device="cuda")
    o, a = obs.reshape(-1, 18)[idx].cpu().numpy(), acs.reshape(-1, 6)[idx].cpu().numpy()
    want = ocn.cost_function(cn_params(d), cn_spec("hc", d), o, a)
    assert_cost_close(cost.reshape(-1)[idx].cpu().numpy(), want)
    np.testing.assert_array_equal(cn.cost_function(o, a), cost.reshape(-1)[idx].cpu().numpy())


def test_unaligned_base_pointer_falls_back():
    """A device view whose base is not 16-byte aligned must take the non-TMA staging path and still be right."""
    d = load_golden("k1_hc_raw_f32")
    cn = make_cn("hc", d)
    n = 1024
    buf_o = th.randn(n * 18 + 1, device="cuda")
    buf_a = th.randn(n * 6 + 1, device="cuda")
    obs, acs = buf_o[1:].reshape(n, 18), buf_a[1:].reshape(n, 6)
    assert obs.data_ptr() % 16 != 0
    out = th.empty(n, device="cuda")
    import ctypes as C
    from icrl_b200 import _lib
    _lib.check(_lib.lib().icrl_cn_forward(C.byref(cn._get_desc()), _lib.ptr(obs), 0, _lib.ptr(acs), n, _lib.ptr(out), 0,
                                          _lib.current_stream()))
    th.cuda.synchronize()
    want = ocn.cost_function(cn_params(d), cn_spec("hc", d), obs.cpu().numpy(), acs.cpu().numpy())
    assert_cost_close(out.cpu().numpy(), want)


def test_tensor_core_variant_matches_goldens():
    """The opt-in mma.sync variant of K1 (ICRL_K1_MMA=1; read once per process) against the same golden fixtures."""
    import os
    import subprocess
    import sys
    env = dict(os.environ, ICRL_K1_MMA="1", ICRL_K1_MMA_CHILD="1")
    if os.environ.get("ICRL_K1_MMA_CHILD"):
        pytest.skip("already inside the child run")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-m", "gpu", "-x", "-k", "golden or checkpoint or ragged or 3d"],
                       env=env, capture_output=True, text=True, timeout=600, cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert " passed" in r.stdout


def test_packed_kernel_matches_goldens():
    """The packed-FP32 kernel (FFMA2, two rows per thread, double-buffered TMA tiles) is the default only for buffers of
    >= 128 rows per SM and nets up to 32 wide; ICRL_K1_PAIR=1 forces it everywhere (every width, ragged and unaligned
    tiles, float64 observations, normalisation, one-hot actions) against the same goldens."""
    import os
    import subprocess
    import sys
    if os.environ.get("ICRL_K1_PAIR_CHILD"):
        pytest.skip("already inside the child run")
    env = dict(os.environ, ICRL_K1_PAIR="1", ICRL_K1_PAIR_CHILD="1")
    r = subprocess.run([sys.executable, "-m", "pytest", os.path.abspath(__file__), "-q", "-m", "gpu", "-x", "-k",
                        "golden or checkpoint or ragged or 3d or unaligned or large"],
                       env=env, capture_output=True, text=True, timeout=600, cwd=os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert " passed" in r.stdout


@pytest.mark.parametrize("shape", ["hc", "lgw", "ant", "point"])
@pytest.mark.parametrize("n", [5, 16, 77, 50_000])
def test_packed_kernel_is_bit_identical_to_the_scalar_kernel(shape, n, monkeypatch):
    """Same IEEE fma sequence per row (bias + sum over k in order): the scalar kernel, the packed kernel and the tiny-batch
    kernel of the per-environment-step calls (n <= 16: one CTA per row, one thread per hidden unit) must agree bit for bit."""
    if shape not in SHAPES:
        pytest.skip(f"no {shape} shape")
    d = load_golden(f"k1_{shape}_norm_f32")
    s = SHAPES[shape]
    cn = make_cn(shape, d)
    rng = np.random.default_rng(n)
    obs = (rng.standard_normal((n, s["obs_dim"])) * 6).astype(np.float32)
    acs = (rng.integers(0, s["acs_dim"], (n, 1)).astype(np.float32) if s["is_discrete"]
           else rng.standard_normal((n, s["acs_dim"])).astype(np.float32) * 1.5)
    monkeypatch.setenv("ICRL_K1_V1", "1")
    monkeypatch.setenv("ICRL_K1_NO_SMALL", "1")
    scalar = cn.cost_function(obs, acs)
    monkeypatch.delenv("ICRL_K1_V1")
    monkeypatch.setenv("ICRL_K1_PAIR", "1")
    packed = cn.cost_function(obs, acs)
    np.testing.assert_array_equal(packed, scalar)
    if n <= 16:
        monkeypatch.delenv("ICRL_K1_NO_SMALL")
        np.testing.assert_array_equal(cn.cost_function(obs, acs), scalar)                       # tiny-batch kernel, zero-copy path
        monkeypatch.setenv("ICRL_K1_NO_ZEROCOPY", "1")
        np.testing.assert_array_equal(cn.cost_function(obs, acs), scalar)                       # ... through staged copies


@pytest.mark.parametrize("name", ["antbroken", "point"])
def test_gail_discriminator_reward_function(name):
    """`cpg --load_gail`: the reference's shipped discriminators loaded by GailDiscriminator.load, evaluated by K1
    (prediction output), against what the reference's own class returns (tests/golden/make_golden.py::golden_gail)."""
    import os
    from icrl_b200.gail_utils import GailDiscriminator
    g = load_golden(f"gail_{name}")
    gail = GailDiscriminator.load(os.path.join(os.path.dirname(__file__), "golden", f"ref_gail_{name}.pt"))
    d = gail.reward_function(g["obs"], g["acs"], apply_log=False)
    assert d.shape == g["d"].shape
    np.testing.assert_allclose(d, g["d"], rtol=COST_RTOL, atol=COST_ATOL)
    np.testing.assert_allclose(gail.reward_function(g["obs"], g["acs"], apply_log=True), g["logd"], rtol=1e-4, atol=1e-5)
    d3 = gail.reward_function(g["obs"][:60].reshape(12, 5, -1), g["acs"][:60].reshape(12, 5, -1), apply_log=False)
    assert d3.shape == g["d3"].shape
    np.testing.assert_allclose(d3, g["d3"], rtol=COST_RTOL, atol=COST_ATOL)
