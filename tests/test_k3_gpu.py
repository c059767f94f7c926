"""GPU parity: K3 (dual GAE) -- bit exact against the reference goldens and the oracle, plus properties at full size."""
import glob
import os

import numpy as np
import pytest
import torch as th

from conftest import GOLDEN, load_golden
from oracle import gae as ogae

pytestmark = pytest.mark.gpu
K3_CASES = sorted(os.path.basename(p)[3:-4] for p in glob.glob(os.path.join(GOLDEN, "k3_*.npz")))
OUT = ("reward_returns", "reward_advantages", "cost_returns", "cost_advantages")


def run_buffer(d, T, E, g):
    from icrl_b200.buffers import RolloutBufferWithCost
    from icrl_b200.spaces import Box
    buf = RolloutBufferWithCost(T, Box(-1, 1, (3,)), Box(-1, 1, (2,)), "cuda", reward_gamma=g[0], reward_gae_lambda=g[1],
                                cost_gamma=g[2], cost_gae_lambda=g[3], n_envs=E)
    for k in ("rewards", "reward_values", "costs", "cost_values", "dones"):
        getattr(buf, k)[:] = d[k]
    buf.compute_returns_and_advantage(th.tensor(d["reward_last_value"]), th.tensor(d["cost_last_value"]), d["last_dones"])
    return buf


@pytest.mark.parametrize("case", K3_CASES)
def test_gae_bit_exact_vs_reference_golden(case):
    d = load_golden(f"k3_{case}")
    T, E = d["rewards"].shape
    buf = run_buffer(d, T, E, [float(x) for x in d["gammas"]])
    for k in OUT:
        got = getattr(buf, k)
        assert got.dtype == np.float32
        np.testing.assert_array_equal(got, d[k], err_msg=k)


def synth(rng, T, E, ep_len, last="mix"):
    d = {k: rng.standard_normal((T, E)).astype(np.float32) for k in ("rewards", "reward_values", "costs", "cost_values")}
    phase = rng.integers(0, ep_len, size=E)
    d["dones"] = (((np.arange(T)[:, None] + phase[None]) % ep_len) == 0).astype(np.float32)
    # row T-1 is the last one the scan reads (it ends step T-2); row 0 is never read
    d["dones"][T - 1, 1::3] = 1.0
    d["dones"][0, 2::3] = 1.0
    d["last_dones"] = {"mix": rng.random(E) < 0.5, "all": np.ones(E, bool), "none": np.zeros(E, bool)}[last]
    d["reward_last_value"] = rng.standard_normal((E, 1)).astype(np.float32)
    d["cost_last_value"] = rng.standard_normal((E, 1)).astype(np.float32)
    return d


# (reward gamma, reward lambda, cost gamma, cost lambda)
GAMMAS = {"d": (0.99, 0.95, 0.97, 0.9), "std": (0.99, 0.95, 0.99, 0.95), "one": (1.0, 1.0, 1.0, 1.0),
          "nolam": (0.9, 0.0, 0.9, 0.0),
          # gamma * lambda is a float64 product cast once: float32(g * l) != float32(g) * float32(l) for both pairs
          "cast": (0.995, 0.98, 0.98, 0.92)}

# Every dual_gae_kernel<NT, CG> instantiation at the E its launch rule picks it for, with T one step below, at and above
# its window length (NT / CG blocks of 8 steps), several windows, and T not a multiple of 8.
GAE_CASES = [  # T, E, episode length, last_dones, gammas
    # <512, 4>: E < 64, 1024-step windows
    (1, 1, 5, "mix", "d"), (2, 33, 3, "mix", "d"), (63, 5, 7, "mix", "d"), (64, 5, 200, "mix", "d"),
    (257, 31, 150, "mix", "d"), (300, 1, 1, "mix", "d"), (1023, 63, 100, "all", "std"), (1024, 7, 1024, "none", "one"),
    (1025, 63, 300, "mix", "nolam"), (2048, 63, 500, "mix", "cast"), (2001, 9, 64, "none", "cast"),
    # <256, 4>: 64 <= E < 1024, 512-step windows
    (1000, 64, 1000, "mix", "d"), (2048, 96, 500, "mix", "d"), (511, 64, 50, "none", "cast"),
    (512, 1023, 700, "all", "one"), (513, 64, 513, "mix", "std"), (2048, 1023, 400, "mix", "nolam"),
    (77, 1023, 9, "mix", "cast"),
    # <256, 8>: 1024 <= E < 4096, 256-step windows; E % 8 != 0 leaves a column tail in the last CTA
    (255, 1024, 30, "mix", "std"), (256, 1025, 256, "none", "cast"), (257, 4095, 100, "all", "nolam"),
    (2048, 1025, 600, "mix", "one"), (1001, 4095, 250, "mix", "cast"),
    # <128, 8>: E >= 4096, 128-step windows (bench.py's ant sweep times T = 2048 here)
    (127, 4096, 40, "mix", "nolam"), (128, 4097, 128, "all", "cast"), (129, 4096, 60, "none", "std"),
    (2048, 4097, 700, "mix", "cast"), (1024, 4096, 1024, "mix", "one"), (203, 4103, 20, "mix", "d"),
]


def _gae_oracle(d, g):
    return ogae.dual_gae(d["rewards"], d["reward_values"], d["costs"], d["cost_values"], d["dones"],
                         d["reward_last_value"], d["cost_last_value"], d["last_dones"], *g)


@pytest.mark.parametrize("T,E,ep,last,gk", GAE_CASES)
def test_gae_bit_exact_vs_oracle_ragged(T, E, ep, last, gk):
    rng = np.random.default_rng(T * 1000 + E)
    d = synth(rng, T, E, ep, last)
    g = GAMMAS[gk]
    if gk == "cast":
        for gamma, lam in (g[:2], g[2:]):
            assert np.float32(gamma * lam) != np.float32(gamma) * np.float32(lam)
    want = _gae_oracle(d, g)
    buf = run_buffer(d, T, E, g)
    for k in OUT:
        np.testing.assert_array_equal(getattr(buf, k), want[k], err_msg=k)


@pytest.mark.parametrize("T,E,no_zero_copy,path", [(64, 5, False, "pinned"), (64, 5, True, "staged"),
                                                   (2048, 64, False, "staged")])
def test_gae_host_entry_matches_device_buffers(T, E, no_zero_copy, path, monkeypatch):
    """icrl_dual_gae_host works on a host-mapped pinned block when inputs and outputs fit 1 MB, else on staged device
    copies (ICRL_K3_NO_ZEROCOPY forces the staged path); both give the bits of icrl_dual_gae on device buffers."""
    from icrl_b200 import _lib
    n_bytes = (5 * T * E + 2 * E) * 4 + E + 4 * T * E * 4
    assert path == ("pinned" if n_bytes <= 1 << 20 and not no_zero_copy else "staged")
    if no_zero_copy:
        monkeypatch.setenv("ICRL_K3_NO_ZEROCOPY", "1")
    d = synth(np.random.default_rng(E), T, E, 40)
    g = GAMMAS["cast"]
    keys = ("rewards", "reward_values", "costs", "cost_values", "dones", "reward_last_value", "cost_last_value")
    ins = [np.ascontiguousarray(d[k], np.float32).reshape(-1) for k in keys] + [d["last_dones"].astype(np.uint8)]
    host = [np.empty(T * E, np.float32) for _ in range(4)]
    L = _lib.lib()
    _lib.check(L.icrl_dual_gae_host(*[_lib.ptr(a) for a in ins], T, E, *g, *[_lib.ptr(o) for o in host],
                                    _lib.current_stream()))
    dev_in = [th.from_numpy(a).cuda() for a in ins]
    dev = [th.empty(T * E, device="cuda") for _ in range(4)]
    _lib.check(L.icrl_dual_gae(*[_lib.ptr(a) for a in dev_in], T, E, *g, *[_lib.ptr(o) for o in dev],
                               _lib.current_stream()))
    th.cuda.synchronize()
    want = _gae_oracle(d, g)
    for k, h, o in zip(("reward_advantages", "reward_returns", "cost_advantages", "cost_returns"), host, dev):
        np.testing.assert_array_equal(h, o.cpu().numpy(), err_msg=k)
        np.testing.assert_array_equal(h.reshape(T, E), want[k], err_msg=k)


def test_gae_full_size_properties():
    """4M transitions (T=2048, E=2048) on device-resident buffers: (i) lambda=1, no dones => advantage + value equals the
    discounted return with bootstrap (buffers.py:508-511 docstring); (ii) returns == advantages + values exactly;
    (iii) a `done` at t+1 cuts every dependence on the future; (iv) columns are independent."""
    import ctypes as C
    from icrl_b200 import _lib
    T, E = 2048, 2048
    g = th.Generator(device="cuda").manual_seed(1)
    r, vr, c, vc = (th.randn(T, E, device="cuda", generator=g) for _ in range(4))
    dones = th.zeros(T, E, device="cuda")
    lvr, lvc = th.randn(E, device="cuda", generator=g), th.randn(E, device="cuda", generator=g)
    last = th.zeros(E, dtype=th.uint8, device="cuda")
    outs = [th.empty(T, E, device="cuda") for _ in range(4)]

    def run(dn):
        _lib.check(_lib.lib().icrl_dual_gae(*[_lib.ptr(x) for x in (r, vr, c, vc, dn, lvr, lvc, last)], T, E, 0.99, 1.0,
                                            0.9, 1.0, *[_lib.ptr(o) for o in outs], _lib.current_stream()))
        th.cuda.synchronize()
        return [o.clone() for o in outs]

    ar, rr, ac, rc = run(dones)
    assert th.equal(rr, ar + vr) and th.equal(rc, ac + vc)
    # discounted return in float64 on a few columns
    cols = [0, 1, 777, E - 1]
    ret = lvr[cols].double()
    R = th.empty(T, len(cols), dtype=th.float64, device="cuda")
    for t in range(T - 1, -1, -1):
        ret = r[t, cols].double() + 0.99 * ret
        R[t] = ret
    assert th.allclose(rr[:, cols].double(), R, rtol=2e-5, atol=2e-5)
    # a done at t0+1 makes [0, t0] independent of everything after t0
    t0 = 1000
    d2 = dones.clone()
    d2[t0 + 1] = 1.0
    ar2 = run(d2)[0]
    r_saved = r[t0 + 1:].clone()
    r[t0 + 1:] += 3.0
    ar3 = run(d2)[0]
    r[t0 + 1:] = r_saved
    assert th.equal(ar2[:t0 + 1], ar3[:t0 + 1]) and not th.equal(ar2[t0 + 1:], ar3[t0 + 1:])
