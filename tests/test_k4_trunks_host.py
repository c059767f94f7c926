"""CPU: per-trunk policy widths (icrl_ppo_cfg.trunk_hidden) at the C ABI -- the flat parameter count agrees with the
reference-layout skeleton, bad widths are refused without touching a GPU with a message naming the trunk, the struct
field sits where the ctypes mirror puts it, and the tests' per-trunk initialisation (k4_trunks_helpers) builds the
skeleton's names and shapes."""
import ctypes as C
import os
import subprocess

import pytest
import torch as th

from conftest import ROOT
from oracle import ppo as oppo


@pytest.fixture(scope="module")
def lib():
    from icrl_b200 import build, _lib
    build.build()
    return _lib.lib()


def cfg_for(D, A, disc, trunks):
    from icrl_b200 import _lib
    cfg = _lib.PpoCfg()
    cfg.obs_dim, cfg.act_dim, cfg.is_discrete = D, A, int(disc)
    cfg.T = cfg.E = 1
    for t, (h0, h1) in enumerate(trunks):
        cfg.trunk_hidden[t][0], cfg.trunk_hidden[t][1] = h0, h1
    return cfg


def skeleton(D, A, disc, trunks):
    from icrl_b200.policies import _PolicyShape
    pi, vf, cvf = (list(t) for t in trunks)
    return _PolicyShape(D, A, disc, pi, vf, cvf, th.nn.Tanh, 0.0, True)


SHAPES = [  # obs_dim, actions, discrete, (pi, vf, cvf), flat parameter count
    (18, 6, False, ((64, 64), (32, 32), (16, 48)), 8638),
    (1, 2, True, ((20, 20), (64, 64), (1, 64)), 5050),
    (113, 8, False, ((64, 64), (64, 32), (48, 64)), None),
    (30, 12, False, ((7, 33), (48, 48), (64, 40)), None),
    (30, 4, False, ((33, 7), (7, 33), (64, 1)), None),
    (128, 16, True, ((1, 1), (64, 64), (2, 3)), None),
]


@pytest.mark.parametrize("D,A,disc,trunks,count", SHAPES)
def test_param_count_matches_the_skeleton(lib, D, A, disc, trunks, count):
    n = sum(p.numel() for p in skeleton(D, A, disc, trunks).parameters())
    if count is not None:
        assert n == count
    assert lib.icrl_ppo_param_count(C.byref(cfg_for(D, A, disc, trunks))) == n
    # hidden[] is ignored once trunk_hidden is set
    cfg = cfg_for(D, A, disc, trunks)
    cfg.hidden[0], cfg.hidden[1] = 65, 0
    assert lib.icrl_ppo_param_count(C.byref(cfg)) == n


def test_zero_trunk_hidden_uses_hidden_for_every_trunk(lib):
    from icrl_b200 import _lib
    cfg = _lib.PpoCfg()
    cfg.obs_dim, cfg.act_dim, cfg.T, cfg.E = 18, 6, 1, 1
    cfg.hidden[0], cfg.hidden[1] = 48, 24
    n = lib.icrl_ppo_param_count(C.byref(cfg))
    assert n == lib.icrl_ppo_param_count(C.byref(cfg_for(18, 6, False, ((48, 24),) * 3)))
    assert n == sum(p.numel() for p in skeleton(18, 6, False, ((48, 24),) * 3).parameters())


@pytest.mark.parametrize("trunk,bad", [(0, (65, 64)), (1, (64, 65)), (2, (0, 64)), (2, (64, 0)), (1, (-1, 8)),
                                       (0, (0, 0))])
def test_bad_trunk_widths_are_refused_without_gpu(lib, trunk, bad):
    trunks = [(64, 64), (32, 32), (16, 48)]
    trunks[trunk] = bad
    assert lib.icrl_ppo_param_count(C.byref(cfg_for(18, 6, False, trunks))) == -1
    msg = lib.icrl_last_error().decode()
    assert f"trunk_hidden[{trunk}] ({('pi', 'vf', 'cvf')[trunk]})" in msg, msg
    # every entry point validates through the same path before any launch
    cfg = cfg_for(18, 6, False, trunks)
    assert lib.icrl_policy_forward(C.byref(cfg), None, None, 4, None, None, None, None) == -1
    assert lib.icrl_ppo_train(C.byref(cfg), None, None, None, None, 0, None, None, None) == -1
    assert lib.icrl_launch_count() == 0


def test_trunk_hidden_offset_matches_the_header(lib, tmp_path):
    from icrl_b200 import _lib
    probe = tmp_path / "probe.c"
    probe.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "icrl_b200.h"\n'
                     'int main(){printf("%zu %zu %zu\\n", offsetof(icrl_ppo_cfg, trunk_hidden), '
                     'sizeof(((icrl_ppo_cfg*)0)->trunk_hidden), sizeof(icrl_ppo_cfg));return 0;}\n')
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(probe), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got == [_lib.PpoCfg.trunk_hidden.offset, _lib.PpoCfg.trunk_hidden.size, C.sizeof(_lib.PpoCfg)]
    assert _lib.PpoCfg.trunk_hidden.offset > _lib.PpoCfg.max_steps.offset     # appended: earlier fields do not move


@pytest.mark.parametrize("D,A,disc,trunks,count", SHAPES)
def test_per_trunk_init_matches_the_skeleton(D, A, disc, trunks, count):
    from k4_trunks_helpers import embed, init_policy_trunks
    P = init_policy_trunks(D, A, disc, trunks, generator=th.Generator().manual_seed(0))
    sk = skeleton(D, A, disc, trunks)
    assert [(n, tuple(p.shape)) for n, p in P.items()] == [(n, tuple(p.shape)) for n, p in sk.named_parameters()]
    assert list(P) == oppo.param_names(disc)
    # the 64-64 embedding keeps every entry and pads with exact zeros
    E = embed(P, D, A, disc)
    for n, p in P.items():
        inner = tuple(slice(0, s) for s in p.shape)
        assert th.equal(E[n][inner], p)
        assert int((E[n] != 0).sum()) == int((p != 0).sum())
