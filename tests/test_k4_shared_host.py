"""CPU: shared trunk layers (icrl_ppo_cfg.n_shared) at the C ABI -- the flat parameter count agrees with the
reference-layout skeleton, bad shapes and data-parallel training are refused without touching a GPU, the struct field
sits where the ctypes mirror puts it, and the skeleton's names, shapes and seeded initial weights are those of an
independently built module with SB3's MlpExtractor structure."""
import ctypes as C
import os
import subprocess

import pytest
import torch as th

import k4_shared_helpers as sh
from conftest import ROOT


@pytest.fixture(scope="module")
def lib():
    from icrl_b200 import build, _lib
    build.build()
    return _lib.lib()


def cfg_for(D, A, disc, arch):
    from icrl_b200 import _lib
    cfg = _lib.PpoCfg()
    cfg.obs_dim, cfg.act_dim, cfg.is_discrete = D, A, int(disc)
    cfg.T = cfg.E = 1
    for t, (h0, h1) in enumerate(sh.trunk_hidden(arch)):
        cfg.trunk_hidden[t][0], cfg.trunk_hidden[t][1] = h0, h1
    cfg.n_shared = len(arch[0])
    return cfg


def skeleton(D, A, disc, arch):
    from icrl_b200.policies import _PolicyShape, _trunks
    shared, pi, vf, cvf, _ = _trunks(sh.net_arch(arch))
    return _PolicyShape(D, A, disc, pi, vf, cvf, th.nn.Tanh, 0.0, True, shared)


SHAPES = [  # obs_dim, actions, discrete, architecture (shared widths, private widths of pi, vf, cvf)
    (18, 6, False, ((64,), (64, 32, 16))),
    (113, 8, False, ((64,), (64, 64, 48))),
    (30, 12, False, ((7,), (33, 48, 64))),
    (18, 6, False, ((64, 64), ())),
    (1, 2, True, ((20, 20), ())),
    (128, 16, True, ((1,), (1, 64, 2))),
    (40, 6, False, ((48, 24), ())),
]


@pytest.mark.parametrize("D,A,disc,arch", SHAPES)
def test_param_count_matches_the_skeleton(lib, D, A, disc, arch):
    sk = skeleton(D, A, disc, arch)
    n = sum(p.numel() for p in sk.parameters())
    assert lib.icrl_ppo_param_count(C.byref(cfg_for(D, A, disc, arch))) == n
    assert [name for name, _ in sk.named_parameters()] == sh.param_names(disc, arch)


@pytest.mark.parametrize("D,A,disc,arch", SHAPES)
def test_skeleton_matches_an_sb3_structured_module(D, A, disc, arch):
    """Names, shapes and seeded initial weights (the reference's creation order and orthogonal init) of the policy's
    skeleton equal those of k4_shared_helpers.SB3Policy, built without icrl_b200."""
    th.manual_seed(5)
    ours = list(skeleton(D, A, disc, arch).named_parameters())
    th.manual_seed(5)
    theirs = list(sh.SB3Policy(D, A, disc, sh.net_arch(arch)).named_parameters())
    assert [(n, tuple(p.shape)) for n, p in ours] == [(n, tuple(p.shape)) for n, p in theirs]
    for (n, a), (_, b) in zip(ours, theirs):
        assert th.equal(a, b), n


def _refused(lib, cfg, what):
    assert lib.icrl_ppo_param_count(C.byref(cfg)) == -1
    msg = lib.icrl_last_error().decode()
    assert what in msg, msg
    assert lib.icrl_policy_forward(C.byref(cfg), None, None, 4, None, None, None, None) == -1
    assert lib.icrl_ppo_train(C.byref(cfg), None, None, None, None, 0, None, None, None) == -1
    assert lib.icrl_launch_count() == 0


@pytest.mark.parametrize("n_shared", [3, -1])
def test_bad_n_shared_is_refused_without_gpu(lib, n_shared):
    cfg = cfg_for(18, 6, False, ((64,), (64, 32, 16)))
    cfg.n_shared = n_shared
    _refused(lib, cfg, f"n_shared = {n_shared}")


@pytest.mark.parametrize("n_shared,trunks,what", [
    (1, ((64, 64), (32, 32), (64, 16)), "equal h0 in every trunk (pi 64, vf 32, cvf 64)"),
    (2, ((64, 64), (64, 64), (64, 16)), "equal h1 in every trunk (pi 64, vf 64, cvf 16)"),
    (2, ((20, 20), (16, 20), (20, 20)), "equal h0 in every trunk (pi 20, vf 16, cvf 20)"),
])
def test_unequal_shared_widths_are_refused_without_gpu(lib, n_shared, trunks, what):
    cfg = cfg_for(18, 6, False, ((64,), (64, 32, 16)))
    for t, (h0, h1) in enumerate(trunks):
        cfg.trunk_hidden[t][0], cfg.trunk_hidden[t][1] = h0, h1
    cfg.n_shared = n_shared
    _refused(lib, cfg, what)


def test_data_parallel_training_is_refused_without_gpu(lib):
    from icrl_b200 import _lib
    cfg = cfg_for(18, 6, False, ((64,), (64, 32, 16)))
    cfg.T, cfg.E, cfg.batch_size, cfg.n_epochs = 64, 4, 64, 1
    dist = _lib.PpoDist()
    dist.rank, dist.world = 0, 2
    fake = C.c_void_p(16)            # never dereferenced: the call is refused first
    for r in range(2):
        dist.recv[r] = dist.flags[r] = fake
    dist.advsums = fake
    data = _lib.PpoData()
    rc = lib.icrl_ppo_train_dist(C.byref(cfg), C.byref(data), fake, fake, fake, 0, fake, fake, C.byref(dist), None)
    assert rc == -1
    msg = lib.icrl_last_error().decode()
    assert "shared policy layers (n_shared = 1) are not supported in data-parallel training (world 2)" in msg, msg
    assert lib.icrl_launch_count() == 0


def test_n_shared_offset_matches_the_header(lib, tmp_path):
    from icrl_b200 import _lib
    probe = tmp_path / "probe.c"
    probe.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "icrl_b200.h"\n'
                     'int main(){printf("%zu %zu %zu\\n", offsetof(icrl_ppo_cfg, n_shared), '
                     'sizeof(((icrl_ppo_cfg*)0)->n_shared), sizeof(icrl_ppo_cfg));return 0;}\n')
    exe = tmp_path / "probe"
    subprocess.run(["gcc", "-I", os.path.join(ROOT, "include"), str(probe), "-o", str(exe)], check=True)
    got = [int(x) for x in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got == [_lib.PpoCfg.n_shared.offset, _lib.PpoCfg.n_shared.size, C.sizeof(_lib.PpoCfg)]
    assert _lib.PpoCfg.n_shared.offset > _lib.PpoCfg.trunk_hidden.offset     # appended: earlier fields do not move
