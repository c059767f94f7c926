"""CPU: the environment limit of icrl_cost_normalize (K5).  The batch moments use numpy's pairwise summation, recursed to
a depth fixed at compile time; every E the host accepts must fit that depth, and the first E beyond the limit is refused
before any CUDA call, with a message naming the limit."""
import os
import re

import numpy as np
import pytest

from conftest import ROOT

K5_SRC = os.path.join(ROOT, "icrl_b200", "csrc", "k5_cost_norm.cu")


@pytest.fixture(scope="module")
def lib():
    from icrl_b200 import build, _lib
    build.build()
    return _lib.lib()


def refusal(lib, E):
    """The error of a call with E environments, which the argument checks must refuse (the pointers are host arrays)."""
    dummy = np.zeros(4, np.float64)
    p = dummy.ctypes.data
    rc = lib.icrl_cost_normalize(p, p, p, 3, E, 0.99, 1e-8, 10.0, 1, 1, p, p, None)
    assert rc != 0
    return lib.icrl_last_error().decode()


def env_limit(lib):
    m = re.search(r"at most (\d+) environments", refusal(lib, 2 ** 31 - 1))
    assert m, "the refusal names the limit"
    return int(m.group(1))


def test_first_refused_env_count_names_the_limit(lib):
    limit = env_limit(lib)
    assert limit == 524288
    launches = lib.icrl_launch_count()
    msg = refusal(lib, limit + 1)
    assert f"at most {limit} environments (got {limit + 1})" in msg, msg
    assert lib.icrl_launch_count() == launches


def test_pairwise_depth_covers_every_accepted_env_count(lib):
    """Replays numpy's split (n2 = n / 2 rounded down to a multiple of 8; blocks of at most 128 are summed directly)
    for every E up to the limit and checks that none needs more levels than np_pairwise_sum<kPwDepth> has."""
    limit = env_limit(lib)
    depth_limit = int(re.search(r"constexpr int kPwDepth = (\d+);", open(K5_SRC).read()).group(1))
    depth = np.zeros(limit + 1, np.int64)
    n = np.arange(129, limit + 1)
    n2 = n // 2 - (n // 2) % 8
    # children are smaller than their parent, so one pass in increasing n fills the table
    for lo in range(129, limit + 1, 64):
        hi = min(lo + 64, limit + 1)
        i = slice(lo - 129, hi - 129)
        depth[lo:hi] = 1 + np.maximum(depth[n2[i]], depth[n[i] - n2[i]])
    assert depth.max() <= depth_limit, (int(depth.max()), int(np.argmax(depth > depth_limit)))
    # 12 levels would not do: the first E that needs 13 is accepted
    assert depth[491529] == 13 and depth[:491529].max() == 12
