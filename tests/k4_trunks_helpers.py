"""Policies with per-trunk widths for the K4 tests, built from oracle.ppo's uniform-width initialisation."""
from collections import OrderedDict

import torch as th

from oracle import ppo as oppo

HEADS = ("action_net", "value_net", "cost_value_net")


def init_policy_trunks(obs_dim, act_dim, is_discrete, trunks, generator=None):
    """oracle.ppo.init_policy with one (h0, h1) pair per trunk (pi, vf, cvf): each trunk and its head come from a uniform
    net of that trunk's widths (the reference's gains, zero biases), in the reference's parameter order."""
    parts = [oppo.init_policy(obs_dim, act_dim, is_discrete, tuple(h), generator=generator) for h in trunks]
    P = OrderedDict()
    for n in oppo.param_names(is_discrete):
        if n == "log_std":
            t = 0
        elif n.startswith("mlp_extractor."):
            t = oppo.TRUNKS.index(n.split(".")[1])
        else:
            t = HEADS.index(n.split(".")[0])
        P[n] = parts[t][n]
    return P


def embed(P, obs_dim, act_dim, is_discrete):
    """Per-trunk tensors -> a uniform 64-64 net, zeros in the extra rows and columns."""
    U = oppo.init_policy(obs_dim, act_dim, is_discrete, (64, 64), generator=th.Generator().manual_seed(0))
    out = OrderedDict()
    for n, p in P.items():
        z = th.zeros_like(U[n])
        z[tuple(slice(0, s) for s in p.shape)] = p
        out[n] = z
    return out
