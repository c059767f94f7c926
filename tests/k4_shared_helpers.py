"""Policies with shared trunk layers (MlpExtractor.shared_net, the reference's -sl) for the K4 tests: the oracle's trunk
with shared layers, the shared parameter layout, the reference's initialisation, and the separate-trunk net that holds
three copies of the shared layers.

An architecture is (shared widths, private widths of pi, vf, cvf): ((s,), (p, v, c)) is net_arch
[s, dict(pi=[p], vf=[v], cvf=[c])] and ((s0, s1), ()) is [s0, s1]."""
import math
from collections import OrderedDict
from itertools import zip_longest

import torch as th
import torch.nn.functional as F
from torch import nn

from oracle import ppo as oppo

HEADS = ("action_net", "value_net", "cost_value_net")
_SEPARATE_TRUNK = oppo._trunk


def net_arch(arch):
    shared, private = arch
    if not private:
        return list(shared)
    return [*shared, dict(zip(("pi", "vf", "cvf"), ([h] for h in private)))]


def trunk_hidden(arch):
    """Effective (h0, h1) of pi, vf and cvf."""
    shared, private = arch
    return tuple((shared[0], shared[1] if len(shared) == 2 else private[t]) for t in range(3))


def param_names(is_discrete, arch):
    """The reference's parameters() order with shared layers: [log_std], shared_net.{0,2}, the private layer of each
    trunk, the heads."""
    shared, private = arch
    names = [] if is_discrete else ["log_std"]
    for layer in range(len(shared)):
        names += [f"mlp_extractor.shared_net.{2 * layer}.weight", f"mlp_extractor.shared_net.{2 * layer}.bias"]
    if private:
        for t in oppo.TRUNKS:
            names += [f"mlp_extractor.{t}.0.weight", f"mlp_extractor.{t}.0.bias"]
    for head in HEADS:
        names += [f"{head}.weight", f"{head}.bias"]
    return names


def trunk(P, name, obs):
    """oracle.ppo._trunk for either layout: shared_net.{0,2}, then the private layers that exist."""
    if "mlp_extractor.shared_net.0.weight" not in P:
        return _SEPARATE_TRUNK(P, name, obs)
    h = obs
    for key in ("mlp_extractor.shared_net.0", "mlp_extractor.shared_net.2", f"mlp_extractor.{name}.0"):
        if f"{key}.weight" in P:
            h = th.tanh(F.linear(h, P[f"{key}.weight"], P[f"{key}.bias"]))
    return h


def init_policy(obs_dim, act_dim, is_discrete, arch, log_std_init=0.0, generator=None):
    """Orthogonal init with the reference's gains (policies.py:693-711): sqrt(2) for every trunk layer, shared or not,
    0.01 / 1 / 1 for the heads, zero biases."""
    shared, private = arch

    def ortho(out_f, in_f, gain):
        w = th.empty(out_f, in_f)
        th.nn.init.orthogonal_(w, gain=gain, generator=generator)
        return w
    P = OrderedDict()
    if not is_discrete:
        P["log_std"] = th.ones(act_dim) * log_std_init
    last = obs_dim
    for layer, h in enumerate(shared):
        P[f"mlp_extractor.shared_net.{2 * layer}.weight"] = ortho(h, last, math.sqrt(2))
        P[f"mlp_extractor.shared_net.{2 * layer}.bias"] = th.zeros(h)
        last = h
    latent = [last] * 3
    if private:
        for t, name in enumerate(oppo.TRUNKS):
            P[f"mlp_extractor.{name}.0.weight"] = ortho(private[t], last, math.sqrt(2))
            P[f"mlp_extractor.{name}.0.bias"] = th.zeros(private[t])
            latent[t] = private[t]
    for (head, out_f, gain), k in zip(((HEADS[0], act_dim, 0.01), (HEADS[1], 1, 1.0), (HEADS[2], 1, 1.0)), latent):
        P[f"{head}.weight"] = ortho(out_f, k, gain)
        P[f"{head}.bias"] = th.zeros(out_f)
    return P


def separate(P, is_discrete, arch):
    """The same function as separate pi / vf / cvf trunks (oracle.ppo's layout): every trunk holds a copy of the shared
    layers."""
    shared, private = arch
    out = OrderedDict()
    for n in oppo.param_names(is_discrete):
        if not n.startswith("mlp_extractor."):
            out[n] = P[n].clone()
            continue
        _, t, layer, kind = n.split(".")
        if layer == "0":
            src = f"mlp_extractor.shared_net.0.{kind}"
        else:
            src = f"mlp_extractor.shared_net.2.{kind}" if len(shared) == 2 else f"mlp_extractor.{t}.0.{kind}"
        out[n] = P[src].clone()
    return out


class SB3MlpExtractor(nn.Module):
    """MlpExtractor's structure (torch_layers.py:129-254), written independently of icrl_b200.policies: integers of
    net_arch are shared layers, created first; a dict after them gives the private pi / vf / cvf layers."""

    def __init__(self, feature_dim, net_arch, activation_fn=nn.Tanh):
        super().__init__()
        shared_net, policy_net, value_net, cost_value_net = [], [], [], []
        policy_only, value_only, cost_only = [], [], []
        last_shared = feature_dim
        for layer in net_arch:
            if isinstance(layer, int):
                shared_net += [nn.Linear(last_shared, layer), activation_fn()]
                last_shared = layer
            else:
                policy_only, value_only, cost_only = layer.get("pi", []), layer.get("vf", []), layer.get("cvf", [])
                break
        last_pi = last_vf = last_cvf = last_shared
        for pi_size, vf_size, cvf_size in zip_longest(policy_only, value_only, cost_only):
            if pi_size is not None:
                policy_net += [nn.Linear(last_pi, pi_size), activation_fn()]
                last_pi = pi_size
            if vf_size is not None:
                value_net += [nn.Linear(last_vf, vf_size), activation_fn()]
                last_vf = vf_size
            if cvf_size is not None:
                cost_value_net += [nn.Linear(last_cvf, cvf_size), activation_fn()]
                last_cvf = cvf_size
        self.latent_dim_pi, self.latent_dim_vf, self.latent_dim_cvf = last_pi, last_vf, last_cvf
        self.shared_net = nn.Sequential(*shared_net)
        self.policy_net = nn.Sequential(*policy_net)
        self.value_net = nn.Sequential(*value_net)
        self.cost_value_net = nn.Sequential(*cost_value_net)


class SB3Policy(nn.Module):
    """ActorTwoCriticsPolicy's modules in the reference's build order (policies.py:659-711): extractor, action_net and
    log_std, value_net, cost_value_net, then orthogonal init with gains sqrt(2) / 0.01 / 1 / 1 and zero biases."""

    def __init__(self, obs_dim, act_out, is_discrete, net_arch, log_std_init=0.0):
        super().__init__()
        self.features_extractor = nn.Flatten()
        self.mlp_extractor = SB3MlpExtractor(obs_dim, net_arch)
        self.action_net = nn.Linear(self.mlp_extractor.latent_dim_pi, act_out)
        if not is_discrete:
            self.log_std = nn.Parameter(th.ones(act_out) * log_std_init)
        self.value_net = nn.Linear(self.mlp_extractor.latent_dim_vf, 1)
        self.cost_value_net = nn.Linear(self.mlp_extractor.latent_dim_cvf, 1)
        for module, gain in ((self.features_extractor, math.sqrt(2)), (self.mlp_extractor, math.sqrt(2)),
                             (self.action_net, 0.01), (self.value_net, 1.0), (self.cost_value_net, 1.0)):
            module.apply(lambda m, gain=gain: self._ortho(m, gain))

    @staticmethod
    def _ortho(module, gain):
        if isinstance(module, nn.Linear):
            nn.init.orthogonal_(module.weight, gain=gain)
            module.bias.data.fill_(0.0)
