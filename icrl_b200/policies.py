"""ActorTwoCriticsPolicy -- host-side mirror of stable_baselines3/common/policies.py:598-779 (MlpPolicy flavour:
FlattenExtractor, three tanh MLP trunks pi/vf/cvf of two layers each, the first or both of them optionally shared
(MlpExtractor.shared_net), DiagGaussian or Categorical head).

Parameters and Adam moments live in flat float32 device tensors in the reference's `parameters()` order; the CUDA
kernels (K4 train step, policy forward) read and update them in place.  A CPU `nn.Module` skeleton with the
reference's exact module/attribute names is kept only to (i) consume the torch RNG in the reference's order at
initialisation, so seeds give identical initial weights, and (ii) import/export `policy.pth`-compatible state_dicts.
"""
import ctypes as C
import math
from functools import partial
from itertools import zip_longest
from typing import Any, Callable, Dict, List, Optional, Tuple

import numpy as np
import torch as th
from torch import nn

from . import _lib
from .constraint_net import _FlatAdam
from .device import resolve_device
from .spaces import is_discrete as _is_discrete


class _MlpExtractorShape(nn.Module):
    """Module skeleton with torch_layers.py:129-254's creation order (shared layers, then pi, vf, cvf layers interleaved)
    and names; a trunk without private layers takes the last shared width as its latent dimension."""

    def __init__(self, feature_dim, shared, pi, vf, cvf, activation_fn):
        super().__init__()
        shared_net, last_shared = [], feature_dim
        for size in shared:
            shared_net += [nn.Linear(last_shared, size), activation_fn()]
            last_shared = size
        nets = {"policy_net": [], "value_net": [], "cost_value_net": []}
        last = {k: last_shared for k in nets}
        for sizes in zip_longest(pi, vf, cvf):
            for key, size in zip(nets, sizes):
                if size is not None:
                    nets[key] += [nn.Linear(last[key], size), activation_fn()]
                    last[key] = size
        self.latent_dim_pi, self.latent_dim_vf, self.latent_dim_cvf = (last[k] for k in nets)
        self.shared_net = nn.Sequential(*shared_net)
        self.policy_net = nn.Sequential(*nets["policy_net"])
        self.value_net = nn.Sequential(*nets["value_net"])
        self.cost_value_net = nn.Sequential(*nets["cost_value_net"])


class _PolicyShape(nn.Module):
    def __init__(self, obs_dim, act_out, discrete, pi, vf, cvf, activation_fn, log_std_init, ortho_init, shared=()):
        super().__init__()
        self.features_extractor = nn.Flatten()
        self.mlp_extractor = _MlpExtractorShape(obs_dim, shared, pi, vf, cvf, activation_fn)
        self.action_net = nn.Linear(self.mlp_extractor.latent_dim_pi, act_out)
        if not discrete:
            self.log_std = nn.Parameter(th.ones(act_out) * log_std_init, requires_grad=True)
        self.value_net = nn.Linear(self.mlp_extractor.latent_dim_vf, 1)
        self.cost_value_net = nn.Linear(self.mlp_extractor.latent_dim_cvf, 1)
        if ortho_init:                                                     # policies.py:693-711
            gains = [(self.features_extractor, np.sqrt(2)), (self.mlp_extractor, np.sqrt(2)), (self.action_net, 0.01),
                     (self.value_net, 1), (self.cost_value_net, 1)]
            for module, gain in gains:
                module.apply(partial(self._init_weights, gain=gain))

    @staticmethod
    def _init_weights(module, gain=1):
        if isinstance(module, (nn.Linear, nn.Conv2d)):
            nn.init.orthogonal_(module.weight, gain=gain)
            module.bias.data.fill_(0.0)


def _trunks(net_arch):
    """net_arch -> (shared widths, pi, vf, cvf private widths, effective (h0, h1) of pi, vf, cvf).  The kernels train two
    tanh layers of width 1..64 under every head: separate trunks [dict(pi=[a, b], vf=[c, d], cvf=[e, f])], one shared
    layer [s, dict(pi=[p], vf=[v], cvf=[c])], or one shared trunk [s0, s1] (a dict there may only hold empty lists)."""
    shared = []
    for layer in net_arch:
        if isinstance(layer, dict):
            break
        shared.append(layer)
    rest = net_arch[len(shared):]
    if len(rest) > 1 or (not shared and len(rest) != 1):
        raise NotImplementedError(f"net_arch {net_arch}: expected shared layer widths followed by at most one dict of "
                                  "pi / vf / cvf layers")
    pi, vf, cvf = (list(rest[0].get(k, [])) if rest else [] for k in ("pi", "vf", "cvf"))
    if not shared:
        for key, sizes in zip(("pi", "vf", "cvf"), (pi, vf, cvf)):
            if len(sizes) != 2 or not all(1 <= int(h) <= 64 for h in sizes):
                raise NotImplementedError(f"net_arch {net_arch}: the {key} trunk {sizes} is not supported; the kernels "
                                          "support two-layer pi / vf / cvf trunks of widths 1..64 each (the reference "
                                          "default is [64, 64])")
        return [], pi, vf, cvf, tuple((int(t[0]), int(t[1])) for t in (pi, vf, cvf))
    if len(shared) > 2 or not all(isinstance(h, int) and 1 <= h <= 64 for h in shared):
        raise NotImplementedError(f"net_arch {net_arch}: the shared layers {shared} are not supported; the kernels "
                                  "support one or two shared layers of widths 1..64")
    for key, sizes in zip(("pi", "vf", "cvf"), (pi, vf, cvf)):
        if len(shared) + len(sizes) != 2 or not all(1 <= int(h) <= 64 for h in sizes):
            raise NotImplementedError(f"net_arch {net_arch}: the {key} trunk, shared {shared} + private {sizes}, is not "
                                      "supported; the kernels support two tanh layers of widths 1..64 under every head "
                                      "(-sl s -pl p -rvl v -cvl c, or -sl s0 s1 with no private layers)")
    effective = tuple((int(shared[0]), int(([*shared[1:], *sizes])[0])) for sizes in (pi, vf, cvf))
    return [int(h) for h in shared], pi, vf, cvf, effective


class ActorTwoCriticsPolicy:
    def __init__(self, observation_space, action_space, lr_schedule: Callable[[float], float],
                 net_arch: Optional[List] = None, activation_fn=nn.Tanh, ortho_init: bool = True, use_sde: bool = False,
                 log_std_init: float = 0.0, full_std: bool = True, sde_net_arch=None, use_expln: bool = False,
                 squash_output: bool = False, features_extractor_class=None, features_extractor_kwargs=None,
                 normalize_images: bool = True, optimizer_class=th.optim.Adam,
                 optimizer_kwargs: Optional[Dict[str, Any]] = None, device="cuda"):
        if use_sde or sde_net_arch is not None or squash_output:
            raise NotImplementedError("gSDE / squashed outputs are not used by the ICRL configs and not implemented")
        if activation_fn is not nn.Tanh:
            raise NotImplementedError("the PPO-Lagrangian kernels implement the reference's Tanh policies only")
        if optimizer_class is not th.optim.Adam:
            raise NotImplementedError("icrl_b200 implements the reference's optimiser (Adam) only")
        if net_arch is None:
            net_arch = [dict(pi=[64, 64], vf=[64, 64], cvf=[64, 64])]
        shared, pi, vf, cvf, trunk_hidden = _trunks(net_arch)
        self.observation_space, self.action_space = observation_space, action_space
        self.net_arch, self.activation_fn, self.ortho_init = net_arch, activation_fn, ortho_init
        self.is_discrete = _is_discrete(action_space)
        self.obs_dim = int(np.prod(observation_space.shape)) if not _is_discrete(observation_space) else 1
        self.act_out = int(action_space.n) if self.is_discrete else int(np.prod(action_space.shape))
        if self.act_out > 16:
            raise NotImplementedError("more than 16 action dimensions")
        self.trunk_hidden = trunk_hidden      # effective {h0, h1} of pi, vf, cvf (shared layers included)
        self.n_shared = len(shared)           # leading layers the three trunks share
        self.log_std_init = log_std_init
        if optimizer_kwargs is None:
            optimizer_kwargs = {"eps": 1e-5}                               # policies.py:357-361
        self.optimizer_class, self.optimizer_kwargs = optimizer_class, optimizer_kwargs
        self.device = resolve_device(device)
        self._shape = _PolicyShape(self.obs_dim, self.act_out, self.is_discrete, pi, vf, cvf, activation_fn,
                                   log_std_init, ortho_init, shared)
        self._slices, off = [], 0
        for _, p in self._shape.named_parameters():
            self._slices.append((off, tuple(p.shape)))
            off += p.numel()
        self.n_params = off
        self._params = th.cat([p.detach().reshape(-1) for p in self._shape.parameters()]).to(self.device)
        self._adam_m = th.zeros_like(self._params)
        self._adam_v = th.zeros_like(self._params)
        self.optimizer = _FlatAdam(self, lr=lr_schedule(1), **optimizer_kwargs)
        cfg = self.make_cfg()
        assert _lib.lib().icrl_ppo_param_count(C.byref(cfg)) == self.n_params, "flat parameter layout mismatch"

    # ---------------------------------------------------------------- parameter plumbing
    def _param_slices(self):
        return self._slices

    def parameter_names(self):
        return [n for n, _ in self._shape.named_parameters()]

    def state_dict(self):
        flat = self._params.detach().cpu()
        with th.no_grad():
            for p, (off, shape) in zip(self._shape.parameters(), self._slices):
                p.copy_(flat[off:off + p.numel()].reshape(shape))
        return self._shape.state_dict()

    def load_state_dict(self, sd, strict=True):
        self._shape.load_state_dict(sd, strict=strict)
        self._params.copy_(th.cat([p.detach().reshape(-1) for p in self._shape.parameters()]))

    def parameters_flat(self) -> th.Tensor:
        return self._params

    @property
    def log_std(self) -> th.Tensor:
        if self.is_discrete:
            raise AttributeError("log_std")
        return self._params[:self.act_out]

    def make_cfg(self, **kw) -> _lib.PpoCfg:
        cfg = _lib.PpoCfg()
        cfg.obs_dim, cfg.act_dim, cfg.is_discrete = self.obs_dim, self.act_out, int(self.is_discrete)
        for t, (h0, h1) in enumerate(self.trunk_hidden):
            cfg.trunk_hidden[t][0], cfg.trunk_hidden[t][1] = h0, h1
        cfg.n_shared = self.n_shared
        cfg.T = cfg.E = 1
        cfg.batch_size = cfg.n_epochs = 1
        g = getattr(self, "optimizer", None)
        if g is not None:
            g = g.param_groups[0]
            cfg.lr, cfg.adam_beta1, cfg.adam_beta2, cfg.adam_eps = g["lr"], g["betas"][0], g["betas"][1], g["eps"]
        for k, v in kw.items():
            setattr(cfg, k, v)
        return cfg

    # ---------------------------------------------------------------- forward passes
    def forward_heads(self, obs: th.Tensor) -> Tuple[th.Tensor, th.Tensor, th.Tensor]:
        """(action mean or logits [n, act_out], reward values [n], cost values [n]) on the device."""
        obs = obs.to(self.device, th.float32).reshape(-1, self.obs_dim).contiguous()
        n = obs.shape[0]
        head = th.empty(n, self.act_out, device=self.device)
        values, cost_values = th.empty(n, device=self.device), th.empty(n, device=self.device)
        cfg = self.make_cfg()
        with th.cuda.device(self.device):
            _lib.check(_lib.lib().icrl_policy_forward(C.byref(cfg), _lib.ptr(self._params), _lib.ptr(obs), n,
                                                      _lib.ptr(head), _lib.ptr(values), _lib.ptr(cost_values),
                                                      _lib.current_stream()))
        return head, values, cost_values

    def _dist_terms(self, head: th.Tensor, actions: th.Tensor, log_std: Optional[th.Tensor] = None):
        """log_prob / entropy with torch.distributions' formulas (distributions.py:143-167, 274-282)."""
        if self.is_discrete:
            logits = head - head.logsumexp(dim=-1, keepdim=True)
            log_prob = logits.gather(-1, actions.long().reshape(-1, 1)).squeeze(-1)
            entropy = -(th.clamp(logits, min=th.finfo(logits.dtype).min) * logits.exp()).sum(-1)
        else:
            scale = th.ones_like(head) * (self.log_std if log_std is None else log_std).to(head.device).exp()
            log_scale = scale.log()
            log_prob = (-((actions - head) ** 2) / (2 * scale ** 2) - log_scale - math.log(math.sqrt(2 * math.pi))).sum(1)
            entropy = (0.5 + 0.5 * math.log(2 * math.pi) + log_scale).sum(1)
        return log_prob, entropy

    def _forward_heads_small(self, obs: th.Tensor):
        """Rollout-time call ([n_envs, obs_dim] host rows, once per environment step): the kernel reads the rows from, and
        writes heads / values to, one host-mapped pinned block (UVA), log_std rides along as a 4*A-byte async copy: one launch
        and ONE synchronisation instead of an upload, three allocations and four blocking downloads.  Returns host tensors."""
        n, D, A = obs.shape[0], self.obs_dim, self.act_out
        need = n * (D + A + 2) + A
        blk = getattr(self, "_pin_block", None)
        if blk is None or blk.numel() < need:
            blk = self._pin_block = th.empty(max(need, 1024), dtype=th.float32).pin_memory()
        o, off = blk[:n * D].view(n, D), n * D
        head, off = blk[off:off + n * A].view(n, A), off + n * A
        values, off = blk[off:off + n], off + n
        cost_values, off = blk[off:off + n], off + n
        log_std = blk[off:off + A]
        o.copy_(obs)
        cfg = getattr(self, "_fwd_cfg", None)          # (the forward reads the shape fields only: built once, ~15 us per make_cfg)
        if cfg is None:
            cfg = self._fwd_cfg = self.make_cfg()

        def launch():
            stream = th.cuda.current_stream()
            _lib.check(_lib.lib().icrl_policy_forward(C.byref(cfg), _lib.ptr(self._params), _lib.ptr(o), n, _lib.ptr(head),
                                                      _lib.ptr(values), _lib.ptr(cost_values), C.c_void_p(stream.cuda_stream)))
            if not self.is_discrete:
                log_std.copy_(self._params[:A], non_blocking=True)
            stream.synchronize()

        if th.cuda.current_device() == self.device.index:
            launch()
        else:
            with th.cuda.device(self.device):
                launch()
        out = blk[n * D:n * (D + A + 2) + A].clone()    # one copy out of the staging block
        head = out[:n * A].view(n, A)
        return head, out[n * A:n * A + n], out[n * A + n:n * A + 2 * n], out[n * A + 2 * n:]

    def forward(self, obs: th.Tensor, deterministic: bool = False):
        """policies.py:716-731: actions, values, cost_values, log_prob.  Heads come from the CUDA forward; sampling uses
        the host torch generator exactly like the reference's CPU `Normal.rsample` / `Categorical.sample`, so a
        given torch seed produces the same exploration noise."""
        obs = th.as_tensor(obs)
        if not obs.is_cuda and obs.numel() <= 64 * self.obs_dim:
            obs = obs.to(th.float32).reshape(-1, self.obs_dim)
            head, values, cost_values, log_std = self._forward_heads_small(obs)
        else:
            head, values, cost_values = self.forward_heads(obs)
            head, values, cost_values = head.cpu(), values.cpu(), cost_values.cpu()
            log_std = None if self.is_discrete else self.log_std.cpu()
        if self.is_discrete:
            probs = th.softmax(head, dim=-1)
            actions = th.argmax(probs, dim=1) if deterministic else th.multinomial(probs, 1).squeeze(-1)
            log_prob, _ = self._dist_terms(head, actions, log_std)
        else:
            # the terms that depend on log_std only change with train(): cached per (log_std bytes, batch shape); the per-step
            # expression below is the reference's, operation for operation (distributions.py:143-167 -> Normal.log_prob)
            c = getattr(self, "_gauss_cache", None)
            if c is None or c[1].shape != head.shape or not th.equal(c[0], log_std):
                scale = th.ones_like(head) * log_std.exp()
                c = self._gauss_cache = (log_std.clone(), scale, scale.log(), 2 * scale ** 2)
            _, std, log_scale, two_var = c
            actions = head if deterministic else head + std * th.empty_like(head).normal_()
            log_prob = (-((actions - head) ** 2) / two_var - log_scale - math.log(math.sqrt(2 * math.pi))).sum(1)
        return actions, values.reshape(-1, 1), cost_values.reshape(-1, 1), log_prob

    __call__ = forward

    def evaluate_actions(self, obs: th.Tensor, actions: th.Tensor):
        """policies.py:752-767 (no autograd: gradients exist only inside the fused K4 kernel)."""
        head, values, cost_values = self.forward_heads(th.as_tensor(obs))
        log_prob, entropy = self._dist_terms(head, th.as_tensor(actions).to(self.device))
        return values.reshape(-1, 1), cost_values.reshape(-1, 1), log_prob, entropy

    def predict(self, observation, state=None, mask=None, deterministic: bool = False):
        obs = np.asarray(observation, dtype=np.float32).reshape(-1, self.obs_dim)
        actions = self.forward(th.as_tensor(obs), deterministic)[0].numpy()
        if not self.is_discrete:
            actions = np.clip(actions, self.action_space.low, self.action_space.high)
        return actions, state
