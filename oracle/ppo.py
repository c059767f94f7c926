"""TEST INFRASTRUCTURE (oracle) -- PPO-Lagrangian minibatch update + dual step (K4).

CPU restatement of
  /root/reference/stable_baselines3/ppo_lag/ppo_lag.py:177-338           (PPOLagrangian.train)
  /root/reference/stable_baselines3/common/policies.py:659-767           (ActorTwoCriticsPolicy)
  /root/reference/stable_baselines3/common/torch_layers.py:129-254       (MlpExtractor, separate pi/vf/cvf trunks)
  /root/reference/stable_baselines3/common/distributions.py:114-192,249-298 (DiagGaussian / Categorical)
  /root/reference/stable_baselines3/common/dual_variable.py:9-57         (Nu / DualVariable)
  /root/reference/stable_baselines3/common/buffers.py:594-627            (minibatch generator)
plus the torch library rules it leans on (Normal.log_prob/entropy, Categorical,
clip_grad_norm_, Adam) as listed in SURVEY §8(a').  Pinned against the unmodified
reference (tests/golden/ppo_*.npz).

The policy is an ordered dict name -> float32 tensor in the reference's
`parameters()` order (SURVEY §8c): [log_std], mlp_extractor.{policy,value,cost_value}_net.{0,2}.{weight,bias},
action_net, value_net, cost_value_net.  Weights are [out, in].
"""
import math
from collections import OrderedDict

import numpy as np
import torch as th
import torch.nn.functional as F

from .cn import adam_init, adam_step  # same Adam rule (torch/optim/adam.py)

TRUNKS = ("policy_net", "value_net", "cost_value_net")


def param_names(is_discrete: bool):
    names = [] if is_discrete else ["log_std"]
    for t in TRUNKS:
        for layer in (0, 2):
            names += [f"mlp_extractor.{t}.{layer}.weight", f"mlp_extractor.{t}.{layer}.bias"]
    for head in ("action_net", "value_net", "cost_value_net"):
        names += [f"{head}.weight", f"{head}.bias"]
    return names


def init_policy(obs_dim, act_dim, is_discrete, hidden=(64, 64), log_std_init=0.0, generator=None):
    """Orthogonal init with the reference's gains (policies.py:693-711): sqrt(2) trunks, 0.01 / 1 / 1 heads, zero bias."""
    P = OrderedDict()
    if not is_discrete:
        P["log_std"] = th.ones(act_dim) * log_std_init

    def ortho(out_f, in_f, gain):
        w = th.empty(out_f, in_f)
        th.nn.init.orthogonal_(w, gain=gain, generator=generator)
        return w
    for t in TRUNKS:
        last = obs_dim
        for layer, h in zip((0, 2), hidden):
            P[f"mlp_extractor.{t}.{layer}.weight"] = ortho(h, last, math.sqrt(2))
            P[f"mlp_extractor.{t}.{layer}.bias"] = th.zeros(h)
            last = h
    for head, out_f, gain in (("action_net", act_dim, 0.01), ("value_net", 1, 1.0), ("cost_value_net", 1, 1.0)):
        P[f"{head}.weight"] = ortho(out_f, hidden[-1], gain)
        P[f"{head}.bias"] = th.zeros(out_f)
    return P


def _trunk(P, name, obs):
    h = th.tanh(F.linear(obs, P[f"mlp_extractor.{name}.0.weight"], P[f"mlp_extractor.{name}.0.bias"]))
    return th.tanh(F.linear(h, P[f"mlp_extractor.{name}.2.weight"], P[f"mlp_extractor.{name}.2.bias"]))


def evaluate_actions(P, obs, actions, is_discrete):
    """policies.py:752-767 -> (values [B,1], cost_values [B,1], log_prob [B], entropy [B])."""
    latent_pi, latent_vf, latent_cvf = (_trunk(P, t, obs) for t in TRUNKS)
    head = F.linear(latent_pi, P["action_net.weight"], P["action_net.bias"])
    if is_discrete:
        # torch.distributions.Categorical(logits=...) : categorical.py:78,151-163
        logits = head - head.logsumexp(dim=-1, keepdim=True)
        probs = F.softmax(logits, dim=-1)
        log_prob = logits.gather(-1, actions.long().reshape(-1, 1)).squeeze(-1)
        entropy = -(th.clamp(logits, min=th.finfo(logits.dtype).min) * probs).sum(-1)
    else:
        # distributions.py:143-167 + torch.distributions.Normal (normal.py:87-101,114-115)
        scale = th.ones_like(head) * P["log_std"].exp()
        var = scale ** 2
        log_scale = scale.log()
        log_prob = (-((actions - head) ** 2) / (2 * var) - log_scale - math.log(math.sqrt(2 * math.pi))).sum(dim=1)
        entropy = (0.5 + 0.5 * math.log(2 * math.pi) + th.log(scale)).sum(dim=1)
    values = F.linear(latent_vf, P["value_net.weight"], P["value_net.bias"])
    cost_values = F.linear(latent_cvf, P["cost_value_net.weight"], P["cost_value_net.bias"])
    return values, cost_values, log_prob, entropy


def policy_forward_mean(P, obs, is_discrete):
    """Deterministic head output (action mean or logits) + both values -- used by rollout-side checks."""
    latent_pi, latent_vf, latent_cvf = (_trunk(P, t, obs) for t in TRUNKS)
    return (F.linear(latent_pi, P["action_net.weight"], P["action_net.bias"]),
            F.linear(latent_vf, P["value_net.weight"], P["value_net.bias"]),
            F.linear(latent_cvf, P["cost_value_net.weight"], P["cost_value_net.bias"]))


def clip_grad_norm(grads, max_norm):
    """torch/nn/utils/clip_grad.py: 2-norm of per-tensor 2-norms; coef = min(max/(tot+1e-6), 1); always multiplied."""
    total = th.linalg.vector_norm(th.stack([th.linalg.vector_norm(g, 2) for g in grads]), 2)
    coef = th.clamp(max_norm / (total + 1e-6), max=1.0)
    return [g * coef for g in grads], total


def minibatch_loss(P, mb, is_discrete, clip_range, nu, ent_coef, reward_vf_coef, cost_vf_coef,
                   clip_range_reward_vf=None, clip_range_cost_vf=None):
    """ppo_lag.py:203-281 for one minibatch `mb` (dict of fp32 tensors).  Returns (loss, stats dict)."""
    actions = mb["actions"]
    if is_discrete:
        actions = actions.long().flatten()
    rv, cv, log_prob, entropy = evaluate_actions(P, mb["observations"], actions, is_discrete)
    rv, cv = rv.flatten(), cv.flatten()
    ra = mb["reward_advantages"] - mb["reward_advantages"].mean()
    ra = ra / (mb["reward_advantages"].std() + 1e-8)              # unbiased std, :218-219
    ca = mb["cost_advantages"] - mb["cost_advantages"].mean()     # centred, NOT rescaled, :222
    ratio = th.exp(log_prob - mb["old_log_prob"])
    pl1 = ra * ratio
    pl2 = ra * th.clamp(ratio, 1 - clip_range, 1 + clip_range)
    policy_loss = -th.min(pl1, pl2).mean()
    policy_loss = policy_loss + nu * th.mean(ca * ratio)          # cost term unclipped, :234-235
    policy_loss = policy_loss / (1 + nu)
    clip_fraction = th.mean((th.abs(ratio - 1) > clip_range).float()).item()
    rv_pred = rv if clip_range_reward_vf is None else mb["old_reward_values"] + th.clamp(
        rv - mb["old_reward_values"], -clip_range_reward_vf, clip_range_reward_vf)
    cv_pred = cv if clip_range_cost_vf is None else mb["old_cost_values"] + th.clamp(
        cv - mb["old_cost_values"], -clip_range_cost_vf, clip_range_cost_vf)
    rv_loss = F.mse_loss(mb["reward_returns"], rv_pred)
    cv_loss = F.mse_loss(mb["cost_returns"], cv_pred)
    entropy_loss = -th.mean(entropy)
    loss = policy_loss + ent_coef * entropy_loss + reward_vf_coef * rv_loss + cost_vf_coef * cv_loss
    stats = {"pg_loss": policy_loss.item(), "clip_fraction": clip_fraction, "reward_value_loss": rv_loss.item(),
             "cost_value_loss": cv_loss.item(), "entropy_loss": entropy_loss.item(), "loss": loss.item(),
             "approx_kl": float(th.mean(mb["old_log_prob"] - log_prob).detach().numpy())}
    return loss, stats


FLAT_FIELDS = ("observations", "actions", "old_log_prob", "old_reward_values", "reward_advantages", "reward_returns",
               "old_cost_values", "cost_advantages", "cost_returns")


def train(P, adam_state, flat, perms, *, is_discrete, batch_size, n_epochs, lr, clip_range, nu,
          ent_coef=0.0, reward_vf_coef=0.5, cost_vf_coef=0.5, max_grad_norm=0.5, target_kl=None,
          clip_range_reward_vf=None, clip_range_cost_vf=None, adam_eps=1e-5, max_steps=None):
    """The epoch/minibatch loop of ppo_lag.py:198-297.

    `flat`: dict of env-major flattened float32 numpy arrays (FLAT_FIELDS; what RolloutBufferWithCost.get
    holds after swap_and_flatten, buffers.py:598-603).  `perms[e]`: the permutation the reference would draw
    for epoch e (np.random.permutation, buffers.py:596) -- generated by the caller so both sides share it.
    Updates P / adam_state in place.  Returns dict with per-step stat lists and early_stop_epoch.
    `max_steps` (bench only) stops after that many optimiser steps.
    """
    names = list(P.keys())
    params = [P[n] for n in names]
    for p in params:
        p.requires_grad_(True)
    n = flat["observations"].shape[0]
    bs = n if batch_size is None else batch_size
    per_step = {k: [] for k in ("pg_loss", "clip_fraction", "reward_value_loss", "cost_value_loss", "entropy_loss",
                                "loss", "approx_kl", "grad_norm")}      # grad_norm: clip_grad_norm_'s pre-clip total norm
    all_kl, early_stop_epoch, steps = [], n_epochs, 0
    done = False
    for epoch in range(n_epochs):
        kls = []
        idx_all = perms[epoch]
        for start in range(0, n, bs):
            idx = idx_all[start:start + bs]
            mb = {k: th.tensor(flat[k][idx]) for k in FLAT_FIELDS}
            for k in FLAT_FIELDS[2:]:
                mb[k] = mb[k].flatten()
            loss, st = minibatch_loss(P, mb, is_discrete, clip_range, nu, ent_coef, reward_vf_coef, cost_vf_coef,
                                      clip_range_reward_vf, clip_range_cost_vf)
            grads = th.autograd.grad(loss, params, allow_unused=True)
            grads = [th.zeros_like(p) if g is None else g for p, g in zip(params, grads)]
            grads, total = clip_grad_norm(grads, max_grad_norm)
            adam_step(params, grads, adam_state, lr, eps=adam_eps)
            for k in st:
                per_step[k].append(st[k])
            per_step["grad_norm"].append(float(total))
            kls.append(st["approx_kl"])
            steps += 1
            if max_steps is not None and steps >= max_steps:
                done = True
                break
        all_kl.append(np.mean(kls))
        if done:
            break
        if target_kl is not None and np.mean(kls) > 1.5 * target_kl:
            early_stop_epoch = epoch
            break
    for p in params:
        p.requires_grad_(False)
    return {"per_step": per_step, "epoch_kl": all_kl, "early_stop_epoch": early_stop_epoch,
            "last_epoch_approx_kl": float(np.mean(kls)), "steps": steps}


# ---------------------------------------------------------------- dual variable (dual_variable.py:9-57)

def dual_init(penalty_init=1.0, clamp_at=None):
    """Nu.__init__: log_nu = log(max(e^p0 - 1, 1e-8)); clamp_at defaults to the *transformed* init (:19-21)."""
    t = np.log(max(np.exp(penalty_init) - 1, 1e-8))
    log_nu = t * th.ones(1)
    return {"log_nu": log_nu, "clamp_at": t if clamp_at is None else clamp_at, "adam": adam_init([log_nu])}


def dual_nu(state):
    return F.softplus(state["log_nu"])


def dual_step(state, cost, alpha, lr):
    """DualVariable.update_parameter (:47-57): loss = -nu*(cost-alpha); Adam(eps=1e-8) step on log_nu; clamp."""
    log_nu = state["log_nu"].requires_grad_(True)
    loss = -F.softplus(log_nu) * (cost - alpha)
    (g,) = th.autograd.grad(loss.sum(), [log_nu])
    log_nu.requires_grad_(False)
    adam_step([log_nu], [g], state["adam"], lr, eps=1e-8)
    log_nu.clamp_(min=np.log(max(np.exp(state["clamp_at"]) - 1, 1e-8)))
    return loss.detach()
