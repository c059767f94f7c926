"""TEST INFRASTRUCTURE (oracle) -- constraint net: K1 (cost forward) and K2 (IS-weighted train).

CPU restatement of /root/reference/icrl/constraint_net.py.  Parity pinned against the
unmodified reference run in the build container (tests/golden/cn_*.npz); the
reference itself has no tests for this path.

Parameters are a flat python list [W0, b0, W1, b1, ..., WL, bL] of float32 torch
tensors, W_i of shape [out, in] (== `network.{0,2,4}.{weight,bias}` in the
reference's state_dict, constraint_net.py:104-107 + torch_layers.py:93-126).
"""
from dataclasses import dataclass, field
from itertools import accumulate
from typing import List, Optional, Sequence

import numpy as np
import torch as th


@dataclass
class CNSpec:
    """The subset of ConstraintNet.__init__ state (constraint_net.py:15-85) that the arithmetic reads."""
    obs_dim: int
    acs_dim: int
    hidden_sizes: Sequence[int]
    is_discrete: bool
    obs_select_dim: Optional[Sequence[int]] = None
    acs_select_dim: Optional[Sequence[int]] = None
    clip_obs: Optional[float] = 10.0
    obs_mean: Optional[np.ndarray] = None
    obs_var: Optional[np.ndarray] = None
    action_low: Optional[np.ndarray] = None
    action_high: Optional[np.ndarray] = None
    eps: float = 1e-5
    regularizer_coeff: float = 0.0
    importance_sampling: bool = True
    per_step_importance_sampling: bool = False
    target_kl_old_new: float = -1
    target_kl_new_old: float = -1
    train_gail_lambda: bool = False
    select_dim: List[int] = field(default_factory=list)

    def __post_init__(self):
        self.select_dim = define_select_dim(self.obs_dim, self.acs_dim, self.obs_select_dim, self.acs_select_dim)

    @property
    def input_dims(self):
        return len(self.select_dim)


def define_select_dim(obs_dim, acs_dim, obs_select_dim, acs_select_dim):
    """constraint_net.py:87-99.  NB: acs_select_dim indices are NOT offset by obs_dim (a1 in SURVEY §8)."""
    sel = []
    if obs_select_dim is None:
        sel += list(range(obs_dim))
    elif obs_select_dim[0] != -1:
        sel += list(obs_select_dim)
    if acs_select_dim is None:
        sel += list(range(acs_dim))
    elif acs_select_dim[0] != -1:
        sel += list(acs_select_dim)
    assert len(sel) > 0
    return sel


def prepare_data(spec: CNSpec, obs: np.ndarray, acs: np.ndarray) -> np.ndarray:
    """constraint_net.py:258-299: normalise+clip obs, one-hot or clip actions, concat, select, cast fp32.

    All arithmetic stays in whatever numpy promotes to (float64 once mean/var or a
    float64 obs is involved), rounded to float32 once at the end -- as the reference.
    """
    if spec.obs_mean is not None and spec.obs_var is not None:        # normalize_obs :275-283
        obs = (obs - spec.obs_mean[None]) / np.sqrt(spec.obs_var[None] + spec.eps)
    if spec.clip_obs is not None:
        obs = np.clip(obs, -spec.clip_obs, spec.clip_obs)
    if spec.is_discrete:                                              # reshape_actions :285-293
        a = acs.astype(int)
        if acs.ndim > 1:
            a = np.squeeze(a, axis=-1)
        acs = np.zeros([acs.shape[0], spec.acs_dim])
        acs[np.arange(a.shape[0]), a] = 1.0
    if spec.action_high is not None and spec.action_low is not None:  # clip_actions :295-299
        acs = np.clip(acs, spec.action_low, spec.action_high)
    x = np.concatenate([obs, acs], axis=-1)[..., spec.select_dim]     # :268, :272-273
    return np.asarray(x, dtype=np.float32)


def forward(params: List[th.Tensor], x: th.Tensor) -> th.Tensor:
    """Linear -> ReLU -> ... -> Linear -> Sigmoid (constraint_net.py:104-107, torch_layers.py:112-123)."""
    n_layers = len(params) // 2
    h = x
    for i in range(n_layers):
        h = th.nn.functional.linear(h, params[2 * i], params[2 * i + 1])
        if i < n_layers - 1:
            h = th.relu(h)
    return th.sigmoid(h)


def cost_function(params, spec: CNSpec, obs: np.ndarray, acs: np.ndarray) -> np.ndarray:
    """constraint_net.py:121-130: cost = 1 - zeta(x), squeezed, numpy float32."""
    assert obs.shape[-1] == spec.obs_dim
    if not spec.is_discrete:
        assert acs.shape[-1] == spec.acs_dim
    x = th.tensor(prepare_data(spec, obs, acs), dtype=th.float32)
    with th.no_grad():
        out = forward(params, x)
    cost = 1 - out.numpy()
    return cost.squeeze(axis=-1)


def compute_is_weights(preds_old: th.Tensor, preds_new: th.Tensor, episode_lengths, eps: float, per_step: bool):
    """constraint_net.py:231-256.  preds are [N,1] fp32.  Returns (is_weights, kl_old_new, kl_new_old).

    per_step -> is_weights has shape [N,1]; per-episode -> shape [N] (this shape
    difference is what causes the N x N broadcast in `train`, see quirk A).
    """
    with th.no_grad():
        n_episodes = len(episode_lengths)
        cumulative = [0] + list(accumulate(int(l) for l in episode_lengths))
        ratio = (preds_new + eps) / (preds_old + eps)
        prod = th.tensor([th.prod(ratio[cumulative[j]:cumulative[j + 1]]) for j in range(n_episodes)])
        normed = n_episodes * prod / (th.sum(prod) + eps)
        if per_step:
            is_weights = ratio / th.mean(ratio)
        else:
            is_weights = th.repeat_interleave(normed, th.as_tensor([int(l) for l in episode_lengths]))
        kl_old_new = th.mean(-th.log(prod + eps))
        prod_mean = th.mean(prod)
        kl_new_old = th.mean((prod - prod_mean) * th.log(prod + eps) / (prod_mean + eps))
    return is_weights, kl_old_new, kl_new_old


def adam_init(params):
    return {"step": 0, "exp_avg": [th.zeros_like(p) for p in params], "exp_avg_sq": [th.zeros_like(p) for p in params]}


def adam_step(params, grads, state, lr, eps=1e-5, betas=(0.9, 0.999)):
    """torch/optim/adam.py `_single_tensor_adam` (CPU path, no amsgrad / weight decay), in place."""
    beta1, beta2 = betas
    state["step"] += 1
    step = state["step"]
    bias_correction1 = 1 - beta1 ** step
    bias_correction2 = 1 - beta2 ** step
    step_size = lr / bias_correction1
    bias_correction2_sqrt = bias_correction2 ** 0.5
    with th.no_grad():
        for p, g, m, v in zip(params, grads, state["exp_avg"], state["exp_avg_sq"]):
            m.lerp_(g, 1 - beta1)
            v.mul_(beta2).addcmul_(g, g, value=1 - beta2)
            denom = (v.sqrt() / bias_correction2_sqrt).add_(eps)
            p.addcdiv_(m, denom, value=-step_size)


def batches(batch_size, nom_size, exp_size):
    """constraint_net.py:301-317 `get`: everything when batch_size is None, else one numpy permutation (global RNG) of
    min(nom_size, exp_size) cut into minibatches -- the SAME indices for the nominal and the expert set."""
    if batch_size is None:
        yield None, None
        return
    size = min(nom_size, exp_size)
    indices = np.random.permutation(size)
    for start in range(0, size, batch_size):
        yield indices[start:start + batch_size], indices[start:start + batch_size]


def loss_terms(spec: CNSpec, nominal_preds: th.Tensor, expert_preds: th.Tensor, is_batch: th.Tensor,
               materialize_broadcast: bool = False):
    """constraint_net.py:193-202: (loss, nominal_loss, expert_loss, regularizer_loss) of one batch.  Works in the dtype
    of the predictions, so a float64 forward gives the float64 loss (and, through autograd, the float64 gradient).
    `is_batch` is the weight tensor as `train` shapes it: [N,1,1] in per-step IS mode (quirk A), [N,1] otherwise."""
    eps = spec.eps
    if spec.train_gail_lambda:                                    # :193-197
        bce = th.nn.BCELoss()
        nominal_loss = bce(nominal_preds, th.zeros(*nominal_preds.size(), dtype=nominal_preds.dtype))
        expert_loss = bce(expert_preds, th.ones(*expert_preds.size(), dtype=expert_preds.dtype))
        regularizer_loss = th.tensor(0)
        loss = nominal_loss + expert_loss
    else:                                                         # :199-202
        expert_loss = th.mean(th.log(expert_preds + eps))
        log_nom = th.log(nominal_preds + eps)
        if is_batch.dim() == 3 and not materialize_broadcast:
            nominal_loss = th.mean(is_batch) * th.mean(log_nom)
        else:
            nominal_loss = th.mean(is_batch * log_nom)
        regularizer_loss = spec.regularizer_coeff * (th.mean(1 - expert_preds) + th.mean(1 - nominal_preds))
        loss = (-expert_loss + nominal_loss) + regularizer_loss
    return loss, nominal_loss, expert_loss, regularizer_loss


def train(params, adam_state, spec: CNSpec, iterations: int, nominal_obs, nominal_acs, episode_lengths,
          expert_obs, expert_acs, lr: float, adam_eps: float = 1e-5, materialize_broadcast: bool = False,
          batch_size: Optional[int] = None):
    """constraint_net.py:137-229; batch_size=None is the full-batch mode the shipped configs use, an int the -cbs
    minibatch mode (permutations from the global numpy RNG, as the reference draws them).

    `spec.obs_mean/obs_var` must already hold this call's normalisation stats (:152-153).
    Quirk A (SURVEY §8 a16): in per-step IS mode the reference multiplies an [N,1,1] weight
    tensor with the [N,1] log-preds, i.e. takes the mean of an [N,N,1] outer product, which
    equals mean(w) * mean(log p).  We use that O(N) identity unless `materialize_broadcast`.
    Returns the `backward/*` metrics dict; params / adam_state are updated in place.
    """
    eps = spec.eps
    nominal = th.tensor(prepare_data(spec, nominal_obs, nominal_acs), dtype=th.float32)
    expert = th.tensor(prepare_data(spec, expert_obs, expert_acs), dtype=th.float32)
    for p in params:
        p.requires_grad_(True)

    if spec.importance_sampling:
        with th.no_grad():
            start_preds = forward(params, nominal).detach()
    early_stop_itr = iterations
    loss = th.tensor(np.inf)
    kl_old_new = kl_new_old = None
    for itr in range(iterations):
        if spec.importance_sampling:
            with th.no_grad():
                current_preds = forward(params, nominal).detach()
            is_weights, kl_old_new, kl_new_old = compute_is_weights(
                start_preds.clone(), current_preds.clone(), episode_lengths, eps, spec.per_step_importance_sampling)
            if ((spec.target_kl_old_new != -1 and kl_old_new > spec.target_kl_old_new) or
                    (spec.target_kl_new_old != -1 and kl_new_old > spec.target_kl_new_old)):
                early_stop_itr = itr
                break
        else:
            is_weights = th.ones(nominal.shape[0])
        for nom_idx, exp_idx in batches(batch_size, nominal.shape[0], expert.shape[0]):      # :180-207
            nominal_batch = nominal if nom_idx is None else nominal[nom_idx]
            expert_batch = expert if exp_idx is None else expert[exp_idx]
            is_batch = (is_weights if nom_idx is None else is_weights[nom_idx])[..., None]
            nominal_preds = forward(params, nominal_batch)
            expert_preds = forward(params, expert_batch)
            loss, nominal_loss, expert_loss, regularizer_loss = loss_terms(spec, nominal_preds, expert_preds, is_batch,
                                                                           materialize_broadcast)
            grads = th.autograd.grad(loss, params)
            adam_step(params, grads, adam_state, lr, eps=adam_eps)

    for p in params:
        p.requires_grad_(False)
    m = {"backward/cn_loss": loss.item(),
         "backward/expert_loss": expert_loss.item(),
         "backward/unweighted_nominal_loss": th.mean(th.log(nominal_preds + eps)).item(),
         "backward/nominal_loss": nominal_loss.item(),
         "backward/regularizer_loss": regularizer_loss.item(),
         "backward/is_mean": th.mean(is_weights).item(),
         "backward/is_max": th.max(is_weights).item(),
         "backward/is_min": th.min(is_weights).item(),
         "backward/nominal_preds_max": th.max(nominal_preds).item(),
         "backward/nominal_preds_min": th.min(nominal_preds).item(),
         "backward/nominal_preds_mean": th.mean(nominal_preds).item(),
         "backward/expert_preds_max": th.max(expert_preds).item(),
         "backward/expert_preds_min": th.min(expert_preds).item(),
         "backward/expert_preds_mean": th.mean(expert_preds).item()}
    if spec.importance_sampling:
        m.update({"backward/kl_old_new": kl_old_new.item(), "backward/kl_new_old": kl_new_old.item(),
                  "backward/early_stop_itr": early_stop_itr})
    return m
