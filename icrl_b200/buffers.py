"""RolloutBufferWithCost -- host-side mirror of stable_baselines3/common/buffers.py:443-627.

The 16 public numpy float32 arrays stay host-resident and authoritative (callbacks mutate them in place at
`on_rollout_end`, icrl/exploration.py:65,311), exactly as in the reference: time-major [n_steps, n_envs, ...]
until the first `get()`, then the ten trained-on fields become env-major flat views.  What changes:

* `compute_returns_and_advantage` runs the dual GAE scan on the GPU (K3, one C-ABI call with host buffers);
* `device_view()` uploads the fields K4 trains on once per rollout (pinned staging -> HBM) in TIME-major layout;
  the PPO kernel translates env-major minibatch indices itself, so no transposed device copy exists;
* `get()` still yields the reference's minibatch samples (host gather) for code that iterates the buffer directly.
"""
import ctypes as C
from typing import Generator, Optional

import numpy as np
import torch as th

from . import _lib
from .device import resolve_device
from .spaces import get_action_dim, get_obs_shape, is_discrete
from .type_aliases import RolloutBufferWithCostSamples

_FLAT_FIELDS = ["orig_observations", "observations", "actions", "log_probs", "reward_values", "reward_advantages",
                "reward_returns", "cost_values", "cost_advantages", "cost_returns"]          # buffers.py:599-601
_TRAIN_FIELDS = ["observations", "actions", "log_probs", "reward_values", "reward_advantages", "reward_returns",
                 "cost_values", "cost_advantages", "cost_returns"]


class RolloutBufferWithCost:
    def __init__(self, buffer_size: int, observation_space, action_space, device="cuda",
                 reward_gamma: float = 0.99, reward_gae_lambda: float = 1, cost_gamma: float = 0.99,
                 cost_gae_lambda: float = 1, n_envs: int = 1):
        self.buffer_size = buffer_size
        self.observation_space, self.action_space = observation_space, action_space
        self.obs_shape = get_obs_shape(observation_space)
        self.action_dim = get_action_dim(action_space)
        self.device = device
        self._dev = None
        self._stage = {}                # persistent pinned / device staging buffers of relabel_costs
        self.n_envs = n_envs
        self.reward_gamma, self.reward_gae_lambda = reward_gamma, reward_gae_lambda
        self.cost_gamma, self.cost_gae_lambda = cost_gamma, cost_gae_lambda
        self.pos, self.full, self.generator_ready = 0, False, False
        self.reset()

    # ---------------------------------------------------------------- storage (buffers.py:468-491)
    def reset(self) -> None:
        T, E = self.buffer_size, self.n_envs
        for name in ("observations", "new_observations", "orig_observations", "new_orig_observations"):
            setattr(self, name, np.zeros((T, E) + self.obs_shape, dtype=np.float32))
        self.actions = np.zeros((T, E, self.action_dim), dtype=np.float32)
        for name in ("dones", "log_probs", "rewards", "reward_returns", "reward_values", "reward_advantages", "costs",
                     "orig_costs", "cost_returns", "cost_values", "cost_advantages"):
            setattr(self, name, np.zeros((T, E), dtype=np.float32))
        self.generator_ready = False
        self.pos, self.full = 0, False

    def size(self) -> int:
        return self.buffer_size if self.full else self.pos

    @staticmethod
    def _np(x):
        return x.detach().cpu().numpy() if isinstance(x, th.Tensor) else np.asarray(x)

    def add(self, obs, orig_obs, new_obs, new_orig_obs, action, reward, cost, orig_cost, done, reward_value,
            cost_value, log_prob) -> None:
        """buffers.py:554-592 (values / log-probs may be torch tensors or arrays)."""
        p = self.pos
        self.observations[p] = np.asarray(obs)
        self.orig_observations[p] = np.asarray(orig_obs)
        self.new_observations[p] = np.asarray(new_obs)
        self.new_orig_observations[p] = np.asarray(new_orig_obs)
        self.actions[p] = np.asarray(action).reshape(self.n_envs, self.action_dim)
        self.dones[p] = np.asarray(done)
        self.log_probs[p] = self._np(log_prob).reshape(-1)
        self.rewards[p] = np.asarray(reward)
        self.reward_values[p] = self._np(reward_value).flatten()
        self.costs[p] = np.asarray(cost)
        self.orig_costs[p] = np.asarray(orig_cost)
        self.cost_values[p] = self._np(cost_value).flatten()
        self.pos += 1
        if self.pos == self.buffer_size:
            self.full = True

    # ---------------------------------------------------------------- K3
    def compute_returns_and_advantage(self, reward_last_value, cost_last_value, dones: np.ndarray) -> None:
        """buffers.py:543-552 -> one fused dual-GAE launch (reward and cost scans share the `dones` reads)."""
        T, E = self.buffer_size, self.n_envs
        rlv = np.ascontiguousarray(self._np(reward_last_value).astype(np.float32).flatten())
        clv = np.ascontiguousarray(self._np(cost_last_value).astype(np.float32).flatten())
        last = np.ascontiguousarray(np.asarray(dones).astype(np.uint8).reshape(-1))
        assert rlv.shape[0] == E and clv.shape[0] == E and last.shape[0] == E
        ins = [np.ascontiguousarray(getattr(self, k), dtype=np.float32)
               for k in ("rewards", "reward_values", "costs", "cost_values", "dones")]
        outs = [np.empty((T, E), dtype=np.float32) for _ in range(4)]
        dev = self._device()
        with th.cuda.device(dev):
            _lib.check(_lib.lib().icrl_dual_gae_host(
                *[_lib.ptr(a) for a in ins], _lib.ptr(rlv), _lib.ptr(clv), _lib.ptr(last), T, E,
                float(self.reward_gamma), float(self.reward_gae_lambda), float(self.cost_gamma),
                float(self.cost_gae_lambda), *[_lib.ptr(o) for o in outs], _lib.current_stream()))
        self.reward_advantages, self.reward_returns, self.cost_advantages, self.cost_returns = outs

    # ---------------------------------------------------------------- K1 + K5 on the whole rollout (SURVEY §8 f1)
    def relabel_costs(self, constraint_net, cost_normalizer, last_dones: np.ndarray) -> None:
        """Fill `orig_costs` / `costs` for the whole rollout after collection, instead of one cost_function call per
        environment step: K1 over [T*E] rows of (orig_observations, actions), then the online statistics of
        `cost_normalizer` (a VecNormalizeWithCost, or None) replayed on the device by icrl_cost_normalize -- bit-exact
        with what vec_cost_wrapper.py:37-41 + vec_normalize.py:232-257 would have produced step by step, because the
        constraint net does not change during collection."""
        T, E = self.buffer_size, self.n_envs
        dev = self._device()
        with th.cuda.device(dev):
            # pinned staging + asynchronous copies on the current stream; ONE synchronisation at the end
            obs = self._h2d("relabel_obs", np.ascontiguousarray(self.orig_observations)).reshape(T * E, -1)
            acs = self.actions
            if not is_discrete(self.action_space):      # the environment (and so the cost wrapper) saw clipped actions
                acs = np.clip(acs, self.action_space.low, self.action_space.high)
            acs = self._h2d("relabel_acs", np.ascontiguousarray(acs, dtype=np.float32)).reshape(T * E, -1)
            if is_discrete(self.action_space):
                acs = acs.reshape(-1)
            orig = constraint_net.cost_function_device(obs, acs).reshape(T, E)
            costs = orig
            vn = cost_normalizer
            state_h = None
            if vn is not None:
                state = np.concatenate([[vn.cost_rms.mean, vn.cost_rms.var, vn.cost_rms.count], vn.cost_ret]).astype(np.float64)
                state_d = self._h2d("relabel_state", state)
                dones_d = self._h2d("relabel_dones", np.ascontiguousarray(self.dones))
                last_d = self._h2d("relabel_last", np.ascontiguousarray(np.asarray(last_dones).astype(np.uint8).reshape(-1)))
                costs = th.empty_like(orig)
                _lib.check(_lib.lib().icrl_cost_normalize(
                    _lib.ptr(orig), _lib.ptr(dones_d), _lib.ptr(last_d), T, E, float(vn.cost_gamma), float(vn.epsilon),
                    float(vn.clip_cost), int(bool(vn.norm_cost)), int(bool(vn.training)), _lib.ptr(state_d),
                    _lib.ptr(costs), _lib.current_stream()))
                state_h = self._d2h("relabel_state_out", state_d)
            orig_h = self._d2h("relabel_orig_out", orig)
            costs_h = orig_h if costs is orig else self._d2h("relabel_costs_out", costs)
            th.cuda.current_stream().synchronize()
            if vn is not None:
                state = state_h.numpy()
                if vn.training:
                    vn.cost_rms.mean, vn.cost_rms.var, vn.cost_rms.count = state[0], state[1], float(state[2])
                vn.cost_ret = state[3:].copy()
            self.orig_costs = orig_h.numpy().copy()
            self.costs = self.orig_costs if costs is orig else costs_h.numpy().copy()
            if vn is not None:
                vn.old_cost = self.orig_costs[-1].copy()

    def _h2d(self, name: str, host: np.ndarray) -> th.Tensor:
        """host array -> persistent pinned staging buffer -> persistent device buffer (asynchronous on the current stream)."""
        slot = self._stage.get(name)
        t = th.from_numpy(host)
        if slot is None or slot[0].shape != t.shape or slot[0].dtype != t.dtype:
            pinned = th.empty(t.shape, dtype=t.dtype).pin_memory()
            slot = (pinned, th.empty(t.shape, dtype=t.dtype, device=self._device()))
            self._stage[name] = slot
        slot[0].copy_(t)
        slot[1].copy_(slot[0], non_blocking=True)
        return slot[1]

    def _d2h(self, name: str, dev_t: th.Tensor) -> th.Tensor:
        """device tensor -> persistent pinned host buffer (asynchronous: valid after the stream is synchronised)."""
        slot = self._stage.get(name)
        if slot is None or slot.shape != dev_t.shape or slot.dtype != dev_t.dtype:
            slot = th.empty(dev_t.shape, dtype=dev_t.dtype).pin_memory()
            self._stage[name] = slot
        slot.copy_(dev_t, non_blocking=True)
        return slot

    def _device(self):
        if self._dev is None:
            self._dev = resolve_device(self.device)
        return self._dev

    # ---------------------------------------------------------------- minibatches (buffers.py:594-627)
    @staticmethod
    def swap_and_flatten(arr: np.ndarray) -> np.ndarray:
        shape = arr.shape
        if len(shape) < 3:
            shape = shape + (1,)
        return arr.swapaxes(0, 1).reshape(shape[0] * shape[1], *shape[2:])

    def _flatten_once(self):
        if not self.generator_ready:
            for name in _FLAT_FIELDS:
                self.__dict__[name] = self.swap_and_flatten(self.__dict__[name])
            self.generator_ready = True

    def get(self, batch_size: Optional[int] = None) -> Generator[RolloutBufferWithCostSamples, None, None]:
        assert self.full, ""
        n = self.buffer_size * self.n_envs
        indices = np.random.permutation(n)
        self._flatten_once()
        if batch_size is None:
            batch_size = n
        start = 0
        while start < n:
            yield self._get_samples(indices[start:start + batch_size])
            start += batch_size

    def to_torch(self, array: np.ndarray, copy: bool = True) -> th.Tensor:
        return th.tensor(array).to(self._device()) if copy else th.as_tensor(array).to(self._device())

    def _get_samples(self, batch_inds: np.ndarray, env=None) -> RolloutBufferWithCostSamples:
        data = (self.orig_observations[batch_inds], self.observations[batch_inds], self.actions[batch_inds],
                self.log_probs[batch_inds].flatten(), self.reward_values[batch_inds].flatten(),
                self.reward_advantages[batch_inds].flatten(), self.reward_returns[batch_inds].flatten(),
                self.cost_values[batch_inds].flatten(), self.cost_advantages[batch_inds].flatten(),
                self.cost_returns[batch_inds].flatten())
        return RolloutBufferWithCostSamples(*tuple(map(self.to_torch, data)))

    # ---------------------------------------------------------------- device staging for K4
    def time_major(self, name: str) -> np.ndarray:
        """The field as [T, E, ...] regardless of whether `get()` has already flattened it to env-major."""
        arr = getattr(self, name)
        if self.generator_ready and name in _FLAT_FIELDS:
            T, E = self.buffer_size, self.n_envs
            arr = arr.reshape(E, T, *arr.shape[1:]).swapaxes(0, 1)
        return arr

    def device_view(self) -> dict:
        """Upload the nine fields PPOLagrangian.train reads (one pinned staging copy + async H2D each).
        Returned tensors are time-major and contiguous; keys follow RolloutBufferWithCostSamples naming."""
        dev = self._device()
        out = {}
        rename = {"log_probs": "old_log_prob", "reward_values": "old_reward_values", "cost_values": "old_cost_values"}
        for name in _TRAIN_FIELDS:
            host = np.ascontiguousarray(self.time_major(name), dtype=np.float32)
            out[rename.get(name, name)] = th.from_numpy(host).pin_memory().to(dev, non_blocking=True)
        return out
