"""PPOLagrangian -- host-side mirror of stable_baselines3/ppo_lag/ppo_lag.py:17-365 and of the
OnPolicyWithCostAlgorithm plumbing it inherits (common/on_policy_algorithm.py:258-497, base_class.py).

`train()` is the learner hot path: the rollout buffer's fields are staged to HBM once, numpy's per-epoch
permutations are drawn on the host (global numpy RNG, as buffers.py:596 does) and ONE persistent cluster kernel
(K4, csrc/k4_ppo_lag.cu) runs every minibatch of every epoch, the global-norm clip, Adam and the target_kl early
stop.  The dual step (dual_variable.py:47-57) follows as a second tiny launch.  `learn()` / `collect_rollouts()`
keep the reference's control flow; env stepping stays on the host (north_star (c)).
"""
import ctypes as C
from collections import deque
import os
import time
from typing import Any, Callable, Dict, Optional, Union

import numpy as np
import torch as th

from . import _lib, logger
from .buffers import RolloutBufferWithCost
from .device import resolve_device
from .dual_variable import DualVariable, PIDLagrangian
from .policies import ActorTwoCriticsPolicy
from .spaces import is_discrete as _is_discrete

POLICIES = {"TwoCriticsMlpPolicy": ActorTwoCriticsPolicy}


def get_schedule_fn(value_schedule):
    """stable_baselines3/common/utils.py:74-91: constants become constant schedules of progress_remaining."""
    if isinstance(value_schedule, (float, int)):
        v = float(value_schedule)
        return lambda _: v
    assert callable(value_schedule)
    return value_schedule


def explained_variance(y_pred: np.ndarray, y_true: np.ndarray) -> np.ndarray:
    """stable_baselines3/common/utils.py:43-59."""
    assert y_true.ndim == 1 and y_pred.ndim == 1
    var_y = np.var(y_true)
    return np.nan if var_y == 0 else 1 - np.var(y_true - y_pred) / var_y


class _NullCallback:
    def init_callback(self, model): pass
    def on_training_start(self, locals_, globals_): pass
    def on_rollout_start(self): pass
    def update_locals(self, locals_): pass
    def on_step(self): return True
    def on_rollout_end(self): pass
    def on_training_end(self): pass


class _CallbackList(_NullCallback):
    def __init__(self, callbacks): self.callbacks = list(callbacks)
    def init_callback(self, model): [c.init_callback(model) for c in self.callbacks]
    def on_training_start(self, l, g): [c.on_training_start(l, g) for c in self.callbacks]
    def on_rollout_start(self): [c.on_rollout_start() for c in self.callbacks]
    def update_locals(self, l): [c.update_locals(l) for c in self.callbacks if hasattr(c, "update_locals")]
    def on_step(self):
        # callbacks.py:186-193: every callback runs (no short circuit), the results are and-ed
        results = [c.on_step() for c in self.callbacks]
        return all(r is not False for r in results)
    def on_rollout_end(self): [c.on_rollout_end() for c in self.callbacks]
    def on_training_end(self): [c.on_training_end() for c in self.callbacks]


def _find_cost_normalizer(env):
    """The VecNormalizeWithCost layer of a wrapped env (None when costs are not normalised)."""
    from .vec_env import VecEnvWrapper, VecNormalizeWithCost
    while isinstance(env, VecEnvWrapper):
        if isinstance(env, VecNormalizeWithCost):
            return env
        env = env.venv
    return None


class PPOLagrangian:
    def __init__(
        self,
        policy: Union[str, type],
        env,
        algo_type: str = 'lagrangian',
        learning_rate: Union[float, Callable] = 3e-4,
        n_steps: int = 2048,
        batch_size: Optional[int] = 64,
        n_epochs: int = 10,
        reward_gamma: float = 0.99,
        reward_gae_lambda: float = 0.95,
        cost_gamma: float = 0.99,
        cost_gae_lambda: float = 0.95,
        clip_range: float = 0.2,
        clip_range_reward_vf: Optional[float] = None,
        clip_range_cost_vf: Optional[float] = None,
        ent_coef: float = 0.0,
        reward_vf_coef: float = 0.5,
        cost_vf_coef: float = 0.5,
        max_grad_norm: float = 0.5,
        use_sde: bool = False,
        sde_sample_freq: int = -1,
        target_kl: Optional[float] = None,
        penalty_initial_value: float = 1,
        penalty_learning_rate: float = 0.01,
        penalty_min_value: Optional[float] = None,
        update_penalty_after: int = 1,
        budget: float = 0.,
        tensorboard_log: Optional[str] = None,
        create_eval_env: bool = False,
        pid_kwargs: Optional[Dict[str, Any]] = None,
        policy_kwargs: Optional[Dict[str, Any]] = None,
        verbose: int = 0,
        seed: Optional[int] = None,
        device: Union[th.device, str] = "auto",
        _init_setup_model: bool = True,
    ):
        if use_sde:
            raise NotImplementedError("gSDE is not used by the ICRL configs and not implemented")
        self.policy_class = POLICIES[policy] if isinstance(policy, str) else policy
        self.env = env
        self.observation_space, self.action_space = env.observation_space, env.action_space
        self.n_envs = getattr(env, "num_envs", 1)
        self.algo_type, self.learning_rate = algo_type, learning_rate
        self.n_steps, self.batch_size, self.n_epochs = n_steps, batch_size, n_epochs
        self.reward_gamma, self.reward_gae_lambda = reward_gamma, reward_gae_lambda
        self.cost_gamma, self.cost_gae_lambda = cost_gamma, cost_gae_lambda
        self.clip_range, self.clip_range_reward_vf, self.clip_range_cost_vf = clip_range, clip_range_reward_vf, clip_range_cost_vf
        self.ent_coef, self.reward_vf_coef, self.cost_vf_coef = ent_coef, reward_vf_coef, cost_vf_coef
        self.max_grad_norm, self.target_kl = max_grad_norm, target_kl
        self.use_sde, self.sde_sample_freq = use_sde, sde_sample_freq
        self.penalty_initial_value, self.penalty_learning_rate = penalty_initial_value, penalty_learning_rate
        self.penalty_min_value, self.update_penalty_after = penalty_min_value, update_penalty_after
        self.budget, self.pid_kwargs = budget, pid_kwargs
        self.policy_kwargs = {} if policy_kwargs is None else policy_kwargs
        self.verbose, self.seed = verbose, seed
        self.device = resolve_device(device)
        self.num_timesteps, self._total_timesteps, self._n_updates = 0, 0, 0
        self._current_progress_remaining = 1
        self._last_obs = self._last_original_obs = self._last_dones = None
        self.start_time = None
        self.rollout_buffer = None
        self.ep_info_buffer = None
        self._staging = {}
        self.comm = None                # data-parallel plumbing (icrl_b200.distributed.PpoComm), see enable_data_parallel()
        if _init_setup_model:
            self._setup_model()
        if os.environ.get("ICRL_DATA_PARALLEL", "0") == "1":
            self.enable_data_parallel()

    # ---------------------------------------------------------------- setup (on_policy_algorithm.py:316-338, ppo_lag.py:145-175)
    def set_random_seed(self, seed: Optional[int] = None) -> None:
        """stable_baselines3/common/utils.py:23-40 + base_class.py:540-558."""
        if seed is None:
            return
        import random
        random.seed(seed)
        np.random.seed(seed)
        th.manual_seed(seed)
        if hasattr(self.action_space, "seed"):
            self.action_space.seed(seed)
        if self.env is not None and hasattr(self.env, "seed"):
            self.env.seed(seed)

    def _setup_model(self) -> None:
        self.lr_schedule = get_schedule_fn(self.learning_rate)
        self.set_random_seed(self.seed)
        self.rollout_buffer = RolloutBufferWithCost(
            self.n_steps, self.observation_space, self.action_space, self.device, reward_gamma=self.reward_gamma,
            reward_gae_lambda=self.reward_gae_lambda, cost_gamma=self.cost_gamma, cost_gae_lambda=self.cost_gae_lambda,
            n_envs=self.n_envs)
        self.policy = self.policy_class(self.observation_space, self.action_space, self.lr_schedule, use_sde=self.use_sde,
                                        device=self.device, **self.policy_kwargs)
        if self.algo_type == 'lagrangian':
            self.dual = DualVariable(self.budget, self.penalty_learning_rate, self.penalty_initial_value,
                                     self.penalty_min_value, device=self.device)
        elif self.algo_type == 'pidlagrangian':
            kw = self.pid_kwargs
            self.dual = PIDLagrangian(alpha=kw['alpha'], penalty_init=kw['penalty_init'], Kp=kw['Kp'], Ki=kw['Ki'],
                                      Kd=kw['Kd'], pid_delay=kw['pid_delay'], delta_p_ema_alpha=kw['delta_p_ema_alpha'],
                                      delta_d_ema_alpha=kw['delta_d_ema_alpha'])
        else:
            raise ValueError("Unrecognized value for argument 'algo_type' in PPOLagrangian")
        self.clip_range = get_schedule_fn(self.clip_range)
        for name in ("clip_range_reward_vf", "clip_range_cost_vf"):
            v = getattr(self, name)
            if v is not None:
                if isinstance(v, (float, int)):
                    assert v > 0, "`clip_range_vf` must be positive, pass `None` to deactivate vf clipping"
                setattr(self, name, get_schedule_fn(v))

    def enable_data_parallel(self, comm=None) -> "PPOLagrangian":
        """Data-parallel train() across the GPUs of one node (SURVEY 8(e); not in the reference, which has no
        distributed path).  One process per GPU under torch.distributed: every rank collects rollouts from ITS OWN
        `n_envs` environments, and train() runs `batch_size` local rows per optimiser step with the gradient all-reduce
        fused into the persistent kernel over NVLink peer memory (global minibatch = world x batch_size).  Parameters
        must start replicated (same seed / checkpoint on every rank); they stay bit-identical afterwards.  Also switched
        on by ICRL_DATA_PARALLEL=1 when the process group is initialised (`torchrun ... run_me.py icrl ...`)."""
        import torch.distributed as dist
        if comm is None:
            if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
                return self
        if self.policy.n_shared:
            raise NotImplementedError(f"data-parallel training of shared policy layers (net_arch "
                                      f"{self.policy.net_arch}) is not implemented")
        if comm is None:
            from .distributed import PpoComm
            with th.cuda.device(self.device):
                comm = PpoComm()
        self.comm = comm
        return self

    def _update_learning_rate(self, optimizer) -> None:
        """base_class.py:213-227."""
        lr = self.lr_schedule(self._current_progress_remaining)
        logger.record("train/learning_rate", lr)
        for g in optimizer.param_groups:
            g["lr"] = lr

    def _update_current_progress_remaining(self, num_timesteps: int, total_timesteps: int) -> None:
        self._current_progress_remaining = 1.0 - float(num_timesteps) / float(total_timesteps)

    # ---------------------------------------------------------------- K4
    def _draw_permutations(self, n: int):
        """One numpy permutation per epoch (buffers.py:596) and the global RNG state after each."""
        perms = np.empty((self.n_epochs, n), dtype=np.int32)
        rng_states = []
        for e in range(self.n_epochs):
            perms[e] = np.random.permutation(n)
            rng_states.append(np.random.get_state())
        return perms, rng_states

    def _speculate_permutations(self, n: int, state_if_all_epochs_run) -> None:
        """While the kernel runs the host is idle: draw the next train()'s permutations from the state the global numpy RNG
        will be in if (a) no epoch is cut by target_kl and (b) nobody touches np.random before the next call.  The next
        call uses them only if the RNG state it finds is exactly that one -- the stream the reference would see is unchanged."""
        if n * self.n_epochs > (1 << 22):       # large buffers: the draw outlasts the kernel and would double the host memory
            self._spec_perms = None
            return
        np.random.set_state(state_if_all_epochs_run)
        perms, states = self._draw_permutations(n)
        self._spec_perms = (n, self.n_epochs, state_if_all_epochs_run, perms, states)

    def _take_speculated_permutations(self, n: int):
        spec, self._spec_perms = getattr(self, "_spec_perms", None), None
        if spec is None or spec[0] != n or spec[1] != self.n_epochs:
            return None, None
        now, base = np.random.get_state(), spec[2]
        same = (now[0] == base[0] and now[2] == base[2] and now[3] == base[3] and now[4] == base[4]
                and np.array_equal(now[1], base[1]))
        if not same:
            return None, None
        np.random.set_state(spec[4][-1])        # where drawing them now would have left the generator
        return spec[3], spec[4]

    def _stage(self, name: str, host: np.ndarray) -> th.Tensor:
        """host array -> persistent pinned staging buffer -> persistent device buffer (async on the current stream)."""
        slot = self._staging.get(name)
        if slot is None or slot[0].shape != host.shape or slot[0].dtype != th.from_numpy(host[:0]).dtype:
            pinned = th.empty(host.shape, dtype=th.from_numpy(host[:0]).dtype).pin_memory()
            slot = (pinned, th.empty(host.shape, dtype=pinned.dtype, device=self.device))
            self._staging[name] = slot
        slot[0].numpy()[...] = host
        slot[1].copy_(slot[0], non_blocking=True)
        return slot[1]

    def train(self) -> None:
        """ppo_lag.py:177-338."""
        self._update_learning_rate(self.policy.optimizer)
        clip_range = self.clip_range(self._current_progress_remaining)
        clip_range_reward_vf = clip_range_cost_vf = None
        if self.clip_range_reward_vf is not None:
            clip_range_reward_vf = self.clip_range_reward_vf(self._current_progress_remaining)
        if self.clip_range_cost_vf is not None:
            clip_range_cost_vf = self.clip_range_cost_vf(self._current_progress_remaining)

        buf = self.rollout_buffer
        assert buf.full, ""
        T, E = buf.buffer_size, buf.n_envs
        n = T * E
        # numpy draws one permutation per epoch that actually runs (buffers.py:596); draw them all, remember the RNG
        # state after each, and rewind to the right one once the device reports where it stopped.
        perms, rng_states = self._take_speculated_permutations(n)
        if perms is None:
            perms, rng_states = self._draw_permutations(n)

        rename = {"log_probs": "old_log_prob", "reward_values": "old_reward_values", "cost_values": "old_cost_values"}
        data = _lib.PpoData()
        keep = []
        for name in ("observations", "actions", "log_probs", "reward_values", "reward_advantages", "reward_returns",
                     "cost_values", "cost_advantages", "cost_returns"):
            dev = self._stage(name, np.ascontiguousarray(buf.time_major(name), dtype=np.float32))
            keep.append(dev)
            setattr(data, rename.get(name, name), dev.data_ptr())
        perm_dev = self._stage("perm", perms)
        data.perm = perm_dev.data_ptr()

        # the multiplier is read on the device (no host round trip before the launch) when it lives there
        nu_on_device = isinstance(self.dual, DualVariable)
        if nu_on_device:
            data.nu_device = self.dual.nu.state[4:5].data_ptr()
        current_penalty = 0.0 if nu_on_device else float(self.dual.nu().item())
        pol = self.policy
        steps_per_epoch = (n + (self.batch_size or n) - 1) // (self.batch_size or n)
        cfg = pol.make_cfg(
            T=T, E=E, batch_size=int(self.batch_size or 0), n_epochs=self.n_epochs,
            has_target_kl=int(self.target_kl is not None), target_kl=float(self.target_kl or 0.0),
            has_clip_vf_reward=int(clip_range_reward_vf is not None), clip_range_reward_vf=float(clip_range_reward_vf or 0.0),
            has_clip_vf_cost=int(clip_range_cost_vf is not None), clip_range_cost_vf=float(clip_range_cost_vf or 0.0),
            clip_range=float(clip_range), ent_coef=float(self.ent_coef), reward_vf_coef=float(self.reward_vf_coef),
            cost_vf_coef=float(self.cost_vf_coef), max_grad_norm=float(self.max_grad_norm), nu=float(current_penalty),
            max_steps=int(getattr(self, "_max_steps", 0)))
        stats = th.zeros(self.n_epochs * steps_per_epoch, _lib.PPO_STATS_PER_STEP, device=self.device)
        result = th.zeros(4, dtype=th.int32, device=self.device)
        dp = self.comm is not None and self.comm.world > 1
        with th.cuda.device(self.device):
            if not dp:
                _lib.check(_lib.lib().icrl_ppo_train(
                    C.byref(cfg), C.byref(data), _lib.ptr(pol._params), _lib.ptr(pol._adam_m), _lib.ptr(pol._adam_v),
                    pol.optimizer.step_count, _lib.ptr(stats), _lib.ptr(result), _lib.current_stream()))
            else:
                # the advantage statistics of ppo_lag.py:218-222 are those of the GLOBAL minibatch: local partial sums ->
                # one small all-reduce; the gradients (and the loss sums) are all-reduced inside the kernel
                advsums = th.zeros(self.n_epochs * steps_per_epoch, 4, dtype=th.float64, device=self.device)
                _lib.check(_lib.lib().icrl_ppo_local_advsums(C.byref(cfg), C.byref(data), _lib.ptr(advsums),
                                                              _lib.current_stream()))
                self.comm.all_reduce_sum(advsums)
                desc = self.comm.descriptor(advsums)
                keep.append(advsums)
                _lib.check(_lib.lib().icrl_ppo_train_dist(
                    C.byref(cfg), C.byref(data), _lib.ptr(pol._params), _lib.ptr(pol._adam_m), _lib.ptr(pol._adam_v),
                    pol.optimizer.step_count, _lib.ptr(stats), _lib.ptr(result), C.byref(desc), _lib.current_stream()))
        # host work that does not depend on the update overlaps the kernel: the reference's public arrays become
        # env-major on the first get() (buffers.py:594-611), the rollout-only logger statistics, and the NEXT call's
        # permutations, drawn speculatively from the RNG state this call leaves behind when no epoch is skipped
        buf._flatten_once()
        self._speculate_permutations(n, rng_states[-1])
        mean_reward_adv = np.mean(buf.reward_advantages.flatten())
        mean_cost_adv = np.mean(buf.cost_advantages.flatten())
        reward_ev = explained_variance(buf.reward_returns.flatten(), buf.reward_values.flatten())
        cost_ev = explained_variance(buf.cost_returns.flatten(), buf.cost_values.flatten())
        average_cost = np.mean(buf.orig_costs)
        total_cost = np.sum(buf.orig_costs)
        if dp:      # the dual step sees the mean cost over every rank's environments
            tot = th.tensor([float(np.sum(buf.orig_costs, dtype=np.float64)), float(buf.orig_costs.size)],
                            dtype=th.float64, device=self.device)
            self.comm.all_reduce_sum(tot)
            tot = tot.cpu()
            average_cost, total_cost = float(tot[0] / tot[1]), float(tot[0])
        result_h = result.cpu()                                   # synchronises
        early_stop_epoch, steps = int(result_h[0]), int(result_h[1])
        if int(result_h[2]) != 0:
            raise _lib.IcrlError("PPO kernel: an exchange wait timed out (a cluster peer or a data-parallel rank did not "
                                 "deliver its gradients); the parameters of this launch are not valid")
        if dp:
            self.comm.advance(steps)
        pol.optimizer.step_count += steps
        epochs_run = min(self.n_epochs, early_stop_epoch + 1)
        np.random.set_state(rng_states[epochs_run - 1])
        st = stats[:steps].cpu().numpy()
        self.last_train_stats = st
        pg_losses, clip_fractions = st[:, 0], st[:, 1]
        reward_value_losses, cost_value_losses, entropy_losses = st[:, 2], st[:, 3], st[:, 4]
        last_epoch_kl = st[(epochs_run - 1) * steps_per_epoch:, 5]
        f32 = np.float32
        last_loss = (f32(st[-1, 0]) + f32(self.ent_coef) * f32(st[-1, 4]) + f32(self.reward_vf_coef) * f32(st[-1, 2])
                     + f32(self.cost_vf_coef) * f32(st[-1, 3]))

        self._n_updates += self.n_epochs
        # dual update with the original (un-normalised) cost, ppo_lag.py:301-306
        if self.update_penalty_after is None or ((self._n_updates / self.n_epochs) % self.update_penalty_after == 0):
            self.dual.update_parameter(average_cost)

        logger.record("train/entropy_loss", np.mean(entropy_losses.astype(np.float64)))
        logger.record("train/policy_gradient_loss", np.mean(pg_losses.astype(np.float64)))
        logger.record("train/reward_value_loss", np.mean(reward_value_losses.astype(np.float64)))
        logger.record("train/cost_value_loss", np.mean(cost_value_losses.astype(np.float64)))
        logger.record("train/approx_kl", np.mean(last_epoch_kl))
        logger.record("train/clip_fraction", np.mean(clip_fractions.astype(np.float64)))
        logger.record("train/loss", float(last_loss))
        logger.record("train/mean_reward_advantages", mean_reward_adv)
        logger.record("train/mean_cost_advantages", mean_cost_adv)
        logger.record("train/reward_explained_variance", reward_ev)
        logger.record("train/cost_explained_variance", cost_ev)
        logger.record("train/nu", self.dual.nu().item())
        logger.record("train/nu_loss", self.dual.loss.item())
        logger.record("train/average_cost", average_cost)
        logger.record("train/total_cost", total_cost)
        logger.record("train/early_stop_epoch", early_stop_epoch)
        if not pol.is_discrete:
            logger.record("train/std", th.exp(pol.log_std).mean().item())
        logger.record("train/n_updates", self._n_updates, exclude="tensorboard")
        logger.record("train/clip_range", clip_range)
        if clip_range_reward_vf is not None:
            logger.record("train/clip_range_reward_vf", clip_range_reward_vf)
        if clip_range_cost_vf is not None:
            logger.record("train/clip_range_cost_vf", clip_range_cost_vf)

    # ---------------------------------------------------------------- rollouts (on_policy_algorithm.py:340-421)
    def _init_callback(self, callback):
        if callback is None:
            callback = _NullCallback()
        elif isinstance(callback, (list, tuple)):
            callback = _CallbackList(callback)
        if hasattr(callback, "init_callback"):
            callback.init_callback(self)
        return callback

    def _setup_learn(self, total_timesteps, callback, reset_num_timesteps=True):
        """base_class.py:479-538 (without eval-env / Monitor plumbing)."""
        self.start_time = time.time()
        if self.ep_info_buffer is None or reset_num_timesteps:      # base_class.py:503-507
            self.ep_info_buffer = deque(maxlen=100)
        if reset_num_timesteps:
            self.num_timesteps = 0
        else:
            total_timesteps += self.num_timesteps
        self._total_timesteps = total_timesteps
        if reset_num_timesteps or self._last_obs is None:
            self._last_obs = self.env.reset()
            self._last_dones = np.zeros((self.n_envs,), dtype=bool)
            self._last_original_obs = (self.env.get_original_obs() if hasattr(self.env, "get_original_obs")
                                       else self._last_obs)
        return total_timesteps, self._init_callback(callback)

    def collect_rollouts(self, env, callback, rollout_buffer, n_rollout_steps: int, cost_function) -> bool:
        assert self._last_obs is not None, "No previous observation was provided"
        n_steps = 0
        rollout_buffer.reset()
        callback.on_rollout_start()
        has_orig_obs = hasattr(env, "get_original_obs")
        discrete = _is_discrete(self.action_space)
        # whole-buffer mode (SURVEY §8 f1): `cost_function` is the ConstraintNet itself -> no per-step cost calls, the
        # rollout is relabelled (K1) and cost-normalised (K5) on the device once collection is over
        relabel = hasattr(cost_function, "cost_function_device")
        while n_steps < n_rollout_steps:
            actions, reward_values, cost_values, log_probs = self.policy.forward(th.as_tensor(np.asarray(self._last_obs)))
            actions = actions.numpy()
            clipped_actions = actions
            if not discrete:
                clipped_actions = np.clip(actions, self.action_space.low, self.action_space.high)
            new_obs, rewards, dones, infos = env.step(clipped_actions)
            orig_obs = env.get_original_obs() if has_orig_obs else new_obs
            if relabel:
                costs = orig_costs = np.zeros(env.num_envs, dtype=np.float32)      # filled for the whole buffer below
            elif type(cost_function) is str:
                costs = np.array([info.get(cost_function, 0) for info in infos])
                orig_costs = env.get_original_cost() if hasattr(env, "get_original_cost") else costs
            else:
                costs = cost_function(orig_obs.copy(), clipped_actions)
                orig_costs = costs
            self.num_timesteps += env.num_envs
            callback.update_locals(locals())
            if callback.on_step() is False:
                return False
            for info in infos:                  # on_policy_algorithm.py:404 -> base_class.py:368-389, after on_step
                if info.get("episode") is not None:
                    self.ep_info_buffer.extend([info["episode"]])
            n_steps += 1
            if discrete:
                actions = actions.reshape(-1, 1)
            rollout_buffer.add(self._last_obs, self._last_original_obs, new_obs, orig_obs, actions, rewards, costs,
                               orig_costs, self._last_dones, reward_values, cost_values, log_probs)
            self._last_obs, self._last_original_obs, self._last_dones = new_obs, orig_obs, dones
        if relabel:
            rollout_buffer.relabel_costs(cost_function, _find_cost_normalizer(env), dones)
        rollout_buffer.compute_returns_and_advantage(reward_values, cost_values, dones=dones)
        callback.on_rollout_end()
        return True

    def learn(self, total_timesteps: int, cost_function: Union[str, Callable], callback=None, log_interval: int = 1,
              eval_env=None, eval_freq: int = -1, n_eval_episodes: int = 5, tb_log_name: str = "PPOLagrangian",
              eval_log_path: Optional[str] = None, reset_num_timesteps: bool = True) -> "PPOLagrangian":
        """on_policy_algorithm.py:430-492."""
        iteration = 0
        total_timesteps, callback = self._setup_learn(total_timesteps, callback, reset_num_timesteps)
        callback.on_training_start(locals(), globals())

        def training_infos(itr):
            elapsed = max(time.time() - self.start_time, 1e-9)
            logger.record("time/iterations", itr, exclude="tensorboard")
            logger.record("time/fps", int(self.num_timesteps / elapsed))
            logger.record("time/time_elapsed", int(elapsed), exclude="tensorboard")
            logger.record("time/total_timesteps", self.num_timesteps, exclude="tensorboard")
            if len(self.ep_info_buffer) > 0 and len(self.ep_info_buffer[0]) > 0:
                extra = {key for ep in self.ep_info_buffer for key in ep} - {'r', 'l', 't'}
                for key in extra:
                    vals = [ep[key] for ep in self.ep_info_buffer]
                    logger.record(f"rollout/ep_{key}_mean", np.mean(vals))
                    logger.record(f"rollout/ep_{key}_max", np.max(vals))
                    logger.record(f"rollout/ep_{key}_min", np.min(vals))
                logger.record("rollout/ep_rew_mean", np.mean([ep["r"] for ep in self.ep_info_buffer]))
                logger.record("rollout/ep_len_mean", np.mean([ep["l"] for ep in self.ep_info_buffer]))

        while self.num_timesteps < total_timesteps:
            if self.collect_rollouts(self.env, callback, self.rollout_buffer, self.n_steps, cost_function) is False:
                break
            iteration += 1
            self._update_current_progress_remaining(self.num_timesteps, total_timesteps)
            if log_interval is not None and iteration % log_interval == 0:
                training_infos(iteration)
                logger.dump(step=self.num_timesteps)
            self.train()
        training_infos(iteration + 1)          # like the reference: left in the logger for the caller (forward/* metrics)
        callback.on_training_end()
        return self

    def predict(self, observation, state=None, mask=None, deterministic: bool = False):
        return self.policy.predict(observation, state, mask, deterministic)

    # ---------------------------------------------------------------- checkpoints (base_class.py:564-700, save_util.py)
    _SAVED_SCALARS = ("algo_type", "learning_rate", "n_steps", "batch_size", "n_epochs", "reward_gamma",
                      "reward_gae_lambda", "cost_gamma", "cost_gae_lambda", "ent_coef", "reward_vf_coef", "cost_vf_coef",
                      "max_grad_norm", "target_kl", "penalty_initial_value", "penalty_learning_rate",
                      "penalty_min_value", "update_penalty_after", "budget", "seed", "n_envs", "num_timesteps",
                      "_total_timesteps", "_n_updates", "_current_progress_remaining", "use_sde", "policy_kwargs",
                      "pid_kwargs")

    def save(self, path: str) -> None:
        """Write the reference's zip layout: `data` (JSON), `policy.pth`, `policy.optimizer.pth`,
        `pytorch_variables.pth`, `_stable_baselines3_version`.  `data` holds plain JSON values only (the reference
        cloudpickles spaces / schedules into it; here the spaces are stored as shape/bounds and the schedules as their
        value at progress 1)."""
        import io, json, zipfile
        path = str(path)
        if not path.endswith(".zip"):
            path += ".zip"
        data = {}
        for k in self._SAVED_SCALARS:
            v = getattr(self, k, None)
            data[k] = v if not callable(v) else float(v(1))
        for k in ("clip_range", "clip_range_reward_vf", "clip_range_cost_vf"):
            v = getattr(self, k)
            data[k] = None if v is None else float(v(1)) if callable(v) else v
        osp, asp = self.observation_space, self.action_space
        data["observation_space"] = dict(shape=list(osp.shape))
        data["action_space"] = (dict(n=int(asp.n)) if _is_discrete(asp) else
                                dict(shape=list(asp.shape), low=np.asarray(asp.low).tolist(),
                                     high=np.asarray(asp.high).tolist()))
        data["policy_class"] = next((k for k, v in POLICIES.items() if v is self.policy_class), "TwoCriticsMlpPolicy")

        def blob(obj):
            buf = io.BytesIO()
            th.save(obj, buf)
            return buf.getvalue()
        variables = {}
        if isinstance(self.dual, DualVariable):
            variables = dict(dual_state=self.dual.nu.state.detach().cpu(), dual_steps=self.dual.steps)
        os_dir = os.path.dirname(path)
        if os_dir:
            os.makedirs(os_dir, exist_ok=True)
        with zipfile.ZipFile(path, "w") as zf:
            zf.writestr("data", json.dumps(data, indent=4, default=str))
            zf.writestr("policy.pth", blob(self.policy.state_dict()))
            zf.writestr("policy.optimizer.pth", blob(self.policy.optimizer.state_dict()))
            zf.writestr("pytorch_variables.pth", blob(variables))
            zf.writestr("_stable_baselines3_version", "0.9.0a2+icrl_b200")

    @classmethod
    def load(cls, path: str, env=None, device="auto", **kwargs) -> "PPOLagrangian":
        """Load a zip written by `save` OR by the reference (its expert `best_model.zip` files): the tensors come
        from `policy.pth` / `policy.optimizer.pth`; hyper-parameters from the plain-JSON entries of `data`; the
        observation / action spaces from `env`, from `data`, or -- for reference zips, whose spaces are cloudpickled
        gym objects -- from the parameter shapes."""
        import io, json, zipfile
        from .spaces import Box, Discrete
        path = str(path)
        if not os.path.exists(path) and os.path.exists(path + ".zip"):
            path += ".zip"
        with zipfile.ZipFile(path) as zf:
            data = json.loads(zf.read("data"))
            sd = th.load(io.BytesIO(zf.read("policy.pth")), map_location="cpu", weights_only=False)
            names = zf.namelist()
            osd = (th.load(io.BytesIO(zf.read("policy.optimizer.pth")), map_location="cpu", weights_only=False)
                   if "policy.optimizer.pth" in names else None)
            variables = (th.load(io.BytesIO(zf.read("pytorch_variables.pth")), map_location="cpu", weights_only=False)
                         if "pytorch_variables.pth" in names else {})

        def plain(k, default=None):
            v = data.get(k, default)
            return default if isinstance(v, dict) and ":serialized:" in v else v
        first = next(k for k in ("mlp_extractor.shared_net.0.weight", "mlp_extractor.policy_net.0.weight") if k in sd)
        obs_dim = sd[first].shape[1]
        act_out = sd["action_net.weight"].shape[0]
        if env is not None:
            osp, asp = env.observation_space, env.action_space
        else:
            o, a = plain("observation_space"), plain("action_space")
            osp = Box(-np.inf, np.inf, shape=tuple(o["shape"]) if o else (obs_dim,))
            if a is not None:
                asp = Discrete(a["n"]) if "n" in a else Box(np.asarray(a["low"], np.float32),
                                                            np.asarray(a["high"], np.float32))
            else:   # reference zip: continuous heads carry log_std; bounds unknown -> unbounded box
                asp = Box(-np.inf, np.inf, shape=(act_out,)) if "log_std" in sd else Discrete(act_out)

        class _Spaces:
            observation_space, action_space, num_envs = osp, asp, int(plain("n_envs", 1) or 1)
        ctor = {k: plain(k) for k in ("algo_type", "learning_rate", "n_steps", "batch_size", "n_epochs", "reward_gamma",
                                      "reward_gae_lambda", "cost_gamma", "cost_gae_lambda", "clip_range",
                                      "clip_range_reward_vf", "clip_range_cost_vf", "ent_coef", "reward_vf_coef",
                                      "cost_vf_coef", "max_grad_norm", "target_kl", "penalty_initial_value",
                                      "penalty_learning_rate", "penalty_min_value", "update_penalty_after", "budget",
                                      "seed", "policy_kwargs", "pid_kwargs") if plain(k) is not None}
        ctor.update(kwargs)
        if ctor.get("algo_type") == "pidlagrangian" and not ctor.get("pid_kwargs"):
            ctor["algo_type"] = "lagrangian"                        # PID state of a reference zip is not recoverable
        seed = ctor.pop("seed", None)
        model = cls(policy=POLICIES.get(plain("policy_class"), ActorTwoCriticsPolicy), env=env or _Spaces(),
                    device=device, seed=None, **ctor)
        model.seed = seed
        if env is None:
            model.env = None
        model.policy.load_state_dict(sd)
        if osd is not None and osd.get("state"):
            model.policy.optimizer.load_state_dict(osd)
        if "dual_state" in variables and isinstance(model.dual, DualVariable):
            model.dual.nu.state.copy_(variables["dual_state"])
            model.dual.steps = int(variables["dual_steps"])
        for k in ("num_timesteps", "_total_timesteps", "_n_updates", "_current_progress_remaining"):
            if plain(k) is not None:
                setattr(model, k, plain(k))
        return model

    def get_parameters(self):
        return {"policy": self.policy.state_dict(), "policy.optimizer": self.policy.optimizer.state_dict()}

    def set_parameters(self, params):
        self.policy.load_state_dict(params["policy"])
        if "policy.optimizer" in params:
            self.policy.optimizer.load_state_dict(params["policy.optimizer"])
