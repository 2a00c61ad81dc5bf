"""Stable-Baselines3 `VecEnv` adapter and a GPU-resident rollout collector for SpinTorqueVectorEnv.

SB3 is not installed in the build image; the adapter implements the documented VecEnv protocol (num_envs, observation_space,
action_space, reset, step_async/step_wait/step, close, env_is_wrapped, get_attr/set_attr/env_method, seed) with NumPy in/out and
same-step auto-reset, `infos[i]['terminal_observation']` and `infos[i]['TimeLimit.truncated']` like SB3's DummyVecEnv, and
subclasses stable_baselines3's VecEnv when it can be imported, so `PPO('MlpPolicy', SB3VecEnvAdapter(env))` works unchanged.

For env counts where SB3's host-side rollout buffer cannot exist (n_steps=2048 x 1M envs x 12 floats = 100 TB), RolloutCollector
keeps a [T, N, ...] ring of observations / actions / rewards / dones on the GPU with SB3-shaped tensors, and optionally the values,
log-probabilities and flags PPO needs together with the GAE advantages computed from them in one kernel, and the shuffled
minibatches of RolloutBuffer.get gathered from them one kernel launch each."""
from __future__ import annotations

import ctypes as C
from typing import Any, Callable, Dict, Iterator, List, NamedTuple, Optional, Sequence

import numpy as np

from .. import _lib
from ..parallel import all_reduce_stats

try:  # pragma: no cover - stable_baselines3 is not in the build image
    from stable_baselines3.common.vec_env import VecEnv as _VecEnvBase
except Exception:  # noqa: BLE001
    _VecEnvBase = object

try:  # pragma: no cover - stable_baselines3 is not in the build image
    from stable_baselines3.common.type_aliases import RolloutBufferSamples
except Exception:  # noqa: BLE001
    class RolloutBufferSamples(NamedTuple):
        """Field names of stable_baselines3.common.type_aliases.RolloutBufferSamples."""
        observations: Any
        actions: Any
        old_values: Any
        old_log_prob: Any
        advantages: Any
        returns: Any

_M64 = (1 << 64) - 1


def _splitmix64(state: int):
    """One step of splitmix64: (next state, output)."""
    state = (state + 0x9E3779B97F4A7C15) & _M64
    z = state
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & _M64
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & _M64
    return state, z ^ (z >> 31)


def minibatch_round_keys(rng_seed: int, env_offset: int, epoch: int) -> List[int]:
    """The 8 round keys of the minibatch permutation of one `RolloutCollector.get()` epoch (include/stg.h,
    stg_rollout_minibatch_f32). A pure function: each of rng_seed, env_offset, epoch (taken mod 2^64) in turn is XORed into a
    64-bit state (initially 0) and the state replaced by splitmix64's output for it; four more splitmix64 outputs from that
    state give keys (low 32 bits, high 32 bits) each. So a seed reproduces every epoch's permutation, and the shards of a
    multi-GPU run (distinct env_offset) shuffle independently."""
    state = 0
    for word in (rng_seed, env_offset, epoch):
        _, state = _splitmix64(state ^ (int(word) & _M64))
    keys = []
    for _ in range(4):
        state, z = _splitmix64(state)
        keys += [z & 0xFFFFFFFF, z >> 32]
    return keys


class SB3VecEnvAdapter(_VecEnvBase):
    def __init__(self, env):
        if not env.autoreset:
            raise ValueError("the SB3 adapter needs an env constructed with autoreset=True")
        self.env = env
        if _VecEnvBase is not object:          # the real SB3 base class: let it set num_envs / spaces / render bookkeeping
            super().__init__(env.num_envs, env.single_observation_space, env.single_action_space)
        self.num_envs = env.num_envs
        self.observation_space = env.single_observation_space
        self.action_space = env.single_action_space
        self.render_mode = None
        self._actions = None
        self.reset_infos: List[Dict[str, Any]] = [{} for _ in range(self.num_envs)]
        self._seed = None

    def reset(self) -> np.ndarray:
        obs, _ = self.env.reset(seed=self._seed)
        self._seed = None
        obs_np = obs.cpu().numpy()
        # host_outputs env: the tensor IS the pinned buffer the next step overwrites, and SB3 keeps reset()'s array as _last_obs
        return obs_np.copy() if obs.device.type == "cpu" else obs_np

    def seed(self, seed: Optional[int] = None) -> List[Optional[int]]:
        self._seed = seed
        return [None if seed is None else seed + i for i in range(self.num_envs)]

    def step_async(self, actions: np.ndarray) -> None:
        self._actions = np.asarray(actions, dtype=np.float32)

    def step_wait(self):
        obs, rew, term, trunc, info = self.env.step(self._actions)
        obs_np = obs.cpu().numpy()
        if obs.device.type == "cpu":          # host_outputs env: the tensor IS the pinned buffer the next step overwrites
            obs_np = obs_np.copy()
        term_np, trunc_np = term.cpu().numpy(), trunc.cpu().numpy()
        dones = term_np | trunc_np
        infos: List[Dict[str, Any]] = [{} for _ in range(self.num_envs)]
        if dones.any():
            fin = info["final_observation"].cpu().numpy()
            for i in np.nonzero(dones)[0]:
                infos[i]["terminal_observation"] = fin[i].copy()
                infos[i]["TimeLimit.truncated"] = bool(trunc_np[i] and not term_np[i])
                infos[i]["is_success"] = bool(term_np[i])
        return obs_np, rew.cpu().numpy().astype(np.float32), dones, infos

    def step(self, actions: np.ndarray):
        self.step_async(actions)
        return self.step_wait()

    def close(self) -> None:
        self.env.close()

    def get_attr(self, attr_name: str, indices=None) -> List[Any]:
        n = self.num_envs if indices is None else len(list(indices))
        return [getattr(self.env, attr_name)] * n

    def set_attr(self, attr_name: str, value: Any, indices=None) -> None:
        setattr(self.env, attr_name, value)

    def env_method(self, method_name: str, *args, indices=None, **kwargs) -> List[Any]:
        n = self.num_envs if indices is None else len(list(indices))
        return [getattr(self.env, method_name)(*args, **kwargs)] * n

    def env_is_wrapped(self, wrapper_class, indices=None) -> List[bool]:
        n = self.num_envs if indices is None else len(list(indices))
        return [False] * n

    def get_images(self) -> Sequence[Optional[np.ndarray]]:
        return [None] * self.num_envs


class RolloutCollector:
    """GPU-resident rollout of `n_steps` env steps: everything stays in HBM, one kernel launch per step plus the policy.
    `policy(obs[N,12] f32 cuda) -> actions[N,2] f32 cuda` (any torch module / callable).

    `store_values=True` keeps what PPO consumes as well: `policy(obs)` then returns `(actions [N,2], values [N] or [N,1],
    log_probs [N])` (SB3's ActorCriticPolicy.forward convention) and `collect(policy, value_fn)` stores `values`, `log_probs`,
    the step's `terminated` / `truncated` flags, `final_values` (`value_fn` on the step's final observations, for all N rows:
    one extra critic forward per step instead of a host synchronisation to find the ended envs) and `last_values` (`value_fn` on
    the observation after the last step). `compute_returns_and_advantage()` then fills `advantages` and `returns` in one kernel
    launch (K6), bootstrapping truncated episodes with V(final observation) like SB3's collect_rollouts. `rewards` stays the
    env's reward. `get(batch_size)` then yields shuffled `RolloutBufferSamples` minibatches like SB3's RolloutBuffer.get (K7).

    `collect(policy)` with an `ActorCriticPolicy` and no `value_fn` (store_values=True) takes the fused path: per step one K9
    launch writes the observations, raw actions, values, log-probs and the env actions, and one masked K9 critic launch
    computes `final_values` on the rows of the envs that ended only (see `_collect_fused`)."""

    def __init__(self, env, n_steps: int, store_observations: bool = True, store_values: bool = False):
        torch = _lib.require_cuda()
        self.env, self.n_steps = env, int(n_steps)
        N, dev = env.num_envs, env.device
        self.store_observations = store_observations
        self.store_values = store_values
        if store_values:
            if not env.autoreset:
                raise ValueError("store_values=True needs an env constructed with autoreset=True (final observations)")
            if env.host_outputs:
                raise ValueError("store_values=True needs the env's outputs on the device (host_outputs=False)")
        if store_observations:
            self.observations = torch.empty(self.n_steps, N, _lib.OBS_DIM, dtype=torch.float32, device=dev)
        self.actions = torch.empty(self.n_steps, N, 2, dtype=torch.float32, device=dev)
        self.rewards = torch.empty(self.n_steps, N, dtype=torch.float32, device=dev)
        self.dones = torch.empty(self.n_steps, N, dtype=torch.bool, device=dev)
        if store_values:
            plane = lambda dtype: torch.empty(self.n_steps, N, dtype=dtype, device=dev)  # noqa: E731
            self.values, self.log_probs, self.final_values = plane(torch.float32), plane(torch.float32), plane(torch.float32)
            self.terminated, self.truncated = plane(torch.bool), plane(torch.bool)
            self.last_values = torch.empty(N, dtype=torch.float32, device=dev)
            self.advantages, self.returns = plane(torch.float32), plane(torch.float32)
            self._values_collected = False
            self._advantages_computed = False
            self._epoch = 0                                 # get() calls so far: the epoch of the next permutation
        self._last_obs = None

    def collect(self, policy: Callable, value_fn: Optional[Callable] = None) -> Dict[str, Any]:
        if self.store_values:
            return self._collect_with_values(policy, value_fn)
        from ..policy import ActorCriticPolicy
        if isinstance(policy, ActorCriticPolicy):
            raise ValueError("an ActorCriticPolicy needs a collector with store_values=True (it returns values and "
                             "log-probabilities, and its actions are in policy units)")
        env = self.env
        if self._last_obs is None:
            self._last_obs, _ = env.reset()
        obs = self._last_obs
        for t in range(self.n_steps):
            if self.store_observations:
                self.observations[t].copy_(obs)
            act = policy(obs)
            self.actions[t].copy_(act)
            obs, rew, term, trunc, _ = env.step(self.actions[t])
            self.rewards[t].copy_(rew)
            self.dones[t].copy_(term | trunc)
        self._last_obs = obs
        return all_reduce_stats(env.stats_tensor())       # one collective per rollout: episode statistics (K5)

    def _collect_with_values(self, policy: Callable, value_fn: Optional[Callable]) -> Dict[str, Any]:
        import torch
        from ..policy import ActorCriticPolicy
        if isinstance(policy, ActorCriticPolicy) and value_fn is None:
            return self._collect_fused(policy)
        if value_fn is None:
            raise ValueError("a collector with store_values=True needs collect(policy, value_fn)")
        env, N = self.env, self.env.num_envs
        self._values_collected = self._advantages_computed = False
        if self._last_obs is None:
            self._last_obs, _ = env.reset()
        obs = self._last_obs
        with torch.no_grad():                              # like SB3's collect_rollouts: the stored planes carry no graph
            for t in range(self.n_steps):
                if self.store_observations:
                    self.observations[t].copy_(obs)
                out = policy(obs)
                if not (isinstance(out, (tuple, list)) and len(out) == 3):
                    raise ValueError("with store_values=True, policy(obs) must return (actions, values, log_probs)")
                act, val, logp = out
                self.actions[t].copy_(act)
                self.values[t].copy_(val.reshape(N))
                self.log_probs[t].copy_(logp.reshape(N))
                obs, rew, term, trunc, info = env.step(self.actions[t])
                self.rewards[t].copy_(rew)
                self.terminated[t].copy_(term)
                self.truncated[t].copy_(trunc)
                self.dones[t].copy_(term | trunc)
                # every row, ended or not: rows of envs that did not end are stale and never read by the GAE kernel
                self.final_values[t].copy_(value_fn(info["final_observation"]).reshape(N))
            self.last_values.copy_(value_fn(obs).reshape(N))
        self._last_obs = obs
        self._values_collected = True
        return all_reduce_stats(env.stats_tensor())

    def _collect_fused(self, policy) -> Dict[str, Any]:
        """The rollout of an ActorCriticPolicy: per step one stg_policy_act_f32 launch writes observations[t], actions[t]
        (raw samples, what evaluate_actions trains on), values[t], log_probs[t] and the env actions, the env steps on those,
        and one stg_policy_value_f32 launch computes final_values[t] on the rows of the envs that ended. The weights are
        packed once per rollout; nothing waits on the host."""
        env, N = self.env, self.env.num_envs
        torch = _lib.require_cuda()
        if torch.device(env.device) != policy.log_std.device or policy.num_envs != N:
            raise ValueError("the policy was built for another env (device or num_envs differ)")
        self._values_collected = self._advantages_computed = False
        if getattr(self, "_env_actions", None) is None:      # the env actions [N,2], allocated by the first fused collect
            self._env_actions = torch.empty(N, 2, dtype=torch.float32, device=env.device)
        if self._last_obs is None:
            self._last_obs, _ = env.reset()
        obs = self._last_obs
        lib = _lib.load()
        with _lib.device_guard(torch, env.device):
            w = policy.pack_weights()
            act, val = policy._args(w, N), policy._args(w, N)
            act.d_env_action = self._env_actions.data_ptr()
            for t in range(self.n_steps):
                act.d_obs = obs.data_ptr()
                act.d_obs_copy = self.observations[t].data_ptr() if self.store_observations else None
                act.d_action, act.d_value = self.actions[t].data_ptr(), self.values[t].data_ptr()
                act.d_log_prob = self.log_probs[t].data_ptr()
                policy._set_draw(act, False)
                _lib.check(lib.stg_policy_act_f32(C.byref(act), env._stream()), "stg_policy_act_f32")
                obs, rew, term, trunc, info = env.step(self._env_actions)
                self.rewards[t].copy_(rew)
                self.terminated[t].copy_(term)
                self.truncated[t].copy_(trunc)
                self.dones[t].copy_(term | trunc)
                val.d_obs, val.d_mask = info["final_observation"].data_ptr(), self.dones[t].data_ptr()
                val.d_value = self.final_values[t].data_ptr()
                _lib.check(lib.stg_policy_value_f32(C.byref(val), env._stream()), "stg_policy_value_f32")
            policy.predict_values(obs, out=self.last_values)
        self._last_obs = obs
        self._values_collected = True
        return all_reduce_stats(env.stats_tensor())

    def compute_returns_and_advantage(self, gamma: float = 0.99, gae_lambda: float = 0.95) -> None:
        """GAE(gamma, gae_lambda) over the stored rollout into `advantages` and `returns` (SB3's
        RolloutBuffer.compute_returns_and_advantage in float32, truncated episodes bootstrapped with `final_values`), one
        launch of stg_rollout_gae_f32 on the env's current stream."""
        if not (self.store_values and self._values_collected):
            raise RuntimeError("compute_returns_and_advantage needs a collector with store_values=True and a collect() first")
        torch = self.env._torch
        a = _lib.StgGaeArgs()
        a.d_reward, a.d_value = self.rewards.data_ptr(), self.values.data_ptr()
        a.d_terminated, a.d_truncated = self.terminated.data_ptr(), self.truncated.data_ptr()
        a.d_final_value, a.d_last_value = self.final_values.data_ptr(), self.last_values.data_ptr()
        a.d_advantage, a.d_return = self.advantages.data_ptr(), self.returns.data_ptr()
        # NumPy's `python_float * float32_array` rounds the scalar to float32 first; gamma * gae_lambda is a double product
        a.gamma, a.gamma_lambda = float(np.float32(gamma)), float(np.float32(gamma * gae_lambda))
        a.n_steps, a.n_envs = self.n_steps, self.env.num_envs
        with _lib.device_guard(torch, self.env.device):
            _lib.check(_lib.load().stg_rollout_gae_f32(C.byref(a), self.env._stream()), "stg_rollout_gae_f32")
        self._advantages_computed = True

    def get(self, batch_size: Optional[int] = None) -> Iterator[RolloutBufferSamples]:
        """One epoch of shuffled minibatches over the n_steps * num_envs stored samples, like SB3's RolloutBuffer.get:
        `RolloutBufferSamples(observations [B,12], actions [B,2], old_values [B], old_log_prob [B], advantages [B],
        returns [B])`, float32 on the env's device. `batch_size=None` yields the whole rollout as one batch; otherwise
        consecutive slices of one permutation, the last one possibly smaller. Every call draws a new permutation: that of
        epoch e = the number of earlier get() calls on this collector, keyed by `minibatch_round_keys(env.rng_seed,
        env.env_offset, e)`. Each batch is one launch of stg_rollout_minibatch_f32 (K7) on the env's current stream into
        newly allocated tensors (one allocation per batch, split into the six fields), so batches kept by the caller are
        never overwritten; iterating never synchronises with the host. Needs store_values=True, store_observations=True
        and compute_returns_and_advantage() after the last collect(); the arguments are checked when get() is called."""
        self._check_get()
        total = self.n_steps * self.env.num_envs
        batch_size = total if batch_size is None else int(batch_size)
        if batch_size <= 0:
            raise ValueError(f"batch_size must be positive, got {batch_size}")
        keys = minibatch_round_keys(self.env.rng_seed, self.env.env_offset, self._epoch)
        self._epoch += 1
        return self._minibatches(keys, batch_size)

    def _check_get(self) -> None:
        if not (self.store_values and self.store_observations):
            raise ValueError("get() needs a collector with store_values=True and store_observations=True")
        if not self._advantages_computed:
            raise RuntimeError("get() needs compute_returns_and_advantage() after the last collect()")

    def rollout_samples(self) -> RolloutBufferSamples:
        """The whole stored rollout as one `RolloutBufferSamples` of flat views: n_steps * num_envs rows in (step, env) order
        (row t * num_envs + i is env i at step t), with no copy, no permutation and no launch. The views alias the collector's
        planes, so the next collect() overwrites them. Preconditions and errors are those of get().

        This is A2C's batch. SB3's A2C.train() iterates `get(batch_size=None)`, which permutes the rows, but its update is
        one sum over all of them: a permutation changes only the order of that sum, which K10 fixes anyway, so the rows are
        used where they lie."""
        self._check_get()
        total = self.n_steps * self.env.num_envs
        return RolloutBufferSamples(self.observations.view(total, _lib.OBS_DIM), self.actions.view(total, 2),
                                    self.values.view(total), self.log_probs.view(total), self.advantages.view(total),
                                    self.returns.view(total))

    def _minibatches(self, keys: List[int], batch_size: int) -> Iterator[RolloutBufferSamples]:
        env = self.env
        torch, N = env._torch, env.num_envs
        total = self.n_steps * N
        a = _lib.StgMinibatchArgs()
        a.d_obs, a.d_action = self.observations.data_ptr(), self.actions.data_ptr()
        a.d_value, a.d_log_prob = self.values.data_ptr(), self.log_probs.data_ptr()
        a.d_advantage, a.d_return = self.advantages.data_ptr(), self.returns.data_ptr()
        a.round_keys[:] = keys
        a.n_steps, a.n_envs = self.n_steps, N
        launch = _lib.load().stg_rollout_minibatch_f32
        for start in range(0, total, batch_size):
            B = min(batch_size, total - start)
            with _lib.device_guard(torch, env.device):
                buf = torch.empty(18 * B, dtype=torch.float32, device=env.device)
                base = buf.data_ptr()           # observations first: 16-B aligned like every allocation
                a.d_obs_out, a.d_action_out, a.d_value_out = base, base + 48 * B, base + 56 * B
                a.d_log_prob_out, a.d_advantage_out, a.d_return_out = base + 60 * B, base + 64 * B, base + 68 * B
                a.start, a.batch = start, B
                _lib.check(launch(C.byref(a), env._stream()), "stg_rollout_minibatch_f32")
            obs, act, val, logp, adv, ret = buf.split([12 * B, 2 * B, B, B, B, B])
            yield RolloutBufferSamples(obs.view(B, _lib.OBS_DIM), act.view(B, 2), val, logp, adv, ret)
