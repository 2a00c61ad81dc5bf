"""`PPO`: Stable-Baselines3's PPO (`learn()` / `train()`) on the GPU vector env, built from the fused parts: the rollout of
RolloutCollector with ActorCriticPolicy (K9), GAE (K6), shuffled minibatches (K7), the minibatch loss and gradient (K10) and
the clipped Adam step with its device-side target_kl gate (K11, ClippedAdam)."""
from __future__ import annotations

import math
from typing import Any, Callable, Dict, List, Optional, Union

import torch

from . import _lib
from .envs import RolloutCollector
from .optim import ClippedAdam
from .parallel import all_reduce_stats, episode_metrics
from .policy import ActorCriticPolicy

Schedule = Union[float, Callable[[float], float]]
_LOG = _lib.ADAM_LOG_SLOTS


def _schedule(value: Optional[Schedule]) -> Optional[Callable[[float], float]]:
    """SB3's get_schedule_fn: a callable of progress_remaining is kept, a number becomes a constant one."""
    if value is None or callable(value):
        return value
    v = float(value)
    return lambda _: v


class PPO:
    """`PPO(policy, env, learning_rate=3e-4, n_steps=2048, batch_size=64, n_epochs=10, gamma=0.99, gae_lambda=0.95,
    clip_range=0.2, clip_range_vf=None, normalize_advantage=True, ent_coef=0.0, vf_coef=0.5, max_grad_norm=0.5,
    target_kl=None, seed=None, policy_kwargs=None)`: SB3's PPO signature and defaults for a SpinTorqueVectorEnv (or a
    VecNormalize around one) with `autoreset=True`, on its device.

    `policy` is "MlpPolicy" (an `ActorCriticPolicy(env, seed=seed, **policy_kwargs)` built after `torch.manual_seed(seed)` when
    a seed is given) or an ActorCriticPolicy built for `env`. `self.rollout_buffer` is a `RolloutCollector(env, n_steps,
    store_values=True)` and `self.policy.optimizer` a ClippedAdam, where SB3 keeps them. `learning_rate`, `clip_range` and
    `clip_range_vf` are numbers or callables of SB3's `progress_remaining`.

    One `learn()` iteration synchronises with the host twice: the episode statistics read by `collect()` and the one read of
    the training log at the end of `train()`; with `target_kl` once more per epoch run, to read the gate. Minibatches enqueued
    after the gate closed in that epoch are computed and then ignored by the optimiser kernel. Each `train()` returns and
    appends to `self.log_history` a dict with SB3's logger keys (`train/...`); `learn()` adds `rollout/...` (of the rollout
    just collected, from the difference of the env's cumulative statistics) and `time/...` to it.

    Raises ValueError for `batch_size < 2` with `normalize_advantage` (SB3 asserts it), a policy of another kind, or an env the
    collector rejects; NotImplementedError under a process group of world size > 1 (each rank would train its own policy)."""

    def __init__(self, policy: Union[str, ActorCriticPolicy], env, learning_rate: Schedule = 3e-4, n_steps: int = 2048,
                 batch_size: int = 64, n_epochs: int = 10, gamma: float = 0.99, gae_lambda: float = 0.95,
                 clip_range: Schedule = 0.2, clip_range_vf: Optional[Schedule] = None, normalize_advantage: bool = True,
                 ent_coef: float = 0.0, vf_coef: float = 0.5, max_grad_norm: Optional[float] = 0.5,
                 target_kl: Optional[float] = None, seed: Optional[int] = None, policy_kwargs: Optional[Dict[str, Any]] = None):
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
            raise NotImplementedError("PPO trains on one rank; data-parallel training across ranks is not implemented")
        if n_steps < 1 or n_epochs < 1 or batch_size < 1:
            raise ValueError(f"n_steps, n_epochs and batch_size must be positive, got {n_steps}, {n_epochs}, {batch_size}")
        if normalize_advantage and batch_size < 2:
            raise ValueError("batch_size must be greater than 1 with normalize_advantage=True (the advantage std of one sample "
                             "is NaN)")
        if isinstance(policy, str):
            if policy != "MlpPolicy":
                raise ValueError(f"the only policy name is 'MlpPolicy', got {policy!r}")
            if seed is not None:
                torch.manual_seed(seed)
            policy = ActorCriticPolicy(env, seed=seed, **(policy_kwargs or {}))
        elif not isinstance(policy, ActorCriticPolicy):
            raise ValueError(f"policy must be 'MlpPolicy' or an ActorCriticPolicy, got {type(policy).__name__}")
        elif policy_kwargs:
            raise ValueError("policy_kwargs apply to 'MlpPolicy' only")
        elif policy.num_envs != env.num_envs or policy.log_std.device != torch.device(env.device):
            raise ValueError("the policy was built for another env (device or num_envs differ)")
        self.env, self.policy = env, policy
        self.n_steps, self.batch_size, self.n_epochs = int(n_steps), int(batch_size), int(n_epochs)
        self.gamma, self.gae_lambda = gamma, gae_lambda
        self.lr_schedule = _schedule(learning_rate)
        self.clip_range, self.clip_range_vf = _schedule(clip_range), _schedule(clip_range_vf)
        self.normalize_advantage, self.ent_coef, self.vf_coef = normalize_advantage, ent_coef, vf_coef
        self.max_grad_norm, self.target_kl, self.seed = max_grad_norm, target_kl, seed
        self.rollout_buffer = RolloutCollector(env, self.n_steps, store_values=True)
        policy.optimizer = ClippedAdam(policy, lr=self.lr_schedule(1.0), eps=1e-5, max_grad_norm=max_grad_norm)
        dev = policy.log_std.device
        self._log = torch.zeros(_lib.ADAM_LOG, dtype=torch.float64, device=dev)
        self._gate = torch.ones(1, dtype=torch.int32, device=dev)
        self.num_timesteps = 0
        self._n_updates = 0
        self._total_timesteps = 0
        self._current_progress_remaining = 1.0
        self._last_stats = all_reduce_stats(env.stats_tensor())
        self.log_history: List[Dict[str, float]] = []

    def learn(self, total_timesteps: int, reset_num_timesteps: bool = True) -> "PPO":
        """SB3's learn(): until num_timesteps reaches total_timesteps, collect n_steps x num_envs samples on the fused path,
        update progress_remaining, compute GAE and train(). With reset_num_timesteps=False, total_timesteps counts from the
        current num_timesteps, as in SB3."""
        if reset_num_timesteps:
            self.num_timesteps = 0
        else:
            total_timesteps += self.num_timesteps
        self._total_timesteps = total_timesteps
        iteration = 0
        col = self.rollout_buffer
        while self.num_timesteps < total_timesteps:
            stats = col.collect(self.policy)
            self.num_timesteps += self.n_steps * self.env.num_envs
            iteration += 1
            self._current_progress_remaining = 1.0 - float(self.num_timesteps) / float(total_timesteps)
            col.compute_returns_and_advantage(self.gamma, self.gae_lambda)
            rollout = episode_metrics({k: stats[k] - self._last_stats[k] for k in _lib.STAT_NAMES})
            self._last_stats = stats
            logs = self.train()
            for k in ("success_rate", "mean_episode_length", "mean_reward", "episodes"):
                logs[f"rollout/{k}"] = rollout[k]
            logs["time/iterations"] = iteration
            logs["time/total_timesteps"] = self.num_timesteps
        return self

    def train(self) -> Dict[str, float]:
        """SB3's train() over the collected rollout: n_epochs epochs of get(batch_size) minibatches, each one ppo_backward
        launch and one ClippedAdam launch that logs its losses and applies the gate. Returns the logged dict."""
        pol, opt, col = self.policy, self.policy.optimizer, self.rollout_buffer
        progress = self._current_progress_remaining
        lr = float(self.lr_schedule(progress))
        for group in opt.param_groups:
            group["lr"] = lr
        clip_range = float(self.clip_range(progress))
        clip_range_vf = None if self.clip_range_vf is None else float(self.clip_range_vf(progress))
        log, gate = self._log, self._gate
        log.zero_()
        gate.fill_(1)
        for _ in range(self.n_epochs):
            log[_LOG["EPOCH_KL"]:_LOG["EPOCH_COUNT"] + 1].zero_()
            for batch in col.get(self.batch_size):
                losses = pol.ppo_backward(batch, clip_range, clip_range_vf, self.ent_coef, self.vf_coef,
                                          self.normalize_advantage)
                opt._step(losses, gate, log, self.target_kl)
            self._n_updates += 1
            if self.target_kl is not None and int(gate.item()) == 0:
                break
        with torch.no_grad():
            values, returns = col.values.reshape(-1), col.returns.reshape(-1)
            var_y = returns.var(correction=0)
            explained_var = torch.where(var_y == 0, math.nan, 1 - (returns - values).var(correction=0) / var_y)
            count = log[_LOG["COUNT"]]
            row = torch.stack([log[_LOG["ENTROPY"]] / count, log[_LOG["PG"]] / count, log[_LOG["VALUE"]] / count,
                               log[_LOG["EPOCH_KL"]] / log[_LOG["EPOCH_COUNT"]], log[_LOG["CLIP"]] / count,
                               log[_LOG["LAST_LOSS"]], explained_var.double(), pol.log_std.exp().mean().double()])
        vals = row.cpu().tolist()
        names = ("entropy_loss", "policy_gradient_loss", "value_loss", "approx_kl", "clip_fraction", "loss",
                 "explained_variance", "std")
        logs = {f"train/{k}": v for k, v in zip(names, vals)}
        logs["train/n_updates"] = self._n_updates
        logs["train/clip_range"] = clip_range
        if clip_range_vf is not None:
            logs["train/clip_range_vf"] = clip_range_vf
        logs["train/learning_rate"] = lr
        self.log_history.append(logs)
        return logs

    def predict(self, obs, deterministic: bool = False):
        """The policy's predict: (env actions, None)."""
        return self.policy.predict(obs, deterministic=deterministic)
