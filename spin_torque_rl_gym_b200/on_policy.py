"""What `PPO` and `A2C` share: the policy built from its name, SB3's `learn()` loop over the fused rollout, the data-parallel
start-up (rank checks and the broadcast of rank 0's weights and optimiser state) and the explained variance of the rollout,
gathered across the ranks with data_parallel."""
from __future__ import annotations

import math
from typing import Any, Callable, Dict, List, Optional, Union

import torch

from . import _lib
from .parallel import all_gather_moments, all_reduce_stats, episode_metrics, world_size
from .policy import ActorCriticPolicy, _adv_moments

Schedule = Union[float, Callable[[float], float]]


def _schedule(value: Optional[Schedule]) -> Optional[Callable[[float], float]]:
    """SB3's get_schedule_fn: a callable of progress_remaining is kept, a number becomes a constant one."""
    if value is None or callable(value):
        return value
    v = float(value)
    return lambda _: v


class OnPolicyAlgorithm:
    """The base of PPO and A2C. A subclass's constructor calls `_ranks`, `_policy` and `_check_data_parallel` to validate,
    sets `env`, `policy` (with its optimizer), `rollout_buffer`, `n_steps`, `gamma`, `gae_lambda`, `data_parallel` and
    `ranks`, then calls `_start`; it implements `train()` and `_rank_agreement()`."""

    _NAME = "OnPolicyAlgorithm"

    # ---- construction ------------------------------------------------------------------------------------------------------
    @classmethod
    def _ranks(cls, data_parallel: bool) -> int:
        """The world size; NotImplementedError for more than one rank without data_parallel."""
        ranks = world_size()
        if ranks > 1 and not data_parallel:
            raise NotImplementedError(f"{cls._NAME}(data_parallel=False) trains on one rank; under a process group of world "
                                      f"size {ranks} pass data_parallel=True to train one policy across the ranks")
        return ranks

    @staticmethod
    def _policy(policy: Union[str, ActorCriticPolicy], env, seed: Optional[int],
                policy_kwargs: Optional[Dict[str, Any]]) -> ActorCriticPolicy:
        """"MlpPolicy" built for `env` after torch.manual_seed(seed), or a given ActorCriticPolicy checked against `env`."""
        if isinstance(policy, str):
            if policy != "MlpPolicy":
                raise ValueError(f"the only policy name is 'MlpPolicy', got {policy!r}")
            if seed is not None:
                torch.manual_seed(seed)
            return ActorCriticPolicy(env, seed=seed, **(policy_kwargs or {}))
        if not isinstance(policy, ActorCriticPolicy):
            raise ValueError(f"policy must be 'MlpPolicy' or an ActorCriticPolicy, got {type(policy).__name__}")
        if policy_kwargs:
            raise ValueError("policy_kwargs apply to 'MlpPolicy' only")
        if policy.num_envs != env.num_envs or policy.log_std.device != torch.device(env.device):
            raise ValueError("the policy was built for another env (device or num_envs differ)")
        return policy

    @classmethod
    def _check_data_parallel(cls, env, ranks: int, batch_size: Optional[int] = None) -> None:
        """The ValueErrors of data_parallel=True that need no collective."""
        from .envs.vec_normalize import VecNormalize
        if batch_size is not None and batch_size % ranks:
            raise ValueError(f"data-parallel {cls._NAME} needs batch_size divisible by the world size {ranks}, got "
                             f"{batch_size}")
        if isinstance(env, VecNormalize) and not env._syncing():
            raise ValueError(f"data-parallel {cls._NAME} needs a VecNormalize that shares its statistics across the ranks "
                             "(sync=None or True), or the ranks would normalise their observations differently")

    def _start(self) -> None:
        """The counters and, with more than one rank, the rank checks and the broadcast; then the first statistics read."""
        self.num_timesteps = 0
        self._n_updates = 0
        self._total_timesteps = 0
        self._current_progress_remaining = 1.0
        if self.ranks > 1:
            self._synchronise_ranks()
        self._last_stats = all_reduce_stats(self.env.stats_tensor())
        self.log_history: List[Dict[str, float]] = []

    def _rank_agreement(self) -> Dict[str, int]:
        """The integers every rank must agree on, by name."""
        raise NotImplementedError

    def _synchronise_ranks(self) -> None:
        """Data-parallel start-up: check that the ranks agree on `_rank_agreement()`, then broadcast rank 0's parameters and
        optimiser state."""
        import torch.distributed as dist
        pol, opt = self.policy, self.policy.optimizer
        agree = self._rank_agreement()
        mine = torch.tensor(list(agree.values()), dtype=torch.int64, device=pol.log_std.device)
        every = all_gather_moments(mine).cpu()
        if not bool((every == every[0]).all()):
            raise ValueError(f"data-parallel {self._NAME} needs the same {', '.join(agree)} on every rank, got "
                             f"{every.tolist()} (rows: ranks)")
        with torch.no_grad():
            for t in [p.data for p in pol.parameters()] + opt.state_tensors():
                dist.broadcast(t, src=0)

    def _seed_int64(self) -> int:
        """The policy's 64-bit seed as an int64."""
        seed = self.policy.seed
        return seed - (1 << 64) if seed >= 1 << 63 else seed

    # ---- SB3's loop --------------------------------------------------------------------------------------------------------
    def learn(self, total_timesteps: int, reset_num_timesteps: bool = True):
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
            self.num_timesteps += self.n_steps * self.env.num_envs * self.ranks
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
        raise NotImplementedError

    @torch.no_grad()
    def _rollout_explained_variance(self):
        """SB3's explained_variance(values, returns) of the stored rollout as a 0-d device tensor (no host read): population
        variances, NaN when Var(returns) is 0; with data_parallel from FP64 moments gathered across the ranks."""
        col = self.rollout_buffer
        values, returns = col.values.reshape(-1), col.returns.reshape(-1)
        if self.data_parallel:
            moments = all_gather_moments(torch.cat([_adv_moments(returns), _adv_moments(returns - values)]))
            return _explained_variance(moments.reshape(-1, 2, _lib.PPO_ADV_MOMENTS))
        var_y = returns.var(correction=0)
        return torch.where(var_y == 0, math.nan, 1 - (returns - values).var(correction=0) / var_y)

    def predict(self, obs, deterministic: bool = False):
        """The policy's predict: (env actions, None)."""
        return self.policy.predict(obs, deterministic=deterministic)


def _explained_variance(moments):
    """1 - Var(returns - values) / Var(returns) (population variances, NaN when Var(returns) is 0) from moments [G, 2, 3]:
    per rank the FP64 (n, mean, M2) of the returns and of returns - values. Each is folded in rank order with K12's merge
    (stg_ppo_adv_merge_f32 gives torch's std with correction 1, whose square ratio is the ratio of the M2)."""
    from .policy import _adv_stats
    std_y, std_d = _adv_stats(moments[:, 0])[1].double(), _adv_stats(moments[:, 1])[1].double()
    return torch.where(std_y == 0, math.nan, 1 - (std_d * std_d) / (std_y * std_y))
