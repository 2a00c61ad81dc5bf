"""`A2C`: Stable-Baselines3's A2C (`learn()` / `train()`) on the GPU vector env, built from the fused parts: the rollout of
RolloutCollector with ActorCriticPolicy (K9), GAE (K6), the loss and gradient of the whole rollout (K10's A2C instance) and
the clipped RMSprop step (K13, ClippedRMSprop) or the clipped Adam step (K11, ClippedAdam)."""
from __future__ import annotations

from typing import Any, Dict, Optional, Union

import torch

from .envs import RolloutCollector
from .on_policy import OnPolicyAlgorithm, Schedule, _schedule
from .optim import ClippedAdam, ClippedRMSprop
from .policy import ActorCriticPolicy


class A2C(OnPolicyAlgorithm):
    """`A2C(policy, env, learning_rate=7e-4, n_steps=5, gamma=0.99, gae_lambda=1.0, ent_coef=0.0, vf_coef=0.5,
    max_grad_norm=0.5, rms_prop_eps=1e-5, use_rms_prop=True, normalize_advantage=False, seed=None, policy_kwargs=None,
    data_parallel=False)`: SB3's A2C signature and defaults for a SpinTorqueVectorEnv (or a VecNormalize around one) with
    `autoreset=True`, on its device. gSDE, other action spaces and rollout buffer classes are not supported.

    `policy` is "MlpPolicy" or an ActorCriticPolicy built for `env`, as for PPO. `self.rollout_buffer` is a
    `RolloutCollector(env, n_steps, store_values=True)`; `self.policy.optimizer` is SB3's choice: with `use_rms_prop` a
    `ClippedRMSprop(alpha=0.99, eps=rms_prop_eps)`, else a `ClippedAdam(eps=1e-5)`, both clipping to `max_grad_norm`.
    `learning_rate` is a number or a callable of SB3's `progress_remaining`.

    `train()` is one update over the whole rollout: one `a2c_backward(rollout_samples())` and one optimiser step. SB3 draws
    that batch through `get(batch_size=None)`, a permutation of the same rows; the update is one sum over them, so only its
    order differs. One `learn()` iteration synchronises with the host twice: the episode statistics read by `collect()` and
    one read of the losses at the end of `train()`. Each `train()` returns and appends to `self.log_history` a dict with SB3's
    A2C logger keys (`train/n_updates`, `explained_variance`, `entropy_loss`, `policy_loss`, `value_loss`, `std`,
    `learning_rate`); `learn()` adds `rollout/...` and `time/...` as PPO's does.

    `data_parallel=True` trains one policy over the G ranks of a process group (K12), each rank holding its shard of the envs
    with the same `num_envs`: the update is that of the union of the ranks' rollouts, bit-identical on every rank, with the
    advantages normalised by the statistics of the union when `normalize_advantage`. The constructor broadcasts rank 0's
    parameters and optimiser state and checks that the ranks agree on `num_envs` and the policy seed; `num_timesteps` and
    `explained_variance` are global. Without a process group, or with world size 1, it runs the same kernels with no
    collective.

    Raises ValueError for `n_steps < 1`, a policy of another kind or an env the collector rejects, and with
    `data_parallel=True` for a VecNormalize that does not share its statistics across the ranks or ranks that disagree;
    NotImplementedError under a process group of world size > 1 without `data_parallel=True`."""

    _NAME = "A2C"

    def __init__(self, policy: Union[str, ActorCriticPolicy], env, learning_rate: Schedule = 7e-4, n_steps: int = 5,
                 gamma: float = 0.99, gae_lambda: float = 1.0, ent_coef: float = 0.0, vf_coef: float = 0.5,
                 max_grad_norm: Optional[float] = 0.5, rms_prop_eps: float = 1e-5, use_rms_prop: bool = True,
                 normalize_advantage: bool = False, seed: Optional[int] = None,
                 policy_kwargs: Optional[Dict[str, Any]] = None, data_parallel: bool = False):
        ranks = self._ranks(data_parallel)
        if n_steps < 1:
            raise ValueError(f"n_steps must be positive, got {n_steps}")
        policy = self._policy(policy, env, seed, policy_kwargs)
        if data_parallel:
            self._check_data_parallel(env, ranks)
        self.data_parallel, self.ranks = bool(data_parallel), ranks if data_parallel else 1
        self.env, self.policy = env, policy
        self.n_steps = int(n_steps)
        self.gamma, self.gae_lambda = gamma, gae_lambda
        self.lr_schedule = _schedule(learning_rate)
        self.normalize_advantage, self.ent_coef, self.vf_coef = normalize_advantage, ent_coef, vf_coef
        self.max_grad_norm, self.rms_prop_eps, self.use_rms_prop, self.seed = max_grad_norm, rms_prop_eps, use_rms_prop, seed
        self.rollout_buffer = RolloutCollector(env, self.n_steps, store_values=True)
        lr = self.lr_schedule(1.0)
        if use_rms_prop:
            policy.optimizer = ClippedRMSprop(policy, lr=lr, alpha=0.99, eps=rms_prop_eps, max_grad_norm=max_grad_norm)
        else:
            policy.optimizer = ClippedAdam(policy, lr=lr, eps=1e-5, max_grad_norm=max_grad_norm)
        self._start()

    def _rank_agreement(self) -> Dict[str, int]:
        return {"num_envs": self.env.num_envs, "policy seed": self._seed_int64()}

    def train(self) -> Dict[str, float]:
        """SB3's A2C.train() over the collected rollout: one a2c_backward launch over every row and one optimiser launch.
        Returns the logged dict."""
        pol, opt = self.policy, self.policy.optimizer
        lr = float(self.lr_schedule(self._current_progress_remaining))
        for group in opt.param_groups:
            group["lr"] = lr
        losses = pol.a2c_backward(self.rollout_buffer.rollout_samples(), self.ent_coef, self.vf_coef,
                                  self.normalize_advantage, data_parallel=self.data_parallel)
        opt.step()
        self._n_updates += 1
        explained_var = self._rollout_explained_variance()
        with torch.no_grad():
            row = torch.stack([explained_var.double(), losses.entropy_loss.double(), losses.policy_loss.double(),
                               losses.value_loss.double(), pol.log_std.exp().mean().double()])
        vals = row.cpu().tolist()
        logs = {"train/n_updates": self._n_updates}
        logs.update({f"train/{k}": v for k, v in zip(("explained_variance", "entropy_loss", "policy_loss", "value_loss",
                                                       "std"), vals)})
        logs["train/learning_rate"] = lr
        self.log_history.append(logs)
        return logs
