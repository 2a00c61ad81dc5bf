"""VecNormalize on the GPU: running observation and return normalisation for SpinTorqueVectorEnv (K8).

Stable-Baselines3's VecNormalize is NumPy on the host and wraps only a VecEnv, so it can neither keep up with 10^5..10^6 envs
nor sit under RolloutCollector. This wrapper keeps SB3's semantics (VecNormalize.step_wait / reset / normalize_obs /
normalize_reward, RunningMeanStd) with the statistics in HBM and three kernel launches per step (include/stg.h, K8), and has
the interface of the vector env that RolloutCollector and SB3VecEnvAdapter use, so both work on it unchanged."""
from __future__ import annotations

import ctypes as C
from typing import Any, Dict, Optional

from .. import _lib
from ..parallel import all_gather_moments


class RunningMeanStdView:
    """SB3's RunningMeanStd fields as float64 device tensors: views into the wrapper's statistics buffer (reading them does
    not synchronise; they change in place with every training step)."""

    def __init__(self, mean, var, count):
        self.mean, self.var, self.count = mean, var, count

    def __repr__(self) -> str:
        return f"RunningMeanStdView(shape={tuple(self.mean.shape)})"


class VecNormalize:
    """`VecNormalize(venv, training=True, norm_obs=True, norm_reward=True, clip_obs=10.0, clip_reward=10.0, gamma=0.99,
    epsilon=1e-8, sync=None)` around a SpinTorqueVectorEnv with device outputs.

    `step(actions)` returns (obs [N,12] f32, reward [N] f64, terminated, truncated, info) like the env, with normalised
    observations, rewards and `info["final_observation"]` rows, in SB3's order: obs_rms is updated with the N returned
    observations (training and norm_obs), the observations and the final observations of ended envs are normalised with the
    updated statistics, `returns = returns * gamma + reward` updates ret_rms (training), the reward is divided by
    sqrt(ret_rms.var + epsilon) (norm_reward), and the returns of ended envs are zeroed. Arithmetic is float64 in SB3's
    expression order; the batch moments accumulate in FP64 (SB3's np.mean / np.var on float32 observations accumulate in float32).
    The outputs are the wrapper's persistent tensors, overwritten by the next step, and nothing in `step` or `reset` waits on
    the host.

    `sync=None` shares the statistics across the ranks of an initialised process group with world size > 1 (one 216-B
    all-gather per step: every rank folds the same moment vectors in rank order, so all ranks hold bit-identical statistics);
    `sync=False` keeps them per rank; `sync=True` gathers whenever a process group is initialised."""

    def __init__(self, venv, training: bool = True, norm_obs: bool = True, norm_reward: bool = True, clip_obs: float = 10.0,
                 clip_reward: float = 10.0, gamma: float = 0.99, epsilon: float = 1e-8, sync: Optional[bool] = None):
        torch = _lib.require_cuda()
        if getattr(venv, "host_outputs", False):
            raise ValueError("VecNormalize needs the env's outputs on the device (host_outputs=False)")
        if tuple(venv.single_observation_space.shape) != (_lib.OBS_DIM,):
            raise ValueError("VecNormalize supports the 12-float SpinTorque-v0 observation only")
        self.venv = venv
        self._torch = torch
        self._lib = _lib.load()
        self.num_envs, self.device = venv.num_envs, venv.device
        self.training, self.norm_obs, self.norm_reward = bool(training), bool(norm_obs), bool(norm_reward)
        self.clip_obs, self.clip_reward = float(clip_obs), float(clip_reward)
        self.gamma, self.epsilon = float(gamma), float(epsilon)
        self.sync = sync
        N, dev, f64 = self.num_envs, self.device, torch.float64
        with torch.cuda.device(dev):
            self._stats = torch.zeros(_lib.VECNORM_STATS, dtype=f64, device=dev)
            self._reset_stats()
            self._returns = torch.zeros(N, dtype=f64, device=dev)
            self._moments = torch.zeros(_lib.VECNORM_MOMENTS, dtype=f64, device=dev)
            self._work = torch.zeros(_lib.VECNORM_WORK_DOUBLES, dtype=f64, device=dev)   # last word: CTA counter, kept 0
            self._obs = torch.zeros(N, _lib.OBS_DIM, dtype=torch.float32, device=dev)
            self._final_obs = torch.zeros(N, _lib.OBS_DIM, dtype=torch.float32, device=dev)
            self._reward = torch.zeros(N, dtype=f64, device=dev)
        s = self._stats
        self.obs_rms = RunningMeanStdView(s[0:12], s[12:24], s[24])
        self.ret_rms = RunningMeanStdView(s[25], s[26], s[27])
        self._raw_obs = self._raw_reward = None
        self._gathered = None                 # keeps the gathered [G, 27] stack alive until the merge has been enqueued

    def _reset_stats(self) -> None:
        s = self._stats                       # RunningMeanStd(): mean 0, var 1, count 1e-4
        s.zero_()
        s[12:24] = 1.0
        s[26] = 1.0
        s[24] = s[27] = 1e-4

    # ---- the vector-env interface RolloutCollector and SB3VecEnvAdapter use ------------------------------------------------
    @property
    def autoreset(self) -> bool:
        return self.venv.autoreset

    @property
    def host_outputs(self) -> bool:
        return False

    @property
    def rng_seed(self) -> int:
        return self.venv.rng_seed

    @property
    def env_offset(self) -> int:
        return self.venv.env_offset

    def stats_tensor(self):
        return self.venv.stats_tensor()

    def _stream(self) -> int:
        return self.venv._stream()

    def close(self) -> None:
        self.venv.close()

    def capture_step(self, actions):
        """Not supported: forwarding it would capture the wrapped env's raw step without the normalisation."""
        raise NotImplementedError("VecNormalize has no capture_step: capture of the normalised step is not implemented")

    def __getattr__(self, name: str):
        """Public attributes the wrapper does not define (spaces, max_steps, episode_stats, ...) come from the wrapped env.
        Private ones do not: the env's state and output buffers behind them (what torch_ops.env_step reads, for one) would
        step the env without the normalisation."""
        if name == "venv" or name.startswith("_"):
            raise AttributeError(f"VecNormalize does not forward {name!r}; the wrapped env is .venv")
        return getattr(self.venv, name)

    # ---- K8 launches -------------------------------------------------------------------------------------------------------
    def _args(self, n: int, flags: int) -> _lib.StgVecNormArgs:
        a = _lib.StgVecNormArgs()
        a.d_stats, a.d_moments, a.d_work = self._stats.data_ptr(), self._moments.data_ptr(), self._work.data_ptr()
        a.gamma, a.epsilon, a.clip_obs, a.clip_reward = self.gamma, self.epsilon, self.clip_obs, self.clip_reward
        a.n_envs, a.n_ranks, a.flags = n, 1, flags
        return a

    def _flags(self) -> int:
        return ((_lib.VECNORM_TRAINING if self.training else 0) | (_lib.VECNORM_NORM_OBS if self.norm_obs else 0)
                | (_lib.VECNORM_NORM_REWARD if self.norm_reward else 0))

    def _syncing(self) -> bool:
        if self.sync is False:
            return False
        import torch.distributed as dist
        if not (dist.is_available() and dist.is_initialized()):
            return False
        return bool(self.sync) or dist.get_world_size() > 1

    def _update(self, a: _lib.StgVecNormArgs, stream: int) -> None:
        """moments -> (all-gather across ranks) -> merge into the statistics, all on `stream`."""
        _lib.check(self._lib.stg_vecnorm_moments_f32(C.byref(a), stream), "stg_vecnorm_moments_f32")
        moments = self._moments
        if self._syncing():
            moments = all_gather_moments(self._moments).contiguous()
        self._gathered = moments
        a.d_moments, a.n_ranks = moments.data_ptr(), moments.numel() // _lib.VECNORM_MOMENTS
        _lib.check(self._lib.stg_vecnorm_merge_f64(C.byref(a), stream), "stg_vecnorm_merge_f64")

    # ---- gymnasium-VectorEnv-style API -------------------------------------------------------------------------------------
    def reset(self, *, seed: Optional[int] = None, options: Optional[Dict[str, Any]] = None, mask=None):
        """Reset the wrapped env and return (normalised obs, info).

        A full reset zeroes every return and, when training with norm_obs, updates obs_rms with the N reset observations (SB3's
        VecNormalize.reset). `reset(mask=...)` zeroes the returns of the masked envs only and does NOT update the statistics:
        the other rows are observations that were already counted when they were returned by the last step."""
        torch = self._torch
        obs, info = self.venv.reset(seed=seed, options=options, mask=mask)
        self._raw_obs = obs
        with _lib.device_guard(torch, self.device):
            stream = self._stream()
            if mask is None:
                self._returns.zero_()
            else:
                mk = torch.as_tensor(mask).to(self.device).to(torch.bool)
                self._returns.masked_fill_(mk, 0.0)
            flags = self._flags()
            if mask is None and self.training and self.norm_obs:
                a = self._args(self.num_envs, flags)
                a.d_obs = obs.data_ptr()
                self._update(a, stream)
            a = self._args(self.num_envs, flags)
            a.d_obs, a.d_obs_out = obs.data_ptr(), self._obs.data_ptr()
            _lib.check(self._lib.stg_vecnorm_apply_f32(C.byref(a), stream), "stg_vecnorm_apply_f32")
        return self._obs, info

    def step(self, actions, noise=None):
        """One env step; see the class docstring for the order of the updates."""
        out = self.venv.step(actions) if noise is None else self.venv.step(actions, noise=noise)
        return self._normalize_step(*out)

    def _normalize_step(self, obs, rew, term, trunc, info):
        """The K8 launches of one step on the wrapped env's outputs (moments, merge when training; apply)."""
        torch = self._torch
        self._raw_obs, self._raw_reward = obs, rew
        final = info.get("final_observation")
        with _lib.device_guard(torch, self.device):
            stream = self._stream()
            flags = self._flags()
            if self.training:
                a = self._args(self.num_envs, flags)
                a.d_obs, a.d_reward, a.d_returns = obs.data_ptr(), rew.data_ptr(), self._returns.data_ptr()
                self._update(a, stream)
            a = self._args(self.num_envs, flags)
            a.d_obs, a.d_obs_out = obs.data_ptr(), self._obs.data_ptr()
            a.d_terminated, a.d_truncated = term.data_ptr(), trunc.data_ptr()
            a.d_reward, a.d_reward_out, a.d_returns = rew.data_ptr(), self._reward.data_ptr(), self._returns.data_ptr()
            if final is not None:
                a.d_final_obs, a.d_final_obs_out = final.data_ptr(), self._final_obs.data_ptr()
            _lib.check(self._lib.stg_vecnorm_apply_f32(C.byref(a), stream), "stg_vecnorm_apply_f32")
        info = dict(info)
        if final is not None:
            info["final_observation"] = self._final_obs
        return self._obs, self._reward, term, trunc, info

    # ---- SB3 accessors -----------------------------------------------------------------------------------------------------
    def get_original_obs(self):
        """The wrapped env's raw observations of the last step or reset. Unlike SB3, which returns a copy, this is the env's
        persistent output tensor (the env's own convention): the next step or reset overwrites it, so clone it to keep it."""
        return self._raw_obs

    def get_original_reward(self):
        """The wrapped env's raw rewards of the last step: the env's persistent output tensor, overwritten by the next step
        (clone it to keep it; SB3 returns a copy)."""
        return self._raw_reward

    def normalize_obs(self, obs):
        """[B,12] observations normalised with the current statistics (not updated): a new float32 tensor."""
        torch = self._torch
        x = torch.as_tensor(obs).to(device=self.device, dtype=torch.float32).reshape(-1, _lib.OBS_DIM).contiguous()
        if x.data_ptr() % 16:
            x = x.clone()
        out = torch.empty_like(x)
        a = self._args(x.shape[0], self._flags())
        a.d_obs, a.d_obs_out = x.data_ptr(), out.data_ptr()
        with _lib.device_guard(torch, self.device):
            _lib.check(self._lib.stg_vecnorm_apply_f32(C.byref(a), self._stream()), "stg_vecnorm_apply_f32")
        return out

    def normalize_reward(self, reward):
        """[B] rewards normalised with the current statistics (not updated): a new float64 tensor."""
        torch = self._torch
        r = torch.as_tensor(reward).to(device=self.device, dtype=torch.float64).reshape(-1).contiguous()
        out = torch.empty_like(r)
        a = self._args(r.shape[0], self._flags())
        a.d_reward, a.d_reward_out = r.data_ptr(), out.data_ptr()
        with _lib.device_guard(torch, self.device):
            _lib.check(self._lib.stg_vecnorm_apply_f32(C.byref(a), self._stream()), "stg_vecnorm_apply_f32")
        return out

    def state_dict(self) -> Dict[str, Any]:
        return {"obs_mean": self.obs_rms.mean.clone(), "obs_var": self.obs_rms.var.clone(),
                "obs_count": self.obs_rms.count.clone(), "ret_mean": self.ret_rms.mean.clone(),
                "ret_var": self.ret_rms.var.clone(), "ret_count": self.ret_rms.count.clone(),
                "returns": self._returns.clone(), "training": self.training, "norm_obs": self.norm_obs,
                "norm_reward": self.norm_reward, "clip_obs": self.clip_obs, "clip_reward": self.clip_reward,
                "gamma": self.gamma, "epsilon": self.epsilon}

    def load_state_dict(self, sd: Dict[str, Any]) -> None:
        for k, t in (("obs_mean", self.obs_rms.mean), ("obs_var", self.obs_rms.var), ("obs_count", self.obs_rms.count),
                     ("ret_mean", self.ret_rms.mean), ("ret_var", self.ret_rms.var), ("ret_count", self.ret_rms.count),
                     ("returns", self._returns)):
            t.copy_(sd[k])
        self.training, self.norm_obs, self.norm_reward = bool(sd["training"]), bool(sd["norm_obs"]), bool(sd["norm_reward"])
        self.clip_obs, self.clip_reward = float(sd["clip_obs"]), float(sd["clip_reward"])
        self.gamma, self.epsilon = float(sd["gamma"]), float(sd["epsilon"])
