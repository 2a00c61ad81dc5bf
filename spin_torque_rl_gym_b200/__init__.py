"""spin_torque_rl_gym_b200 — B200-native batched LLGS hot path of Spin-Torque RL-Gym.

Host layer (Python/PyTorch) mirroring the reference's env / solver / device API for the per-step
Landau-Lifshitz-Gilbert-Slonczewski integration, on top of hand-written sm_100a CUDA kernels behind the C-ABI of
include/stg.h (libstg.so). See DESIGN.md.

    import spin_torque_rl_gym_b200 as stg
    env = stg.make('SpinTorque-v0', device_type='stt_mram')                    # reference single-env API
    venv = stg.make('SpinTorque-v0', num_envs=1 << 20, device='cuda:0')        # one kernel launch per step for 1M envs
"""
__version__ = "0.1.0"

from . import _lib, build, params  # noqa: F401
from .envs import (RolloutCollector, SB3VecEnvAdapter, SpinTorqueArrayEnv, SpinTorqueArrayVectorEnv,  # noqa: F401
                   SpinTorqueEnv, SpinTorqueVectorEnv, VecNormalize, make, register_with_gymnasium)
from .parallel import all_gather_moments, all_reduce_stats, shard_range  # noqa: F401
from .policy import A2CLosses, ActorCriticPolicy, PPOLosses  # noqa: F401
from .optim import ClippedAdam, ClippedRMSprop  # noqa: F401
from .ppo import PPO  # noqa: F401
from .a2c import A2C  # noqa: F401

register_with_gymnasium()
