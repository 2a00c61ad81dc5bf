from .vector_env import SpinTorqueVectorEnv  # noqa: F401
from .array_env import SpinTorqueArrayVectorEnv  # noqa: F401
from .spin_torque_env import SpinTorqueArrayEnv, SpinTorqueEnv, make, register_with_gymnasium  # noqa: F401
from .sb3_vec_env import RolloutCollector, SB3VecEnvAdapter  # noqa: F401
from .vec_normalize import RunningMeanStdView, VecNormalize  # noqa: F401
