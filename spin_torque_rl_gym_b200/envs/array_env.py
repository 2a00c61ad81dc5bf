"""SpinTorqueArrayVectorEnv — N SpinTorqueArray-v0 crossbar arrays stepped by one kernel launch (K3).

Host-side mirror of the reference's SpinTorqueArrayEnv (spin_torque_gym/envs/array_env.py:20-755) for observation_mode='array'
with the same constructor kwargs, batched over `num_envs` arrays. One CTA per array; the coupling matrix is computed on the
host exactly like the reference (envs/array_env.py:289-318) and shared by all arrays."""
from __future__ import annotations

import ctypes as C
from typing import Any, Dict, Optional, Tuple, Union

import numpy as np

from .. import _lib, params as _params
from ..spaces import Box, batch_box

MU0 = 4 * np.pi * 1e-7


def compute_coupling_matrix(n_rows: int, n_cols: int, coupling_strength: float, coupling_type: str) -> np.ndarray:
    """envs/array_env.py:289-318 (distances in grid units). Evaluated with the reference's scalar expressions
    (np.float64 ** 3 and array ** 3 round differently), once per distinct (|dr|, |dc|) offset."""
    n = n_rows * n_cols
    table = {}
    for dr in range(n_rows):
        for dc in range(n_cols):
            distance = np.sqrt(dr ** 2 + dc ** 2)
            v = 0.0
            if coupling_type == "dipolar":
                if distance > 0:
                    v = coupling_strength / (distance ** 3)
            elif coupling_type == "exchange":
                if distance == 1:
                    v = coupling_strength
            elif coupling_type == "stray_field":
                if distance > 0:
                    v = coupling_strength / (distance ** 2)
            table[(dr, dc)] = v
    out = np.zeros((n, n))
    for i in range(n):
        ir, ic = divmod(i, n_cols)
        for j in range(n):
            if i != j:
                jr, jc = divmod(j, n_cols)
                out[i, j] = table[(abs(ir - jr), abs(ic - jc))]
    return out


def array_params(array_size: Tuple[int, int], device_type: str, device_params: Dict[str, Any], action_mode: str,
                 max_steps: int, max_current: float, max_duration: float, success_threshold: float,
                 energy_penalty_weight: float) -> _lib.StgArrayParams:
    """K3's parameter block (StgArrayParams) for one array configuration: the device's field and resistance constants
    as the reference's device classes derive them from device_params."""
    p = _lib.StgArrayParams()
    p.n_rows, p.n_cols = array_size
    p.action_mode = _lib.ARRAY_MODES[action_mode]
    p.device_kind = _params.DEVICE_KINDS[device_type]
    p.max_steps = int(max_steps)
    ms = float(device_params.get("saturation_magnetization", 800e3))
    p.hk = 2 * float(device_params.get("uniaxial_anisotropy", 1e6)) / (MU0 * ms)
    p.saturation_magnetization = ms
    p.easy_axis = _lib.c_double3(*np.asarray(device_params.get("easy_axis", [0, 0, 1]), dtype=float))
    st = _params.make_param_struct(device_type, device_params, max_steps=max_steps, max_current=max_current,
                                   max_duration=max_duration, temperature=300.0, thermal=False,
                                   success_threshold=success_threshold, energy_penalty_weight=energy_penalty_weight)
    if p.device_kind != _lib.DEV_STT:
        ar = float(device_params.get("aspect_ratio", 1.0))
        nx, ny = (1.0 / (1.0 + ar), ar / (1.0 + ar)) if ar >= 1.0 else (ar / (1.0 + ar), 1.0 / (1.0 + ar))
        p.demag_n = _lib.c_double3(nx, ny, 1.0 - nx - ny)
    ref = np.asarray(device_params.get("reference_magnetization", [0, 0, 1]), dtype=float)
    p.reference_magnetization = _lib.c_double3(*(ref / np.linalg.norm(ref)))
    p.resistance_parallel, p.resistance_antiparallel = st.resistance_parallel, st.resistance_antiparallel
    p.series_resistance, p.area = st.series_resistance, st.area
    p.max_current, p.max_duration = float(max_current), float(max_duration)
    p.success_threshold, p.energy_penalty_weight = float(success_threshold), float(energy_penalty_weight)
    return p


class SpinTorqueArrayVectorEnv:
    metadata = {"render_modes": [], "autoreset_mode": "same_step"}

    def __init__(self, num_envs: int = 1, array_size: Tuple[int, int] = (4, 4), device_type: str = "stt_mram",
                 device_params: Optional[Dict[str, Any]] = None, target_pattern: Optional[np.ndarray] = None,
                 max_steps: int = 200, max_current: float = 2e6, max_duration: float = 5e-9, temperature: float = 300.0,
                 include_thermal_fluctuations: bool = True, include_coupling: bool = True, coupling_strength: float = 0.1,
                 coupling_type: str = "dipolar", reward_components: Optional[Dict[str, Dict]] = None,
                 action_mode: str = "individual", observation_mode: str = "array", success_threshold: float = 0.9,
                 energy_penalty_weight: float = 0.1, render_mode: Optional[str] = None, seed: Optional[int] = None, *,
                 device: Union[str, Any] = "cuda", rng_seed: Optional[int] = None, array_offset: int = 0,
                 autoreset: bool = True, collect_stats: bool = True, one_warp_kernel: bool = False,
                 host_outputs: bool = False):
        torch = _lib.require_cuda()
        self.one_warp_kernel = bool(one_warp_kernel)      # STG_F_ARRAY_ONE_WARP: A/B against the four-arrays-per-warp kernel
        # host_outputs: obs / final_obs / reward / terminated / truncated live in PINNED HOST memory, the kernel writes them there
        # directly (for consumers on the CPU); step() then synchronises the stream before it returns (as SpinTorqueVectorEnv)
        self.host_outputs = bool(host_outputs)
        self._args_cache = None
        self._torch = torch
        self._lib = _lib.load()
        if action_mode not in _lib.ARRAY_MODES:
            raise ValueError(f"Unknown action mode: {action_mode}")
        if observation_mode != "array":
            raise ValueError("only observation_mode='array' is implemented")
        if reward_components is not None:
            raise ValueError("custom reward_components are Python callables and cannot run in the kernel")
        self.num_envs = int(num_envs)
        self.array_size = tuple(array_size)
        self.n_rows, self.n_cols = self.array_size
        self.n_devices = self.n_rows * self.n_cols
        if self.n_devices > 1024:
            raise ValueError("at most 1024 devices per array")
        self.device_type = device_type
        self.max_steps, self.max_current, self.max_duration = int(max_steps), float(max_current), float(max_duration)
        self.temperature = temperature          # the reference builds a thermal model and never uses it (:103-108)
        self.include_coupling, self.coupling_strength, self.coupling_type = include_coupling, coupling_strength, coupling_type
        self.action_mode, self.observation_mode = action_mode, observation_mode
        self.success_threshold, self.energy_penalty_weight = float(success_threshold), float(energy_penalty_weight)
        self.autoreset, self.collect_stats = bool(autoreset), bool(collect_stats)
        self.array_offset = int(array_offset)
        if rng_seed is None:
            rng_seed = 0 if seed is None else int(seed)
        self.rng_seed = int(rng_seed) & 0xFFFFFFFFFFFFFFFF
        self.device = torch.device(device)
        if self.device.type != "cuda":
            raise _lib.StgError("SpinTorqueArrayVectorEnv requires a CUDA device (no CPU fallback)")
        if self.device.index is None:
            self.device = torch.device("cuda", torch.cuda.current_device())
        if device_params is None:
            device_params = _params.default_device_parameters("stt_mram")     # envs/array_env.py:155-171
        _params.check_device_constructible(device_type, device_params)
        self.device_params = dict(device_params)

        self._params_struct = array_params(self.array_size, device_type, device_params, action_mode, self.max_steps,
                                           self.max_current, self.max_duration, self.success_threshold,
                                           self.energy_penalty_weight)

        N, D, dev, f64 = self.num_envs, self.n_devices, self.device, torch.float64
        if target_pattern is None:
            tp = np.zeros((self.n_rows, self.n_cols, 3))
            ii, jj = np.indices((self.n_rows, self.n_cols))
            tp[..., 2] = np.where((ii + jj) % 2 == 0, 1.0, -1.0)               # checkerboard (:173-180)
        else:
            tp = np.asarray(target_pattern, dtype=float)
            if tp.shape != (self.n_rows, self.n_cols, 3):
                raise ValueError(f"Target pattern shape must be {(self.n_rows, self.n_cols, 3)}")
        self.target_pattern = tp.copy()
        with torch.cuda.device(dev):
            self.coupling_matrix = compute_coupling_matrix(self.n_rows, self.n_cols, coupling_strength, coupling_type) \
                if include_coupling else None
            self._coupling = torch.from_numpy(self.coupling_matrix).to(dev) if include_coupling else None
            self._pattern = torch.zeros(N, D, 3, dtype=f64, device=dev)
            self._pattern[..., 2] = 1.0
            self._target = torch.from_numpy(tp.reshape(1, D, 3)).to(dev).repeat(N, 1, 1).contiguous()
            self._total_energy = torch.zeros(N, dtype=f64, device=dev)
            self._step_count = torch.zeros(N, dtype=torch.int32, device=dev)
            self._episode = torch.zeros(N, dtype=torch.int32, device=dev)
            def out_buf(shape, dtype):
                if self.host_outputs:
                    return torch.zeros(shape, dtype=dtype).pin_memory()
                return torch.zeros(shape, dtype=dtype, device=dev)
            self._obs = out_buf((N, self.n_rows, self.n_cols, 6), torch.float32)
            self._final_obs = out_buf((N, self.n_rows, self.n_cols, 6), torch.float32)
            self._reward = out_buf((N,), f64)
            self._terminated = out_buf((N,), torch.uint8)
            self._truncated = out_buf((N,), torch.uint8)
            self._step_energy = torch.zeros(N, dtype=f64, device=dev)
            self._similarity = torch.zeros(N, dtype=f64, device=dev)
            self._stats = torch.zeros(_lib.STAT_REPLICAS, _lib.NSTATS, dtype=f64, device=dev)
            self._stats_folded = torch.zeros(_lib.NSTATS, dtype=f64, device=dev)
            self._adim = 2 if action_mode == "global" else 3
            self._action_dev = torch.zeros(N, self._adim, dtype=torch.float32, device=dev)
        self._needs_reset = True
        self.gpu_launches = 0
        hi0 = {"individual": self.n_devices - 1, "row": self.n_rows - 1, "column": self.n_cols - 1}.get(action_mode)
        if action_mode == "global":
            self.single_action_space = Box(low=np.array([-self.max_current, 0]),
                                           high=np.array([self.max_current, self.max_duration]), dtype=np.float32)
        else:
            self.single_action_space = Box(low=np.array([0, -self.max_current, 0]),
                                           high=np.array([hi0, self.max_current, self.max_duration]), dtype=np.float32)
        self.single_observation_space = Box(low=-1, high=1, shape=(self.n_rows, self.n_cols, 6), dtype=np.float32)
        self.action_space = batch_box(self.single_action_space, N)
        self.observation_space = batch_box(self.single_observation_space, N)

    def _args(self) -> _lib.StgArrayStepArgs:
        """Argument block of both entry points. Every buffer is allocated once in the constructor, so the block is built
        once and only the fields that can change between calls (seed, flags, action pointer) are rewritten."""
        a = self._args_cache
        if a is not None:
            a.seed = self.rng_seed
            return a
        a = _lib.StgArrayStepArgs()
        a.params = self._params_struct
        a.d_coupling = _lib.ptr(self._coupling)
        a.d_pattern, a.d_target = self._pattern.data_ptr(), self._target.data_ptr()
        a.d_total_energy, a.d_step_count, a.d_episode = (self._total_energy.data_ptr(), self._step_count.data_ptr(),
                                                         self._episode.data_ptr())
        a.d_obs, a.d_reward = _lib.ptr(self._obs), _lib.ptr(self._reward)
        a.d_terminated, a.d_truncated = _lib.ptr(self._terminated), _lib.ptr(self._truncated)
        a.d_step_energy, a.d_similarity = self._step_energy.data_ptr(), self._similarity.data_ptr()
        a.d_final_obs = _lib.ptr(self._final_obs) if self.autoreset else None
        a.d_stats = self._stats.data_ptr() if self.collect_stats else None
        a.seed, a.array_offset, a.n_arrays = self.rng_seed, self.array_offset, self.num_envs
        a.action_stride = self._adim
        a.flags = (_lib.F_AUTORESET if self.autoreset else 0) | (_lib.F_ARRAY_ONE_WARP if self.one_warp_kernel else 0)
        self._args_cache = a
        # zero-copy bool views of the u8 flag buffers (a .bool() per step is an extra kernel launch each)
        self._terminated_b = self._terminated.view(self._torch.bool)
        self._truncated_b = self._truncated.view(self._torch.bool)
        return a

    def _stream(self):
        return self._torch.cuda.current_stream(self.device).cuda_stream

    def reset(self, *, seed: Optional[int] = None, options: Optional[Dict[str, Any]] = None, mask=None):
        torch = self._torch
        options = options or {}
        if seed is not None:
            self.rng_seed = int(seed) & 0xFFFFFFFFFFFFFFFF
            self._episode.zero_()
        N, D = self.num_envs, self.n_devices
        keep = []
        if "target_pattern" in options:
            t = torch.as_tensor(np.asarray(options["target_pattern"], dtype=np.float64)).to(self.device)
            self._target.copy_(t.reshape(-1, D, 3).expand(N, D, 3))
        p0 = None
        if "initial_pattern" in options:
            p0 = torch.as_tensor(np.asarray(options["initial_pattern"], dtype=np.float64)).to(self.device)
            p0 = p0.reshape(-1, D, 3).expand(N, D, 3).contiguous()
            keep.append(p0)
        mk = None
        if mask is not None:
            mk = torch.as_tensor(mask).to(self.device).to(torch.uint8).contiguous()
            keep.append(mk)
        a = self._args()
        with torch.cuda.device(self.device):
            _lib.check(self._lib.stg_array_reset(C.byref(a), _lib.ptr(mk), _lib.ptr(p0), self._stream()), "stg_array_reset")
        self.gpu_launches += 1
        self._needs_reset = False
        self._keep = keep
        self._sync_host_outputs()
        return self._obs, {}

    def step(self, actions):
        torch = self._torch
        if self._needs_reset:
            raise RuntimeError("Environment must be reset before calling step")
        N = self.num_envs
        if isinstance(actions, torch.Tensor) and actions.device == self.device and actions.dtype == torch.float32 \
                and actions.is_contiguous() and tuple(actions.shape) == (N, self._adim):
            act = actions
        else:
            src = actions if isinstance(actions, torch.Tensor) else torch.as_tensor(np.asarray(actions, dtype=np.float32))
            self._action_dev.copy_(src.to(torch.float32).reshape(N, self._adim))
            act = self._action_dev
        a = self._args()
        a.d_action = act.data_ptr()
        with _lib.device_guard(torch, self.device):
            _lib.check(self._lib.stg_array_step_f64(C.byref(a), self._stream()), "stg_array_step_f64")
        self.gpu_launches += 1
        info = {"step_energy": self._step_energy, "pattern_similarity": self._similarity,
                "total_energy": self._total_energy, "step_count": self._step_count}
        if self.autoreset:
            info["final_observation"] = self._final_obs
        self._sync_host_outputs()
        return self._obs, self._reward, self._terminated_b, self._truncated_b, info

    def _sync_host_outputs(self) -> None:
        """host_outputs: the kernel wrote obs / reward / flags into pinned host memory; readable once the stream has drained."""
        if self.host_outputs and not self._torch.cuda.is_current_stream_capturing():
            self._torch.cuda.current_stream(self.device).synchronize()

    @property
    def current_pattern(self):
        """[N, rows, cols, 3] float64 (a view of the device state)."""
        return self._pattern.view(self.num_envs, self.n_rows, self.n_cols, 3)

    def _fold_stats(self):
        """Column sums of the replicated statistics buffer (include/stg.h, STG_STAT_REPLICAS) into one [NSTATS] vector."""
        torch = self._torch
        with _lib.device_guard(torch, self.device):
            _lib.check(self._lib.stg_stats_fold_f64(self._stats.data_ptr(), self._stats_folded.data_ptr(), 0,
                                                    torch.cuda.current_stream(self.device).cuda_stream), "stg_stats_fold_f64")
        return self._stats_folded

    def episode_stats(self, reset: bool = False) -> Dict[str, float]:
        """Accumulated episode statistics of this rank (dict of python floats; one D2H of 64 bytes)."""
        vals = self._fold_stats().cpu().tolist()
        if reset:
            self._stats.zero_()
        return dict(zip(_lib.STAT_NAMES, vals))

    def stats_tensor(self):
        """[NSTATS] float64 CUDA tensor of the statistics accumulated so far: the input of the one all-reduce per rollout.
        It is a folded copy (overwritten by the next call); use reset_stats() to start a new accumulation."""
        return self._fold_stats()

    def reset_stats(self) -> None:
        self._stats.zero_()

    def close(self):
        pass
