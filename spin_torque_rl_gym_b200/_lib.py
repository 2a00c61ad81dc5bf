"""ctypes binding of libstg.so (include/stg.h). The product path has NO CPU fallback: if the library is missing or
CUDA is unavailable, calls raise."""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

from . import build as _build

c_double3 = C.c_double * 3

# flags / enums (include/stg.h)
F_THERMAL_PHILOX = 0x01
F_THERMAL_INJECT = 0x02
F_AUTORESET = 0x04
F_EULER = 0x08
F_SORTED = 0x10
F_AXIS_Z = 0x20
F_VECTORIZED_PLAN = 0x40
F_NO_PAIR = 0x80
F_ARRAY_ONE_WARP = 0x100
F_PAIR_ALWAYS = 0x200
F_STREAM_PHILOX10 = 0x400
DEV_STT, DEV_SOT, DEV_VCMA = 0, 1, 2
NSTATS = 8
STAT_REPLICAS = 256      # include/stg.h STG_STAT_REPLICAS: the step kernels spread their atomics over this many copies
STAT_NAMES = ("steps", "substeps", "terminated", "truncated", "energy", "reward", "guard", "episode_length")
FOLDED_DOUBLES = 40
SORT_WORK_INTS = 8192 + 8
REDO_HEADER = 4          # include/stg.h STG_REDO_HEADER
STATUS_GUARD, STATUS_INVALID_PARAMS, STATUS_REDONE_F64 = 1, 2, 4
OBS_DIM = 12
# K8 VecNormalize (include/stg.h STG_VECNORM_*)
VECNORM_MOMENTS = 27      # moment vector (n, mean[13], M2[13]): 12 observation columns and the return
VECNORM_STATS = 28        # obs_rms mean [0, 12), var [12, 24), count 24; ret_rms mean 25, var 26, count 27
VECNORM_MAX_CTAS = 296
VECNORM_WORK_DOUBLES = VECNORM_MAX_CTAS * VECNORM_MOMENTS + 1
VECNORM_TRAINING, VECNORM_NORM_OBS, VECNORM_NORM_REWARD = 0x1, 0x2, 0x4
# K9 ActorCriticPolicy (include/stg.h STG_POLICY_*): offsets into the packed weight buffer, in floats
POLICY_LAYOUT = {"PI_W1": 0, "PI_B1": 768, "PI_W2": 832, "PI_B2": 4928, "VF_W1": 4992, "VF_B1": 5760, "VF_W2": 5824,
                 "VF_B2": 9920, "ACT_W": 9984, "ACT_B": 10112, "VAL_W": 10114, "VAL_B": 10178, "LOG_STD": 10179,
                 "STD": 10181, "LOG_SCALE": 10183}
POLICY_PARAMS = 10181
POLICY_FLOATS = 10188
POLICY_DETERMINISTIC = 0x1
# K10 PPO gradient (include/stg.h STG_PPO_*)
PPO_TILE = 128
PPO_MAX_CTAS = 296
PPO_PART = 10192          # doubles per CTA partial: gradient sums in the d_grad layout, then the loss sums
PPO_PART_LOSS = 10181
PPO_LOSSES = 6
PPO_CLIP_VF = 0x1
# K12 data-parallel PPO (include/stg.h)
PPO_PART_COUNT = 10185    # the row count within a sums vector
PPO_ADV_MOMENTS = 3       # (n, mean, M2) of the raw advantages
PPO_ADV_THREADS = 1024
# K11 clipped Adam (include/stg.h STG_ADAM_*)
ADAM_THREADS = 1024
ADAM_TENSORS = 13
ADAM_LOG = 8
ADAM_LOG_SLOTS = {"PG": 0, "VALUE": 1, "ENTROPY": 2, "CLIP": 3, "COUNT": 4, "EPOCH_KL": 5, "EPOCH_COUNT": 6, "LAST_LOSS": 7}
ADAM_CLIP, ADAM_TARGET_KL = 0x1, 0x2
# K13 clipped RMSprop (include/stg.h STG_RMSPROP_*)
RMSPROP_CLIP = 0x1


def ppo_grid(batch: int) -> int:
    """STG_PPO_GRID(batch): CTAs of stg_policy_ppo_grad_f32, a function of the batch size alone."""
    return 0 if batch <= 0 else min((batch + PPO_TILE - 1) // PPO_TILE, PPO_MAX_CTAS)


def ppo_work_doubles(batch: int) -> int:
    """STG_PPO_WORK_DOUBLES(batch)."""
    return ppo_grid(batch) * PPO_PART


class StgSttParams(C.Structure):
    _fields_ = [
        ("damping", C.c_double), ("saturation_magnetization", C.c_double), ("uniaxial_anisotropy", C.c_double),
        ("volume", C.c_double), ("polarization", C.c_double), ("easy_axis", c_double3),
        ("reference_magnetization", c_double3), ("resistance_parallel", C.c_double),
        ("resistance_antiparallel", C.c_double), ("area", C.c_double), ("series_resistance", C.c_double),
        ("temperature", C.c_double), ("applied_field", c_double3), ("max_current", C.c_double),
        ("max_duration", C.c_double), ("success_threshold", C.c_double), ("energy_penalty_weight", C.c_double),
        ("max_step", C.c_double), ("max_steps", C.c_int32), ("device_kind", C.c_int32), ("thermal", C.c_int32),
        ("solver_valid", C.c_int32),
    ]


class StgSttFolded(C.Structure):
    _fields_ = [("v", C.c_double * FOLDED_DOUBLES)]


class StgSttState(C.Structure):
    _fields_ = [("m", C.c_void_p), ("target", C.c_void_p), ("total_energy", C.c_void_p), ("last_action", C.c_void_p),
                ("step_count", C.c_void_p), ("episode", C.c_void_p)]


class StgSttStepOut(C.Structure):
    _fields_ = [("obs", C.c_void_p), ("reward", C.c_void_p), ("terminated", C.c_void_p), ("truncated", C.c_void_p),
                ("step_energy", C.c_void_p), ("n_sub", C.c_void_p), ("status", C.c_void_p), ("final_obs", C.c_void_p),
                ("stats", C.c_void_p)]


class StgSttStepArgs(C.Structure):
    _fields_ = [("d_table", C.c_void_p), ("d_param_index", C.c_void_p), ("state", StgSttState),
                ("d_action", C.c_void_p), ("out", StgSttStepOut), ("d_noise", C.c_void_p),
                ("noise_stride", C.c_int64), ("d_perm", C.c_void_p), ("d_target_table", C.c_void_p),
                ("seed", C.c_uint64), ("env_offset", C.c_uint64), ("n_envs", C.c_int64), ("n_sets", C.c_int32),
                ("n_targets", C.c_int32), ("flags", C.c_uint32), ("reserved", C.c_uint32), ("d_redo", C.c_void_p)]


class StgSttResetArgs(C.Structure):
    _fields_ = [("d_table", C.c_void_p), ("d_param_index", C.c_void_p), ("state", StgSttState),
                ("d_mask", C.c_void_p), ("d_m0", C.c_void_p), ("d_target0", C.c_void_p),
                ("d_target_table", C.c_void_p), ("d_obs", C.c_void_p), ("seed", C.c_uint64),
                ("env_offset", C.c_uint64), ("n_envs", C.c_int64), ("n_sets", C.c_int32), ("n_targets", C.c_int32)]


class StgSttSolveArgs(C.Structure):
    _fields_ = [("d_table", C.c_void_p), ("d_param_index", C.c_void_p), ("d_m0", C.c_void_p),
                ("d_pulse", C.c_void_p), ("d_m_out", C.c_void_p), ("d_traj", C.c_void_p), ("traj_stride", C.c_int64),
                ("d_n_sub", C.c_void_p), ("d_guard", C.c_void_p), ("d_noise", C.c_void_p),
                ("noise_stride", C.c_int64), ("seed", C.c_uint64), ("env_offset", C.c_uint64), ("n_envs", C.c_int64),
                ("n_sets", C.c_int32), ("flags", C.c_uint32), ("d_current_grid", C.c_void_p), ("d_field_grid", C.c_void_p),
                ("grid_stride", C.c_int64), ("grid_envs", C.c_int32), ("reserved", C.c_int32)]


class StgDeviceParams(C.Structure):
    _fields_ = [("kind", C.c_int32), ("reserved", C.c_int32), ("saturation_magnetization", C.c_double),
                ("uniaxial_anisotropy", C.c_double), ("mu0", C.c_double), ("easy_axis", c_double3),
                ("demag_n", c_double3), ("vcma_coefficient", C.c_double), ("dielectric_thickness", C.c_double),
                ("breakdown_voltage", C.c_double), ("tau_dl_factor", C.c_double), ("tau_fl_factor", C.c_double),
                ("resistance_parallel", C.c_double), ("resistance_antiparallel", C.c_double),
                ("reference_magnetization", c_double3), ("series_resistance", C.c_double)]


class StgLlgParams(C.Structure):
    _fields_ = [("gamma", C.c_double), ("mu0", C.c_double), ("alpha", C.c_double),
                ("saturation_magnetization", C.c_double), ("uniaxial_anisotropy", C.c_double), ("volume", C.c_double),
                ("easy_axis", c_double3), ("demag_n", c_double3), ("exchange_coeff", C.c_double), ("h_th", C.c_double),
                ("c_dl_p", C.c_double), ("c_fl_p", C.c_double), ("p_hat", c_double3), ("c_dl_s", C.c_double),
                ("c_fl_s", C.c_double), ("sigma", c_double3), ("vcma_coefficient", C.c_double),
                ("dielectric_thickness", C.c_double), ("breakdown_voltage", C.c_double), ("use_vcma", C.c_int32),
                ("reserved", C.c_int32)]


class StgRk45Args(C.Structure):
    _fields_ = [("d_table", C.c_void_p), ("d_param_index", C.c_void_p), ("d_m0", C.c_void_p), ("d_t_end", C.c_void_p),
                ("d_current", C.c_void_p), ("d_t_pulse", C.c_void_p), ("d_happ", C.c_void_p), ("d_voltage", C.c_void_p),
                ("d_y_out", C.c_void_p), ("d_n_accepted", C.c_void_p), ("d_n_rejected", C.c_void_p),
                ("d_n_rhs", C.c_void_p), ("d_status", C.c_void_p), ("d_t_reached", C.c_void_p), ("d_traj", C.c_void_p),
                ("traj_stride", C.c_int64), ("d_noise", C.c_void_p), ("noise_stride", C.c_int64), ("rtol", C.c_double),
                ("atol", C.c_double), ("max_step", C.c_double), ("max_attempts", C.c_int64), ("seed", C.c_uint64),
                ("env_offset", C.c_uint64), ("n_envs", C.c_int64), ("n_sets", C.c_int32), ("flags", C.c_uint32),
                ("d_perm", C.c_void_p), ("d_t_start", C.c_void_p), ("d_seg_t", C.c_void_p), ("d_seg_current", C.c_void_p),
                ("d_seg_field", C.c_void_p), ("n_seg", C.c_int32), ("seg_rows", C.c_int32)]


class StgThermalAnalyticsArgs(C.Structure):
    _fields_ = [("d_temperature", C.c_void_p), ("d_ku", C.c_void_p), ("d_volume", C.c_void_p), ("d_damping", C.c_void_p),
                ("d_ms", C.c_void_p), ("d_barrier", C.c_void_p), ("d_out", C.c_void_p), ("k_b", C.c_double),
                ("mu0", C.c_double), ("gamma", C.c_double), ("attempt_frequency", C.c_double),
                ("measurement_time", C.c_double), ("failure_rate", C.c_double), ("n_t", C.c_int32), ("n_dev", C.c_int32)]


ARRAY_MODES = {"individual": 0, "row": 1, "column": 2, "global": 3}


class StgArrayParams(C.Structure):
    _fields_ = [("n_rows", C.c_int32), ("n_cols", C.c_int32), ("action_mode", C.c_int32), ("device_kind", C.c_int32),
                ("max_steps", C.c_int32), ("reserved", C.c_int32), ("hk", C.c_double),
                ("saturation_magnetization", C.c_double), ("easy_axis", c_double3), ("demag_n", c_double3),
                ("resistance_parallel", C.c_double), ("resistance_antiparallel", C.c_double),
                ("reference_magnetization", c_double3), ("series_resistance", C.c_double), ("area", C.c_double),
                ("max_current", C.c_double), ("max_duration", C.c_double), ("success_threshold", C.c_double),
                ("energy_penalty_weight", C.c_double)]


class StgArrayStepArgs(C.Structure):
    _fields_ = [("params", StgArrayParams), ("d_coupling", C.c_void_p), ("d_pattern", C.c_void_p),
                ("d_target", C.c_void_p), ("d_total_energy", C.c_void_p), ("d_step_count", C.c_void_p),
                ("d_episode", C.c_void_p), ("d_action", C.c_void_p), ("d_obs", C.c_void_p), ("d_reward", C.c_void_p),
                ("d_terminated", C.c_void_p), ("d_truncated", C.c_void_p), ("d_step_energy", C.c_void_p),
                ("d_similarity", C.c_void_p), ("d_final_obs", C.c_void_p), ("d_stats", C.c_void_p), ("seed", C.c_uint64),
                ("array_offset", C.c_uint64), ("n_arrays", C.c_int64), ("action_stride", C.c_int32), ("flags", C.c_uint32)]


class StgGaeArgs(C.Structure):
    _fields_ = [("d_reward", C.c_void_p), ("d_value", C.c_void_p), ("d_terminated", C.c_void_p),
                ("d_truncated", C.c_void_p), ("d_final_value", C.c_void_p), ("d_last_value", C.c_void_p),
                ("d_advantage", C.c_void_p), ("d_return", C.c_void_p), ("gamma", C.c_float),
                ("gamma_lambda", C.c_float), ("n_steps", C.c_int64), ("n_envs", C.c_int64)]


class StgMinibatchArgs(C.Structure):
    _fields_ = [("d_obs", C.c_void_p), ("d_obs_out", C.c_void_p), ("d_action", C.c_void_p), ("d_action_out", C.c_void_p),
                ("d_value", C.c_void_p), ("d_value_out", C.c_void_p), ("d_log_prob", C.c_void_p),
                ("d_log_prob_out", C.c_void_p), ("d_advantage", C.c_void_p), ("d_advantage_out", C.c_void_p),
                ("d_return", C.c_void_p), ("d_return_out", C.c_void_p), ("round_keys", C.c_uint32 * 8),
                ("n_steps", C.c_int64), ("n_envs", C.c_int64), ("start", C.c_int64), ("batch", C.c_int64)]


class StgVecNormArgs(C.Structure):
    _fields_ = [("d_obs", C.c_void_p), ("d_final_obs", C.c_void_p), ("d_terminated", C.c_void_p),
                ("d_truncated", C.c_void_p), ("d_reward", C.c_void_p), ("d_returns", C.c_void_p), ("d_stats", C.c_void_p),
                ("d_moments", C.c_void_p), ("d_work", C.c_void_p), ("d_obs_out", C.c_void_p),
                ("d_final_obs_out", C.c_void_p), ("d_reward_out", C.c_void_p), ("gamma", C.c_double),
                ("epsilon", C.c_double), ("clip_obs", C.c_double), ("clip_reward", C.c_double), ("n_envs", C.c_int64),
                ("n_ranks", C.c_int32), ("flags", C.c_uint32)]


class StgPolicyArgs(C.Structure):
    _fields_ = [("d_obs", C.c_void_p), ("d_weights", C.c_void_p), ("d_mask", C.c_void_p), ("d_obs_copy", C.c_void_p),
                ("d_action", C.c_void_p), ("d_env_action", C.c_void_p), ("d_value", C.c_void_p), ("d_log_prob", C.c_void_p),
                ("action_low", C.c_float * 2), ("action_high", C.c_float * 2), ("key", C.c_uint32 * 2),
                ("draw", C.c_uint64), ("env_offset", C.c_uint64), ("n_envs", C.c_int64), ("flags", C.c_uint32),
                ("reserved", C.c_uint32)]


class StgPpoArgs(C.Structure):
    _fields_ = [("d_weights", C.c_void_p), ("d_obs", C.c_void_p), ("d_action", C.c_void_p), ("d_old_value", C.c_void_p),
                ("d_old_log_prob", C.c_void_p), ("d_advantage", C.c_void_p), ("d_return", C.c_void_p),
                ("d_adv_stats", C.c_void_p), ("d_grad", C.c_void_p), ("d_losses", C.c_void_p), ("d_work", C.c_void_p),
                ("clip_range", C.c_float), ("ratio_lo", C.c_float), ("ratio_hi", C.c_float), ("clip_range_vf", C.c_float),
                ("ent_coef", C.c_float), ("vf_coef", C.c_float), ("flags", C.c_uint32), ("reserved", C.c_uint32),
                ("batch", C.c_int64)]


class StgAdamArgs(C.Structure):
    _fields_ = [("d_param", C.c_void_p * ADAM_TENSORS), ("d_grad", C.c_void_p), ("d_exp_avg", C.c_void_p),
                ("d_exp_avg_sq", C.c_void_p), ("d_step", C.c_void_p), ("d_losses", C.c_void_p), ("d_gate", C.c_void_p),
                ("d_log", C.c_void_p), ("lr", C.c_double), ("beta1", C.c_double), ("beta2", C.c_double), ("eps", C.c_double),
                ("max_grad_norm", C.c_double), ("target_kl", C.c_double), ("flags", C.c_uint32), ("reserved", C.c_uint32)]


class StgRmspropArgs(C.Structure):
    _fields_ = [("d_param", C.c_void_p * ADAM_TENSORS), ("d_grad", C.c_void_p), ("d_square_avg", C.c_void_p),
                ("d_step", C.c_void_p), ("lr", C.c_double), ("alpha", C.c_double), ("eps", C.c_double),
                ("max_grad_norm", C.c_double), ("flags", C.c_uint32), ("reserved", C.c_uint32)]


class StgEnergyParams(C.Structure):
    _fields_ = [("mu0", C.c_double), ("saturation_magnetization", C.c_double), ("volume", C.c_double),
                ("uniaxial_anisotropy", C.c_double), ("easy_axis", c_double3), ("demag_factors", c_double3)]


# every symbol include/stg.h declares: (name, restype, argtypes)
SYMBOLS = {
    "stg_abi_version": (C.c_int, []),
    "stg_stt_thermal_pair_dispatch": (C.c_int, [C.c_int64, C.c_uint32, C.c_int]),
    "stg_error_string": (C.c_char_p, [C.c_int]),
    "stg_stt_fold": (C.c_int, [C.POINTER(StgSttParams), C.c_int32, C.POINTER(StgSttFolded)]),
    "stg_stt_all_axis_z": (C.c_int, [C.POINTER(StgSttFolded), C.c_int32]),
    "stg_stt_step_f32": (C.c_int, [C.POINTER(StgSttStepArgs), C.c_void_p]),
    "stg_stt_step_f64": (C.c_int, [C.POINTER(StgSttStepArgs), C.c_void_p]),
    "stg_stt_reset": (C.c_int, [C.POINTER(StgSttResetArgs), C.c_void_p]),
    "stg_stt_sort_by_substeps": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_int64, C.c_void_p]),
    "stg_stt_solve_f32": (C.c_int, [C.POINTER(StgSttSolveArgs), C.c_void_p]),
    "stg_stt_solve_f64": (C.c_int, [C.POINTER(StgSttSolveArgs), C.c_void_p]),
    "stg_llgs_rk45_f64": (C.c_int, [C.POINTER(StgRk45Args), C.c_void_p]),
    "stg_llgs_rk45_cost_f64": (C.c_int, [C.POINTER(StgRk45Args), C.c_void_p, C.c_void_p]),
    "stg_llgs_rk45_sort_f64": (C.c_int, [C.POINTER(StgRk45Args), C.c_void_p, C.c_void_p, C.c_void_p]),
    "stg_array_step_f64": (C.c_int, [C.POINTER(StgArrayStepArgs), C.c_void_p]),
    "stg_array_reset": (C.c_int, [C.POINTER(StgArrayStepArgs), C.c_void_p, C.c_void_p, C.c_void_p]),
    "stg_device_field_f64": (C.c_int, [C.POINTER(StgDeviceParams), C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                       C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "stg_device_resistance_f64": (C.c_int, [C.POINTER(StgDeviceParams), C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p,
                                            C.c_void_p]),
    "stg_device_sot_torque_f64": (C.c_int, [C.POINTER(StgDeviceParams), C.c_void_p, C.c_int32, C.c_void_p,
                                            C.POINTER(C.c_double), C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "stg_vcma_anisotropy_f64": (C.c_int, [C.POINTER(StgDeviceParams), C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "stg_thermal_analytics_f64": (C.c_int, [C.POINTER(StgThermalAnalyticsArgs), C.c_void_p]),
    "stg_thermal_field_f64": (C.c_int, [C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_uint64, C.c_uint64,
                                        C.c_uint64, C.c_int64, C.c_void_p]),
    "stg_energy_landscape_f64": (C.c_int, [C.POINTER(StgEnergyParams), C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                           C.c_void_p, C.c_int64, C.c_void_p]),
    "stg_stats_reduce_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_int64, C.c_void_p, C.c_void_p]),
    "stg_stats_fold_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "stg_host_device_pointer": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "stg_vec3_op_f64": (C.c_int, [C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                  C.c_int64, C.c_void_p]),
    "stg_phase_diagram_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_double, C.c_double, C.c_void_p,
                                        C.c_void_p]),
    "stg_rollout_gae_f32": (C.c_int, [C.POINTER(StgGaeArgs), C.c_void_p]),
    "stg_rollout_minibatch_f32": (C.c_int, [C.POINTER(StgMinibatchArgs), C.c_void_p]),
    "stg_vecnorm_moments_f32": (C.c_int, [C.POINTER(StgVecNormArgs), C.c_void_p]),
    "stg_vecnorm_merge_f64": (C.c_int, [C.POINTER(StgVecNormArgs), C.c_void_p]),
    "stg_vecnorm_apply_f32": (C.c_int, [C.POINTER(StgVecNormArgs), C.c_void_p]),
    "stg_policy_act_f32": (C.c_int, [C.POINTER(StgPolicyArgs), C.c_void_p]),
    "stg_policy_value_f32": (C.c_int, [C.POINTER(StgPolicyArgs), C.c_void_p]),
    "stg_policy_ppo_grad_f32": (C.c_int, [C.POINTER(StgPpoArgs), C.c_void_p]),
    "stg_policy_ppo_sums_f32": (C.c_int, [C.POINTER(StgPpoArgs), C.c_void_p, C.c_void_p]),
    "stg_policy_ppo_finish_f32": (C.c_int, [C.POINTER(StgPpoArgs), C.c_void_p, C.c_int32, C.c_void_p]),
    "stg_ppo_adv_moments_f64": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "stg_ppo_adv_merge_f32": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "stg_policy_adam_f32": (C.c_int, [C.POINTER(StgAdamArgs), C.c_void_p]),
    "stg_policy_a2c_grad_f32": (C.c_int, [C.POINTER(StgPpoArgs), C.c_void_p]),
    "stg_policy_a2c_sums_f32": (C.c_int, [C.POINTER(StgPpoArgs), C.c_void_p, C.c_void_p]),
    "stg_policy_rmsprop_f32": (C.c_int, [C.POINTER(StgRmspropArgs), C.c_void_p]),
    "stg_probe_fma": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
}

ABI_VERSION = 7          # include/stg.h STG_ABI_VERSION (2: sampled current / field grids; 3: replicated statistics buffer;
                         # 4: zero-row counters of stg_device_field_f64 / stg_device_resistance_f64; 5: StgRk45Args.d_perm;
                         # 6: StgSttStepArgs.d_redo, status bit 2)
_LIB: Optional[C.CDLL] = None


class StgError(RuntimeError):
    pass


def lib_path() -> str:
    # STG_LIB_PATH: load an alternative build of libstg.so (kernel tuning experiments); default is the in-tree library
    return os.environ.get("STG_LIB_PATH") or _build.LIB_PATH


def load(build_if_missing: bool = True) -> C.CDLL:
    """Load libstg.so (building it in-tree with nvcc first if it is missing or stale). Raises if impossible."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if build_if_missing and path == _build.LIB_PATH and _build.needs_build():
        try:
            _build.build()
        except Exception as exc:  # a stale but present library is still usable on a box without nvcc
            if not os.path.exists(path):
                raise StgError(f"libstg.so is missing and could not be built: {exc}") from exc
    if not os.path.exists(path):
        raise StgError(f"{path} not found: the CUDA extension is required (no CPU fallback)")
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    if lib.stg_abi_version() != ABI_VERSION:
        raise StgError(f"libstg.so ABI version {lib.stg_abi_version()} != {ABI_VERSION} expected by this package "
                       "(stale build? run __graft_entry__.build())")
    _LIB = lib
    return lib


def check(rc: int, what: str = "stg call") -> None:
    if rc != 0:
        msg = load().stg_error_string(rc).decode()
        raise StgError(f"{what} failed with code {rc}: {msg}")


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise StgError("CUDA device required: spin_torque_rl_gym_b200 has no CPU fallback for the LLGS hot path")
    return torch


class _NullGuard:
    def __enter__(self):
        return None

    def __exit__(self, *exc):
        return False


_NULL_GUARD = _NullGuard()


def device_guard(torch, device):
    """`torch.cuda.device(device)` only when it is not already the current device (the context switch costs several
    microseconds per call, which is visible in small-batch env steps)."""
    idx = device.index
    if idx is None or torch.cuda.current_device() == idx:
        return _NULL_GUARD
    return torch.cuda.device(device)


def ptr(t) -> Optional[int]:
    """Device pointer of a torch tensor (None -> NULL). A pinned CPU tensor yields the device-side address of its mapped
    host memory (kernels may write their outputs there directly)."""
    if t is None:
        return None
    if t.device.type == "cpu":
        if not t.is_pinned():
            raise StgError("a CPU tensor handed to a kernel must be pinned")
        out = C.c_void_p()
        check(load().stg_host_device_pointer(t.data_ptr(), C.byref(out)), "stg_host_device_pointer")
        return out.value
    return t.data_ptr()
