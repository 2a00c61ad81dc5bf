/* stg.h — C-ABI of the B200-native batched LLGS hot path (libstg.so).
 *
 * The reference (danieleschmidt/spin-torque-rl-gym) is pure Python and has no FFI; these entry points are what a
 * ctypes binding in the reference would call in place of its per-env NumPy loops. Each entry point names the reference
 * interface it replaces (paths relative to /root/reference/spin_torque_gym/).
 *
 * Conventions
 *   - Plain C: pointers + sizes only. All `d_*` pointers are DEVICE pointers owned by the caller (PyTorch tensors in the
 *     host layer). The library allocates nothing persistent and keeps no state between calls (re-entrant).
 *   - Every call is asynchronous on `stream` (a cudaStream_t passed as void*; NULL = legacy default stream). No hidden
 *     synchronisation.
 *   - Return value: 0 ok; <0 bad argument (STG_E_*); >0 a cudaError_t from the launch. Numerical failures of individual
 *     envs are reported per env in status[] and never as an error code.
 *   - State is kept in FP64 struct-of-arrays planes regardless of the arithmetic type; `_f32` / `_f64` select the type the
 *     RHS / integrator stages are computed in.
 */
#ifndef STG_H_
#define STG_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define STG_ABI_VERSION 7

/* error codes */
#define STG_OK 0
#define STG_E_NULL (-1)      /* required pointer is NULL        */
#define STG_E_SIZE (-2)      /* negative / inconsistent size    */
#define STG_E_ENUM (-3)      /* unknown enum / flag combination */
#define STG_E_ALIGN (-4)     /* pointer not aligned as required */

/* device kinds: which compute_resistance() formula the env uses (devices/stt_mram.py:78-94,
 * devices/sot_mram.py:196-228, devices/vcma_mram.py:236-257) */
#define STG_DEV_STT 0
#define STG_DEV_SOT 1
#define STG_DEV_VCMA 2

/* integrators of SimpleLLGSSolver (physics/simple_solver.py:254-295) */
#define STG_INT_RK4 0
#define STG_INT_EULER 1

/* step flags */
#define STG_F_THERMAL_PHILOX 0x01u   /* thermal field from the in-kernel stream: Philox4x32-10 keyed by seed, counter =   *
                                      * (global env id, episode, step, block); the RK4 paths seed one xoshiro128++ state  *
                                      * per env-step from block 0 of it (llgs_core.cuh, ThermalSource)                    */
#define STG_F_THERMAL_INJECT 0x02u   /* thermal field from the caller's noise tensor (parity / debugging)          */
#define STG_F_AUTORESET 0x04u        /* envs that terminate/truncate are reset in the same call (SB3 VecEnv rule)  */
#define STG_F_EULER 0x08u            /* SimpleLLGSSolver(method='euler') instead of 'rk4'                          */
#define STG_F_SORTED 0x10u           /* d_perm holds an env permutation (e.g. sorted by substep count)             */
#define STG_F_AXIS_Z 0x20u           /* caller asserts stg_stt_all_axis_z(): kernels drop structurally-zero terms   */
#define STG_F_NO_PAIR 0x80u          /* stg_stt_step_f32: one env per thread instead of the packed two-envs-per-thread FFMA2
                                        kernel (identical results; for comparisons)                                 */
#define STG_F_PAIR_ALWAYS 0x200u     /* stg_stt_step_f32 with STG_F_THERMAL_PHILOX: take the two-envs-per-thread kernel at every batch
                                        size (by default it is dispatched from 262,144 envs, where it is the faster one; identical
                                        results per env either way)                                                  */
#define STG_F_STREAM_PHILOX10 0x400u  /* stg_stt_step_*, with STG_F_THERMAL_PHILOX and RK4: every word of the thermal stream from
                                        Philox4x32-10 (counter-based down to the substep: three blocks per two substeps) instead of
                                        the default Philox-seeded xoshiro128++ expansion; 10.4 against 8.6 ms per 1M-env step     */
#define STG_F_ARRAY_ONE_WARP 0x100u  /* stg_array_step_f64: force the one-warp-per-array kernel (the default for 8 <= devices <= 128
                                      * is four arrays per warp, eight lanes each; both are bit-identical) */
#define STG_F_VECTORIZED_PLAN 0x40u  /* stg_stt_solve_*: n = max(10, int(t_end/max_step)) — VectorizedSolver.solve_batch's step
                                        policy (utils/vectorized_operations.py:55-57) instead of SimpleLLGSSolver's        */

/* Raw physical parameters of one device parameter set (FP64, SI units). Mirrors the `device_params` dict read by
 * SimpleLLGSSolver._compute_dmdt/_compute_effective_field (physics/simple_solver.py:310-315, 358-380) plus the env
 * configuration of SpinTorqueEnv.__init__ (envs/spin_torque_env.py:36-53). */
typedef struct StgSttParams {
    double damping;                  /* alpha                                                     */
    double saturation_magnetization; /* Ms  [A/m]                                                 */
    double uniaxial_anisotropy;      /* Ku  [J/m^3]                                               */
    double volume;                   /* V   [m^3]                                                 */
    double polarization;             /* P                                                         */
    double easy_axis[3];             /* normalised by the library like the solver does (:319)     */
    double reference_magnetization[3];
    double resistance_parallel;      /* R_P  [Ohm]                                                */
    double resistance_antiparallel;  /* R_AP [Ohm]                                                */
    double area;                     /* A [m^2], default 1e-14 (envs/spin_torque_env.py:476)      */
    double series_resistance;        /* SOT: 0.1*rho/(t_HM*A*1e-12) (devices/sot_mram.py:219-226) */
    double temperature;              /* K                                                         */
    double applied_field[3];         /* constant H_app [A/m] (env passes 0)                       */
    double max_current;              /* A/m^2 (env clip, :430)                                    */
    double max_duration;             /* s     (env clip, :431)                                    */
    double success_threshold;        /* alignment threshold (:353)                                */
    double energy_penalty_weight;    /* w_E (:193)                                                */
    double max_step;                 /* SimpleLLGSSolver.max_step, 1e-12 (:29)                    */
    int32_t max_steps;               /* episode length (:372)                                     */
    int32_t device_kind;             /* STG_DEV_*                                                 */
    int32_t thermal;                 /* include_thermal_fluctuations                              */
    int32_t solver_valid;            /* 0: RobustLLGSSolver input validation fails => m never moves
                                        (utils/robust_solver.py:152-190, SURVEY A3)               */
} StgSttParams;

/* Folded per-parameter-set constants consumed by the kernels (produced on the host by stg_stt_fold, uploaded once by the
 * caller). Opaque to callers: treat as STG_FOLDED_BYTES bytes. */
#define STG_FOLDED_DOUBLES 40
#define STG_FOLDED_BYTES (STG_FOLDED_DOUBLES * 8)
typedef struct StgSttFolded {
    double v[STG_FOLDED_DOUBLES];
} StgSttFolded;

/* Per-env state, FP64 SoA planes of length n_envs (device pointers). Mirrors SpinTorqueEnv's instance state
 * (envs/spin_torque_env.py:133-139). */
typedef struct StgSttState {
    double* m;           /* [3][n]  current_magnetization (plane-major: mx[n], my[n], mz[n]) */
    double* target;      /* [3][n]  target_magnetization                                    */
    double* total_energy;/* [n]                                                             */
    double* last_action; /* [2][n]  (J, T) after clipping                                   */
    int32_t* step_count; /* [n]                                                             */
    int32_t* episode;    /* [n]     episodes completed (advances the Philox reset stream)   */
} StgSttState;

/* Outputs of one env step (device pointers; any may be NULL except obs/reward/terminated/truncated). */
typedef struct StgSttStepOut {
    float* obs;          /* [n][12] f32, _get_observation (envs/spin_torque_env.py:500-520)           */
    double* reward;      /* [n]     CompositeReward default + clip (envs/spin_torque_env.py:184-207)    */
    uint8_t* terminated; /* [n]                                                                        */
    uint8_t* truncated;  /* [n]                                                                        */
    double* step_energy; /* [n]     energy_consumed (:474-480)                                         */
    int32_t* n_sub;      /* [n]     substeps integrated (physics/simple_solver.py:137-139)              */
    int32_t* status;     /* [n]     0 ok; bit0 non-finite/zero-norm guard fired (m kept); bit1 solver
                                    validation failed (solver_valid==0); bit2 (STG_STATUS_REDONE_F64)
                                    stg_stt_step_f32 repeated this env with FP64 stages (see d_redo)   */
    float* final_obs;    /* [n][12] with STG_F_AUTORESET: observation before the reset (terminal_observation). Only the rows of
                            envs whose episode ended in this step (terminated | truncated) are written; the others keep their
                            previous contents */
    double* stats;       /* [STG_STAT_REPLICAS][STG_NSTATS] accumulated with atomics (K5 input), see below */
} StgSttStepOut;

#define STG_STATUS_GUARD 1
#define STG_STATUS_INVALID_PARAMS 2
#define STG_STATUS_REDONE_F64 4

/* stats vector layout (all doubles, SUM-reducible across ranks) */
#define STG_STAT_STEPS 0        /* env-steps executed                */
#define STG_STAT_SUBSTEPS 1     /* LLGS substeps integrated          */
#define STG_STAT_TERMINATED 2   /* episodes ended by success         */
#define STG_STAT_TRUNCATED 3    /* episodes ended by max_steps       */
#define STG_STAT_ENERGY 4       /* sum of step energies [J]          */
#define STG_STAT_REWARD 5       /* sum of rewards                    */
#define STG_STAT_GUARD 6        /* env-steps whose guard fired       */
#define STG_STAT_EPLEN 7        /* sum of lengths of ended episodes  */
#define STG_NSTATS 8
/* The step kernels ADD into d_stats with FP64 atomics. A single 64-byte vector puts every atomic of a launch on one L2 line
 * (measured on the crossbar step, 16,384 arrays: 114,688 atomics on one line took the step from 43 us to 91 us; the 1M-env
 * K1 step, whose atomics are spread over 14 ms, did not change), so the buffer holds STG_STAT_REPLICAS copies of the vector
 * and CTA b adds to copy b % STG_STAT_REPLICAS. A statistic is the column sum over the
 * copies (stg_stats_fold_f64). The caller zeroes the whole buffer once per rollout. */
#define STG_STAT_REPLICAS 256

/* Argument block of one batched env step. Host struct (passed by pointer, copied into the kernel's parameter space);
 * every d_* member is a device pointer.
 *   d_table        [n_sets] folded parameter sets; d_param_index [n] int32 or NULL (all envs use set 0)
 *   d_action       [n][2] f32 (J, T) as produced by the policy; clipped like SafetyWrapper + _parse_action
 *   d_noise        STG_F_THERMAL_INJECT: [n][noise_stride][S][3] f64 N(0,1) samples, S=4 (rk4) or 1 (euler), in the order
 *                  the reference draws them: (substep, stage, xyz) (physics/simple_solver.py:381); an env that integrates
 *                  more than noise_stride substeps reuses the last row (no out-of-bounds read)
 *   d_perm         STG_F_SORTED: [n] int32 env indices processed by consecutive threads (stg_stt_sort_by_substeps)
 *   d_target_table STG_F_AUTORESET: [n_targets][3] f64 target_states (envs/spin_torque_env.py:117-120)
 *   seed, env_offset: Philox key / global env id of local env 0 (rank sharding keeps streams independent of #GPUs)
 *   d_redo         stg_stt_step_f32, STG_F_AXIS_Z, RK4, without STG_F_THERMAL_PHILOX: int32 workspace of STG_REDO_HEADER + n
 *                  entries (contents irrelevant on entry). The FP32 stages track a conditioning bound per trajectory
 *                  (csrc/llgs_core.cuh: CondTrack); an env whose bound exceeds the FP32 contract (1e-4 on m, energy, reward:
 *                  trajectories held near an unstable polar angle for thousands of substeps, ~0.2 % of uniformly random
 *                  (state, pulse <= 5 ns) samples) is not stepped by the FP32 kernel but appended to this list, and a second,
 *                  compacted launch in the same call steps the listed envs with FP64 stages (status bit 2). Results do not
 *                  depend on the order of the list. Required (STG_E_NULL) for those launches; ignored otherwise. */
#define STG_REDO_HEADER 4
typedef struct StgSttStepArgs {
    const StgSttFolded* d_table;
    const int32_t* d_param_index;
    StgSttState state;
    const float* d_action;
    StgSttStepOut out;
    const double* d_noise;
    int64_t noise_stride;
    const int32_t* d_perm;
    const double* d_target_table;
    uint64_t seed;
    uint64_t env_offset;
    int64_t n_envs;
    int32_t n_sets;
    int32_t n_targets;
    uint32_t flags;
    uint32_t reserved;
    int32_t* d_redo;
} StgSttStepArgs;

/* Argument block of a batched reset (envs/spin_torque_env.py:250-308) of the envs with d_mask[i]!=0 (all if NULL).
 *   d_m0 / d_target0: optional [n][3] f64 explicit options['initial_state'] / ['target_state'] (normalised here);
 *   NULL => m0 = normalise(N(0,1)^3) from Philox, target drawn uniformly from d_target_table [n_targets][3].
 *   d_obs: [n][12] f32, rows of the reset envs are overwritten with the reset observation (may be NULL). */
typedef struct StgSttResetArgs {
    const StgSttFolded* d_table;
    const int32_t* d_param_index;
    StgSttState state;
    const uint8_t* d_mask;
    const double* d_m0;
    const double* d_target0;
    const double* d_target_table;
    float* d_obs;
    uint64_t seed;
    uint64_t env_offset;
    int64_t n_envs;
    int32_t n_sets;
    int32_t n_targets;
} StgSttResetArgs;

/* Argument block of a batched SimpleLLGSSolver.solve for rectangular pulses (physics/simple_solver.py:71-191):
 *   d_m0 [n][3] f64; d_pulse [n][3] f64 rows (J, t_pulse, t_end): current_func(t) = J if t <= t_pulse else 0 on (0, t_end);
 *   d_m_out [n][3] f64 last trajectory row; d_traj NULL or [n][traj_stride][3] f64 (rows 0..n_sub);
 *   d_n_sub [n] int32 out (may be NULL); d_guard [n] int32 out (may be NULL): 1 if the non-finite guard fired.
 * Arbitrary current_func / field_func callables cannot cross into a kernel; the host samples them at the stage times the
 * reference evaluates them at, (t_i, t_i + dt/2, t_i + dt) with t = linspace(0, t_end, n_sub + 1), dt = t_end / n_sub
 * (physics/simple_solver.py:137-145, 278-295), and passes the samples:
 *   d_current_grid NULL or [grid_envs][grid_stride][3] f64       J at the three times (replaces d_pulse's J, t_pulse)
 *   d_field_grid   NULL or [grid_envs][grid_stride][3][3] f64    H_app (A/m) at the three times (added to the table's field)
 *   grid_envs = 1 (one grid shared by every trajectory) or n_envs; substeps beyond grid_stride reuse the last row.
 * With either grid the solve runs the FP64 general-geometry stages (both entry points). */
typedef struct StgSttSolveArgs {
    const StgSttFolded* d_table;
    const int32_t* d_param_index;
    const double* d_m0;
    const double* d_pulse;
    double* d_m_out;
    double* d_traj;
    int64_t traj_stride;
    int32_t* d_n_sub;
    int32_t* d_guard;
    const double* d_noise;
    int64_t noise_stride;
    uint64_t seed;
    uint64_t env_offset;
    int64_t n_envs;
    int32_t n_sets;
    uint32_t flags;
    const double* d_current_grid;
    const double* d_field_grid;
    int64_t grid_stride;
    int32_t grid_envs;
    int32_t reserved;
} StgSttSolveArgs;

int stg_abi_version(void);
/* 1 if stg_stt_step_f32 (STG_F_AXIS_Z, RK4, STG_F_THERMAL_PHILOX) takes the two-envs-per-thread kernel for n_envs envs and these
 * flags on a GPU with sm_count SMs (<= 0: the current device), else 0. Both kernels give the same bits per env; this is the
 * dispatch rule of stt_kernels.cu made visible to tests and tools. */
int stg_stt_thermal_pair_dispatch(int64_t n_envs, uint32_t flags, int sm_count);
const char* stg_error_string(int code);

/* Host-side: fold n raw parameter sets into kernel constants (pure CPU, no CUDA call). Replaces the per-RHS-call
 * dict lookups + constant recomputation of physics/simple_solver.py:310-319, 358-380. */
int stg_stt_fold(const StgSttParams* params, int32_t n_sets, StgSttFolded* out);
/* 1 if every folded set has easy_axis == (0,0,1) and zero applied field (then STG_F_AXIS_Z may be passed). */
int stg_stt_all_axis_z(const StgSttFolded* folded_host, int32_t n_sets);

/* One SpinTorqueEnv.step for n_envs envs. Replaces envs/spin_torque_env.py:310-407 together with
 * utils/robust_solver.py:75 -> physics/simple_solver.py:71-191, devices/*:compute_resistance,
 * rewards/composite_reward.py:65-126 and the SafetyWrapper clamps (utils/monitoring.py:288-348). */
int stg_stt_step_f32(const StgSttStepArgs* args, void* stream);
int stg_stt_step_f64(const StgSttStepArgs* args, void* stream);

int stg_stt_reset(const StgSttResetArgs* args, void* stream);

/* Counting sort of envs by substep count (descending) so that warps are homogeneous when pulse durations differ
 * (physics/simple_solver.py:137-139 gives n in [10, 5000]). d_perm [n] int32 out; d_work >= STG_SORT_WORK_INTS int32
 * scratch (zeroed by the call). When every env has the same substep count the identity permutation is written, so the
 * sorted launch keeps coalesced accesses. The order inside one bin is unspecified; results never depend on it. */
#define STG_SORT_BINS 8192
#define STG_SORT_WORK_INTS (STG_SORT_BINS + 8)
int stg_stt_sort_by_substeps(const StgSttFolded* d_table, int32_t n_sets, const int32_t* d_param_index,
                             const float* d_action, int32_t* d_perm, int32_t* d_work, int64_t n_envs, void* stream);

int stg_stt_solve_f32(const StgSttSolveArgs* args, void* stream);
int stg_stt_solve_f64(const StgSttSolveArgs* args, void* stream);

/* ---- K2: adaptive RK45 (SciPy-compatible Dormand-Prince 5(4)) on the generalised LLGS right-hand side --------------------
 * One parameter set of the generalised RHS (FP64). LLGSSolver form (physics/llgs_solver.py:92-126, 182-237):
 *   H   = H_app + (2K/(mu0 Ms)) (m.e) e - Ms N (.) m + exchange_coeff m + h_th xi
 *   tau = J [ c_dl_p m x (m x p) + c_fl_p (m x p) + c_dl_s (sigma x m) + c_fl_s sigma ]      (0 when |J| < 1e-12)
 *   dm  = -gamma m x H;  dm += alpha m x dm;  dm += tau                     with m = y/|y| inside the RHS
 * STT (LLGSSolver._compute_spin_torques): c_dl_p = P gamma/(2 Ms V), c_fl_p = 0.1 c_dl_p, p = z^.
 * SOT (devices/sot_mram.py:163-194): c_dl_s / c_fl_s = tau_dl_factor / tau_fl_factor, sigma = z^ x J^.
 * VCMA (devices/vcma_mram.py:122-147): use_vcma = 1, K = K_eff(V) from the per-env voltage. */
typedef struct StgLlgParams {
    double gamma;
    double mu0;
    double alpha;
    double saturation_magnetization;
    double uniaxial_anisotropy;
    double volume;
    double easy_axis[3];             /* used as given (LLGSSolver does not normalise it)                          */
    double demag_n[3];               /* params['demag_factors'] (default 0,0,1) or N(aspect_ratio)                */
    double exchange_coeff;           /* (2 A_ex/(mu0 Ms))*0.1 if A_ex > 0 else 0 (physics/llgs_solver.py:204-209) */
    double h_th;                     /* sqrt(2 alpha k_B T/(gamma mu0 Ms V)), k_B = 1.380649e-23; 0 = no noise    */
    double c_dl_p, c_fl_p;
    double p_hat[3];
    double c_dl_s, c_fl_s;
    double sigma[3];
    double vcma_coefficient, dielectric_thickness, breakdown_voltage;
    int32_t use_vcma;
    int32_t reserved;
} StgLlgParams;

/* Argument block of a batched LLGSSolver.solve(m_initial, (t_start, t_end), params, current_func, field_func, thermal_noise,
 * temperature) with current_func(t) = J if t <= t_pulse else 0 and a constant H_app per trajectory, or - n_seg > 0 - with
 * piecewise-constant current_func / field_func tables evaluated at the controller's data-dependent stage times:
 *   d_seg_t       [seg_rows][n_seg]       ascending segment ends; segment k is (t_{k-1}, t_k] (right-closed, like `t <= t_pulse`),
 *                                         segment n_seg is everything after the last end
 *   d_seg_current [seg_rows][n_seg + 1]   current density of each segment (replaces d_current / d_t_pulse)
 *   d_seg_field   [seg_rows][n_seg + 1][3] applied field of each segment, or NULL (= d_happ)
 *   seg_rows      1 (one table shared by every trajectory) or n_envs
 *   d_t_start     [n] or NULL (= 0): solve_ivp integrates in absolute time (its minimum step is 10 ulp(t)); t_end > t_start
 *   d_table [n_sets] (DEVICE copy of StgLlgParams), d_param_index [n] or NULL
 *   d_m0 [n][3]; d_t_end [n]; d_current [n] or NULL; d_t_pulse [n] or NULL (= always on); d_happ [n][3] or NULL;
 *   d_voltage [n] or NULL
 *   outputs: d_y_out [n][3] raw end state (sol.y[:, -1]); d_n_accepted / d_n_rejected / d_n_rhs / d_status [n] int32
 *            (status bit0 step size too small (SciPy failure), bit1 trajectory buffer overflow, bit2 max_attempts reached,
 *            bit3 non-finite error norm); d_t_reached [n];
 *            d_traj NULL or [n][traj_stride][6] rows (t, m_x, m_y, m_z normalised, energy, |tau_DL|+|tau_FL|) for row 0 (t=0)
 *            and every accepted step, as LLGSSolver returns them (physics/llgs_solver.py:146-180)
 *   thermal: STG_F_THERMAL_PHILOX (counter = RHS evaluation index) or STG_F_THERMAL_INJECT with d_noise [n][noise_stride][3]
 *            consumed one row per RHS evaluation in call order (select_initial_step's two evaluations included). */
typedef struct StgRk45Args {
    const StgLlgParams* d_table;
    const int32_t* d_param_index;
    const double* d_m0;
    const double* d_t_end;
    const double* d_current;
    const double* d_t_pulse;
    const double* d_happ;
    const double* d_voltage;
    double* d_y_out;
    int32_t* d_n_accepted;
    int32_t* d_n_rejected;
    int32_t* d_n_rhs;
    int32_t* d_status;
    double* d_t_reached;
    double* d_traj;
    int64_t traj_stride;
    const double* d_noise;
    int64_t noise_stride;
    double rtol, atol, max_step;
    int64_t max_attempts;            /* safety bound on attempted steps per trajectory (0 = 1e6)                  */
    uint64_t seed;
    uint64_t env_offset;
    int64_t n_envs;
    int32_t n_sets;
    uint32_t flags;
    const int32_t* d_perm;           /* NULL or [n]: thread s integrates trajectory d_perm[s]; every array above stays indexed by
                                      * the trajectory, as does the Philox id (sort by (parameter set, t_end) for homogeneous warps) */
    const double* d_t_start;
    const double* d_seg_t;
    const double* d_seg_current;
    const double* d_seg_field;
    int32_t n_seg;
    int32_t seg_rows;
} StgRk45Args;

int stg_llgs_rk45_f64(const StgRk45Args* args, void* stream);
/* Estimated attempted steps per trajectory (d_cost [n]), the sort key for d_perm: (t_end - t_start) * max(1 / max_step,
 * 8 * (gamma |H_eff(m0)| + torque rate)). Reads the inputs of the argument block only. */
int stg_llgs_rk45_cost_f64(const StgRk45Args* args, double* d_cost, void* stream);
/* d_perm [n] int32 out: the trajectories counting-sorted by (parameter set, estimated cost descending, 1.5 % bins) - three small
 * launches; d_work >= STG_SORT_WORK_INTS int32. Pass the result as args->d_perm of stg_llgs_rk45_f64. */
int stg_llgs_rk45_sort_f64(const StgRk45Args* args, int32_t* d_perm, int32_t* d_work, void* stream);

/* ---- K3: SpinTorqueArray-v0 (envs/array_env.py) ------------------------------------------------------------------------- */
#define STG_ARRAY_INDIVIDUAL 0
#define STG_ARRAY_ROW 1
#define STG_ARRAY_COLUMN 2
#define STG_ARRAY_GLOBAL 3
#define STG_ARRAY_MAX_DEVICES 1024

typedef struct StgArrayParams {
    int32_t n_rows, n_cols;
    int32_t action_mode;             /* STG_ARRAY_*                                                                 */
    int32_t device_kind;             /* STG_DEV_*: which compute_effective_field / compute_resistance form          */
    int32_t max_steps;               /* 200 (envs/array_env.py:36)                                                  */
    int32_t reserved;
    double hk;                       /* 2 K_u / (mu0 Ms)                                                            */
    double saturation_magnetization;
    double easy_axis[3];             /* as given (devices/stt_mram.py:68-72)                                        */
    double demag_n[3];               /* SOT/VCMA shape factors; zeros for STT                                       */
    double resistance_parallel, resistance_antiparallel;
    double reference_magnetization[3];   /* normalised                                                              */
    double series_resistance;
    double area;
    double max_current, max_duration;
    double success_threshold, energy_penalty_weight;
} StgArrayParams;

/* One step of n_arrays independent crossbar arrays (envs/array_env.py:358-411). D = n_rows*n_cols devices per array.
 *   d_coupling  [D][D] f64 coupling matrix (envs/array_env.py:289-318) or NULL (include_coupling=False)
 *   d_pattern   [n][D][3] f64 current_pattern (updated in place); d_target [n][D][3] f64
 *   d_action    [n][3] f32 (idx, J, T); `global` mode: [n][2] f32 (J, T) with action_stride = 2
 *   outputs     d_obs [n][D][6] f32 (pattern, target), d_reward/d_step_energy/d_similarity [n] f64, flags [n] u8
 *   STG_F_AUTORESET: arrays that terminate/truncate are reset in the same call (random unit vectors from the Philox stream,
 *   target kept), d_final_obs receives the pre-reset observation (rows of arrays that keep running are not written). */
typedef struct StgArrayStepArgs {
    StgArrayParams params;
    const double* d_coupling;
    double* d_pattern;
    const double* d_target;
    double* d_total_energy;
    int32_t* d_step_count;
    int32_t* d_episode;
    const float* d_action;
    float* d_obs;
    double* d_reward;
    uint8_t* d_terminated;
    uint8_t* d_truncated;
    double* d_step_energy;
    double* d_similarity;
    float* d_final_obs;
    double* d_stats;                 /* [STG_STAT_REPLICAS][STG_NSTATS] (see StgSttStepOut.stats) or NULL           */
    uint64_t seed;
    uint64_t array_offset;
    int64_t n_arrays;
    int32_t action_stride;
    uint32_t flags;
} StgArrayStepArgs;

int stg_array_step_f64(const StgArrayStepArgs* args, void* stream);
/* Reset of the arrays with d_mask[i] != 0 (all if NULL): per-device normalised N(0,1)^3 from the Philox stream, or the rows
 * of d_pattern0 [n][D][3] (options['initial_pattern'], stored as given); counters zeroed; observation written. */
int stg_array_reset(const StgArrayStepArgs* args, const uint8_t* d_mask, const double* d_pattern0, void* stream);

/* ---- K4: batched device-class operations (FP64, one row per device state) -------------------------------------------------
 * Host struct passed by pointer; mirrors what the reference's device constructors cache (devices/sot_mram.py:61-76,
 * devices/vcma_mram.py:60-84). easy_axis is used AS GIVEN (the device methods do not normalise it);
 * reference_magnetization must already be normalised by the caller. */
typedef struct StgDeviceParams {
    int32_t kind;                    /* STG_DEV_*                                                                 */
    int32_t reserved;
    double saturation_magnetization;
    double uniaxial_anisotropy;
    double mu0;                      /* 4*pi*1e-7 (devices/base_device.py:30)                                     */
    double easy_axis[3];
    double demag_n[3];               /* (N_x, N_y, N_z) of devices/sot_mram.py:114-132; zeros for STT             */
    double vcma_coefficient;         /* VCMA: xi [J/(V m)]                                                        */
    double dielectric_thickness;     /* VCMA: t_d [m]                                                             */
    double breakdown_voltage;        /* VCMA: V_bd [V]                                                            */
    double tau_dl_factor;            /* SOT: damping_like_efficiency * j_s_efficiency                             */
    double tau_fl_factor;            /* SOT: field_like_efficiency * j_s_efficiency                               */
    double resistance_parallel;
    double resistance_antiparallel;
    double reference_magnetization[3];
    double series_resistance;        /* SOT: 0.1 * sheet_resistance_hm / (area*1e-12)                             */
} StgDeviceParams;

/* device.compute_effective_field(m, H_app[, V]) for n rows (devices/stt_mram.py:56-76, sot_mram.py:78-112,
 * vcma_mram.py:86-120). d_happ: NULL (zero), 1 row (broadcast) or n rows; d_voltage: VCMA only, NULL = 0 V.
 * d_zero_rows: NULL, or one int32 the kernel ADDS the number of STT rows with |m| < 1e-12 to: the reference raises
 * "Magnetization vector cannot be zero" for those (devices/base_device.py:112-114); the caller reads 4 bytes instead of
 * scanning its input. */
int stg_device_field_f64(const StgDeviceParams* p, const double* d_m, const double* d_happ, int32_t happ_rows,
                         const double* d_voltage, double* d_out, int64_t n, int32_t* d_zero_rows, void* stream);
/* device.compute_resistance(m) (devices/stt_mram.py:78-94, sot_mram.py:196-228, vcma_mram.py:236-257); d_zero_rows as above. */
int stg_device_resistance_f64(const StgDeviceParams* p, const double* d_m, double* d_out, int64_t n, int32_t* d_zero_rows,
                              void* stream);
/* SOTMRAMDevice.compute_spin_torque(J, m, direction) (devices/sot_mram.py:163-194); current_direction: 3 host doubles. */
int stg_device_sot_torque_f64(const StgDeviceParams* p, const double* d_current, int32_t current_rows, const double* d_m,
                              const double* current_direction, double* d_tau_dl, double* d_tau_fl, int64_t n, void* stream);
/* VCMAMRAMDevice._compute_effective_anisotropy(V) (devices/vcma_mram.py:122-147). */
int stg_vcma_anisotropy_f64(const StgDeviceParams* p, const double* d_voltage, double* d_out, int64_t n, void* stream);
/* ThermalFluctuations.generate_thermal_field (physics/thermal_model.py:75-137) for n devices: white noise (d_state NULL)
 * or Ornstein-Uhlenbeck x <- decay*x + sqrt(1-decay^2)*xi on d_state [n][3]; out = strength * x. Philox counter =
 * (offset + row, call_index). */
int stg_thermal_field_f64(double strength, double decay, double* d_state, double* d_out, uint64_t seed, uint64_t offset,
                          uint64_t call_index, int64_t n, void* stream);

/* ThermalFluctuations analytics (physics/thermal_model.py:46-73 compute_noise_strength, :139-258 compute_thermal_barrier /
 * compute_switching_probability / compute_retention_time, i.e. the body of generate_temperature_sweep :274-336) on a grid of
 * n_t temperatures x n_dev devices in one launch.
 *   d_temperature [n_t]; d_ku, d_volume, d_damping, d_ms [n_dev]; d_barrier [n_dev] energy barriers in J or NULL (= K_u V)
 *   d_out [4][n_t][n_dev]: stability factor, switching probability over measurement_time, retention time [s] at failure_rate,
 *                          noise strength [A/m]; T <= 0 gives (inf, 0, inf, 0) like the reference */
typedef struct StgThermalAnalyticsArgs {
    const double* d_temperature;
    const double* d_ku;
    const double* d_volume;
    const double* d_damping;
    const double* d_ms;
    const double* d_barrier;
    double* d_out;
    double k_b, mu0, gamma;          /* 1.380649e-23, 4 pi 1e-7, 2.21e5 (physics/thermal_model.py:31-33, 50) */
    double attempt_frequency, measurement_time, failure_rate;
    int32_t n_t, n_dev;
} StgThermalAnalyticsArgs;
int stg_thermal_analytics_f64(const StgThermalAnalyticsArgs* args, void* stream);

/* EnergyLandscape.compute_energy / compute_energy_gradient (physics/energy_landscape.py:36-104) for n states: m is
 * normalised, E = Zeeman + uniaxial + demag, gradient = H_app + H_anis + H_demag. Either output may be NULL. */
typedef struct StgEnergyParams {
    double mu0, saturation_magnetization, volume, uniaxial_anisotropy;
    double easy_axis[3];             /* as given                                   */
    double demag_factors[3];         /* params['demag_factors'], default (0, 0, 1) */
} StgEnergyParams;
int stg_energy_landscape_f64(const StgEnergyParams* p, const double* d_m, const double* d_happ, int32_t happ_rows,
                             double* d_energy, double* d_gradient, int64_t n, void* stream);

/* K5 standalone (the step kernels fuse the same reduction into their epilogue): ADD the statistics of n env-step results to
 * d_stats [STG_NSTATS] f64 (ONE vector, not the replicated buffer of the step kernels: this kernel reduces inside each CTA and
 * issues one atomic set per CTA; caller zeroes it once per rollout; reference analogue: EnvironmentMonitor's rolling sums,
 * utils/monitoring.py:89-116,180-229). Every input is [n] and may be NULL (its statistic then stays untouched, STEPS always
 * counts n): d_reward f64, d_step_energy f64, d_terminated / d_truncated u8, d_n_sub i32 substeps of the step, d_status i32
 * (bit0 = guard fired), d_step_count i32 step counter AFTER the step (summed into EPLEN where the episode ended). */
int stg_stats_reduce_f64(const double* d_reward, const double* d_step_energy, const uint8_t* d_terminated,
                         const uint8_t* d_truncated, const int32_t* d_n_sub, const int32_t* d_status, const int32_t* d_step_count,
                         int64_t n, double* d_stats, void* stream);
/* Column sums of the replicated statistics buffer of the step kernels: d_out[q] (+)= sum_r d_replicas[r][q], q < STG_NSTATS
 * (accumulate != 0 adds to d_out, 0 overwrites). d_out is what one all-reduce(SUM) per rollout exchanges between ranks. */
int stg_stats_fold_f64(const double* d_replicas, double* d_out, int32_t accumulate, void* stream);
/* Device-side address of a pinned, mapped host allocation. Every OUTPUT array of the step / reset entry points (obs,
 * final_obs, reward, terminated, truncated, ...) is write-only for the kernels, so it may live in pinned host memory: the
 * kernels then deliver results over PCIe while they run (posted writes, overlapped), instead of a serialised device-to-host
 * copy after the launch. The caller synchronises the stream before reading. */
int stg_host_device_pointer(void* host_ptr, void** device_ptr);

/* VectorizedMagneticsOperations (utils/vectorized_operations.py:288-393), n rows of 3 doubles, NumPy's operation order:
 *   CROSS           out[n][3] = a x b                              (batch_cross_product :292-303)
 *   DOT             out[n]    = sum(a*b, axis=1)                   (batch_dot_product   :305-316)
 *   NORMALIZE       out[n][3] = a / max(||a||, 1e-12), b unused    (batch_normalize     :318-330)
 *   ANIS_ENERGY     out[n]    = -p0*p1*(a.b)^2, p0 = K_u[n], p1 = volume[n], b = easy axis (batch_energy_computation :332-364)
 *   TMR_RESISTANCE  out[n]    = max(p0 (1 + ((p1-p0)/p0)(1 - a.b)/2), p0/2), p0 = R_P[n], p1 = R_AP[n]
 *                                                                  (batch_resistance_computation :366-393)
 * d_b holds 1 row (broadcast) or n rows. */
enum { STG_VEC3_CROSS = 0, STG_VEC3_DOT = 1, STG_VEC3_NORMALIZE = 2, STG_VEC3_ANIS_ENERGY = 3, STG_VEC3_TMR_RESISTANCE = 4 };
int stg_vec3_op_f64(int32_t op, const double* d_a, const double* d_b, int32_t b_rows, const double* d_p0, const double* d_p1,
                    double* d_out, int64_t n, void* stream);
/* EnergyLandscape.generate_phase_diagram (physics/energy_landscape.py:282-340): out[n_fields][n_currents] =
 * 1 if |field_i| > h_k - |beta * current_j| else 0, beta = P*2.21e5/(2 Ms V), h_k = 2 K_u/(mu0 Ms) (host doubles). */
int stg_phase_diagram_f64(const double* d_currents, const double* d_fields, int32_t n_currents, int32_t n_fields, double beta,
                          double h_k, double* d_out, void* stream);

/* ---- K6: generalised advantage estimation over a stored rollout ----------------------------------------------------------
 * Replaces Stable-Baselines3's RolloutBuffer.compute_returns_and_advantage together with the TimeLimit.truncated bootstrap of
 * OnPolicyAlgorithm.collect_rollouts (`rewards[idx] += gamma * terminal_value`), in float32 and SB3's expression order, every
 * product and sum rounded on its own (no contraction; spin_torque_rl_gym_b200/csrc/rollout_core.cuh). Every plane is
 * [n_steps][n_envs] row-major (time-major), device memory:
 *   d_reward f32        the env's reward of step t
 *   d_value f32         V(obs_t)
 *   d_terminated u8, d_truncated u8   the step's flags (nonzero = set; both may be set)
 *   d_final_value f32   V(final_observation_t); read only where truncated && !terminated, other entries may hold anything (NaN)
 *   d_last_value f32 [n_envs]          V of the observation after step n_steps - 1
 *   d_advantage f32 out; d_return f32 out (= advantage + value) or NULL
 * With done_t = term_t | trunc_t, nnt_t = 1 - done_t, v_next = value_{t+1} (d_last_value at the last step), adv_{n_steps} = 0:
 *   r_t = reward_t + gamma * final_value_t where trunc_t && !term_t (else reward_t)
 *   adv_t = ((r_t + (gamma * v_next) * nnt_t) - value_t) + (gamma_lambda * nnt_t) * adv_{t+1}
 * gamma = float32(gamma), gamma_lambda = float32(gamma * gae_lambda) with the product in double: what SB3's NumPy evaluates.
 * Errors: args NULL -> STG_E_NULL; a negative size -> STG_E_SIZE; n_steps == 0 or n_envs == 0 -> STG_OK without a launch;
 * then any NULL pointer except d_return -> STG_E_NULL. */
typedef struct StgGaeArgs {
    const float* d_reward;
    const float* d_value;
    const uint8_t* d_terminated;
    const uint8_t* d_truncated;
    const float* d_final_value;
    const float* d_last_value;
    float* d_advantage;
    float* d_return;
    float gamma;
    float gamma_lambda;
    int64_t n_steps;
    int64_t n_envs;
} StgGaeArgs;
int stg_rollout_gae_f32(const StgGaeArgs* args, void* stream);

/* ---- K7: one shuffled PPO minibatch gathered from a stored rollout ---------------------------------------------------------
 * Replaces the fancy indexing of Stable-Baselines3's RolloutBuffer.get / _get_samples (`self.observations[batch_inds]`, ...)
 * for one minibatch of a uniform random permutation of the n_steps * n_envs samples, without materialising the permutation.
 * Source planes are the collector's time-major device planes; destinations are dense rows:
 *   d_obs [n_steps][n_envs][12] -> d_obs_out [batch][12]     (both 16-B aligned, else STG_E_ALIGN)
 *   d_action [n_steps][n_envs][2] -> d_action_out [batch][2] (both 8-B aligned, else STG_E_ALIGN)
 *   d_value, d_log_prob, d_advantage, d_return [n_steps][n_envs] -> [batch]
 * With M = n_steps * n_envs, output row k (0 <= k < batch) is a copy of sample f = rollout_permute(round_keys, M, start + k),
 * the flat time-major index f = t * n_envs + i (spin_torque_rl_gym_b200/csrc/rollout_core.cuh): a balanced 8-round Feistel
 * network over the smallest even number b >= 2 of bits with 2^b >= M, round r = (murmur3 fmix32(right ^ round_keys[r])) masked
 * to b/2 bits, cycle-walked into [0, M). It is a bijection of [0, M) for every key set, so positions 0 .. M-1 taken in
 * consecutive minibatches visit every sample exactly once. SB3 permutes the env-major flattening (i * n_steps + t) instead;
 * for a uniform random permutation the two orders differ only by a fixed relabelling of the samples. Values are copied bit
 * for bit, never converted. The keys come from the caller (RolloutCollector derives them from the env's seed, env_offset
 * and the epoch), so the library needs no random state.
 * Each (source, destination) pair is either both NULL (that plane is skipped) or both set.
 * Errors, in this order: args NULL -> STG_E_NULL; a negative size, n_steps * n_envs overflowing or above 2^62 -> STG_E_SIZE;
 * batch == 0 or an empty rollout -> STG_OK without a launch; start + batch > n_steps * n_envs -> STG_E_SIZE; a pair with
 * only one pointer set, or no pair set -> STG_E_NULL; a misaligned observation or action pointer -> STG_E_ALIGN. */
typedef struct StgMinibatchArgs {
    const float* d_obs;
    float* d_obs_out;
    const float* d_action;
    float* d_action_out;
    const float* d_value;
    float* d_value_out;
    const float* d_log_prob;
    float* d_log_prob_out;
    const float* d_advantage;
    float* d_advantage_out;
    const float* d_return;
    float* d_return_out;
    uint32_t round_keys[8];
    int64_t n_steps;
    int64_t n_envs;
    int64_t start;   /* first permutation position of this minibatch */
    int64_t batch;   /* rows in it */
} StgMinibatchArgs;
int stg_rollout_minibatch_f32(const StgMinibatchArgs* args, void* stream);

/* ---- K8: VecNormalize, running observation and return normalisation of the STT vector env -------------------------------
 * Replaces Stable-Baselines3's VecNormalize.step_wait / reset / normalize_obs / normalize_reward with RunningMeanStd, in float64
 * and SB3's expression order (spin_torque_rl_gym_b200/csrc/vecnorm_core.cuh). A wrapped step is three launches on one stream,
 * with an optional gather of the moment vectors across ranks between the first two:
 *   stg_vecnorm_moments_f32  with d_reward set: d_returns = d_returns * gamma + d_reward (two roundings). Then the moments of the
 *                            n rows of the 12 observation columns and of the return column (zero when d_reward is NULL, which
 *                            leaves d_returns untouched) are reduced in FP64 into d_moments[0 .. STG_VECNORM_MOMENTS).
 *                            The reduction order is fixed: STG_VECNORM_GRID(n) CTAs write partials into d_work, the last CTA
 *                            folds them in a fixed tree, so the bits depend only on n and the data.
 *   stg_vecnorm_merge_f64    folds the n_ranks moment vectors d_moments [n_ranks][STG_VECNORM_MOMENTS] in rank order (Chan's
 *                            pairwise update) and applies RunningMeanStd.update_from_moments in place to d_stats: to obs_rms when
 *                            flags has TRAINING and NORM_OBS, to ret_rms when flags has TRAINING and d_reward is set (d_reward is
 *                            not read). One CTA, so no CTA reads statistics another one writes.
 *   stg_vecnorm_apply_f32    with the statistics in d_stats (not updated):
 *                            d_obs_out = clip((d_obs - mean) / sqrt(var + epsilon), +-clip_obs) computed in f64 and rounded to f32
 *                            (a copy without NORM_OBS); the same for the rows of d_final_obs of envs with terminated | truncated
 *                            into d_final_obs_out (other rows are neither read nor written);
 *                            d_reward_out = clip(d_reward / sqrt(ret_var + epsilon), +-clip_reward) (a copy without NORM_REWARD);
 *                            d_returns of envs with terminated | truncated set to 0 (when d_returns and the flags are set).
 *                            Each (input, output) pair may be skipped with both pointers NULL.
 * Moment vector (doubles): [0] n, [1 + f] mean, [1 + 13 + f] M2 = sum of squared deviations, f = 0..11 observation columns, 12 the
 * return. Statistics (doubles): obs_rms mean [0..12), var [12..24), count [24]; ret_rms mean [25], var [26], count [27]; SB3 starts
 * them at mean 0, var 1, count 1e-4. d_work: STG_VECNORM_WORK_DOUBLES doubles whose last 8 bytes hold a CTA counter that must be
 * zero before the first call (every call leaves it zero); it serves one stream at a time.
 * Only the 12-float STT observation is supported. d_obs, d_final_obs and both observation outputs are 16-B aligned.
 * Errors, in this order: args NULL -> STG_E_NULL; n_envs < 0 -> STG_E_SIZE; n_envs == 0 -> STG_OK without a launch; a
 * required pointer NULL or a half-set pair -> STG_E_NULL; a misaligned observation pointer -> STG_E_ALIGN. The merge reads no
 * per-env array and ignores n_envs: n_ranks < 1 -> STG_E_SIZE.
 * Required: moments d_obs, d_moments, d_work, and d_returns with d_reward; merge d_moments, d_stats; apply d_stats, at least one
 * pair, d_terminated and d_truncated with the final pair. */
#define STG_VECNORM_FEATURES 13
#define STG_VECNORM_MOMENTS 27
#define STG_VECNORM_STATS 28
#define STG_VECNORM_OBS_MEAN 0
#define STG_VECNORM_OBS_VAR 12
#define STG_VECNORM_OBS_COUNT 24
#define STG_VECNORM_RET_MEAN 25
#define STG_VECNORM_RET_VAR 26
#define STG_VECNORM_RET_COUNT 27
#define STG_VECNORM_THREADS 256
#define STG_VECNORM_MAX_CTAS 296
#define STG_VECNORM_GRID(n) ((n) <= 0 ? 0 : ((n) + STG_VECNORM_THREADS - 1) / STG_VECNORM_THREADS < STG_VECNORM_MAX_CTAS \
                             ? ((n) + STG_VECNORM_THREADS - 1) / STG_VECNORM_THREADS : STG_VECNORM_MAX_CTAS)
#define STG_VECNORM_WORK_DOUBLES (STG_VECNORM_MAX_CTAS * STG_VECNORM_MOMENTS + 1)
#define STG_VECNORM_TRAINING 0x1u
#define STG_VECNORM_NORM_OBS 0x2u
#define STG_VECNORM_NORM_REWARD 0x4u
typedef struct StgVecNormArgs {
    const float* d_obs;              /* [n][12] raw observations                                     */
    const float* d_final_obs;        /* [n][12] raw final observations (rows of ended envs) or NULL   */
    const uint8_t* d_terminated;     /* [n]                                                          */
    const uint8_t* d_truncated;      /* [n]                                                          */
    const double* d_reward;          /* [n] raw reward or NULL                                       */
    double* d_returns;               /* [n] discounted returns                                       */
    double* d_stats;                 /* [STG_VECNORM_STATS]                                          */
    double* d_moments;               /* moments: [STG_VECNORM_MOMENTS] out; merge: [n_ranks][...] in  */
    double* d_work;                  /* [STG_VECNORM_WORK_DOUBLES]                                   */
    float* d_obs_out;                /* [n][12]                                                      */
    float* d_final_obs_out;          /* [n][12]                                                      */
    double* d_reward_out;            /* [n]                                                          */
    double gamma, epsilon, clip_obs, clip_reward;
    int64_t n_envs;
    int32_t n_ranks;
    uint32_t flags;                  /* STG_VECNORM_*                                                */
} StgVecNormArgs;
int stg_vecnorm_moments_f32(const StgVecNormArgs* args, void* stream);
int stg_vecnorm_merge_f64(const StgVecNormArgs* args, void* stream);
int stg_vecnorm_apply_f32(const StgVecNormArgs* args, void* stream);

/* ---- K9: ActorCriticPolicy rollout inference (Stable-Baselines3's PPO MlpPolicy) ------------------------------------------
 * The forward pass of SB3's ActorCriticPolicy for PPO's MlpPolicy on the 12-float observation and the 2-float action:
 * separate actor and critic MLPs 12 -> 64 -> 64 (tanh), action_net 64 -> 2 (the Gaussian mean), value_net 64 -> 1, and a
 * state-independent log_std. The kernels are specialised for this architecture. Arithmetic: FP32, per env
 * (spin_torque_rl_gym_b200/csrc/policy_core.cuh):
 *   every layer output o is acc = b[o], then acc = fma(x[k], W[k][o], acc) for k = 0, 1, ..., K-1 in that order (no split-K),
 *   hidden outputs go through tanhf (full precision);
 *   eps0, eps1 = box_muller(Philox4x32-10 with key (key[0], key[1]) at counter (gid lo, gid hi, draw lo, draw hi)), words 0
 *   and 1, gid = env_offset + i (llgs_core.cuh's Philox and box_muller);
 *   a_d = mean_d + eps_d * std_d (two roundings), or mean_d with STG_POLICY_DETERMINISTIC;
 *   log_prob = sum over d of ((-((a_d - mean_d)^2) / (2 * std_d^2) - log_std_d) - log(sqrt(2 pi))), torch's
 *   Normal.log_prob term by term with each operation rounded on its own and IEEE division; log_std_d = the packed LOG_SCALE;
 *   env_action_d = lo_d + (hi_d - lo_d) * ((clip(a_d, -1, 1) + 1) / 2), each operation rounded on its own.
 * So every env's outputs depend only on its own row, the weights and (key, gid, draw): not on n, the launch geometry or the
 * partition of the envs over launches or GPUs.
 *
 * Weights: one buffer of STG_POLICY_FLOATS floats, 16-B aligned, at the offsets below. Matrices are k-major: W[k][o] (input k,
 * output o) at W + k * n_out + o, i.e. the transpose of torch's Linear.weight [out][in]. STD = exp(log_std) and LOG_SCALE =
 * log(STD) are computed by the caller (torch) when the buffer is packed; the last three floats are padding.
 *
 *   stg_policy_act_f32    reads d_obs [n][12]; writes whichever of d_obs_copy [n][12] (a copy of d_obs), d_action [n][2]
 *                         (the raw sample), d_env_action [n][2], d_value [n], d_log_prob [n] is not NULL. d_mask is ignored.
 *   stg_policy_value_f32  the critic only: d_value [i] = V(d_obs[i]) for every row i with d_mask[i] != 0 (u8 [n]; NULL: all
 *                         rows). Other rows are neither read nor written. Each CTA compacts the selected rows of its windows
 *                         before computing them, so the work scales with the number of selected rows.
 * Errors, in this order: args NULL -> STG_E_NULL; n_envs < 0 -> STG_E_SIZE; n_envs == 0 -> STG_OK without a launch; d_obs or
 * d_weights NULL, act without any output, value with d_value NULL -> STG_E_NULL; d_obs, d_weights or d_obs_copy not 16-B
 * aligned, d_action or d_env_action not 8-B aligned -> STG_E_ALIGN; flags other than STG_POLICY_DETERMINISTIC -> STG_E_ENUM. */
#define STG_POLICY_OBS 12
#define STG_POLICY_HIDDEN 64
#define STG_POLICY_ACTIONS 2
#define STG_POLICY_PI_W1 0          /* [12][64]  mlp_extractor.policy_net.0.weight, transposed */
#define STG_POLICY_PI_B1 768        /* [64]      mlp_extractor.policy_net.0.bias              */
#define STG_POLICY_PI_W2 832        /* [64][64]  mlp_extractor.policy_net.2.weight, transposed */
#define STG_POLICY_PI_B2 4928       /* [64]                                                   */
#define STG_POLICY_VF_W1 4992       /* [12][64]  mlp_extractor.value_net.0.weight, transposed  */
#define STG_POLICY_VF_B1 5760
#define STG_POLICY_VF_W2 5824       /* [64][64]  mlp_extractor.value_net.2.weight, transposed  */
#define STG_POLICY_VF_B2 9920
#define STG_POLICY_ACT_W 9984       /* [64][2]   action_net.weight, transposed                 */
#define STG_POLICY_ACT_B 10112      /* [2]                                                    */
#define STG_POLICY_VAL_W 10114      /* [64]      value_net.weight                             */
#define STG_POLICY_VAL_B 10178      /* [1]                                                    */
#define STG_POLICY_LOG_STD 10179    /* [2]       log_std                                      */
#define STG_POLICY_STD 10181        /* [2]       exp(log_std)                                 */
#define STG_POLICY_LOG_SCALE 10183  /* [2]       log(exp(log_std))                            */
#define STG_POLICY_PARAMS 10181     /* SB3's parameters: everything before STD                */
#define STG_POLICY_FLOATS 10188
#define STG_POLICY_DETERMINISTIC 0x1u
typedef struct StgPolicyArgs {
    const float* d_obs;              /* [n][12]                                                      */
    const float* d_weights;          /* [STG_POLICY_FLOATS]                                          */
    const uint8_t* d_mask;           /* value: [n] or NULL                                           */
    float* d_obs_copy;               /* act: [n][12] or NULL                                         */
    float* d_action;                 /* act: [n][2] or NULL                                          */
    float* d_env_action;             /* act: [n][2] or NULL                                          */
    float* d_value;                  /* [n]; act: or NULL                                            */
    float* d_log_prob;               /* act: [n] or NULL                                             */
    float action_low[2];             /* the env's action Box, for d_env_action                      */
    float action_high[2];
    uint32_t key[2];                 /* Philox key of the action noise                               */
    uint64_t draw;                   /* noise draw index: one per sampling launch                    */
    uint64_t env_offset;             /* global id of row 0                                           */
    int64_t n_envs;
    uint32_t flags;                  /* STG_POLICY_DETERMINISTIC                                     */
    uint32_t reserved;
} StgPolicyArgs;
int stg_policy_act_f32(const StgPolicyArgs* args, void* stream);
int stg_policy_value_f32(const StgPolicyArgs* args, void* stream);

/* ---- K10: PPO loss and gradient of the ActorCriticPolicy (Stable-Baselines3's PPO.train() minibatch step) ---------------
 * For one minibatch of B rows (the RolloutBufferSamples planes, device memory) and the K9 weight buffer, computes the loss of
 * SB3's PPO.train() and its gradient with respect to every parameter: what `loss.backward()` leaves in `.grad`.
 * Per row i, in FP32:
 *   forward: K9's arithmetic exactly (the same fma chains in ascending k, tanhf, pol_log_prob_term), so values_i and
 *            logp_i are bit-equal to stg_policy_act_f32's for the same weights, observation and action;
 *   A_i = (adv_i - mean) / (std + 1e-8f) with mean = d_adv_stats[0], std = d_adv_stats[1] (each operation IEEE-rounded:
 *         torch's `(adv - adv.mean()) / (adv.std() + 1e-8)` bit for bit), or adv_i when d_adv_stats is NULL;
 *   ratio_i = expf(logp_i - old_log_prob_i); c_i = min(max(ratio_i, ratio_lo), ratio_hi);
 *   pmin_i = min(A_i * ratio_i, A_i * c_i);  clipped_i = |ratio_i - 1| > clip_range;
 *   vpred_i = values_i, or old_value_i + clamp(values_i - old_value_i, -clip_range_vf, clip_range_vf) with STG_PPO_CLIP_VF;
 *   kl_i = (ratio_i - 1) - (logp_i - old_log_prob_i).
 * Losses (d_losses, 6 floats, in this order; sums over rows in FP64, the rest in FP64 and rounded once):
 *   [0] loss = policy_loss + ent_coef * entropy_loss + vf_coef * value_loss   [1] policy_loss = -sum(pmin) / B
 *   [2] value_loss = sum((return - vpred)^2) / B   [3] entropy_loss = -sum_d(float32(0.5 + 0.5 log 2 pi) + LOG_SCALE_d)
 *   [4] approx_kl = sum(kl) / B   [5] clip_fraction = count(clipped) / B
 * Gradient: torch autograd's rules. torch.min sends half the gradient to each side at a tie (A_i * ratio_i == A_i * c_i
 * compared in FP32); clamp passes it on the closed interval. So d pmin / d ratio = A_i where A_i * ratio_i < A_i * c_i or
 * (a tie with ratio_lo <= ratio_i <= ratio_hi), A_i / 2 at a tie outside it, 0 otherwise; the value clip likewise. Through
 * ratio = exp(.), Normal.log_prob with scale = exp(log_std) and the tanh layers; the entropy adds -ent_coef to each log_std.
 * Each layer's weight gradient is summed over a tile of STG_PPO_TILE rows in FP32 (fma chains in ascending row), the tile sums
 * are accumulated in FP64 per CTA, and a second launch folds the STG_PPO_GRID(B) CTA partials in CTA order in FP64 and scales
 * them by 1/B (the actor) or 2 vf_coef/B (the critic) before one rounding to FP32. No floating-point atomics: the bits of the
 * gradient and of the losses depend only on B, the weights and the data, not on the device, the stream or the addresses.
 *
 * d_grad: STG_POLICY_PARAMS floats, torch's parameter layout: every parameter at the offset of its K9 buffer slot (the
 * STG_PPO_GRAD_* offsets equal STG_POLICY_*) but with matrices in Linear.weight's [out][in] order. It is overwritten.
 * d_work: STG_PPO_WORK_DOUBLES(B) doubles; CTA b's partial is [b * STG_PPO_PART, (b + 1) * STG_PPO_PART): gradient sums in
 * the d_grad layout, then the four loss sums at STG_PPO_PART_LOSS (pmin, squared value error, kl, clipped count).
 * The Python caller computes ratio_lo = float32(1 - clip_range), ratio_hi = float32(1 + clip_range) in double first.
 * Errors, in this order: args NULL -> STG_E_NULL; batch < 1 -> STG_E_SIZE; any pointer other than d_adv_stats NULL ->
 * STG_E_NULL; d_weights or d_obs not 16-B aligned, d_action or d_work not 8-B aligned, any other pointer not 4-B aligned ->
 * STG_E_ALIGN; flags other than STG_PPO_CLIP_VF -> STG_E_ENUM. */
#define STG_PPO_TILE 128
#define STG_PPO_MAX_CTAS 296
#define STG_PPO_GRID(b) ((b) <= 0 ? 0 : ((b) + STG_PPO_TILE - 1) / STG_PPO_TILE < STG_PPO_MAX_CTAS \
                         ? ((b) + STG_PPO_TILE - 1) / STG_PPO_TILE : STG_PPO_MAX_CTAS)
#define STG_PPO_PART 10192          /* doubles per CTA partial                                       */
#define STG_PPO_PART_LOSS 10181     /* the four loss sums within a partial                           */
#define STG_PPO_WORK_DOUBLES(b) ((int64_t)STG_PPO_GRID(b) * STG_PPO_PART)
#define STG_PPO_LOSSES 6
#define STG_PPO_GRAD_PI_W1 0        /* [64][12]  d mlp_extractor.policy_net.0.weight */
#define STG_PPO_GRAD_PI_B1 768
#define STG_PPO_GRAD_PI_W2 832      /* [64][64]  */
#define STG_PPO_GRAD_PI_B2 4928
#define STG_PPO_GRAD_VF_W1 4992     /* [64][12]  d mlp_extractor.value_net.0.weight  */
#define STG_PPO_GRAD_VF_B1 5760
#define STG_PPO_GRAD_VF_W2 5824     /* [64][64]  */
#define STG_PPO_GRAD_VF_B2 9920
#define STG_PPO_GRAD_ACT_W 9984     /* [2][64]   d action_net.weight             */
#define STG_PPO_GRAD_ACT_B 10112
#define STG_PPO_GRAD_VAL_W 10114    /* [1][64]   d value_net.weight              */
#define STG_PPO_GRAD_VAL_B 10178
#define STG_PPO_GRAD_LOG_STD 10179  /* [2]       d log_std                       */
#define STG_PPO_CLIP_VF 0x1u
typedef struct StgPpoArgs {
    const float* d_weights;          /* [STG_POLICY_FLOATS] the K9 buffer                            */
    const float* d_obs;              /* [B][12]                                                      */
    const float* d_action;           /* [B][2] raw actions (policy units)                            */
    const float* d_old_value;        /* [B]                                                          */
    const float* d_old_log_prob;     /* [B]                                                          */
    const float* d_advantage;        /* [B]                                                          */
    const float* d_return;           /* [B]                                                          */
    const float* d_adv_stats;        /* [2] mean, std of d_advantage, or NULL: no normalisation       */
    float* d_grad;                   /* [STG_POLICY_PARAMS] out                                      */
    float* d_losses;                 /* [STG_PPO_LOSSES] out                                         */
    double* d_work;                  /* [STG_PPO_WORK_DOUBLES(B)]                                    */
    float clip_range, ratio_lo, ratio_hi, clip_range_vf;
    float ent_coef, vf_coef;
    uint32_t flags;                  /* STG_PPO_CLIP_VF                                              */
    uint32_t reserved;
    int64_t batch;
} StgPpoArgs;
int stg_policy_ppo_grad_f32(const StgPpoArgs* args, void* stream);

/* ---- K11: clipped Adam step of the ActorCriticPolicy (clip_grad_norm_ + torch.optim.Adam, SB3's PPO optimiser) -----------
 * One launch of one CTA over the STG_POLICY_PARAMS parameters in the K10 gradient layout, in this order:
 * 1. Gate. With d_gate set and *d_gate == 0: nothing is read or written. Otherwise, with d_losses and d_log set, the K10 losses
 *    of the minibatch are logged (in FP64): d_log[LOG_PG, LOG_VALUE, LOG_ENTROPY, LOG_CLIP] += d_losses[1, 2, 3, 5],
 *    d_log[LOG_COUNT] += 1, d_log[LOG_EPOCH_KL] += d_losses[4], d_log[LOG_EPOCH_COUNT] += 1, d_log[LOG_LAST_LOSS] = d_losses[0].
 *    Then, with STG_ADAM_TARGET_KL, if (double)d_losses[4] > 1.5 * target_kl: *d_gate = 0 and the update is skipped (SB3
 *    checks approx_kl before backward() and the step; the minibatch that trips the gate is logged).
 * 2. Clip (STG_ADAM_CLIP). sum = the FP64 sum of (double)g * (double)g over d_grad: thread t of STG_ADAM_THREADS adds the
 *    elements t, t + STG_ADAM_THREADS, ... in ascending order (each product and sum rounded), then a tree halves the partials
 *    (partial[t] += partial[t + h] for h = STG_ADAM_THREADS / 2, ..., 1). No atomics: the bits depend only on the gradient.
 *    total_norm = float32(sqrt(sum)); clip_coef = float32(1 / float32(total_norm + 1e-6f)) * float32(max_grad_norm) (torch
 *    evaluates `max_norm / t` as t.reciprocal() * max_norm); clip_coef = 1 if it is > 1 (NaN stays NaN). Every element is
 *    multiplied by clip_coef, also when it is 1, and written back to d_grad: clip_grad_norm_'s in-place result.
 * 3. Adam: torch.optim.Adam's single-tensor update (no weight decay, no amsgrad, not maximize). *d_step += 1.0f (float32);
 *    s = (double)*d_step; bc1 = 1 - pow(beta1, s), bc2 = 1 - pow(beta2, s) in FP64; these scalars are rounded to float32 once:
 *      w1 = float32(1 - beta1), b2 = float32(beta2), w2 = float32(1 - beta2), eps_f = float32(eps),
 *      step_size = float32(lr / bc1), bc2_sqrt = float32(sqrt(bc2)).
 *    (pow is CUDA's double pow, accurate to 2 ulp: in rare steps these two scalars may differ in their last bit from a host
 *    evaluation with a correctly rounded pow.)
 *    Per element, in float32 with every operation IEEE-rounded on its own (no contraction):
 *      m = w1 < 0.5f ? m + w1 * (g - m) : g - (g - m) * (1 - w1)      (torch's lerp formula)
 *      v = v * b2 + (w2 * g) * g                                       (mul_, then addcmul_)
 *      denom = sqrt(v) / bc2_sqrt + eps_f
 *      p = p - (step_size * m) / denom                                 (addcdiv_ with value = -step_size)
 *    with g the clipped gradient. The element at offset i of the K10 layout is parameter segment s (the last STG_PPO_GRAD_*
 *    offset <= i) and is read and written at d_param[s][i - offset_s].
 * d_log: STG_ADAM_LOG doubles at the STG_ADAM_LOG_* slots. The caller zeroes it before the first minibatch of PPO.train() and
 * zeroes the two per-epoch slots at the start of every epoch: SB3 logs the means of pg, value and entropy losses and clip
 * fractions over every minibatch evaluated, approx_kl over the last epoch, and the loss of the last minibatch evaluated.
 * Errors, in this order: args NULL -> STG_E_NULL; a d_param, d_grad, d_exp_avg, d_exp_avg_sq or d_step pointer NULL ->
 * STG_E_NULL; a float or int32 pointer not 4-B aligned or d_log not 8-B aligned -> STG_E_ALIGN; flags other than
 * STG_ADAM_CLIP | STG_ADAM_TARGET_KL -> STG_E_ENUM; STG_ADAM_TARGET_KL with d_losses or d_gate NULL -> STG_E_NULL. */
#define STG_ADAM_THREADS 1024
#define STG_ADAM_TENSORS 13        /* the parameters, in STG_PPO_GRAD_* order                         */
#define STG_ADAM_LOG 8             /* d_log layout, below                                             */
#define STG_ADAM_LOG_PG 0          /* sum of policy_loss over the minibatches logged                  */
#define STG_ADAM_LOG_VALUE 1       /* sum of value_loss                                               */
#define STG_ADAM_LOG_ENTROPY 2     /* sum of entropy_loss                                             */
#define STG_ADAM_LOG_CLIP 3        /* sum of clip_fraction                                            */
#define STG_ADAM_LOG_COUNT 4       /* minibatches logged                                              */
#define STG_ADAM_LOG_EPOCH_KL 5    /* sum of approx_kl over the minibatches logged in this epoch       */
#define STG_ADAM_LOG_EPOCH_COUNT 6 /* minibatches logged in this epoch                                */
#define STG_ADAM_LOG_LAST_LOSS 7   /* loss of the last minibatch logged                               */
#define STG_ADAM_CLIP 0x1u         /* clip the global L2 norm to max_grad_norm                        */
#define STG_ADAM_TARGET_KL 0x2u    /* gate on d_losses[4] (approx_kl) > 1.5 * target_kl               */
typedef struct StgAdamArgs {
    float* d_param[STG_ADAM_TENSORS];  /* each parameter's own contiguous storage (the nn.Parameter data) */
    float* d_grad;                     /* [STG_POLICY_PARAMS] K10 layout; clipped in place, as clip_grad_norm_ does */
    float* d_exp_avg;                  /* [STG_POLICY_PARAMS] */
    float* d_exp_avg_sq;               /* [STG_POLICY_PARAMS] */
    float* d_step;                     /* [1] Adam's step count, float32 as torch keeps it */
    const float* d_losses;             /* [STG_PPO_LOSSES] K10's losses of this minibatch, or NULL */
    int32_t* d_gate;                   /* [1] 1 open / 0 closed, or NULL */
    double* d_log;                     /* [STG_ADAM_LOG] or NULL */
    double lr, beta1, beta2, eps, max_grad_norm, target_kl;
    uint32_t flags, reserved;
} StgAdamArgs;
int stg_policy_adam_f32(const StgAdamArgs* args, void* stream);

/* FMA-pipe throughput probe (bench.py's measured FP32/FP64 roofline denominator): blocks*256 threads x iters*64 FMAs.
 * f64 = 0: FFMA, 1: DFMA, 2: packed FFMA2 (iters*64 instructions = iters*128 FMAs per thread).
 * d_out: >= blocks*256 elements of the probed type (8 bytes each for modes 1, 2; never written in practice). */
int stg_probe_fma(void* d_out, int32_t blocks, int32_t iters, int32_t f64, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* STG_H_ */
