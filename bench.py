#!/usr/bin/env python
"""bench.py — LLGS hot-path benchmark (driver contract: one JSON line on stdout from rank 0).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

`--dump-outputs DIR` (e.g. bench_outputs/) writes what the last timed step returned as DIR/<name>.npy, so that two builds run
with the same arguments (hence the same inputs) can be compared output for output.

A "step" is one env.step() of every env of the workload = one launch of the fused K1 kernel per GPU.
Workload (config.workload): BASELINE configs[1] physics — SpinTorque-v0, stt_mram reference defaults, T = 300 K thermal
fluctuations from the in-kernel stream (xoshiro128++ seeded per env-step from Philox4x32-10), RK4 fixed dt (pulse 1 ns -> 999 substeps per step), random current
densities — at the env count the metric is quoted on: 1,048,576 envs per GPU (weak scaling: every rank owns that many).

  value      LLGS substeps/s, whole job, actions/state/obs resident in HBM (device-timed, max over ranks)
  e2e        same metric through the public API (SpinTorqueVectorEnv.step) with HOST numpy actions: pinned H2D of the
             actions and D2H of obs/reward/flags inside the timed region
  roofline   dominant kernel (stt_env_step_kernel) against the FP32 FMA pipe (the path is not HBM- or tensor-bound)
  cpu_baseline  the reference's CPU path on the box's host cores, bounded sample: the LIVE reference (sanitised
             SpinTorqueEnv.step, one process per core, kind "reference") when a checkout is reachable (tools/time_live_reference.py
             probes $STG_REFERENCE, baseline/_ref, oracle/_ref, /root/reference), else the C restatement of the same algorithm
             (oracle/c, kind "port"); the port's figure is reported in both cases

`--impl reference` times that CPU path alone, on all host cores (rank 0 only under torchrun). The reference is a pure-Python
package whose own packaging installs 3 of its 62 modules, so it does not travel to the GPU box (DESIGN.md §5): there the arm is
the port and its line says why.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

N_ENVS_PER_GPU = 1 << 20
PULSE_S = 1e-9                 # float32(1e-9) floors to 999 substeps (physics/simple_solver.py:137-139)
FLOP_RK4_THERMAL = 329         # SURVEY §8(d): algorithmic flops per RK4 substep, thermal on
FLOP_RK4 = 301
# FP32 flops the dispatched thermal kernel EXECUTES per env-substep (FFMA2 = 4, FMUL2 / FADD2 = 2 per instruction and two envs;
# SASS instruction mix of its substep loop, profiles/r02_sass_stats.txt): 190 in the four RK4 stages, the combination, the
# renormalisation and the compensated state update + 42 in Box-Muller. The e = z stage drops the structural zeros of the 329.
FLOP_RK4_THERMAL_EXECUTED = 232
# one launch of the headline kernel at 1,048,576 envs x 999 substeps under `ncu --set full` (profiles/, condensed CSV):
# dram__bytes_read.sum + dram__bytes_write.sum and the pipe utilisations (pct of peak sustained active)
# (profiles/r02_ncu_stt_env_step_pair_f32_thermal1_xoshiro.csv; 85.8 MB read + 116.2 MB written: the FP64 state planes and the
# per-step diagnostics make it 1.3x the 150 B per env-step of SURVEY 8(d); 23 GB/s, irrelevant against the FP32 pipes)
NCU_TRAFFIC_BYTES = 202.0e6
NCU_PIPES = {"fma": 52.0, "fma_heavy": 51.7, "xu": 66.6, "alu": 40.6, "fp64": 1.2, "issue_slots_busy": 58.2,
             "warp_instructions_per_env_substep": 176.0}
BYTES_PER_ENV_STEP = 150       # SURVEY §8(d): algorithmic HBM bytes per env-step
FP32_LANES_PER_SM, N_SM = 128, 148
DUMP_ROWS = 1 << 18            # --dump-outputs: envs kept from a larger batch (fixed sample), ~42 MB of .npy files


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f), "measured"
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:  # noqa: BLE001
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:  # noqa: BLE001
            self.proc.kill()
        try:
            rows = [r.split(",") for r in open(self.path).read().strip().splitlines() if r.strip()]
            sm = [float(r[1]) for r in rows]
            out["samples"] = len(sm)
            if sm:
                out["sm_mhz"] = float(np.median(sm))
                out["sm_max_mhz"] = float(rows[0][2])
                out["power_w_max"] = max(float(r[3]) for r in rows)
                names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                for k, nm in enumerate(names):
                    if any(r[5 + k].strip().lower().startswith("active") for r in rows):
                        out["reasons"].append(nm)
        except Exception:  # noqa: BLE001
            pass
        finally:
            try:
                os.unlink(self.path)
            except OSError:
                pass
        return out


def make_actions(n, seed):
    """Synthetic random pulse sequences: J ~ U(-Jm, Jm) in the well-conditioned regime (SURVEY §8d), fixed 1 ns duration."""
    rng = np.random.default_rng(seed)
    a = np.empty((n, 2), np.float32)
    a[:, 0] = rng.uniform(-1.1e-6, 1.1e-6, n)
    a[:, 1] = PULSE_S
    return a


def dump_outputs(path, step_out, n):
    """Write what env.step returned (obs, reward, terminated, truncated and the info tensors, rows = envs) as path/<name>.npy:
    obs-shaped arrays in float32, the rest in float64, for a fixed sample of DUMP_ROWS envs (env_index.npy) when n is larger."""
    import torch
    obs, reward, terminated, truncated, info = step_out
    idx = np.arange(n) if n <= DUMP_ROWS else np.sort(np.random.default_rng(0).choice(n, DUMP_ROWS, replace=False))
    rows = torch.from_numpy(idx).to(obs.device)
    os.makedirs(path, exist_ok=True)
    arrays = dict(env_index=idx, obs=obs, reward=reward, terminated=terminated, truncated=truncated, **info)
    for name, a in arrays.items():
        if torch.is_tensor(a):
            a = a.index_select(0, rows).cpu().numpy()
        np.save(os.path.join(path, name + ".npy"), a.astype(np.float32 if a.dtype == np.float32 else np.float64))


ENV_KW = dict(device_type="stt_mram", max_current=1.1e-6, temperature=300.0, include_thermal_fluctuations=True,
              integrator="rk4", autoreset=True, sort_by_substeps=False)   # fixed pulse duration: nothing to sort


# ----------------------------------------------------------------------------------------------------------------------
def cpu_port_rate(n_sample: int, steps: int, threads: int, thermal: bool = True):
    """LLGS substeps/s of the C restatement (oracle/c) on `threads` host threads over `steps` steps of n_sample envs."""
    from oracle.c_oracle import COracleEnv
    env = COracleEnv(n_sample, max_current=1.1e-6, include_thermal=thermal, temperature=300.0, nthreads=threads)
    rng = np.random.default_rng(0)
    env.reset(rng.normal(size=(n_sample, 3)), np.array([0.0, 0.0, 1.0]))
    act = make_actions(n_sample, 1)
    sub = 0
    t0 = time.perf_counter()
    for _ in range(steps):
        env.step(act)
        sub += int(env.substeps)
    dt = time.perf_counter() - t0
    return sub / dt, n_sample * steps / dt, dt


def python_port_rate(max_seconds: float = 4.0):
    """Substeps/s of the NumPy restatement (what the reference's interpreter-bound loop costs), one core."""
    from oracle.stt_oracle import SttOracleEnv
    env = SttOracleEnv(max_current=1.1e-6, include_thermal=False)
    env.reset(np.array([0.3, 0.2, 0.9]), np.array([0.0, 0.0, 1.0]))
    t0 = time.perf_counter()
    sub = 0
    while time.perf_counter() - t0 < max_seconds:
        _, _, _, _, info = env.step(np.array([5e-7, 5e-10], np.float32))
        sub += info["n_sub"]
    return sub / (time.perf_counter() - t0)


def live_reference_rate(seconds: float, thermal: bool = True):
    """The live reference's own SpinTorqueEnv.step, one process per host core (tools/time_live_reference.py in a subprocess:
    the workers are spawned processes and must not inherit a CUDA context). Returns the tool's dict; ['available'] False with a
    reason when no checkout is reachable on this box."""
    cmd = [sys.executable, os.path.join(ROOT, "tools", "time_live_reference.py"), "--json", "--seconds", str(seconds)]
    if not thermal:
        cmd.append("--no-thermal")
    try:
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=seconds * 4 + 240)
        return json.loads(out.stdout.strip().splitlines()[-1])
    except Exception as exc:  # noqa: BLE001
        return {"available": False, "why": f"time_live_reference.py failed: {exc!r}"}


def run_reference(args, rank):
    """`--impl reference`: the reference's CPU implementation of the path on all host cores. Rank 0 only."""
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    live = live_reference_rate(min(60.0, max(5.0, 1.0 * args.steps)))
    if live.get("available"):
        sub_rate, env_rate = live["substeps_per_s"], live["env_steps_per_s"]
        n_sample, kind = live["procs"], "reference"
        ms_per_step = 1e3 * live["procs"] / env_rate                 # one env.step of each process's env
        sample = (f"live reference at {live['path']}: {live['procs']} processes (one SpinTorqueEnv each, sanitised) x "
                  f"{live['seconds_per_proc']:.0f} s = {live['env_steps']} env.step x 999 RK4 substeps, thermal on")
        cores = live["procs"]
        extra = {"vectorized_solver": live.get("vectorized_solver")}
    else:
        n_sample = 2048 * threads          # bounded sample: ~0.5 s of CPU work per step on all host threads
        for _ in range(args.warmup):
            cpu_port_rate(max(threads, n_sample // 8), 1, threads)
        sub_rate, env_rate, dt = cpu_port_rate(n_sample, args.steps, threads)
        ms_per_step, kind, cores = 1e3 * dt / args.steps, "port", threads
        sample = (f"{n_sample} envs x {args.steps} steps x 999 RK4 substeps, thermal on, C restatement oracle/c on {threads} "
                  f"threads (live reference not reachable: {live.get('why')})")
        extra = {}
    line = {
        "impl": "reference", "metric": "llgs_substeps_per_sec", "value": sub_rate, "unit": "LLGS substeps/s",
        "env_steps_per_s": env_rate, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.gpus, n_sample, "bounded sample of the same workload"),
        "cpu_baseline": dict({"value": sub_rate, "unit": "LLGS substeps/s", "cores": cores, "kind": kind, "sample": sample},
                             **extra),
        "e2e": {"value": sub_rate, "unit": "LLGS substeps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def workload_config(n_gpus, n_envs_per_gpu, note=""):
    return {
        "workload": "SpinTorque-v0 stt_mram (reference default device), T=300K thermal (in-kernel stream: Philox-seeded xoshiro128++), RK4 fixed dt, "
                    "1 ns pulses = 999 substeps/step, random J in the well-conditioned regime (BASELINE configs[1] physics "
                    "at the metric's 1M envs per GPU)" + (f"; {note}" if note else ""),
        "envs_per_gpu": n_envs_per_gpu, "total_envs": n_envs_per_gpu * n_gpus, "substeps_per_env_step": 999,
        "parallelism": f"env-sharded x{n_gpus}, no data-path collective; stats all-reduce once per rollout",
        "l2": "state+io per step (~200 MB at 1M envs) exceeds the 126 MB L2; kernel is FP32-pipe bound",
    }


# ----------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs-per-gpu", type=int, default=N_ENVS_PER_GPU)
    ap.add_argument("--total-envs", type=int, default=0,
                    help="strong scaling (SURVEY 8e): fixed total env count split evenly over the ranks; the line says "
                         "'scaling': 'strong'. Default 0 = weak scaling with --envs-per-gpu on every rank")
    ap.add_argument("--dtype", default="f32", choices=["f32", "f64"])
    ap.add_argument("--no-thermal", action="store_true", help="secondary workload: thermal off (301 flop/substep)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the secondary measurements (thermal-off, f64, probe)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (rank 0's envs) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    from spin_torque_rl_gym_b200 import SpinTorqueVectorEnv, _lib
    from spin_torque_rl_gym_b200.parallel import all_reduce_stats

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    n_gpus = world
    n_local = args.envs_per_gpu
    if args.total_envs:
        if args.total_envs % n_gpus:
            raise SystemExit(f"--total-envs {args.total_envs} does not divide over {n_gpus} ranks")
        n_local = args.total_envs // n_gpus
    scaling = "strong" if args.total_envs else "weak"
    tdtype = torch.float32 if args.dtype == "f32" else torch.float64
    thermal = not args.no_thermal
    kw = dict(ENV_KW, include_thermal_fluctuations=thermal)
    flop_sub = FLOP_RK4_THERMAL if thermal else FLOP_RK4

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    action_gen = torch.Generator(device=dev)
    action_gen.manual_seed(4321 + rank)

    def fresh_actions(act):
        """Random pulse sequences: a fresh current density per env and step, drawn on the device from a seeded generator, so
        that the same arguments give the same inputs (the duration stays the metric's 1 ns = 999 substeps). One torch fill
        kernel per step inside the timed region; not counted in gpu_launches."""
        act[:, 0].uniform_(-1.1e-6, 1.1e-6, generator=action_gen)

    def timed_device_steps(env, act, steps, warmup):
        """Device time of `steps` env steps after `warmup` untimed ones: (ms, kernel launches, what the last step returned)."""
        for _ in range(warmup):
            fresh_actions(act)
            env.step(act)
        barrier()
        l0 = env.gpu_launches
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fresh_actions(act)
            out = env.step(act)
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t[0])
        return ms, env.gpu_launches - l0, out

    # ---- headline: device-resident ------------------------------------------------------------------------------------
    env = SpinTorqueVectorEnv(num_envs=n_local, device=dev, dtype=tdtype, rng_seed=1234, env_offset=rank * n_local, **kw)
    env.reset(seed=1234)
    act_host = make_actions(n_local, 100 + rank)
    act = torch.from_numpy(act_host).to(dev)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms, launches, last_step = timed_device_steps(env, act, args.steps, args.warmup)
    stats = all_reduce_stats(env.stats_tensor())          # one collective per rollout (K5): episode statistics
    clocks = sampler.stop() if rank == 0 else {}
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last_step, n_local)
    sub_per_step = n_local * 999 * n_gpus
    value = sub_per_step * args.steps / (ms * 1e-3)
    env_steps = n_local * n_gpus * args.steps / (ms * 1e-3)
    kernel_ms = ms / args.steps                             # one K1 launch per step per GPU

    # ---- e2e: public API, host actions in, host results out ------------------------------------------------------------
    # host_outputs=True: obs / reward / terminated / truncated live in pinned host memory and the step kernel writes them there
    # directly while it runs (posted PCIe writes), so no device-to-host copy is serialised after the launch; the actions go
    # host -> device from pinned memory inside step(); step() returns once the stream has drained, i.e. the results are readable.
    env_h = SpinTorqueVectorEnv(num_envs=n_local, device=dev, dtype=tdtype, rng_seed=1234, env_offset=rank * n_local,
                                host_outputs=True, **kw)
    env_h.reset(seed=1234)
    # a different host action array every step (four pinned buffers of random pulses used in turn)
    act_ring = [torch.from_numpy(make_actions(n_local, 200 + 10 * rank + k)).pin_memory() for k in range(4)]

    def e2e_step(k):
        o, r, te, tr, _ = env_h.step(act_ring[k & 3])        # H2D of the actions + kernel + results in host memory + sync
        return float(r[0]) + float(o[0, 0]) + float(te[0]) + float(tr[0])      # the caller reads the host buffers every step

    for k in range(args.warmup):
        e2e_step(k)
    barrier()
    ended0 = env_h.episode_stats()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(args.steps):
        e2e_step(k)
    e1.record()
    barrier()
    ended1 = env_h.episode_stats()
    # rows of final_obs cross PCIe only for the envs whose episode ended in the step (include/stg.h StgSttStepOut.final_obs)
    resets_per_step = ((ended1["terminated"] + ended1["truncated"]) - (ended0["terminated"] + ended0["truncated"])) / args.steps
    if world > 1:
        t = torch.tensor([resets_per_step], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        resets_per_step = float(t[0])
    e2e_ms = max(e0.elapsed_time(e1), 0.0)
    if world > 1:
        t = torch.tensor([e2e_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_ms = float(t[0])
    e2e_value = sub_per_step * args.steps / (e2e_ms * 1e-3)

    # ---- secondary measurements (rank 0, N=1 only) ---------------------------------------------------------------------
    extras = {}
    peaks, peaks_src = _peaks()
    sm_max_mhz = float(peaks.get("sm_max_mhz", 1965.0))
    fp32_peak_theory = N_SM * FP32_LANES_PER_SM * 2 * sm_max_mhz * 1e6 / 1e12
    fma_probe_tflops = None
    if rank == 0 and not args.no_extras:
        lib = _lib.load()
        buf = torch.empty(N_SM * 16 * 256, dtype=torch.float32, device=dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        best = 0.0
        for it in range(6):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            _lib.check(lib.stg_probe_fma(buf.data_ptr(), N_SM * 16, 4096, 0, stream))
            e1.record()
            torch.cuda.synchronize(dev)
            if it:
                best = max(best, N_SM * 16 * 256 * 4096 * 64 * 2 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
        fma_probe_tflops = best
        for mode, key in ((2, "ffma2_probe_tflops"), (1, "dfma_probe_tflops")):
            best2 = 0.0
            per_iter = 128 if mode == 2 else 64
            buf64 = torch.empty(N_SM * 16 * 256, dtype=torch.float64, device=dev)
            for it in range(4):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                _lib.check(lib.stg_probe_fma(buf64.data_ptr(), N_SM * 16, 4096, mode, stream))
                e1.record()
                torch.cuda.synchronize(dev)
                if it:
                    best2 = max(best2, N_SM * 16 * 256 * 4096 * per_iter * 2 / (e0.elapsed_time(e1) * 1e-3) / 1e12)
            extras[key] = best2
        if world == 1:
            def variant(name, n, **over):
                e = SpinTorqueVectorEnv(num_envs=n, device=dev, rng_seed=1234,
                                        **dict(kw, **{k: v for k, v in over.items() if k != "dtype"}),
                                        dtype=over.get("dtype", tdtype))
                e.reset(seed=1234)
                a = torch.from_numpy(make_actions(n, 7)).to(dev)
                m, _, _ = timed_device_steps(e, a, max(3, args.steps // 2), 3)
                extras[name] = n * 999 * max(3, args.steps // 2) / (m * 1e-3)
                del e
            variant("substeps_per_s_thermal_off", n_local, include_thermal_fluctuations=False)
            variant("substeps_per_s_65536_envs", 65536)
            # same workload with every word of the thermal stream from Philox4x32-10 (thermal_stream='philox': counter-based down
            # to the substep; the headline uses the default stream, xoshiro128++ seeded per env-step from that Philox stream)
            variant("substeps_per_s_all_philox_stream", n_local, thermal_stream="philox")
            variant("substeps_per_s_f64_thermal", n_local // 4, dtype=torch.float64)
            variant("substeps_per_s_f64_thermal_off", n_local // 4, dtype=torch.float64, include_thermal_fluctuations=False)
            try:       # BASELINE configs[2], configs[3] and the ragged-duration variant of configs[1] (tools/bench_extra.py)
                from tools.bench_extra import collect
                extras["other_configs"] = collect(dev)
            except Exception as exc:  # noqa: BLE001 - secondary numbers must never break the contract line
                extras["other_configs_error"] = repr(exc)

    # ---- multi-GPU extras (every rank takes part): strong scaling at the north star's total, a short configs[4] rollout -----
    if world > 1 and not args.no_extras and not args.total_envs:
        total = N_ENVS_PER_GPU                                   # 1,048,576 envs over all ranks (131,072 per GPU at N = 8)
        if total % world == 0:
            n_s = total // world
            env_s = SpinTorqueVectorEnv(num_envs=n_s, device=dev, dtype=tdtype, rng_seed=1234, env_offset=rank * n_s, **kw)
            env_s.reset(seed=1234)
            act_s = torch.from_numpy(make_actions(n_s, 300 + rank)).to(dev)
            ms_s, _, _ = timed_device_steps(env_s, act_s, args.steps, args.warmup)
            if rank == 0:
                extras["strong_scaling_total_1048576"] = {
                    "envs_per_gpu": n_s, "ms_per_step": ms_s / args.steps,
                    "substeps_per_s": total * 999 * args.steps / (ms_s * 1e-3),
                    "env_steps_per_s": total * args.steps / (ms_s * 1e-3)}
            del env_s
        # BASELINE configs[4]: 1M+ envs sharded over the ranks feeding an SB3-shaped rollout buffer; policy = fixed random MLP,
        # pulse durations from the policy (ragged substep counts, counting sort active), statistics all-reduced once at the end.
        # n_steps is cut to 128 of the 2048 so that the bench stays short; tools/rollout_bench.py runs the full length.
        from spin_torque_rl_gym_b200 import RolloutCollector
        n_r, n_steps_r = N_ENVS_PER_GPU // world if N_ENVS_PER_GPU % world == 0 else 131072, 128
        env_r = SpinTorqueVectorEnv(num_envs=n_r, device=dev, dtype=tdtype, rng_seed=7, env_offset=rank * n_r,
                                    **dict(kw, sort_by_substeps="auto"))
        gen = torch.Generator(device=dev).manual_seed(0)
        w1 = torch.randn(12, 64, device=dev, generator=gen) * 0.3
        w2 = torch.randn(64, 2, device=dev, generator=gen) * 0.3

        def policy(obs):
            h = torch.tanh(obs @ w1) @ w2
            a2 = torch.empty(obs.shape[0], 2, device=dev)
            a2[:, 0] = torch.tanh(h[:, 0]) * 1.1e-6
            a2[:, 1] = torch.sigmoid(h[:, 1]) * 1e-9 + 1e-11
            return a2

        RolloutCollector(env_r, n_steps=2, store_observations=False).collect(policy)       # warm-up
        col = RolloutCollector(env_r, n_steps=n_steps_r)
        env_r.reset(seed=7)
        env_r.reset_stats()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        st_r = col.collect(policy)                              # includes the one NCCL all-reduce of the statistics vector
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        if rank == 0:
            ms_r = float(t[0])
            extras["rollout_configs4"] = {
                "envs_total": n_r * world, "envs_per_gpu": n_r, "n_steps": n_steps_r, "rollout_ms": ms_r,
                "env_steps_per_s": n_r * world * n_steps_r / (ms_r * 1e-3), "substeps_per_s": st_r["substeps"] / (ms_r * 1e-3),
                "episodes": st_r["episodes"], "success_rate": st_r["success_rate"],
                "note": "policy-chosen pulse durations (ragged substeps, sorted launch), obs/actions/rewards/dones stored per step, "
                        "stats all-reduced via NCCL once at the end; 128 of the 2048 steps of BASELINE configs[4]"}
        del env_r, col

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        threads = os.cpu_count() or 1
        n_sample = 8192 * threads
        cpu_port_rate(max(threads, n_sample // 64), 1, threads, thermal)
        cpu_steps = 8                                  # 131072 envs x 8 steps on 16 threads: ~13 s
        rate, _, dt = cpu_port_rate(n_sample, cpu_steps, threads, thermal)
        port = {"value": rate, "unit": "LLGS substeps/s", "cores": threads,
                "sample": f"{n_sample} envs x {cpu_steps} steps x 999 RK4 substeps (thermal {'on' if thermal else 'off'}), "
                          f"C restatement oracle/c on {threads} threads, {dt:.1f} s",
                "python_port_substeps_per_s_1core": python_port_rate(3.0)}
        live = live_reference_rate(10.0, thermal)
        if live.get("available"):
            cpu_baseline = {"value": live["substeps_per_s"], "unit": "LLGS substeps/s", "cores": live["procs"], "kind": "reference",
                            "sample": f"live reference at {live['path']}: sanitised SpinTorqueEnv.step, {live['procs']} processes x "
                                      f"{live['seconds_per_proc']:.0f} s = {live['env_steps']} env.step x 999 RK4 substeps",
                            "env_steps_per_s": live["env_steps_per_s"], "vectorized_solver": live.get("vectorized_solver"),
                            "port": port}
        else:
            cpu_baseline = dict(port, kind="port", reference_unavailable=live.get("why"))

    if rank == 0:
        achieved = value / n_gpus * flop_sub / 1e12            # per-GPU algorithmic TFLOP/s of the dominant kernel
        headline = n_local == N_ENVS_PER_GPU and thermal and args.dtype == "f32"
        executed = value / n_gpus * FLOP_RK4_THERMAL_EXECUTED / 1e12 if thermal and args.dtype == "f32" else None
        line = {
            "metric": "llgs_substeps_per_sec", "value": value, "unit": "LLGS substeps/s",
            "env_steps_per_s": env_steps, "n_gpus": n_gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": scaling, "vs_baseline": None,
            "dtype": args.dtype + " stages, " + ("compensated f32 state inside a step, " if thermal and args.dtype == "f32" else "")
                     + "f64 state between steps", "data": "synthetic",
            "config": workload_config(n_gpus, n_local),
            "e2e": {"value": e2e_value, "unit": "LLGS substeps/s", "ms_per_step": e2e_ms / args.steps,
                    "h2d_bytes_per_step": n_local * 8 * n_gpus,
                    "d2h_bytes_per_step": int(n_local * (48 + 8 + 2) * n_gpus + 48 * resets_per_step),
                    "final_obs_rows_per_step": resets_per_step,
                    "api": "SpinTorqueVectorEnv(host_outputs=True).step(pinned host actions, a different array every step): H2D of "
                           "the actions, the kernel writes obs / reward / terminated / truncated (58 B per env) and the final_obs rows "
                           "of ended episodes (48 B each) into pinned host memory, stream synchronised every step"},
            "gpu_launches": launches,
            "roofline": {
                # the path is FP32-pipe bound (no contraction, 2,000 flop/B): the contract's "hbm" | "tensor" do not apply; the HBM
                # figure is reported beside it
                "bound": "fp32_fma",
                "kernel": "stt_env_step_pair_kernel<1> (two envs per thread on FFMA2, axis z, in-kernel thermal stream, RK4)" if thermal and args.dtype == "f32"
                          else "stt_env_step_kernel",
                "achieved": achieved, "peak": fp32_peak_theory, "unit": "TFLOP/s", "frac": achieved / fp32_peak_theory,
                "peak_source": "theoretical 148 SM x 128 FP32 lanes x 2 x sm_max_mhz (MEASURED_PEAKS.json carries no FP32 figure)",
                "peak_fma_probe": fma_probe_tflops,
                "frac_of_fma_probe": achieved / fma_probe_tflops if fma_probe_tflops else None,
                "algorithmic_flop_per_substep": flop_sub, "executed_flop_per_substep": FLOP_RK4_THERMAL_EXECUTED if executed else None,
                "executed_tflops": executed, "executed_frac": executed / fp32_peak_theory if executed else None,
                "substeps_per_launch": n_local * 999, "kernel_ms": kernel_ms,
                # the thermal stream of the headline: xoshiro128++ seeded per env-step from the env-step's Philox4x32-10 stream;
                # the same workload with every word from Philox4x32-10 (thermal_stream='philox', measured in extras at N = 1)
                "thermal_stream": "xoshiro128++ seeded per env-step from Philox4x32-10 (default)" if thermal else None,
                "frac_with_all_philox_stream": (extras["substeps_per_s_all_philox_stream"] * flop_sub / 1e12 / fp32_peak_theory
                                                if "substeps_per_s_all_philox_stream" in extras else None),
                # pipe utilisation and DRAM traffic of one launch at this size from the ncu --set full capture of the shipped kernel
                # (profiles/r02_ncu_stt_env_step_pair_f32_thermal1_xoshiro.csv)
                "pipes_pct_from_ncu": NCU_PIPES if headline else None,
                "traffic": NCU_TRAFFIC_BYTES if headline else None,
                "hbm": {"achieved_gbs": n_local * BYTES_PER_ENV_STEP / (kernel_ms * 1e-3) / 1e9,
                        "peak_gbs": peaks.get("hbm_gbs"), "peak_source": peaks_src},
            },
            "cpu_baseline": cpu_baseline,
            "clocks": clocks,
            "episode_stats": stats,
            "extras": extras,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
