#!/usr/bin/env python
"""K8 (VecNormalize): CUDA-event time of the launches a wrapped step adds after K1, their algorithmic HBM bandwidth, and, in
the same run, an eager torch float64 implementation of the same update with its outputs compared to tolerance.

    python tools/vecnorm_bench.py [--envs 4096 131072 1048576] [--steps 30] [--warmup 5] [--out FILE]

Every timed window follows a real K1 step (`SpinTorqueVectorEnv.step`, the bench's env configuration with max_steps=20 so that
episodes end), so L2 holds what K1 just wrote, as in training. Algorithmic bytes per step: 72 per env for the moments launch
(48 B observation, reward, return read and written), 114 per env for the apply launch (observation read and written, reward
read and written, two flag bytes) and 104 per ended env (final row read and written, return zeroed). At 1,048,576 envs the 50 MB
observation plane K1 wrote fits in the 126 MB L2, so part of the traffic may never reach HBM; the fraction of peak is stated
against HBM all the same. K1 is enqueued without a host synchronisation and runs for hundreds of microseconds, so the host has
enqueued the K8 launches before the device reaches them: every window is device time.

Where the time goes, per size, in further steps of the same env:
  - events between the launches (moments | merge | apply), so each window is one kernel plus the gap before it;
  - the apply launch once with the normalisation flags cleared (the same loads and stores, the values copied): the difference
    to the normalising apply is the cost of the FP64 arithmetic (the IEEE divisions and square roots);
  - a separate torch.profiler pass (not timed otherwise) for the kernel durations alone; window minus kernel is the launch gap. With two or more GPUs visible, a `torchrun --nproc-per-node=2` run of `--nccl-worker` checks that
sync=True leaves bit-identical statistics on both ranks."""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ctypes as C  # noqa: E402

import spin_torque_rl_gym_b200 as stg  # noqa: E402
from spin_torque_rl_gym_b200 import _lib  # noqa: E402

HBM_PEAK_GBS = 6554.9          # the B200's measured HBM bandwidth the project quotes (SURVEY §8d, MEASURED_PEAKS.json)
ENV_KW = dict(max_current=1.1e-6, temperature=300.0, include_thermal_fluctuations=True, max_steps=20)


def actions(n, dev, g):
    act = torch.empty(n, 2, device=dev)
    act[:, 0] = (torch.rand(n, generator=g, device=dev) * 2 - 1) * 1.1e-6
    act[:, 1] = torch.rand(n, generator=g, device=dev) * 1e-9 + 1e-11
    return act


class TorchVecNormalize:
    """SB3's VecNormalize step in eager torch float64 ops on the device (the obvious GPU port)."""

    def __init__(self, n, dev, gamma=0.99, eps=1e-8, clip=10.0):
        f64 = torch.float64
        self.om, self.ov, self.oc = torch.zeros(12, dtype=f64, device=dev), torch.ones(12, dtype=f64, device=dev), 1e-4
        self.rm, self.rv, self.rc = torch.zeros((), dtype=f64, device=dev), torch.ones((), dtype=f64, device=dev), 1e-4
        self.returns = torch.zeros(n, dtype=f64, device=dev)
        self.gamma, self.eps, self.clip = gamma, eps, clip

    @staticmethod
    def _update(mean, var, count, x):
        bm, bv, bc = x.mean(0), x.var(0, unbiased=False), x.shape[0]
        delta = bm - mean
        tot = count + bc
        new_mean = mean + delta * bc / tot
        m2 = var * count + bv * bc + delta * delta * count * bc / tot
        return new_mean, m2 / tot, bc + count

    def reset(self, obs):
        self.returns.zero_()
        self.om, self.ov, self.oc = self._update(self.om, self.ov, self.oc, obs.double())

    def step(self, obs, rew, term, trunc, final):
        x = obs.double()
        self.om, self.ov, self.oc = self._update(self.om, self.ov, self.oc, x)
        scale = torch.sqrt(self.ov + self.eps)
        o = ((x - self.om) / scale).clamp(-self.clip, self.clip).float()
        ended = term | trunc
        f = torch.where(ended[:, None], ((final.double() - self.om) / scale).clamp(-self.clip, self.clip).float(), final)
        self.returns = self.returns * self.gamma + rew
        self.rm, self.rv, self.rc = self._update(self.rm, self.rv, self.rc, self.returns)
        r = (rew / torch.sqrt(self.rv + self.eps)).clamp(-self.clip, self.clip)
        self.returns.masked_fill_(ended, 0.0)
        return o, r, f


def median(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2]


def k8_split(norm, out, ev, apply_flags=None):
    """The launches of VecNormalize._normalize_step for a training step without sync, one by one, with an event after each:
    ev[0] | moments | ev[1] | merge | ev[2] | apply | ev[3]. `apply_flags` overrides the apply launch's flags (0: copy)."""
    obs, rew, term, trunc, info = out
    lib, stream, flags = norm._lib, norm._stream(), norm._flags()
    a = norm._args(norm.num_envs, flags)
    a.d_obs, a.d_reward, a.d_returns = obs.data_ptr(), rew.data_ptr(), norm._returns.data_ptr()
    ev[0].record()
    _lib.check(lib.stg_vecnorm_moments_f32(C.byref(a), stream), "stg_vecnorm_moments_f32")
    ev[1].record()
    _lib.check(lib.stg_vecnorm_merge_f64(C.byref(a), stream), "stg_vecnorm_merge_f64")
    ev[2].record()
    a = norm._args(norm.num_envs, flags if apply_flags is None else apply_flags)
    a.d_obs, a.d_obs_out = obs.data_ptr(), norm._obs.data_ptr()
    a.d_terminated, a.d_truncated = term.data_ptr(), trunc.data_ptr()
    a.d_reward, a.d_reward_out, a.d_returns = rew.data_ptr(), norm._reward.data_ptr(), norm._returns.data_ptr()
    a.d_final_obs, a.d_final_obs_out = info["final_observation"].data_ptr(), norm._final_obs.data_ptr()
    _lib.check(lib.stg_vecnorm_apply_f32(C.byref(a), stream), "stg_vecnorm_apply_f32")
    ev[3].record()


def breakdown(venv, norm, steps, dev, g):
    """Per-launch event windows, the copy-only apply, and kernel durations from a torch.profiler pass (see the docstring)."""
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    win = {"moments": [], "merge": [], "apply": [], "apply_copy_only": []}
    for s in range(2 * steps):
        out = venv.step(actions(venv.num_envs, dev, g))
        copy = s % 2 == 1                     # alternate the normalising and the copy-only apply
        k8_split(norm, out, ev, apply_flags=0 if copy else None)
        torch.cuda.synchronize()
        if not copy:
            win["moments"].append(ev[0].elapsed_time(ev[1]) * 1e3)
            win["merge"].append(ev[1].elapsed_time(ev[2]) * 1e3)
        win["apply_copy_only" if copy else "apply"].append(ev[2].elapsed_time(ev[3]) * 1e3)
    res = {"event_window_us_median": {k: round(median(v), 2) for k, v in win.items()}}
    try:
        from torch.profiler import ProfilerActivity, profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(5):
                out = venv.step(actions(venv.num_envs, dev, g))
                norm._normalize_step(*out)
            torch.cuda.synchronize()
        kern = {}
        for e in prof.key_averages():
            if "vecnorm" in e.key:
                total = getattr(e, "device_time_total", None)
                if total is None:
                    total = getattr(e, "cuda_time_total", 0.0)
                kern[e.key] = round(total / max(e.count, 1), 2)
        res["profiler_kernel_us_mean"] = kern
    except Exception as exc:  # noqa: BLE001
        res["profiler_kernel_us_mean"] = f"torch.profiler failed: {exc}"
    return res


def bench_size(n, steps, warmup, dev):
    venv = stg.make("SpinTorque-v0", num_envs=n, device=dev, rng_seed=1234, **ENV_KW)
    norm = stg.VecNormalize(venv)
    ref = TorchVecNormalize(n, dev)
    g = torch.Generator(device=dev).manual_seed(n)
    obs, _ = norm.reset(seed=1234)
    ref.reset(norm.get_original_obs())
    t_k1, t_k8, t_torch, ended = [], [], [], []
    err = {"obs": 0.0, "reward": 0.0, "final": 0.0, "obs_mean_rel": 0.0, "obs_var_rel": 0.0, "ret_var_rel": 0.0}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
    for s in range(warmup + steps):
        act = actions(n, dev, g)
        ev[0].record()
        out = venv.step(act)
        ev[1].record()
        o, r, te, tr, info = norm._normalize_step(*out)
        ev[2].record()
        ev[3].record()
        ro, rr, rf = ref.step(out[0], out[1], te, tr, venv._final_obs)
        ev[4].record()
        torch.cuda.synchronize()
        if s < warmup:
            continue
        t_k1.append(ev[0].elapsed_time(ev[1]) * 1e3)
        t_k8.append(ev[1].elapsed_time(ev[2]) * 1e3)
        t_torch.append(ev[3].elapsed_time(ev[4]) * 1e3)
        e = te | tr
        ended.append(int(e.sum()))
        err["obs"] = max(err["obs"], float((o - ro).abs().max()))
        err["reward"] = max(err["reward"], float((r - rr).abs().max()))
        if ended[-1]:
            err["final"] = max(err["final"], float((info["final_observation"][e] - rf[e]).abs().max()))
        rel = lambda a, b: float(((a - b).abs() / b.abs().clamp_min(1e-300)).max())      # noqa: E731
        err["obs_mean_rel"] = max(err["obs_mean_rel"], rel(norm.obs_rms.mean, ref.om))
        err["obs_var_rel"] = max(err["obs_var_rel"], rel(norm.obs_rms.var, ref.ov))
        err["ret_var_rel"] = max(err["ret_var_rel"], rel(norm.ret_rms.var, ref.rv))
    k8 = median(t_k8)
    mean_ended = sum(ended) / len(ended)
    split = breakdown(venv, norm, steps, dev, g)
    alg_bytes = n * (72 + 114) + mean_ended * 104
    return {
        "envs": n, "steps_timed": steps, "k1_step_us_median": round(median(t_k1), 2),
        "k8_us_median": round(k8, 2), "k8_us_min": round(min(t_k8), 2), "k8_us_max": round(max(t_k8), 2),
        "k8_share_of_k1_step": round(k8 / median(t_k1), 5),
        "torch_f64_us_median": round(median(t_torch), 2), "speedup_vs_torch": round(median(t_torch) / k8, 2),
        "ended_envs_per_step_mean": round(mean_ended, 1), "algorithmic_bytes_per_step": int(alg_bytes),
        "algorithmic_GBps": round(alg_bytes / (k8 * 1e-6) / 1e9, 1),
        "fraction_of_hbm_peak": round(alg_bytes / (k8 * 1e-6) / 1e9 / HBM_PEAK_GBS, 3),
        "max_abs_diff_vs_torch": {k: err[k] for k in ("obs", "reward", "final")},
        "max_rel_diff_stats_vs_torch": {k: err[k] for k in ("obs_mean_rel", "obs_var_rel", "ret_var_rel")},
        "torch_outputs_within_tolerance": err["obs"] <= 1e-5 and err["reward"] <= 1e-5 and err["final"] <= 1e-5
        and all(err[k] <= 1e-9 for k in ("obs_mean_rel", "obs_var_rel", "ret_var_rel")),
        "moments_bytes_per_step": 72 * n, "apply_bytes_per_step": int(114 * n + 104 * mean_ended),
        "breakdown": split,
    }


def nccl_worker():
    import torch.distributed as dist
    dist.init_process_group("nccl")
    rank, world = dist.get_rank(), dist.get_world_size()
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    n = 65536
    venv = stg.make("SpinTorque-v0", num_envs=n, device=dev, rng_seed=1234, env_offset=rank * n, **ENV_KW)
    norm = stg.VecNormalize(venv, sync=True)
    g = torch.Generator(device=dev).manual_seed(rank)
    norm.reset(seed=1234)
    for _ in range(8):
        norm.step(actions(n, dev, g))
    stats = [torch.empty_like(norm._stats) for _ in range(world)]
    dist.all_gather(stats, norm._stats.clone())
    if rank == 0:
        same = all(torch.equal(s.view(torch.int64), stats[0].view(torch.int64)) for s in stats)
        print("NCCL_RESULT " + json.dumps({"world_size": world, "steps": 8, "envs_per_rank": n,
                                           "statistics_bit_identical_on_all_ranks": same,
                                           "obs_count": float(stats[0][24])}), flush=True)
    dist.destroy_process_group()


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as exc:  # noqa: BLE001
        return f"unknown ({exc})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, nargs="+", default=[4096, 131072, 1048576])
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    ap.add_argument("--nccl-worker", action="store_true")
    args = ap.parse_args()
    if args.nccl_worker:
        return nccl_worker()
    if not torch.cuda.is_available():
        raise SystemExit("vecnorm_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    res = {"gpu": gpu_info(), "hbm_peak_GBps": HBM_PEAK_GBS, "env": ENV_KW,
           "timing": "CUDA events around the K8 launches (moments, merge, apply) after each real K1 step, device time (K1 is "
                     "still running when the host has enqueued K8); median over the timed steps after warm-up",
           "sizes": [bench_size(n, args.steps, args.warmup, dev) for n in args.envs]}
    if torch.cuda.device_count() >= 2:
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
               "127.0.0.1", "--master-port", "29561", os.path.abspath(__file__), "--nccl-worker"]
        p = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
        line = [l for l in p.stdout.splitlines() if l.startswith("NCCL_RESULT ")]
        res["nccl_sync"] = json.loads(line[0][12:]) if line else {"error": p.stderr[-2000:]}
    else:
        res["nccl_sync"] = f"unverified: {torch.cuda.device_count()} GPU visible, the NCCL path of sync=True was not run"
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
