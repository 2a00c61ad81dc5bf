#!/usr/bin/env python
"""K6 (stg_rollout_gae_f32): CUDA-event time of the GAE kernel over a stored [T, N] rollout, its algorithmic HBM bandwidth,
and, in the same run, an eager torch loop over time computing the same float32 recurrence (with a bit-for-bit comparison).

    python tools/gae_bench.py [--steps 2048] [--envs 4096 131072 1048576] [--reps 30] [--out FILE]

Inputs are generated on the device from a seed. The flags follow a max_steps=100 rollout: every env starts at a random point of
its episode, terminates with probability 0.2 % per step and is truncated when its episode reaches 100 steps, so about 1 % of the
(step, env) entries are bootstrapped with a final value; the other final values are NaN (stale rows, never read).
Algorithmic bytes: 18 per (step, env) (reward, value, return, advantage f32; two u8 flags) plus 4 per bootstrapped entry.
N = 4,096 moves 151 MB per launch, about the 126 MB of L2, so part of it may be served from there between launches.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from spin_torque_rl_gym_b200 import _lib  # noqa: E402

HBM_PEAK_GBS = 6554.9          # the B200's measured HBM bandwidth the project quotes (SURVEY §8d, MEASURED_PEAKS.json)
MAX_STEPS, P_TERM = 100, 0.002


def make_inputs(T, N, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    reward = torch.randn(T, N, generator=g, device=dev)
    value = torch.randn(T, N, generator=g, device=dev)
    final_value = torch.randn(T, N, generator=g, device=dev)
    last_value = torch.randn(N, generator=g, device=dev)
    term = torch.empty(T, N, dtype=torch.bool, device=dev)
    trunc = torch.empty(T, N, dtype=torch.bool, device=dev)
    count = torch.randint(0, MAX_STEPS, (N,), generator=g, device=dev)
    for t in range(T):
        count += 1
        torch.lt(torch.rand(N, generator=g, device=dev), P_TERM, out=term[t])
        torch.ge(count, MAX_STEPS, out=trunc[t])
        count.masked_fill_(term[t] | trunc[t], 0)
    boot = trunc & ~term
    final_value.masked_fill_(~boot, float("nan"))
    return reward, value, term.view(torch.uint8), trunc.view(torch.uint8), final_value, last_value, int(boot.sum())


def gae_kernel(planes, adv, ret, gamma, gae_lambda):
    reward, value, term, trunc, final_value, last_value = planes
    a = _lib.StgGaeArgs()
    a.d_reward, a.d_value = reward.data_ptr(), value.data_ptr()
    a.d_terminated, a.d_truncated = term.data_ptr(), trunc.data_ptr()
    a.d_final_value, a.d_last_value = final_value.data_ptr(), last_value.data_ptr()
    a.d_advantage, a.d_return = adv.data_ptr(), ret.data_ptr()
    a.gamma, a.gamma_lambda = float(np.float32(gamma)), float(np.float32(gamma * gae_lambda))
    a.n_steps, a.n_envs = reward.shape
    _lib.check(_lib.load().stg_rollout_gae_f32(C.byref(a), torch.cuda.current_stream().cuda_stream), "stg_rollout_gae_f32")


def gae_torch(planes, adv, ret, gamma, gae_lambda):
    """The same recurrence as eager torch float32 ops, one op per rounding (no fused multiply-add anywhere)."""
    reward, value, term, trunc, final_value, last_value = planes
    g, gl = float(np.float32(gamma)), float(np.float32(gamma * gae_lambda))
    last = torch.zeros_like(last_value)
    v_next = last_value
    for t in reversed(range(reward.shape[0])):
        te, tr = term[t].bool(), trunc[t].bool()
        r = torch.where(tr & ~te, reward[t] + g * final_value[t], reward[t])
        nnt = 1.0 - (te | tr).float()
        delta = (r + (g * v_next) * nnt) - value[t]
        last = delta + (gl * nnt) * last
        adv[t] = last
        v_next = value[t]
    torch.add(adv, value, out=ret)


def events_ms(fn, reps):
    times = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    return times


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=2048)
    ap.add_argument("--envs", type=int, nargs="+", default=[4096, 131072, 1048576])
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--torch-reps", type=int, default=2)
    ap.add_argument("--gamma", type=float, default=0.99)
    ap.add_argument("--gae-lambda", type=float, default=0.95)
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("gae_bench.py measures the CUDA kernel: no CUDA device")
    if a.reps < 20:
        raise SystemExit("--reps must be at least 20")
    dev = torch.device("cuda", 0)
    smi = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True).stdout.strip()
    res = {"gpu": torch.cuda.get_device_name(dev), "nvidia_smi": smi, "hbm_peak_gbs": HBM_PEAK_GBS, "n_steps": a.steps,
           "gamma": a.gamma, "gae_lambda": a.gae_lambda, "reps": a.reps, "sizes": []}
    for N in a.envs:
        *planes, n_boot = make_inputs(a.steps, N, dev, seed=N)
        adv, ret = torch.empty_like(planes[0]), torch.empty_like(planes[0])
        run = lambda: gae_kernel(planes, adv, ret, a.gamma, a.gae_lambda)        # noqa: E731
        events_ms(run, a.warmup)
        k = events_ms(run, a.reps)
        adv_t, ret_t = torch.empty_like(adv), torch.empty_like(ret)
        tl = events_ms(lambda: gae_torch(planes, adv_t, ret_t, a.gamma, a.gae_lambda), 1 + a.torch_reps)[1:]
        elems = a.steps * N
        nbytes = 18 * elems + 4 * n_boot
        med = float(np.median(k))
        row = {"n_envs": N, "elements": elems, "bootstrapped": n_boot, "algorithmic_bytes": nbytes,
               "kernel_ms_median": med, "kernel_ms_min": float(np.min(k)), "kernel_ms_max": float(np.max(k)),
               "hbm_gbs_algorithmic": nbytes / (med * 1e-3) / 1e9,
               "frac_of_hbm_peak": nbytes / (med * 1e-3) / 1e9 / HBM_PEAK_GBS,
               "torch_loop_ms": float(np.median(tl)), "speedup_vs_torch_loop": float(np.median(tl)) / med,
               "bit_equal_advantage": bool(torch.equal(adv, adv_t)), "bit_equal_return": bool(torch.equal(ret, ret_t)),
               "finite": bool(torch.isfinite(adv).all())}
        res["sizes"].append(row)
        print(json.dumps(row), file=sys.stderr, flush=True)
        del planes, adv, ret, adv_t, ret_t
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
