#!/usr/bin/env python
"""K7 (stg_rollout_minibatch_f32): CUDA-event time of one whole epoch of RolloutCollector.get(batch_size), against the torch
version of the same sampler in the same run: torch.randperm over all T * N samples each epoch, then six index_select per
minibatch.

    python tools/minibatch_bench.py [--steps 2048] [--envs 131072 393216] [--batch 4096 65536 1048576] [--epochs 3] [--out FILE]

The rollout is collected on the device from a seed (SpinTorque-v0, seeded env and a fixed random linear actor-critic), then
GAE fills advantages and returns. Every timed epoch runs its batches back to back and drops each one after the yield, as a PPO
epoch does after the gradient step; the time is CUDA events around the epoch, the host loop included. N = 131,072 is the
per-GPU shard of the 8-GPU configuration; 393,216 makes T * N = 3 x 2^28 samples, which is not a power of 4, so the kernel's
permutation cycle-walks (4/3 network passes per sample on average, none at 2^28). The planes (20 GB and up) are far larger
than the 126 MB L2, so the random reads come from HBM.
Bytes per sample: algorithmic 72 read (48 observation, 8 action, 4 x 4 scalars) + 72 written; sector-granular 224 read
(2 + 1 + 4 sectors of 32 B) + 72 written.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import spin_torque_rl_gym_b200 as stg  # noqa: E402
from spin_torque_rl_gym_b200.envs.sb3_vec_env import RolloutBufferSamples  # noqa: E402

HBM_PEAK_GBS = 6554.9          # the B200's measured HBM bandwidth the project quotes (SURVEY §8d, MEASURED_PEAKS.json)
ALG_BYTES, SECTOR_BYTES = 72 + 72, 224 + 72


def make_collector(T, N, dev, seed):
    env = stg.make("SpinTorque-v0", num_envs=N, device=dev, max_steps=100, max_current=1.1e-6, rng_seed=seed)
    g = torch.Generator(device=dev).manual_seed(seed)
    w1 = torch.randn(12, 16, generator=g, device=dev) * 0.3
    wa = torch.randn(16, 2, generator=g, device=dev) * 0.3
    wv = torch.randn(16, 1, generator=g, device=dev) * 0.3

    def value_fn(o):
        return torch.tanh(o @ w1) @ wv

    def policy(o):
        out = torch.tanh(o @ w1) @ wa
        act = torch.stack([torch.tanh(out[:, 0]) * 1.1e-6, torch.sigmoid(out[:, 1]) * 1e-10 + 1e-11], 1)
        return act, value_fn(o), -(out * out).sum(1)

    col = stg.RolloutCollector(env, n_steps=T, store_values=True)
    col.collect(policy, value_fn)
    col.compute_returns_and_advantage()
    return col


def torch_epoch(col, batch_size):
    """The torch sampler: a fresh randperm, then one index_select per plane per minibatch."""
    M = col.n_steps * col.env.num_envs
    planes = (col.observations.view(M, 12), col.actions.view(M, 2), col.values.view(M), col.log_probs.view(M),
              col.advantages.view(M), col.returns.view(M))
    perm = torch.randperm(M, device=col.env.device)
    for s in range(0, M, batch_size):
        idx = perm[s:s + batch_size]
        yield RolloutBufferSamples(*[p.index_select(0, idx) for p in planes])


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


def drain(it):
    for _ in it:
        pass


def check_epoch(col, it):
    """Untimed: an epoch visits every sample once (the float64 sums of |advantage| and |observation| over the epoch equal
    those of the planes up to summation order, and the sample count is T * N)."""
    def abs_sum(x):                                      # step by step: no float64 copy of a whole plane
        return sum(x[t].abs().sum(dtype=torch.float64) for t in range(x.shape[0]))
    n = 0
    adv = torch.zeros((), dtype=torch.float64, device=col.env.device)
    obs = torch.zeros_like(adv)
    for b in it:
        n += len(b.advantages)
        adv += b.advantages.abs().sum(dtype=torch.float64)
        obs += b.observations.abs().sum(dtype=torch.float64)
    ok_adv = torch.isclose(adv, abs_sum(col.advantages), rtol=1e-9, atol=0)
    ok_obs = torch.isclose(obs, abs_sum(col.observations), rtol=1e-9, atol=0)
    return bool(n == col.advantages.numel() and ok_adv and ok_obs)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=2048)
    ap.add_argument("--envs", type=int, nargs="+", default=[131072, 393216])
    ap.add_argument("--batch", type=int, nargs="+", default=[4096, 65536, 1048576])
    ap.add_argument("--epochs", type=int, default=3, help="timed epochs per case, after one warm-up epoch")
    ap.add_argument("--out", default=None, help="also write the JSON result here")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("minibatch_bench.py measures the CUDA kernel: no CUDA device")
    dev = torch.device("cuda", 0)
    smi = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True).stdout.strip()
    res = {"gpu": torch.cuda.get_device_name(dev), "nvidia_smi": smi, "hbm_peak_gbs": HBM_PEAK_GBS, "n_steps": a.steps,
           "epochs": a.epochs, "bytes_per_sample_algorithmic": ALG_BYTES, "bytes_per_sample_sectors": SECTOR_BYTES,
           "cases": []}
    for N in a.envs:
        col = make_collector(a.steps, N, dev, seed=N)
        M = a.steps * N
        randperm = events_ms(lambda: torch.randperm(M, device=dev), 1 + a.epochs)[1:]
        for B in a.batch:
            kern = events_ms(lambda: drain(col.get(B)), 1 + a.epochs)[1:]
            base = events_ms(lambda: drain(torch_epoch(col, B)), 1 + a.epochs)[1:]
            k, t = float(np.median(kern)), float(np.median(base))
            row = {"n_envs": N, "samples": M, "batch_size": B, "batches": -(-M // B),
                   "kernel_epoch_ms": k, "kernel_epoch_ms_all": kern, "torch_epoch_ms": t, "torch_epoch_ms_all": base,
                   "torch_randperm_ms": float(np.median(randperm)), "speedup_vs_torch": t / k,
                   "kernel_gbs_algorithmic": ALG_BYTES * M / (k * 1e-3) / 1e9,
                   "kernel_gbs_sectors": SECTOR_BYTES * M / (k * 1e-3) / 1e9,
                   "kernel_frac_of_hbm_peak_algorithmic": ALG_BYTES * M / (k * 1e-3) / 1e9 / HBM_PEAK_GBS,
                   "kernel_us_per_batch": k * 1e3 / -(-M // B),
                   "kernel_epoch_visits_every_sample": check_epoch(col, col.get(B)),
                   "torch_epoch_visits_every_sample": check_epoch(col, torch_epoch(col, B))}
            res["cases"].append(row)
            print(json.dumps(row), file=sys.stderr, flush=True)
        del col
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
