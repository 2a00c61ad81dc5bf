#!/usr/bin/env python
"""K11 (ClippedAdam) and stg.PPO: the optimiser step, a PPO epoch and a full learn() iteration, against the torch optimiser
(`clip_grad_norm_(0.5)` + `Adam(fused=True)`) in the same run, and a 30-iteration learning curve.

    python tools/ppo_train_bench.py [--envs 65536] [--steps 16] [--batches 4096 65536 1048576] [--reps 20] [--out FILE]

The setup is tools/ppo_grad_bench.py's, so the figures compare with its epochs: a fresh ActorCriticPolicy collects `--steps` x
`--envs` samples from a VecNormalize'd SpinTorqueVectorEnv (max_steps=40) on the fused path, GAE, then the weights are
perturbed; losses with clip_range_vf=0.2, ent_coef=0.01. Reported:
  - optimiser step: one ClippedAdam.step() (one K11 launch) against clip_grad_norm_(0.5) + Adam(fused=True).step() on the same
    K10 gradient; CUDA events around each call, synchronised per repetition (so host launch time is inside), median of
    `--reps` after warm-up;
  - epoch: every get(B) minibatch with ppo_backward and either optimiser, from identical weights, each run twice alternating
    (CUDA events around the epoch), and the largest parameter difference between the two after the first run;
  - iteration: one PPO.learn iteration with n_epochs=10 at batch sizes 4,096 and 65,536, split into collect, GAE and train
    (host clock, each part ending in a device synchronise; train() ends in its own read of the log);
  - learning curve: rollout/success_rate and rollout/mean_reward of PPO("MlpPolicy", seed=0, n_steps=16, batch_size=65,536)
    over 30 iterations on fresh envs; reported, not judged."""
import argparse
import copy
import json
import os
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import spin_torque_rl_gym_b200 as stg  # noqa: E402
from tools.policy_bench import gpu_info, timed  # noqa: E402

KW = dict(clip_range=0.2, clip_range_vf=0.2, ent_coef=0.01, vf_coef=0.5)


def make_env(envs, seed=2024):
    return stg.VecNormalize(stg.make("SpinTorque-v0", num_envs=envs, device="cuda:0", max_steps=40, rng_seed=seed))


def torch_optimiser(pol):
    adam = torch.optim.Adam(pol.parameters(), lr=3e-4, eps=1e-5, fused=True)

    def step():
        torch.nn.utils.clip_grad_norm_(pol.parameters(), 0.5)
        adam.step()
    return step


def epoch_ms(pol, batches, step):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    torch.cuda.synchronize()
    ev[0].record()
    for b in batches:
        pol.ppo_backward(b, **KW)
        step()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1])


def bench_step(pol, col, reps, warmup):
    b = next(iter(col.get(4096)))
    k11, ref = copy.deepcopy(pol), copy.deepcopy(pol)
    k11.ppo_backward(b, **KW)
    ref.ppo_backward(b, **KW)
    opt = stg.ClippedAdam(k11)
    t_k11 = timed(opt.step, reps, warmup)
    t_torch = timed(torch_optimiser(ref), reps, warmup)
    return {"clipped_adam_us_median": round(t_k11[0], 2), "clipped_adam_us_min": round(t_k11[1], 2),
            "torch_clip_adam_fused_us_median": round(t_torch[0], 2), "torch_clip_adam_fused_us_min": round(t_torch[1], 2),
            "saving_us": round(t_torch[0] - t_k11[0], 2)}


def bench_epoch(pol, col, B):
    batches = list(col.get(B))
    for fused in (True, False):                                  # warm-up of both optimiser paths
        w = copy.deepcopy(pol)
        epoch_ms(w, batches[:2], stg.ClippedAdam(w).step if fused else torch_optimiser(w))
    runs = {"clipped_adam": [], "torch": []}
    for rep in range(2):
        a, t = copy.deepcopy(pol), copy.deepcopy(pol)
        runs["clipped_adam"].append(epoch_ms(a, batches, stg.ClippedAdam(a).step))
        runs["torch"].append(epoch_ms(t, batches, torch_optimiser(t)))
        if rep == 0:
            diff = max(float((p - q).abs().max() / q.abs().max()) for p, q in zip(a.parameters(), t.parameters()))
    n = len(batches)
    best_a, best_t = min(runs["clipped_adam"]), min(runs["torch"])
    return {"batch": B, "minibatches": n, "epoch_clipped_adam_ms": [round(x, 2) for x in runs["clipped_adam"]],
            "epoch_torch_optimiser_ms": [round(x, 2) for x in runs["torch"]],
            "saving_per_minibatch_us": round((best_t - best_a) * 1e3 / n, 2),
            "clipped_adam_no_slower": all(x <= y for x, y in zip(runs["clipped_adam"], runs["torch"])),
            "param_max_rel_diff_after_one_epoch": diff}


def bench_iteration(envs, steps, B):
    env = make_env(envs, seed=7)
    model = stg.PPO("MlpPolicy", env, n_steps=steps, batch_size=B, n_epochs=10, seed=0, clip_range_vf=0.2, ent_coef=0.01)
    model.learn(envs * steps)                                    # warm-up iteration (first reset, allocations)
    col = model.rollout_buffer
    out = {}
    for rep in range(2):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        col.collect(model.policy)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        col.compute_returns_and_advantage(model.gamma, model.gae_lambda)
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        logs = model.train()
        t3 = time.perf_counter()
        out = {"batch": B, "minibatches_per_epoch": -(-envs * steps // B), "collect_ms": round((t1 - t0) * 1e3, 2),
               "gae_ms": round((t2 - t1) * 1e3, 2), "train_ms": round((t3 - t2) * 1e3, 2),
               "iteration_ms": round((t3 - t0) * 1e3, 2), "repetition": rep,
               "train_logs": {k: v for k, v in logs.items()}}
    return out


def learning_curve(envs, steps, iterations):
    env = make_env(envs, seed=11)
    model = stg.PPO("MlpPolicy", env, n_steps=steps, batch_size=65536, n_epochs=10, seed=0)
    t0 = time.perf_counter()
    model.learn(iterations * envs * steps)
    torch.cuda.synchronize()
    return {"iterations": iterations, "seconds": round(time.perf_counter() - t0, 2),
            "success_rate": [round(l["rollout/success_rate"], 5) for l in model.log_history],
            "mean_reward": [round(l["rollout/mean_reward"], 5) for l in model.log_history],
            "episodes": [l["rollout/episodes"] for l in model.log_history],
            "approx_kl": [l["train/approx_kl"] for l in model.log_history],
            "explained_variance": [l["train/explained_variance"] for l in model.log_history]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--batches", type=int, nargs="+", default=[4096, 65536, 1048576])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--iterations", type=int, default=30)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ppo_train_bench needs a CUDA device")
    if max(args.batches) > args.envs * args.steps:
        raise SystemExit("every batch size must fit in one rollout of --envs x --steps samples")
    info = gpu_info()
    env = make_env(args.envs)
    torch.manual_seed(0)
    pol = stg.ActorCriticPolicy(env, log_std_init=-0.5)
    col = stg.RolloutCollector(env, n_steps=args.steps, store_values=True)
    col.collect(pol)
    col.compute_returns_and_advantage(gamma=0.99, gae_lambda=0.95)
    with torch.no_grad():
        g = torch.Generator(device="cuda:0").manual_seed(1)
        for p in pol.parameters():
            p.add_(torch.randn(p.shape, generator=g, device=p.device) * 0.03 * (p.abs().mean() + 0.05))
    res = {"gpu": info, "envs": args.envs, "steps": args.steps, "loss_settings": KW,
           "optimiser_step": bench_step(pol, col, args.reps, args.warmup),
           "epochs": [bench_epoch(pol, col, B) for B in args.batches]}
    del col, env
    res["iterations"] = [bench_iteration(args.envs, args.steps, B) for B in (4096, 65536)]
    res["learning_curve"] = learning_curve(args.envs, args.steps, args.iterations)
    res["gpu_after"] = gpu_info()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
