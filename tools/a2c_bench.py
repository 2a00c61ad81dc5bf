#!/usr/bin/env python
"""K10's A2C instance (a2c_backward), K13 (ClippedRMSprop) and stg.A2C at SB3's A2C defaults: the whole-rollout loss and
gradient, the optimiser step and one learn() iteration, against eager torch in the same run.

    python tools/a2c_bench.py [--envs 1048576] [--steps 5] [--reps 20] [--warmup 5] [--out FILE]

Setup: a fresh ActorCriticPolicy collects `--steps` x `--envs` samples (SB3's A2C default n_steps=5) from a VecNormalize'd
SpinTorqueVectorEnv (max_steps=40) on the fused path, GAE with gae_lambda=1.0, then the weights are perturbed; ent_coef=0.01,
vf_coef=0.5. Reported:
  - backward: a2c_backward over the whole rollout (rollout_samples(), n_steps x N rows) against eager torch on the same rows
    (evaluate_actions, SB3's A2C loss, backward()), and the largest gradient difference relative to each tensor's largest
    entry; CUDA events around each call, synchronised per repetition, median of `--reps` after `--warmup`;
  - optimiser step: ClippedRMSprop.step() (one K13 launch) against clip_grad_norm_(0.5) + RMSprop(alpha=0.99, eps=1e-5,
    foreach=False and foreach=True) on the same gradient;
  - iteration: one A2C.learn iteration split into collect, GAE and train (host clock, each part ending in a device
    synchronise; train() ends in its own read of the losses), after one warm-up iteration."""
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

KW = dict(ent_coef=0.01, vf_coef=0.5)


def make_env(envs, seed=2024):
    return stg.VecNormalize(stg.make("SpinTorque-v0", num_envs=envs, device="cuda:0", max_steps=40, rng_seed=seed))


def eager_a2c_backward(pol, b):
    """SB3's A2C.train() loss and backward() in eager torch."""
    pol.zero_grad(set_to_none=True)
    values, log_prob, entropy = pol.evaluate_actions(b.observations, b.actions)
    policy_loss = -(b.advantages * log_prob).mean()
    value_loss = torch.nn.functional.mse_loss(b.returns, values.flatten())
    loss = policy_loss + KW["ent_coef"] * -torch.mean(entropy) + KW["vf_coef"] * value_loss
    loss.backward()


def bench_backward(pol, col, reps, warmup):
    b = col.rollout_samples()
    fused, eager = copy.deepcopy(pol), copy.deepcopy(pol)
    t_fused = timed(lambda: fused.a2c_backward(b, **KW), reps, warmup)
    t_eager = timed(lambda: eager_a2c_backward(eager, b), reps, warmup)
    diff = max(float((p.grad - q.grad).abs().max() / q.grad.abs().max()) for p, q in zip(fused.parameters(),
                                                                                          eager.parameters()))
    return {"rows": b.observations.shape[0], "a2c_backward_us_median": round(t_fused[0], 1),
            "a2c_backward_us_min": round(t_fused[1], 1), "eager_torch_us_median": round(t_eager[0], 1),
            "eager_torch_us_min": round(t_eager[1], 1), "speedup_median": round(t_eager[0] / t_fused[0], 2),
            "grad_max_rel_diff_vs_eager": diff}


def torch_rmsprop(pol, foreach):
    opt = torch.optim.RMSprop(pol.parameters(), lr=7e-4, alpha=0.99, eps=1e-5, foreach=foreach)

    def step():
        torch.nn.utils.clip_grad_norm_(pol.parameters(), 0.5)
        opt.step()
    return step


def bench_step(pol, col, reps, warmup):
    b = col.rollout_samples()
    k13, ref1, ref2 = (copy.deepcopy(pol) for _ in range(3))
    for x in (k13, ref1, ref2):
        x.a2c_backward(b, **KW)
    t_k13 = timed(stg.ClippedRMSprop(k13).step, reps, warmup)
    t_single = timed(torch_rmsprop(ref1, False), reps, warmup)
    t_foreach = timed(torch_rmsprop(ref2, True), reps, warmup)
    return {"clipped_rmsprop_us_median": round(t_k13[0], 2), "clipped_rmsprop_us_min": round(t_k13[1], 2),
            "torch_clip_rmsprop_single_tensor_us_median": round(t_single[0], 2),
            "torch_clip_rmsprop_foreach_us_median": round(t_foreach[0], 2)}


def bench_iteration(envs, steps):
    env = make_env(envs, seed=7)
    model = stg.A2C("MlpPolicy", env, n_steps=steps, seed=0, **KW)
    model.learn(envs * steps)                                    # warm-up iteration (first reset, allocations)
    col = model.rollout_buffer
    out = []
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
        out.append({"repetition": rep, "collect_ms": round((t1 - t0) * 1e3, 2), "gae_ms": round((t2 - t1) * 1e3, 2),
                    "train_ms": round((t3 - t2) * 1e3, 2), "iteration_ms": round((t3 - t0) * 1e3, 2),
                    "train_logs": dict(logs)})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("a2c_bench needs a CUDA device")
    info = gpu_info()
    env = make_env(args.envs)
    torch.manual_seed(0)
    pol = stg.ActorCriticPolicy(env, log_std_init=-0.5)
    col = stg.RolloutCollector(env, n_steps=args.steps, store_values=True)
    col.collect(pol)
    col.compute_returns_and_advantage(gamma=0.99, gae_lambda=1.0)
    with torch.no_grad():
        g = torch.Generator(device="cuda:0").manual_seed(1)
        for p in pol.parameters():
            p.add_(torch.randn(p.shape, generator=g, device=p.device) * 0.03 * (p.abs().mean() + 0.05))
    res = {"gpu": info, "envs": args.envs, "steps": args.steps, "loss_settings": KW,
           "backward": bench_backward(pol, col, args.reps, args.warmup),
           "optimiser_step": bench_step(pol, col, args.reps, args.warmup)}
    del col, env
    torch.cuda.empty_cache()
    res["iterations"] = bench_iteration(args.envs, args.steps)
    res["gpu_after"] = gpu_info()
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
