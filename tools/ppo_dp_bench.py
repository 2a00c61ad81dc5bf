#!/usr/bin/env python
"""K12 (ActorCriticPolicy.ppo_backward(data_parallel=True), PPO(data_parallel=True)): what the data-parallel minibatch path
costs.

    python tools/ppo_dp_bench.py [--envs 65536] [--steps 16] [--batches 4096 65536 1048576] [--reps 30] [--out FILE]
    torchrun --nproc-per-node=G tools/ppo_dp_bench.py --learn [--envs 65536] [--out FILE]

One process (no process group, world size 1): per batch size B, CUDA-event medians after warm-up of
  - k10: ppo_backward(b): torch's adv.mean() / adv.std(), the K10 launch and its fold;
  - k12: ppo_backward(b, data_parallel=True): advantage moments, merge, sums (K10's launch and the raw fold) and finish, with
         no collective;
  - moments, merge: stg_ppo_adv_moments_f64 and stg_ppo_adv_merge_f32 alone.
The batches come from a real rollout (a fresh ActorCriticPolicy on a VecNormalize'd SpinTorqueVectorEnv, max_steps=40,
`--steps` x `--envs` samples, weights then perturbed); clip_range_vf=0.2, ent_coef=0.01. The two paths' gradients are
compared in the same run (they differ only by the rounding of the advantage mean and std: torch's float32 reduction against
FP64 moments rounded once).

With `--learn` under torchrun (NCCL, one GPU per rank): weak scaling of one PPO(data_parallel=True).learn() iteration with
`--envs` envs per rank, n_steps=16, batch_size = 65,536 x G, 10 epochs: the time of collect (with GAE), of train, and of one
all_gather of the 10,192-double sums vector alone. Rank 0 writes the result."""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import spin_torque_rl_gym_b200 as stg  # noqa: E402
from spin_torque_rl_gym_b200 import _lib  # noqa: E402
from spin_torque_rl_gym_b200.policy import _adv_moments, _adv_stats  # noqa: E402
from tools.policy_bench import gpu_info, timed  # noqa: E402

KW = dict(clip_range=0.2, clip_range_vf=0.2, ent_coef=0.01, vf_coef=0.5)
BYTES_PER_MINIBATCH = 8 * (_lib.PPO_ADV_MOMENTS + _lib.PPO_PART)       # gathered from each rank


def one_gpu(args, dev):
    env = stg.VecNormalize(stg.make("SpinTorque-v0", num_envs=args.envs, device=dev, max_steps=40, rng_seed=5))
    torch.manual_seed(5)
    pol = stg.ActorCriticPolicy(env, log_std_init=-0.5)
    col = stg.RolloutCollector(env, n_steps=args.steps, store_values=True)
    col.collect(pol)
    col.compute_returns_and_advantage(0.99, 0.95)
    g = torch.Generator(device=dev).manual_seed(1)
    with torch.no_grad():
        for p in pol.parameters():
            p.add_(torch.randn(p.shape, generator=g, device=dev) * 0.03 * (p.abs().mean() + 0.05))
    rows = []
    for B in args.batches:
        b = next(iter(col.get(B)))
        k10 = timed(lambda: pol.ppo_backward(b, **KW), args.reps, 5)
        ref = pol._grad.clone()
        k12 = timed(lambda: pol.ppo_backward(b, data_parallel=True, **KW), args.reps, 5)
        diff = float((pol._grad - ref).abs().max() / ref.abs().max())
        m = _adv_moments(b.advantages)
        mom = timed(lambda: _adv_moments(b.advantages), args.reps, 5)
        mrg = timed(lambda: _adv_stats(m), args.reps, 5)
        row = {"batch": B, "k10_us": k10[0], "k12_us": k12[0], "k12_over_k10": k12[0] / k10[0], "moments_us": mom[0],
               "merge_us": mrg[0], "k10_min_us": k10[1], "k12_min_us": k12[1], "grad_max_rel_diff": diff}
        print(json.dumps(row), flush=True)
        rows.append(row)
    return {"mode": "one_gpu", "envs": args.envs, "steps": args.steps, "reps": args.reps, "rows": rows}


def learn(args, dev):
    import torch.distributed as dist
    from spin_torque_rl_gym_b200.parallel import all_gather_moments
    rank, G = dist.get_rank(), dist.get_world_size()
    env = stg.VecNormalize(stg.make("SpinTorque-v0", num_envs=args.envs, device=dev, max_steps=40, rng_seed=5,
                                    env_offset=rank * args.envs))
    model = stg.PPO("MlpPolicy", env, n_steps=16, batch_size=65536 * G, n_epochs=10, seed=0, data_parallel=True)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    out = []
    for it in range(3):                                 # the first iteration is warm-up
        dist.barrier()
        ev[0].record()
        model.rollout_buffer.collect(model.policy)
        model.rollout_buffer.compute_returns_and_advantage(0.99, 0.95)
        ev[1].record()
        model.train()
        ev[2].record()
        torch.cuda.synchronize()
        if it:
            out.append((ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])))
    sums = torch.zeros(_lib.PPO_PART, dtype=torch.float64, device=dev)
    gather = timed(lambda: all_gather_moments(sums), args.reps, 5)
    res = {"mode": "learn", "world_size": G, "envs_per_rank": args.envs, "collect_ms": min(o[0] for o in out),
           "train_ms": min(o[1] for o in out), "sums_all_gather_us": gather[0],
           "minibatches_per_train": 10 * (16 * args.envs) // 65536}
    return res if rank == 0 else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--batches", type=int, nargs="+", default=[4096, 65536, 1048576])
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--learn", action="store_true")
    ap.add_argument("--out")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ppo_dp_bench needs a CUDA device")
    if args.learn:
        import torch.distributed as dist
        dist.init_process_group("nccl")
        dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", 0)))
        torch.cuda.set_device(dev)
        res = learn(args, dev)
        dist.destroy_process_group()
    else:
        dev = torch.device("cuda", 0)
        res = one_gpu(args, dev)
    if res is None:
        return
    res.update(gpu=gpu_info(), bytes_gathered_per_minibatch_per_rank=BYTES_PER_MINIBATCH)
    print(json.dumps(res))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
