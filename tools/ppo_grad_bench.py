#!/usr/bin/env python
"""K10 (ActorCriticPolicy.ppo_backward): CUDA-event time of SB3's PPO minibatch loss and gradient on the fused path against
eager torch on the same batches, the fused path's share of the FP32 FMA peak by algorithmic flops, and the gradient
agreement of the two paths in the same run.

    python tools/ppo_grad_bench.py [--envs 65536] [--steps 16] [--batches 4096 65536 1048576] [--reps 20] [--out FILE]

The batches come from a real rollout: a fresh ActorCriticPolicy collects `--steps` x `--envs` samples from a VecNormalize'd
SpinTorqueVectorEnv (max_steps=40) on the fused path, then compute_returns_and_advantage() and get(B). The weights are then
perturbed (so that ratios differ from 1 and both branches of the clipped surrogate occur); clip_range_vf=0.2, ent_coef=0.01.
Per batch size B:
  - ppo_backward: the advantage statistics (two torch reductions), the K10 launch and its fold, as one call;
  - kernels: the K10 launch and its fold alone on the same arguments;
  - eager: zero_grad, evaluate_actions, SB3's loss written out, backward;
  - an epoch of each path over all get(B) minibatches with clip_grad_norm_(0.5) and Adam(fused=True), from identical weights.
Algorithmic flops per sample: forward 19,840 (K9's count) and backward 2 x 18,304 MACs (the weight and bias gradients of
every layer, the input gradients of every layer but the first), 56,448 in all; 72 bytes of samples are read per row, so the
kernel is bound by the FP32 pipe. The FP32 peak is 148 SMs x 128 FMA lanes x 2 flops x the card's maximum SM clock as
nvidia-smi reports it. Each timed window is one call, synchronised, medians after warm-up."""
import argparse
import copy
import ctypes as C
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import spin_torque_rl_gym_b200 as stg  # noqa: E402
from spin_torque_rl_gym_b200 import _lib  # noqa: E402
from tools.policy_bench import gpu_info, timed  # noqa: E402

H, OBS = 64, 12
FLOPS_FORWARD = 2 * (OBS * H + H * H + H * 2) + 2 * (OBS * H + H * H + H)
MACS_BACKWARD = sum(H * H + H * H + OBS * H + 2 * H * n_out for n_out in (2, 1))
FLOPS_PER_SAMPLE = FLOPS_FORWARD + 2 * MACS_BACKWARD
BYTES_PER_SAMPLE = 4 * (OBS + 2 + 4)
KW = dict(clip_range=0.2, clip_range_vf=0.2, ent_coef=0.01, vf_coef=0.5)


def eager_backward(pol, b):
    """SB3's PPO.train() step for one minibatch up to loss.backward(), in torch."""
    values, log_prob, entropy = pol.evaluate_actions(b.observations, b.actions)
    values = values.flatten()
    adv = b.advantages
    if len(adv) > 1:
        adv = (adv - adv.mean()) / (adv.std() + 1e-8)
    ratio = torch.exp(log_prob - b.old_log_prob)
    policy_loss = -torch.min(adv * ratio, adv * torch.clamp(ratio, 1 - KW["clip_range"], 1 + KW["clip_range"])).mean()
    vpred = b.old_values + torch.clamp(values - b.old_values, -KW["clip_range_vf"], KW["clip_range_vf"])
    value_loss = torch.nn.functional.mse_loss(b.returns, vpred)
    loss = policy_loss + KW["ent_coef"] * -torch.mean(entropy) + KW["vf_coef"] * value_loss
    pol.zero_grad(set_to_none=True)
    loss.backward()


def epoch_ms(pol, batches, fused):
    opt = torch.optim.Adam(pol.parameters(), lr=3e-4, eps=1e-5, fused=True)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    torch.cuda.synchronize()
    ev[0].record()
    for b in batches:
        if fused:
            pol.ppo_backward(b, **KW)
        else:
            eager_backward(pol, b)
        torch.nn.utils.clip_grad_norm_(pol.parameters(), 0.5)
        opt.step()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1])


def kernel_args(pol, b):
    """StgPpoArgs of ppo_backward for batch b (what the call builds), with the buffers kept alive."""
    n = b.observations.shape[0]
    keep = [torch.stack([b.advantages.mean(), b.advantages.std()]), torch.empty(6, device=b.returns.device),
            torch.empty(_lib.ppo_work_doubles(n), dtype=torch.float64, device=b.returns.device),
            torch.empty(_lib.POLICY_PARAMS, device=b.returns.device), pol.pack_weights()]
    a = _lib.StgPpoArgs()
    a.d_weights, a.d_obs, a.d_action = keep[4].data_ptr(), b.observations.data_ptr(), b.actions.data_ptr()
    a.d_old_value, a.d_old_log_prob = b.old_values.data_ptr(), b.old_log_prob.data_ptr()
    a.d_advantage, a.d_return, a.d_adv_stats = b.advantages.data_ptr(), b.returns.data_ptr(), keep[0].data_ptr()
    a.d_losses, a.d_work, a.d_grad = keep[1].data_ptr(), keep[2].data_ptr(), keep[3].data_ptr()
    a.clip_range, a.ratio_lo, a.ratio_hi = KW["clip_range"], 1 - KW["clip_range"], 1 + KW["clip_range"]
    a.clip_range_vf, a.flags = KW["clip_range_vf"], _lib.PPO_CLIP_VF
    a.ent_coef, a.vf_coef, a.batch = KW["ent_coef"], KW["vf_coef"], n
    return a, keep


def bench_batch(pol, col, B, reps, warmup, peak):
    batches = list(col.get(B))
    b = batches[0]
    t_call = timed(lambda: pol.ppo_backward(b, **KW), reps, warmup)
    a, keep = kernel_args(pol, b)
    lib, stream = _lib.load(), torch.cuda.current_stream().cuda_stream
    t_kern = timed(lambda: _lib.check(lib.stg_policy_ppo_grad_f32(C.byref(a), stream)), reps, warmup)
    eager = copy.deepcopy(pol)
    t_eager = timed(lambda: eager_backward(eager, b), reps, warmup)
    pol.ppo_backward(b, **KW)
    eager_backward(eager, b)
    agree = {}
    for (name, p), q in zip(pol.named_parameters(), eager.parameters()):
        agree[name] = float((p.grad - q.grad).abs().max() / q.grad.abs().max().clamp_min(1e-30))
    flops = B * FLOPS_PER_SAMPLE
    res = {"batch": B, "minibatches_per_epoch": len(batches),
           "ppo_backward_us_median": round(t_call[0], 2), "ppo_backward_us_min": round(t_call[1], 2),
           "k10_and_fold_us_median": round(t_kern[0], 2),
           "k10_and_fold_share_of_fp32_peak": round(flops / (t_kern[0] * 1e-6) / peak, 3),
           "ppo_backward_share_of_fp32_peak": round(flops / (t_call[0] * 1e-6) / peak, 3),
           "eager_us_median": round(t_eager[0], 2),
           "speedup_vs_eager": round(t_eager[0] / t_call[0], 2),
           "grad_max_rel_diff_fused_vs_eager": max(agree.values()), "grad_rel_diff_by_parameter": agree}
    start = copy.deepcopy(pol)
    fused_pol, eager_pol = copy.deepcopy(start), copy.deepcopy(start)
    epoch_ms(copy.deepcopy(start), batches[:2], True)                   # warm-up of the optimiser paths
    epoch_ms(copy.deepcopy(start), batches[:2], False)
    res["epoch_fused_ms"] = round(epoch_ms(fused_pol, batches, True), 2)
    res["epoch_eager_ms"] = round(epoch_ms(eager_pol, batches, False), 2)
    res["epoch_speedup"] = round(res["epoch_eager_ms"] / res["epoch_fused_ms"], 2)
    res["epoch_param_max_rel_diff"] = max(float((p - q).abs().max() / q.abs().max()) for p, q in
                                          zip(fused_pol.parameters(), eager_pol.parameters()))
    del keep
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=16)
    ap.add_argument("--batches", type=int, nargs="+", default=[4096, 65536, 1048576])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("ppo_grad_bench needs a CUDA device")
    if max(args.batches) > args.envs * args.steps:
        raise SystemExit("every batch size must fit in one rollout of --envs x --steps samples")
    dev = torch.device("cuda", 0)
    info = gpu_info()
    env = stg.VecNormalize(stg.make("SpinTorque-v0", num_envs=args.envs, device=dev, max_steps=40, rng_seed=2024))
    torch.manual_seed(0)
    pol = stg.ActorCriticPolicy(env, log_std_init=-0.5)
    col = stg.RolloutCollector(env, n_steps=args.steps, store_values=True)
    col.collect(pol)
    col.compute_returns_and_advantage(gamma=0.99, gae_lambda=0.95)
    with torch.no_grad():
        g = torch.Generator(device=dev).manual_seed(1)
        for p in pol.parameters():
            p.add_(torch.randn(p.shape, generator=g, device=dev) * 0.03 * (p.abs().mean() + 0.05))
    res = {"gpu": info, "envs": args.envs, "steps": args.steps, "samples_per_rollout": args.envs * args.steps,
           "flops_per_sample": {"forward": FLOPS_FORWARD, "backward": 2 * MACS_BACKWARD, "total": FLOPS_PER_SAMPLE},
           "bytes_per_sample": BYTES_PER_SAMPLE, "loss_settings": KW,
           "timing": "CUDA events around each call, synchronised per repetition, median after warm-up; device time. "
                     "Epochs are one call each over every get(B) minibatch of the rollout, after a two-batch warm-up.",
           "sizes": [bench_batch(pol, col, B, args.reps, args.warmup, info["fp32_peak_TFLOPs"] * 1e12)
                     for B in args.batches]}
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
