#!/usr/bin/env python
"""K9 (ActorCriticPolicy): CUDA-event time of the fused policy launches on real env observations, their share of the FP32
FMA peak by algorithmic flops, and, in the same run, the same work done eagerly in torch with its outputs compared.

    python tools/policy_bench.py [--envs 131072 1048576] [--reps 20] [--warmup 5] [--n-steps 128] [--out FILE]

Per size, on a SpinTorqueVectorEnv with max_steps=100 (thermal noise on):
  - one 128-step `RolloutCollector.collect(policy)` on the fused path first (it warms everything up and leaves the env in
    steady state, past the first truncation at step 100), from which the mean number of ended envs per step is taken;
  - the act launch (stg_policy_act_f32 with all five outputs) on the env's current observations, `--reps` times;
  - the masked critic launch (stg_policy_value_f32) on the env's final observations with a mask of the measured end rate
    (rows drawn at random), and with every row selected;
  - the eager torch step: the module's layers, torch.distributions.Normal sampling and log_prob, the rescale, the four copies
    into collector planes, and the critic over all N final rows (what a collector with a torch policy and value_fn does);
  - the K1 env step alone, with the policy's env actions;
  - a full 128-step collect() with each path, timed with events around the call (device time of the whole rollout).
Algorithmic flops per env: actor 2 (12*64 + 64*64 + 64*2) = 9,984, critic 2 (12*64 + 64*64 + 64) = 9,856, together 19,840
(tanh, sampling and the rescale are not counted). The FP32 peak is 148 SMs x 128 FMA lanes x 2 flops x the card's maximum
SM clock as nvidia-smi reports it. Each timed window is one launch, timed separately, medians reported; the 50 MB of
observations at 1,048,576 envs fit in L2, so the act launch reads them from there after the first repetition."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import spin_torque_rl_gym_b200 as stg  # noqa: E402
from spin_torque_rl_gym_b200 import _lib  # noqa: E402

FLOPS_ACTOR, FLOPS_CRITIC = 2 * (12 * 64 + 64 * 64 + 64 * 2), 2 * (12 * 64 + 64 * 64 + 64)
SMS, FMA_LANES = 148, 128


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                       capture_output=True, text=True, timeout=60).stdout.strip().splitlines()
    name, power, clock = [s.strip() for s in q[0].split(",")]
    return {"name": name, "power_limit_W": float(power), "max_sm_clock_MHz": float(clock),
            "fp32_peak_TFLOPs": SMS * FMA_LANES * 2 * float(clock) * 1e6 / 1e12}


def median(xs):
    xs = sorted(xs)
    return xs[len(xs) // 2]


def timed(fn, reps, warmup):
    """Median and minimum microseconds of fn() between two events, each repetition synchronised."""
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    out = []
    for r in range(warmup + reps):
        ev[0].record()
        fn()
        ev[1].record()
        torch.cuda.synchronize()
        if r >= warmup:
            out.append(ev[0].elapsed_time(ev[1]) * 1e3)
    return median(out), min(out)


class EagerStep:
    """The policy's step in eager torch, writing the collector planes like RolloutCollector's generic path."""

    def __init__(self, pol, n, dev):
        self.pol = pol
        self.planes = [torch.empty(n, 12, device=dev), torch.empty(n, 2, device=dev), torch.empty(n, device=dev),
                       torch.empty(n, device=dev), torch.empty(n, device=dev)]

    def policy(self, obs):
        pol = self.pol
        latent_pi, latent_vf = pol.mlp_extractor(obs)
        mean = pol.action_net(latent_pi)
        dist = torch.distributions.Normal(mean, torch.ones_like(mean) * pol.log_std.exp())
        a = dist.rsample()
        return a, pol.scale_action(a), pol.value_net(latent_vf), dist.log_prob(a).sum(dim=1)

    def critic(self, obs):
        return self.pol.value_net(self.pol.mlp_extractor.forward_critic(obs))

    def __call__(self, obs, final_obs):
        with torch.no_grad():
            a, env_a, v, lp = self.policy(obs)
            o_p, a_p, v_p, lp_p, f_p = self.planes
            o_p.copy_(obs)
            a_p.copy_(a)
            v_p.copy_(v.reshape(-1))
            lp_p.copy_(lp)
            f_p.copy_(self.critic(final_obs).reshape(-1))
            return env_a


def bench_size(n, reps, warmup, n_steps, dev):
    venv = stg.make("SpinTorque-v0", num_envs=n, device=dev, rng_seed=2024, max_steps=100)
    torch.manual_seed(0)
    pol = stg.ActorCriticPolicy(venv, log_std_init=-0.5)
    col = stg.RolloutCollector(venv, n_steps=n_steps, store_values=True)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

    def collect_us(fn):
        torch.cuda.synchronize()
        ev[0].record()
        fn()
        ev[1].record()
        torch.cuda.synchronize()
        return ev[0].elapsed_time(ev[1]) * 1e3

    collect_us(lambda: col.collect(pol))                                   # warm-up, and past the first truncation
    t_fused = collect_us(lambda: col.collect(pol))
    ended = col.dones.sum(1).float()
    end_rate = float(ended.mean()) / n
    obs = venv._obs
    final = venv._final_obs
    lib = _lib.load()
    w = pol.pack_weights()
    bufs = [torch.empty(n, 12, device=dev), torch.empty(n, 2, device=dev), torch.empty(n, 2, device=dev),
            torch.empty(n, device=dev), torch.empty(n, device=dev), torch.full((n,), float("nan"), device=dev)]
    act = pol._args(w, n)
    act.d_obs, act.d_obs_copy, act.d_action, act.d_env_action = obs.data_ptr(), *(b.data_ptr() for b in bufs[:3])
    act.d_value, act.d_log_prob = bufs[3].data_ptr(), bufs[4].data_ptr()
    stream = torch.cuda.current_stream(dev).cuda_stream
    g = torch.Generator(device=dev).manual_seed(n)
    mask_rate = (torch.rand(n, generator=g, device=dev) < end_rate).to(torch.uint8)
    mask_all = torch.ones(n, dtype=torch.uint8, device=dev)
    val = pol._args(w, n)
    val.d_obs, val.d_value = final.data_ptr(), bufs[5].data_ptr()

    def act_launch():
        _lib.check(lib.stg_policy_act_f32(C.byref(act), stream))

    def value_launch(mask):
        val.d_mask = mask.data_ptr()
        _lib.check(lib.stg_policy_value_f32(C.byref(val), stream))

    t_act = timed(act_launch, reps, warmup)
    t_val_rate = timed(lambda: value_launch(mask_rate), reps, warmup)
    t_val_all = timed(lambda: value_launch(mask_all), reps, warmup)
    eager = EagerStep(pol, n, dev)
    t_eager = timed(lambda: eager(obs, final), reps, warmup)
    env_actions = bufs[2].clone()
    t_k1 = timed(lambda: venv.step(env_actions), reps, warmup)
    # outputs of both paths on the same inputs (the env has stepped: fresh observations)
    act_launch()
    value_launch(mask_all)
    with torch.no_grad():
        _, _, v_e, _ = eager.policy(obs)
        _, lp_e, _ = pol.evaluate_actions(obs, bufs[1])
        fv_e = eager.critic(final)[:, 0]
        det = pol(obs, deterministic=True)[0]
        mean_e = pol.action_net(pol.mlp_extractor.forward_actor(obs))
    torch.cuda.synchronize()
    diffs = {"value": float((bufs[3] - v_e[:, 0]).abs().max()), "log_prob": float((bufs[4] - lp_e).abs().max()),
             "final_value": float((bufs[5] - fv_e).abs().max()), "mean": float((det - mean_e).abs().max()),
             "obs_copy": float((bufs[0] - obs).abs().max()),
             "env_action_vs_scale_action": float((bufs[2] - pol.scale_action(bufs[1])).abs().max())}

    def eager_policy(o):
        a, env_a, v, lp = eager.policy(o)
        return env_a, v, lp

    t_eager_collect = collect_us(lambda: col.collect(eager_policy, eager.critic))
    peak = INFO["fp32_peak_TFLOPs"] * 1e12
    flops_act = n * (FLOPS_ACTOR + FLOPS_CRITIC)
    fused_step = t_act[0] + t_val_rate[0]
    return {
        "envs": n, "reps": reps, "ended_envs_per_step_mean": round(end_rate * n, 1), "end_rate": round(end_rate, 5),
        "act_us_median": round(t_act[0], 2), "act_us_min": round(t_act[1], 2),
        "act_algorithmic_TFLOPs": round(flops_act / (t_act[0] * 1e-6) / 1e12, 2),
        "act_share_of_fp32_peak": round(flops_act / (t_act[0] * 1e-6) / peak, 3),
        "value_masked_at_end_rate_us_median": round(t_val_rate[0], 2),
        "value_all_rows_us_median": round(t_val_all[0], 2),
        "value_all_rows_share_of_fp32_peak": round(n * FLOPS_CRITIC / (t_val_all[0] * 1e-6) / peak, 3),
        "fused_policy_us_per_step": round(fused_step, 2),
        "eager_torch_us_per_step": round(t_eager[0], 2),
        "policy_speedup_vs_eager": round(t_eager[0] / fused_step, 2),
        "k1_step_us_median": round(t_k1[0], 2),
        "collect_steps": n_steps,
        "collect_fused_ms": round(t_fused / 1e3, 2), "collect_eager_ms": round(t_eager_collect / 1e3, 2),
        "collect_fused_us_per_step": round(t_fused / n_steps, 2),
        "collect_eager_us_per_step": round(t_eager_collect / n_steps, 2),
        "collect_speedup": round(t_eager_collect / t_fused, 3),
        "policy_share_of_fused_collect": round(fused_step * n_steps / t_fused, 3),
        "max_abs_diff_fused_vs_eager": diffs,
    }


INFO = {}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, nargs="+", default=[131072, 1048576])
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--n-steps", type=int, default=128)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("policy_bench needs a CUDA device")
    dev = torch.device("cuda", 0)
    INFO.update(gpu_info())
    res = {"gpu": INFO, "flops_per_env": {"actor": FLOPS_ACTOR, "critic": FLOPS_CRITIC},
           "timing": "CUDA events around each launch or call, synchronised per repetition, median after warm-up; device "
                     "time. Collect times are one call each, after a warm-up collect.",
           "sizes": [bench_size(n, args.reps, args.warmup, args.n_steps, dev) for n in args.envs]}
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(text + "\n")


if __name__ == "__main__":
    main()
