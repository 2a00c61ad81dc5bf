"""K12 and PPO(data_parallel=True): one policy trained over G ranks, the K10 gradient and the advantage statistics of each
minibatch folded across the ranks in rank order.

The specification: the loss, gradient and advantage normalisation of the union of the ranks' minibatches, bit-identical on
every rank; with one rank, exactly K10 (stg_policy_ppo_grad_f32)."""
import ctypes as C
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from spin_torque_rl_gym_b200 import _lib
from tests.helpers import ROOT
from tests.test_ppo_train import StubCollector, StubEnv, _close
from tests.test_actor_critic_policy import FakeEnv, _random_policy

HEADER = os.path.join(ROOT, "include", "stg.h")
CSRC = os.path.join(ROOT, "spin_torque_rl_gym_b200", "csrc")
E_NULL, E_SIZE, E_ENUM, E_ALIGN = -1, -2, -3, -4


# ---------------------------------------------------------------------------------------------------- CPU ---------------

def test_k12_constants_and_signatures_match_the_header(tmp_path):
    consts = dict(STG_PPO_PART_COUNT=_lib.PPO_PART_COUNT, STG_PPO_ADV_MOMENTS=_lib.PPO_ADV_MOMENTS,
                  STG_PPO_ADV_THREADS=_lib.PPO_ADV_THREADS, STG_PPO_PART=_lib.PPO_PART, STG_PPO_PART_LOSS=_lib.PPO_PART_LOSS,
                  STG_ABI_VERSION=7)
    lines = ['#include <stdio.h>', f'#include "{HEADER}"', 'int main(void){']
    lines += [f'printf("{c} %lld\\n", (long long)({c}));' for c in consts]
    lines.append('return 0;}')
    src = tmp_path / "k12.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "k12"
    subprocess.run(["gcc", str(src), "-o", str(exe)], check=True)
    # the entry points' types, checked by the compiler
    types = tmp_path / "k12_types.c"
    types.write_text("\n".join([
        f'#include "{HEADER}"',
        'int (*s)(const StgPpoArgs*, double*, void*) = stg_policy_ppo_sums_f32;',
        'int (*f)(const StgPpoArgs*, const double*, int32_t, void*) = stg_policy_ppo_finish_f32;',
        'int (*m)(const float*, int64_t, double*, void*) = stg_ppo_adv_moments_f64;',
        'int (*g)(const double*, int32_t, float*, void*) = stg_ppo_adv_merge_f32;']))
    subprocess.run(["gcc", "-fsyntax-only", "-Werror=incompatible-pointer-types", str(types)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split("\n") if l)
    for c, v in consts.items():
        assert int(got[c]) == v, c
    # the count slot follows the four loss sums and lies inside a partial
    assert _lib.PPO_PART_COUNT == _lib.PPO_PART_LOSS + 4 < _lib.PPO_PART
    text = open(HEADER).read()
    want = {"stg_policy_ppo_sums_f32": 3, "stg_policy_ppo_finish_f32": 4, "stg_ppo_adv_moments_f64": 4,
            "stg_ppo_adv_merge_f32": 4}
    for name, nargs in want.items():
        decl = re.search(rf"int {name}\(([^)]*)\);", text)
        assert decl and len(decl.group(1).split(",")) == nargs == len(_lib.SYMBOLS[name][1]), name


def _ppo_args(**over):
    B = 0x10000
    a = _lib.StgPpoArgs()
    a.d_weights, a.d_obs, a.d_action, a.d_old_value, a.d_old_log_prob = B, B * 2, B * 3, B * 4, B * 5
    a.d_advantage, a.d_return, a.d_work = B * 6, B * 7, B * 8
    a.d_grad, a.d_losses = B * 9, B * 10
    a.batch = 256
    for k, v in over.items():
        setattr(a, k, v)
    return a


def test_k12_argument_errors_in_documented_order():
    lib = _lib.load()
    B = 0x10000
    sums = lambda d_sums=B * 11, **kw: lib.stg_policy_ppo_sums_f32(C.byref(_ppo_args(**kw)), d_sums, None)  # noqa: E731
    assert lib.stg_policy_ppo_sums_f32(None, B, None) == E_NULL
    assert sums(batch=0) == E_SIZE and sums(batch=0, d_sums=None) == E_SIZE          # size before pointers
    assert sums(d_sums=None) == E_NULL
    for k in ("d_weights", "d_obs", "d_action", "d_old_value", "d_old_log_prob", "d_advantage", "d_return", "d_work"):
        assert sums(**{k: None}) == E_NULL, k
    assert sums(d_obs=None, d_weights=B + 4) == E_NULL                              # pointers before alignment
    for k, off in (("d_weights", 8), ("d_obs", 4), ("d_action", 4), ("d_work", 4), ("d_advantage", 2), ("d_adv_stats", 1)):
        base = getattr(_ppo_args(), k) or B
        assert sums(**{k: base + off}) == E_ALIGN, k
    assert sums(d_sums=B * 11 + 4) == E_ALIGN
    assert sums(d_sums=B * 11 + 4, flags=2) == E_ALIGN                              # alignment before flags
    assert sums(flags=2) == E_ENUM
    # d_grad and d_losses are not used by the sums
    assert sums(flags=2, d_grad=None, d_losses=None) == E_ENUM
    fin = lambda d_sums=B * 11, ranks=2, **kw: lib.stg_policy_ppo_finish_f32(C.byref(_ppo_args(**kw)), d_sums, ranks, None)  # noqa: E731,E501
    assert lib.stg_policy_ppo_finish_f32(None, B, 1, None) == E_NULL
    assert fin(ranks=0) == E_SIZE and fin(ranks=-1, d_sums=None) == E_SIZE
    for k in ("d_weights", "d_grad", "d_losses"):
        assert fin(**{k: None}) == E_NULL, k
    assert fin(d_sums=None) == E_NULL
    assert fin(d_grad=None, d_weights=B + 4) == E_NULL
    assert fin(d_weights=B + 8) == E_ALIGN and fin(d_sums=B + 4) == E_ALIGN and fin(d_losses=B * 10 + 2) == E_ALIGN
    mom = lib.stg_ppo_adv_moments_f64
    assert mom(B, -1, None, None) == E_SIZE
    assert mom(B, 4, None, None) == E_NULL and mom(None, 4, B, None) == E_NULL
    assert mom(B + 2, 4, B, None) == E_ALIGN and mom(B, 4, B + 4, None) == E_ALIGN
    mrg = lib.stg_ppo_adv_merge_f32
    assert mrg(B, 0, B, None) == E_SIZE and mrg(None, 0, None, None) == E_SIZE
    assert mrg(None, 2, B, None) == E_NULL and mrg(B, 2, None, None) == E_NULL
    assert mrg(B + 4, 2, B, None) == E_ALIGN and mrg(B, 2, B + 2, None) == E_ALIGN


@pytest.fixture(scope="module")
def host_merge(tmp_path_factory):
    """policy_core.cuh's K12 moments and merge compiled for the host with g++."""
    d = tmp_path_factory.mktemp("k12_host")
    src = d / "k12_host.cpp"
    src.write_text(r'''#include "policy_core.cuh"
using namespace stg;
// the advantages cut into `ranks` parts at cuts[0..ranks]: each part's moments (one thread), then the merge in rank order
extern "C" void stats(const float* adv, const long long* cuts, int ranks, float* out) {
  static double m[64 * 3];
  for (int r = 0; r < ranks; ++r) pol_adv_moments(adv + cuts[r], 0, cuts[r + 1] - cuts[r], 1, m + 3 * r);
  pol_adv_stats(m, ranks, out);
}
''')
    so = d / "k12_host.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-I", CSRC, str(src), "-o", str(so)], check=True)
    lib = C.CDLL(str(so))
    lib.stats.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]
    return lib


def _ulps(a, b):
    """distance in float32 units in the last place (finite values of one sign)"""
    ia, ib = np.float32(a).view(np.int32).astype(np.int64), np.float32(b).view(np.int32).astype(np.int64)
    return abs(int(ia) - int(ib))


def test_host_advantage_merge_matches_numpy_float64(host_merge):
    rng = np.random.default_rng(12)
    cases = []
    for n, scale, shift in ((5000, 1.0, 0.0), (4096, 30.0, 100.0), (7, 1e-3, -2.0), (2, 1.0, 0.5), (1000, 1.0, 1e3)):
        adv = (rng.standard_normal(n) * scale + shift).astype(np.float32)
        for cuts in ([0, n], [0, n // 2, n], [0, 0, n // 3, n // 3, n - 1, n, n], [0] + sorted(rng.integers(0, n, 6)) + [n],
                     [0, 1, 2, n] if n > 2 else [0, 1, n]):
            cases.append((adv, np.asarray(cuts, np.int64)))
    for adv, cuts in cases:
        out = np.zeros(2, np.float32)
        host_merge.stats(adv.ctypes.data, cuts.ctypes.data, len(cuts) - 1, out.ctypes.data)
        x = adv.astype(np.float64)
        assert _ulps(out[0], np.float32(x.mean())) <= 1, (len(adv), cuts, out[0], x.mean())
        assert _ulps(out[1], np.float32(x.std(ddof=1))) <= 1, (len(adv), cuts, out[1], x.std(ddof=1))
    # one row in all (torch: NaN std) and none at all (NaN mean and std), with empty ranks around it
    out = np.zeros(2, np.float32)
    one = np.array([3.5], np.float32)
    host_merge.stats(one.ctypes.data, np.array([0, 0, 1, 1], np.int64).ctypes.data, 3, out.ctypes.data)
    assert out[0] == 3.5 and np.isnan(out[1])
    host_merge.stats(one.ctypes.data, np.array([0, 0, 0], np.int64).ctypes.data, 2, out.ctypes.data)
    assert np.isnan(out).all()


def test_ppo_data_parallel_argument_errors(monkeypatch):
    import torch.distributed as dist
    import spin_torque_rl_gym_b200 as stg
    from spin_torque_rl_gym_b200 import ppo as ppo_mod
    from spin_torque_rl_gym_b200.envs.vec_normalize import VecNormalize
    monkeypatch.setattr(ppo_mod, "RolloutCollector", StubCollector)
    env = StubEnv()
    pol = _random_policy(env, 31)
    monkeypatch.setattr(dist, "is_initialized", lambda: True)
    monkeypatch.setattr(dist, "get_world_size", lambda group=None: 2)
    with pytest.raises(NotImplementedError, match="data_parallel=True"):
        stg.PPO(pol, env, batch_size=64)
    with pytest.raises(ValueError, match="divisible"):
        stg.PPO(pol, env, batch_size=63, data_parallel=True)

    class Unsynced(VecNormalize):
        def __init__(self, venv):                                                 # the wrapper's fields, no device
            self.venv, self.sync = venv, False

    norm = Unsynced(env)
    assert not norm._syncing() and norm.num_envs == env.num_envs
    with pytest.raises(ValueError, match="VecNormalize"):
        stg.PPO(pol, norm, batch_size=64, data_parallel=True)


# ---------------------------------------------------------------------------------------------------- GPU ---------------

def _synthetic_batch(dev, n, seed):
    """RolloutBufferSamples of n rows with values in the ranges a rollout produces."""
    import torch
    from spin_torque_rl_gym_b200.envs.sb3_vec_env import RolloutBufferSamples
    g = torch.Generator(device=dev).manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g, device=dev)                    # noqa: E731
    obs = r(n, 12).clamp(-3, 3)
    act = r(n, 2) * 0.6
    return RolloutBufferSamples(obs, act, r(n) * 0.5, r(n) * 0.3 - 1.5, r(n) * 2.0 + 0.3, r(n))


def _losses(l):
    return np.array([float(x) for x in l], np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("clip_vf", [None, 0.2])
def test_cuda_sums_then_finish_of_one_rank_equal_k10_bitwise(cuda_device, clip_vf):
    import torch
    from tests.test_ppo_grad import _perturb
    pol = _random_policy(FakeEnv(device=str(cuda_device)), 32)
    _perturb(pol, 2)
    kw = dict(clip_range=0.2, clip_range_vf=clip_vf, ent_coef=0.01, vf_coef=0.5)
    for n in (1, 127, 128, 4096, 65536, 1048576):
        b = _synthetic_batch(cuda_device, n, n)
        want_l = _losses(pol.ppo_backward(b, normalize_advantage=n > 1, **kw))
        want = pol._grad.clone()
        stats = torch.stack([b.advantages.mean(), b.advantages.std()]) if n > 1 else None
        pol._grad.fill_(float("nan"))
        sums = pol._ppo_sums(b, stats, **kw)
        got_l = _losses(pol._ppo_finish(sums[None], kw["ent_coef"], kw["vf_coef"]))
        assert torch.equal(pol._grad.view(torch.int32), want.view(torch.int32)), n
        assert np.array_equal(got_l.view(np.int32), want_l.view(np.int32)), (n, got_l, want_l)
        assert float(sums[_lib.PPO_PART_COUNT]) == n
        assert bool((sums[_lib.PPO_PART_COUNT + 1:] == 0).all())
        for p, off in pol._grad_slots():
            assert p.grad.data_ptr() == pol._grad.data_ptr() + 4 * off


@pytest.fixture(scope="module")
def dp_minibatch(cuda_device):
    """One real minibatch of 65,536 rows from a fused rollout, with perturbed weights."""
    import spin_torque_rl_gym_b200 as stg
    from tests.test_ppo_grad import _perturb, _rollout
    env, pol, col = _rollout(stg, cuda_device, 8192, 8)
    _perturb(pol, 3)
    return pol, next(iter(col.get(None)))


def _split(b, cuts):
    from spin_torque_rl_gym_b200.envs.sb3_vec_env import RolloutBufferSamples
    return [RolloutBufferSamples(*(t[lo:hi].contiguous().clone() for t in b)) for lo, hi in zip(cuts, cuts[1:])]


@pytest.mark.gpu
@pytest.mark.parametrize("G", [2, 3, 8])
def test_cuda_ranks_simulated_in_one_process_match_the_whole_batch(dp_minibatch, G):
    import torch
    from spin_torque_rl_gym_b200.policy import _adv_moments, _adv_stats
    pol, b = dp_minibatch
    n = b.observations.shape[0]
    cuts = [n * r // G for r in range(G + 1)]
    aligned = all(c % _lib.PPO_TILE == 0 for c in cuts)
    parts = _split(b, cuts)
    stats = _adv_stats(torch.stack([_adv_moments(p.advantages) for p in parts]))
    x = b.advantages.double()
    for got, want in zip(stats.cpu().numpy(), (x.mean().item(), x.std().item())):
        assert _ulps(got, np.float32(want)) <= 1, (G, got, want)
    kw = dict(clip_range=0.2, clip_range_vf=0.2, ent_coef=0.01, vf_coef=0.5)
    want_l = _losses(pol._ppo_finish(pol._ppo_sums(b, stats, **kw)[None], 0.01, 0.5))     # K10 on the whole batch
    want = pol._grad.clone()
    sums = torch.stack([pol._ppo_sums(p, stats, **kw) for p in parts])
    got_l = _losses(pol._ppo_finish(sums, 0.01, 0.5))
    got = pol._grad.clone()
    for p, off in pol._grad_slots():
        k = p.numel()
        _close(got[off:off + k].cpu(), want[off:off + k].cpu(), 1e-6, f"G={G} offset {off}")
    assert np.abs(got_l - want_l).max() <= 1e-6 * max(1.0, np.abs(want_l).max()), (got_l, want_l)
    if aligned:
        ulps = (got.view(torch.int32).long() - want.view(torch.int32).long()).abs()
        print(f"G={G}: {int((ulps > 0).sum())} of {got.numel()} gradient elements differ (FP64 order), max {int(ulps.max())} ulp")
        assert int(ulps.max()) <= 1


WORKER = r'''
import os, sys, json
sys.path.insert(0, sys.argv[1])
out, backend = sys.argv[2], sys.argv[3]
import torch, torch.distributed as dist
import spin_torque_rl_gym_b200 as stg
dist.init_process_group(backend)
rank, world = dist.get_rank(), dist.get_world_size()
dev = torch.device("cuda", rank % torch.cuda.device_count())
torch.cuda.set_device(dev)
N = 4096

def env(**kw):
    return stg.make("SpinTorque-v0", num_envs=N, device=dev, max_steps=40, rng_seed=7, env_offset=rank * N, **kw)

def save(name, model, col):
    torch.save({"state": {k: v.cpu() for k, v in model.policy.state_dict().items()}, "log": model.log_history,
                "obs": col.observations.cpu(), "act": col.actions.cpu(), "rew": col.rewards.cpu()},
               os.path.join(out, f"{name}_{rank}.pt"))

# (a) raw env without the thermal field, one minibatch = the whole global rollout
m = stg.PPO("MlpPolicy", env(include_thermal_fluctuations=False), n_steps=8, batch_size=8 * N * world, n_epochs=3, seed=3, data_parallel=True,
            policy_kwargs=dict(log_std_init=-0.5))
m.learn(8 * N * world)
save("a", m, m.rollout_buffer)
# (b) 16 minibatches per epoch and target_kl
m = stg.PPO("MlpPolicy", env(), learning_rate=1e-3, n_steps=8, batch_size=4096, n_epochs=10, seed=3, target_kl=1e-4,
            data_parallel=True)
m.learn(8 * N * world)
save("b", m, m.rollout_buffer)
# (c) VecNormalize shared across the ranks and the seven-line loop
norm = stg.VecNormalize(env(), sync=None)
torch.manual_seed(100 + rank)                                  # different initial weights: rank 0's are broadcast below
pol = stg.ActorCriticPolicy(norm, seed=11)
for p in pol.parameters():
    dist.broadcast(p.data, src=0)
opt = stg.ClippedAdam(pol, lr=3e-4, max_grad_norm=0.5)
col = stg.RolloutCollector(norm, n_steps=8, store_values=True)
for it in range(2):
    col.collect(pol); col.compute_returns_and_advantage()
    for epoch in range(2):
        for b in col.get(2048):
            losses = pol.ppo_backward(b, data_parallel=True)
            opt.step()
torch.save({"state": {k: v.cpu() for k, v in pol.state_dict().items()}, "vn": norm._stats.cpu(),
            "loss": float(losses.loss)}, os.path.join(out, f"c_{rank}.pt"))
torch.cuda.synchronize()
dist.destroy_process_group()
print("DONE", rank)
'''


def _run_ranks(tmp_path, backend, port):
    script = tmp_path / "dp_worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), str(script), ROOT, str(tmp_path), backend]
    res = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=900)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-5000:]
    import torch
    return {k: [torch.load(tmp_path / f"{k}_{r}.pt", weights_only=False) for r in range(2)] for k in "abc"}


def _same_state(s0, s1):
    import torch
    return all(torch.equal(s0[k].view(torch.int32), s1[k].view(torch.int32)) for k in s0)


def _check_ranks(got, cuda_device):
    import torch
    import spin_torque_rl_gym_b200 as stg
    a, b, c = got["a"], got["b"], got["c"]
    for run in (a, b):
        assert _same_state(run[0]["state"], run[1]["state"])
        assert json.dumps(run[0]["log"]) == json.dumps(run[1]["log"])              # every value, bit for bit
    # (a) against one process over all 8,192 envs with the same seeds (resets and action noise keyed by global env id)
    env = stg.make("SpinTorque-v0", num_envs=8192, device=cuda_device, max_steps=40, rng_seed=7,
                   include_thermal_fluctuations=False)
    ref = stg.PPO("MlpPolicy", env, n_steps=8, batch_size=8 * 8192, n_epochs=3, seed=3, policy_kwargs=dict(log_std_init=-0.5))
    ref.learn(8 * 8192)
    col = ref.rollout_buffer
    for r in range(2):
        sl = slice(r * 4096, (r + 1) * 4096)
        for k, plane in (("obs", col.observations), ("act", col.actions), ("rew", col.rewards)):
            # the rollouts of 2 x 4,096 and 1 x 8,192 envs agree to rounding, not bit for bit (on a B200, about 0.25 % of
            # the observation, 5 % of the action and 1 % of the reward elements differ); the counts are printed
            want = plane[:, sl].cpu()
            print(f"rank {r} {k}: {int((a[r][k] != want).sum())} of {want.numel()} elements differ from one process")
            _close(a[r][k], want, 1e-5, f"rollout {k} of rank {r}")
    for k, v in ref.policy.state_dict().items():
        _close(a[0]["state"][k], v.cpu(), 1e-5, k)
    want, log = ref.log_history[0], a[0]["log"][0]
    assert log["time/total_timesteps"] == want["time/total_timesteps"] == 8 * 8192
    for k in ("train/policy_gradient_loss", "train/value_loss", "train/entropy_loss", "train/loss", "train/std",
              "train/explained_variance"):
        assert abs(log[k] - want[k]) <= 1e-4 * abs(want[k]) + 1e-6, (k, log[k], want[k])
    assert log["train/approx_kl"] == pytest.approx(want["train/approx_kl"], rel=1e-3, abs=1e-7)
    # (b) the gate trips on the same minibatch everywhere
    assert b[0]["log"][0]["train/n_updates"] == b[1]["log"][0]["train/n_updates"] < 10
    # (c) VecNormalize statistics and weights identical across the ranks
    assert torch.equal(c[0]["vn"], c[1]["vn"]) and _same_state(c[0]["state"], c[1]["state"])
    assert c[0]["loss"] == c[1]["loss"]


@pytest.mark.gpu
def test_cuda_two_ranks_gloo_train_one_policy(cuda_device, tmp_path):
    _check_ranks(_run_ranks(tmp_path, "gloo", 29541), cuda_device)


@pytest.mark.gpu
def test_cuda_two_ranks_nccl_train_one_policy(cuda_device, tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("NCCL needs one GPU per rank; fewer than 2 GPUs are visible")
    _check_ranks(_run_ranks(tmp_path, "nccl", 29543), cuda_device)
