"""K11 (stg_policy_adam_f32, ClippedAdam) and stg.PPO: SB3's PPO optimiser step and its learn() / train() loop.

The specification of K11 is `torch.nn.utils.clip_grad_norm_` followed by `torch.optim.Adam` (single-tensor update) with the
operation order and roundings of include/stg.h; that of PPO is Stable-Baselines3's PPO.train() written out literally in torch
(`evaluate_actions`, the loss, `backward`, `clip_grad_norm_`, `torch.optim.Adam`)."""
import copy
import ctypes as C
import math
import os
import subprocess
import warnings

import numpy as np
import pytest

from spin_torque_rl_gym_b200 import _lib
from tests.helpers import ROOT
from tests.test_actor_critic_policy import FakeEnv, _random_policy
from tests.test_ppo_grad import _fields, _perturb, _venv, sb3_ppo_loss

HEADER = os.path.join(ROOT, "include", "stg.h")
CSRC = os.path.join(ROOT, "spin_torque_rl_gym_b200", "csrc")
SEGMENTS = ("PI_W1", "PI_B1", "PI_W2", "PI_B2", "VF_W1", "VF_B1", "VF_W2", "VF_B2", "ACT_W", "ACT_B", "VAL_W", "VAL_B",
            "LOG_STD")
SHAPES = ((64, 12), (64,), (64, 64), (64,), (64, 12), (64,), (64, 64), (64,), (2, 64), (2,), (1, 64), (1,), (2,))
# logged train/ values against the literal SB3 reference: relative, with an absolute floor for values near zero (the policy
# loss and approx_kl are means of O(1) float32 terms over 4,096 rows, which eager torch sums with errors of order 1e-7)
LOG_RTOL, LOG_ATOL = 1e-4, 1e-6


def _close(got, want, tol=1e-5, what=""):
    """max |got - want| <= tol * max |want| (both tensors or arrays)."""
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    scale = float(np.abs(want).max())
    err = float(np.abs(got - want).max())
    assert err <= tol * max(scale, 1e-30), (what, err, scale)


# ---------------------------------------------------------------------------------------------------- host build ----------

@pytest.fixture(scope="module")
def host_adam(tmp_path_factory):
    """optim_core.cuh compiled for the host with g++: the kernel's work on flat arrays, serially."""
    d = tmp_path_factory.mktemp("adam_host")
    src = d / "adam_host.cpp"
    src.write_text(r'''#include "optim_core.cuh"
using namespace stg;
extern "C" double sumsq(const float* g) {
  static double part[kAdamThreads];
  for (int t = 0; t < kAdamThreads; ++t) part[t] = adam_norm_chain(g, STG_POLICY_PARAMS, t);
  return adam_norm_tree(part);
}
extern "C" void step(float* p, float* g, float* m, float* v, float* count, double lr, double b1, double b2, double eps,
                     double max_norm, int clip) {
  const float coef = clip ? adam_clip_coef(sumsq(g), max_norm) : 1.0f;
  *count = Pk<float>::add(*count, 1.0f);
  const AdamCoef c = adam_coef(*count, lr, b1, b2, eps);
  for (int s = 0; s < STG_ADAM_TENSORS; ++s)
    for (int i = adam_offset(s); i < adam_offset(s + 1); ++i) {
      if (clip) g[i] = Pk<float>::mul(g[i], coef);
      p[i] = adam_element(p[i], g[i], m[i], v[i], c);
    }
}
''')
    so = d / "adam_host.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-I", CSRC, str(src), "-o", str(so)], check=True)
    lib = C.CDLL(str(so))
    dp, dd = C.c_void_p, C.c_double
    lib.sumsq.restype, lib.sumsq.argtypes = dd, [dp]
    lib.step.argtypes = [dp] * 5 + [dd] * 5 + [C.c_int]
    return lib


def numpy_step(p, g, m, v, count, lr, b1, b2, eps, max_norm):
    """include/stg.h's K11 contract restated in NumPy (float32 arrays, every operation rounded): returns the new
    (p, g, m, v, count) and the total norm."""
    f = np.float32
    T, n = _lib.ADAM_THREADS, _lib.POLICY_PARAMS
    total = None
    if max_norm is not None:
        g64 = np.zeros(-(-n // T) * T)
        g64[:n] = g.astype(np.float64)
        part = np.zeros(T)
        for k in range(len(g64) // T):
            part = part + g64[k * T:(k + 1) * T] * g64[k * T:(k + 1) * T]
        h = T // 2
        while h >= 1:
            part[:h] = part[:h] + part[h:2 * h]
            h //= 2
        total = f(np.sqrt(part[0]))
        coef = (f(1) / (total + f(1e-6))) * f(max_norm)
        coef = f(1) if coef > 1 else coef
        g = g * coef
    count = f(count + f(1))
    s = float(count)
    bc1, bc2 = 1 - b1 ** s, 1 - b2 ** s
    w1, fb2, w2, feps = f(1 - b1), f(b2), f(1 - b2), f(eps)
    ss, bc2s = f(lr / bc1), f(math.sqrt(bc2))
    d = g - m
    m = m + w1 * d if w1 < f(0.5) else g - d * (f(1) - w1)
    v = v * fb2 + (w2 * g) * g
    denom = np.sqrt(v) / bc2s + feps
    p = p - (ss * m) / denom
    return p, g, m, v, count, total


@pytest.mark.parametrize("max_norm", [0.5, None, 1e4])
def test_core_matches_numpy_bitwise_and_torch_cpu(host_adam, max_norm):
    import torch
    rng = np.random.default_rng(3)
    n = _lib.POLICY_PARAMS
    p = rng.normal(size=n).astype(np.float32)
    m, v = np.zeros(n, np.float32), np.zeros(n, np.float32)
    count = np.zeros(1, np.float32)
    np_state = (p.copy(), m.copy(), v.copy(), np.float32(0))
    params = [torch.nn.Parameter(torch.from_numpy(p[_lib.POLICY_LAYOUT[k]:_lib.POLICY_LAYOUT[k] + int(np.prod(s))]
                                                  .reshape(s).copy())) for k, s in zip(SEGMENTS, SHAPES)]
    opt = torch.optim.Adam(params, lr=3e-4, eps=1e-5, foreach=False)
    clipped = 0
    sign, mag = rng.choice([-1.0, 1.0], size=n), rng.choice([1e-4, 0.01, 0.05], size=n)   # a gradient with a direction
    for it in range(50):
        lr = 3e-4 if it < 25 else 1e-3
        for grp in opt.param_groups:
            grp["lr"] = lr
        g = (sign * (1 + 0.5 * rng.normal(size=n)) * mag * (0.15 if it % 3 else 0.4)).astype(np.float32)
        g[rng.random(n) < 0.01] = 0.0
        for q, k in zip(params, SEGMENTS):
            q.grad = torch.from_numpy(g[_lib.POLICY_LAYOUT[k]:_lib.POLICY_LAYOUT[k] + q.numel()].reshape(q.shape).copy())
        gh = g.copy()
        host_adam.step(p.ctypes.data, gh.ctypes.data, m.ctypes.data, v.ctypes.data, count.ctypes.data, lr, 0.9, 0.999, 1e-5,
                       0.0 if max_norm is None else max_norm, max_norm is not None)
        np_p, np_g, np_m, np_v, np_c, total = numpy_step(*np_state[:1], g.copy(), *np_state[1:3], np_state[3], lr, 0.9, 0.999,
                                                         1e-5, max_norm)
        np_state = (np_p, np_m, np_v, np_c)
        assert np.array_equal(p, np_p) and np.array_equal(gh, np_g) and np.array_equal(m, np_m) and np.array_equal(v, np_v)
        assert count[0] == np_c == it + 1
        if max_norm is not None:
            tn = torch.nn.utils.clip_grad_norm_(params, max_norm, foreach=False)
            clipped += float(tn) > max_norm
            assert abs(float(tn) - float(total)) <= 1e-6 * float(total)
        opt.step()
        for q, k in zip(params, SEGMENTS):
            o = _lib.POLICY_LAYOUT[k]
            _close(p[o:o + q.numel()], q.detach().numpy().ravel(), what=("param", k, it))
            _close(gh[o:o + q.numel()], q.grad.numpy().ravel(), what=("grad", k, it))
            st = opt.state[q]
            _close(m[o:o + q.numel()], st["exp_avg"].numpy().ravel(), what=("exp_avg", k, it))
            _close(v[o:o + q.numel()], st["exp_avg_sq"].numpy().ravel(), what=("exp_avg_sq", k, it))
            assert float(st["step"]) == count[0]
    if max_norm == 0.5:
        assert 0 < clipped < 50                                             # clipping both active and inactive
    elif max_norm == 1e4:
        assert clipped == 0


def test_adam_args_layout_and_constants(tmp_path):
    fields = [f for f, _ in _lib.StgAdamArgs._fields_]
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', 'int main(void){',
             'printf("size %zu\\n", sizeof(StgAdamArgs));']
    lines += [f'printf("{f} %zu\\n", offsetof(StgAdamArgs, {f}));' for f in fields]
    consts = dict(STG_ADAM_THREADS=_lib.ADAM_THREADS, STG_ADAM_TENSORS=_lib.ADAM_TENSORS, STG_ADAM_LOG=_lib.ADAM_LOG,
                  STG_ADAM_CLIP=_lib.ADAM_CLIP, STG_ADAM_TARGET_KL=_lib.ADAM_TARGET_KL, STG_ABI_VERSION=7)
    consts.update({f"STG_ADAM_LOG_{k}": v for k, v in _lib.ADAM_LOG_SLOTS.items()})
    lines += [f'printf("{c} %lld\\n", (long long)({c}));' for c in consts]
    lines.append('return 0;}')
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", str(src), "-o", str(exe)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split("\n") if l)
    assert int(got["size"]) == C.sizeof(_lib.StgAdamArgs)
    for f in fields:
        assert int(got[f]) == getattr(_lib.StgAdamArgs, f).offset, f
    for c, v in consts.items():
        assert int(got[c]) == v, c
    assert sorted(_lib.ADAM_LOG_SLOTS.values()) == list(range(_lib.ADAM_LOG))


def _adam_args(**over):
    B = 0x10000
    a = _lib.StgAdamArgs()
    for s in range(_lib.ADAM_TENSORS):
        a.d_param[s] = B * (s + 1)
    a.d_grad, a.d_exp_avg, a.d_exp_avg_sq, a.d_step = B * 20, B * 21, B * 22, B * 23
    for k, v in over.items():
        if k.startswith("d_param"):
            a.d_param[int(k[7:])] = v
        else:
            setattr(a, k, v)
    return a


def test_adam_argument_validation():
    f = _lib.load().stg_policy_adam_f32
    call = lambda **kw: f(C.byref(_adam_args(**kw)), None)                  # noqa: E731
    B = 0x10000
    assert f(None, None) == -1                                               # STG_E_NULL
    for k in ["d_param0", "d_param7", "d_param12", "d_grad", "d_exp_avg", "d_exp_avg_sq", "d_step"]:
        assert call(**{k: None}) == -1, k
    assert call(d_param3=None, d_grad=B * 20 + 2) == -1                      # pointers before alignment
    for k, off in (("d_param5", 2), ("d_grad", 1), ("d_exp_avg", 2), ("d_exp_avg_sq", 3), ("d_step", 2)):
        base = getattr(_adam_args(), "d_param")[int(k[7:])] if k.startswith("d_param") else getattr(_adam_args(), k)
        assert call(**{k: base + off}) == -4, k                              # STG_E_ALIGN
    assert call(d_losses=B + 2) == -4 and call(d_gate=B + 1) == -4 and call(d_log=B + 4) == -4
    assert call(d_log=B + 4, flags=4) == -4                                  # alignment before flags
    assert call(flags=4) == -3 and call(flags=0x7) == -3                     # STG_E_ENUM
    assert call(flags=2, d_losses=B, d_gate=None) == -1                      # a flag without its pointers
    assert call(flags=2, d_losses=None, d_gate=B) == -1
    assert call(flags=6, d_losses=None) == -3                                # unknown flags before the flag's pointers


def test_clipped_adam_python_errors():
    import torch
    import spin_torque_rl_gym_b200 as stg
    pol = _random_policy(FakeEnv(), 21)
    with pytest.raises(ValueError):
        stg.ClippedAdam(torch.nn.Linear(2, 2))
    opt = stg.ClippedAdam(pol)
    with pytest.raises(ValueError):
        opt.step()                                                           # no .grad at all
    for p in pol.parameters():
        p.grad = torch.zeros_like(p)
    pol.value_net.bias.grad = None
    with pytest.raises(ValueError):
        opt.step()                                                           # one .grad missing
    pol.value_net.bias.grad = torch.zeros_like(pol.value_net.bias)
    with pytest.raises(_lib.StgError):
        opt.step()                                                           # well-formed, but on the CPU
    for key, bad in (("weight_decay", 0.01), ("amsgrad", True), ("maximize", True), ("decoupled_weight_decay", True),
                     ("betas", (0.9, 1.0))):
        good = opt.param_groups[0][key]
        opt.param_groups[0][key] = bad                                       # settings K11 does not implement
        with pytest.raises(ValueError):
            opt.step()
        opt.param_groups[0][key] = good
        with pytest.raises(ValueError):
            opt.load_state_dict(torch.optim.Adam(pol.parameters(), **{key: bad}).state_dict())
    with pytest.raises(ValueError):
        opt.add_param_group({"params": [torch.nn.Parameter(torch.zeros(3))]})   # a foreign parameter
    foreign = stg.ClippedAdam(pol)
    foreign.param_groups[0]["params"][4] = torch.nn.Parameter(torch.zeros(64, 12))
    with pytest.raises(ValueError):
        foreign.step()
    # state dicts: torch.optim.Adam's format; unequal per-parameter steps do not load
    ref = torch.optim.Adam(pol.parameters(), lr=3e-4, eps=1e-5)
    sd = ref.state_dict()
    assert set(opt.state_dict()["param_groups"][0]) == set(sd["param_groups"][0]) | {"max_grad_norm"}
    sd = {"state": {i: {"step": torch.tensor(float(3 + (i == 5))), "exp_avg": torch.zeros_like(p),
                        "exp_avg_sq": torch.zeros_like(p)} for i, p in enumerate(pol.parameters())},
          "param_groups": sd["param_groups"]}
    with pytest.raises(ValueError):
        opt.load_state_dict(sd)
    sd["state"][5]["step"] = torch.tensor(3.0)
    opt.load_state_dict(sd)
    assert float(opt._step_count) == 3.0
    del sd["state"][2]
    with pytest.raises(ValueError):
        opt.load_state_dict(sd)                                              # a parameter without state has step 0


class StubEnv(FakeEnv):
    autoreset, host_outputs = True, False

    def stats_tensor(self):
        import torch
        return torch.zeros(_lib.NSTATS, dtype=torch.float64)


class StubCollector:
    """What PPO reads from RolloutCollector, on the CPU: cumulative statistics growing by a fixed amount per collect()."""

    def __init__(self, env, n_steps, store_values=True):
        import torch
        self.env, self.n_steps, self.k = env, n_steps, 0
        self.values, self.returns = torch.zeros(n_steps, env.num_envs), torch.ones(n_steps, env.num_envs)
        self.returns[0, 0] = 3.0

    def collect(self, policy):
        self.k += 1
        per = dict(steps=32, substeps=0, terminated=3, truncated=1, energy=0, reward=16, guard=0, episode_length=40)
        return {name: float(self.k * per[name]) for name in _lib.STAT_NAMES}

    def compute_returns_and_advantage(self, gamma, gae_lambda):
        pass

    def get(self, batch_size):
        return iter([None, None])


def test_ppo_schedules_and_progress_remaining(monkeypatch):
    import torch
    import spin_torque_rl_gym_b200 as stg
    from spin_torque_rl_gym_b200 import ppo as ppo_mod
    from spin_torque_rl_gym_b200.policy import PPOLosses
    monkeypatch.setattr(ppo_mod, "RolloutCollector", StubCollector)
    monkeypatch.setattr(stg.ClippedAdam, "_step", lambda self, *a, **k: None)
    env = StubEnv()
    pol = _random_policy(env, 22)
    monkeypatch.setattr(pol, "ppo_backward", lambda *a, **k: PPOLosses(*torch.zeros(6).unbind()))
    seen = {"lr": [], "cr": [], "vf": []}

    def rec(key, value):
        return lambda progress: seen[key].append(progress) or value

    model = stg.PPO(pol, env, learning_rate=rec("lr", 1e-3), n_steps=4, batch_size=8, n_epochs=2, clip_range=rec("cr", 0.1),
                    clip_range_vf=rec("vf", 0.3))
    assert model.rollout_buffer.n_steps == 4 and isinstance(pol.optimizer, stg.ClippedAdam)
    assert seen["lr"] == [1.0] and pol.optimizer.param_groups[0]["lr"] == 1e-3      # the optimiser starts at lr_schedule(1)
    assert model.learn(100) is model
    want = [1.0 - float(32 * k) / 100.0 for k in (1, 2, 3, 4)]                      # SB3: 1 - num_timesteps / total
    assert seen["lr"] == [1.0] + want and seen["cr"] == want and seen["vf"] == want
    model.learn(50, reset_num_timesteps=False)                                       # total counts from 128: 178
    want2 = [1.0 - float(t) / 178.0 for t in (160, 192)]
    assert seen["cr"] == want + want2
    logs = model.log_history
    assert len(logs) == 6 and [l["time/iterations"] for l in logs] == [1, 2, 3, 4, 1, 2]
    assert [l["train/n_updates"] for l in logs] == [2, 4, 6, 8, 10, 12]
    assert logs[-1]["time/total_timesteps"] == 192 and logs[0]["train/learning_rate"] == 1e-3
    assert logs[0]["train/clip_range"] == 0.1 and logs[0]["train/clip_range_vf"] == 0.3
    for l in logs:                                                                   # per rollout, not cumulative
        assert l["rollout/episodes"] == 4 and l["rollout/success_rate"] == 0.75
        assert l["rollout/mean_episode_length"] == 10 and l["rollout/mean_reward"] == 0.5
    y = model.rollout_buffer.returns.double().flatten()
    assert logs[0]["train/explained_variance"] == pytest.approx(1 - float(((y - 0).var(unbiased=False))) /
                                                                float(y.var(unbiased=False)))
    assert logs[0]["train/std"] == pytest.approx(float(pol.log_std.detach().exp().mean()))
    assert set(logs[0]) >= {f"train/{k}" for k in ("entropy_loss", "policy_gradient_loss", "value_loss", "approx_kl",
                                                     "clip_fraction", "loss", "explained_variance", "std")}
    assert "train/clip_range_vf" not in stg.PPO(pol, env, n_steps=4).train()


def test_ppo_argument_errors(monkeypatch):
    import torch
    import spin_torque_rl_gym_b200 as stg
    from spin_torque_rl_gym_b200 import ppo as ppo_mod
    monkeypatch.setattr(ppo_mod, "RolloutCollector", StubCollector)
    env = StubEnv()
    pol = _random_policy(env, 23)
    for kw in (dict(batch_size=1), dict(batch_size=0, normalize_advantage=False), dict(n_epochs=0), dict(n_steps=0)):
        with pytest.raises(ValueError):
            stg.PPO(pol, env, **kw)
    stg.PPO(pol, env, batch_size=1, normalize_advantage=False)
    for bad in ("CnnPolicy", torch.nn.Linear(12, 2)):
        with pytest.raises(ValueError):
            stg.PPO(bad, env)
    with pytest.raises(ValueError):
        stg.PPO(pol, StubEnv(n=16))                                                  # built for another env
    with pytest.raises(ValueError):
        stg.PPO(pol, env, policy_kwargs=dict(log_std_init=-1.0))
    with pytest.raises(ValueError):
        stg.PPO("MlpPolicy", env, policy_kwargs=dict(net_arch=[32, 32]))
    import torch.distributed as dist
    monkeypatch.setattr(dist, "is_initialized", lambda: True)
    monkeypatch.setattr(dist, "get_world_size", lambda group=None: 2)
    with pytest.raises(NotImplementedError):
        stg.PPO(pol, env)


# ---------------------------------------------------------------------------------------------------- GPU ---------------

def _collector(stg, dev, n, T, seed=5, log_std_init=-0.5):
    import torch
    env = _venv(stg, dev, n, seed=seed)
    torch.manual_seed(seed)
    pol = stg.ActorCriticPolicy(env, log_std_init=log_std_init)
    col = stg.RolloutCollector(env, n_steps=T, store_values=True)
    col.collect(pol)
    col.compute_returns_and_advantage(gamma=0.99, gae_lambda=0.95)
    return env, pol, col


def _compare_to_torch(pol, opt, ref, ropt, tol=1e-5):
    sd = opt.state_dict()
    for i, ((name, p), q) in enumerate(zip(pol.named_parameters(), ref.parameters())):
        _close(p.detach().cpu(), q.detach().cpu(), tol, name)
        _close(p.grad.cpu(), q.grad.cpu(), tol, name + ".grad")
        st = ropt.state[q]
        _close(sd["state"][i]["exp_avg"].cpu(), st["exp_avg"].cpu(), tol, name + ".exp_avg")
        _close(sd["state"][i]["exp_avg_sq"].cpu(), st["exp_avg_sq"].cpu(), tol, name + ".exp_avg_sq")
        assert float(sd["state"][i]["step"]) == float(st["step"])


def _torch_step(ref, ropt, grads, max_norm):
    for q, g in zip(ref.parameters(), grads):
        q.grad = g.clone()
    tn = None
    if max_norm is not None:
        tn = float(torch_clip(ref.parameters(), max_norm))
    ropt.step()
    return tn


def torch_clip(params, max_norm):
    import torch
    return torch.nn.utils.clip_grad_norm_(params, max_norm, foreach=False)


@pytest.fixture(scope="module")
def train_rollout(cuda_device):
    import spin_torque_rl_gym_b200 as stg
    env, pol, col = _collector(stg, cuda_device, 8192, 8)
    _perturb(pol, 1)
    return env, pol, col


@pytest.mark.gpu
@pytest.mark.parametrize("max_norm", [0.5, None])
def test_cuda_clipped_adam_matches_torch(train_rollout, max_norm):
    import torch
    import spin_torque_rl_gym_b200 as stg
    _, pol0, col = train_rollout
    pol = copy.deepcopy(pol0)
    ref = copy.deepcopy(pol0)
    opt = stg.ClippedAdam(pol, max_grad_norm=max_norm)
    ropt = torch.optim.Adam(ref.parameters(), lr=3e-4, eps=1e-5, foreach=False)
    batches = list(col.get(4096))
    clipped = 0
    for it in range(30):
        if it == 15:
            for g in opt.param_groups + ropt.param_groups:
                g["lr"] = 2e-3
        pol.ppo_backward(batches[it % len(batches)], clip_range_vf=0.2, ent_coef=0.01)
        if it % 3 == 2:
            pol._grad.mul_(100.0)                                # a larger gradient, so that clipping is active at 0.5
        tn = _torch_step(ref, ropt, [p.grad for p in pol.parameters()], max_norm)
        opt.step()
        clipped += tn is not None and tn > max_norm
        _compare_to_torch(pol, opt, ref, ropt)
    print(f"max_grad_norm={max_norm}: clipping active in {clipped} of 30 steps")
    if max_norm is not None:
        assert clipped > 0


@pytest.mark.gpu
def test_cuda_k11_bitwise_equal_to_host_core(train_rollout, host_adam):
    """The kernel against optim_core.cuh built with g++ on the same K10 gradients, bit for bit."""
    import torch
    import spin_torque_rl_gym_b200 as stg
    _, pol0, col = train_rollout
    pol = copy.deepcopy(pol0)
    opt = stg.ClippedAdam(pol, lr=1e-3)
    batches = list(col.get(8192))

    def flat(tensors):
        return torch.cat([t.detach().reshape(-1) for t in tensors]).cpu().numpy()
    slots = [p for p, _ in pol._grad_slots()]                    # the K10 layout, in offset order
    p = flat(slots)
    m, v, count = np.zeros_like(p), np.zeros_like(p), np.zeros(1, np.float32)
    for it in range(20):
        pol.ppo_backward(batches[it % len(batches)], clip_range_vf=0.2, ent_coef=0.01)
        if it % 3 == 2:
            pol._grad.mul_(100.0)                                # clipping active in some steps
        g = pol._grad.cpu().numpy().copy()
        opt.step()
        host_adam.step(p.ctypes.data, g.ctypes.data, m.ctypes.data, v.ctypes.data, count.ctypes.data, 1e-3, 0.9, 0.999, 1e-5,
                       0.5, 1)
        assert np.array_equal(flat(slots), p) and np.array_equal(pol._grad.cpu().numpy(), g), it
        assert np.array_equal(opt._exp_avg.cpu().numpy(), m) and np.array_equal(opt._exp_avg_sq.cpu().numpy(), v), it
        assert float(opt._step_count) == count[0] == it + 1


@pytest.mark.gpu
def test_cuda_state_dict_round_trip_with_torch_adam(train_rollout):
    import torch
    import spin_torque_rl_gym_b200 as stg
    _, pol0, col = train_rollout
    batches = list(col.get(8192))
    pol, ref = copy.deepcopy(pol0), copy.deepcopy(pol0)
    opt = stg.ClippedAdam(pol, lr=1e-3)
    ropt = torch.optim.Adam(ref.parameters(), lr=1e-3, eps=1e-5, foreach=False)
    for it in range(4):                                          # ClippedAdam's state -> torch.optim.Adam
        pol.ppo_backward(batches[it])
        opt.step()
    sd = opt.state_dict()
    tsd = ropt.state_dict()
    assert set(sd) == set(tsd) and set(sd["param_groups"][0]) == set(tsd["param_groups"][0]) | {"max_grad_norm"}
    assert all(set(s) == {"step", "exp_avg", "exp_avg_sq"} and s["step"].dtype == torch.float32 and s["step"].device.type ==
               "cpu" for s in sd["state"].values())
    with torch.no_grad():
        for p, q in zip(pol.parameters(), ref.parameters()):
            q.copy_(p)
    ropt.load_state_dict(sd)
    for it in range(5):
        pol.ppo_backward(batches[it % len(batches)])
        _torch_step(ref, ropt, [p.grad for p in pol.parameters()], 0.5)
        opt.step()
    _compare_to_torch(pol, opt, ref, ropt)
    # torch.optim.Adam's state -> a new ClippedAdam on a copy
    pol2 = copy.deepcopy(ref)
    opt2 = stg.ClippedAdam(pol2, lr=5.0)
    opt2.load_state_dict(ropt.state_dict())
    assert opt2.param_groups[0]["lr"] == 1e-3 and opt2.param_groups[0]["max_grad_norm"] == 0.5
    for it in range(5):
        pol2.ppo_backward(batches[it % len(batches)])
        _torch_step(ref, ropt, [p.grad for p in pol2.parameters()], 0.5)
        opt2.step()
    _compare_to_torch(pol2, opt2, ref, ropt)


@pytest.mark.gpu
def test_cuda_eager_gradients_through_the_staging_buffer(train_rollout):
    import torch
    import spin_torque_rl_gym_b200 as stg
    _, pol0, col = train_rollout
    b = next(iter(col.get(16384)))
    direct, staged, eager = (copy.deepcopy(pol0) for _ in range(3))
    opts = [stg.ClippedAdam(x, max_grad_norm=0.1) for x in (direct, staged, eager)]
    for it in range(3):
        direct.ppo_backward(b, ent_coef=0.01)
        for p, q in zip(direct.parameters(), staged.parameters()):
            q.grad = p.grad.clone()                              # K10's gradient, but in tensors of their own
        before = [q.grad for q in staged.parameters()]
        eager.zero_grad()
        sb3_ppo_loss(eager, *_fields(b), ent_coef=0.01)[0].backward()
        for o in opts:
            o.step()
        for (name, p), q, e in zip(direct.named_parameters(), staged.parameters(), eager.parameters()):
            assert torch.equal(p, q) and torch.equal(p.grad, q.grad), name      # the staging path is the same step
            _close(e.detach().cpu(), p.detach().cpu(), 1e-5, name)
            _close(e.grad.cpu(), p.grad.cpu(), 1e-5, name + ".grad")          # clipped values copied back
        assert all(q.grad is g for q, g in zip(staged.parameters(), before))


@pytest.mark.gpu
def test_cuda_adam_deterministic_and_no_host_sync(train_rollout):
    import torch
    import spin_torque_rl_gym_b200 as stg
    _, pol0, col = train_rollout
    batches = list(col.get(4096))
    pol = copy.deepcopy(pol0)
    opt = stg.ClippedAdam(pol)
    for b in batches[:3]:
        pol.ppo_backward(b)
        opt.step()
    pol.ppo_backward(batches[3])
    start = (copy.deepcopy(pol.state_dict()), pol._grad.clone(), opt._exp_avg.clone(), opt._exp_avg_sq.clone(),
             opt._step_count.clone())

    def restore(p, o):
        p.load_state_dict(start[0])
        p._grad.copy_(start[1])
        o._exp_avg.copy_(start[2]); o._exp_avg_sq.copy_(start[3]); o._step_count.copy_(start[4])

    def result(p, o):
        return torch.cat([x.detach().reshape(-1) for x in p.parameters()] + [p._grad, o._exp_avg, o._exp_avg_sq,
                                                                                o._step_count])
    opt.step()
    first = result(pol, opt).clone()
    restore(pol, opt)
    opt.step()
    assert torch.equal(first, result(pol, opt))
    other = copy.deepcopy(pol0)                                  # other addresses
    other_opt = stg.ClippedAdam(other)
    other.ppo_backward(batches[0])
    restore(other, other_opt)
    other_opt.step()
    assert torch.equal(first, result(other, other_opt))
    restore(pol, opt)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        opt.step()
    torch.cuda.current_stream().wait_stream(side)
    assert torch.equal(first, result(pol, opt))
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for b in batches:
            pol.ppo_backward(b)
            opt.step()
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert float(opt._step_count) == 4 + len(batches)


# ---- PPO.train() against SB3's train() written out ------------------------------------------------------------------------

def sb3_train(pol, epochs, lr, max_grad_norm=0.5, target_kl=None, **kw):
    """SB3's PPO.train() over the given minibatches (a list per epoch), literally, in torch: the logged dict and the
    approx_kl of every minibatch evaluated."""
    import torch
    opt = torch.optim.Adam(pol.parameters(), lr=lr, eps=1e-5, foreach=False)
    pg, vl, el, cf, kls = [], [], [], [], []
    n_updates, steps, continue_training = 0, 0, True
    for batches in epochs:
        approx_kl_divs = []
        for b in batches:
            loss, parts = sb3_ppo_loss(pol, *_fields(b), **kw)
            pg.append(float(parts[1])); vl.append(float(parts[2])); el.append(float(parts[3])); cf.append(float(parts[5]))
            approx_kl_divs.append(float(parts[4])); kls.append(float(parts[4]))
            last_loss = float(loss)
            if target_kl is not None and float(parts[4]) > 1.5 * target_kl:
                continue_training = False
                break
            opt.zero_grad()
            loss.backward()
            torch.nn.utils.clip_grad_norm_(pol.parameters(), max_grad_norm, foreach=False)
            opt.step()
            steps += 1
        n_updates += 1
        if not continue_training:
            break
    logs = {"train/entropy_loss": np.mean(el), "train/policy_gradient_loss": np.mean(pg), "train/value_loss": np.mean(vl),
            "train/approx_kl": np.mean(approx_kl_divs), "train/clip_fraction": np.mean(cf), "train/loss": last_loss,
            "train/std": float(pol.log_std.detach().exp().mean()), "train/n_updates": n_updates}
    return logs, kls, steps


def _explained_variance(col):
    y_pred, y_true = col.values.flatten().cpu().numpy(), col.returns.flatten().cpu().numpy()
    return float(1 - np.var(y_true - y_pred) / np.var(y_true))


def _ppo_after_collect(stg, dev, n_epochs, lr, **kw):
    """A PPO on 2048 envs with one rollout of 8 steps collected and GAE done, weights perturbed; the minibatches its train()
    will draw, per epoch (get() is re-wound, so train() draws the same permutations)."""
    env = _venv(stg, dev, 2048, seed=9)
    model = stg.PPO("MlpPolicy", env, learning_rate=lr, n_steps=8, batch_size=4096, n_epochs=n_epochs, seed=4,
                    policy_kwargs=dict(log_std_init=-0.5), **kw)
    col = model.rollout_buffer
    col.collect(model.policy)
    col.compute_returns_and_advantage(0.99, 0.95)
    e0 = col._epoch
    epochs = [list(col.get(4096)) for _ in range(n_epochs)]
    col._epoch = e0
    assert len(epochs[0]) == 4
    return model, epochs


@pytest.mark.gpu
def test_cuda_ppo_train_matches_sb3_train(cuda_device):
    import spin_torque_rl_gym_b200 as stg
    kw = dict(clip_range=0.2, clip_range_vf=0.2, ent_coef=0.01)
    model, epochs = _ppo_after_collect(stg, cuda_device, 3, 1e-3, **kw)
    ref = copy.deepcopy(model.policy)
    want, _, steps = sb3_train(ref, epochs, 1e-3, **kw)
    got = model.train()
    for (name, p), q in zip(model.policy.named_parameters(), ref.parameters()):
        _close(p.detach().cpu(), q.detach().cpu(), 1e-4, name)
    assert float(model.policy.optimizer._step_count) == steps == 12
    want["train/explained_variance"] = _explained_variance(model.rollout_buffer)
    for k, v in want.items():
        assert abs(got[k] - v) <= LOG_RTOL * abs(v) + LOG_ATOL, (k, got[k], v)
    assert got["train/clip_range"] == 0.2 and got["train/clip_range_vf"] == 0.2 and got["train/learning_rate"] == 1e-3
    assert 0.0 < got["train/clip_fraction"] and got["train/approx_kl"] > 0.0


@pytest.mark.gpu
def test_cuda_ppo_target_kl_gate(cuda_device):
    import torch
    import spin_torque_rl_gym_b200 as stg
    kw = dict(clip_range=0.2, ent_coef=0.01)
    lr, n_epochs = 1e-3, 6
    model, epochs = _ppo_after_collect(stg, cuda_device, n_epochs, lr, **kw)
    _, kls, _ = sb3_train(copy.deepcopy(model.policy), epochs, lr, **kw)
    per = len(epochs[0])
    # the first minibatch of epoch >= 1 whose approx_kl exceeds every earlier one: the reference trips there
    j = next((j for j in range(per, len(kls)) if kls[j] > max(kls[:j]) * 1.001), None)
    assert j is not None, kls
    target_kl = (max(kls[:j]) + kls[j]) / 2 / 1.5
    ref = copy.deepcopy(model.policy)
    want, kls_ref, steps = sb3_train(ref, epochs, lr, target_kl=target_kl, **kw)
    assert len(kls_ref) == j + 1 and steps == j and want["train/n_updates"] == j // per + 1
    model.target_kl = target_kl
    got = model.train()
    assert got["train/n_updates"] == want["train/n_updates"] and model._n_updates == j // per + 1
    assert float(model.policy.optimizer._step_count) == steps
    assert int(model._gate) == 0
    for k in ("train/approx_kl", "train/loss", "train/policy_gradient_loss", "train/clip_fraction"):
        assert abs(got[k] - want[k]) <= LOG_RTOL * abs(want[k]) + LOG_ATOL, (k, got[k], want[k])
    for (name, p), q in zip(model.policy.named_parameters(), ref.parameters()):
        _close(p.detach().cpu(), q.detach().cpu(), 1e-4, name)
    print(f"target_kl {target_kl:.3e}: tripped at minibatch {j % per} of epoch {j // per}")


@pytest.mark.gpu
def test_cuda_ppo_reproducible_from_the_seed(cuda_device):
    import torch
    import spin_torque_rl_gym_b200 as stg
    runs = []
    for _ in range(2):
        env = _venv(stg, cuda_device, 4096, seed=11)
        model = stg.PPO("MlpPolicy", env, n_steps=8, batch_size=8192, n_epochs=2, seed=3, clip_range_vf=0.3, ent_coef=0.01)
        model.learn(3 * 8 * 4096)
        opt = model.policy.optimizer
        runs.append(([p.detach().clone() for p in model.policy.parameters()], opt._exp_avg.clone(), opt._exp_avg_sq.clone(),
                     opt._step_count.clone(), copy.deepcopy(model.log_history)))
    a, b = runs
    assert all(torch.equal(x, y) for x, y in zip(a[0], b[0]))
    assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2]) and torch.equal(a[3], b[3])
    assert len(a[4]) == len(b[4]) == 3
    for la, lb in zip(a[4], b[4]):
        # the env's reward statistic is a float64 sum of per-step atomics, whose order varies between runs
        assert la.pop("rollout/mean_reward") == pytest.approx(lb.pop("rollout/mean_reward"), rel=1e-12)
        assert repr(la) == repr(lb)


@pytest.mark.gpu
def test_cuda_ppo_learn_syncs_twice_and_next_rollout_uses_new_weights(cuda_device):
    import torch
    import spin_torque_rl_gym_b200 as stg
    env = _venv(stg, cuda_device, 4096, seed=13)
    model = stg.PPO("MlpPolicy", env, n_steps=8, batch_size=4096, n_epochs=3, seed=1)
    model.learn(8 * 4096)                                       # the first iteration resets the env
    before = [p.detach().clone() for p in model.policy.parameters()]
    torch.cuda.synchronize()
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        torch.cuda.set_sync_debug_mode("warn")
        try:
            model.learn(8 * 4096, reset_num_timesteps=False)
        finally:
            torch.cuda.set_sync_debug_mode("default")
    syncs = [w for w in caught if "synchroniz" in str(w.message)]
    assert len(syncs) == 2, [str(w.message) for w in syncs]
    logs = model.log_history[-1]
    assert logs["time/total_timesteps"] == 2 * 8 * 4096 and logs["train/n_updates"] == 6
    assert all(k in logs for k in ("rollout/success_rate", "rollout/mean_episode_length", "rollout/mean_reward",
                                   "rollout/episodes"))
    assert any(not torch.equal(p, q) for p, q in zip(model.policy.parameters(), before))
    col = model.rollout_buffer
    col.collect(model.policy)
    with torch.no_grad():
        v, lp, _ = model.policy.evaluate_actions(col.observations[0], col.actions[0])
    assert float((v[:, 0] - col.values[0]).abs().max()) <= 1e-5
    assert float((lp - col.log_probs[0]).abs().max()) <= 1e-5
    actions, _ = model.predict(col.observations[0], deterministic=True)
    assert actions.shape == (4096, 2)


@pytest.mark.gpu
def test_cuda_ppo_rejects_env_the_collector_rejects(cuda_device):
    import spin_torque_rl_gym_b200 as stg
    env = stg.make("SpinTorque-v0", num_envs=64, device=cuda_device, autoreset=False)
    with pytest.raises(ValueError):
        stg.PPO("MlpPolicy", env)
