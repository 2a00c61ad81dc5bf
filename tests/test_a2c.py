"""K10's A2C instance (stg_policy_a2c_grad_f32 / stg_policy_a2c_sums_f32, ActorCriticPolicy.a2c_backward), K13
(stg_policy_rmsprop_f32, ClippedRMSprop) and stg.A2C.

The specification of the gradient is Stable-Baselines3's A2C.train() loss (`evaluate_actions`, `-(advantages *
log_prob).mean()`, `mse_loss(returns, values)`, the entropy loss) differentiated by torch autograd in float64; that of K13 is
`torch.nn.utils.clip_grad_norm_` followed by `torch.optim.RMSprop` (single-tensor update) with include/stg.h's roundings; that
of A2C is SB3's A2C.train() written out literally in torch."""
import copy
import ctypes as C
import json
import os
import subprocess
import sys
import warnings

import numpy as np
import pytest

from spin_torque_rl_gym_b200 import _lib
from tests.helpers import ROOT
from tests.test_actor_critic_policy import FakeEnv, _random_policy
from tests.test_ppo_grad import _p, _venv, check_grads, grads_by_name, host_ppo, synthetic_batch  # noqa: F401
from tests.test_ppo_train import LOG_RTOL, LOG_ATOL, SEGMENTS, SHAPES, StubEnv, _close, torch_clip

HEADER = os.path.join(ROOT, "include", "stg.h")
CSRC = os.path.join(ROOT, "spin_torque_rl_gym_b200", "csrc")
E_NULL, E_SIZE, E_ENUM, E_ALIGN = -1, -2, -3, -4
A2C_LOSS_NAMES = ("loss", "policy_loss", "value_loss", "entropy_loss")


# ---------------------------------------------------------------------------------------------------- SB3, restated -------

def sb3_a2c_loss(pol, obs, actions, advantages, returns, ent_coef=0.0, vf_coef=0.5, normalize_advantage=False):
    """A2C.train()'s loss of the rollout, as SB3 writes it, on `pol` (any dtype): (loss, [loss, policy_loss, value_loss,
    entropy_loss])."""
    import torch
    values, log_prob, entropy = pol.evaluate_actions(obs, actions)
    values = values.flatten()
    if normalize_advantage:
        advantages = (advantages - advantages.mean()) / (advantages.std() + 1e-8)
    policy_loss = -(advantages * log_prob).mean()
    value_loss = torch.nn.functional.mse_loss(returns, values)
    entropy_loss = -torch.mean(entropy)
    loss = policy_loss + ent_coef * entropy_loss + vf_coef * value_loss
    return loss, [loss, policy_loss, value_loss, entropy_loss]


def _a2c_fields(b):
    return (b.observations, b.actions, b.advantages, b.returns)


def reference_a2c_grads(pol, fields, **kw):
    """float64 autograd of sb3_a2c_loss on a double copy of `pol` with the float32 values: ({name: grad}, losses)."""
    ref = copy.deepcopy(pol).double()
    ref.extract_features = lambda obs: obs
    for p in ref.parameters():
        p.grad = None
    loss, parts = sb3_a2c_loss(ref, *(t.double() for t in fields), **kw)
    loss.backward()
    return {n: p.grad.detach() for n, p in ref.named_parameters()}, [float(v.detach()) for v in parts]


def check_a2c_losses(got, want, tol=1e-5):
    for name, g, w in zip(A2C_LOSS_NAMES, got, want):
        assert abs(float(g) - w) <= tol * max(1.0, abs(w)), (name, float(g), w)


# ---------------------------------------------------------------------------------------------------- host builds ---------

def _gxx(tmp_path_factory, name, code):
    d = tmp_path_factory.mktemp(name)
    src = d / f"{name}.cpp"
    src.write_text(code)
    so = d / f"{name}.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-I", CSRC, str(src), "-o", str(so)], check=True)
    return C.CDLL(str(so))


@pytest.fixture(scope="module")
def host_a2c(tmp_path_factory):
    """policy_core.cuh's pol_backward_row<kLossA2c> and the fold's scaling compiled for the host with g++."""
    lib = _gxx(tmp_path_factory, "a2c_host", r'''#include "policy_core.cuh"
using namespace stg;
extern "C" void a2c(const float* w, const float* obs, const float* act, const float* adv, const float* ret, int64_t n,
                    float ent_coef, float vf_coef, float* grad, float* losses) {
  const PolPpoCoef c{0.0f, 0.0f, 0.0f, 0.0f, false};
  static double g[STG_POLICY_PARAMS];
  double sums[4] = {0, 0, 0, 0};
  for (int p = 0; p < STG_POLICY_PARAMS; ++p) g[p] = 0.0;
  for (int64_t i = 0; i < n; ++i)
    pol_backward_row<kLossA2c>(w, obs + 12 * i, act + 2 * i, NAN, NAN, adv[i], ret[i], c, g, sums);
  for (int p = 0; p < STG_POLICY_PARAMS; ++p) grad[p] = pol_ppo_grad_value(p, g[p], n, ent_coef, vf_coef);
  pol_ppo_losses(sums, w, n, ent_coef, vf_coef, losses);
}
''')
    dp, i64, f32 = C.c_void_p, C.c_int64, C.c_float
    lib.a2c.argtypes = [dp] * 5 + [i64, f32, f32, dp, dp]
    return lib


def host_a2c_step(lib, ppo_lib, pol, fields, ent_coef=0.0, vf_coef=0.5, normalize_advantage=False):
    """The host core on float32 CPU planes (obs, act, adv, ret): ({name: grad}, the six losses)."""
    import torch
    from tests.test_actor_critic_policy import _packed_numpy
    w, _ = _packed_numpy(pol)
    obs, act, adv, ret = (np.ascontiguousarray(t.numpy(), np.float32) for t in fields)
    n = len(obs)
    if normalize_advantage and n > 1:
        a = torch.from_numpy(adv)
        stats = np.array([float(a.mean()), float(a.std())], np.float32)
        adv_n = np.empty_like(adv)
        ppo_lib.advantage(_p(adv), n, _p(stats), _p(adv_n))
        adv = adv_n
    grad, losses = np.empty(_lib.POLICY_PARAMS, np.float32), np.empty(6, np.float32)
    lib.a2c(_p(w), _p(obs), _p(act), _p(adv), _p(ret), n, ent_coef, vf_coef, _p(grad), _p(losses))
    return grads_by_name(pol, grad), losses


@pytest.fixture(scope="module")
def host_rmsprop(tmp_path_factory):
    """optim_core.cuh's K13 arithmetic compiled for the host with g++: the kernel's work on flat arrays, serially."""
    lib = _gxx(tmp_path_factory, "rmsprop_host", r'''#include "optim_core.cuh"
using namespace stg;
extern "C" double sumsq(const float* g) {
  static double part[kAdamThreads];
  for (int t = 0; t < kAdamThreads; ++t) part[t] = adam_norm_chain(g, STG_POLICY_PARAMS, t);
  return adam_norm_tree(part);
}
extern "C" void step(float* p, float* g, float* sq, float* count, double lr, double alpha, double eps, double max_norm,
                     int clip) {
  const float coef = clip ? adam_clip_coef(sumsq(g), max_norm) : 1.0f;
  *count = Pk<float>::add(*count, 1.0f);
  const RmspropCoef c = rmsprop_coef(lr, alpha, eps);
  for (int s = 0; s < STG_ADAM_TENSORS; ++s)
    for (int i = adam_offset(s); i < adam_offset(s + 1); ++i) {
      if (clip) g[i] = Pk<float>::mul(g[i], coef);
      p[i] = rmsprop_element(p[i], g[i], sq[i], c);
    }
}
''')
    dp, dd = C.c_void_p, C.c_double
    lib.sumsq.restype, lib.sumsq.argtypes = dd, [dp]
    lib.step.argtypes = [dp] * 4 + [dd] * 4 + [C.c_int]
    return lib


def numpy_rmsprop(p, g, sq, count, lr, alpha, eps, max_norm):
    """include/stg.h's K13 contract restated in NumPy (float32 arrays, every operation rounded): the new (p, g, sq, count)
    and the total norm."""
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
    sq = sq * f(alpha) + (f(1 - alpha) * g) * g
    avg = np.sqrt(sq) + f(eps)
    p = p - (f(lr) * g) / avg
    return p, g, sq, count, total


# ---------------------------------------------------------------------------------------------------- CPU ---------------

@pytest.mark.parametrize("kw", [dict(), dict(ent_coef=0.01), dict(normalize_advantage=True),
                                dict(normalize_advantage=True, ent_coef=0.01, vf_coef=0.25)])
def test_core_a2c_backward_matches_float64_autograd(host_ppo, host_a2c, kw):  # noqa: F811
    pol = _random_policy(FakeEnv(), 41)
    obs, act, _, _, adv, ret = synthetic_batch(host_ppo, pol, 3000, 7, zero_adv=0.1)
    adv[:100] = -adv[:100].abs()
    fields = (obs, act, adv, ret)
    assert float(adv.min()) < 0 < float(adv.max()) and int((adv == 0).sum()) > 0     # zero and negative advantages
    got, losses = host_a2c_step(host_a2c, host_ppo, pol, fields, **kw)
    want, want_losses = reference_a2c_grads(pol, fields, **kw)
    check_grads(got, want, tol=2e-5)
    check_a2c_losses(losses, want_losses)
    assert losses[4] == 0.0 and losses[5] == 0.0                                      # no kl, no clip fraction


def test_core_a2c_single_row_and_zero_advantages(host_ppo, host_a2c):  # noqa: F811
    import torch
    pol = _random_policy(FakeEnv(), 42)
    for seed in (1, 2, 3):
        obs, act, _, _, adv, ret = synthetic_batch(host_ppo, pol, 1, seed)              # B = 1: never normalised
        if seed == 2:
            adv = -adv.abs()
        for kw in (dict(), dict(ent_coef=0.01, normalize_advantage=True)):
            got, losses = host_a2c_step(host_a2c, host_ppo, pol, (obs, act, adv, ret), **kw)
            want, want_losses = reference_a2c_grads(pol, (obs, act, adv, ret), **{**kw, "normalize_advantage": False})
            check_grads(got, want)
            check_a2c_losses(losses, want_losses)
    # all advantages zero: the actor's gradient is zero and the policy loss -0.0 / 0.0
    obs, act, _, _, adv, ret = synthetic_batch(host_ppo, pol, 300, 4)
    adv = torch.zeros_like(adv)
    got, losses = host_a2c_step(host_a2c, host_ppo, pol, (obs, act, adv, ret))
    assert float(got["action_net.weight"].abs().max()) == 0.0 and float(got["log_std"].abs().max()) == 0.0
    assert losses[1] == 0.0
    want, _ = reference_a2c_grads(pol, (obs, act, adv, ret))
    check_grads({k: v for k, v in got.items() if k != "log_std"}, {k: v for k, v in want.items() if k != "log_std"})


@pytest.mark.parametrize("max_norm", [0.5, None, 1e4])
def test_rmsprop_core_matches_numpy_bitwise_and_torch_cpu(host_rmsprop, max_norm):
    import torch
    rng = np.random.default_rng(5)
    n = _lib.POLICY_PARAMS
    p = rng.normal(size=n).astype(np.float32)
    sq, count = np.zeros(n, np.float32), np.zeros(1, np.float32)
    np_state = (p.copy(), sq.copy(), np.float32(0))
    params = [torch.nn.Parameter(torch.from_numpy(p[_lib.POLICY_LAYOUT[k]:_lib.POLICY_LAYOUT[k] + int(np.prod(s))]
                                                  .reshape(s).copy())) for k, s in zip(SEGMENTS, SHAPES)]
    opt = torch.optim.RMSprop(params, lr=7e-4, alpha=0.99, eps=1e-5, foreach=False)
    clipped = 0
    sign, mag = rng.choice([-1.0, 1.0], size=n), rng.choice([1e-4, 0.01, 0.05], size=n)
    for it in range(50):
        lr = 7e-4 if it < 25 else 2e-3
        for grp in opt.param_groups:
            grp["lr"] = lr
        g = (sign * (1 + 0.5 * rng.normal(size=n)) * mag * (0.15 if it % 3 else 0.4)).astype(np.float32)
        g[rng.random(n) < 0.01] = 0.0
        for q, k in zip(params, SEGMENTS):
            q.grad = torch.from_numpy(g[_lib.POLICY_LAYOUT[k]:_lib.POLICY_LAYOUT[k] + q.numel()].reshape(q.shape).copy())
        gh = g.copy()
        host_rmsprop.step(p.ctypes.data, gh.ctypes.data, sq.ctypes.data, count.ctypes.data, lr, 0.99, 1e-5,
                          0.0 if max_norm is None else max_norm, max_norm is not None)
        np_p, np_g, np_sq, np_c, total = numpy_rmsprop(np_state[0], g.copy(), np_state[1], np_state[2], lr, 0.99, 1e-5,
                                                       max_norm)
        np_state = (np_p, np_sq, np_c)
        assert np.array_equal(p, np_p) and np.array_equal(gh, np_g) and np.array_equal(sq, np_sq), it
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
            _close(sq[o:o + q.numel()], st["square_avg"].numpy().ravel(), what=("square_avg", k, it))
            assert float(st["step"]) == count[0]
    if max_norm == 0.5:
        assert 0 < clipped < 50                                             # clipping both active and inactive
    elif max_norm == 1e4:
        assert clipped == 0


def test_rmsprop_args_layout_constants_and_signatures(tmp_path):
    fields = [f for f, _ in _lib.StgRmspropArgs._fields_]
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', 'int main(void){',
             'printf("size %zu\\n", sizeof(StgRmspropArgs));']
    lines += [f'printf("{f} %zu\\n", offsetof(StgRmspropArgs, {f}));' for f in fields]
    consts = dict(STG_RMSPROP_CLIP=_lib.RMSPROP_CLIP, STG_ADAM_TENSORS=_lib.ADAM_TENSORS, STG_ADAM_THREADS=_lib.ADAM_THREADS,
                  STG_ABI_VERSION=7)
    lines += [f'printf("{c} %lld\\n", (long long)({c}));' for c in consts]
    lines.append('return 0;}')
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", str(src), "-o", str(exe)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split("\n") if l)
    assert int(got["size"]) == C.sizeof(_lib.StgRmspropArgs)
    for f in fields:
        assert int(got[f]) == getattr(_lib.StgRmspropArgs, f).offset, f
    for c, v in consts.items():
        assert int(got[c]) == v, c
    types = tmp_path / "types.c"
    types.write_text("\n".join([
        f'#include "{HEADER}"',
        'int (*g)(const StgPpoArgs*, void*) = stg_policy_a2c_grad_f32;',
        'int (*s)(const StgPpoArgs*, double*, void*) = stg_policy_a2c_sums_f32;',
        'int (*r)(const StgRmspropArgs*, void*) = stg_policy_rmsprop_f32;']))
    subprocess.run(["gcc", "-fsyntax-only", "-Werror=incompatible-pointer-types", str(types)], check=True)
    for name, nargs in (("stg_policy_a2c_grad_f32", 2), ("stg_policy_a2c_sums_f32", 3), ("stg_policy_rmsprop_f32", 2)):
        assert len(_lib.SYMBOLS[name][1]) == nargs, name


def _ppo_args(**over):
    B = 0x10000
    a = _lib.StgPpoArgs()
    a.d_weights, a.d_obs, a.d_action = B, B * 2, B * 3
    a.d_advantage, a.d_return, a.d_work = B * 6, B * 7, B * 8
    a.d_grad, a.d_losses = B * 9, B * 10
    a.batch = 256
    for k, v in over.items():
        setattr(a, k, v)
    return a


def test_a2c_argument_errors_in_documented_order():
    lib = _lib.load()
    B = 0x10000
    for entry in ("grad", "sums"):
        if entry == "grad":
            f = lib.stg_policy_a2c_grad_f32
            call = lambda d_sums=None, **kw: f(C.byref(_ppo_args(**kw)), None)                      # noqa: E731
            assert f(None, None) == E_NULL
            req = ("d_weights", "d_obs", "d_action", "d_advantage", "d_return", "d_grad", "d_losses", "d_work")
        else:
            f = lib.stg_policy_a2c_sums_f32
            call = lambda d_sums=B * 11, **kw: f(C.byref(_ppo_args(**kw)), d_sums, None)           # noqa: E731
            assert f(None, B, None) == E_NULL
            assert call(d_sums=None) == E_NULL and call(d_sums=None, batch=0) == E_SIZE
            req = ("d_weights", "d_obs", "d_action", "d_advantage", "d_return", "d_work")
            assert call(d_grad=None, d_losses=None, flags=1) == E_ENUM            # d_grad and d_losses are not needed
            assert call(d_sums=B * 11 + 4) == E_ALIGN and call(d_sums=B * 11 + 4, flags=1) == E_ALIGN
        assert call(batch=0) == E_SIZE and call(batch=-1, d_obs=None) == E_SIZE   # size before pointers
        for k in req:
            assert call(**{k: None}) == E_NULL, (entry, k)
        assert call(d_obs=None, d_weights=B + 4) == E_NULL                       # pointers before alignment
        for k, off in (("d_weights", 8), ("d_obs", 4), ("d_action", 4), ("d_work", 4), ("d_advantage", 2),
                       ("d_return", 1), ("d_adv_stats", 2)):
            base = getattr(_ppo_args(), k) or B
            assert call(**{k: base + off}) == E_ALIGN, (entry, k)
        # the old planes are not read: NULL or misaligned is accepted (checked up to the flags, which come last)
        assert call(d_old_value=None, d_old_log_prob=None, flags=1) == E_ENUM
        assert call(d_old_value=B + 1, d_old_log_prob=B + 2, flags=1) == E_ENUM
        assert call(d_obs=B * 2 + 4, flags=1) == E_ALIGN                           # alignment before flags
        for flags in (_lib.PPO_CLIP_VF, 2, 0x80000000):
            assert call(flags=flags) == E_ENUM, (entry, flags)                    # A2C has no value clip
    r = lib.stg_policy_rmsprop_f32

    def rms(**over):
        a = _lib.StgRmspropArgs()
        for s in range(_lib.ADAM_TENSORS):
            a.d_param[s] = B * (s + 1)
        a.d_grad, a.d_square_avg, a.d_step = B * 20, B * 21, B * 22
        for k, v in over.items():
            if k.startswith("d_param"):
                a.d_param[int(k[7:])] = v
            else:
                setattr(a, k, v)
        return r(C.byref(a), None)
    assert r(None, None) == E_NULL
    for k in ("d_param0", "d_param6", "d_param12", "d_grad", "d_square_avg", "d_step"):
        assert rms(**{k: None}) == E_NULL, k
    assert rms(d_param2=None, d_grad=B * 20 + 2) == E_NULL                       # pointers before alignment
    for k, off in (("d_param5", 2), ("d_grad", 1), ("d_square_avg", 2), ("d_step", 3)):
        base = B * (int(k[7:]) + 1) if k.startswith("d_param") else {"d_grad": B * 20, "d_square_avg": B * 21,
                                                                       "d_step": B * 22}[k]
        assert rms(**{k: base + off}) == E_ALIGN, k
    assert rms(d_step=B * 22 + 2, flags=2) == E_ALIGN                            # alignment before flags
    assert rms(flags=2) == E_ENUM and rms(flags=3) == E_ENUM


def test_clipped_rmsprop_python_errors():
    import torch
    import spin_torque_rl_gym_b200 as stg
    pol = _random_policy(FakeEnv(), 43)
    with pytest.raises(ValueError):
        stg.ClippedRMSprop(torch.nn.Linear(2, 2))
    for kw in (dict(lr=-1e-3), dict(alpha=-0.1), dict(eps=-1e-8)):                # torch rejects these too
        with pytest.raises(ValueError):
            stg.ClippedRMSprop(pol, **kw)
        with pytest.raises(ValueError):
            torch.optim.RMSprop(pol.parameters(), **kw)
    opt = stg.ClippedRMSprop(pol)
    assert opt.param_groups[0]["lr"] == 7e-4 and opt.param_groups[0]["alpha"] == 0.99 and opt.param_groups[0]["eps"] == 1e-5
    with pytest.raises(ValueError):
        opt.step()                                                                # no .grad at all
    for p in pol.parameters():
        p.grad = torch.zeros_like(p)
    with pytest.raises(_lib.StgError):
        opt.step()                                                                # well-formed, but on the CPU
    for key, bad in (("momentum", 0.9), ("centered", True), ("weight_decay", 0.01), ("maximize", True), ("lr", -1.0)):
        good = opt.param_groups[0][key]
        opt.param_groups[0][key] = bad                                            # settings K13 does not implement
        with pytest.raises(ValueError):
            opt.step()
        opt.param_groups[0][key] = good
        if key != "lr":
            with pytest.raises(ValueError):
                opt.load_state_dict(torch.optim.RMSprop(pol.parameters(), **{key: bad}).state_dict())
    with pytest.raises(ValueError):
        opt.add_param_group({"params": [torch.nn.Parameter(torch.zeros(3))]})
    # state dicts: torch.optim.RMSprop's format, both ways
    ref = torch.optim.RMSprop(pol.parameters(), lr=7e-4, alpha=0.99, eps=1e-5)
    assert set(opt.state_dict()["param_groups"][0]) == set(ref.state_dict()["param_groups"][0]) | {"max_grad_norm"}
    sd = {"state": {i: {"step": torch.tensor(4.0), "square_avg": torch.full_like(p, 0.25)}
                    for i, p in enumerate(pol.parameters())}, "param_groups": ref.state_dict()["param_groups"]}
    opt.load_state_dict(sd)
    assert float(opt._step_count) == 4.0 and bool((opt._square_avg == 0.25).all())
    out = opt.state_dict()
    assert set(out["state"][3]) == {"step", "square_avg"} and out["param_groups"][0]["max_grad_norm"] == 0.5
    ref.load_state_dict(out)
    assert float(ref.state[next(iter(pol.parameters()))]["step"]) == 4.0
    sd["state"][5]["step"] = torch.tensor(5.0)
    with pytest.raises(ValueError):
        opt.load_state_dict(sd)                                                   # unequal steps
    sd["state"][5] = {"step": torch.tensor(4.0), "square_avg": torch.zeros(1), "momentum_buffer": torch.zeros(1)}
    with pytest.raises(ValueError):
        opt.load_state_dict(sd)                                                   # momentum state
    assert len(opt.state_tensors()) == 2


def test_a2c_backward_python_errors():
    import torch
    from spin_torque_rl_gym_b200.envs.sb3_vec_env import RolloutBufferSamples
    pol = _random_policy(FakeEnv(), 44)

    def samples(n=8, **over):
        t = dict(observations=torch.zeros(n, 12), actions=torch.zeros(n, 2), old_values=None, old_log_prob=None,
                 advantages=torch.zeros(n), returns=torch.zeros(n))
        t.update(over)
        return RolloutBufferSamples(**t)

    with pytest.raises(_lib.StgError):
        pol.a2c_backward(samples())                     # well-formed (the old planes are not needed), but on the CPU
    for bad in (samples(0), samples(observations=torch.zeros(8, 13)), samples(actions=torch.zeros(8, 3)),
                samples(returns=torch.zeros(7)), samples(advantages=torch.zeros(8, dtype=torch.float64)),
                samples(advantages=torch.zeros(8, 1)), samples(returns=np.zeros(8, np.float32))):
        with pytest.raises(ValueError):
            pol.a2c_backward(bad)


class StubCollector:
    """What A2C reads from RolloutCollector, on the CPU."""

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
        self.gae = (gamma, gae_lambda)

    def rollout_samples(self):
        return "rollout"


def test_a2c_defaults_log_keys_and_errors(monkeypatch):
    import torch
    import spin_torque_rl_gym_b200 as stg
    from spin_torque_rl_gym_b200 import a2c as a2c_mod
    from spin_torque_rl_gym_b200.policy import A2CLosses
    monkeypatch.setattr(a2c_mod, "RolloutCollector", StubCollector)
    monkeypatch.setattr(stg.ClippedRMSprop, "_step", lambda self: None)
    monkeypatch.setattr(stg.ClippedAdam, "_step", lambda self, *a, **k: None)
    env = StubEnv()
    pol = _random_policy(env, 45)
    seen = []
    monkeypatch.setattr(pol, "a2c_backward", lambda s, *a, **k: seen.append((s, a, k)) or
                        A2CLosses(*torch.tensor([0.5, 0.1, 0.2, -2.5]).unbind()))
    lrs = []
    model = stg.A2C(pol, env, learning_rate=lambda p: lrs.append(p) or 1e-3, ent_coef=0.01)
    opt = pol.optimizer
    assert isinstance(opt, stg.ClippedRMSprop) and model.n_steps == 5 and model.gae_lambda == 1.0
    assert opt.param_groups[0]["alpha"] == 0.99 and opt.param_groups[0]["eps"] == 1e-5
    assert opt.param_groups[0]["max_grad_norm"] == 0.5 and opt.param_groups[0]["lr"] == 1e-3
    assert model.learn(300) is model
    assert model.rollout_buffer.gae == (0.99, 1.0)
    assert lrs == [1.0] + [1.0 - 40 * k / 300 for k in range(1, 9)]                 # 5 steps x 8 envs per iteration
    assert seen[0] == ("rollout", (0.01, 0.5, False), {"data_parallel": False}) and len(seen) == 8
    logs = model.log_history
    assert [l["train/n_updates"] for l in logs] == list(range(1, 9)) and logs[-1]["time/total_timesteps"] == 320
    assert set(logs[0]) == {"train/n_updates", "train/explained_variance", "train/entropy_loss", "train/policy_loss",
                            "train/value_loss", "train/std", "train/learning_rate", "rollout/success_rate",
                            "rollout/mean_episode_length", "rollout/mean_reward", "rollout/episodes", "time/iterations",
                            "time/total_timesteps"}
    assert logs[0]["train/policy_loss"] == pytest.approx(0.1) and logs[0]["train/entropy_loss"] == -2.5
    assert logs[0]["rollout/episodes"] == 4 and logs[0]["train/learning_rate"] == 1e-3
    assert logs[0]["train/explained_variance"] == pytest.approx(0.0, abs=1e-12)  # values 0: 1 - Var(y) / Var(y)
    adam = stg.A2C(pol, env, use_rms_prop=False, max_grad_norm=0.3).policy.optimizer
    assert isinstance(adam, stg.ClippedAdam) and adam.param_groups[0]["eps"] == 1e-5
    assert adam.param_groups[0]["lr"] == 7e-4 and adam.param_groups[0]["max_grad_norm"] == 0.3
    assert stg.A2C(pol, env, rms_prop_eps=1e-3).policy.optimizer.param_groups[0]["eps"] == 1e-3
    with pytest.raises(ValueError):
        stg.A2C(pol, env, n_steps=0)
    for bad in ("CnnPolicy", torch.nn.Linear(12, 2)):
        with pytest.raises(ValueError):
            stg.A2C(bad, env)
    with pytest.raises(ValueError):
        stg.A2C(pol, StubEnv(n=16))
    with pytest.raises(ValueError):
        stg.A2C(pol, env, policy_kwargs=dict(log_std_init=-1.0))
    with pytest.raises(ValueError):
        stg.A2C(pol, env, rms_prop_eps=-1.0)


def test_a2c_data_parallel_argument_errors(monkeypatch):
    import torch.distributed as dist
    import spin_torque_rl_gym_b200 as stg
    from spin_torque_rl_gym_b200 import a2c as a2c_mod
    from spin_torque_rl_gym_b200.envs.vec_normalize import VecNormalize
    monkeypatch.setattr(a2c_mod, "RolloutCollector", StubCollector)
    env = StubEnv()
    pol = _random_policy(env, 46)
    monkeypatch.setattr(dist, "is_initialized", lambda: True)
    monkeypatch.setattr(dist, "get_world_size", lambda group=None: 2)
    with pytest.raises(NotImplementedError, match="data_parallel=True"):
        stg.A2C(pol, env)

    class Unsynced(VecNormalize):
        def __init__(self, venv):
            self.venv, self.sync = venv, False

    with pytest.raises(ValueError, match="VecNormalize"):
        stg.A2C(pol, Unsynced(env), data_parallel=True)


# ---------------------------------------------------------------------------------------------------- GPU ---------------

def _a2c_rollout(stg, dev, n, T, seed=5):
    """A collector with one fused A2C rollout (gae_lambda = 1) of a policy with perturbed weights."""
    import torch
    from tests.test_ppo_grad import _perturb
    env = _venv(stg, dev, n, seed=seed)
    torch.manual_seed(seed)
    pol = stg.ActorCriticPolicy(env, log_std_init=-0.5)
    col = stg.RolloutCollector(env, n_steps=T, store_values=True)
    col.collect(pol)
    col.compute_returns_and_advantage(gamma=0.99, gae_lambda=1.0)
    _perturb(pol, 1)
    return env, pol, col


def _grads(pol):
    return {n: p.grad.detach().clone() for n, p in pol.named_parameters()}


@pytest.fixture(scope="module")
def big_a2c_rollout(cuda_device):
    """SB3's A2C default n_steps = 5 over 1,048,576 VecNormalize'd envs: 5,242,880 rows."""
    import spin_torque_rl_gym_b200 as stg
    return _a2c_rollout(stg, cuda_device, 1 << 20, 5)


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 4096, 1048576, "rollout"])
def test_cuda_a2c_gradient_matches_float64_autograd(big_a2c_rollout, B):
    import torch
    from spin_torque_rl_gym_b200.envs.sb3_vec_env import RolloutBufferSamples
    _, pol, col = big_a2c_rollout
    whole = col.rollout_samples()
    assert whole.observations.data_ptr() == col.observations.data_ptr() and whole.returns.shape == (5 << 20,)
    if B == "rollout":
        batch = whole
    else:
        idx = torch.randperm(5 << 20, generator=torch.Generator().manual_seed(B))[:B].to(whole.observations.device)
        batch = RolloutBufferSamples(*(t[idx] for t in whole))
    for kw in (dict(ent_coef=0.01), dict(normalize_advantage=True, vf_coef=0.25)):
        losses = pol.a2c_backward(batch, **kw)
        got = _grads(pol)
        want, want_losses = reference_a2c_grads(pol, _a2c_fields(batch),
                                                **{**kw, "normalize_advantage": kw.get("normalize_advantage", False)
                                                   and B != 1})
        worst = check_grads(got, want)
        check_a2c_losses(losses, want_losses)
        print(f"B={B} {sorted(kw.items())}: A2C max rel err {worst:.2e}")
        del want


@pytest.fixture(scope="module")
def a2c_rollout(cuda_device):
    import spin_torque_rl_gym_b200 as stg
    return _a2c_rollout(stg, cuda_device, 16384, 5)


@pytest.mark.gpu
def test_cuda_a2c_deterministic_and_no_host_sync(a2c_rollout):
    import torch
    from spin_torque_rl_gym_b200.envs.sb3_vec_env import RolloutBufferSamples
    _, pol, col = a2c_rollout
    batch = col.rollout_samples()
    kw = dict(ent_coef=0.01, normalize_advantage=True)
    l1 = torch.stack(pol.a2c_backward(batch, **kw)).clone()
    g1 = pol._grad.clone()
    assert torch.equal(torch.stack(pol.a2c_backward(batch, **kw)), l1) and torch.equal(g1, pol._grad)
    moved = RolloutBufferSamples(*(torch.cat([torch.zeros(1, *t.shape[1:], device=t.device), t])[1:] for t in batch))
    pol.a2c_backward(moved, **kw)                        # other addresses, misaligned (copied inside)
    assert torch.equal(g1, pol._grad)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        l3 = torch.stack(pol.a2c_backward(batch, **kw))
    torch.cuda.current_stream().wait_stream(side)
    assert torch.equal(g1, pol._grad) and torch.equal(l1, l3)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        pol.a2c_backward(batch, **kw, data_parallel=True)  # K12's FP64-moment statistics: last bits differ from torch's
        pol.a2c_backward(batch, **kw)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert torch.equal(g1, pol._grad)
    for p, off in pol._grad_slots():
        assert p.grad.data_ptr() == pol._grad.data_ptr() + 4 * off


@pytest.mark.gpu
def test_cuda_a2c_sums_then_finish(a2c_rollout):
    import torch
    from spin_torque_rl_gym_b200.envs.sb3_vec_env import RolloutBufferSamples
    _, pol, col = a2c_rollout
    b = col.rollout_samples()
    n = b.observations.shape[0]
    for n_rows in (1, 127, 4096, n):
        part = RolloutBufferSamples(*(t[:n_rows] for t in b))
        want_l = torch.stack(pol.a2c_backward(part, ent_coef=0.01, vf_coef=0.5)).cpu()
        want = pol._grad.clone()
        pol._grad.fill_(float("nan"))
        sums = pol._ppo_sums(part, None, ent_coef=0.01, vf_coef=0.5, loss="a2c")
        got_l = pol._ppo_finish(sums[None], 0.01, 0.5)
        assert torch.equal(pol._grad.view(torch.int32), want.view(torch.int32)), n_rows
        assert torch.equal(torch.stack(got_l[:4]).cpu().view(torch.int32), want_l.view(torch.int32)), n_rows
        assert float(got_l[4]) == 0.0 and float(got_l[5]) == 0.0
        assert float(sums[_lib.PPO_PART_COUNT]) == n_rows
    stats = torch.stack([b.advantages.mean(), b.advantages.std()])
    whole = pol._ppo_finish(pol._ppo_sums(b, stats, ent_coef=0.01, loss="a2c")[None], 0.01, 0.5)
    want, want_l = pol._grad.clone(), torch.stack(whole).cpu()
    for G in (2, 8):
        cuts = [n * r // G for r in range(G + 1)]
        assert all(c % _lib.PPO_TILE == 0 for c in cuts)
        sums = torch.stack([pol._ppo_sums(RolloutBufferSamples(*(t[lo:hi] for t in b)), stats, ent_coef=0.01, loss="a2c")
                            for lo, hi in zip(cuts, cuts[1:])])
        got_l = torch.stack(pol._ppo_finish(sums, 0.01, 0.5)).cpu()
        for p, off in pol._grad_slots():
            _close(pol._grad[off:off + p.numel()].cpu(), want[off:off + p.numel()].cpu(), 1e-6, f"G={G} offset {off}")
        assert float((got_l - want_l).abs().max()) <= 1e-6 * max(1.0, float(want_l.abs().max()))


def _torch_rmsprop_step(ref, ropt, grads, max_norm):
    for q, g in zip(ref.parameters(), grads):
        q.grad = g.clone()
    tn = None if max_norm is None else float(torch_clip(ref.parameters(), max_norm))
    ropt.step()
    return tn


def _compare_rmsprop(pol, opt, ref, ropt, tol=1e-5):
    sd = opt.state_dict()
    for i, ((name, p), q) in enumerate(zip(pol.named_parameters(), ref.parameters())):
        _close(p.detach().cpu(), q.detach().cpu(), tol, name)
        _close(p.grad.cpu(), q.grad.cpu(), tol, name + ".grad")
        _close(sd["state"][i]["square_avg"].cpu(), ropt.state[q]["square_avg"].cpu(), tol, name + ".square_avg")
        assert float(sd["state"][i]["step"]) == float(ropt.state[q]["step"])


def _chunks(col, k=4):
    from spin_torque_rl_gym_b200.envs.sb3_vec_env import RolloutBufferSamples
    b = col.rollout_samples()
    n = b.observations.shape[0]
    return [RolloutBufferSamples(*(t[n * i // k:n * (i + 1) // k] for t in b)) for i in range(k)]


@pytest.mark.gpu
def test_cuda_rmsprop_bitwise_equal_to_host_core(a2c_rollout, host_rmsprop):
    import torch
    import spin_torque_rl_gym_b200 as stg
    _, pol0, col = a2c_rollout
    pol = copy.deepcopy(pol0)
    opt = stg.ClippedRMSprop(pol, lr=1e-3)
    parts = _chunks(col)
    slots = [p for p, _ in pol._grad_slots()]
    flat = lambda ts: torch.cat([t.detach().reshape(-1) for t in ts]).cpu().numpy()   # noqa: E731
    p, sq, count = flat(slots), np.zeros(_lib.POLICY_PARAMS, np.float32), np.zeros(1, np.float32)
    for it in range(20):
        pol.a2c_backward(parts[it % len(parts)], ent_coef=0.01)
        if it % 3 == 2:
            pol._grad.mul_(100.0)                                  # clipping active in some steps
        g = pol._grad.cpu().numpy().copy()
        opt.step()
        host_rmsprop.step(p.ctypes.data, g.ctypes.data, sq.ctypes.data, count.ctypes.data, 1e-3, 0.99, 1e-5, 0.5, 1)
        assert np.array_equal(flat(slots), p) and np.array_equal(pol._grad.cpu().numpy(), g), it
        assert np.array_equal(opt._square_avg.cpu().numpy(), sq) and float(opt._step_count) == count[0] == it + 1


@pytest.mark.gpu
@pytest.mark.parametrize("max_norm", [0.5, None])
def test_cuda_rmsprop_matches_torch(a2c_rollout, max_norm):
    import torch
    import spin_torque_rl_gym_b200 as stg
    _, pol0, col = a2c_rollout
    pol, ref = copy.deepcopy(pol0), copy.deepcopy(pol0)
    opt = stg.ClippedRMSprop(pol, max_grad_norm=max_norm)
    ropt = torch.optim.RMSprop(ref.parameters(), lr=7e-4, alpha=0.99, eps=1e-5, foreach=False)
    parts = _chunks(col)
    clipped = 0
    for it in range(30):
        if it == 15:
            for g in opt.param_groups + ropt.param_groups:
                g["lr"] = 2e-3
        pol.a2c_backward(parts[it % len(parts)], ent_coef=0.01)
        if it % 3 == 2:
            pol._grad.mul_(100.0)
        tn = _torch_rmsprop_step(ref, ropt, [p.grad for p in pol.parameters()], max_norm)
        opt.step()
        clipped += tn is not None and tn > max_norm
        _compare_rmsprop(pol, opt, ref, ropt)
    if max_norm is not None:
        assert 0 < clipped < 30


@pytest.mark.gpu
def test_cuda_rmsprop_state_dict_round_trip_and_staging(a2c_rollout):
    import torch
    import spin_torque_rl_gym_b200 as stg
    _, pol0, col = a2c_rollout
    parts = _chunks(col)
    pol, ref = copy.deepcopy(pol0), copy.deepcopy(pol0)
    opt = stg.ClippedRMSprop(pol, lr=1e-3)
    ropt = torch.optim.RMSprop(ref.parameters(), lr=1e-3, alpha=0.99, eps=1e-5, foreach=False)
    for it in range(3):                                            # ClippedRMSprop's state -> torch.optim.RMSprop
        pol.a2c_backward(parts[it])
        opt.step()
    with torch.no_grad():
        for p, q in zip(pol.parameters(), ref.parameters()):
            q.copy_(p)
    ropt.load_state_dict(opt.state_dict())
    for it in range(4):
        pol.a2c_backward(parts[it % 4])
        _torch_rmsprop_step(ref, ropt, [p.grad for p in pol.parameters()], 0.5)
        opt.step()
    _compare_rmsprop(pol, opt, ref, ropt)
    pol2 = copy.deepcopy(ref)                                      # torch.optim.RMSprop's state -> a new ClippedRMSprop
    opt2 = stg.ClippedRMSprop(pol2, lr=5.0)
    opt2.load_state_dict(ropt.state_dict())
    assert opt2.param_groups[0]["lr"] == 1e-3 and opt2.param_groups[0]["max_grad_norm"] == 0.5
    for it in range(4):
        pol2.a2c_backward(parts[it % 4])
        _torch_rmsprop_step(ref, ropt, [p.grad for p in pol2.parameters()], 0.5)
        opt2.step()
    _compare_rmsprop(pol2, opt2, ref, ropt)
    # eager .grad tensors go through the staging buffer and take the same step
    direct, staged = copy.deepcopy(pol0), copy.deepcopy(pol0)
    opts = [stg.ClippedRMSprop(x, max_grad_norm=0.1) for x in (direct, staged)]
    for it in range(3):
        direct.a2c_backward(parts[it], ent_coef=0.01)
        for p, q in zip(direct.parameters(), staged.parameters()):
            q.grad = p.grad.clone()
        before = [q.grad for q in staged.parameters()]
        for o in opts:
            o.step()
        for (name, p), q in zip(direct.named_parameters(), staged.parameters()):
            assert torch.equal(p, q) and torch.equal(p.grad, q.grad), name
        assert all(q.grad is g for q, g in zip(staged.parameters(), before))
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        direct.a2c_backward(parts[0])
        opts[0].step()
    finally:
        torch.cuda.set_sync_debug_mode("default")


# ---- A2C.train() against SB3's train() written out ------------------------------------------------------------------------

def sb3_a2c_train(pol, samples, lr, use_rms_prop, rms_prop_eps=1e-5, max_grad_norm=0.5, **kw):
    """SB3's A2C.train() over the rollout, literally, in torch: the logged losses."""
    import torch
    if use_rms_prop:
        opt = torch.optim.RMSprop(pol.parameters(), lr=lr, alpha=0.99, eps=rms_prop_eps, weight_decay=0, foreach=False)
    else:
        opt = torch.optim.Adam(pol.parameters(), lr=lr, eps=1e-5, foreach=False)
    return opt, _sb3_a2c_update(pol, opt, samples, max_grad_norm, **kw)


def _sb3_a2c_update(pol, opt, samples, max_grad_norm=0.5, **kw):
    import torch
    loss, parts = sb3_a2c_loss(pol, *_a2c_fields(samples), **kw)
    opt.zero_grad()
    loss.backward()
    torch.nn.utils.clip_grad_norm_(pol.parameters(), max_grad_norm, foreach=False)
    opt.step()
    return {"train/entropy_loss": float(parts[3]), "train/policy_loss": float(parts[1]),
            "train/value_loss": float(parts[2]), "train/std": float(pol.log_std.detach().exp().mean())}


@pytest.mark.gpu
@pytest.mark.parametrize("use_rms_prop", [True, False])
def test_cuda_a2c_train_matches_sb3_train(cuda_device, use_rms_prop):
    import spin_torque_rl_gym_b200 as stg
    from tests.test_ppo_train import _explained_variance
    env = _venv(stg, cuda_device, 4096, seed=9)
    kw = dict(ent_coef=0.01, normalize_advantage=use_rms_prop)
    model = stg.A2C("MlpPolicy", env, n_steps=5, seed=4, use_rms_prop=use_rms_prop, policy_kwargs=dict(log_std_init=-0.5),
                    **kw)
    ref, opt = copy.deepcopy(model.policy), None
    col = model.rollout_buffer
    for it in range(3):
        col.collect(model.policy)
        col.compute_returns_and_advantage(0.99, 1.0)
        samples = next(iter(col.get(None)))                 # SB3's batch: a permutation of the rollout
        if opt is None:
            opt, want = sb3_a2c_train(ref, samples, 7e-4, use_rms_prop, **kw)
        else:
            want = _sb3_a2c_update(ref, opt, samples, **kw)
        got = model.train()
        for (name, p), q in zip(model.policy.named_parameters(), ref.parameters()):
            _close(p.detach().cpu(), q.detach().cpu(), 1e-4, (it, name))
        want["train/explained_variance"] = _explained_variance(col)
        for k, v in want.items():
            assert abs(got[k] - v) <= LOG_RTOL * abs(v) + LOG_ATOL, (it, k, got[k], v)
        assert got["train/n_updates"] == it + 1 and got["train/learning_rate"] == 7e-4
    assert float(model.policy.optimizer._step_count) == 3


@pytest.mark.gpu
def test_cuda_a2c_reproducible_from_the_seed(cuda_device):
    import torch
    import spin_torque_rl_gym_b200 as stg
    runs = []
    for _ in range(2):
        env = _venv(stg, cuda_device, 4096, seed=11)
        model = stg.A2C("MlpPolicy", env, seed=3, ent_coef=0.01, normalize_advantage=True)
        model.learn(4 * 5 * 4096)
        opt = model.policy.optimizer
        runs.append(([p.detach().clone() for p in model.policy.parameters()], opt._square_avg.clone(),
                     opt._step_count.clone(), copy.deepcopy(model.log_history)))
    a, b = runs
    assert all(torch.equal(x, y) for x, y in zip(a[0], b[0]))
    assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2]) and len(a[3]) == len(b[3]) == 4
    for la, lb in zip(a[3], b[3]):
        assert la.pop("rollout/mean_reward") == pytest.approx(lb.pop("rollout/mean_reward"), rel=1e-12)
        assert repr(la) == repr(lb)


@pytest.mark.gpu
def test_cuda_a2c_learn_syncs_twice_and_next_rollout_uses_new_weights(cuda_device):
    import torch
    import spin_torque_rl_gym_b200 as stg
    env = _venv(stg, cuda_device, 4096, seed=13)
    model = stg.A2C("MlpPolicy", env, seed=1)
    model.learn(5 * 4096)                                   # the first iteration resets the env
    before = [p.detach().clone() for p in model.policy.parameters()]
    torch.cuda.synchronize()
    with warnings.catch_warnings(record=True) as caught:
        warnings.simplefilter("always")
        torch.cuda.set_sync_debug_mode("warn")
        try:
            model.learn(5 * 4096, reset_num_timesteps=False)
        finally:
            torch.cuda.set_sync_debug_mode("default")
    syncs = [w for w in caught if "synchroniz" in str(w.message)]
    assert len(syncs) == 2, [str(w.message) for w in syncs]
    logs = model.log_history[-1]
    assert logs["time/total_timesteps"] == 2 * 5 * 4096 and logs["train/n_updates"] == 2
    assert any(not torch.equal(p, q) for p, q in zip(model.policy.parameters(), before))
    col = model.rollout_buffer
    col.collect(model.policy)
    with torch.no_grad():
        v, lp, _ = model.policy.evaluate_actions(col.observations[0], col.actions[0])
    assert float((v[:, 0] - col.values[0]).abs().max()) <= 1e-5
    assert float((lp - col.log_probs[0]).abs().max()) <= 1e-5
    assert model.predict(col.observations[0], deterministic=True)[0].shape == (4096, 2)


WORKER = r'''
import os, sys
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

def save(name, model):
    opt = model.policy.optimizer
    torch.save({"state": {k: v.cpu() for k, v in model.policy.state_dict().items()}, "log": model.log_history,
                "opt": [t.cpu() for t in opt.state_tensors()]}, os.path.join(out, f"{name}_{rank}.pt"))

torch.manual_seed(100 + rank)                       # different initial weights unless broadcast
m = stg.A2C("MlpPolicy", env(), seed=3, ent_coef=0.01, data_parallel=True)
m.learn(3 * 5 * N * world)
save("a", m)
m = stg.A2C("MlpPolicy", stg.VecNormalize(env(), sync=None), seed=5, use_rms_prop=False, normalize_advantage=True,
            data_parallel=True)
m.learn(3 * 5 * N * world)
save("b", m)
torch.cuda.synchronize()
dist.destroy_process_group()
print("DONE", rank)
'''


def _run_ranks(tmp_path, backend, port):
    script = tmp_path / "a2c_dp_worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", str(port), str(script), ROOT, str(tmp_path), backend]
    res = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=900)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-5000:]
    import torch
    return {k: [torch.load(tmp_path / f"{k}_{r}.pt", weights_only=False) for r in range(2)] for k in "ab"}


def _check_ranks(got):
    import torch
    for name, run in got.items():
        s0, s1 = run[0]["state"], run[1]["state"]
        assert all(torch.equal(s0[k].view(torch.int32), s1[k].view(torch.int32)) for k in s0), name
        assert all(torch.equal(x.view(torch.int32), y.view(torch.int32)) for x, y in zip(run[0]["opt"], run[1]["opt"])), name
        assert json.dumps(run[0]["log"]) == json.dumps(run[1]["log"]), name          # every value, bit for bit
        assert len(run[0]["log"]) == 3 and run[0]["log"][-1]["time/total_timesteps"] == 3 * 5 * 4096 * 2
        assert float(run[0]["opt"][-1]) == 3.0


@pytest.mark.gpu
def test_cuda_a2c_two_ranks_gloo_train_one_policy(cuda_device, tmp_path):
    _check_ranks(_run_ranks(tmp_path, "gloo", 29561))


@pytest.mark.gpu
def test_cuda_a2c_two_ranks_nccl_train_one_policy(cuda_device, tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("NCCL needs one GPU per rank; fewer than 2 GPUs are visible")
    _check_ranks(_run_ranks(tmp_path, "nccl", 29563))
