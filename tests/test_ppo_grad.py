"""K10: SB3's PPO loss and its gradient through the MlpPolicy (stg_policy_ppo_grad_f32, ActorCriticPolicy.ppo_backward).

The specification is Stable-Baselines3's PPO.train() for one minibatch: `evaluate_actions`, the clipped surrogate, the
(optionally clipped) value loss and the entropy loss, differentiated by torch autograd. The reference here is that loss
written literally and run in float64 on a copy of the module cast to double, with the same float32 inputs."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from spin_torque_rl_gym_b200 import _lib
from tests.helpers import ROOT
from tests.test_actor_critic_policy import FakeEnv, _random_policy, _packed_numpy

HEADER = os.path.join(ROOT, "include", "stg.h")
CSRC = os.path.join(ROOT, "spin_torque_rl_gym_b200", "csrc")
LOSS_NAMES = ("loss", "policy_loss", "value_loss", "entropy_loss", "approx_kl", "clip_fraction")


# ---------------------------------------------------------------------------------------------------- SB3, restated -------

def sb3_ppo_loss(pol, obs, actions, old_values, old_log_prob, advantages, returns, clip_range=0.2, clip_range_vf=None,
                 ent_coef=0.0, vf_coef=0.5, normalize_advantage=True):
    """PPO.train()'s loss of one minibatch, as SB3 writes it, on `pol` (any dtype): (loss, [the six PPOLosses values])."""
    import torch
    values, log_prob, entropy = pol.evaluate_actions(obs, actions)
    values = values.flatten()
    if normalize_advantage and len(advantages) > 1:
        advantages = (advantages - advantages.mean()) / (advantages.std() + 1e-8)
    ratio = torch.exp(log_prob - old_log_prob)
    policy_loss_1 = advantages * ratio
    policy_loss_2 = advantages * torch.clamp(ratio, 1 - clip_range, 1 + clip_range)
    policy_loss = -torch.min(policy_loss_1, policy_loss_2).mean()
    clip_fraction = torch.mean((torch.abs(ratio - 1) > clip_range).float())
    if clip_range_vf is None:
        values_pred = values
    else:
        values_pred = old_values + torch.clamp(values - old_values, -clip_range_vf, clip_range_vf)
    value_loss = torch.nn.functional.mse_loss(returns, values_pred)
    entropy_loss = -torch.mean(entropy)
    loss = policy_loss + ent_coef * entropy_loss + vf_coef * value_loss
    with torch.no_grad():
        log_ratio = log_prob - old_log_prob
        approx_kl = torch.mean((torch.exp(log_ratio) - 1) - log_ratio)
    return loss, [loss, policy_loss, value_loss, entropy_loss, approx_kl, clip_fraction]


def reference_grads(pol, batch, **kw):
    """float64 autograd of sb3_ppo_loss on a double copy of `pol` with the batch's float32 values: ({name: grad}, losses)."""
    import copy
    import torch
    ref = copy.deepcopy(pol).double()
    ref.extract_features = lambda obs: obs                 # SB3's float cast of the observations would undo the double copy
    for p in ref.parameters():
        p.grad = None
    loss, parts = sb3_ppo_loss(ref, *(t.double() for t in batch), **kw)
    loss.backward()
    return {n: p.grad.detach() for n, p in ref.named_parameters()}, [float(v.detach()) for v in parts]


def check_grads(got, want, tol=1e-4):
    """max |g - g64| <= tol * max |g64| for every parameter tensor; returns the worst ratio."""
    worst = 0.0
    for name, g64 in want.items():
        scale = float(g64.abs().max())
        err = float((got[name].double().to(g64.device) - g64).abs().max())
        assert err <= tol * scale, (name, err, scale)
        worst = max(worst, err / scale if scale > 0 else 0.0)
    return worst


def check_losses(got, want, tol=1e-5):
    for name, g, w in zip(LOSS_NAMES, got, want):
        assert abs(float(g) - w) <= tol * max(1.0, abs(w)), (name, float(g), w)


# ---------------------------------------------------------------------------------------------------- host build ----------

@pytest.fixture(scope="module")
def host_ppo(tmp_path_factory):
    """policy_core.cuh's K10 per-row arithmetic compiled for the host with g++."""
    d = tmp_path_factory.mktemp("ppo_host")
    src = d / "ppo_host.cpp"
    src.write_text(r'''#include "policy_core.cuh"
using namespace stg;
extern "C" void eval(const float* w, const float* obs, const float* act, int64_t n, float* value, float* logp) {
  for (int64_t i = 0; i < n; ++i) {
    float h1[64], h2[64];
    const float* x = obs + 12 * i;
    for (int o = 0; o < 64; ++o) h1[o] = tanhf(pol_dot(x, 12, w + STG_POLICY_VF_W1, 64, o, w[STG_POLICY_VF_B1 + o]));
    for (int o = 0; o < 64; ++o) h2[o] = tanhf(pol_dot(h1, 64, w + STG_POLICY_VF_W2, 64, o, w[STG_POLICY_VF_B2 + o]));
    value[i] = pol_dot(h2, 64, w + STG_POLICY_VAL_W, 1, 0, w[STG_POLICY_VAL_B]);
    for (int o = 0; o < 64; ++o) h1[o] = tanhf(pol_dot(x, 12, w + STG_POLICY_PI_W1, 64, o, w[STG_POLICY_PI_B1 + o]));
    for (int o = 0; o < 64; ++o) h2[o] = tanhf(pol_dot(h1, 64, w + STG_POLICY_PI_W2, 64, o, w[STG_POLICY_PI_B2 + o]));
    float lp = 0.0f;
    for (int d = 0; d < 2; ++d) {
      const float m = pol_dot(h2, 64, w + STG_POLICY_ACT_W, 2, d, w[STG_POLICY_ACT_B + d]);
      const float t = pol_log_prob_term(act[2 * i + d], m, w[STG_POLICY_STD + d], w[STG_POLICY_LOG_SCALE + d]);
      lp = d == 0 ? t : Pk<float>::add(lp, t);
    }
    logp[i] = lp;
  }
}
extern "C" void advantage(const float* adv, int64_t n, const float* stats, float* out) {
  for (int64_t i = 0; i < n; ++i) out[i] = pol_ppo_advantage(adv[i], stats);
}
extern "C" void ppo(const float* w, const float* obs, const float* act, const float* old_v, const float* old_lp,
                    const float* adv, const float* ret, int64_t n, float clip_range, float lo, float hi, float clip_vf,
                    int clip_value, float ent_coef, float vf_coef, float* grad, float* losses) {
  const PolPpoCoef c{clip_range, lo, hi, clip_vf, clip_value != 0};
  static double g[STG_POLICY_PARAMS];
  double sums[4] = {0, 0, 0, 0};
  for (int p = 0; p < STG_POLICY_PARAMS; ++p) g[p] = 0.0;
  for (int64_t i = 0; i < n; ++i)
    pol_backward_row(w, obs + 12 * i, act + 2 * i, old_v[i], old_lp[i], adv[i], ret[i], c, g, sums);
  for (int p = 0; p < STG_POLICY_PARAMS; ++p) grad[p] = pol_ppo_grad_value(p, g[p], n, ent_coef, vf_coef);
  pol_ppo_losses(sums, w, n, ent_coef, vf_coef, losses);
}
''')
    so = d / "ppo_host.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-I", CSRC, str(src), "-o", str(so)], check=True)
    lib = C.CDLL(str(so))
    dp, i64, f32 = C.c_void_p, C.c_int64, C.c_float
    lib.eval.argtypes = [dp, dp, dp, i64, dp, dp]
    lib.advantage.argtypes = [dp, i64, dp, dp]
    lib.ppo.argtypes = [dp] * 7 + [i64, f32, f32, f32, f32, C.c_int, f32, f32, dp, dp]
    return lib


def _p(a):
    return a.ctypes.data


def grads_by_name(pol, flat):
    """{parameter name: its gradient} from a flat buffer in the STG_PPO_GRAD_* layout."""
    import torch
    flat = torch.as_tensor(flat)
    names = {id(p): n for n, p in pol.named_parameters()}
    return {names[id(p)]: flat[off:off + p.numel()].view(p.shape) for p, off in pol._grad_slots()}


def host_ppo_step(lib, pol, batch, clip_range=0.2, clip_range_vf=None, ent_coef=0.0, vf_coef=0.5, normalize_advantage=True):
    """The host core on a float32 CPU batch: ({name: grad}, losses)."""
    import torch
    w, _ = _packed_numpy(pol)
    obs, act, old_v, old_lp, adv, ret = (np.ascontiguousarray(t.numpy(), np.float32) for t in batch)
    n = len(obs)
    if normalize_advantage and n > 1:
        a = torch.from_numpy(adv)
        stats = np.array([float(a.mean()), float(a.std())], np.float32)
        adv_n = np.empty_like(adv)
        lib.advantage(_p(adv), n, _p(stats), _p(adv_n))
        assert np.array_equal(adv_n, ((a - a.mean()) / (a.std() + 1e-8)).numpy())      # torch's float32 bits
        adv = adv_n
    grad, losses = np.empty(_lib.POLICY_PARAMS, np.float32), np.empty(6, np.float32)
    lib.ppo(_p(w), _p(obs), _p(act), _p(old_v), _p(old_lp), _p(adv), _p(ret), n, clip_range, 1.0 - clip_range,
            1.0 + clip_range, clip_range_vf or 0.0, clip_range_vf is not None, ent_coef, vf_coef, _p(grad), _p(losses))
    return grads_by_name(pol, grad), losses


def synthetic_batch(lib, pol, n, seed, ratio_set=(0.5, 0.7, 0.9, 1.0, 1.1, 1.35, 1.6), zero_adv=0.0):
    """A float32 CPU batch whose ratios are drawn from ratio_set (1.0: old_log_prob = the core's log-prob exactly, a tie),
    whose value offsets lie on both sides of the value clip 0.3 and away from it, and a fraction zero_adv of zero advantages."""
    import torch
    rng = np.random.default_rng(seed)
    w, _ = _packed_numpy(pol)
    obs = (rng.normal(size=(n, 12)) * rng.choice([0.3, 1.0, 2.0], size=(n, 12))).astype(np.float32)
    act = (rng.normal(size=(n, 2)) * 0.8).astype(np.float32)
    value, logp = np.empty(n, np.float32), np.empty(n, np.float32)
    lib.eval(_p(w), _p(obs), _p(act), n, _p(value), _p(logp))
    r = rng.choice(ratio_set, size=n)
    old_lp = np.where(r == 1.0, logp, (logp.astype(np.float64) - np.log(r))).astype(np.float32)
    old_v = (value + rng.choice([-0.6, -0.1, 0.05, 0.5], size=n)).astype(np.float32)
    adv = (rng.normal(size=n) * 2 + 0.3).astype(np.float32)
    adv[rng.random(n) < zero_adv] = 0.0
    ret = (value + rng.normal(size=n)).astype(np.float32)
    return [torch.from_numpy(a) for a in (obs, act, old_v, old_lp, adv, ret)]


# ---------------------------------------------------------------------------------------------------- CPU ---------------

@pytest.mark.parametrize("kw", [dict(), dict(clip_range_vf=0.3), dict(ent_coef=0.01), dict(normalize_advantage=False),
                                dict(clip_range=0.25, clip_range_vf=0.3, ent_coef=0.05, vf_coef=0.7)])
def test_core_backward_matches_float64_autograd(host_ppo, kw):
    pol = _random_policy(FakeEnv(), 11)
    batch = synthetic_batch(host_ppo, pol, 3000, 1, zero_adv=0.0 if kw.get("normalize_advantage", True) else 0.1)
    got, losses = host_ppo_step(host_ppo, pol, batch, **kw)
    want, want_losses = reference_grads(pol, batch, **kw)
    check_grads(got, want, tol=2e-5)
    check_losses(losses, want_losses)
    assert 0.1 < want_losses[5] < 0.9                                       # rows on both branches of the min


def test_core_backward_single_row_and_special_rows(host_ppo):
    pol = _random_policy(FakeEnv(), 12)
    for ratio_set in ((1.0,), (0.5,), (1.6,)):
        batch = synthetic_batch(host_ppo, pol, 1, 2, ratio_set=ratio_set)   # B = 1: no normalisation
        for kw in (dict(), dict(clip_range_vf=0.3, ent_coef=0.02)):
            got, losses = host_ppo_step(host_ppo, pol, batch, **kw)
            want, want_losses = reference_grads(pol, batch, **kw)
            check_grads(got, want)                  # one row: FP32's action - mean cancels, nothing averages it out
            check_losses(losses, want_losses)
    # ties only (ratio exactly 1): approx_kl and clip_fraction exactly 0, the gradient the unclipped one
    batch = synthetic_batch(host_ppo, pol, 500, 3, ratio_set=(1.0,))
    got, losses = host_ppo_step(host_ppo, pol, batch)
    assert losses[4] == 0.0 and losses[5] == 0.0
    check_grads(got, reference_grads(pol, batch)[0])
    # zero advantages (no normalisation): the policy gradient of those rows is zero on every branch
    batch = synthetic_batch(host_ppo, pol, 400, 4, zero_adv=1.0)
    got, losses = host_ppo_step(host_ppo, pol, batch, normalize_advantage=False)
    assert float(got["action_net.weight"].abs().max()) == 0.0 and losses[1] == 0.0
    want, _ = reference_grads(pol, batch, normalize_advantage=False)
    check_grads({k: v for k, v in got.items() if k != "log_std"}, {k: v for k, v in want.items() if k != "log_std"})


def test_ppo_args_layout_constants_and_grid(tmp_path):
    fields = [f for f, _ in _lib.StgPpoArgs._fields_]
    sizes = [1, 127, 128, 129, 4097, 37888, 37889, 65536, 1 << 20, 0, -5]
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', 'int main(void){',
             'printf("size %zu\\n", sizeof(StgPpoArgs));']
    lines += [f'printf("{f} %zu\\n", offsetof(StgPpoArgs, {f}));' for f in fields]
    lines += [f'printf("grid{i} %lld\\n", (long long)STG_PPO_GRID((int64_t){b}));' for i, b in enumerate(sizes)]
    lines += [f'printf("work{i} %lld\\n", (long long)STG_PPO_WORK_DOUBLES((int64_t){b}));' for i, b in enumerate(sizes)]
    consts = dict(STG_PPO_TILE=_lib.PPO_TILE, STG_PPO_MAX_CTAS=_lib.PPO_MAX_CTAS, STG_PPO_PART=_lib.PPO_PART,
                  STG_PPO_PART_LOSS=_lib.PPO_PART_LOSS, STG_PPO_LOSSES=_lib.PPO_LOSSES, STG_PPO_CLIP_VF=_lib.PPO_CLIP_VF,
                  STG_ABI_VERSION=7)
    consts.update({f"STG_PPO_GRAD_{k}": v for k, v in _lib.POLICY_LAYOUT.items() if k not in ("STD", "LOG_SCALE")})
    lines += [f'printf("{c} %lld\\n", (long long)({c}));' for c in consts]
    lines.append('return 0;}')
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", str(src), "-o", str(exe)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split("\n") if l)
    assert int(got["size"]) == C.sizeof(_lib.StgPpoArgs)
    for f in fields:
        assert int(got[f]) == getattr(_lib.StgPpoArgs, f).offset, f
    for c, v in consts.items():
        assert int(got[c]) == v, c
    # known answers: one CTA per 128-row tile up to 296 CTAs (two per SM of a 148-SM B200), whatever the device
    want_grid = [1, 1, 1, 2, 33, 296, 296, 296, 296, 0, 0]
    for i, (b, g) in enumerate(zip(sizes, want_grid)):
        assert int(got[f"grid{i}"]) == g == _lib.ppo_grid(b), b
        assert int(got[f"work{i}"]) == g * 10192 == _lib.ppo_work_doubles(b), b
    assert _lib.PPO_PART_LOSS == _lib.POLICY_PARAMS and _lib.PPO_PART >= _lib.PPO_PART_LOSS + 4 and _lib.PPO_PART % 2 == 0


def _ppo_args(**ptrs):
    a = _lib.StgPpoArgs()
    a.batch = ptrs.pop("batch", 4)
    for k, v in ptrs.items():
        setattr(a, k, v)
    return a


def test_ppo_argument_validation():
    f = _lib.load().stg_policy_ppo_grad_f32
    call = lambda a: f(C.byref(a), None)                                    # noqa: E731
    B = 0x10000
    req = ("d_weights", "d_obs", "d_action", "d_old_value", "d_old_log_prob", "d_advantage", "d_return", "d_grad",
           "d_losses", "d_work")
    ok = {k: B * (i + 1) for i, k in enumerate(req)}
    assert f(None, None) == -1                                              # STG_E_NULL
    assert call(_ppo_args(batch=0, **ok)) == -2                             # STG_E_SIZE: an empty batch has no loss
    assert call(_ppo_args(batch=-1)) == -2                                  # size before pointers
    for k in req:
        assert call(_ppo_args(**dict(ok, **{k: None}))) == -1, k
    assert call(_ppo_args(batch=-1, **dict(ok, d_obs=B + 4))) == -2
    for k, off in (("d_weights", 8), ("d_obs", 4), ("d_action", 4), ("d_work", 4), ("d_old_value", 2), ("d_return", 1),
                   ("d_adv_stats", 2), ("d_grad", 2), ("d_losses", 1)):
        assert call(_ppo_args(**dict(ok, **{k: ok.get(k, B) + off}))) == -4, k   # STG_E_ALIGN
    assert call(_ppo_args(flags=2, **dict(ok, d_obs=B + 4))) == -4          # alignment before flags
    assert call(_ppo_args(flags=2, **ok)) == -3                             # STG_E_ENUM
    assert call(_ppo_args(d_weights=None, **{k: v for k, v in ok.items() if k != "d_weights"}, flags=2)) == -1


def test_ppo_backward_python_errors():
    import torch
    from spin_torque_rl_gym_b200.envs.sb3_vec_env import RolloutBufferSamples
    pol = _random_policy(FakeEnv(), 13)

    def samples(n=8, **over):
        t = dict(observations=torch.zeros(n, 12), actions=torch.zeros(n, 2), old_values=torch.zeros(n),
                 old_log_prob=torch.zeros(n), advantages=torch.zeros(n), returns=torch.zeros(n))
        t.update(over)
        return RolloutBufferSamples(**t)

    with pytest.raises(_lib.StgError):
        pol.ppo_backward(samples())                                          # well-formed, but on the CPU
    for bad in (samples(0), samples(observations=torch.zeros(8, 13)), samples(actions=torch.zeros(8, 3)),
                samples(returns=torch.zeros(7)), samples(old_values=torch.zeros(8, 1)),
                samples(advantages=torch.zeros(8, dtype=torch.float64)), samples(observations=torch.zeros(12)),
                samples(actions=torch.zeros(8, 2, dtype=torch.float16)), samples(returns=np.zeros(8, np.float32))):
        with pytest.raises(ValueError):
            pol.ppo_backward(bad)


# ---------------------------------------------------------------------------------------------------- GPU ---------------

def _venv(stg, dev, n, max_steps=40, seed=5):
    return stg.VecNormalize(stg.make("SpinTorque-v0", num_envs=n, device=dev, max_steps=max_steps, rng_seed=seed))


def _rollout(stg, dev, n, T, seed=5):
    """A collector with one fused rollout of a fresh policy, GAE done."""
    import torch
    env = _venv(stg, dev, n, seed=seed)
    torch.manual_seed(seed)
    pol = stg.ActorCriticPolicy(env, log_std_init=-0.5)
    col = stg.RolloutCollector(env, n_steps=T, store_values=True)
    col.collect(pol)
    col.compute_returns_and_advantage(gamma=0.99, gae_lambda=0.95)
    return env, pol, col


def _perturb(pol, seed, scale=0.03):
    import torch
    g = torch.Generator(device=pol.log_std.device).manual_seed(seed)
    with torch.no_grad():
        for p in pol.parameters():
            p.add_(torch.randn(p.shape, generator=g, device=p.device) * scale * (p.abs().mean() + 0.05))


def _fields(b):
    return (b.observations, b.actions, b.old_values, b.old_log_prob, b.advantages, b.returns)


def _clear_of(x, candidates, margin=1e-5):
    """A clip range c such that no |x| lies within `margin` of c: the first of the candidates that is, else the midpoint of the
    widest gap between consecutive sorted |x| in their top decile (below the 99.99th percentile, so rows lie on both sides of
    it). With 10^6 rows every fixed candidate has rows within 1e-5 of it; the tail has gaps."""
    import torch
    d = torch.sort(x.abs().flatten()).values
    c = next((c for c in candidates if float((d - c).abs().min()) > margin), None)
    if c is None and len(d) > 100:
        i0, i1 = int(0.9 * (len(d) - 1)), int(0.9999 * (len(d) - 1))
        gaps = d[i0 + 1:i1 + 1] - d[i0:i1]
        k = int(torch.argmax(gaps))
        if float(gaps[k]) > 2 * margin:
            c = float((d[i0 + k] + d[i0 + k + 1]) / 2)
    assert c is not None and float((d - c).abs().min()) > margin, "no clip range clear of every row by 1e-5"
    return c


def _pick_clip(pol, batch, candidates, vf_candidates):
    """clip_range and clip_range_vf such that no row's float64 ratio or value offset lies within 1e-5 of a clip boundary, where
    FP32 could take the other branch (one such row is worth about 1/sqrt(B) of the gradient)."""
    import copy
    import torch
    ref = copy.deepcopy(pol).double()
    ref.extract_features = lambda obs: obs
    with torch.no_grad():
        v, lp, _ = ref.evaluate_actions(batch.observations.double(), batch.actions.double())
        ratio = torch.exp(lp - batch.old_log_prob.double())
        dv = v.flatten() - batch.old_values.double()
    return _clear_of(ratio - 1, candidates), _clear_of(dv, vf_candidates)


def _grads(pol):
    return {n: p.grad.detach().clone() for n, p in pol.named_parameters()}


def _torch32_grads(pol, batch, **kw):
    import copy
    ref = copy.deepcopy(pol)
    for p in ref.parameters():
        p.grad = None
    loss, _ = sb3_ppo_loss(ref, *_fields(batch), **kw)
    loss.backward()
    return {n: p.grad.detach() for n, p in ref.named_parameters()}


@pytest.fixture(scope="module")
def big_rollout(cuda_device):
    import spin_torque_rl_gym_b200 as stg
    env, pol, col = _rollout(stg, cuda_device, 65536, 16)                   # 1,048,576 samples
    _perturb(pol, 1)
    return env, pol, col


@pytest.mark.gpu
@pytest.mark.parametrize("B", [1, 127, 4097, 65536, 1048576])
def test_cuda_gradient_matches_float64_autograd(big_rollout, B):
    _, pol, col = big_rollout
    batch = next(iter(col.get(B)))
    cr, vf = _pick_clip(pol, batch, (0.2, 0.15, 0.25, 0.1, 0.3), (0.2, 0.15, 0.25, 0.1, 0.3))
    for kw in (dict(clip_range=cr, ent_coef=0.01), dict(clip_range=cr, clip_range_vf=vf, normalize_advantage=False)):
        losses = pol.ppo_backward(batch, **kw)
        got = _grads(pol)
        want, want_losses = reference_grads(pol, _fields(batch), **kw)
        worst = check_grads(got, want)
        check_losses(losses, want_losses)
        t32 = check_grads(_torch32_grads(pol, batch, **kw), want, tol=1.0)
        print(f"B={B} {sorted(kw.items())}: K10 max rel err {worst:.2e}, torch float32 autograd {t32:.2e}, "
              f"clip_fraction {want_losses[5]:.3f}")
        if B >= 4097:
            assert 0.0 < want_losses[5] < 1.0                                # both branches of the min occur


@pytest.mark.gpu
def test_cuda_first_epoch_is_exact(cuda_device):
    import torch
    import spin_torque_rl_gym_b200 as stg
    _, pol, col = _rollout(stg, cuda_device, 4096, 8)
    batches = list(col.get(4096))
    assert len(batches) == 8
    for b in batches:
        losses = pol.ppo_backward(b, clip_range_vf=0.2)
        assert float(losses.approx_kl) == 0.0 and float(losses.clip_fraction) == 0.0
    want, want_losses = reference_grads(pol, _fields(batches[-1]), clip_range_vf=0.2)
    check_grads(_grads(pol), want)
    check_losses(losses, want_losses)


@pytest.mark.gpu
def test_cuda_deterministic_and_no_host_sync(big_rollout):
    import torch
    _, pol, col = big_rollout
    batch = next(iter(col.get(100003)))
    kw = dict(clip_range_vf=0.2, ent_coef=0.01)
    l1 = torch.stack(pol.ppo_backward(batch, **kw)).clone()
    g1 = pol._grad.clone()
    l2 = torch.stack(pol.ppo_backward(batch, **kw))
    assert torch.equal(g1, pol._grad) and torch.equal(l1, l2)
    # the same batch at other addresses, one of them misaligned (copied inside)
    from spin_torque_rl_gym_b200.envs.sb3_vec_env import RolloutBufferSamples
    moved = RolloutBufferSamples(*(torch.cat([torch.zeros(1, *t.shape[1:], device=t.device), t])[1:] for t in _fields(batch)))
    assert moved.returns.data_ptr() % 16 != 0
    pol.ppo_backward(moved, **kw)
    assert torch.equal(g1, pol._grad)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        l3 = torch.stack(pol.ppo_backward(batch, **kw))
    torch.cuda.current_stream().wait_stream(side)
    assert torch.equal(g1, pol._grad) and torch.equal(l1, l3)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        pol.ppo_backward(batch, **kw)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert torch.equal(g1, pol._grad)
    # .grad are views into the one buffer, reassigned after zero_grad(set_to_none=True)
    pol.zero_grad(set_to_none=True)
    pol.ppo_backward(batch, **kw)
    for p, off in pol._grad_slots():
        assert p.grad.data_ptr() == pol._grad.data_ptr() + 4 * off and p.grad.is_contiguous()


@pytest.mark.gpu
def test_cuda_training_matches_eager_torch(cuda_device):
    import copy
    import torch
    import spin_torque_rl_gym_b200 as stg
    _, pol, col = _rollout(stg, cuda_device, 8192, 16)
    batches = list(col.get(8192))
    eager = copy.deepcopy(pol)
    opt_f = torch.optim.SGD(pol.parameters(), lr=0.05)
    opt_e = torch.optim.SGD(eager.parameters(), lr=0.05)
    kw = dict(clip_range_vf=0.2, ent_coef=0.01)
    for b in batches:
        pol.ppo_backward(b, **kw)
        opt_f.step()
        opt_e.zero_grad()
        sb3_ppo_loss(eager, *_fields(b), **kw)[0].backward()
        opt_e.step()
    for (name, p), q in zip(pol.named_parameters(), eager.parameters()):
        assert float((p - q).detach().abs().max()) <= 1e-4 * float(q.detach().abs().max()), name
    # a short Adam + clip_grad_norm_ iteration, then the next rollout acts with the updated weights
    opt = torch.optim.Adam(pol.parameters(), lr=3e-4, eps=1e-5, fused=True)
    before = [p.detach().clone() for p in pol.parameters()]
    for b in col.get(16384):
        losses = pol.ppo_backward(b)
        torch.nn.utils.clip_grad_norm_(pol.parameters(), 0.5)
        opt.step()
    assert torch.isfinite(torch.stack(losses)).all()
    assert any(not torch.equal(p, q) for p, q in zip(pol.parameters(), before))
    col.collect(pol)
    with torch.no_grad():
        v, lp, _ = pol.evaluate_actions(col.observations[0], col.actions[0])
    assert float((v[:, 0] - col.values[0]).abs().max()) <= 1e-5
    assert float((lp - col.log_probs[0]).abs().max()) <= 1e-5
