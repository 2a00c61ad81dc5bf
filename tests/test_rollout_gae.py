"""K6: generalised advantage estimation over a stored rollout (stg_rollout_gae_f32, RolloutCollector(store_values=True)).

The specification is Stable-Baselines3's float32 computation, restated below in NumPy exactly as SB3 writes it: the
TimeLimit.truncated bootstrap of OnPolicyAlgorithm.collect_rollouts followed by RolloutBuffer.compute_returns_and_advantage.
Every comparison is np.array_equal."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from spin_torque_rl_gym_b200 import _lib
from tests.helpers import ROOT

HEADER = os.path.join(ROOT, "include", "stg.h")
CSRC = os.path.join(ROOT, "spin_torque_rl_gym_b200", "csrc")


def sb3_gae(reward, value, terminated, truncated, final_value, last_value, gamma, gae_lambda):
    """SB3's float32 loop. `final_value` is read only at truncated-but-not-terminated entries (the others may be NaN)."""
    T, _ = reward.shape
    rewards = reward.astype(np.float32).copy()
    values = value.astype(np.float32)
    dones = (terminated | truncated).astype(np.float32)
    for t in range(T):                                   # collect_rollouts: rewards[idx] += self.gamma * terminal_value
        idx = np.nonzero(truncated[t] & ~terminated[t])[0]
        rewards[t, idx] += gamma * final_value[t, idx]
    advantages = np.zeros_like(rewards)
    last_gae_lam = 0
    for step in reversed(range(T)):                      # RolloutBuffer.compute_returns_and_advantage
        if step == T - 1:
            next_non_terminal = 1.0 - dones[T - 1]
            next_values = last_value.astype(np.float32)
        else:
            next_non_terminal = 1.0 - dones[step]        # episode_starts[step + 1] is the done flag of step `step`
            next_values = values[step + 1]
        delta = rewards[step] + gamma * next_values * next_non_terminal - values[step]
        last_gae_lam = delta + gamma * gae_lambda * next_non_terminal * last_gae_lam
        advantages[step] = last_gae_lam
    return advantages, advantages + values


def make_case(T, N, flags, seed):
    rng = np.random.default_rng(seed)
    reward = rng.normal(size=(T, N)).astype(np.float32)
    value = (rng.normal(size=(T, N)) * 3).astype(np.float32)
    if flags == "none":
        term = np.zeros((T, N), bool)
        trunc = np.zeros((T, N), bool)
    elif flags == "all":
        term = rng.random((T, N)) < 0.5
        trunc = ~term | (rng.random((T, N)) < 0.3)      # every step ends an episode, some with both flags
    else:
        term = rng.random((T, N)) < 0.05
        trunc = rng.random((T, N)) < 0.1                 # independent: some steps carry both flags
    final_value = (rng.normal(size=(T, N)) * 3).astype(np.float32)
    final_value[~(trunc & ~term)] = np.nan               # stale rows: must never reach an output
    last_value = rng.normal(size=N).astype(np.float32)
    return reward, value, term, trunc, final_value, last_value


CASES = [(T, flags) for T in (1, 2, 37, 256) for flags in ("all", "none", "mixed")]
COEFS = [(0.99, 0.95), (0.997, 0.9)]


def test_gae_args_layout_matches_the_c_header(tmp_path):
    fields = ["d_reward", "d_value", "d_terminated", "d_truncated", "d_final_value", "d_last_value", "d_advantage", "d_return",
              "gamma", "gamma_lambda", "n_steps", "n_envs"]
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', 'int main(void){',
             'printf("size %zu\\n", sizeof(StgGaeArgs));']
    lines += [f'printf("{f} %zu\\n", offsetof(StgGaeArgs, {f}));' for f in fields]
    lines.append('return 0;}')
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", str(src), "-o", str(exe)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split("\n") if l)
    assert int(got["size"]) == C.sizeof(_lib.StgGaeArgs)
    for f in fields:
        assert int(got[f]) == getattr(_lib.StgGaeArgs, f).offset, f


def test_gae_argument_validation():
    lib = _lib.load()
    assert lib.stg_rollout_gae_f32(None, None) == -1                       # STG_E_NULL
    a = _lib.StgGaeArgs()
    a.n_steps, a.n_envs = -1, 4
    assert lib.stg_rollout_gae_f32(C.byref(a), None) == -2                 # STG_E_SIZE
    a.n_steps, a.n_envs = 4, -1
    assert lib.stg_rollout_gae_f32(C.byref(a), None) == -2
    for t, n in ((0, 4), (4, 0), (0, 0)):                                  # empty: nothing to launch
        a.n_steps, a.n_envs = t, n
        assert lib.stg_rollout_gae_f32(C.byref(a), None) == 0
    a.n_steps, a.n_envs = 4, 4
    assert lib.stg_rollout_gae_f32(C.byref(a), None) == -1                 # no buffers
    names = ["d_reward", "d_value", "d_terminated", "d_truncated", "d_final_value", "d_last_value", "d_advantage"]
    for missing in names:                                                   # every required pointer is checked
        for f in names:
            setattr(a, f, None if f == missing else 0x1000)
        assert lib.stg_rollout_gae_f32(C.byref(a), None) == -1, missing


@pytest.fixture(scope="module")
def host_gae(tmp_path_factory):
    """rollout_core.cuh compiled for the host with contraction ALLOWED: gae_step must still round every operation."""
    d = tmp_path_factory.mktemp("gae_host")
    src = d / "gae_host.cpp"
    src.write_text('#include "rollout_core.cuh"\n'
                   'extern "C" void gae_host(const float* r, const float* v, const uint8_t* te, const uint8_t* tr, const float* fv,\n'
                   '                         const float* lv, float* adv, float* ret, float g, float gl, long T, long N) {\n'
                   '  for (long i = 0; i < N; ++i) {\n'
                   '    float vn = lv[i], a = 0.0f;\n'
                   '    for (long t = T - 1; t >= 0; --t) {\n'
                   '      const long o = t * N + i;\n'
                   '      a = stg::gae_step(r[o], v[o], vn, te[o] != 0, tr[o] != 0, fv[o], g, gl, a, ret[o]);\n'
                   '      vn = v[o]; adv[o] = a;\n'
                   '    }\n'
                   '  }\n'
                   '}\n')
    so = d / "gae_host.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-mfma", "-ffp-contract=fast", "-fPIC", "-shared", "-I", CSRC, str(src),
                    "-o", str(so)], check=True)
    lib = C.CDLL(str(so))
    lib.gae_host.argtypes = [C.c_void_p] * 8 + [C.c_float, C.c_float, C.c_long, C.c_long]

    def run(reward, value, term, trunc, final_value, last_value, gamma, gae_lambda):
        T, N = reward.shape
        te, tr = np.ascontiguousarray(term, np.uint8), np.ascontiguousarray(trunc, np.uint8)
        adv, ret = np.empty((T, N), np.float32), np.empty((T, N), np.float32)
        ins = [np.ascontiguousarray(x) for x in (reward, value)] + [te, tr] + \
              [np.ascontiguousarray(x) for x in (final_value, last_value)]
        lib.gae_host(*[x.ctypes.data for x in ins], adv.ctypes.data, ret.ctypes.data, float(np.float32(gamma)),
                     float(np.float32(gamma * gae_lambda)), T, N)
        return adv, ret
    return run


@pytest.mark.parametrize("T,flags", CASES)
def test_host_build_of_the_recurrence_equals_sb3(host_gae, T, flags):
    for k, (gamma, lam) in enumerate(COEFS):
        case = make_case(T, 333, flags, seed=T * 7 + k)
        want_adv, want_ret = sb3_gae(*case, gamma, lam)
        adv, ret = host_gae(*case, gamma, lam)
        assert np.isfinite(adv).all() and np.array_equal(adv, want_adv)
        assert np.array_equal(ret, want_ret)
        assert np.isnan(case[4]).any()                                      # stale final values, to be skipped


# ---------------------------------------------------------------------------------------------------- GPU --------------------

def _gae_on_device(torch, planes, gamma, gae_lambda, with_return=True):
    reward, value, term, trunc, final_value, last_value = planes
    T, N = reward.shape
    adv = torch.empty(T, N, dtype=torch.float32, device=reward.device)
    ret = torch.empty_like(adv) if with_return else None
    a = _lib.StgGaeArgs()
    a.d_reward, a.d_value = reward.data_ptr(), value.data_ptr()
    a.d_terminated, a.d_truncated = term.data_ptr(), trunc.data_ptr()
    a.d_final_value, a.d_last_value = final_value.data_ptr(), last_value.data_ptr()
    a.d_advantage, a.d_return = adv.data_ptr(), (ret.data_ptr() if with_return else None)
    a.gamma, a.gamma_lambda = float(np.float32(gamma)), float(np.float32(gamma * gae_lambda))
    a.n_steps, a.n_envs = T, N
    _lib.check(_lib.load().stg_rollout_gae_f32(C.byref(a), torch.cuda.current_stream().cuda_stream), "stg_rollout_gae_f32")
    return adv, ret


def _to_device(torch, dev, case):
    reward, value, term, trunc, final_value, last_value = case
    f = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)         # noqa: E731
    return (f(reward), f(value), f(term.astype(np.uint8)), f(trunc.astype(np.uint8)), f(final_value), f(last_value))


@pytest.mark.gpu
@pytest.mark.parametrize("N", [1, 1000, 4097])
def test_cuda_gae_kernel_equals_sb3(cuda_device, N):
    import torch
    for T, flags in CASES:
        for k, (gamma, lam) in enumerate(COEFS):
            case = make_case(T, N, flags, seed=N * 1000 + T * 7 + k)
            want_adv, want_ret = sb3_gae(*case, gamma, lam)
            adv, ret = _gae_on_device(torch, _to_device(torch, cuda_device, case), gamma, lam, with_return=(k == 0))
            assert np.array_equal(adv.cpu().numpy(), want_adv), (T, flags, N)
            if ret is not None:
                assert np.array_equal(ret.cpu().numpy(), want_ret), (T, flags, N)


@pytest.mark.gpu
def test_cuda_gae_kernel_full_rollout_shard(cuda_device):
    """BASELINE configs[4]'s per-GPU shard: 2048 steps x 131,072 envs."""
    import torch
    case = make_case(2048, 131072, "mixed", seed=11)
    want_adv, want_ret = sb3_gae(*case, 0.99, 0.95)
    adv, ret = _gae_on_device(torch, _to_device(torch, cuda_device, case), 0.99, 0.95)
    assert np.array_equal(adv.cpu().numpy(), want_adv) and np.array_equal(ret.cpu().numpy(), want_ret)


@pytest.mark.gpu
def test_cuda_gae_kernel_int64_offsets(cuda_device):
    """2049 steps x 1,048,576 envs = 2,148,532,224 elements > 2^31 (about 47 GB of planes), generated on the device; 1,024
    env columns, the last one included, checked against the NumPy restatement (the recurrence is per column: exact)."""
    import torch
    T, N = 2049, 1 << 20
    g = torch.Generator(device=cuda_device).manual_seed(5)
    reward = torch.randn(T, N, generator=g, device=cuda_device)
    value = torch.randn(T, N, generator=g, device=cuda_device)
    term = (torch.rand(T, N, generator=g, device=cuda_device) < 0.005).view(torch.uint8)
    trunc = (torch.rand(T, N, generator=g, device=cuda_device) < 0.01).view(torch.uint8)
    final_value = torch.randn(T, N, generator=g, device=cuda_device)
    final_value.masked_fill_((trunc > term).logical_not_(), float("nan"))
    last_value = torch.randn(N, generator=g, device=cuda_device)
    adv, ret = _gae_on_device(torch, (reward, value, term, trunc, final_value, last_value), 0.99, 0.95)
    cols = np.unique(np.concatenate([np.random.default_rng(0).choice(N, 1022, replace=False), [0, N - 1]]))
    idx = torch.from_numpy(cols).to(cuda_device)
    pick = lambda x: x.index_select(-1, idx).cpu().numpy()                 # noqa: E731
    want_adv, want_ret = sb3_gae(pick(reward), pick(value), pick(term).astype(bool), pick(trunc).astype(bool),
                                 pick(final_value), pick(last_value), 0.99, 0.95)
    assert np.array_equal(pick(adv), want_adv) and np.array_equal(pick(ret), want_ret)
    assert np.isfinite(want_adv).all()


def _actor_critic(torch, dev):
    gen = torch.Generator(device=dev).manual_seed(0)
    w1 = torch.randn(12, 32, generator=gen, device=dev) * 0.3
    wa = torch.randn(32, 2, generator=gen, device=dev) * 0.3
    wv = torch.randn(32, 1, generator=gen, device=dev) * 0.3

    def actor(o):
        out = torch.tanh(o @ w1) @ wa
        act = torch.empty(o.shape[0], 2, device=dev)
        act[:, 0] = torch.tanh(out[:, 0]) * 1.1e-6
        act[:, 1] = torch.sigmoid(out[:, 1]) * 1e-9 + 1e-11
        return act, -(out * out).sum(1)

    def value_fn(o):
        return torch.tanh(o @ w1) @ wv                                      # [N, 1]

    def policy(o):
        act, logp = actor(o)
        return act, value_fn(o), logp
    return actor, value_fn, policy


@pytest.mark.gpu
def test_rollout_collector_values_and_gae_end_to_end(cuda_device):
    import torch
    import spin_torque_rl_gym_b200 as stg
    n, T = 512, 16
    mk = lambda: stg.make("SpinTorque-v0", num_envs=n, device=cuda_device, max_steps=5, max_current=1.1e-6, rng_seed=3)  # noqa: E731
    actor, value_fn, policy = _actor_critic(torch, cuda_device)
    col = stg.RolloutCollector(mk(), n_steps=T, store_values=True)
    col.collect(policy, value_fn)
    col.compute_returns_and_advantage()
    pl = {k: getattr(col, k).cpu().numpy() for k in ("rewards", "values", "terminated", "truncated", "final_values",
                                                      "last_values", "advantages", "returns", "dones", "log_probs")}
    assert pl["truncated"].sum() >= n and np.array_equal(pl["dones"], pl["terminated"] | pl["truncated"])
    want_adv, want_ret = sb3_gae(pl["rewards"], pl["values"], pl["terminated"], pl["truncated"], pl["final_values"],
                                 pl["last_values"], 0.99, 0.95)
    assert np.array_equal(pl["advantages"], want_adv) and np.array_equal(pl["returns"], want_ret)
    col.compute_returns_and_advantage(gamma=0.9, gae_lambda=0.8)
    want_adv, _ = sb3_gae(pl["rewards"], pl["values"], pl["terminated"], pl["truncated"], pl["final_values"],
                          pl["last_values"], 0.9, 0.8)
    assert np.array_equal(col.advantages.cpu().numpy(), want_adv)

    # the same rollout stepped by hand: flags, final observations, rewards, values and log-probabilities
    env = mk()
    obs, _ = env.reset()
    for t in range(T):
        act, logp = actor(obs)
        assert np.array_equal(pl["values"][t], value_fn(obs).reshape(n).cpu().numpy())
        assert np.array_equal(pl["log_probs"][t], logp.cpu().numpy())
        obs, rew, term, trunc, info = env.step(act)
        te, tr = term.cpu().numpy(), trunc.cpu().numpy()
        assert np.array_equal(pl["terminated"][t], te) and np.array_equal(pl["truncated"][t], tr)
        assert np.array_equal(pl["rewards"][t], rew.float().cpu().numpy())
        fin = value_fn(info["final_observation"]).reshape(n).cpu().numpy()
        assert np.array_equal(pl["final_values"][t][tr], fin[tr])
    assert np.array_equal(pl["last_values"], value_fn(obs).reshape(n).cpu().numpy())

    # rewards are the env's rewards, exactly what the default collector stores for the same seed and actions
    plain = stg.RolloutCollector(mk(), n_steps=T)
    plain.collect(lambda o: actor(o)[0])
    assert torch.equal(plain.rewards, col.rewards) and torch.equal(plain.actions, col.actions)


@pytest.mark.gpu
def test_rollout_collector_default_is_unchanged_and_errors(cuda_device):
    import torch
    import spin_torque_rl_gym_b200 as stg
    env = stg.make("SpinTorque-v0", num_envs=64, device=cuda_device, max_steps=5, max_current=1.1e-6, rng_seed=3)
    actor, value_fn, policy = _actor_critic(torch, cuda_device)
    plain = stg.RolloutCollector(env, n_steps=4)
    for name in ("values", "log_probs", "final_values", "terminated", "truncated", "last_values", "advantages", "returns"):
        assert not hasattr(plain, name), name
    plain.collect(lambda o: actor(o)[0])
    with pytest.raises(RuntimeError):
        plain.compute_returns_and_advantage()
    col = stg.RolloutCollector(env, n_steps=4, store_values=True)
    with pytest.raises(RuntimeError):
        col.compute_returns_and_advantage()                                 # nothing collected yet
    with pytest.raises(ValueError):
        col.collect(policy)                                                 # no value_fn
    with pytest.raises(ValueError):
        col.collect(lambda o: actor(o)[0], value_fn)                        # actions only
    with pytest.raises(ValueError):
        stg.RolloutCollector(stg.make("SpinTorque-v0", num_envs=64, device=cuda_device, autoreset=False), 4, store_values=True)
    with pytest.raises(ValueError):
        stg.RolloutCollector(stg.make("SpinTorque-v0", num_envs=64, device=cuda_device, host_outputs=True), 4,
                             store_values=True)
