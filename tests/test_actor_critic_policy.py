"""K9: ActorCriticPolicy on the GPU (stg_policy_act_f32 / stg_policy_value_f32, stg.ActorCriticPolicy, the fused rollout path).

The specification is Stable-Baselines3's ActorCriticPolicy for PPO's MlpPolicy with a DiagGaussianDistribution, restated below
in NumPy float64 as SB3 and torch write it. The kernel's forward pass is FP32 fma chains, compared within 1e-5; sampling is
Philox4x32-10 + llgs_core.cuh's Box-Muller at counter (global env id, draw), restated in NumPy; the rescale to the env's Box
is compared bit for bit against its float32 restatement."""
import ctypes as C
import math
import os
import subprocess

import numpy as np
import pytest

from spin_torque_rl_gym_b200 import _lib
from tests.helpers import ROOT

HEADER = os.path.join(ROOT, "include", "stg.h")
CSRC = os.path.join(ROOT, "spin_torque_rl_gym_b200", "csrc")
M32 = 0xFFFFFFFF

# the state_dict keys of stable_baselines3's ActorCriticPolicy for PPO('MlpPolicy') on a Box action space, in its order
SB3_KEYS = ["log_std",
            "mlp_extractor.policy_net.0.weight", "mlp_extractor.policy_net.0.bias",
            "mlp_extractor.policy_net.2.weight", "mlp_extractor.policy_net.2.bias",
            "mlp_extractor.value_net.0.weight", "mlp_extractor.value_net.0.bias",
            "mlp_extractor.value_net.2.weight", "mlp_extractor.value_net.2.bias",
            "action_net.weight", "action_net.bias", "value_net.weight", "value_net.bias"]


# ---------------------------------------------------------------------------------------------------- SB3, restated -------

def sb3_forward(sd, obs):
    """SB3's MlpPolicy forward in float64: (mean_actions [N,2], values [N])."""
    g = {k: np.asarray(v, np.float64) for k, v in sd.items()}
    x = np.asarray(obs, np.float64)
    pi = np.tanh(x @ g["mlp_extractor.policy_net.0.weight"].T + g["mlp_extractor.policy_net.0.bias"])
    pi = np.tanh(pi @ g["mlp_extractor.policy_net.2.weight"].T + g["mlp_extractor.policy_net.2.bias"])
    vf = np.tanh(x @ g["mlp_extractor.value_net.0.weight"].T + g["mlp_extractor.value_net.0.bias"])
    vf = np.tanh(vf @ g["mlp_extractor.value_net.2.weight"].T + g["mlp_extractor.value_net.2.bias"])
    return pi @ g["action_net.weight"].T + g["action_net.bias"], (vf @ g["value_net.weight"].T + g["value_net.bias"])[:, 0]


def diag_gaussian_log_prob(mean, log_std, actions):
    """DiagGaussianDistribution.log_prob: torch's Normal.log_prob summed over the action dimensions."""
    std = np.exp(log_std)
    return (-((actions - mean) ** 2) / (2 * std ** 2) - np.log(std) - math.log(math.sqrt(2 * math.pi))).sum(1)


def diag_gaussian_entropy(log_std, n):
    """DiagGaussianDistribution.entropy: torch's Normal.entropy summed over the action dimensions."""
    return np.full(n, (0.5 + 0.5 * math.log(2 * math.pi) + np.asarray(log_std, np.float64)).sum())


def rescale_f32(a, lo, hi):
    """Clip to [-1, 1], then gymnasium's RescaleAction, in float32 with each operation rounded on its own."""
    a, lo, hi = np.asarray(a, np.float32), np.asarray(lo, np.float32), np.asarray(hi, np.float32)
    c = np.clip(a, np.float32(-1), np.float32(1))
    return lo + (hi - lo) * ((c + np.float32(1)) / np.float32(2))


def philox(k0, k1, c0, c1, c2, c3):
    """Philox4x32-10 over uint64 arrays holding 32-bit words (llgs_core.cuh's Philox)."""
    c0, c1, c2, c3 = (np.asarray(c, np.uint64) & np.uint64(M32) for c in (c0, c1, c2, c3))
    k0, k1 = int(k0), int(k1)
    for _ in range(10):
        p0 = np.uint64(0xD2511F53) * c0
        p1 = np.uint64(0xCD9E8D57) * c2
        h0, l0, h1, l1 = p0 >> np.uint64(32), p0 & np.uint64(M32), p1 >> np.uint64(32), p1 & np.uint64(M32)
        c0, c1, c2, c3 = h1 ^ c1 ^ np.uint64(k0), l1, h0 ^ c3 ^ np.uint64(k1), l0
        k0, k1 = (k0 + 0x9E3779B9) & M32, (k1 + 0xBB67AE85) & M32
    return c0, c1, c2, c3


def host_eps(key, gids, draw):
    """The two normals of each env (box_muller of Philox words 0 and 1 at counter (gid lo, gid hi, draw lo, draw hi)), with
    the float32 roundings of the uniform and of the angle restated and the transcendental functions in float64."""
    gids = np.asarray(gids, np.uint64)
    w0, w1, _, _ = philox(key[0], key[1], gids, gids >> np.uint64(32), np.full_like(gids, draw & M32),
                          np.full_like(gids, draw >> 32))
    a = (w0.astype(np.float32).astype(np.float64) * 2.0 ** -32 + 2.0 ** -33).astype(np.float32).astype(np.float64)
    r = np.sqrt(-2.0 * np.log(a))
    twopi = np.float64(np.float32(6.283185307179586))
    f = 1.0 + (w1 >> np.uint64(9)).astype(np.float64) * 2.0 ** -23
    ang = (f * twopi - twopi).astype(np.float32).astype(np.float64)
    return np.stack([r * np.cos(ang), r * np.sin(ang)], 1)


# ---------------------------------------------------------------------------------------------------- host build ----------

@pytest.fixture(scope="module")
def host_core(tmp_path_factory):
    """policy_core.cuh compiled for the host with g++."""
    d = tmp_path_factory.mktemp("policy_host")
    src = d / "policy_host.cpp"
    src.write_text('#include "policy_core.cuh"\n'
                   'using namespace stg;\n'
                   'extern "C" void forward(const float* w, const float* obs, int64_t n, uint32_t k0, uint32_t k1,\n'
                   '                        uint64_t offset, uint64_t draw, int sample, float* mean, float* act, float* value,\n'
                   '                        float* logp) {\n'
                   '  for (int64_t i = 0; i < n; ++i)\n'
                   '    pol_forward_row(w, obs + 12 * i, k0, k1, offset + i, draw, sample != 0, mean + 2 * i, act + 2 * i,\n'
                   '                    value[i], logp[i]); }\n'
                   'extern "C" void eps(uint32_t k0, uint32_t k1, uint64_t gid0, int64_t n, uint64_t draw, float* out) {\n'
                   '  for (int64_t i = 0; i < n; ++i) pol_eps(k0, k1, gid0 + i, draw, out[2 * i], out[2 * i + 1]); }\n'
                   'extern "C" void rescale(const float* a, int64_t n, const float* lo, const float* hi, float* out) {\n'
                   '  for (int64_t i = 0; i < 2 * n; ++i) out[i] = pol_rescale(a[i], lo[i & 1], hi[i & 1]); }\n')
    so = d / "policy_host.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-I", CSRC, str(src), "-o", str(so)], check=True)
    lib = C.CDLL(str(so))
    dp, i64, u32, u64 = C.c_void_p, C.c_int64, C.c_uint32, C.c_uint64
    lib.forward.argtypes = [dp, dp, i64, u32, u32, u64, u64, C.c_int, dp, dp, dp, dp]
    lib.eps.argtypes = [u32, u32, u64, i64, u64, dp]
    lib.rescale.argtypes = [dp, i64, dp, dp, dp]
    return lib


def _p(a):
    return a.ctypes.data


def host_draws(lib, key, gid0, n, draw):
    out = np.empty((n, 2), np.float32)
    lib.eps(key[0], key[1], gid0, n, draw, _p(out))
    return out


class FakeEnv:
    """What ActorCriticPolicy reads from an env, on the CPU (the torch methods need no GPU)."""

    def __init__(self, n=8, obs_dim=12, act_dim=2, device="cpu"):
        from spin_torque_rl_gym_b200.spaces import Box
        self.num_envs, self.device, self.env_offset, self.rng_seed = n, device, 0, 7
        self.single_observation_space = Box(low=-np.inf, high=np.inf, shape=(obs_dim,), dtype=np.float32)
        hi = np.array([2e6, 5e-9][:act_dim] + [1.0] * max(0, act_dim - 2))
        lo = np.array([-2e6, 0.0][:act_dim] + [-1.0] * max(0, act_dim - 2))
        self.single_action_space = Box(low=lo, high=hi, dtype=np.float32)


def _random_policy(env, seed, log_std=(-0.4, 0.3)):
    """A policy with SB3's initialisation, then every parameter perturbed, so no layer is near its orthogonal init."""
    import torch
    import spin_torque_rl_gym_b200 as stg
    torch.manual_seed(seed)
    pol = stg.ActorCriticPolicy(env)
    with torch.no_grad():
        for name, p in pol.named_parameters():
            if name != "log_std":
                p.add_(torch.randn_like(p) * 0.2)
        pol.log_std.copy_(torch.tensor(log_std))
    return pol


def _packed_numpy(pol):
    """The STG_POLICY_* buffer of a CPU module, built independently of pack_weights."""
    sd = {k: v.detach().cpu().numpy().astype(np.float32) for k, v in pol.state_dict().items()}
    L = _lib.POLICY_LAYOUT
    w = np.zeros(_lib.POLICY_FLOATS, np.float32)
    for pre, net in (("PI", "policy_net"), ("VF", "value_net")):
        w[L[pre + "_W1"]:L[pre + "_W1"] + 768] = sd[f"mlp_extractor.{net}.0.weight"].T.ravel()
        w[L[pre + "_B1"]:L[pre + "_B1"] + 64] = sd[f"mlp_extractor.{net}.0.bias"]
        w[L[pre + "_W2"]:L[pre + "_W2"] + 4096] = sd[f"mlp_extractor.{net}.2.weight"].T.ravel()
        w[L[pre + "_B2"]:L[pre + "_B2"] + 64] = sd[f"mlp_extractor.{net}.2.bias"]
    w[L["ACT_W"]:L["ACT_W"] + 128] = sd["action_net.weight"].T.ravel()
    w[L["ACT_B"]:L["ACT_B"] + 2] = sd["action_net.bias"]
    w[L["VAL_W"]:L["VAL_W"] + 64] = sd["value_net.weight"].ravel()
    w[L["VAL_B"]] = sd["value_net.bias"][0]
    w[L["LOG_STD"]:L["LOG_STD"] + 2] = sd["log_std"]
    std = np.exp(sd["log_std"]).astype(np.float32)
    w[L["STD"]:L["STD"] + 2] = std
    w[L["LOG_SCALE"]:L["LOG_SCALE"] + 2] = np.log(std).astype(np.float32)
    return w, sd


# ---------------------------------------------------------------------------------------------------- CPU ---------------

def test_core_forward_matches_the_sb3_restatement(host_core):
    pol = _random_policy(FakeEnv(), 0)
    w, sd = _packed_numpy(pol)
    packed = pol.pack_weights().numpy()                                     # the torch.cat packing, here on the CPU
    L = _lib.POLICY_LAYOUT
    assert np.array_equal(packed[:L["STD"]], w[:L["STD"]]) and not packed[L["LOG_SCALE"] + 2:].any()
    assert np.allclose(packed[L["STD"]:], w[L["STD"]:], rtol=1e-6, atol=0)
    rng = np.random.default_rng(0)
    n = 5000
    obs = (rng.normal(size=(n, 12)) * rng.choice([0.1, 1.0, 3.0], size=(n, 12))).astype(np.float32)
    mean, act, val, lp = (np.empty((n, 2), np.float32), np.empty((n, 2), np.float32), np.empty(n, np.float32),
                          np.empty(n, np.float32))
    key = (0x12345678, 0x9ABCDEF0)
    ref_mean, ref_val = sb3_forward(sd, obs)
    for sample in (0, 1):
        host_core.forward(_p(w), _p(obs), n, key[0], key[1], 100, 3, sample, _p(mean), _p(act), _p(val), _p(lp))
        assert np.abs(mean - ref_mean).max() <= 1e-5
        assert np.abs(val - ref_val).max() <= 1e-5
        assert np.abs(lp - diag_gaussian_log_prob(ref_mean, sd["log_std"], act.astype(np.float64))).max() <= 1e-5
        if sample:
            eps = host_draws(host_core, key, 100, n, 3)
            assert np.abs((act - mean.astype(np.float64)) / np.exp(sd["log_std"].astype(np.float64)) - eps).max() <= 1e-5
            assert np.array_equal(act, (mean + eps * w[_lib.POLICY_LAYOUT["STD"]:][:2]).astype(np.float32))
        else:
            assert np.array_equal(act, mean)


def test_host_restatement_of_the_draws_matches_the_core(host_core):
    key = (0xDEADBEEF, 0x01234567)
    for gid0, draw in ((0, 0), ((1 << 32) - 3, 5), (1 << 40, (1 << 33) + 1)):
        got = host_draws(host_core, key, gid0, 1000, draw)
        want = host_eps(key, np.arange(1000, dtype=np.uint64) + np.uint64(gid0), draw)
        assert np.abs(got - want).max() <= 1e-5


def test_noise_draws_are_standard_normal_and_uncorrelated(host_core):
    from scipy import stats
    from spin_torque_rl_gym_b200.policy import policy_noise_key
    key = policy_noise_key(11)
    e = host_draws(host_core, key, 0, 500_000, 0)
    x = e.ravel().astype(np.float64)                                         # 10^6 draws
    assert abs(x.mean()) < 5e-3 and abs(x.var() - 1.0) < 5e-3
    assert stats.kstest(x, "norm").pvalue > 1e-3
    lim = 6 / math.sqrt(len(e))
    assert abs(np.corrcoef(e[:-1, 0], e[1:, 0])[0, 1]) < lim                 # neighbouring gids
    assert abs(np.corrcoef(e[:, 0], e[:, 1])[0, 1]) < lim                    # the two dimensions of one env
    nxt = host_draws(host_core, key, 0, 500_000, 1)
    assert abs(np.corrcoef(e[:, 0], nxt[:, 0])[0, 1]) < lim                  # consecutive draws
    assert abs(np.corrcoef(e[:, 1], nxt[:, 1])[0, 1]) < lim


def test_noise_key_known_answers_and_domain_separation():
    from spin_torque_rl_gym_b200.policy import POLICY_NOISE_TAG, policy_noise_key
    from spin_torque_rl_gym_b200.envs.sb3_vec_env import _splitmix64
    assert _splitmix64(0)[1] == 0xE220A8397B1DCDAF                            # splitmix64's published first output
    assert POLICY_NOISE_TAG == 0x316573696F6E394B                            # b"K9noise1", little-endian
    assert policy_noise_key(0) == (0xACA1DA2B, 0x52F1B053)
    assert policy_noise_key(12345) == (0xEE69D2F4, 0x9EDA0AEE)
    assert policy_noise_key((1 << 64) - 1) == policy_noise_key(-1)
    keys = set()
    for seed in list(range(2000)) + [(1 << 64) - 1, 1 << 63]:
        k = policy_noise_key(seed)
        assert k != (seed & M32, (seed >> 32) & M32)                        # the env's thermal / reset key
        keys.add(k)
    assert len(keys) == 2002


def test_evaluate_actions_and_entropy_match_the_sb3_restatement():
    import torch
    pol = _random_policy(FakeEnv(), 1)
    sd = {k: v.detach().numpy() for k, v in pol.state_dict().items()}
    rng = np.random.default_rng(1)
    obs = rng.normal(size=(300, 12)).astype(np.float32)
    act = (rng.normal(size=(300, 2)) * 2).astype(np.float32)
    values, log_prob, entropy = pol.evaluate_actions(torch.from_numpy(obs), torch.from_numpy(act))
    assert values.shape == (300, 1) and log_prob.shape == (300,) and entropy.shape == (300,)
    assert log_prob.requires_grad and values.requires_grad                  # PPO trains through it
    ref_mean, ref_val = sb3_forward(sd, obs)
    assert np.abs(values.detach().numpy()[:, 0] - ref_val).max() <= 1e-5
    assert np.abs(log_prob.detach().numpy() - diag_gaussian_log_prob(ref_mean, sd["log_std"], act)).max() <= 1e-5
    assert np.abs(entropy.detach().numpy() - diag_gaussian_entropy(sd["log_std"], 300)).max() <= 1e-5
    dist = pol.get_distribution(torch.from_numpy(obs))
    assert np.abs(dist.mode().detach().numpy() - ref_mean).max() <= 1e-5
    env_act, state = pol.predict(torch.from_numpy(obs), deterministic=True)
    assert state is None
    assert np.array_equal(env_act.numpy(), rescale_f32(dist.mode().detach().numpy(), [-2e6, 0], [2e6, 5e-9]))
    assert np.array_equal(pol.scale_action(torch.from_numpy(act)).numpy(), rescale_f32(act, [-2e6, 0], [2e6, 5e-9]))


def test_rescale_of_the_core_is_the_float32_restatement(host_core):
    rng = np.random.default_rng(2)
    a = np.concatenate([rng.normal(size=(10000, 2)) * 1.5, [[-1, 1], [1, -1], [0, 0], [-0.0, 1e-30], [5, -5]]])
    a = a.astype(np.float32)
    lo, hi = np.array([-2e6, 0], np.float32), np.array([2e6, 5e-9], np.float32)
    out = np.empty_like(a)
    host_core.rescale(_p(a), len(a), _p(lo), _p(hi), _p(out))
    assert np.array_equal(out, rescale_f32(a, lo, hi))
    assert out[:, 0].min() == -2e6 and out[:, 1].min() == 0 and out[:, 1].max() == np.float32(5e-9)


def test_state_dict_is_sb3s_and_only_the_default_architecture_is_accepted():
    import torch
    from torch import nn
    import spin_torque_rl_gym_b200 as stg
    pol = stg.ActorCriticPolicy(FakeEnv())
    sd = pol.state_dict()
    assert list(sd) == SB3_KEYS
    shapes = {k: tuple(v.shape) for k, v in sd.items()}
    assert shapes["mlp_extractor.policy_net.0.weight"] == (64, 12) and shapes["action_net.weight"] == (2, 64)
    assert shapes["value_net.weight"] == (1, 64) and shapes["log_std"] == (2,)
    assert sum(v.numel() for v in sd.values()) == _lib.POLICY_PARAMS == 10181
    other = _random_policy(FakeEnv(), 3)
    pol.load_state_dict(other.state_dict(), strict=True)
    assert all(torch.equal(a, b) for a, b in zip(pol.state_dict().values(), other.state_dict().values()))
    # SB3's initialisation: orthogonal with gains sqrt(2) / 0.01 / 1, zero biases, log_std = log_std_init
    torch.manual_seed(0)
    init = stg.ActorCriticPolicy(FakeEnv(), log_std_init=-0.5)
    w = init.mlp_extractor.value_net[2].weight.detach()
    assert torch.allclose(w @ w.T, 2 * torch.eye(64), atol=1e-5)
    a = init.action_net.weight.detach()
    assert torch.allclose(a @ a.T, 1e-4 * torch.eye(2), atol=1e-9)
    assert torch.allclose(init.value_net.weight.detach().norm(), torch.tensor(1.0))
    assert all(float(b.detach().abs().max()) == 0 for n_, b in init.named_parameters() if n_.endswith("bias"))
    assert torch.equal(init.log_std.detach(), torch.full((2,), -0.5))
    torch.manual_seed(0)
    again = stg.ActorCriticPolicy(FakeEnv(), log_std_init=-0.5)
    assert all(torch.equal(x, y) for x, y in zip(init.state_dict().values(), again.state_dict().values()))
    # the defaults spelled out are accepted; anything else is not
    stg.ActorCriticPolicy(FakeEnv(), net_arch=dict(pi=[64, 64], vf=[64, 64]), activation_fn=nn.Tanh)
    for kw in (dict(net_arch=dict(pi=[32, 32], vf=[32, 32])), dict(net_arch=dict(pi=[64, 64, 64], vf=[64, 64, 64])),
               dict(net_arch=dict(pi=[64, 64], vf=[128, 128])), dict(net_arch=[256, 256]), dict(activation_fn=nn.ReLU)):
        with pytest.raises(ValueError):
            stg.ActorCriticPolicy(FakeEnv(), **kw)
    for env in (FakeEnv(obs_dim=13), FakeEnv(act_dim=3)):
        with pytest.raises(ValueError):
            stg.ActorCriticPolicy(env)
    # the product path is CUDA-only
    with pytest.raises(_lib.StgError):
        pol(torch.zeros(4, 12))
    with pytest.raises(_lib.StgError):
        pol.predict_values(torch.zeros(4, 12))


def test_policy_args_layout_and_constants_match_the_c_header(tmp_path):
    fields = [f for f, _ in _lib.StgPolicyArgs._fields_]
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', 'int main(void){',
             'printf("size %zu\\n", sizeof(StgPolicyArgs));']
    lines += [f'printf("{f} %zu\\n", offsetof(StgPolicyArgs, {f}));' for f in fields]
    consts = {f"STG_POLICY_{k}": v for k, v in _lib.POLICY_LAYOUT.items()}
    consts.update(STG_POLICY_PARAMS=_lib.POLICY_PARAMS, STG_POLICY_FLOATS=_lib.POLICY_FLOATS,
                  STG_POLICY_DETERMINISTIC=_lib.POLICY_DETERMINISTIC, STG_POLICY_OBS=12, STG_POLICY_HIDDEN=64,
                  STG_POLICY_ACTIONS=2, STG_ABI_VERSION=7)
    lines += [f'printf("{c} %lld\\n", (long long)({c}));' for c in consts]
    lines.append('return 0;}')
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", str(src), "-o", str(exe)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split("\n") if l)
    assert int(got["size"]) == C.sizeof(_lib.StgPolicyArgs)
    for f in fields:
        assert int(got[f]) == getattr(_lib.StgPolicyArgs, f).offset, f
    for c, v in consts.items():
        assert int(got[c]) == v, c
    L = _lib.POLICY_LAYOUT                                                  # the layout is dense, in SB3's parameter order
    sizes = [768, 64, 4096, 64, 768, 64, 4096, 64, 128, 2, 64, 1, 2, 2, 2]
    assert list(L.values()) == list(np.cumsum([0] + sizes[:-1]))
    assert L["LOG_SCALE"] + 2 <= _lib.POLICY_FLOATS and _lib.POLICY_FLOATS % 4 == 0
    assert all(L[k] % 4 == 0 for k in ("PI_W1", "PI_B1", "PI_W2", "PI_B2", "VF_W1", "VF_B1", "VF_W2", "VF_B2"))


def _pargs(n=4, **ptrs):
    a = _lib.StgPolicyArgs()
    a.n_envs = n
    for k, v in ptrs.items():
        setattr(a, k, v)
    return a


def test_policy_argument_validation():
    lib = _lib.load()
    act, val = lib.stg_policy_act_f32, lib.stg_policy_value_f32
    call = lambda f, a: f(C.byref(a), None)                                 # noqa: E731
    B = 0x10000
    for f in (act, val):
        assert f(None, None) == -1                                          # STG_E_NULL
        assert call(f, _pargs(-1, d_obs=B, d_weights=B, d_value=B)) == -2   # STG_E_SIZE
        assert call(f, _pargs(0)) == 0                                      # empty: STG_OK without a launch
        assert call(f, _pargs(d_weights=B, d_value=B)) == -1
        assert call(f, _pargs(d_obs=B, d_value=B)) == -1
        ok = dict(d_obs=B, d_weights=B * 2, d_value=B * 3)
        for field, off in (("d_obs", 4), ("d_weights", 8)):
            assert call(f, _pargs(**dict(ok, **{field: ok[field] + off}))) == -4, field   # STG_E_ALIGN
        assert call(f, _pargs(flags=2, **ok)) == -3                         # STG_E_ENUM
    assert call(act, _pargs(d_obs=B, d_weights=B)) == -1                    # no output at all
    assert call(val, _pargs(d_obs=B, d_weights=B, d_log_prob=B)) == -1      # the critic needs d_value
    base = dict(d_obs=B, d_weights=B, d_log_prob=B)
    assert call(act, _pargs(d_obs_copy=B + 4, **base)) == -4
    assert call(act, _pargs(d_action=B + 4, **base)) == -4
    assert call(act, _pargs(d_env_action=B + 12, **base)) == -4


def test_plain_collector_refuses_an_actor_critic_policy():
    import spin_torque_rl_gym_b200 as stg
    col = stg.RolloutCollector.__new__(stg.RolloutCollector)
    col.store_values = False
    with pytest.raises(ValueError):
        col.collect(stg.ActorCriticPolicy(FakeEnv()))


# ---------------------------------------------------------------------------------------------------- GPU ---------------

def _venv(stg, dev, n, max_steps=100, seed=5, **kw):
    return stg.make("SpinTorque-v0", num_envs=n, device=dev, max_steps=max_steps, rng_seed=seed, **kw)


def _obs(torch, dev, n, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    scale = torch.tensor([0.3, 1.0, 3.0] * 4, device=dev)
    return torch.randn(n, 12, generator=g, device=dev) * scale


def _torch_layers(pol, obs):
    """The module's own torch layers: (mean_actions [N,2], values [N])."""
    import torch
    with torch.no_grad():
        latent_pi, latent_vf = pol.mlp_extractor(obs)
        return pol.action_net(latent_pi), pol.value_net(latent_vf)[:, 0]


def _act_launch(pol, obs, draw, env_offset=None, deterministic=False):
    """One stg_policy_act_f32 launch with every output: (action, env_action, value, log_prob)."""
    import torch
    n = obs.shape[0]
    out = [torch.empty(n, 2, device=obs.device), torch.empty(n, 2, device=obs.device), torch.empty(n, device=obs.device),
           torch.empty(n, device=obs.device)]
    a = pol._args(pol.pack_weights(), n)
    a.d_obs, a.d_action, a.d_env_action = obs.data_ptr(), out[0].data_ptr(), out[1].data_ptr()
    a.d_value, a.d_log_prob, a.draw = out[2].data_ptr(), out[3].data_ptr(), draw
    if env_offset is not None:
        a.env_offset = env_offset
    a.flags = _lib.POLICY_DETERMINISTIC if deterministic else 0
    pol._launch(_lib.load().stg_policy_act_f32, a, "stg_policy_act_f32")
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 33, 4097, 131072, 1048576])
def test_cuda_kernel_matches_the_torch_layers(cuda_device, n):
    import torch
    import spin_torque_rl_gym_b200 as stg
    dev = cuda_device
    env = _venv(stg, dev, 1)
    pol = _random_policy(env, 4)
    obs = _obs(torch, dev, n, n)
    mean_t, val_t = _torch_layers(pol, obs)
    det_a, det_v, det_lp = pol(obs, deterministic=True)
    assert pol.noise_draws == 0
    actions, values, log_probs = pol(obs)
    assert pol.noise_draws == 1
    assert actions.shape == (n, 2) and values.shape == (n, 1) and log_probs.shape == (n,)
    assert not (actions.requires_grad or values.requires_grad or log_probs.requires_grad)
    assert float((values[:, 0] - val_t).abs().max()) <= 1e-5
    assert float((det_a - mean_t).abs().max()) <= 1e-5                     # deterministic: the means
    assert torch.equal(det_v, values)
    std = pol.log_std.detach().exp().double()
    eps = (actions.double() - det_a.double()) / std
    want = host_eps(pol.noise_key(), np.arange(n, dtype=np.uint64) + np.uint64(env.env_offset), 0)
    # box_muller takes the radius from lg2.approx (absolute error <= 2^-22): r^2 = -2 ln2 lg2(u) is off by up to 2.2e-7, so
    # r by up to 1.1e-7 / r, which exceeds 1e-5 in the rare rows with r < 0.011 (about 6e-5 of them)
    err = np.abs(eps.cpu().numpy() - want)
    r = np.hypot(want[:, 0], want[:, 1])[:, None]
    assert bool((err <= 1e-5 + 2e-7 / r).all())
    assert float(np.median(err)) <= 1e-6 and float((err > 1e-5).mean()) <= 1e-4
    with torch.no_grad():
        _, lp_t, _ = pol.evaluate_actions(obs, actions)
        _, lp_det, _ = pol.evaluate_actions(obs, det_a)
    assert float((log_probs - lp_t).abs().max()) <= 1e-5
    assert float((det_lp - lp_det).abs().max()) <= 1e-5
    # the env actions of a launch with every output are the float32 rescale of its raw actions, bit for bit
    act, env_act, val, lp = _act_launch(pol, obs, 1)
    assert torch.equal(act, pol(obs)[0]) and torch.equal(val, values[:, 0])
    lo, hi = env.single_action_space.low, env.single_action_space.high
    assert np.array_equal(env_act.cpu().numpy(), rescale_f32(act.cpu().numpy(), lo, hi))
    assert torch.equal(env_act, pol.scale_action(act))
    if n > 1000:
        assert float(act.abs().max()) > 1.0                                  # the clip is exercised


@pytest.mark.gpu
def test_cuda_samples_are_invariant_to_sharding_and_reproduce(cuda_device):
    import torch
    import spin_torque_rl_gym_b200 as stg
    dev, n, parts = cuda_device, 1 << 20, 4
    env = _venv(stg, dev, 1, seed=21)
    pol = _random_policy(env, 5)
    obs = _obs(torch, dev, n, 9)
    whole = _act_launch(pol, obs, 7)
    m = n // parts
    shards = [_act_launch(pol, obs[k * m:(k + 1) * m].clone(), 7, env_offset=k * m) for k in range(parts)]
    for q in range(4):
        assert torch.equal(whole[q], torch.cat([s[q] for s in shards]))
    # the same seed and weights reproduce; the next draw differs
    twin = stg.ActorCriticPolicy(env, seed=21)
    twin.load_state_dict(pol.state_dict())
    assert twin.noise_key() == pol.noise_key()
    a1, v1, l1 = pol(obs[:4096])
    b1, w1, k1 = twin(obs[:4096])
    assert torch.equal(a1, b1) and torch.equal(v1, w1) and torch.equal(l1, k1)
    a2 = pol(obs[:4096])[0]
    assert not torch.equal(a1, a2) and float((a1 - a2).abs().mean()) > 0.5
    other = stg.ActorCriticPolicy(env, seed=22)
    other.load_state_dict(pol.state_dict())
    assert not torch.equal(other(obs[:4096])[0], a1)


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 4097, 100003])
def test_cuda_masked_value_writes_exactly_the_masked_rows(cuda_device, n):
    import torch
    import spin_torque_rl_gym_b200 as stg
    dev = cuda_device
    pol = _random_policy(_venv(stg, dev, 1), 6)
    obs = _obs(torch, dev, n, 3)
    full = pol.predict_values(obs)
    _, ref = _torch_layers(pol, obs)
    assert full.shape == (n, 1) and float((full[:, 0] - ref).abs().max()) <= 1e-5
    g = torch.Generator(device=dev).manual_seed(n)
    for p in (0.0, 0.02, 0.5, 1.0):
        mask = torch.rand(n, generator=g, device=dev) < p
        for dtype in (torch.bool, torch.uint8):
            out = torch.full((n,), float("nan"), device=dev)
            assert pol.predict_values(obs, mask=mask.to(dtype), out=out) is out
            assert torch.equal(out[mask], full[mask, 0])
            assert bool(out[~mask].isnan().all())
    assert bool(pol.predict_values(obs, mask=torch.zeros(n, dtype=torch.bool, device=dev)).isnan().all())


def _ppo_env(stg, dev, n, max_steps):
    return stg.VecNormalize(_venv(stg, dev, n, max_steps=max_steps))


@pytest.mark.gpu
def test_cuda_fused_collector_on_vec_normalize(cuda_device, monkeypatch):
    import torch
    import spin_torque_rl_gym_b200 as stg
    from spin_torque_rl_gym_b200.envs import sb3_vec_env
    dev, n, T = cuda_device, 4096, 12
    norm = _ppo_env(stg, dev, n, 5)
    pol = _random_policy(norm, 7)
    rec = []
    venv_step, norm_step = norm.venv.step, norm.step

    def recording_venv_step(actions, noise=None):
        rec.append({"env_action": actions.clone()})
        return venv_step(actions)

    def recording_norm_step(actions):
        out = norm_step(actions)
        rec[-1].update(final=out[4]["final_observation"].clone(), done=(out[2] | out[3]).clone(), obs=out[0].clone())
        return out

    norm.venv.step, norm.step = recording_venv_step, recording_norm_step
    col = stg.RolloutCollector(norm, n_steps=T, store_values=True)
    with pytest.raises(ValueError):
        stg.RolloutCollector(norm, n_steps=2).collect(pol)                  # store_values=False
    torch.cuda.synchronize()
    # the episode statistics collect() returns are read on the host once per rollout; everything before them must not sync
    monkeypatch.setattr(sb3_vec_env, "all_reduce_stats", lambda stats: stats)
    torch.cuda.set_sync_debug_mode("error")
    try:
        col.collect(pol)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert len(rec) == T and pol.noise_draws == T
    lo, hi = norm.single_action_space.low, norm.single_action_space.high
    ended = 0
    for t in range(T):
        r = rec[t]
        # actions[t] are the raw samples; the env stepped on their rescale
        assert np.array_equal(r["env_action"].cpu().numpy(), rescale_f32(col.actions[t].cpu().numpy(), lo, hi))
        with torch.no_grad():
            v, lp, _ = pol.evaluate_actions(col.observations[t], col.actions[t])
        assert float((v[:, 0] - col.values[t]).abs().max()) <= 1e-5
        assert float((lp - col.log_probs[t]).abs().max()) <= 1e-5
        done = r["done"]
        assert torch.equal(col.dones[t], done)
        if bool(done.any()):
            _, fv = _torch_layers(pol, r["final"][done])
            assert float((col.final_values[t][done] - fv).abs().max()) <= 1e-5
        ended += int(done.sum())
        if t + 1 < T:
            assert torch.equal(col.observations[t + 1], r["obs"])
    assert ended > 0
    # the env's last_action plane holds the (clamped) env actions of the last step where the episode did not end
    la = norm.venv._last_action.cpu().numpy()
    ea = rec[-1]["env_action"].cpu().numpy().astype(np.float64)
    keep = ~rec[-1]["done"].cpu().numpy()
    assert np.array_equal(la[0][keep], np.clip(ea[keep, 0], -norm.max_current, norm.max_current))
    assert np.array_equal(la[1][keep], np.clip(ea[keep, 1], 1e-12, norm.max_duration))
    _, lv = _torch_layers(pol, rec[-1]["obs"])
    assert float((col.last_values - lv).abs().max()) <= 1e-5


@pytest.mark.gpu
def test_cuda_ppo_iteration(cuda_device):
    import torch
    import spin_torque_rl_gym_b200 as stg
    dev, n, T = cuda_device, 8192, 8
    norm = _ppo_env(stg, dev, n, 4)
    torch.manual_seed(0)
    pol = stg.ActorCriticPolicy(norm, log_std_init=-0.5)
    opt = torch.optim.Adam(pol.parameters(), lr=3e-4, eps=1e-5)
    col = stg.RolloutCollector(norm, n_steps=T, store_values=True)
    col.collect(pol)
    col.compute_returns_and_advantage(gamma=0.99, gae_lambda=0.95)
    first = True
    for batch in col.get(4096):
        values, log_prob, entropy = pol.evaluate_actions(batch.observations, batch.actions)
        ratio = torch.exp(log_prob - batch.old_log_prob)
        if first:
            assert float((ratio - 1).abs().max().detach()) <= 1e-5         # the rollout's log-probs are the training ones
            assert float((values[:, 0] - batch.old_values).abs().max().detach()) <= 1e-5
            first = False
        adv = (batch.advantages - batch.advantages.mean()) / (batch.advantages.std() + 1e-8)
        policy_loss = -torch.min(adv * ratio, adv * torch.clamp(ratio, 0.8, 1.2)).mean()
        loss = policy_loss + 0.5 * torch.nn.functional.mse_loss(batch.returns, values[:, 0]) - 0.0 * entropy.mean()
        opt.zero_grad()
        loss.backward()
        opt.step()
    before = col.values[0].clone()
    obs0 = col._last_obs.clone()
    col.collect(pol)                                                        # repacks: the updated weights
    _, v_new = _torch_layers(pol, col.observations[0])
    assert torch.equal(col.observations[0], obs0)
    assert float((col.values[0] - v_new).abs().max()) <= 1e-5
    assert not torch.equal(col.values[0], before)
    with torch.no_grad():
        _, lp, _ = pol.evaluate_actions(col.observations[T - 1], col.actions[T - 1])
    assert float((lp - col.log_probs[T - 1]).abs().max()) <= 1e-5
