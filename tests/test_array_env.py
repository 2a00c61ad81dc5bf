"""K3 SpinTorqueArray-v0: oracle pinned bit-exactly to the live-reference goldens; the kernel's arithmetic (host build on CPU,
CUDA kernel on the GPU) against both. FP64, tolerance 1e-9 (the sums follow NumPy's order, so it is usually bit-identical)."""
import ctypes as C
import os

import numpy as np
import pytest

from oracle.array_oracle import ArrayOracleEnv
from spin_torque_rl_gym_b200 import _lib
from tests.helpers import GOLDEN

G = np.load(os.path.join(GOLDEN, "array_env.npz"))
CASES = {"ind8": ((8, 8), "individual", {}), "row8": ((8, 8), "row", {}), "col8": ((8, 8), "column", {}),
         "glob8": ((8, 8), "global", {}),
         "stray35": ((3, 5), "row", dict(coupling_type="stray_field", coupling_strength=0.25, max_steps=10))}


@pytest.mark.parametrize("name", list(CASES))
def test_oracle_bit_exact(name):
    size, mode, kw = CASES[name]
    env = ArrayOracleEnv(array_size=size, action_mode=mode, **kw)
    assert np.array_equal(env.coupling, G[f"{name}/coupling"])
    assert np.array_equal(env.reset(G[f"{name}/p0"]), G[f"{name}/obs"][0])
    for k, a in enumerate(G[f"{name}/actions"]):
        o, r, te, tr, info = env.step(a.copy())
        assert np.array_equal(env.pattern, G[f"{name}/pattern"][k + 1])
        assert np.array_equal(o, G[f"{name}/obs"][k + 1]) and r == G[f"{name}/reward"][k]
        assert te == G[f"{name}/terminated"][k] and tr == G[f"{name}/truncated"][k]
        assert info["energy"] == G[f"{name}/energy"][k] and info["similarity"] == G[f"{name}/similarity"][k]


def _host_env(size, mode, kw):
    """StgArrayStepArgs over NumPy buffers driven through tests/hostsim (same helpers as the CUDA kernel)."""
    from spin_torque_rl_gym_b200.envs.array_env import array_params, compute_coupling_matrix
    from spin_torque_rl_gym_b200 import params as P
    from tests.hostsim.harness import lib
    D = size[0] * size[1]
    p = array_params(size, "stt_mram", P.default_device_parameters("stt_mram"), mode, kw.get("max_steps", 200), 2e6, 5e-9,
                     0.9, 0.1)
    coup = compute_coupling_matrix(size[0], size[1], kw.get("coupling_strength", 0.1), kw.get("coupling_type", "dipolar"))
    st = dict(coup=np.ascontiguousarray(coup), pattern=np.zeros((1, D, 3)), target=np.zeros((1, D, 3)),
              te=np.zeros(1), sc=np.zeros(1, np.int32), ep=np.zeros(1, np.int32), obs=np.zeros((1, D, 6), np.float32),
              rew=np.zeros(1), term=np.zeros(1, np.uint8), trunc=np.zeros(1, np.uint8), en=np.zeros(1), sim=np.zeros(1))
    ii, jj = np.indices(size)
    st["target"][0, :, 2] = np.where((ii + jj) % 2 == 0, 1.0, -1.0).reshape(-1)

    def step(action):
        act = np.ascontiguousarray(action, np.float32)
        a = _lib.StgArrayStepArgs()
        a.params = p
        a.d_coupling, a.d_pattern, a.d_target = st["coup"].ctypes.data, st["pattern"].ctypes.data, st["target"].ctypes.data
        a.d_total_energy, a.d_step_count, a.d_episode = st["te"].ctypes.data, st["sc"].ctypes.data, st["ep"].ctypes.data
        a.d_action, a.d_obs, a.d_reward = act.ctypes.data, st["obs"].ctypes.data, st["rew"].ctypes.data
        a.d_terminated, a.d_truncated = st["term"].ctypes.data, st["trunc"].ctypes.data
        a.d_step_energy, a.d_similarity = st["en"].ctypes.data, st["sim"].ctypes.data
        a.n_arrays, a.action_stride = 1, len(act)
        lib().hostsim_array_step(C.byref(a))
    return st, step, coup


@pytest.mark.parametrize("name", list(CASES))
def test_kernel_arithmetic_on_host(name):
    size, mode, kw = CASES[name]
    st, step, coup = _host_env(size, mode, kw)
    assert np.array_equal(coup, G[f"{name}/coupling"])
    st["pattern"][0] = G[f"{name}/p0"].reshape(-1, 3)
    for k, a in enumerate(G[f"{name}/actions"]):
        step(a)
        ref = G[f"{name}/pattern"][k + 1].reshape(-1, 3)
        assert np.abs(st["pattern"][0] - ref).max() < 1e-12, (name, k)
        assert np.array_equal(st["obs"][0].reshape(size + (6,)), G[f"{name}/obs"][k + 1])
        assert st["rew"][0] == pytest.approx(G[f"{name}/reward"][k], rel=1e-12)
        assert st["en"][0] == pytest.approx(G[f"{name}/energy"][k], rel=1e-12)
        assert st["sim"][0] == pytest.approx(G[f"{name}/similarity"][k], rel=1e-12, abs=1e-15)
        assert bool(st["term"][0]) == G[f"{name}/terminated"][k] and bool(st["trunc"][0]) == G[f"{name}/truncated"][k]


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(CASES))
def test_cuda_array_env_matches_reference(name, cuda_device):
    from spin_torque_rl_gym_b200 import SpinTorqueArrayVectorEnv
    size, mode, kw = CASES[name]
    n = 3                                    # the same episode in three arrays of the batch
    env = SpinTorqueArrayVectorEnv(num_envs=n, array_size=size, action_mode=mode, device=cuda_device, autoreset=False, **kw)
    assert np.array_equal(env.coupling_matrix, G[f"{name}/coupling"])
    obs, _ = env.reset(options={"initial_pattern": G[f"{name}/p0"]})
    assert np.array_equal(obs.cpu().numpy()[1], G[f"{name}/obs"][0])
    for k, a in enumerate(G[f"{name}/actions"]):
        o, r, te, tr, info = env.step(np.tile(a, (n, 1)))
        pat = env.current_pattern.cpu().numpy()
        assert np.abs(pat - G[f"{name}/pattern"][k + 1][None]).max() < 1e-9, (name, k)
        assert np.array_equal(o.cpu().numpy()[2], G[f"{name}/obs"][k + 1])
        assert np.allclose(r.cpu().numpy(), G[f"{name}/reward"][k], rtol=1e-9)
        assert np.allclose(info["step_energy"].cpu().numpy(), G[f"{name}/energy"][k], rtol=1e-9)
        assert bool(te[0]) == G[f"{name}/terminated"][k] and bool(tr[0]) == G[f"{name}/truncated"][k]


@pytest.mark.gpu
def test_cuda_array_env_batch_vs_oracle_and_full_size(cuda_device):
    """BASELINE config[3]: 8x8 dipolar crossbars. 64 arrays x 20 random steps against the oracle, then 16,384 arrays for the
    size-independent properties (unit vectors, batch independence, auto-reset, statistics)."""
    import torch
    from spin_torque_rl_gym_b200 import SpinTorqueArrayVectorEnv
    rng = np.random.default_rng(4)
    n, size = 64, (8, 8)
    p0 = rng.normal(size=(n,) + size + (3,))
    p0 /= np.linalg.norm(p0, axis=-1, keepdims=True)
    env = SpinTorqueArrayVectorEnv(num_envs=n, array_size=size, action_mode="row", device=cuda_device, autoreset=False)
    env.reset(options={"initial_pattern": p0})
    oras = []
    for i in range(n):
        o = ArrayOracleEnv(array_size=size, action_mode="row")
        o.reset(p0[i])
        oras.append(o)
    for s in range(20):
        act = np.stack([rng.uniform(0, 7.49, n), rng.uniform(-2e6, 2e6, n), rng.uniform(0, 5e-9, n)], 1).astype(np.float32)
        o, r, te, tr, info = env.step(act)
        ref = [ora.step(act[i].copy()) for i, ora in enumerate(oras)]
        pat = env.current_pattern.cpu().numpy()
        assert np.abs(pat - np.stack([ora.pattern for ora in oras])).max() < 1e-9
        assert np.allclose(r.cpu().numpy(), [x[1] for x in ref], rtol=1e-9)
        assert np.array_equal(te.cpu().numpy(), [x[2] for x in ref])
    N = 16384
    big = SpinTorqueArrayVectorEnv(num_envs=N, array_size=size, action_mode="individual", device=cuda_device, max_steps=4,
                                   rng_seed=5)
    obs, _ = big.reset(seed=5)
    pat0 = big.current_pattern.clone()
    assert float((pat0.norm(dim=-1) - 1).abs().max()) < 1e-12
    assert abs(float(pat0.mean())) < 0.01
    act = torch.zeros(N, 3, dtype=torch.float32, device=cuda_device)
    act[:, 0] = torch.arange(N, device=cuda_device) % 64
    act[:, 1] = 1.5e6
    act[:, 2] = 2e-9
    ended = 0
    for s in range(4):
        o, r, te, tr, info = big.step(act)
        ended += int((te | tr).sum())
        assert torch.isfinite(r).all() and float((big.current_pattern.norm(dim=-1) - 1).abs().max()) < 1e-12
    st = big.episode_stats()
    assert st["steps"] == 4 * N and st["terminated"] + st["truncated"] == ended and ended >= N
    assert torch.all(info["step_count"] == 0)            # max_steps=4 truncated every array in the last step


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["individual", "row", "column", "global"])
def test_cuda_array_kernels_bit_identical(mode, cuda_device):
    """The default kernel (four arrays per warp, eight lanes each: NumPy's pairwise accumulators live in the lanes) and the
    one-warp-per-array kernel produce the same bits: state, observation, reward, energy, similarity, flags, statistics.
    Grids cover a multiple of 8 (8x8), remainders (3x3 = 8+1, 4x5 = 16+4, 10x12 = 120), the device counts whose shared-memory
    stride needs no padding (2x4, 4x6, 10x12: the last group's scratch ends exactly at the allocation), both fall-back sizes
    (2x3 < 8, 12x12 > 128) and batches that are not a multiple of 4; auto-reset on, so reset draws are compared too."""
    import torch
    from spin_torque_rl_gym_b200 import SpinTorqueArrayVectorEnv
    for size, n in (((8, 8), 1003), ((3, 3), 257), ((4, 5), 130), ((10, 12), 66), ((2, 4), 35), ((4, 6), 21), ((2, 3), 33),
                    ((12, 12), 9)):
        rng = np.random.default_rng(100 * ["individual", "row", "column", "global"].index(mode) + 10 * size[0] + size[1])
        envs = [SpinTorqueArrayVectorEnv(num_envs=n, array_size=size, action_mode=mode, device=cuda_device, max_steps=3,
                                         rng_seed=7, autoreset=True, one_warp_kernel=flag) for flag in (False, True)]
        for e in envs:
            e.reset(seed=7)
        assert torch.equal(envs[0].current_pattern, envs[1].current_pattern)
        nd = size[0] * size[1]
        for s in range(5):
            if mode == "global":
                act = np.stack([rng.uniform(-2e6, 2e6, n), rng.uniform(0, 5e-9, n)], 1)
            else:
                hi = {"individual": nd, "row": size[0], "column": size[1]}[mode]
                act = np.stack([rng.uniform(-0.5, hi + 0.5, n), rng.uniform(-2e6, 2e6, n), rng.uniform(0, 5e-9, n)], 1)
            act[::7, -2 if mode != "global" else 1] = 0.0              # |J| <= 1e-12: device untouched, no energy
            act = act.astype(np.float32)
            outs = [e.step(act.copy()) for e in envs]
            (o0, r0, te0, tr0, i0), (o1, r1, te1, tr1, i1) = outs
            assert torch.equal(o0, o1) and torch.equal(r0, r1) and torch.equal(te0, te1) and torch.equal(tr0, tr1), (size, s)
            assert torch.equal(envs[0].current_pattern, envs[1].current_pattern), (size, s)
            for k in ("step_energy", "pattern_similarity", "step_count", "final_observation"):
                assert torch.equal(i0[k], i1[k]), (size, s, k)
        s0, s1 = envs[0].episode_stats(), envs[1].episode_stats()
        for k in ("steps", "substeps", "terminated", "truncated", "episode_length"):
            assert s0[k] == s1[k], (size, k)
        assert s0["energy"] == pytest.approx(s1["energy"], rel=1e-12) and s0["truncated"] > 0
