"""K7: shuffled PPO minibatches gathered from a stored rollout (stg_rollout_minibatch_f32, RolloutCollector.get).

The permutation is checked on a host build of rollout_core.cuh (bijection, uniformity, independence of neighbouring
positions); the kernel and the collector are checked against torch indexing at the host build's indices, bit for bit."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy import stats

from spin_torque_rl_gym_b200 import _lib
from spin_torque_rl_gym_b200.envs.sb3_vec_env import RolloutBufferSamples, _splitmix64, minibatch_round_keys
from tests.helpers import ROOT

HEADER = os.path.join(ROOT, "include", "stg.h")
CSRC = os.path.join(ROOT, "spin_torque_rl_gym_b200", "csrc")
PLANES = ("obs", "action", "value", "log_prob", "advantage", "return")
KEY_SETS = [minibatch_round_keys(seed, off, ep) for seed, off, ep in ((0, 0, 0), (1, 0, 0), (1, 4096, 0), (7, 0, 3))]


@pytest.fixture(scope="module")
def host_permute(tmp_path_factory):
    """rollout_core.cuh's permutation compiled for the host: run(keys, M, start, count) -> int64 [count]."""
    d = tmp_path_factory.mktemp("perm_host")
    src = d / "perm_host.cpp"
    src.write_text('#include "rollout_core.cuh"\n'
                   'extern "C" void perm_host(const uint32_t* keys, int64_t M, int64_t start, int64_t n, int64_t* out) {\n'
                   '  for (int64_t k = 0; k < n; ++k) out[k] = stg::rollout_permute(keys, M, start + k);\n'
                   '}\n'
                   'extern "C" void perm_positions_many(const uint32_t* keys, int64_t n_keys, int64_t M, int64_t* out) {\n'
                   '  for (int64_t s = 0; s < n_keys; ++s)\n'
                   '    for (int64_t p = 0; p < M; ++p) out[s * M + p] = stg::rollout_permute(keys + 8 * s, M, p);\n'
                   '}\n'
                   'extern "C" int half_bits(int64_t M) { return stg::rollout_permute_half_bits(M); }\n')
    so = d / "perm_host.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-I", CSRC, str(src), "-o", str(so)], check=True)
    lib = C.CDLL(str(so))
    lib.perm_host.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p]
    lib.perm_positions_many.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p]
    lib.half_bits.argtypes = [C.c_int64]

    class Host:
        @staticmethod
        def run(keys, M, start=0, count=None):
            count = M - start if count is None else count
            k = np.asarray(keys, np.uint32)
            out = np.empty(count, np.int64)
            lib.perm_host(k.ctypes.data, M, start, count, out.ctypes.data)
            return out

        @staticmethod
        def many(key_sets, M):
            k = np.ascontiguousarray(np.asarray(key_sets, np.uint32))
            out = np.empty((len(key_sets), M), np.int64)
            lib.perm_positions_many(k.ctypes.data, len(key_sets), M, out.ctypes.data)
            return out

        half_bits = staticmethod(lib.half_bits)
    return Host


# ---------------------------------------------------------------------------------------------------- CPU --------------------

@pytest.mark.parametrize("M,half", [(1, 1), (2, 1), (4, 1), (5, 2), (16, 2), (17, 3), (1 << 28, 14), ((1 << 28) + 1, 15),
                                    (2049 << 20, 16), (1 << 62, 31)])
def test_half_width(host_permute, M, half):
    assert host_permute.half_bits(M) == half


@pytest.mark.parametrize("M", [1, 2, 3, 5, 1000, 4097, 65536, 65537, (1 << 20) + 3])
def test_permutation_is_a_bijection(host_permute, M):
    perms = [host_permute.run(keys, M) for keys in KEY_SETS]
    for p in perms:
        assert np.array_equal(np.sort(p), np.arange(M))
    if M >= 5:                                                              # different keys, different permutations
        for i in range(len(perms)):
            for j in range(i):
                assert not np.array_equal(perms[i], perms[j]), (M, i, j)
    # a slice is the same positions of the same permutation
    assert np.array_equal(host_permute.run(KEY_SETS[0], M, start=M // 2, count=M - M // 2), perms[0][M // 2:])


def test_permutation_at_the_largest_domain(host_permute):
    M = 1 << 62
    p = host_permute.run(KEY_SETS[1], M, start=M - 1000, count=1000)
    assert ((p >= 0) & (p < M)).all() and len(np.unique(p)) == 1000


@pytest.fixture(scope="module")
def images_1024(host_permute):
    """pi_e(p) for the 10^4 permutations of epochs 0 .. 9999 (seed 3, env_offset 0) of M = 1024 samples: [10^4, 1024]."""
    keys = [minibatch_round_keys(3, 0, e) for e in range(10_000)]
    return host_permute.many(keys, 1024)


def test_image_of_every_position_is_uniform(images_1024):
    S, M = images_1024.shape
    for p in range(M):
        counts = np.bincount(images_1024[:, p], minlength=M)
        _, pval = stats.chisquare(counts)
        assert pval > 1e-6, (p, pval)                                       # ~0.001 family-wise over the 1024 positions


def test_consecutive_positions_are_uncorrelated(images_1024):
    S, M = images_1024.shape
    x = images_1024.astype(np.float64)
    a, b = x[:, :-1] - x[:, :-1].mean(0), x[:, 1:] - x[:, 1:].mean(0)
    r = (a * b).sum(0) / np.sqrt((a * a).sum(0) * (b * b).sum(0))
    assert np.abs(r).max() < 5 / np.sqrt(S), np.abs(r).max()
    # joint of (pi(p), pi(p+1)) in 16 x 16 cells, pooled over p, against a uniform draw of two distinct samples
    hi = images_1024 >> 6
    cells = np.bincount((hi[:, :-1] * 16 + hi[:, 1:]).ravel(), minlength=256)
    n = cells.sum()
    expect = np.full((16, 16), 64.0 * 64.0)
    np.fill_diagonal(expect, 64.0 * 63.0)
    expect = expect.ravel() / expect.sum() * n
    _, pval = stats.chisquare(cells, expect)
    assert pval > 1e-6, pval


def test_minibatch_args_layout_matches_the_c_header(tmp_path):
    fields = [f for p in PLANES for f in (f"d_{p}", f"d_{p}_out")] + ["round_keys", "n_steps", "n_envs", "start", "batch"]
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', 'int main(void){',
             'printf("size %zu\\n", sizeof(StgMinibatchArgs));',
             'printf("keys %zu\\n", sizeof(((StgMinibatchArgs*)0)->round_keys));']
    lines += [f'printf("{f} %zu\\n", offsetof(StgMinibatchArgs, {f}));' for f in fields]
    lines.append('return 0;}')
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", str(src), "-o", str(exe)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split("\n") if l)
    assert int(got["size"]) == C.sizeof(_lib.StgMinibatchArgs)
    assert int(got["keys"]) == C.sizeof(C.c_uint32 * 8)
    for f in fields:
        assert int(got[f]) == getattr(_lib.StgMinibatchArgs, f).offset, f


def _args(T=4, N=4, start=0, batch=4, planes=PLANES, base=0x1000):
    a = _lib.StgMinibatchArgs()
    for i, p in enumerate(planes):
        setattr(a, f"d_{p}", base + 0x100000 * i)
        setattr(a, f"d_{p}_out", base + 0x100000 * i + 0x80000)
    a.n_steps, a.n_envs, a.start, a.batch = T, N, start, batch
    return a


def test_minibatch_argument_validation():
    lib = _lib.load()
    call = lambda a: lib.stg_rollout_minibatch_f32(C.byref(a), None)      # noqa: E731
    assert lib.stg_rollout_minibatch_f32(None, None) == -1                 # STG_E_NULL
    for kw in ({"T": -1}, {"N": -1}, {"start": -1}, {"batch": -1}):       # STG_E_SIZE: negative sizes
        assert call(_args(**kw)) == -2, kw
    assert call(_args(T=1 << 32, N=1 << 32)) == -2                         # T * N overflows int64
    assert call(_args(T=(1 << 31) + 1, N=1 << 31)) == -2                   # T * N > 2^62
    assert call(_args(T=1 << 31, N=1 << 31, start=(1 << 62) - 1, batch=2)) == -2
    assert call(_args(start=15, batch=2)) == -2                            # start + batch > T * N
    for kw in ({"batch": 0}, {"T": 0}, {"N": 0}, {"T": 0, "N": 0}):       # STG_OK without a launch
        assert call(_args(**kw)) == 0, kw
    assert call(_args(planes=())) == -1                                    # no plane at all
    for p in PLANES:                                                       # a half-set pair
        for side in (f"d_{p}", f"d_{p}_out"):
            a = _args()
            setattr(a, side, None)
            assert call(a) == -1, side
    for field, off in (("d_obs", 8), ("d_obs_out", 4), ("d_action", 4), ("d_action_out", 2)):
        a = _args()
        setattr(a, field, getattr(a, field) + off)
        assert call(a) == -4, field                                        # STG_E_ALIGN


def test_round_keys_are_a_pure_function_of_seed_offset_and_epoch():
    k = minibatch_round_keys(12345, 0, 0)
    assert len(k) == 8 and all(isinstance(x, int) and 0 <= x < 1 << 32 for x in k)
    assert k == minibatch_round_keys(12345, 0, 0)
    others = [minibatch_round_keys(12346, 0, 0), minibatch_round_keys(12345, 131072, 0), minibatch_round_keys(12345, 0, 1),
              minibatch_round_keys(0, 12345, 0), minibatch_round_keys(0, 0, 12345)]
    assert all(o != k for o in others) and len({tuple(o) for o in others}) == len(others)
    assert minibatch_round_keys(-1, 0, 0) == minibatch_round_keys((1 << 64) - 1, 0, 0)        # words are taken mod 2^64
    # pinned: a seed keeps reproducing the same shuffles across releases (splitmix64's first output from state 0 is
    # 0xE220A8397B1DCDAF in its reference implementation)
    assert _splitmix64(0) == (0x9E3779B97F4A7C15, 0xE220A8397B1DCDAF)
    assert minibatch_round_keys(0, 0, 0) == [0xAAC80268, 0x2130748A, 0x79CE5090, 0x0CC78FB9, 0xFBA6B4AC, 0xAB9AA3DA, 0x6B3B1DD2,
                                             0xB0C750A8]


def test_samples_tuple_has_sb3_field_names():
    assert RolloutBufferSamples._fields == ("observations", "actions", "old_values", "old_log_prob", "advantages", "returns")


# ---------------------------------------------------------------------------------------------------- GPU --------------------

def _random_bits(torch, dev, shape, gen):
    """float32 planes of random bit patterns (NaNs, infinities and subnormals included): the gather must copy bits."""
    return torch.randint(-(1 << 31), 1 << 31, shape, dtype=torch.int64, device=dev, generator=gen).to(torch.int32) \
        .view(torch.float32)


def _bits(x):
    import torch
    return x.view(torch.int32)


def _launch(torch, planes, outs, keys, T, N, start, batch):
    a = _lib.StgMinibatchArgs()
    for p in PLANES:
        if p in planes:
            setattr(a, f"d_{p}", planes[p].data_ptr())
            setattr(a, f"d_{p}_out", outs[p].data_ptr())
    a.round_keys[:] = keys
    a.n_steps, a.n_envs, a.start, a.batch = T, N, start, batch
    _lib.check(_lib.load().stg_rollout_minibatch_f32(C.byref(a), torch.cuda.current_stream().cuda_stream),
               "stg_rollout_minibatch_f32")


def _windows(M, B):
    """(start, batch): the first, a middle and the last (possibly partial) minibatch of size B."""
    last = (M - 1) // B * B
    return sorted({(0, min(B, M)), (min(M // 2 // B * B, last), min(B, M - min(M // 2 // B * B, last))), (last, M - last)})


@pytest.mark.gpu
@pytest.mark.parametrize("T,N", [(1, 1), (37, 1000), (256, 4097)])
def test_cuda_minibatch_kernel_equals_torch_indexing(cuda_device, host_permute, T, N):
    import torch
    M = T * N
    gen = torch.Generator(device=cuda_device).manual_seed(M)
    width = {"obs": 12, "action": 2}
    planes = {p: _random_bits(torch, cuda_device, (T, N, width[p]) if p in width else (T, N), gen) for p in PLANES}
    for keys in KEY_SETS[:2]:
        for B in (1, 1000, 65536):
            for start, batch in _windows(M, B):
                idx = torch.from_numpy(host_permute.run(keys, M, start, batch)).to(cuda_device)
                want = {p: planes[p].reshape(M, -1)[idx].reshape((batch, width[p]) if p in width else (batch,))
                        for p in PLANES}
                outs = {p: torch.empty_like(want[p]) for p in PLANES}
                _launch(torch, planes, outs, keys, T, N, start, batch)
                for p in PLANES:
                    assert torch.equal(_bits(outs[p]), _bits(want[p])), (p, B, start, batch)
    # one plane at a time, the other pairs NULL: only that output is written
    start, batch = _windows(M, 1000)[-1]
    idx = torch.from_numpy(host_permute.run(KEY_SETS[0], M, start, batch)).to(cuda_device)
    for p in PLANES:
        want = planes[p].reshape(M, -1)[idx].reshape((batch, width[p]) if p in width else (batch,))
        outs = {q: torch.full((batch, width[q]) if q in width else (batch,), -7.0, device=cuda_device) for q in PLANES}
        _launch(torch, {p: planes[p]}, {p: outs[p]}, KEY_SETS[0], T, N, start, batch)
        assert torch.equal(_bits(outs[p]), _bits(want)), p
        for q in PLANES:
            if q != p:
                assert bool((outs[q] == -7.0).all()), (p, q)


@pytest.mark.gpu
def test_cuda_minibatch_kernel_int64_offsets(cuda_device, host_permute):
    """2049 steps x 1,048,576 envs = 2,148,532,224 samples > 2^31, advantage plane only (8.6 GB)."""
    import torch
    T, N = 2049, 1 << 20
    M = T * N
    gen = torch.Generator(device=cuda_device).manual_seed(9)
    adv = torch.randn(T, N, generator=gen, device=cuda_device)
    keys = KEY_SETS[3]
    B = 65536
    for start, batch in _windows(M, B):
        idx_np = host_permute.run(keys, M, start, batch)
        idx = torch.from_numpy(idx_np).to(cuda_device)
        out = torch.empty(batch, device=cuda_device)
        _launch(torch, {"advantage": adv}, {"advantage": out}, keys, T, N, start, batch)
        assert torch.equal(_bits(out), _bits(adv.view(-1)[idx])), (start, batch)
    assert (host_permute.run(keys, M, M - B, B) >= 1 << 31).any()          # the last window reaches past 2^31


def _actor_critic(torch, dev):
    gen = torch.Generator(device=dev).manual_seed(0)
    w1 = torch.randn(12, 32, generator=gen, device=dev) * 0.3
    wa = torch.randn(32, 2, generator=gen, device=dev) * 0.3
    wv = torch.randn(32, 1, generator=gen, device=dev) * 0.3

    def value_fn(o):
        return torch.tanh(o @ w1) @ wv

    def policy(o):
        out = torch.tanh(o @ w1) @ wa
        act = torch.empty(o.shape[0], 2, device=dev)
        act[:, 0] = torch.tanh(out[:, 0]) * 1.1e-6
        act[:, 1] = torch.sigmoid(out[:, 1]) * 1e-9 + 1e-11
        return act, value_fn(o), -(out * out).sum(1)
    return value_fn, policy


def _collector(stg, torch, dev, n=512, T=16, seed=3, **kw):
    env = stg.make("SpinTorque-v0", num_envs=n, device=dev, max_steps=5, max_current=1.1e-6, rng_seed=seed)
    value_fn, policy = _actor_critic(torch, dev)
    col = stg.RolloutCollector(env, n_steps=T, store_values=True, **kw)
    col.collect(policy, value_fn)
    col.compute_returns_and_advantage()
    return col, value_fn, policy


def _epoch(col, batch_size):
    import torch
    batches = list(col.get(batch_size))
    cat = RolloutBufferSamples(*[torch.cat([getattr(b, f) for b in batches]) for f in RolloutBufferSamples._fields])
    return batches, cat


@pytest.mark.gpu
def test_rollout_collector_get_end_to_end(cuda_device, host_permute):
    import torch
    import spin_torque_rl_gym_b200 as stg
    col, _, _ = _collector(stg, torch, cuda_device)
    twin, _, _ = _collector(stg, torch, cuda_device)
    T, N = col.n_steps, col.env.num_envs
    M = T * N
    flat = RolloutBufferSamples(col.observations.reshape(M, 12), col.actions.reshape(M, 2), col.values.reshape(M),
                                col.log_probs.reshape(M), col.advantages.reshape(M), col.returns.reshape(M))
    epoch = 0
    for bs in (None, 1, 7, 1000, M, M + 5):
        first, cat = _epoch(col, bs)
        idx = torch.from_numpy(host_permute.run(minibatch_round_keys(col.env.rng_seed, col.env.env_offset, epoch), M))
        idx = idx.to(cuda_device)
        for f in RolloutBufferSamples._fields:
            assert torch.equal(getattr(cat, f), getattr(flat, f)[idx]), (bs, f)
        b = M if bs is None else bs
        assert [len(x.advantages) for x in first] == [b] * (M // b) + ([M % b] if M % b else []), bs
        for x in first[:2]:
            B = len(x.advantages)
            assert x.observations.shape == (B, 12) and x.actions.shape == (B, 2)
            assert all(getattr(x, f).shape == (B,) for f in RolloutBufferSamples._fields[2:])
            assert all(getattr(x, f).dtype == torch.float32 and getattr(x, f).device == cuda_device for f in x._fields)
        second, cat2 = _epoch(col, bs)                                     # the next epoch: another permutation
        assert not torch.equal(cat2.advantages, cat.advantages)
        assert torch.equal(torch.sort(cat2.advantages).values, torch.sort(cat.advantages).values)
        for ref, got in ((first, _epoch(twin, bs)[0]), (second, _epoch(twin, bs)[0])):  # same seed, same epochs
            for x, y in zip(ref, got):
                assert all(torch.equal(getattr(x, f), getattr(y, f)) for f in x._fields), bs
        epoch += 2
    # a batch kept by the caller is not overwritten by later batches or epochs
    kept = next(iter(col.get(100)))
    snapshot = [getattr(kept, f).clone() for f in kept._fields]
    list(col.get(100))
    assert all(torch.equal(s, getattr(kept, f)) for s, f in zip(snapshot, kept._fields))


@pytest.mark.gpu
def test_rollout_collector_get_does_not_synchronise(cuda_device):
    import torch
    import spin_torque_rl_gym_b200 as stg
    col, _, _ = _collector(stg, torch, cuda_device)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        n = sum(1 for _ in col.get(1000)) + sum(1 for _ in col.get())
    finally:
        torch.cuda.set_sync_debug_mode("default")
    assert n == 9 + 1


@pytest.mark.gpu
def test_rollout_collector_get_errors(cuda_device):
    import torch
    import spin_torque_rl_gym_b200 as stg
    env = stg.make("SpinTorque-v0", num_envs=64, device=cuda_device, max_steps=5, max_current=1.1e-6, rng_seed=3)
    value_fn, policy = _actor_critic(torch, cuda_device)
    plain = stg.RolloutCollector(env, n_steps=4)
    assert set(vars(plain)) == {"env", "n_steps", "store_observations", "store_values", "observations", "actions", "rewards",
                                "dones", "_last_obs"}
    plain.collect(lambda o: policy(o)[0])
    with pytest.raises(ValueError):
        plain.get()                                                         # no values stored
    no_obs = stg.RolloutCollector(env, n_steps=4, store_observations=False, store_values=True)
    no_obs.collect(policy, value_fn)
    no_obs.compute_returns_and_advantage()
    with pytest.raises(ValueError):
        no_obs.get()                                                        # no observations stored
    col = stg.RolloutCollector(env, n_steps=4, store_values=True)
    with pytest.raises(RuntimeError):
        col.get()                                                           # nothing collected
    col.collect(policy, value_fn)
    with pytest.raises(RuntimeError):
        col.get()                                                           # no GAE yet
    col.compute_returns_and_advantage()
    assert len(list(col.get(64))) == 4
    col.collect(policy, value_fn)
    with pytest.raises(RuntimeError):
        col.get()                                                           # a new rollout without its GAE
    col.compute_returns_and_advantage()
    for bad in (0, -1):
        with pytest.raises(ValueError):
            col.get(bad)
