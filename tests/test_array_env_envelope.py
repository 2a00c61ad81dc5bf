"""K3 (SpinTorqueArrayVectorEnv) over everything it accepts: 1 to 1,024 devices, the three device kinds, the three coupling
types or none, the four action modes, edge actions and every reset path.

Three levels are compared. The oracle (oracle/array_oracle.py, pinned bit-exactly to the reference) is the semantics. The
host build of array_core.cuh (tests/hostsim) must agree with it to 1e-12. The CUDA kernels must equal the host build bit for
bit (array_kernels.cu: the 8-lane kernel's sums and device update are the host sequence, lane by lane), and the oracle to
1e-12 on a sample of each batch. The GPU sizes reach every launch branch of stg_array_step_f64: the one-warp kernel below 8
and above 128 devices (NumPy's recursive pairwise sum), the 8-lane kernel's non-VEC (odd device count), generic VEC and
<64, VEC> builds, both sides of the 48 KB shared-memory line of a launch without the opt-in (1x876, 1x877, 2x439) and the
1,024-device maximum, where the reset kernel uses exactly 48 KB."""
import ctypes as C
import functools

import numpy as np
import pytest

from oracle.array_oracle import ArrayOracleEnv, checkerboard, coupling_matrix
from spin_torque_rl_gym_b200 import _lib, params as P
from spin_torque_rl_gym_b200.envs.array_env import array_params, compute_coupling_matrix

KINDS = ("stt_mram", "sot_mram", "vcma_mram")
COUPLINGS = ("dipolar", "exchange", "stray_field", None)        # None: include_coupling=False
MODES = ("individual", "row", "column", "global")
STRENGTH = 1e4           # coupling fields of ~1 % of the anisotropy field, so that a wrong coupling sum moves the pattern
MAX_CURRENT, MAX_DURATION = 2e6, 5e-9
TOL = 1e-12
# kind x coupling with the four modes spread so that every kind and every coupling meets every mode once
SWEEP = [(k, c, MODES[(j + j // 4) % 4]) for j, (k, c) in enumerate((k, c) for k in KINDS for c in COUPLINGS)]


def device_params(kind):
    dp = P.default_device_parameters(kind)
    if kind == "sot_mram":
        dp["aspect_ratio"] = 2.0          # unequal in-plane demagnetising factors, both branches of the shape formula
    elif kind == "vcma_mram":
        dp["aspect_ratio"] = 0.5
    return dp


@functools.lru_cache(maxsize=None)
def _oracle_coupling(size, coupling):
    return coupling_matrix(*size, STRENGTH, coupling)


def make_oracle(size, kind, coupling, mode, max_steps, pattern, target):
    """A fresh oracle array. Its coupling matrix (O(nd^2) Python, seconds at 1,024 devices) is computed once per size and
    coupling type and shared read-only."""
    o = ArrayOracleEnv(array_size=size, device_type=kind, device_params=device_params(kind), max_steps=max_steps,
                       max_current=MAX_CURRENT, max_duration=MAX_DURATION, include_coupling=False, action_mode=mode)
    if coupling is not None:
        o.include_coupling, o.coupling = True, _oracle_coupling(size, coupling)
    o.reset(pattern.reshape(size + (3,)), target.reshape(size + (3,)))
    return o


@functools.lru_cache(maxsize=None)
def _coupling(size, coupling):
    return None if coupling is None else np.ascontiguousarray(compute_coupling_matrix(*size, STRENGTH, coupling))


class HostArrays:
    """n arrays stepped by the host build of K3's core, with the env's buffer layout. It has no autoreset: the caller
    restarts ended arrays itself."""

    def __init__(self, size, kind, coupling, mode, max_steps, pattern, target):
        from tests.hostsim.harness import lib
        self.lib = lib()
        self.p = array_params(size, kind, device_params(kind), mode, max_steps, MAX_CURRENT, MAX_DURATION, 0.9, 0.1)
        self.coupling = _coupling(size, coupling)
        n, D = pattern.shape[:2]
        self.pattern = np.ascontiguousarray(pattern, dtype=np.float64).copy()
        self.target = np.ascontiguousarray(target, dtype=np.float64).copy()
        self.total_energy, self.step_count, self.episode = np.zeros(n), np.zeros(n, np.int32), np.zeros(n, np.int32)
        self.obs = np.zeros((n, D, 6), np.float32)
        self.reward, self.energy, self.similarity = np.zeros(n), np.zeros(n), np.zeros(n)
        self.terminated, self.truncated = np.zeros(n, np.uint8), np.zeros(n, np.uint8)

    def step(self, act):
        act = np.ascontiguousarray(act, np.float32)
        a = _lib.StgArrayStepArgs()
        a.params = self.p
        a.d_coupling = None if self.coupling is None else self.coupling.ctypes.data
        a.d_pattern, a.d_target = self.pattern.ctypes.data, self.target.ctypes.data
        a.d_total_energy, a.d_step_count, a.d_episode = (self.total_energy.ctypes.data, self.step_count.ctypes.data,
                                                         self.episode.ctypes.data)
        a.d_action, a.d_obs, a.d_reward = act.ctypes.data, self.obs.ctypes.data, self.reward.ctypes.data
        a.d_terminated, a.d_truncated = self.terminated.ctypes.data, self.truncated.ctypes.data
        a.d_step_energy, a.d_similarity = self.energy.ctypes.data, self.similarity.ctypes.data
        a.n_arrays, a.action_stride = len(act), act.shape[1]
        self.lib.hostsim_array_step(C.byref(a))


def unit_vectors(rng, shape):
    v = rng.normal(size=shape + (3,))
    return v / np.linalg.norm(v, axis=-1, keepdims=True)


def top_index(size, mode):
    return {"individual": size[0] * size[1] - 1, "row": size[0] - 1, "column": size[1] - 1}[mode]


def random_actions(rng, n, size, mode):
    if mode == "global":          # [J, T] is read as [index, J]: half the rows put a real current where T goes
        second = np.where(rng.random(n) < 0.5, rng.uniform(0, MAX_DURATION, n), rng.uniform(-MAX_CURRENT, MAX_CURRENT, n))
        return np.stack([rng.uniform(-MAX_CURRENT, MAX_CURRENT, n), second], 1).astype(np.float32)
    hi = top_index(size, mode)
    return np.stack([rng.uniform(-0.5, hi + 0.99, n), rng.uniform(-MAX_CURRENT, MAX_CURRENT, n),
                     rng.uniform(0, MAX_DURATION, n)], 1).astype(np.float32)


def edge_actions(size, mode):
    """One edge case per row. NaN, +-inf and out-of-range values of every component; |J| <= 1e-12 leaves the devices
    untouched at no energy; a NaN current does the same; a NaN duration propagates NaN into the driven devices."""
    nan, inf, J, T = np.nan, np.inf, 1.3e6, 2e-9
    if mode == "global":
        rows = [[0.0, J], [1e6, T], [nan, T], [inf, -J], [0.0, inf], [0.0, -inf], [0.0, 0.0], [0.0, 1e-12],
                [0.0, -5e-13], [0.0, nan], [0.0, 1e-11], [0.0, 3 * MAX_CURRENT]]
    else:
        hi = top_index(size, mode)
        rows = [[-3.0, J, T], [hi + 7.0, J, T], [hi + 0.5, J, T], [nan, J, T], [-inf, J, T], [inf, J, T],
                [0.0, inf, T], [0.0, -inf, T], [0.0, 0.0, T], [hi, 1e-12, T], [hi, -5e-13, T], [0.0, nan, T],
                [0.0, J, 0.0], [0.0, -J, -1e-9], [hi, J, 3 * MAX_DURATION], [0.0, J, inf], [0.0, J, nan],
                [hi, nan, nan], [0.0, 0.0, nan]]
    return np.asarray(rows, np.float32)


def oracle_action(a):
    """The reference raises on a NaN index (int(nan)); K3 takes index 0 (DESIGN.md, K3's action semantics)."""
    a = a.copy()
    if len(a) == 3 and np.isnan(a[0]):
        a[0] = 0.0
    return a


def assert_near(got, want, tol, what, rel=False):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    assert np.array_equal(np.isnan(got), np.isnan(want)), what
    ok = ~np.isnan(want)
    scale = np.abs(want[ok]) if rel else np.maximum(1.0, np.abs(want[ok]))
    err = np.abs(got[ok] - want[ok])
    assert np.all(err <= tol * scale), (what, float(err.max()) if err.size else 0.0)


def check_against_oracle(i, ora, ref, pattern, obs, reward, energy, similarity, terminated, truncated, what):
    o, r, te, tr, info = ref
    assert_near(pattern, ora.pattern.reshape(-1, 3), TOL, (what, i, "pattern"))
    assert np.array_equal(obs.reshape(o.shape), o, equal_nan=True), (what, i, "obs")
    assert_near(reward, r, TOL, (what, i, "reward"))
    assert_near(energy, info["energy"], TOL, (what, i, "energy"), rel=True)
    assert_near(similarity, info["similarity"], TOL, (what, i, "similarity"))
    assert bool(terminated) == te and bool(truncated) == tr, (what, i, "flags")


def start_state(rng, n, size, kind_index=0):
    """Per-array start patterns and targets: a checkerboard, random unit vectors, and the start pattern itself (those arrays
    end with success after one step in most modes, so that episodes end at different steps)."""
    nd = size[0] * size[1]
    p0 = unit_vectors(rng, (n, nd))
    tgt = np.repeat(checkerboard(*size).reshape(1, nd, 3), n, 0)
    sel = (np.arange(n) + kind_index) % 5
    tgt[sel == 1] = p0[sel == 1]
    tgt[sel == 2] = unit_vectors(rng, (int((sel == 2).sum()), nd))
    return p0, tgt


# ---- host build against the oracle (no GPU) ---------------------------------------------------------------------------------
CPU_SIZES = [(1, 1), (1, 7), (2, 3), (3, 3), (4, 5), (8, 16), (3, 43), (9, 15), (16, 16)]


@pytest.mark.parametrize("size", CPU_SIZES + [(32, 32)], ids=lambda s: f"{s[0]}x{s[1]}")
def test_host_build_matches_oracle(size):
    """Every kind x coupling x mode; a few random steps each. At 32x32 one step of one configuration: the oracle's coupling
    matrix alone takes seconds there, and a step of the whole array as long."""
    nd = size[0] * size[1]
    steps = 1 if nd > 256 else (2 if nd >= 128 else 3)
    n = 1 if nd >= 128 else 2
    cases = [(k, c, m) for k in KINDS for c in COUPLINGS for m in MODES] if nd <= 256 else [("sot_mram", "dipolar", "row")]
    for ci, (kind, coupling, mode) in enumerate(cases):
        rng = np.random.default_rng([nd, ci])
        p0, tgt = start_state(rng, n, size, ci)
        host = HostArrays(size, kind, coupling, mode, 2, p0, tgt)
        oras = [make_oracle(size, kind, coupling, mode, 2, p0[i], tgt[i]) for i in range(n)]
        for s in range(steps):
            act = random_actions(rng, n, size, mode)
            host.step(act)
            for i, ora in enumerate(oras):
                check_against_oracle(i, ora, ora.step(act[i].copy()), host.pattern[i], host.obs[i], host.reward[i],
                                     host.energy[i], host.similarity[i], host.terminated[i], host.truncated[i],
                                     (size, kind, coupling, mode, s))


@pytest.mark.parametrize("mode", MODES)
def test_host_build_edge_actions_match_oracle(mode):
    """NaN, infinite, zero and out-of-range actions follow the reference (a NaN index aside, see oracle_action)."""
    for size in ((1, 1), (2, 3), (4, 5), (3, 43)):
        acts = edge_actions(size, mode)
        n = len(acts)
        rng = np.random.default_rng(size[0] * 100 + size[1])
        p0, tgt = start_state(rng, n, size)
        host = HostArrays(size, "stt_mram", "dipolar", mode, 200, p0, tgt)
        host.step(acts)
        for i in range(n):
            ora = make_oracle(size, "stt_mram", "dipolar", mode, 200, p0[i], tgt[i])
            check_against_oracle(i, ora, ora.step(oracle_action(acts[i])), host.pattern[i], host.obs[i], host.reward[i],
                                 host.energy[i], host.similarity[i], host.terminated[i], host.truncated[i],
                                 (size, mode, acts[i]))


# ---- CUDA kernels against the host build (bit for bit) and the oracle -------------------------------------------------------
# Representative size of each kernel: every kind x coupling. The other sizes: all four modes, kind and coupling rotating.
KERNEL_SIZES = [(2, 3), (3, 3), (4, 5), (8, 8), (9, 15)]
EDGE_SIZES = [(1, 1), (1, 127), (1, 8), (8, 16), (3, 43), (1, 876), (1, 877), (2, 439), (32, 32)]
GPU_CASES = [(s, k, c, m) for s in KERNEL_SIZES for k, c, m in SWEEP] + \
    [(s, *SWEEP[(5 * j + q) % 12][:2], m) for j, s in enumerate(EDGE_SIZES) for q, m in enumerate(MODES)]


def _gpu_env(cuda_device, size, kind, coupling, mode, n, max_steps, **kw):
    from spin_torque_rl_gym_b200 import SpinTorqueArrayVectorEnv
    return SpinTorqueArrayVectorEnv(num_envs=n, array_size=size, device_type=kind, device_params=device_params(kind),
                                    include_coupling=coupling is not None, coupling_type=coupling or "dipolar",
                                    coupling_strength=STRENGTH, action_mode=mode, max_steps=max_steps,
                                    max_current=MAX_CURRENT, max_duration=MAX_DURATION, device=cuda_device, **kw)


def _np(t):
    return t.detach().cpu().numpy()


def _same(got, want, what):
    assert np.array_equal(np.asarray(got), np.asarray(want), equal_nan=True), what


def _obs_of(pattern, target):
    return np.concatenate([pattern, target], -1).astype(np.float32)


@pytest.mark.gpu
@pytest.mark.parametrize("size,kind,coupling,mode", GPU_CASES,
                         ids=[f"{s[0]}x{s[1]}-{k[:4]}-{c}-{m}" for s, k, c, m in GPU_CASES])
def test_cuda_matches_host_build_and_oracle(size, kind, coupling, mode, cuda_device):
    """A batch of distinct arrays (a count that is not a multiple of 4) for five steps with max_steps=3 and autoreset:
    every output equals the host build bit for bit, the first, a middle and the last array follow the oracle, the autoreset
    draws equal the reset kernel's draws for the same episode, and the episode statistics are the sums of the steps."""
    import torch
    nd = size[0] * size[1]
    n = 37 if nd <= 256 else 7
    steps, max_steps = 5, 3
    rng = np.random.default_rng([nd, KINDS.index(kind), COUPLINGS.index(coupling), MODES.index(mode)])
    p0, tgt = start_state(rng, n, size, KINDS.index(kind))
    env = _gpu_env(cuda_device, size, kind, coupling, mode, n, max_steps, rng_seed=11)
    twin = _gpu_env(cuda_device, size, kind, None, mode, n, max_steps, rng_seed=11, autoreset=False)
    if coupling is not None:
        _same(env.coupling_matrix, _oracle_coupling(size, coupling), "coupling matrix")
    rows = (n, nd, 3)
    obs, _ = env.reset(options={"initial_pattern": p0.reshape((n,) + size + (3,)),
                                "target_pattern": tgt.reshape((n,) + size + (3,))})
    twin.reset(options={"initial_pattern": p0.reshape((n,) + size + (3,))})
    _same(_np(obs).reshape(n, nd, 6), _obs_of(p0, tgt), "reset obs")
    host = HostArrays(size, kind, coupling, mode, max_steps, p0, tgt)
    sample = (0, n // 2, n - 1)
    oras = {i: make_oracle(size, kind, coupling, mode, max_steps, p0[i], tgt[i]) for i in sample}
    oracle_steps = steps if nd <= 256 else 1          # an oracle step of a whole 1x877 array takes over a second
    count = {"individual": 1, "row": size[1], "column": size[0], "global": nd}[mode]
    want = dict.fromkeys(("steps", "substeps", "terminated", "truncated", "energy", "reward", "episode_length"), 0.0)
    for s in range(steps):
        act = random_actions(rng, n, size, mode)
        o, r, te, tr, info = env.step(torch.from_numpy(act).to(cuda_device))
        host.step(act)
        what = (size, kind, coupling, mode, s)
        ended = (host.terminated | host.truncated).astype(bool)
        _same(_np(r), host.reward, (what, "reward"))
        _same(_np(te), host.terminated.astype(bool), (what, "terminated"))
        _same(_np(tr), host.truncated.astype(bool), (what, "truncated"))
        _same(_np(info["step_energy"]), host.energy, (what, "step_energy"))
        _same(_np(info["pattern_similarity"]), host.similarity, (what, "similarity"))
        _same(_np(info["step_count"]), np.where(ended, 0, host.step_count), (what, "step_count"))
        _same(_np(info["total_energy"]), np.where(ended, 0.0, host.total_energy), (what, "total_energy"))
        pat, ob = _np(env.current_pattern).reshape(rows), _np(o).reshape(n, nd, 6)
        _same(pat[~ended], host.pattern[~ended], (what, "pattern"))
        _same(ob[~ended], host.obs[~ended], (what, "obs"))
        _same(_np(info["final_observation"]).reshape(n, nd, 6)[ended], host.obs[ended], (what, "final_observation"))
        for i in sample:
            if s < oracle_steps:
                check_against_oracle(i, oras[i], oras[i].step(act[i].copy()), pat[i] if not ended[i] else host.pattern[i],
                                     host.obs[i], _np(r)[i], _np(info["step_energy"])[i],
                                     _np(info["pattern_similarity"])[i], _np(te)[i], _np(tr)[i], what)
        want["steps"] += n
        want["substeps"] += 10.0 * count * n
        want["terminated"] += float(host.terminated.sum())
        want["truncated"] += float((host.truncated & ~host.terminated).sum())
        want["energy"] += float(host.energy.sum())
        want["reward"] += float(host.reward.sum())
        want["episode_length"] += float(host.step_count[ended].sum())
        if ended.any():
            # the autoreset draw: unit vectors, the reset kernel's draw for the same (seed, array, episode), target kept
            mask = torch.from_numpy(ended).to(cuda_device)
            twin.reset(mask=mask)
            twin_pat = _np(twin.current_pattern).reshape(rows)
            _same(pat[ended], twin_pat[ended], (what, "autoreset draw vs reset draw"))
            assert np.abs(np.linalg.norm(pat[ended], axis=-1) - 1).max() < 1e-12, what
            _same(ob[ended], _obs_of(pat[ended], tgt[ended]), (what, "obs after autoreset"))
            host.pattern[ended] = pat[ended]
            host.step_count[ended], host.total_energy[ended] = 0, 0.0
            for i in sample:
                if ended[i]:
                    oras[i].reset(pat[i].reshape(size + (3,)), tgt[i].reshape(size + (3,)))
    got = env.episode_stats()
    for k in ("steps", "substeps", "terminated", "truncated", "episode_length"):
        assert got[k] == want[k], (k, got[k], want[k])
    assert got["truncated"] > 0
    for k in ("energy", "reward"):          # atomics in any order
        assert got[k] == pytest.approx(want[k], rel=1e-12, abs=1e-12), k


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
def test_cuda_edge_actions(mode, cuda_device):
    """The edge actions of test_host_build_edge_actions_match_oracle through both kernels at a size of every launch branch:
    bit for bit against the host build, against the oracle, untouched devices where |J| <= 1e-12 or J is NaN, and a
    global-mode step that ignores its first component. Autoreset is off: several rows end with success (start pattern equal
    to the target, no current), and their end state is what is compared."""
    import torch
    for size in ((1, 1), (2, 3), (3, 3), (1, 8), (4, 5), (8, 8), (3, 43)):
        nd = size[0] * size[1]
        acts = edge_actions(size, mode)
        if mode == "global":       # same start pattern, same second component, different first: same result
            acts = np.concatenate([acts, [[-7.0, 1.3e6]]]).astype(np.float32)
        n = len(acts)
        rng = np.random.default_rng(size[0] * 1000 + size[1])
        p0, tgt = start_state(rng, n, size)
        if mode == "global":
            p0[-1], tgt[-1] = p0[0], tgt[0]
        host = HostArrays(size, "stt_mram", "dipolar", mode, 200, p0, tgt)
        host.step(acts)
        for one_warp in (False, True):
            what = (size, mode, "one-warp kernel" if one_warp else "default kernel")
            env = _gpu_env(cuda_device, size, "stt_mram", "dipolar", mode, n, 200, autoreset=False,
                           one_warp_kernel=one_warp)
            env.reset(options={"initial_pattern": p0.reshape((n,) + size + (3,)),
                               "target_pattern": tgt.reshape((n,) + size + (3,))})
            o, r, te, tr, info = env.step(torch.from_numpy(acts).to(cuda_device))
            pat, ob = _np(env.current_pattern).reshape(n, nd, 3), _np(o).reshape(n, nd, 6)
            energy, sim = _np(info["step_energy"]), _np(info["pattern_similarity"])
            for name, got, want in (("pattern", pat, host.pattern), ("obs", ob, host.obs), ("reward", _np(r), host.reward),
                                    ("energy", energy, host.energy), ("similarity", sim, host.similarity),
                                    ("terminated", _np(te), host.terminated.astype(bool)),
                                    ("truncated", _np(tr), host.truncated.astype(bool))):
                _same(got, want, (what, name))
            for i in range(n):
                cur = acts[i][1]
                if np.isnan(cur) or abs(cur) <= 1e-12:
                    assert energy[i] == 0.0 and np.array_equal(pat[i], p0[i]), (what, acts[i])
            if mode == "global":
                _same(pat[-1], pat[0], (what, "global ignores its first component"))
                _same(_np(r)[-1], _np(r)[0], (what, "global ignores its first component"))
        for i in range(n):
            ora = make_oracle(size, "stt_mram", "dipolar", mode, 200, p0[i], tgt[i])
            check_against_oracle(i, ora, ora.step(oracle_action(acts[i])), pat[i], ob[i], _np(r)[i], energy[i], sim[i],
                                 _np(te)[i], _np(tr)[i], (size, mode, acts[i]))


def _reset_surface_env(cuda_device, size, n, max_steps=200, **kw):
    return _gpu_env(cuda_device, size, "stt_mram", "dipolar", "individual", n, max_steps, **kw)


@pytest.mark.gpu
@pytest.mark.parametrize("size", [(2, 3), (4, 5), (8, 8), (1, 877)], ids=lambda s: f"{s[0]}x{s[1]}")
def test_cuda_reset_surface(size, cuda_device):
    """reset(mask=...) redraws only the masked arrays and advances their episode counters; a constructor target_pattern
    reaches the observation and the reward; two envs of N/2 arrays with array_offset 0 and N/2 draw, at reset and at
    autoreset, exactly what one N-array env draws."""
    import torch
    nd, n = size[0] * size[1], 10
    rng = np.random.default_rng(nd)
    target = unit_vectors(rng, size)
    env = _reset_surface_env(cuda_device, size, n, target_pattern=target, rng_seed=3)
    obs, _ = env.reset(seed=3)
    pat0 = _np(env.current_pattern).reshape(n, nd, 3)
    assert np.abs(np.linalg.norm(pat0, axis=-1) - 1).max() < 1e-12
    _same(_np(obs).reshape(n, nd, 6), _obs_of(pat0, np.repeat(target.reshape(1, nd, 3), n, 0)), "target in obs")
    act = random_actions(rng, n, size, "individual")
    o, r, te, tr, info = env.step(torch.from_numpy(act).to(cuda_device))
    host = HostArrays(size, "stt_mram", "dipolar", "individual", 200, pat0, np.repeat(target.reshape(1, nd, 3), n, 0))
    host.step(act)
    _same(_np(r), host.reward, "reward with a custom target")
    _same(_np(env.current_pattern).reshape(n, nd, 3), host.pattern, "pattern with a custom target")
    before, ep0 = _np(env.current_pattern).reshape(n, nd, 3), _np(env._episode)
    mask = np.arange(n) % 3 == 1
    env.reset(mask=mask)
    after, ep1 = _np(env.current_pattern).reshape(n, nd, 3), _np(env._episode)
    _same(after[~mask], before[~mask], "unmasked arrays keep their pattern")
    assert not np.any(np.all(after[mask] == before[mask], axis=(1, 2))), "masked arrays draw a new pattern"
    _same(ep1, ep0 + mask, "episode counters")
    _same(_np(env._step_count), np.where(mask, 0, 1), "step counters")

    def draws(num_envs, offset):
        e = _reset_surface_env(cuda_device, size, num_envs, rng_seed=9, array_offset=offset, max_steps=1)
        e.reset(seed=9)
        first = _np(e.current_pattern).copy()
        e.step(torch.from_numpy(random_actions(np.random.default_rng(0), num_envs, size, "individual")).to(cuda_device))
        return first, _np(e.current_pattern)          # max_steps=1: every array was redrawn by the autoreset

    whole = draws(n, 0)
    halves = [draws(n // 2, 0), draws(n // 2, n // 2)]
    for k in range(2):
        _same(np.concatenate([h[k] for h in halves]), whole[k], ("array_offset sharding", k))


@pytest.mark.gpu
@pytest.mark.parametrize("size", KERNEL_SIZES, ids=lambda s: f"{s[0]}x{s[1]}")
def test_cuda_coupling_sum_skips_the_device_itself(size, cuda_device):
    """The reference's coupling sum runs over j != i. The env's coupling matrices have a zero diagonal, which hides a
    kernel that multiplies it instead; with a nonzero diagonal in the shared buffer, every kernel must still skip it."""
    import torch
    nd, n = size[0] * size[1], 6
    rng = np.random.default_rng(nd + 1)
    p0, tgt = start_state(rng, n, size)
    env = _gpu_env(cuda_device, size, "stt_mram", "dipolar", "global", n, 200)
    coupling = _coupling(size, "dipolar").copy()
    np.fill_diagonal(coupling, 3 * STRENGTH)
    env._coupling.copy_(torch.from_numpy(coupling))
    env.reset(options={"initial_pattern": p0.reshape((n,) + size + (3,)), "target_pattern": tgt.reshape((n,) + size + (3,))})
    act = random_actions(rng, n, size, "global")
    o, r, te, tr, info = env.step(torch.from_numpy(act).to(cuda_device))
    host = HostArrays(size, "stt_mram", "dipolar", "global", 200, p0, tgt)
    host.coupling = coupling
    host.step(act)
    _same(_np(env.current_pattern).reshape(n, nd, 3), host.pattern, "pattern")
    _same(_np(r), host.reward, "reward")
    ora = make_oracle(size, "stt_mram", "dipolar", "global", 200, p0[0], tgt[0])
    ora.coupling = coupling
    ref = ora.step(act[0].copy())
    check_against_oracle(0, ora, ref, host.pattern[0], host.obs[0], host.reward[0], host.energy[0], host.similarity[0],
                         host.terminated[0], host.truncated[0], (size, "nonzero diagonal"))
