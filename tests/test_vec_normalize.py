"""K8: VecNormalize on the GPU (stg_vecnorm_moments_f32 / stg_vecnorm_merge_f64 / stg_vecnorm_apply_f32, stg.VecNormalize).

The specification is Stable-Baselines3's VecNormalize with RunningMeanStd, restated below in NumPy as SB3 writes it and fed
float64 data. update_from_moments, the normalisations and the return update are compared bit for bit (np.array_equal); the
batch moments are a parallel reduction, equal to np.mean / np.var up to FP64 summation order."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

from spin_torque_rl_gym_b200 import _lib
from tests.helpers import ROOT

HEADER = os.path.join(ROOT, "include", "stg.h")
CSRC = os.path.join(ROOT, "spin_torque_rl_gym_b200", "csrc")


# ---------------------------------------------------------------------------------------------------- SB3, restated -------

class RunningMeanStd:
    """stable_baselines3.common.running_mean_std.RunningMeanStd."""

    def __init__(self, epsilon=1e-4, shape=()):
        self.mean = np.zeros(shape, np.float64)
        self.var = np.ones(shape, np.float64)
        self.count = epsilon

    def update(self, arr):
        batch_mean = np.mean(arr, axis=0)
        batch_var = np.var(arr, axis=0)
        batch_count = arr.shape[0]
        self.update_from_moments(batch_mean, batch_var, batch_count)

    def update_from_moments(self, batch_mean, batch_var, batch_count):
        delta = batch_mean - self.mean
        tot_count = self.count + batch_count
        new_mean = self.mean + delta * batch_count / tot_count
        m_a = self.var * self.count
        m_b = batch_var * batch_count
        m_2 = m_a + m_b + np.square(delta) * self.count * batch_count / (self.count + batch_count)
        new_var = m_2 / (self.count + batch_count)
        new_count = batch_count + self.count
        self.mean = new_mean
        self.var = new_var
        self.count = new_count


class SB3VecNormalize:
    """VecNormalize.reset / step_wait / normalize_obs / normalize_reward / _update_reward over arrays: obs [N,12] float64,
    reward [N] float64, dones [N] bool, final [N,12] float64 (SB3 reads infos[i]['terminal_observation'] of done envs)."""

    def __init__(self, n, training=True, norm_obs=True, norm_reward=True, clip_obs=10.0, clip_reward=10.0, gamma=0.99,
                 epsilon=1e-8):
        self.obs_rms, self.ret_rms = RunningMeanStd(shape=(12,)), RunningMeanStd(shape=())
        self.training, self.norm_obs, self.norm_reward = training, norm_obs, norm_reward
        self.clip_obs, self.clip_reward, self.gamma, self.epsilon = clip_obs, clip_reward, gamma, epsilon
        self.returns = np.zeros(n)

    def _normalize_obs(self, obs, obs_rms):
        return np.clip((obs - obs_rms.mean) / np.sqrt(obs_rms.var + self.epsilon), -self.clip_obs, self.clip_obs)

    def normalize_obs(self, obs):
        if self.norm_obs:
            return self._normalize_obs(obs, self.obs_rms).astype(np.float32)
        return obs.astype(np.float32)

    def normalize_reward(self, reward):
        if self.norm_reward:
            reward = np.clip(reward / np.sqrt(self.ret_rms.var + self.epsilon), -self.clip_reward, self.clip_reward)
        return reward

    def _update_reward(self, reward):
        self.returns = self.returns * self.gamma + reward
        self.ret_rms.update(self.returns)

    def reset(self, obs):
        self.returns = np.zeros(len(obs))
        if self.training and self.norm_obs:
            self.obs_rms.update(obs)
        return self.normalize_obs(obs)

    def step(self, obs, reward, dones, final):
        if self.training and self.norm_obs:
            self.obs_rms.update(obs)
        obs = self.normalize_obs(obs)
        if self.training:
            self._update_reward(reward)
        reward = self.normalize_reward(reward)
        final = self.normalize_obs(final[dones])
        self.returns[dones] = 0
        return obs, reward, final


# ---------------------------------------------------------------------------------------------------- host build ----------

@pytest.fixture(scope="module")
def host_core(tmp_path_factory):
    """vecnorm_core.cuh compiled for the host with g++."""
    d = tmp_path_factory.mktemp("vecnorm_host")
    src = d / "vecnorm_host.cpp"
    src.write_text('#include "vecnorm_core.cuh"\n'
                   'using namespace stg;\n'
                   'extern "C" void upd(double* mean, double* var, double count, const double* bm, const double* bv, double bc,\n'
                   '                    int64_t n) { for (int64_t k = 0; k < n; ++k) vn_update_from_moments(mean[k], var[k], count,\n'
                   '                                                                                      bm[k], bv[k], bc); }\n'
                   'extern "C" void norm_obs(const float* x, int64_t n, const double* mean, const double* var, double eps,\n'
                   '                         double clip, float* out) {\n'
                   '  for (int64_t i = 0; i < n; ++i) for (int f = 0; f < 12; ++f)\n'
                   '    out[i * 12 + f] = vn_norm_obs(x[i * 12 + f], mean[f], vn_scale(var[f], eps), clip); }\n'
                   'extern "C" void norm_reward(const double* r, int64_t n, double var, double eps, double clip, double* out) {\n'
                   '  for (int64_t i = 0; i < n; ++i) out[i] = vn_norm_reward(r[i], vn_scale(var, eps), clip); }\n'
                   'extern "C" void returns(double* ret, double gamma, const double* r, int64_t n) {\n'
                   '  for (int64_t i = 0; i < n; ++i) ret[i] = vn_return(ret[i], gamma, r[i]); }\n'
                   '// the moment vector of rows [n][13] the way one thread of the moments kernel accumulates them\n'
                   'extern "C" void moments(const double* x, int64_t n, double* out) {\n'
                   '  double s1[13] = {0}, s2[13] = {0};\n'
                   '  out[0] = (double)n;\n'
                   '  for (int f = 0; f < 13; ++f) {\n'
                   '    const double x0 = n ? x[f] : 0.0;\n'
                   '    for (int64_t i = 0; i < n; ++i) { const double d = x[i * 13 + f] - x0; s1[f] += d; s2[f] += d * d; }\n'
                   '    vn_shifted_to_moments((double)n, x0, s1[f], s2[f], out[1 + f], out[14 + f]);\n'
                   '  } }\n'
                   'extern "C" void fold(const double* v, int g, double* out) { vn_fold(v, g, out); }\n')
    so = d / "vecnorm_host.so"
    subprocess.run(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-I", CSRC, str(src), "-o", str(so)], check=True)
    lib = C.CDLL(str(so))
    dp, i64 = C.c_void_p, C.c_int64
    lib.upd.argtypes = [dp, dp, C.c_double, dp, dp, C.c_double, i64]
    lib.norm_obs.argtypes = [dp, i64, dp, dp, C.c_double, C.c_double, dp]
    lib.norm_reward.argtypes = [dp, i64, C.c_double, C.c_double, C.c_double, dp]
    lib.returns.argtypes = [dp, C.c_double, dp, i64]
    lib.moments.argtypes = [dp, i64, dp]
    lib.fold.argtypes = [dp, C.c_int, dp]
    lib.path = str(so)
    return lib


def _p(a):
    return a.ctypes.data


def host_moments(lib, rows):
    rows = np.ascontiguousarray(rows, np.float64)
    out = np.empty(27)
    lib.moments(_p(rows), len(rows), _p(out))
    return out


def host_fold(lib, vecs):
    vecs = np.ascontiguousarray(vecs, np.float64)
    out = np.empty(27)
    lib.fold(_p(vecs), len(vecs), _p(out))
    return out


# ---------------------------------------------------------------------------------------------------- CPU ---------------

def test_vecnorm_args_layout_and_constants_match_the_c_header(tmp_path):
    fields = [f for f, _ in _lib.StgVecNormArgs._fields_]
    consts = ["STG_VECNORM_FEATURES", "STG_VECNORM_MOMENTS", "STG_VECNORM_STATS", "STG_VECNORM_OBS_VAR",
              "STG_VECNORM_OBS_COUNT", "STG_VECNORM_RET_MEAN", "STG_VECNORM_RET_VAR", "STG_VECNORM_RET_COUNT",
              "STG_VECNORM_MAX_CTAS", "STG_VECNORM_WORK_DOUBLES", "STG_VECNORM_TRAINING", "STG_VECNORM_NORM_OBS",
              "STG_VECNORM_NORM_REWARD", "STG_ABI_VERSION"]
    lines = ['#include <stdio.h>', '#include <stddef.h>', f'#include "{HEADER}"', 'int main(void){',
             'printf("size %zu\\n", sizeof(StgVecNormArgs));']
    lines += [f'printf("{f} %zu\\n", offsetof(StgVecNormArgs, {f}));' for f in fields]
    lines += [f'printf("{c} %lld\\n", (long long)({c}));' for c in consts]
    lines += [f'printf("grid{n} %lld\\n", (long long)STG_VECNORM_GRID((long long){n}));' for n in (0, 1, 256, 257, 75776, 75777, 1 << 20)]
    lines.append('return 0;}')
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", str(src), "-o", str(exe)], check=True)
    got = dict(l.split() for l in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split("\n") if l)
    assert int(got["size"]) == C.sizeof(_lib.StgVecNormArgs)
    for f in fields:
        assert int(got[f]) == getattr(_lib.StgVecNormArgs, f).offset, f
    assert int(got["STG_VECNORM_MOMENTS"]) == _lib.VECNORM_MOMENTS == 27 and int(got["STG_VECNORM_FEATURES"]) == 13
    assert int(got["STG_VECNORM_STATS"]) == _lib.VECNORM_STATS == 28
    assert [int(got[c]) for c in consts[3:8]] == [12, 24, 25, 26, 27]
    assert int(got["STG_VECNORM_MAX_CTAS"]) == _lib.VECNORM_MAX_CTAS
    assert int(got["STG_VECNORM_WORK_DOUBLES"]) == _lib.VECNORM_WORK_DOUBLES
    assert [int(got[c]) for c in consts[10:13]] == [_lib.VECNORM_TRAINING, _lib.VECNORM_NORM_OBS, _lib.VECNORM_NORM_REWARD]
    assert int(got["STG_ABI_VERSION"]) == _lib.ABI_VERSION == 7
    assert [int(got[f"grid{n}"]) for n in (0, 1, 256, 257, 75776, 75777, 1 << 20)] == [0, 1, 1, 2, 296, 296, 296]


def _vargs(n=4, **ptrs):
    a = _lib.StgVecNormArgs()
    a.n_envs, a.n_ranks = n, 1
    for k, v in ptrs.items():
        setattr(a, k, v)
    return a


def test_vecnorm_argument_validation():
    lib = _lib.load()
    mom, mrg, app = lib.stg_vecnorm_moments_f32, lib.stg_vecnorm_merge_f64, lib.stg_vecnorm_apply_f32
    call = lambda f, a: f(C.byref(a), None)                                 # noqa: E731
    B = 0x10000
    for f in (mom, mrg, app):
        assert f(None, None) == -1                                          # STG_E_NULL
    # moments
    ok = dict(d_obs=B, d_moments=B * 2, d_work=B * 3)
    assert call(mom, _vargs(-1, **ok)) == -2                                # STG_E_SIZE
    assert call(mom, _vargs(0, **ok)) == 0 and call(mom, _vargs(0)) == 0    # empty batch: STG_OK without a launch
    for k in ok:
        assert call(mom, _vargs(**{q: v for q, v in ok.items() if q != k})) == -1, k
    assert call(mom, _vargs(d_reward=B * 4, **ok)) == -1                    # reward without returns
    assert call(mom, _vargs(**dict(ok, d_obs=B + 8))) == -4                 # STG_E_ALIGN
    # merge (n_envs is not read: it checks n_ranks)
    a = _vargs(d_moments=B, d_stats=B)
    a.n_ranks = 0
    assert call(mrg, a) == -2
    assert call(mrg, _vargs(d_moments=B)) == -1 and call(mrg, _vargs(d_stats=B)) == -1
    # apply
    assert call(app, _vargs(-1, d_stats=B, d_obs=B, d_obs_out=B)) == -2
    assert call(app, _vargs(0)) == 0
    assert call(app, _vargs(d_obs=B, d_obs_out=B)) == -1                    # no statistics
    assert call(app, _vargs(d_stats=B)) == -1                               # no pair at all
    for half in ("d_obs", "d_obs_out", "d_final_obs", "d_final_obs_out", "d_reward", "d_reward_out"):
        assert call(app, _vargs(d_stats=B, d_terminated=B, d_truncated=B, **{half: B})) == -1, half
    assert call(app, _vargs(d_stats=B, d_final_obs=B, d_final_obs_out=B)) == -1             # final rows need the flags
    assert call(app, _vargs(d_stats=B, d_reward=B, d_reward_out=B, d_terminated=B)) == -1   # one flag array only
    for field in ("d_obs", "d_obs_out", "d_final_obs", "d_final_obs_out"):
        a = _vargs(d_stats=B, d_obs=B, d_obs_out=B, d_final_obs=B, d_final_obs_out=B, d_terminated=B, d_truncated=B)
        setattr(a, field, getattr(a, field) + 4)
        assert call(app, a) == -4, field


def _rng_stats(rng, shape):
    mean = rng.normal(size=shape) * rng.choice([1e-3, 1.0, 1e3], size=shape)
    var = rng.exponential(size=shape) * rng.choice([1e-12, 1e-2, 1.0, 1e4], size=shape)
    return mean, var


def test_update_from_moments_is_bit_equal(host_core):
    rng = np.random.default_rng(0)
    for count, bc in ((1e-4, 65536.0), (1e-4 + 65536, 65536.0), (123456789.0001, 3.0), (7.5, 1048576.0)):
        mean, var = _rng_stats(rng, 1000)
        bm, bv = _rng_stats(rng, 1000)
        ref = RunningMeanStd(shape=(1000,))
        ref.mean, ref.var, ref.count = mean.copy(), var.copy(), count
        ref.update_from_moments(bm, bv, int(bc))
        m, v = mean.copy(), var.copy()
        host_core.upd(_p(m), _p(v), count, _p(bm), _p(bv), bc, 1000)
        assert np.array_equal(m, ref.mean) and np.array_equal(v, ref.var), count
        assert ref.count == bc + count


def test_normalisations_and_return_update_are_bit_equal(host_core):
    rng = np.random.default_rng(1)
    ref = SB3VecNormalize(4096, clip_obs=5.0, clip_reward=3.0, gamma=0.995)
    ref.obs_rms.mean, ref.obs_rms.var = _rng_stats(rng, 12)
    ref.obs_rms.var[7] = 1e-17                                              # a constant column: scale ~ sqrt(eps)
    ref.ret_rms.var = 0.37
    obs = (rng.normal(size=(4096, 12)) * 10 ** rng.uniform(-3, 3, size=(4096, 12))).astype(np.float32)
    obs[:5] = [np.inf], [-np.inf], [0.0], [-0.0], [np.float32(1e30)]
    want = ref.normalize_obs(obs.astype(np.float64))
    assert (np.abs(want) == 5.0).any() and (np.abs(want) < 5.0).any()      # values beyond +-clip on both sides
    got = np.empty_like(obs)
    host_core.norm_obs(_p(obs), 4096, _p(ref.obs_rms.mean), _p(ref.obs_rms.var), 1e-8, 5.0, _p(got))
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    reward = rng.normal(size=4096) * 10 ** rng.uniform(-3, 2, size=4096)
    got_r = np.empty(4096)
    host_core.norm_reward(_p(reward), 4096, float(ref.ret_rms.var), 1e-8, 3.0, _p(got_r))
    assert np.array_equal(got_r, ref.normalize_reward(reward))
    ret = rng.normal(size=4096) * 100
    ref.returns = ret.copy()
    ref._update_reward(reward)
    host_core.returns(_p(ret), 0.995, _p(reward), 4096)
    assert np.array_equal(ret, ref.returns)


@pytest.mark.parametrize("splits", [[1000], [1, 999], [500, 500], [37, 0, 963], [256] * 3 + [232], [0, 1000]])
def test_chan_fold_of_split_batches_equals_one_batch(host_core, splits):
    rng = np.random.default_rng(len(splits))
    x = rng.normal(size=(sum(splits), 13)) * np.array([1e-3, 1, 1e3] * 4 + [50]) + np.array([0, 5, -1e4] * 4 + [1e3])
    x[:, 7] = 1.0                                                           # constant column (o[7] = T / 300)
    parts, lo = [], 0
    for s in splits:
        parts.append(host_moments(host_core, x[lo:lo + s]))
        lo += s
    v = host_fold(host_core, parts)
    assert v[0] == len(x)
    assert np.allclose(v[1:14], x.mean(0), rtol=1e-12, atol=1e-18)
    assert np.allclose(v[14:] / v[0], x.var(0), rtol=1e-12, atol=0)
    assert v[1 + 7] == 1.0 and v[14 + 7] == 0.0                             # exact for a constant column
    assert np.array_equal(host_fold(host_core, parts), v)
    empty = host_moments(host_core, x[:0])
    assert np.array_equal(empty, np.zeros(27))
    assert np.array_equal(host_fold(host_core, [empty] + parts + [empty]), v)     # empty vectors change no bit


GLOO_WORKER = r'''
import ctypes as C, json, sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import torch, torch.distributed as dist
from spin_torque_rl_gym_b200.parallel import all_gather_moments
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
lib = C.CDLL(sys.argv[2])
lib.moments.argtypes = [C.c_void_p, C.c_int64, C.c_void_p]
lib.fold.argtypes = [C.c_void_p, C.c_int, C.c_void_p]
x = np.random.default_rng(rank).normal(size=(1000 + 7 * rank, 13)) * (rank + 1)
local = np.empty(27)
lib.moments(x.ctypes.data, len(x), local.ctypes.data)
g = all_gather_moments(torch.from_numpy(local)).numpy()
folded = np.empty(27)
lib.fold(np.ascontiguousarray(g).ctypes.data, len(g), folded.ctypes.data)
with open(f"{sys.argv[3]}/rank{rank}.json", "w") as fh:
    json.dump({"rank": rank, "shape": list(g.shape), "local": local.tobytes().hex(), "rows": [r.tobytes().hex() for r in g],
               "folded": folded.tobytes().hex()}, fh)
dist.destroy_process_group()
'''


def test_all_gather_moments_world_size_2(tmp_path, host_core):
    import json
    import torch
    from spin_torque_rl_gym_b200.parallel import all_gather_moments
    v = torch.arange(27, dtype=torch.float64)
    assert torch.equal(all_gather_moments(v), v[None])                     # no process group: no collective
    script = tmp_path / "worker.py"
    script.write_text(GLOO_WORKER)
    env = dict(os.environ, MASTER_ADDR="127.0.0.1")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr", "127.0.0.1",
           "--master-port", "29541", str(script), ROOT, host_core.path, str(tmp_path)]
    res = subprocess.run(cmd, capture_output=True, text=True, env=env, timeout=240)
    assert res.returncode == 0, res.stderr[-2000:]
    outs = [json.loads((tmp_path / f"rank{r}.json").read_text()) for r in range(2)]
    assert [o["rank"] for o in outs] == [0, 1]
    for o in outs:
        assert o["shape"] == [2, 27]
        assert o["rows"] == [outs[0]["local"], outs[1]["local"]]            # rank order
    assert outs[0]["folded"] == outs[1]["folded"]                           # both ranks fold identical bits
    x = np.concatenate([np.random.default_rng(r).normal(size=(1000 + 7 * r, 13)) * (r + 1) for r in range(2)])
    folded = np.frombuffer(bytes.fromhex(outs[0]["folded"]))
    assert folded[0] == len(x) and np.allclose(folded[1:14], x.mean(0), rtol=1e-12, atol=1e-15)
    assert np.allclose(folded[14:] / folded[0], x.var(0), rtol=1e-12)


# ---------------------------------------------------------------------------------------------------- GPU ---------------

def _dev_args(torch, n, flags, **tensors):
    a = _lib.StgVecNormArgs()
    a.gamma, a.epsilon, a.clip_obs, a.clip_reward = 0.99, 1e-8, 10.0, 10.0
    a.n_envs, a.n_ranks, a.flags = n, 1, flags
    for k, t in tensors.items():
        setattr(a, k, None if t is None else t.data_ptr())
    return a


def _stats_tensor(torch, dev, obs_rms, ret_rms):
    s = np.concatenate([obs_rms.mean, obs_rms.var, [obs_rms.count, ret_rms.mean, ret_rms.var, ret_rms.count]])
    return torch.from_numpy(s).to(dev)


def _run(torch, fn, a):
    _lib.check(fn(C.byref(a), torch.cuda.current_stream().cuda_stream), "stg_vecnorm")


@pytest.mark.gpu
@pytest.mark.parametrize("n", [1, 1000, 65536 + 17])
def test_cuda_apply_with_given_statistics_is_bit_equal(cuda_device, n):
    import torch
    lib = _lib.load()
    rng = np.random.default_rng(n)
    ref = SB3VecNormalize(n, clip_obs=4.0, clip_reward=2.5)
    ref.obs_rms.mean, ref.obs_rms.var = _rng_stats(rng, 12)
    ref.ret_rms.mean, ref.ret_rms.var = 0.3, 0.81
    obs = (rng.normal(size=(n, 12)) * 10 ** rng.uniform(-3, 3, size=(n, 12))).astype(np.float32)
    final = (rng.normal(size=(n, 12)) * 10).astype(np.float32)
    term, trunc = rng.random(n) < 0.2, rng.random(n) < 0.2
    ended = term | trunc
    reward = rng.normal(size=n) * 5
    returns = rng.normal(size=n)
    d = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(cuda_device)         # noqa: E731
    t_obs, t_final, t_rew, t_ret = d(obs), d(final), d(reward), d(returns)
    t_te, t_tr = d(term.astype(np.uint8)), d(trunc.astype(np.uint8))
    o_obs = torch.full((n, 12), -7.0, device=cuda_device)
    o_fin = torch.full((n, 12), -7.0, device=cuda_device)
    o_rew = torch.empty(n, dtype=torch.float64, device=cuda_device)
    stats = _stats_tensor(torch, cuda_device, ref.obs_rms, ref.ret_rms)
    stats_before = stats.clone()
    a = _dev_args(torch, n, _lib.VECNORM_TRAINING | _lib.VECNORM_NORM_OBS | _lib.VECNORM_NORM_REWARD, d_obs=t_obs,
                  d_obs_out=o_obs, d_final_obs=t_final, d_final_obs_out=o_fin, d_terminated=t_te, d_truncated=t_tr,
                  d_reward=t_rew, d_reward_out=o_rew, d_returns=t_ret, d_stats=stats)
    a.clip_obs, a.clip_reward = 4.0, 2.5
    _run(torch, lib.stg_vecnorm_apply_f32, a)
    want_obs = ref.normalize_obs(obs.astype(np.float64))
    assert np.array_equal(o_obs.cpu().numpy().view(np.uint32), want_obs.view(np.uint32))
    got_fin = o_fin.cpu().numpy()
    assert np.array_equal(got_fin[ended].view(np.uint32), ref.normalize_obs(final[ended].astype(np.float64)).view(np.uint32))
    assert (got_fin[~ended] == -7.0).all()                                  # rows of running envs are not written
    assert np.array_equal(o_rew.cpu().numpy(), ref.normalize_reward(reward))
    want_ret = returns.copy()
    want_ret[ended] = 0
    assert np.array_equal(t_ret.cpu().numpy(), want_ret)
    assert torch.equal(stats, stats_before)                                 # apply never updates the statistics
    # without NORM_OBS / NORM_REWARD: copies
    a.flags = 0
    _run(torch, lib.stg_vecnorm_apply_f32, a)
    assert torch.equal(o_obs, t_obs) and torch.equal(o_rew, t_rew)


def _moments_and_merge(torch, dev, obs, reward, returns, stats, work, flags, moments=None):
    lib = _lib.load()
    n = obs.shape[0]
    mom = torch.empty(27, dtype=torch.float64, device=dev) if moments is None else moments
    a = _dev_args(torch, n, flags, d_obs=obs, d_reward=reward, d_returns=returns, d_stats=stats, d_moments=mom, d_work=work)
    _run(torch, lib.stg_vecnorm_moments_f32, a)
    _run(torch, lib.stg_vecnorm_merge_f64, a)
    return mom


@pytest.mark.gpu
@pytest.mark.parametrize("n", [200, 1000, 100003, 1 << 20])
def test_cuda_moments_are_deterministic_and_match_numpy(cuda_device, n):
    import torch
    dev = cuda_device
    g = torch.Generator(device=dev).manual_seed(n)
    obs = torch.randn(n, 12, generator=g, device=dev) * 3 + 1
    obs[:, 7] = 1.0
    reward = torch.randn(n, generator=g, device=dev, dtype=torch.float64)
    ret0 = torch.randn(n, generator=g, device=dev, dtype=torch.float64)
    init = _stats_tensor(torch, dev, RunningMeanStd(shape=(12,)), RunningMeanStd())
    flags = _lib.VECNORM_TRAINING | _lib.VECNORM_NORM_OBS
    work = torch.zeros(_lib.VECNORM_WORK_DOUBLES, dtype=torch.float64, device=dev)
    runs = []
    for _ in range(2):
        stats, ret = init.clone(), ret0.clone()
        mom = _moments_and_merge(torch, dev, obs, reward, ret, stats, work, flags)
        runs.append((mom.clone(), stats.clone(), ret.clone()))
    for x, y in zip(*runs):
        assert torch.equal(x.view(torch.int64), y.view(torch.int64))
    assert float(work[-1]) == 0.0                                           # the CTA counter is left at zero
    mom, stats, ret = (t.cpu().numpy() for t in runs[0])
    want_ret = ret0.cpu().numpy() * 0.99 + reward.cpu().numpy()
    assert np.array_equal(ret, want_ret)
    x = np.concatenate([obs.cpu().numpy().astype(np.float64), want_ret[:, None]], 1)
    assert mom[0] == n
    assert np.allclose(mom[1:14], x.mean(0), rtol=1e-12, atol=1e-300)
    assert np.allclose(mom[14:] / n, x.var(0), rtol=1e-12, atol=1e-300)
    assert mom[1 + 7] == 1.0 and mom[14 + 7] == 0.0
    ref_o, ref_r = RunningMeanStd(shape=(12,)), RunningMeanStd()
    ref_o.update(x[:, :12])
    ref_r.update(x[:, 12])
    assert np.allclose(stats[:12], ref_o.mean, rtol=1e-12, atol=1e-300) and np.allclose(stats[12:24], ref_o.var, rtol=1e-12)
    assert stats[24] == ref_o.count and stats[27] == ref_r.count
    assert np.isclose(stats[25], ref_r.mean, rtol=1e-12) and np.isclose(stats[26], ref_r.var, rtol=1e-12)


@pytest.mark.gpu
def test_cuda_merge_of_shards_equals_the_whole_batch(cuda_device):
    import torch
    dev, n = cuda_device, 300001
    lib = _lib.load()
    g = torch.Generator(device=dev).manual_seed(5)
    obs = torch.randn(n, 12, generator=g, device=dev) * 2 - 3
    reward = torch.randn(n, generator=g, device=dev, dtype=torch.float64)
    init = _stats_tensor(torch, dev, RunningMeanStd(shape=(12,)), RunningMeanStd())
    flags = _lib.VECNORM_TRAINING | _lib.VECNORM_NORM_OBS
    work = torch.zeros(_lib.VECNORM_WORK_DOUBLES, dtype=torch.float64, device=dev)
    whole = init.clone()
    _moments_and_merge(torch, dev, obs, reward, torch.zeros(n, dtype=torch.float64, device=dev), whole, work, flags)
    h = 123457                                                               # unequal shards, not a multiple of the block
    stack = torch.empty(2, 27, dtype=torch.float64, device=dev)
    for r, (lo, hi) in enumerate(((0, h), (h, n))):
        a = _dev_args(torch, hi - lo, flags, d_obs=obs[lo:hi], d_reward=reward[lo:hi],
                      d_returns=torch.zeros(hi - lo, dtype=torch.float64, device=dev), d_moments=stack[r], d_work=work)
        _run(torch, lib.stg_vecnorm_moments_f32, a)
    merged = []
    for _ in range(2):
        s = init.clone()
        a = _dev_args(torch, n, flags, d_moments=stack, d_stats=s, d_reward=reward)
        a.n_ranks = 2
        _run(torch, lib.stg_vecnorm_merge_f64, a)
        merged.append(s)
    assert torch.equal(merged[0].view(torch.int64), merged[1].view(torch.int64))     # same stack, same bits
    assert torch.allclose(merged[0], whole, rtol=1e-12, atol=1e-300)


def _venv(stg, dev, n, max_steps=5, seed=3, **kw):
    return stg.make("SpinTorque-v0", num_envs=n, device=dev, max_steps=max_steps, max_current=1.1e-6, rng_seed=seed, **kw)


def _actions(torch, dev, n, g):
    act = torch.empty(n, 2, device=dev)
    act[:, 0] = (torch.rand(n, generator=g, device=dev) * 2 - 1) * 1.1e-6
    act[:, 1] = torch.rand(n, generator=g, device=dev) * 1e-9 + 1e-11
    return act


def _check_stats(norm, ref, rtol=1e-12):
    s = norm._stats.cpu().numpy()
    # means: 1e-15 absolute as well, for columns whose mean is near zero (only the summation order differs)
    assert np.allclose(s[:12], ref.obs_rms.mean, rtol=rtol, atol=1e-15)
    assert np.allclose(s[12:24], ref.obs_rms.var, rtol=rtol, atol=1e-300)
    assert np.isclose(s[25], ref.ret_rms.mean, rtol=rtol, atol=1e-15) and np.isclose(s[26], ref.ret_rms.var, rtol=rtol)
    assert s[24] == ref.obs_rms.count and s[27] == ref.ret_rms.count


def _sequence(stg, torch, dev, n, steps, tol=1e-5, **opts):
    venv = _venv(stg, dev, n)
    norm = stg.VecNormalize(venv, **opts)
    ref = SB3VecNormalize(n, **opts)
    g = torch.Generator(device=dev).manual_seed(11)
    obs, _ = norm.reset(seed=3)
    want = ref.reset(norm.get_original_obs().cpu().numpy().astype(np.float64))
    assert np.abs(obs.cpu().numpy() - want).max() <= tol
    _check_stats(norm, ref)
    ended_total = 0
    for _ in range(steps):
        obs, rew, term, trunc, info = norm.step(_actions(torch, dev, n, g))
        dones = (term | trunc).cpu().numpy()
        ended_total += int(dones.sum())
        raw_final = venv._final_obs.cpu().numpy().astype(np.float64)
        w_obs, w_rew, w_fin = ref.step(norm.get_original_obs().cpu().numpy().astype(np.float64),
                                       norm.get_original_reward().cpu().numpy(), dones, raw_final)
        assert np.abs(obs.cpu().numpy() - w_obs).max() <= tol
        assert np.abs(rew.cpu().numpy() - w_rew).max() <= tol
        assert np.abs(info["final_observation"].cpu().numpy()[dones] - w_fin).max(initial=0.0) <= tol
        assert np.allclose(norm._returns.cpu().numpy(), ref.returns, rtol=1e-12, atol=1e-300)
        _check_stats(norm, ref)
    assert ended_total > 0
    return norm, ref


@pytest.mark.gpu
def test_cuda_sequence_matches_sb3_restatement(cuda_device):
    import torch
    import spin_torque_rl_gym_b200 as stg
    norm, ref = _sequence(stg, torch, cuda_device, 65536, 64)
    assert ref.obs_rms.count > 65 * 65536


@pytest.mark.gpu
@pytest.mark.parametrize("opts", [dict(training=False), dict(norm_obs=False), dict(norm_reward=False),
                                  dict(clip_obs=0.5, clip_reward=0.1, gamma=0.9, epsilon=1e-4)])
def test_cuda_options_follow_sb3(cuda_device, opts):
    import torch
    import spin_torque_rl_gym_b200 as stg
    norm, ref = _sequence(stg, torch, cuda_device, 4096, 8, **opts)
    if opts.get("training") is False:
        assert ref.obs_rms.count == 1e-4 and ref.ret_rms.count == 1e-4


@pytest.mark.gpu
def test_cuda_wrapper_interface_state_dict_and_no_sync(cuda_device):
    import torch
    import spin_torque_rl_gym_b200 as stg
    dev, n = cuda_device, 4096
    venv = _venv(stg, dev, n)
    norm = stg.VecNormalize(venv)
    assert norm.num_envs == n and norm.device == venv.device and norm.autoreset and not norm.host_outputs
    assert norm.rng_seed == venv.rng_seed and norm.env_offset == venv.env_offset and norm._torch is torch
    assert norm.single_observation_space is venv.single_observation_space and norm.max_steps == 5   # forwarded
    for rms, shape in ((norm.obs_rms, (12,)), (norm.ret_rms, ())):
        assert rms.mean.shape == shape and rms.var.shape == shape and rms.count.shape == ()
        assert all(t.dtype == torch.float64 and t.device == venv.device for t in (rms.mean, rms.var, rms.count))
    g = torch.Generator(device=dev).manual_seed(2)
    acts = [_actions(torch, dev, n, g) for _ in range(6)]
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        norm.reset(seed=4)
        for a in acts[:3]:
            norm.step(a)
        norm.normalize_obs(venv._obs)
        norm.normalize_reward(venv._reward)
    finally:
        torch.cuda.set_sync_debug_mode("default")
    count = 1e-4
    for _ in range(4):
        count = n + count
    assert float(norm.obs_rms.count) == count
    # normalize_* use the current statistics and the kernel of step()
    o = norm.normalize_obs(norm.get_original_obs())
    assert torch.equal(o, norm._obs)
    # a state_dict round trip reproduces the next step bit for bit
    sd_env, sd = venv.state_dict(), norm.state_dict()
    first = [t.clone() for t in norm.step(acts[3])[:2]] + [norm._stats.clone(), norm._returns.clone()]
    venv.load_state_dict(sd_env)
    norm.load_state_dict(sd)
    again = [t.clone() for t in norm.step(acts[3])[:2]] + [norm._stats.clone(), norm._returns.clone()]
    for x, y in zip(first, again):
        assert torch.equal(x, y)
    # masked reset: returns of the masked envs zeroed, statistics untouched
    stats = norm._stats.clone()
    ret = norm._returns.clone()
    mask = torch.zeros(n, dtype=torch.bool, device=dev)
    mask[::3] = True
    norm.reset(mask=mask)
    assert torch.equal(norm._stats, stats)
    assert torch.equal(norm._returns, torch.where(mask, torch.zeros_like(ret), ret))
    # errors
    with pytest.raises(ValueError):
        stg.VecNormalize(_venv(stg, dev, 16, host_outputs=True))
    with pytest.raises(NotImplementedError):
        norm.capture_step(acts[0])                                          # would capture the raw step
    with pytest.raises(AttributeError):
        norm._m                                                             # the env's private state is not forwarded
    # autoreset=False: no final rows
    plain = stg.VecNormalize(_venv(stg, dev, 64, autoreset=False))
    plain.reset(seed=1)
    _, _, _, _, info = plain.step(_actions(torch, dev, 64, g))
    assert "final_observation" not in info


@pytest.mark.gpu
def test_cuda_sb3_adapter_returns_normalised_terminal_observations(cuda_device):
    import torch
    import spin_torque_rl_gym_b200 as stg
    dev, n = cuda_device, 256
    norm = stg.VecNormalize(_venv(stg, dev, n, max_steps=2))
    sb3 = stg.SB3VecEnvAdapter(norm)
    obs = sb3.reset()
    assert np.array_equal(obs, norm._obs.cpu().numpy())
    rng = np.random.default_rng(0)
    ended = 0
    for _ in range(4):
        act = np.stack([rng.uniform(-1.1e-6, 1.1e-6, n), rng.uniform(1e-11, 1e-9, n)], 1).astype(np.float32)
        obs, rew, dones, infos = sb3.step(act)
        assert np.array_equal(obs, norm._obs.cpu().numpy())
        assert np.array_equal(rew, norm._reward.cpu().numpy().astype(np.float32))
        fin, raw = norm._final_obs.cpu().numpy(), norm.venv._final_obs.cpu().numpy()
        for i in np.nonzero(dones)[0]:
            assert np.array_equal(infos[i]["terminal_observation"], fin[i])
            assert not np.array_equal(fin[i], raw[i])
        ended += int(dones.sum())
    assert ended >= n                                                       # max_steps=2: every env ends at least once


@pytest.mark.gpu
def test_cuda_rollout_collector_on_the_wrapper(cuda_device):
    import torch
    import spin_torque_rl_gym_b200 as stg
    dev, n, T = cuda_device, 512, 16
    norm = stg.VecNormalize(_venv(stg, dev, n))
    gen = torch.Generator(device=dev).manual_seed(0)
    w1 = torch.randn(12, 32, generator=gen, device=dev) * 0.3
    wa = torch.randn(32, 2, generator=gen, device=dev) * 0.3

    def value_fn(o):
        return o[:, 9].clone()                                              # one observation column

    def policy(o):
        out = torch.tanh(o @ w1) @ wa
        act = torch.empty(o.shape[0], 2, device=dev)
        act[:, 0] = torch.tanh(out[:, 0]) * 1.1e-6
        act[:, 1] = torch.sigmoid(out[:, 1]) * 1e-9 + 1e-11
        return act, value_fn(o), -(out * out).sum(1)

    rec = []
    step = norm.step

    def recording_step(actions):
        out = step(actions)
        rec.append((out[0].clone(), out[1].clone(), out[4]["final_observation"].clone(), (out[2] | out[3]).clone()))
        return out

    norm.step = recording_step
    col = stg.RolloutCollector(norm, n_steps=T, store_values=True)
    col.collect(policy, value_fn)
    assert len(rec) == T
    assert sum(int(r[3].sum()) for r in rec) > 0
    for t in range(T):
        obs, rew, fin, _ = rec[t]
        assert torch.equal(col.rewards[t], rew.float())
        assert torch.equal(col.final_values[t], fin[:, 9])                  # V(normalised final observation)
        if t + 1 < T:
            assert torch.equal(col.observations[t + 1], obs)
    assert torch.equal(col.last_values, rec[-1][0][:, 9])
    assert float(col.observations.abs().max()) <= 10.0                      # clipped: these are normalised observations
    col.compute_returns_and_advantage()
    batches = list(col.get(1024))
    assert len(batches) == T * n // 1024 and batches[0].observations.shape == (1024, 12)
