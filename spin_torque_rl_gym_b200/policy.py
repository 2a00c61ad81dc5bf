"""Stable-Baselines3's PPO `MlpPolicy` for the GPU vector env, with rollout inference fused into one kernel launch (K9).

`ActorCriticPolicy` has the parameters, initialisation and torch methods of SB3's ActorCriticPolicy for a Box observation and a
Box action (net_arch pi=[64, 64], vf=[64, 64], tanh, FlattenExtractor, DiagGaussianDistribution with a state-independent
log_std), so SB3 state dicts load into it and back. Its `forward` and `predict_values`, which a rollout calls over all N envs
every step, run as single launches of stg_policy_act_f32 / stg_policy_value_f32 (include/stg.h); `evaluate_actions` is plain
torch with autograd. `ppo_backward` computes SB3's PPO.train() loss of a minibatch and writes every parameter's gradient in
one launch of stg_policy_ppo_grad_f32 plus a fold (K10)."""
from __future__ import annotations

import ctypes as C
import math
from typing import NamedTuple, Optional, Tuple

import numpy as np
import torch
from torch import nn

from . import _lib
from .envs.sb3_vec_env import _M64, _splitmix64

# domain tag of the action-noise key: "K9noise1" read as a little-endian 64-bit word
POLICY_NOISE_TAG = int.from_bytes(b"K9noise1", "little")
_DEFAULT_NET_ARCH = dict(pi=[64, 64], vf=[64, 64])


def policy_noise_key(seed: int) -> Tuple[int, int]:
    """The Philox key (low, high 32-bit words) of the action noise of an ActorCriticPolicy with this seed. A pure function:
    POLICY_NOISE_TAG and then the seed (mod 2^64) are in turn XORed into a 64-bit state (initially 0) and the state replaced by
    splitmix64's output for it; one more splitmix64 output from that state is the key. The tag keeps it apart from the env's
    thermal and reset noise, whose key is the seed itself."""
    state = 0
    for word in (POLICY_NOISE_TAG, seed):
        _, state = _splitmix64(state ^ (int(word) & _M64))
    _, z = _splitmix64(state)
    return z & 0xFFFFFFFF, z >> 32


class PPOLosses(NamedTuple):
    """The losses of one PPO minibatch with Stable-Baselines3's PPO.train() definitions, each a 0-d float32 tensor on the
    device: loss = policy_loss + ent_coef * entropy_loss + vf_coef * value_loss, approx_kl = mean((ratio - 1) - log ratio),
    clip_fraction = mean(|ratio - 1| > clip_range)."""
    loss: torch.Tensor
    policy_loss: torch.Tensor
    value_loss: torch.Tensor
    entropy_loss: torch.Tensor
    approx_kl: torch.Tensor
    clip_fraction: torch.Tensor


# the sample planes ppo_backward reads: (RolloutBufferSamples field, trailing shape, required alignment in bytes)
_PPO_PLANES = (("observations", (_lib.OBS_DIM,), 16), ("actions", (2,), 8), ("old_values", (), 4),
               ("old_log_prob", (), 4), ("advantages", (), 4), ("returns", (), 4))


class MlpExtractor(nn.Module):
    """SB3's MlpExtractor for net_arch pi=[64, 64], vf=[64, 64] and tanh."""

    def __init__(self, feature_dim: int):
        super().__init__()
        self.policy_net = nn.Sequential(nn.Linear(feature_dim, 64), nn.Tanh(), nn.Linear(64, 64), nn.Tanh())
        self.value_net = nn.Sequential(nn.Linear(feature_dim, 64), nn.Tanh(), nn.Linear(64, 64), nn.Tanh())
        self.latent_dim_pi = self.latent_dim_vf = 64

    def forward(self, features):
        return self.forward_actor(features), self.forward_critic(features)

    def forward_actor(self, features):
        return self.policy_net(features)

    def forward_critic(self, features):
        return self.value_net(features)


class DiagGaussianDistribution:
    """SB3's DiagGaussianDistribution: independent Normals over the action dimensions, log-probability and entropy summed."""

    def __init__(self, mean_actions, log_std):
        self.distribution = torch.distributions.Normal(mean_actions, torch.ones_like(mean_actions) * log_std.exp())

    def log_prob(self, actions):
        return self.distribution.log_prob(actions).sum(dim=1)

    def entropy(self):
        return self.distribution.entropy().sum(dim=1)

    def sample(self):
        return self.distribution.rsample()

    def mode(self):
        return self.distribution.mean

    def get_actions(self, deterministic: bool = False):
        return self.mode() if deterministic else self.sample()


class ActorCriticPolicy(nn.Module):
    """`ActorCriticPolicy(env, log_std_init=0.0, ortho_init=True, seed=None)`: SB3's PPO MlpPolicy for `env` (a
    SpinTorqueVectorEnv or a VecNormalize around one), on the env's device.

    The module has SB3's structure and parameter names (mlp_extractor.policy_net / value_net, action_net, value_net, log_std),
    so `load_state_dict(sb3_model.policy.state_dict())` works with strict=True and so does the reverse. Initialisation is
    SB3's: orthogonal weights with gain sqrt(2) for the extractor, 0.01 for action_net and 1 for value_net, zero biases, log_std
    = log_std_init. The kernels are specialised for this architecture: any other `net_arch` or `activation_fn` raises
    ValueError, as do observation or action spaces other than the env's 12 and 2 floats.

    Actions are in policy units: SB3 with `RescaleAction(env, -1, 1)` in front of the env. `scale_action` maps them to the env's
    Box (clip to [-1, 1], then rescale); the fused rollout path of RolloutCollector does that in the kernel.

    Action noise is Philox4x32-10 keyed by `noise_key()` (a function of `seed`, default the env's rng_seed) at counter (global
    env id, `noise_draws`): every sampling launch uses the current `noise_draws` and increments it. So samples depend on the
    seed, the env's global id and the draw, not on the torch RNG or on how the envs are split over launches or GPUs. The
    packed weight buffer and `noise_draws` are not part of `state_dict`."""

    def __init__(self, env, log_std_init: float = 0.0, ortho_init: bool = True, seed: Optional[int] = None,
                 net_arch=None, activation_fn=nn.Tanh):
        super().__init__()
        if net_arch is not None and net_arch not in (_DEFAULT_NET_ARCH, [64, 64]):
            raise ValueError(f"only net_arch={_DEFAULT_NET_ARCH} is supported (the K9 kernel is specialised for it), got "
                             f"{net_arch!r}")
        if activation_fn is not nn.Tanh:
            raise ValueError(f"only activation_fn=nn.Tanh is supported (the K9 kernel is specialised for it), got "
                             f"{activation_fn!r}")
        obs_shape = tuple(env.single_observation_space.shape)
        space = env.single_action_space
        if obs_shape != (_lib.OBS_DIM,) or tuple(space.shape) != (2,):
            raise ValueError(f"ActorCriticPolicy needs a 12-float observation and a 2-float action, got {obs_shape} and "
                             f"{tuple(space.shape)}")
        self.num_envs, self.device = env.num_envs, torch.device(env.device)
        self.env_offset = int(env.env_offset)
        self.seed = int(env.rng_seed if seed is None else seed) & _M64
        self.noise_draws = 0
        self.action_space = space
        self.ortho_init = ortho_init
        self.features_extractor = nn.Flatten()
        self.mlp_extractor = MlpExtractor(_lib.OBS_DIM)
        self.action_net = nn.Linear(64, 2)
        self.log_std = nn.Parameter(torch.ones(2) * log_std_init, requires_grad=True)
        self.value_net = nn.Linear(64, 1)
        if ortho_init:
            gains = ((self.mlp_extractor, math.sqrt(2)), (self.action_net, 0.01), (self.value_net, 1.0))
            for module, gain in gains:
                for m in module.modules():
                    if isinstance(m, nn.Linear):
                        nn.init.orthogonal_(m.weight, gain=gain)
                        m.bias.data.fill_(0.0)
        self.to(self.device)
        self._low = np.asarray(space.low, np.float32)
        self._high = np.asarray(space.high, np.float32)
        self._action_low = torch.as_tensor(self._low, device=self.device)
        self._action_high = torch.as_tensor(self._high, device=self.device)
        self._packed = None
        self._pad = None
        self._grad = None

    # ---- SB3's torch methods -----------------------------------------------------------------------------------------------
    def extract_features(self, obs):
        return self.features_extractor(obs.float())

    def _get_action_dist_from_latent(self, latent_pi) -> DiagGaussianDistribution:
        return DiagGaussianDistribution(self.action_net(latent_pi), self.log_std)

    def get_distribution(self, obs) -> DiagGaussianDistribution:
        return self._get_action_dist_from_latent(self.mlp_extractor.forward_actor(self.extract_features(obs)))

    def evaluate_actions(self, obs, actions):
        """(values [N,1], log_prob [N], entropy [N]) of `actions` (policy units) under the current weights, with autograd:
        SB3's evaluate_actions, which PPO's loss is built from."""
        latent_pi, latent_vf = self.mlp_extractor(self.extract_features(obs))
        distribution = self._get_action_dist_from_latent(latent_pi)
        log_prob = distribution.log_prob(actions)
        values = self.value_net(latent_vf)
        return values, log_prob, distribution.entropy()

    def predict(self, obs, deterministic: bool = False):
        """SB3's predict on a RescaleAction(-1, 1) env, in torch: (env actions [N,2], None). Sampling draws from the torch
        RNG like SB3; the clip to [-1, 1] and the rescale are `scale_action`."""
        with torch.no_grad():
            actions = self.get_distribution(obs).get_actions(deterministic=deterministic)
            return self.scale_action(actions), None

    def scale_action(self, actions):
        """Env actions of raw policy actions: lo + (hi - lo) * ((clip(a, -1, 1) + 1) / 2) in float32, each operation rounded
        on its own (SB3's clip to the [-1, 1] Box, then gymnasium's RescaleAction)."""
        lo, hi = self._action_low, self._action_high
        return lo + (hi - lo) * ((actions.float().clamp(-1.0, 1.0) + 1.0) / 2.0)

    # ---- K9 ------------------------------------------------------------------------------------------------------------------
    def noise_key(self) -> Tuple[int, int]:
        return policy_noise_key(self.seed)

    @torch.no_grad()
    def pack_weights(self):
        """Write every parameter, exp(log_std) and log(exp(log_std)) into the persistent device buffer of include/stg.h's
        STG_POLICY_* layout (matrices transposed to k-major) with one torch.cat, and return it."""
        dev = self.log_std.device
        if self._packed is None or self._packed.device != dev:
            self._packed = torch.empty(_lib.POLICY_FLOATS, dtype=torch.float32, device=dev)
            self._pad = torch.zeros(_lib.POLICY_FLOATS - _lib.POLICY_PARAMS - 4, dtype=torch.float32, device=dev)
        pi, vf = self.mlp_extractor.policy_net, self.mlp_extractor.value_net
        std = self.log_std.exp()
        torch.cat([pi[0].weight.t().reshape(-1), pi[0].bias, pi[2].weight.t().reshape(-1), pi[2].bias,
                   vf[0].weight.t().reshape(-1), vf[0].bias, vf[2].weight.t().reshape(-1), vf[2].bias,
                   self.action_net.weight.t().reshape(-1), self.action_net.bias, self.value_net.weight.reshape(-1),
                   self.value_net.bias, self.log_std, std, std.log(), self._pad], out=self._packed)
        return self._packed

    def _obs_rows(self, obs):
        if not isinstance(obs, torch.Tensor) or obs.device.type != "cuda":
            raise _lib.StgError("ActorCriticPolicy.forward / predict_values need a CUDA tensor (no CPU fallback)")
        if obs.device != self.log_std.device:
            raise ValueError(f"observations on {obs.device}, policy on {self.log_std.device}")
        obs = obs.reshape(-1, _lib.OBS_DIM)
        if obs.dtype != torch.float32 or not obs.is_contiguous() or obs.data_ptr() % 16:
            obs = obs.to(torch.float32).contiguous().clone()
        return obs

    def _args(self, weights, n: int) -> _lib.StgPolicyArgs:
        a = _lib.StgPolicyArgs()
        a.d_weights = weights.data_ptr()
        a.action_low[:] = [float(v) for v in self._low]
        a.action_high[:] = [float(v) for v in self._high]
        a.key[:] = list(self.noise_key())
        a.env_offset = self.env_offset
        a.n_envs = n
        return a

    def _launch(self, fn, a, what: str) -> None:
        dev = self.log_std.device
        with _lib.device_guard(torch, dev):
            _lib.check(fn(C.byref(a), torch.cuda.current_stream(dev).cuda_stream), what)

    def forward(self, obs, deterministic: bool = False):
        """SB3's forward in one launch of stg_policy_act_f32: (actions [N,2] in policy units, values [N,1], log_probs [N]).
        Row i is env `env_offset + i` for the noise. No autograd graph. Repacks the weights first."""
        obs = self._obs_rows(obs)
        n = obs.shape[0]
        w = self.pack_weights()
        actions = torch.empty(n, 2, dtype=torch.float32, device=obs.device)
        values = torch.empty(n, 1, dtype=torch.float32, device=obs.device)
        log_probs = torch.empty(n, dtype=torch.float32, device=obs.device)
        a = self._args(w, n)
        a.d_obs, a.d_action, a.d_value, a.d_log_prob = obs.data_ptr(), actions.data_ptr(), values.data_ptr(), log_probs.data_ptr()
        self._set_draw(a, deterministic)
        self._launch(_lib.load().stg_policy_act_f32, a, "stg_policy_act_f32")
        return actions, values, log_probs

    def _set_draw(self, a: _lib.StgPolicyArgs, deterministic: bool) -> None:
        if deterministic:
            a.flags = _lib.POLICY_DETERMINISTIC
        else:
            a.draw = self.noise_draws
            self.noise_draws += 1

    def predict_values(self, obs, mask=None, out=None):
        """V(obs) in one launch of stg_policy_value_f32: the critic only. `mask` (bool / uint8 [N] on the device): only rows
        where it is nonzero are computed and written; the other rows of `out` are left as they are (NaN in a new tensor).
        `out`: float32 contiguous tensor of N elements to write into; default a new [N,1]. Returns `out`. Repacks the weights."""
        obs = self._obs_rows(obs)
        n = obs.shape[0]
        if out is None:
            out = torch.empty(n, 1, dtype=torch.float32, device=obs.device) if mask is None \
                else torch.full((n, 1), math.nan, dtype=torch.float32, device=obs.device)
        elif out.dtype != torch.float32 or not out.is_contiguous() or out.numel() != n or out.device != obs.device:
            raise ValueError(f"out must be a contiguous float32 tensor of {n} elements on {obs.device}")
        a = self._args(self.pack_weights(), n)
        a.d_obs, a.d_value = obs.data_ptr(), out.data_ptr()
        if mask is not None:
            if mask.dtype not in (torch.bool, torch.uint8) or mask.numel() != n or mask.device != obs.device:
                raise ValueError(f"mask must be a bool or uint8 tensor of {n} elements on {obs.device}")
            mask = mask.contiguous()
            a.d_mask = mask.data_ptr()
        self._launch(_lib.load().stg_policy_value_f32, a, "stg_policy_value_f32")
        return out

    # ---- K10 -----------------------------------------------------------------------------------------------------------------
    def _grad_slots(self):
        """(parameter, offset of its gradient in the flat buffer): include/stg.h's STG_PPO_GRAD_* offsets."""
        L, pi, vf = _lib.POLICY_LAYOUT, self.mlp_extractor.policy_net, self.mlp_extractor.value_net
        return ((pi[0].weight, L["PI_W1"]), (pi[0].bias, L["PI_B1"]), (pi[2].weight, L["PI_W2"]), (pi[2].bias, L["PI_B2"]),
                (vf[0].weight, L["VF_W1"]), (vf[0].bias, L["VF_B1"]), (vf[2].weight, L["VF_W2"]), (vf[2].bias, L["VF_B2"]),
                (self.action_net.weight, L["ACT_W"]), (self.action_net.bias, L["ACT_B"]),
                (self.value_net.weight, L["VAL_W"]), (self.value_net.bias, L["VAL_B"]), (self.log_std, L["LOG_STD"]))

    def _ppo_planes(self, samples):
        obs = samples.observations
        n = obs.shape[0] if isinstance(obs, torch.Tensor) and obs.dim() == 2 else 0
        if n < 1:
            raise ValueError("ppo_backward needs samples.observations of shape [B, 12] with B >= 1, got "
                             f"{tuple(obs.shape) if isinstance(obs, torch.Tensor) else type(obs).__name__}")
        planes = [getattr(samples, name) for name, _, _ in _PPO_PLANES]
        for t, (name, tail, _) in zip(planes, _PPO_PLANES):
            if not isinstance(t, torch.Tensor) or t.dtype != torch.float32 or tuple(t.shape) != (n,) + tail:
                got = (t.dtype, tuple(t.shape)) if isinstance(t, torch.Tensor) else type(t).__name__
                raise ValueError(f"samples.{name} must be a float32 tensor of shape {(n,) + tail}, got {got}")
        if obs.device.type != "cuda":
            raise _lib.StgError("ActorCriticPolicy.ppo_backward needs CUDA tensors (no CPU fallback)")
        dev = self.log_std.device
        for i, (t, (name, _, align)) in enumerate(zip(planes, _PPO_PLANES)):
            if t.device != dev:
                raise ValueError(f"samples.{name} is on {t.device}, the policy on {dev}")
            if not t.is_contiguous() or t.data_ptr() % align:
                planes[i] = t.contiguous().clone()
        return n, planes

    def ppo_backward(self, samples, clip_range: float = 0.2, clip_range_vf: Optional[float] = None,
                     ent_coef: float = 0.0, vf_coef: float = 0.5, normalize_advantage: bool = True) -> PPOLosses:
        """SB3's PPO.train() loss of one minibatch with the current weights, and the gradient of every parameter: the result
        of `optimizer.zero_grad(); loss.backward()`, in one launch of stg_policy_ppo_grad_f32 and its fold (K10).

        `samples`: a RolloutBufferSamples as RolloutCollector.get() yields it (float32, B >= 1 rows, on the policy's device);
        misaligned or non-contiguous planes are copied first. With `normalize_advantage` and B > 1 the advantages are
        normalised as SB3 does, `(adv - adv.mean()) / (adv.std() + 1e-8)`, bit for bit (the mean and std by torch, the rest
        per row in the kernel). The weights are repacked first, so an optimiser step since the last call is seen.

        Every parameter's `.grad` is set to a view into one flat gradient buffer the policy owns, and that buffer is
        OVERWRITTEN on every call: gradients are not accumulated, and a `.grad` kept from an earlier call changes. The views
        are reassigned on every call, so `zero_grad(set_to_none=True)` between calls does no harm. Gradient clipping and the
        optimiser step are the caller's (`torch.nn.utils.clip_grad_norm_`, `torch.optim.Adam`). Returns PPOLosses; nothing
        is read back to the host, so early stopping on approx_kl costs the caller one synchronisation.
        Raises StgError without CUDA, ValueError for an empty batch or planes of the wrong shape, dtype or device."""
        n, planes = self._ppo_planes(samples)
        dev = self.log_std.device
        with _lib.device_guard(torch, dev):
            w = self.pack_weights()
            if self._grad is None or self._grad.device != dev:
                self._grad = torch.empty(_lib.POLICY_PARAMS, dtype=torch.float32, device=dev)
            stats = None
            if normalize_advantage and n > 1:
                adv = planes[4]
                stats = torch.stack([adv.mean(), adv.std()])
            losses = torch.empty(_lib.PPO_LOSSES, dtype=torch.float32, device=dev)
            work = torch.empty(_lib.ppo_work_doubles(n), dtype=torch.float64, device=dev)
            a = _lib.StgPpoArgs()
            a.d_weights = w.data_ptr()
            a.d_obs, a.d_action, a.d_old_value, a.d_old_log_prob, a.d_advantage, a.d_return = (t.data_ptr() for t in planes)
            a.d_adv_stats = None if stats is None else stats.data_ptr()
            a.d_grad, a.d_losses, a.d_work = self._grad.data_ptr(), losses.data_ptr(), work.data_ptr()
            cr = float(clip_range)
            a.clip_range, a.ratio_lo, a.ratio_hi = cr, 1.0 - cr, 1.0 + cr     # rounded to float32 as torch.clamp does
            if clip_range_vf is not None:
                a.flags = _lib.PPO_CLIP_VF
                a.clip_range_vf = float(clip_range_vf)
            a.ent_coef, a.vf_coef = float(ent_coef), float(vf_coef)
            a.batch = n
            self._launch(_lib.load().stg_policy_ppo_grad_f32, a, "stg_policy_ppo_grad_f32")
        for p, off in self._grad_slots():
            p.grad = self._grad[off:off + p.numel()].view_as(p)
        return PPOLosses(*losses.unbind())
