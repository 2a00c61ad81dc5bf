"""`ClippedAdam`: Stable-Baselines3's PPO optimiser step for the ActorCriticPolicy, clip_grad_norm_ + torch.optim.Adam, in one
launch of stg_policy_adam_f32 (K11, include/stg.h)."""
from __future__ import annotations

from typing import Optional

import torch

from . import _lib
from .policy import ActorCriticPolicy, PPOLosses

_STATE_KEYS = ("step", "exp_avg", "exp_avg_sq")
# torch.optim.Adam's settings that change its result and that K11 does not implement, with the only value K11 accepts
_FIXED = {"weight_decay": 0, "amsgrad": False, "maximize": False, "decoupled_weight_decay": False}


def _check_group(group) -> None:
    """ValueError for a parameter group K11 would not step as torch.optim.Adam does."""
    for key, want in _FIXED.items():
        if group.get(key, want) != want:
            raise ValueError(f"ClippedAdam implements Adam with {key}={want!r} only, got {group[key]!r}")
    if not 0.0 <= float(group["betas"][0]) < 1.0 or not 0.0 <= float(group["betas"][1]) < 1.0:
        raise ValueError(f"ClippedAdam needs betas in [0, 1), got {group['betas']!r}")


class ClippedAdam(torch.optim.Optimizer):
    """`ClippedAdam(policy, lr=3e-4, betas=(0.9, 0.999), eps=1e-5, max_grad_norm=0.5)`: `clip_grad_norm_(policy.parameters(),
    max_grad_norm)` followed by `torch.optim.Adam(policy.parameters(), lr, betas, eps).step()` (single-tensor update, no weight
    decay), as one kernel launch over an ActorCriticPolicy. The defaults are SB3's PPO optimiser and its `max_grad_norm`;
    `max_grad_norm=None` does not clip. The order of operations and the roundings are include/stg.h's K11 contract.

    `step()` reads `param_groups[0]["lr"]` on every call, so SB3-style schedules that set `param_group["lr"]` work. When every
    `.grad` is the view `policy.ppo_backward` set, the kernel reads the policy's flat gradient buffer; otherwise the `.grad`
    tensors (eager autograd through `evaluate_actions`, say) are gathered into a staging buffer with one torch.cat and, when
    clipping, the clipped values are copied back, so `.grad` ends as clip_grad_norm_ leaves it. A parameter without `.grad`
    raises ValueError. `step()` never synchronises with the host.

    The moments live in flat device buffers in the K10 layout and the step count in one device float32 shared by every
    parameter. `state_dict()` / `load_state_dict()` use torch.optim.Adam's format (parameters indexed in `policy.parameters()`
    order, `step` a float32 CPU scalar tensor per parameter, Adam's param-group keys plus `max_grad_norm`), so a state dict
    saved from `torch.optim.Adam(policy.parameters())` loads here and the reverse; per-parameter steps that differ raise
    ValueError. Adam's settings K11 does not implement (weight_decay, amsgrad, maximize, decoupled_weight_decay) raise
    ValueError when a state dict sets them or when step() finds them changed in the parameter group."""

    def __init__(self, policy: ActorCriticPolicy, lr: float = 3e-4, betas=(0.9, 0.999), eps: float = 1e-5,
                 max_grad_norm: Optional[float] = 0.5):
        if not isinstance(policy, ActorCriticPolicy):
            raise ValueError(f"ClippedAdam needs an ActorCriticPolicy, got {type(policy).__name__}")
        params = list(policy.parameters())
        dev = policy.log_std.device
        for p in params:
            if p.dtype != torch.float32 or not p.is_contiguous() or p.device != dev:
                raise ValueError("ClippedAdam needs contiguous float32 parameters on the policy's device")
        defaults = dict(lr=lr, betas=tuple(betas), eps=eps, weight_decay=0, amsgrad=False, maximize=False, foreach=None,
                        capturable=False, differentiable=False, fused=None, decoupled_weight_decay=False,
                        max_grad_norm=max_grad_norm)
        self.policy = policy
        self._ready = False
        super().__init__(params, defaults)
        self._ready = True
        self._slots = policy._grad_slots()
        self._exp_avg = torch.zeros(_lib.POLICY_PARAMS, dtype=torch.float32, device=dev)
        self._exp_avg_sq = torch.zeros(_lib.POLICY_PARAMS, dtype=torch.float32, device=dev)
        self._step_count = torch.zeros(1, dtype=torch.float32, device=dev)
        self._stage = None

    def add_param_group(self, param_group):
        if getattr(self, "_ready", True):
            raise ValueError("ClippedAdam owns exactly its policy's parameters; it takes no other parameter group")
        super().add_param_group(param_group)

    # ---- the step ------------------------------------------------------------------------------------------------------------
    def _check_params(self):
        group = self.param_groups[0]
        want = list(self.policy.parameters())
        if len(self.param_groups) != 1 or len(group["params"]) != len(want) or \
                any(p is not q for p, q in zip(group["params"], want)):
            raise ValueError("ClippedAdam's parameters are no longer its policy's parameters")
        dev = self.policy.log_std.device
        for p, _ in self._slots:
            if p.dtype != torch.float32 or not p.is_contiguous() or p.device != dev:
                raise ValueError("ClippedAdam needs contiguous float32 parameters on the policy's device")
            if p.grad is None:
                raise ValueError("every parameter needs a .grad before ClippedAdam.step() (ppo_backward or backward())")

    def _grad_buffer(self):
        """The flat gradient in the K10 layout: the policy's own buffer when every .grad is its view, else the staging buffer
        filled from the .grad tensors with one torch.cat (then `True` as second value)."""
        flat = self.policy._grad
        if flat is not None and all(p.grad.data_ptr() == flat.data_ptr() + 4 * off and p.grad.is_contiguous()
                                    and p.grad.shape == p.shape for p, off in self._slots):
            return flat, False
        for p, _ in self._slots:
            if p.grad.shape != p.shape or p.grad.dtype != torch.float32 or p.grad.device != p.device:
                raise ValueError("every .grad must be a float32 tensor of its parameter's shape and device")
        if self._stage is None:
            self._stage = torch.empty(_lib.POLICY_PARAMS, dtype=torch.float32, device=self._exp_avg.device)
        torch.cat([p.grad.reshape(-1) for p, _ in self._slots], out=self._stage)
        return self._stage, True

    @torch.no_grad()
    def step(self, closure=None):
        """One clip_grad_norm_ + Adam step: one launch of stg_policy_adam_f32."""
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        self._step()
        return loss

    def _step(self, losses: Optional[PPOLosses] = None, gate: Optional[torch.Tensor] = None,
              log: Optional[torch.Tensor] = None, target_kl: Optional[float] = None) -> None:
        """The launch behind step(), with PPO.train()'s extras: `losses` (ppo_backward's PPOLosses of this minibatch), `gate`
        (int32 [1] device tensor: 1 open, 0 closed) and `log` (float64 [STG_ADAM_LOG] device tensor) as include/stg.h
        describes; with `target_kl` the kernel closes the gate instead of stepping when approx_kl > 1.5 * target_kl."""
        self._check_params()
        _check_group(self.param_groups[0])
        if self._exp_avg.device.type != "cuda":
            raise _lib.StgError("ClippedAdam.step needs the policy on a CUDA device (no CPU fallback)")
        grad, staged = self._grad_buffer()
        group = self.param_groups[0]
        a = _lib.StgAdamArgs()
        for s, (p, _) in enumerate(self._slots):
            a.d_param[s] = p.data_ptr()
        a.d_grad, a.d_exp_avg, a.d_exp_avg_sq = grad.data_ptr(), self._exp_avg.data_ptr(), self._exp_avg_sq.data_ptr()
        a.d_step = self._step_count.data_ptr()
        keep = None
        if losses is not None:
            keep = losses_tensor(losses)
            a.d_losses = keep.data_ptr()
        a.d_gate = None if gate is None else gate.data_ptr()
        a.d_log = None if log is None else log.data_ptr()
        a.lr = float(group["lr"])
        a.beta1, a.beta2 = (float(b) for b in group["betas"])
        a.eps = float(group["eps"])
        if group["max_grad_norm"] is not None:
            a.flags |= _lib.ADAM_CLIP
            a.max_grad_norm = float(group["max_grad_norm"])
        if target_kl is not None:
            a.flags |= _lib.ADAM_TARGET_KL
            a.target_kl = float(target_kl)
        self.policy._launch(_lib.load().stg_policy_adam_f32, a, "stg_policy_adam_f32")
        if staged and group["max_grad_norm"] is not None:
            for p, off in self._slots:
                p.grad.copy_(grad[off:off + p.numel()].view_as(p))
        del keep

    # ---- torch.optim.Adam's state dict -----------------------------------------------------------------------------------------
    def _offsets(self):
        """(parameter, its offset in the flat buffers) in policy.parameters() order."""
        off = {id(p): o for p, o in self._slots}
        return [(p, off[id(p)]) for p in self.param_groups[0]["params"]]

    def state_dict(self):
        group = {k: v for k, v in self.param_groups[0].items() if k != "params"}
        params = self._offsets()
        group["params"] = list(range(len(params)))
        step = self._step_count.detach().to("cpu").reshape(())
        state = {}
        if float(step) > 0:
            for i, (p, o) in enumerate(params):
                state[i] = {"step": step.clone(), "exp_avg": self._exp_avg[o:o + p.numel()].view_as(p).clone(),
                            "exp_avg_sq": self._exp_avg_sq[o:o + p.numel()].view_as(p).clone()}
        return {"state": state, "param_groups": [group]}

    def load_state_dict(self, state_dict):
        groups = state_dict["param_groups"]
        params = self._offsets()
        if len(groups) != 1 or len(groups[0]["params"]) != len(params):
            raise ValueError(f"ClippedAdam has one parameter group of {len(params)} parameters")
        _check_group(groups[0])
        state = state_dict["state"]
        steps = set()
        for i in range(len(params)):
            st = state.get(groups[0]["params"][i])
            if st is None:
                steps.add(0.0)
                continue
            if any(k not in st for k in _STATE_KEYS) or set(st) - set(_STATE_KEYS):
                raise ValueError(f"the state of parameter {i} needs exactly {_STATE_KEYS} (no amsgrad)")
            steps.add(float(st["step"]))
        if len(steps) > 1:
            raise ValueError(f"ClippedAdam keeps one step count for all parameters; the state dict has {sorted(steps)}")
        with torch.no_grad():
            for i, (p, o) in enumerate(params):
                st = state.get(groups[0]["params"][i])
                for buf, key in ((self._exp_avg, "exp_avg"), (self._exp_avg_sq, "exp_avg_sq")):
                    dst = buf[o:o + p.numel()]
                    if st is None:
                        dst.zero_()
                    else:
                        src = torch.as_tensor(st[key])
                        if src.numel() != p.numel():
                            raise ValueError(f"{key} of parameter {i} has {src.numel()} elements, the parameter {p.numel()}")
                        dst.copy_(src.reshape(-1))
            self._step_count.fill_(steps.pop())
        new = {k: v for k, v in groups[0].items() if k != "params"}
        new.setdefault("max_grad_norm", self.param_groups[0]["max_grad_norm"])
        self.param_groups[0].update(new)
        if isinstance(self.param_groups[0]["betas"], list):
            self.param_groups[0]["betas"] = tuple(self.param_groups[0]["betas"])


def losses_tensor(losses) -> torch.Tensor:
    """The [STG_PPO_LOSSES] float32 device tensor behind ppo_backward's PPOLosses (its fields are consecutive views of it),
    or a stacked copy when they are not."""
    if isinstance(losses, torch.Tensor):
        t = losses
    elif len(losses) != _lib.PPO_LOSSES:
        raise ValueError(f"losses must be ppo_backward's PPOLosses or a float32 tensor of {_lib.PPO_LOSSES} elements")
    elif all(x.dtype == torch.float32 and x.device == losses[0].device and x.data_ptr() == losses[0].data_ptr() + 4 * i
             for i, x in enumerate(losses)):
        t = losses[0].as_strided((_lib.PPO_LOSSES,), (1,))
    else:
        t = torch.stack([x.reshape(()) for x in losses]).to(torch.float32)
    if t.dtype != torch.float32 or t.numel() != _lib.PPO_LOSSES or not t.is_contiguous():
        raise ValueError(f"losses must be ppo_backward's PPOLosses or a float32 tensor of {_lib.PPO_LOSSES} elements")
    return t
