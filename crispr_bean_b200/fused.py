"""What the three fused SVI engines share: `svi.SviEngine` (sorting), `survival_fused.SurvivalFusedEngine` and
`tiling_fused.TilingFusedEngine`.

`svi_config` builds the `BeanSviConfig` all three pass to their C entry point (it needs no GPU), and `FusedEngine` holds the loss
buffer and the run / gradient loop around that entry point.  Each engine adds its own buffers, C state and `_launch`.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

from . import _lib
from .halt import NonfiniteWatch

PRIOR_FIELDS = (("mu_loc", "mu_prior_loc_v"), ("mu_scale", "mu_prior_scale_v"), ("sd_loc", "sd_prior_loc_v"),
                ("sd_scale", "sd_prior_scale_v"))


def pi_dtype(dtype, pi_a0, control_timepoint=None, promote: bool = False) -> torch.dtype:
    """The dtype `pi` has in the reference, at whose eps torch's Multinomial clamps probabilities.

    promote=False (sorting, tiling): pi carries pi_a0's dtype -- float64 out of the fit, float32 with the fallback
    coefficients -- and is float64 when the engine computes in float64 or pi_a0 is not a floating tensor.
    promote=True (survival): the reference evaluates pi exp(mu t_c) in the promoted dtype of (dtype, pi_a0,
    control_timepoint), over those that are tensors."""
    if promote:
        for t in (pi_a0, control_timepoint):
            if torch.is_tensor(t):
                dtype = torch.promote_types(dtype, t.dtype)
        return dtype
    if dtype == torch.float64 or not (torch.is_tensor(pi_a0) and pi_a0.is_floating_point()):
        return torch.float64
    return pi_a0.dtype


def svi_config(*, lr: float, gamma: float, num_steps: int, seed: int, ll_const: float, guide_offset: int = 0,
               variant_offset: int = 0, sd_scale: float = 1.0, sd_priors: bool = True, prior_params: Optional[dict] = None,
               n_variants: int = 0, unit: str = "variants", device="cpu", dtype=torch.float32, pi_a0=None,
               control_timepoint=None, promote: bool = False):
    """The BeanSviConfig of a fused engine and the per-variant prior tensors {key: (n_variants,) tensor}.

    Priors: Laplace(0, 1) on mu and LogNormal(0, sd_scale) on sd unless `prior_params` (`bean run --prior-params`, run.py:480-542)
    gives scalars or per-variant tensors (n_variants,) / (n_variants, 1); a mu key makes the mu prior Normal.  With
    sd_priors=False (survival: no sd site) the sd keys are ignored.  ClippedAdam: lr_t = lr * gamma^(t / num_steps)
    (run.py:367).  The Multinomial clamp is the eps of `pi_dtype(dtype, pi_a0, control_timepoint, promote)`.  The caller sets
    model, sd_is_sqrt and fit_noise."""
    c = _lib.BeanSviConfig()
    c.model, c.apply_update = _lib.MODEL_MIXTURE_NORMAL, 1
    c.mu_prior_normal, c.mu_prior_loc, c.mu_prior_scale = 0, 0.0, 1.0
    c.sd_prior_loc, c.sd_prior_scale = 0.0, float(sd_scale)
    prior_v = {}
    if prior_params:
        def put(key):
            val = prior_params[key]
            if torch.is_tensor(val) and val.numel() > 1:
                if val.numel() != n_variants:
                    raise ValueError(f"prior_params[{key!r}] has {val.numel()} entries for {n_variants} {unit}")
                prior_v[key] = val.detach().reshape(-1).to(device=device, dtype=dtype).contiguous()
            else:
                setattr(c, f"{key[:2]}_prior_{key[3:]}", float(val))

        if "mu_loc" in prior_params or "mu_scale" in prior_params:
            c.mu_prior_normal = 1
        for key in ("mu_loc", "mu_scale") + (("sd_loc", "sd_scale") if sd_priors else ()):
            if key in prior_params:
                put(key)
    c.lr0, c.lrd = float(lr), float(gamma) ** (1.0 / max(int(num_steps), 1))
    c.beta1, c.beta2, c.adam_eps, c.clip = 0.9, 0.999, 1e-8, 10.0
    c.ll_const, c.seed = ll_const, int(seed)
    c.prob_clamp_eps = float(torch.finfo(pi_dtype(dtype, pi_a0, control_timepoint, promote)).eps)
    c.guide_offset, c.variant_offset = int(guide_offset), int(variant_offset)
    return c, prior_v


def set_prior_pointers(state, prior_v: Dict[str, torch.Tensor]) -> None:
    """The `*_prior_v` fields of a C state struct from `svi_config`'s per-variant tensors (the others stay NULL)."""
    for key, field in PRIOR_FIELDS:
        if key in prior_v:
            setattr(state, field, prior_v[key].data_ptr())


def dist_active(group) -> bool:
    import torch.distributed as dist

    return dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1


class FusedEngine(NonfiniteWatch):
    """Base of the fused engines.  `_setup` allocates the loss buffer; a subclass sets `cfg` and its C state, and implements
    `_launch(first, n_steps, noise, apply_update)` -> the injected buffers to keep alive, and `_grads()` -> {name: gradient}."""

    def _setup(self, device, dtype, num_steps: int):
        self.lib = _lib.lib()
        self.device, self.dtype = torch.device(device), dtype
        self.num_steps = int(num_steps)
        self.counter = torch.zeros((1,), dtype=torch.int32, device=self.device)
        # one spare slot: `gradients()` evaluates a step without updating and writes its loss at index `step`, which is
        # num_steps after a complete run
        self.loss = torch.zeros((max(self.num_steps, 1) + 1,), dtype=torch.float64, device=self.device)
        self.step = 0

    def _put(self, keep: list, struct, field: str, tensor: torch.Tensor, shape: tuple, dtype=None):
        """Injected noise: `tensor` on the device in the engine's dtype (or `dtype`), checked against `shape`, into `field`."""
        t = tensor.to(device=self.device, dtype=dtype or self.dtype).contiguous()
        assert tuple(t.shape) == shape, (field, tuple(t.shape), shape)
        setattr(struct, field, t.data_ptr())
        keep.append(t)

    def run(self, n_steps: int, noise: Optional[Dict[str, torch.Tensor]] = None, apply_update: bool = True):
        """Advance `n_steps` SVI steps (asynchronously); injected `noise` applies to every one of them."""
        if self.step + n_steps > self.loss.numel() - (1 if apply_update else 0):
            raise ValueError("loss buffer exhausted: construct the engine with a larger num_steps")
        first = self.step
        self.cfg.apply_update = 1 if apply_update else 0
        self._keep = self._launch(first, n_steps, noise, apply_update)  # alive until the stream has consumed them
        if apply_update:
            self.step += n_steps
        return self.loss[first:first + n_steps]

    def gradients(self, noise=None) -> Dict[str, torch.Tensor]:
        """Loss and its gradient w.r.t. the unconstrained parameters at the current point (no update)."""
        loss = self.run(1, noise=noise, apply_update=False)
        out = {"loss": loss[0].clone()}
        out.update({k: g.clone() for k, g in self._grads().items()})
        return out

    def losses(self):
        return self.loss[: self.step].cpu()
