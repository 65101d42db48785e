"""Device-resident SVI engine for the variant sorting models (host side of `bean_svi_run_*`).

Holds the unconstrained parameters and ClippedAdam moments as torch CUDA tensors (plumbing) and
advances them with the fused CUDA step; there is no per-step host synchronisation -- the loss of
every step lands in a device buffer that is read once (reference: `float(loss)` sync per step,
bean/model/run.py:377-380).
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import torch

from . import _lib
from .device_pack import DeviceScreen, row_constants
from .fused import FusedEngine, set_prior_pointers, svi_config

_RUN = {torch.float32: "bean_svi_run_f32", torch.float64: "bean_svi_run_f64"}
VAR_PARAM_NAMES = ("mu_loc", "mu_scale", "sd_loc", "sd_scale")  # rows of var_params; scales stored as log


class SviEngine(FusedEngine):
    """Parameters + optimiser state + the fused step for one (screen, model) pair on one GPU.

    model: "Normal" | "ControlNormal" | "MixtureNormal".  Parameter names, shapes and initial values
    follow the pyro guides (model.py:754-875; SURVEY App. A.5): mu_loc=0, mu_scale=1, sd_loc=0,
    sd_scale=1, alpha_pi=alpha_prior.
    """

    def __init__(self, data, model: str = "MixtureNormal", device="cuda", dtype=torch.float32,
                 use_bcmatch: bool = True, num_steps: int = 2000, initial_lr: float = 0.01, gamma: float = 0.1,
                 seed: int = 101, alpha_prior: float = 1.0, sd_scale: float = 0.01, mask_thres: int = 10,
                 prior_params: Optional[dict] = None, screen: Optional[DeviceScreen] = None,
                 guide_offset: int = 0, variant_offset: int = 0, scale_by_accessibility: bool = False,
                 fit_noise: bool = False):
        if model not in ("Normal", "ControlNormal", "MixtureNormal"):
            raise ValueError(f"SviEngine does not implement model {model!r}")
        self._setup(device, dtype, num_steps)
        self.model = model
        self.mixture = model == "MixtureNormal"
        use_bcmatch = bool(use_bcmatch) and getattr(data, "X_bcmatch_masked", None) is not None
        self.screen = screen or DeviceScreen(data, self.device, dtype=dtype, use_bcmatch=use_bcmatch, mask_thres=mask_thres)
        G, R = self.screen.n_guides, self.screen.n_reps
        dev, kw = self.device, dict(device=self.device, dtype=dtype)
        if model == "ControlNormal":  # one shared (mu, sd) for all guides (model.py:178-181)
            self.T = 1
            self.guide_variant = torch.zeros(G, dtype=torch.int32, device=dev)
            self.variant_ptr = torch.tensor([0, G], dtype=torch.int32, device=dev)
        else:
            self.T = int(data.n_targets)
            self.guide_variant = data.guide_variant.to(dev).contiguous()
            self.variant_ptr = data.variant_ptr.to(dev).contiguous()
        T = self.T
        self.var_params = torch.zeros((4, T), **kw)  # mu_loc = 0, log mu_scale = 0, sd_loc = 0, log sd_scale = 0
        self.var_m, self.var_v = torch.zeros((4, T), **kw), torch.zeros((4, T), **kw)
        self.var_grad = torch.zeros((4, T), **kw)
        self.d_guide = torch.zeros((2, G), **kw)
        ll_const = self.screen.ll_const
        if self.mixture:
            self.alpha_u = torch.full((G, 2), float(alpha_prior), **kw).log()
            self.alpha_m, self.alpha_v = torch.zeros((G, 2), **kw), torch.zeros((G, 2), **kw)
            self.alpha_grad = torch.zeros((G, 2), **kw)
            ac = data.allele_counts_control  # (R, C, G, 2); the model observes condition 0 of the control
            if ac.shape[1] != 1:
                raise NotImplementedError("more than one control condition")
            self.allele_counts = ac.to(dev, non_blocking=True)[:, 0].to(dtype).contiguous()  # (R, G, 2)
            self.pi_a0 = torch.as_tensor(data.pi_a0).to(**kw).contiguous()
            # data-only part of the Multinomial log-pmf, masked like the site (model.py:455, :470-474)
            mconst, _ = row_constants(self.allele_counts, with_xlogx=False)  # (R, G)
            ll_const += float((mconst * (self.screen.row_mask != 0)).sum())
        self.acc = bool(scale_by_accessibility) and self.mixture
        self.fit_noise = bool(fit_noise) and self.acc
        if self.acc:
            if getattr(data, "guide_accessibility", None) is None:
                raise ValueError("scale_by_accessibility needs data.guide_accessibility (accessibility_col)")
            # _scale_edited_pi: pi * exp(b) * accessibility^a with a = 0.2513, b = -1.9458 (utils.py:79-103)
            acc = torch.as_tensor(data.guide_accessibility).double()
            self.acc_k = (math.exp(-1.9458) * acc.pow(0.2513)).to(**kw).contiguous()
            self.noise_u = torch.stack([torch.zeros(G, dtype=torch.float64), torch.full((G,), 0.655, dtype=torch.float64).log()]).to(**kw).contiguous()
            self.noise_m, self.noise_v = torch.zeros((2, G), **kw), torch.zeros((2, G), **kw)
            self.noise_grad = torch.zeros((2, G), **kw)
        self.partial = torch.zeros((self.lib.bean_svi_num_partials(G, T),), dtype=torch.float64, device=dev)

        c, self._prior_v = svi_config(lr=initial_lr, gamma=gamma, num_steps=self.num_steps, seed=seed, ll_const=ll_const,
                                      guide_offset=guide_offset, variant_offset=variant_offset,
                                      sd_scale=1.0 if model == "ControlNormal" else float(sd_scale), prior_params=prior_params,
                                      n_variants=T, device=dev, dtype=dtype, pi_a0=getattr(data, "pi_a0", None))
        c.model = _lib.MODEL_MIXTURE_NORMAL if self.mixture else _lib.MODEL_NORMAL
        c.sd_is_sqrt = 1 if model == "Normal" else 0
        c.fit_noise = 1 if self.fit_noise else 0
        self.cfg = c

        s = _lib.BeanSviState()
        s.n_variants, s.loss_capacity = T, self.loss.numel()
        s.guide_variant, s.variant_ptr = self.guide_variant.data_ptr(), self.variant_ptr.data_ptr()
        if self.mixture:
            s.allele_counts, s.pi_a0 = self.allele_counts.data_ptr(), self.pi_a0.data_ptr()
            s.alpha_u, s.alpha_m, s.alpha_v = self.alpha_u.data_ptr(), self.alpha_m.data_ptr(), self.alpha_v.data_ptr()
            s.alpha_grad = self.alpha_grad.data_ptr()
        s.var_params, s.var_m, s.var_v = self.var_params.data_ptr(), self.var_m.data_ptr(), self.var_v.data_ptr()
        s.d_guide, s.var_grad = self.d_guide.data_ptr(), self.var_grad.data_ptr()
        s.partial, s.counter, s.loss = self.partial.data_ptr(), self.counter.data_ptr(), self.loss.data_ptr()
        if self.mixture:  # hand-over scratch of the two-kernel guide step (include/bean_b200.h: pw, dconc)
            self.pw = torch.empty((R, G, 4), **kw)
            self.dconc = torch.empty((G, 4), **kw)
            s.pw, s.dconc = self.pw.data_ptr(), self.dconc.data_ptr()
        set_prior_pointers(s, self._prior_v)
        if self.acc:
            s.acc_k = self.acc_k.data_ptr()
            s.noise_u, s.noise_m, s.noise_v = self.noise_u.data_ptr(), self.noise_m.data_ptr(), self.noise_v.data_ptr()
            s.noise_grad = self.noise_grad.data_ptr()
        s.nonfinite_step = self._init_nonfinite()
        self.state = s

    # ---------------------------------------------------------------------------------------------
    def _launch(self, first, n_steps, noise, apply_update):
        n, keep = None, []
        if noise is not None:
            n = _lib.BeanSviNoise()
            if noise.get("record"):  # have the kernels write out the Philox draws they used
                kw = dict(device=self.device, dtype=self.dtype)
                self.eps_used = torch.zeros((2, self.T), **kw)
                n.eps_out = self.eps_used.data_ptr()
                if self.mixture:
                    self.pi_used = torch.zeros((self.screen.n_guides, self.screen.n_reps, 2), **kw)
                    n.pi_out = self.pi_used.data_ptr()
            if "eps_mu" in noise:
                self._put(keep, n, "eps_mu", noise["eps_mu"].reshape(-1), (self.T,))
                self._put(keep, n, "eps_sd", noise["eps_sd"].reshape(-1), (self.T,))
            if self.acc and "eps_noise" in noise:
                self._put(keep, n, "eps_noise", noise["eps_noise"].reshape(-1), (self.screen.n_guides,))
            if self.mixture and "pi" in noise:
                pi = noise["pi"]
                if pi.dim() == 4:  # reference layout (R, 1, G, 2)
                    pi = pi[:, 0].permute(1, 0, 2)
                self._put(keep, n, "pi", pi, (self.screen.n_guides, self.screen.n_reps, 2))
        stream = torch.cuda.current_stream(self.device).cuda_stream
        rc = getattr(self.lib, _RUN[self.dtype])(self.screen.c, self.state, self.cfg, n, first, n_steps, stream)
        _lib.check(rc, _RUN[self.dtype])
        return keep

    def _snapshot_tensors(self):
        out = [self.var_params, self.var_m, self.var_v]
        if self.mixture:
            out += [self.alpha_u, self.alpha_m, self.alpha_v]
        if self.acc:
            out += [self.noise_u, self.noise_m, self.noise_v]
        return out

    def _grads(self):
        out = dict(zip(VAR_PARAM_NAMES, self.var_grad))
        if self.mixture:
            out["alpha_pi"] = self.alpha_grad
        if self.fit_noise:
            out["noise_loc"], out["noise_scale"] = self.noise_grad[0], self.noise_grad[1]
        return out

    def params(self) -> Dict[str, torch.Tensor]:
        """Constrained parameter values under the reference's names and shapes (pyro param store)."""
        T = self.T
        shape = () if self.model == "ControlNormal" else (T, 1)
        vp = self.var_params
        out = {"mu_loc": vp[0].reshape(shape).clone(), "mu_scale": vp[1].exp().reshape(shape),
               "sd_loc": vp[2].reshape(shape).clone(), "sd_scale": vp[3].exp().reshape(shape)}
        if self.mixture:
            out["alpha_pi"] = self.alpha_u.exp()
        if self.fit_noise:
            out["noise_loc"], out["noise_scale"] = self.noise_u[0].clone(), self.noise_u[1].exp()
        return out
