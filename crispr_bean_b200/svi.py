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
from .halt import NonfiniteWatch

_RUN = {torch.float32: "bean_svi_run_f32", torch.float64: "bean_svi_run_f64"}
VAR_PARAM_NAMES = ("mu_loc", "mu_scale", "sd_loc", "sd_scale")  # rows of var_params; scales stored as log


class SviEngine(NonfiniteWatch):
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
                 fit_noise: bool = False, split: bool = True):
        if model not in ("Normal", "ControlNormal", "MixtureNormal"):
            raise ValueError(f"SviEngine does not implement model {model!r}")
        self.lib = _lib.lib()
        self.model, self.dtype, self.device = model, dtype, torch.device(device)
        self.num_steps = int(num_steps)
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
        self.counter = torch.zeros((1,), dtype=torch.int32, device=dev)
        # one spare slot: `gradients()` evaluates a step without updating and writes its loss at index `step`, which is
        # num_steps after a complete run
        self.loss = torch.zeros((max(self.num_steps, 1) + 1,), dtype=torch.float64, device=dev)
        self.step = 0

        c = _lib.BeanSviConfig()
        c.model = _lib.MODEL_MIXTURE_NORMAL if self.mixture else _lib.MODEL_NORMAL
        c.sd_is_sqrt = 1 if model == "Normal" else 0
        c.apply_update = 1
        c.fit_noise = 1 if self.fit_noise else 0
        c.mu_prior_normal, c.mu_prior_loc, c.mu_prior_scale = 0, 0.0, 1.0
        c.sd_prior_loc, c.sd_prior_scale = 0.0, (1.0 if model == "ControlNormal" else float(sd_scale))
        self._prior_v = {}
        if prior_params:
            # scalars or per-variant tensors (T,) / (T, 1), as `bean build-prior` writes them (run.py:480-542)
            def put(key, field):
                val = prior_params[key]
                if torch.is_tensor(val) and val.numel() > 1:
                    if val.numel() != T:
                        raise ValueError(f"prior_params[{key!r}] has {val.numel()} entries for {T} variants")
                    self._prior_v[key] = val.detach().reshape(-1).to(**kw).contiguous()
                else:
                    setattr(c, field, float(val))

            if "mu_loc" in prior_params or "mu_scale" in prior_params:
                c.mu_prior_normal = 1
                c.mu_prior_loc, c.mu_prior_scale = 0.0, 1.0
                for key in ("mu_loc", "mu_scale"):
                    if key in prior_params:
                        put(key, f"mu_prior_{key[3:]}")
            for key in ("sd_loc", "sd_scale"):
                if key in prior_params:
                    put(key, f"sd_prior_{key[3:]}")
        c.lr0, c.lrd = float(initial_lr), float(gamma) ** (1.0 / max(self.num_steps, 1))
        c.beta1, c.beta2, c.adam_eps, c.clip = 0.9, 0.999, 1e-8, 10.0
        c.ll_const, c.seed = ll_const, int(seed)
        # Multinomial prob clamp: eps of the dtype pi has in the reference = dtype of pi_a0 (float64 out of the fit)
        pa0 = getattr(data, "pi_a0", None)
        ref_dtype = torch.float64 if (dtype == torch.float64 or pa0 is None or not torch.is_tensor(pa0)) else pa0.dtype
        c.prob_clamp_eps = float(torch.finfo(ref_dtype).eps)
        c.guide_offset, c.variant_offset = int(guide_offset), int(variant_offset)
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
        self.split = bool(split) and self.mixture
        if self.split:  # scratch of the two-kernel guide step (include/bean_b200.h: pw, dconc)
            self.pw = torch.empty((R, G, 4), **kw)
            self.dconc = torch.empty((G, 4), **kw)
            s.pw, s.dconc = self.pw.data_ptr(), self.dconc.data_ptr()
        for key, field in (("mu_loc", "mu_prior_loc_v"), ("mu_scale", "mu_prior_scale_v"), ("sd_loc", "sd_prior_loc_v"),
                           ("sd_scale", "sd_prior_scale_v")):
            if key in self._prior_v:
                setattr(s, field, self._prior_v[key].data_ptr())
        if self.acc:
            s.acc_k = self.acc_k.data_ptr()
            s.noise_u, s.noise_m, s.noise_v = self.noise_u.data_ptr(), self.noise_m.data_ptr(), self.noise_v.data_ptr()
            s.noise_grad = self.noise_grad.data_ptr()
        s.nonfinite_step = self._init_nonfinite()
        self.state = s

    # ---------------------------------------------------------------------------------------------
    def _noise_struct(self, noise: Optional[Dict[str, torch.Tensor]]):
        if noise is None:
            return None, ()
        kw = dict(device=self.device, dtype=self.dtype)
        n, keep = _lib.BeanSviNoise(), []
        if noise.get("record"):  # have the kernels write out the Philox draws they used
            self.eps_used = torch.zeros((2, self.T), **kw)
            n.eps_out = self.eps_used.data_ptr()
            if self.mixture:
                self.pi_used = torch.zeros((self.screen.n_guides, self.screen.n_reps, 2), **kw)
                n.pi_out = self.pi_used.data_ptr()
        if "eps_mu" in noise:
            em = noise["eps_mu"].reshape(-1).to(**kw).contiguous()
            es = noise["eps_sd"].reshape(-1).to(**kw).contiguous()
            assert em.numel() == self.T == es.numel()
            n.eps_mu, n.eps_sd = em.data_ptr(), es.data_ptr()
            keep += [em, es]
        if self.acc and "eps_noise" in noise:
            en = noise["eps_noise"].reshape(-1).to(**kw).contiguous()
            assert en.numel() == self.screen.n_guides
            n.eps_noise = en.data_ptr()
            keep.append(en)
        if self.mixture and "pi" in noise:
            pi = noise["pi"]
            if pi.dim() == 4:  # reference layout (R, 1, G, 2)
                pi = pi[:, 0].permute(1, 0, 2)
            pi = pi.to(**kw).contiguous()
            assert pi.shape == (self.screen.n_guides, self.screen.n_reps, 2)
            n.pi = pi.data_ptr()
            keep.append(pi)
        return n, keep

    def run(self, n_steps: int, noise: Optional[Dict[str, torch.Tensor]] = None, apply_update: bool = True):
        """Advance `n_steps` SVI steps (asynchronously); injected `noise` applies to every one of them."""
        if self.step + n_steps > self.loss.numel() - (1 if apply_update else 0):
            raise ValueError("loss buffer exhausted: construct the engine with a larger num_steps")
        n, keep = self._noise_struct(noise)
        self.cfg.apply_update = 1 if apply_update else 0
        stream = torch.cuda.current_stream(self.device).cuda_stream
        rc = getattr(self.lib, _RUN[self.dtype])(self.screen.c, self.state, self.cfg, n, self.step, n_steps, stream)
        _lib.check(rc, _RUN[self.dtype])
        first = self.step
        if apply_update:
            self.step += n_steps
        self._keep = keep  # keep injected buffers alive until the stream has consumed them
        return self.loss[first:first + n_steps]

    def _snapshot_tensors(self):
        out = [self.var_params, self.var_m, self.var_v]
        if self.mixture:
            out += [self.alpha_u, self.alpha_m, self.alpha_v]
        if self.acc:
            out += [self.noise_u, self.noise_m, self.noise_v]
        return out

    def gradients(self, noise=None) -> Dict[str, torch.Tensor]:
        """Loss and its gradient w.r.t. the unconstrained parameters at the current point (no update)."""
        loss = self.run(1, noise=noise, apply_update=False)
        out = {"loss": loss[0].clone()}
        for i, k in enumerate(VAR_PARAM_NAMES):
            out[k] = self.var_grad[i].clone()
        if self.mixture:
            out["alpha_pi"] = self.alpha_grad.clone()
        if self.fit_noise:
            out["noise_loc"], out["noise_scale"] = self.noise_grad[0].clone(), self.noise_grad[1].clone()
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

    def losses(self):
        return self.loss[: self.step].cpu()
