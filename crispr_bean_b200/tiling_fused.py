"""Device-resident SVI engine of the tiling sorting program (MultiMixtureNormal): host side of `bean_svi_tiling_run_*`.

One step = `svi.step` of bean/model/run.py:376-380 for bean/model/model.py:550-751 / :878-962 in three kernel launches
(per-edit draws, warp-per-guide kernel with a lane per allele, per-edit reduction + update; include/bean_b200.h), no torch
op and no host round trip per step.  Parameter names, shapes and initial values follow the pyro guide (model.py:893-937):
mu_loc = 0, mu_scale = 1, sd_loc = 0, sd_scale = 1 (E,), alpha_pi = alpha_prior (G, A) with epsilon at non-existent alleles.

Takes designs with at most 32 alleles per guide (one lane per allele: filtered allele tables; wider raw tables and
`--scale-by-acc` stay on `generic.TilingSviEngine`) -- see `supports()`.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

from . import _lib
from .device_pack import DeviceScreen, row_constants
from .halt import NonfiniteWatch
from .tiling import AlleleMap

_RUN = {torch.float32: "bean_svi_tiling_run_f32", torch.float64: "bean_svi_tiling_run_f64"}
MAX_ALLELES = 32


def supports(data, scale_by_accessibility: bool = False) -> bool:
    return (not scale_by_accessibility) and 2 <= int(data.n_max_alleles) <= MAX_ALLELES


class TilingFusedEngine(NonfiniteWatch):
    def __init__(self, data, device="cuda", dtype=torch.float32, use_bcmatch: bool = True, num_steps: int = 2000,
                 initial_lr: float = 0.01, gamma: float = 0.1, seed: int = 101, alpha_prior: float = 1.0, sd_scale: float = 0.01,
                 epsilon: float = 1e-5, prior_params: Optional[dict] = None, guide_offset: int = 0, group=None):
        if not torch.cuda.is_available():
            raise _lib.BeanError("TilingFusedEngine needs a CUDA device: there is no CPU fallback")
        if not supports(data):
            raise ValueError(f"the fused tiling step takes 2..{MAX_ALLELES} alleles per guide (got {data.n_max_alleles})")
        self.lib = _lib.lib()
        self.model, self.dtype, self.device = "MultiMixtureNormal", dtype, torch.device(device)
        # guides sharded over the ranks of `group` (dist.shard_data): `data` is this rank's guide block with ALL edits of the screen
        self.group, self.sharded = group, _dist_active(group)
        self.replicated_params = ("mu_loc", "mu_scale", "sd_loc", "sd_scale")  # per edit: identical on every rank
        self.num_steps = int(num_steps)
        use_bcmatch = bool(use_bcmatch) and getattr(data, "X_bcmatch_masked", None) is not None
        self.screen = DeviceScreen(data, self.device, dtype=dtype, use_bcmatch=use_bcmatch, mask_thres=10)
        G, R, A, E = data.n_guides, data.n_reps, int(data.n_max_alleles), int(data.n_edits)
        self.G, self.R, self.A, self.E = G, R, A, E
        dev, kw = self.device, dict(device=self.device, dtype=dtype)
        self.amap = AlleleMap(data.allele_ptr.numpy(), data.allele_edit.numpy(), G, A, E, dev)
        self.allele_mask = data.allele_mask.to(dev)
        self.allele_mask_u8 = self.allele_mask.to(torch.uint8).contiguous()
        self.pi_a0 = torch.as_tensor(data.pi_a0).to(device=dev, dtype=torch.float64).contiguous()
        ac = data.allele_counts_control  # (R, C, G, A)
        self.C = int(ac.shape[1])
        self.counts = ac.to(dev).to(dtype).contiguous()
        self.edit_params = torch.zeros((4, E), **kw)
        self.edit_m, self.edit_v, self.edit_grad = torch.zeros((4, E), **kw), torch.zeros((4, E), **kw), torch.zeros((4, E), **kw)
        a0 = torch.full((G, A), float(alpha_prior), **kw)
        a0[~self.allele_mask] = float(epsilon)
        self.alpha_u = a0.log()
        self.alpha_m, self.alpha_v, self.alpha_grad = torch.zeros((G, A), **kw), torch.zeros((G, A), **kw), torch.zeros((G, A), **kw)
        self.mu_e, self.sd_e = torch.zeros(E, **kw), torch.ones(E, **kw)
        self.d_slot = torch.zeros((2, G * (A - 1)), **kw)
        self.partial = torch.zeros(self.lib.bean_svi_tiling_num_partials(G, E), dtype=torch.float64, device=dev)
        self.counter = torch.zeros(1, dtype=torch.int32, device=dev)
        self.loss = torch.zeros(max(self.num_steps, 1) + 1, dtype=torch.float64, device=dev)
        self.step = 0
        # data-only parts of the ELBO: Dirichlet-Multinomial rows + the reporter Multinomial's coefficient (under repguide_mask)
        mconst, _ = row_constants(self.counts, with_xlogx=False)  # (R, C, G)
        ll_const = self.screen.ll_const + float((mconst * (self.screen.row_mask != 0).unsqueeze(1)).sum())

        c = _lib.BeanSviConfig()
        c.model, c.sd_is_sqrt, c.apply_update, c.fit_noise = _lib.MODEL_MIXTURE_NORMAL, 0, 1, 0
        c.mu_prior_normal, c.mu_prior_loc, c.mu_prior_scale = 0, 0.0, 1.0
        c.sd_prior_loc, c.sd_prior_scale = 0.0, float(sd_scale)
        self._prior_v = {}
        if prior_params:  # scalars or per-edit tensors, as for the variant programs (run.py:480-542)
            def put(key, field):
                val = prior_params[key]
                if torch.is_tensor(val) and val.numel() > 1:
                    if val.numel() != E:
                        raise ValueError(f"prior_params[{key!r}] has {val.numel()} entries for {E} edits")
                    self._prior_v[key] = val.detach().reshape(-1).to(**kw).contiguous()
                else:
                    setattr(c, field, float(val))

            if "mu_loc" in prior_params or "mu_scale" in prior_params:
                c.mu_prior_normal = 1
                for key in ("mu_loc", "mu_scale"):
                    if key in prior_params:
                        put(key, f"mu_prior_{key[3:]}")
            for key in ("sd_loc", "sd_scale"):
                if key in prior_params:
                    put(key, f"sd_prior_{key[3:]}")
        c.lr0, c.lrd = float(initial_lr), float(gamma) ** (1.0 / max(self.num_steps, 1))
        c.beta1, c.beta2, c.adam_eps, c.clip = 0.9, 0.999, 1e-8, 10.0
        c.ll_const, c.seed = ll_const, int(seed)
        c.guide_offset = int(guide_offset)
        # pi carries pi_a0's dtype in the reference (float64 out of the fit, float32 with the fallback coefficients): torch's
        # Multinomial clamps probabilities at that dtype's eps and its Dirichlet sampler at that dtype's smallest normal number
        pa0 = getattr(data, "pi_a0", None)
        ref_dtype = pa0.dtype if (torch.is_tensor(pa0) and pa0.is_floating_point()) else torch.float64
        if dtype == torch.float64:
            ref_dtype = torch.float64
        c.prob_clamp_eps = float(torch.finfo(ref_dtype).eps)
        self.cfg = c

        s = _lib.BeanTilingState()
        s.map = C_pointer(self.amap.c)
        s.n_controls, s.loss_capacity = self.C, self.loss.numel()
        s.allele_mask, s.pi_a0, s.counts = self.allele_mask_u8.data_ptr(), self.pi_a0.data_ptr(), self.counts.data_ptr()
        s.edit_params, s.edit_m, s.edit_v, s.edit_grad = (t.data_ptr() for t in (self.edit_params, self.edit_m, self.edit_v, self.edit_grad))
        s.alpha_u, s.alpha_m, s.alpha_v, s.alpha_grad = (t.data_ptr() for t in (self.alpha_u, self.alpha_m, self.alpha_v, self.alpha_grad))
        s.mu_e, s.sd_e, s.d_slot = self.mu_e.data_ptr(), self.sd_e.data_ptr(), self.d_slot.data_ptr()
        s.partial, s.counter, s.loss = self.partial.data_ptr(), self.counter.data_ptr(), self.loss.data_ptr()
        for key, field in (("mu_loc", "mu_prior_loc_v"), ("mu_scale", "mu_prior_scale_v"), ("sd_loc", "sd_prior_loc_v"),
                           ("sd_scale", "sd_prior_scale_v")):
            if key in self._prior_v:
                setattr(s, field, self._prior_v[key].data_ptr())
        s.epsilon, s.pi_tiny = float(epsilon), float(torch.finfo(ref_dtype).tiny)
        if self.sharded:
            import torch.distributed as dist

            self.edit_sum = torch.zeros((2, E), **kw)
            self.edit_iota = torch.arange(E + 1, dtype=torch.int32, device=dev)
            s.edit_sum, s.edit_iota = self.edit_sum.data_ptr(), self.edit_iota.data_ptr()
            s.edit_term_weight = 1.0 if dist.get_rank(group) == 0 else 0.0  # the per-edit ELBO terms count once
        s.nonfinite_step = self._init_nonfinite()
        self.state = s

    # ---------------------------------------------------------------------------------------------
    def _noise_struct(self, noise):
        if noise is None:
            return None, ()
        kw = dict(device=self.device, dtype=self.dtype)
        n, keep = _lib.BeanTilingNoise(), []
        if noise.get("record"):
            self.eps_used = torch.zeros((2, self.E), **kw)
            self.pi_used = torch.zeros((self.R, self.G, self.A), device=self.device, dtype=torch.float64)
            n.eps_out, n.pi_out = self.eps_used.data_ptr(), self.pi_used.data_ptr()
        if "eps_mu" in noise:
            em = noise["eps_mu"].reshape(-1).to(**kw).contiguous()
            es = noise["eps_sd"].reshape(-1).to(**kw).contiguous()
            assert em.numel() == self.E == es.numel()
            n.eps_mu, n.eps_sd = em.data_ptr(), es.data_ptr()
            keep += [em, es]
        if "pi" in noise:
            pi = noise["pi"]
            if pi.dim() == 4:  # reference layout (R, 1, G, A)
                pi = pi[:, 0]
            pi = pi.to(device=self.device, dtype=torch.float64).contiguous()
            assert tuple(pi.shape) == (self.R, self.G, self.A), tuple(pi.shape)
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
        run = getattr(self.lib, _RUN[self.dtype])
        if not self.sharded:
            _lib.check(run(self.screen.c, self.state, self.cfg, n, self.step, n_steps, stream), _RUN[self.dtype])
        else:
            # per step: this shard's guides -> per-edit gradient sums; one all-reduce of 2 E numbers (edits are shared between
            # guides of different shards); then every rank updates every edit from the same sums
            import torch.distributed as dist

            for t in range(self.step, self.step + n_steps):
                self.cfg.phases = 1
                _lib.check(run(self.screen.c, self.state, self.cfg, n, t, 1, stream), _RUN[self.dtype])
                dist.all_reduce(self.edit_sum, group=self.group)
                self.cfg.phases = 2
                _lib.check(run(self.screen.c, self.state, self.cfg, n, t, 1, stream), _RUN[self.dtype])
            self.cfg.phases = 0
        first = self.step
        if apply_update:
            self.step += n_steps
        self._keep = keep
        return self.loss[first:first + n_steps]

    def _snapshot_tensors(self):
        return [self.edit_params, self.edit_m, self.edit_v, self.alpha_u, self.alpha_m, self.alpha_v]

    def gradients(self, noise=None) -> Dict[str, torch.Tensor]:
        """Loss and its gradient w.r.t. the unconstrained parameters at the current point (no update)."""
        loss = self.run(1, noise=noise, apply_update=False)
        out = {"loss": loss[0].clone(), "alpha_pi": self.alpha_grad.clone()}
        for i, k in enumerate(("mu_loc", "mu_scale", "sd_loc", "sd_scale")):
            out[k] = self.edit_grad[i].clone()
        return out

    def params(self) -> Dict[str, torch.Tensor]:
        """Constrained parameter values under the reference's names and shapes."""
        ep = self.edit_params
        alpha = torch.where(self.allele_mask, self.alpha_u.exp(), torch.full_like(self.alpha_u, float(self.state.epsilon)))
        return {"mu_loc": ep[0].clone(), "mu_scale": ep[1].exp(), "sd_loc": ep[2].clone(), "sd_scale": ep[3].exp(), "alpha_pi": alpha}

    def losses(self):
        return self.loss[: self.step].cpu()


def _dist_active(group) -> bool:
    import torch.distributed as dist

    return dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1


def C_pointer(struct):
    import ctypes

    return ctypes.pointer(struct)
