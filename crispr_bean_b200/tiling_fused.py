"""Device-resident SVI engine of the tiling sorting program (MultiMixtureNormal): host side of `bean_svi_tiling_run_*`.

One step = `svi.step` of bean/model/run.py:376-380 for bean/model/model.py:550-751 / :878-962 in three kernel launches
(per-edit draws, warp-per-guide kernel with a lane per allele, per-edit reduction + update; include/bean_b200.h), no torch
op and no host round trip per step.  Parameter names, shapes and initial values follow the pyro guide (model.py:893-937):
mu_loc = 0, mu_scale = 1, sd_loc = 0, sd_scale = 1 (E,), alpha_pi = alpha_prior (G, A) with epsilon at non-existent alleles.

Takes designs with at most 32 alleles per guide (one lane per allele: filtered allele tables; wider raw tables and
`--scale-by-acc` stay on `generic.TilingSviEngine`) -- see `supports()`.
"""
from __future__ import annotations

import ctypes
from typing import Dict, Optional

import torch

from . import _lib
from .device_pack import DeviceScreen, row_constants
from .fused import FusedEngine, dist_active, pi_dtype, set_prior_pointers, svi_config
from .tiling import AlleleMap

_RUN = {torch.float32: "bean_svi_tiling_run_f32", torch.float64: "bean_svi_tiling_run_f64"}
MAX_ALLELES = 32


def supports(data, scale_by_accessibility: bool = False) -> bool:
    return (not scale_by_accessibility) and 2 <= int(data.n_max_alleles) <= MAX_ALLELES


class TilingFusedEngine(FusedEngine):
    def __init__(self, data, device="cuda", dtype=torch.float32, use_bcmatch: bool = True, num_steps: int = 2000,
                 initial_lr: float = 0.01, gamma: float = 0.1, seed: int = 101, alpha_prior: float = 1.0, sd_scale: float = 0.01,
                 epsilon: float = 1e-5, prior_params: Optional[dict] = None, guide_offset: int = 0, group=None):
        if not torch.cuda.is_available():
            raise _lib.BeanError("TilingFusedEngine needs a CUDA device: there is no CPU fallback")
        if not supports(data):
            raise ValueError(f"the fused tiling step takes 2..{MAX_ALLELES} alleles per guide (got {data.n_max_alleles})")
        self._setup(device, dtype, num_steps)
        self.model = "MultiMixtureNormal"
        # guides sharded over the ranks of `group` (dist.shard_data): `data` is this rank's guide block with ALL edits of the screen
        self.group, self.sharded = group, dist_active(group)
        self.replicated_params = ("mu_loc", "mu_scale", "sd_loc", "sd_scale")  # per edit: identical on every rank
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
        # data-only parts of the ELBO: Dirichlet-Multinomial rows + the reporter Multinomial's coefficient (under repguide_mask)
        mconst, _ = row_constants(self.counts, with_xlogx=False)  # (R, C, G)
        ll_const = self.screen.ll_const + float((mconst * (self.screen.row_mask != 0).unsqueeze(1)).sum())

        # pi carries pi_a0's dtype in the reference (float64 out of the fit, float32 with the fallback coefficients): torch's
        # Multinomial clamps probabilities at that dtype's eps and its Dirichlet sampler at that dtype's smallest normal number
        pa0 = getattr(data, "pi_a0", None)
        c, self._prior_v = svi_config(lr=initial_lr, gamma=gamma, num_steps=self.num_steps, seed=seed, ll_const=ll_const,
                                      guide_offset=guide_offset, sd_scale=float(sd_scale), prior_params=prior_params,
                                      n_variants=E, unit="edits", device=dev, dtype=dtype, pi_a0=pa0)
        c.sd_is_sqrt, c.fit_noise = 0, 0
        self.cfg = c

        s = _lib.BeanTilingState()
        s.map = ctypes.pointer(self.amap.c)
        s.n_controls, s.loss_capacity = self.C, self.loss.numel()
        s.allele_mask, s.pi_a0, s.counts = self.allele_mask_u8.data_ptr(), self.pi_a0.data_ptr(), self.counts.data_ptr()
        s.edit_params, s.edit_m, s.edit_v, s.edit_grad = (t.data_ptr() for t in (self.edit_params, self.edit_m, self.edit_v, self.edit_grad))
        s.alpha_u, s.alpha_m, s.alpha_v, s.alpha_grad = (t.data_ptr() for t in (self.alpha_u, self.alpha_m, self.alpha_v, self.alpha_grad))
        s.mu_e, s.sd_e, s.d_slot = self.mu_e.data_ptr(), self.sd_e.data_ptr(), self.d_slot.data_ptr()
        s.partial, s.counter, s.loss = self.partial.data_ptr(), self.counter.data_ptr(), self.loss.data_ptr()
        set_prior_pointers(s, self._prior_v)
        s.epsilon, s.pi_tiny = float(epsilon), float(torch.finfo(pi_dtype(dtype, pa0)).tiny)
        if self.sharded:
            import torch.distributed as dist

            self.edit_sum = torch.zeros((2, E), **kw)
            self.edit_iota = torch.arange(E + 1, dtype=torch.int32, device=dev)
            s.edit_sum, s.edit_iota = self.edit_sum.data_ptr(), self.edit_iota.data_ptr()
            s.edit_term_weight = 1.0 if dist.get_rank(group) == 0 else 0.0  # the per-edit ELBO terms count once
        s.nonfinite_step = self._init_nonfinite()
        self.state = s

    # ---------------------------------------------------------------------------------------------
    def _launch(self, first, n_steps, noise, apply_update):
        n, keep = None, []
        if noise is not None:
            n = _lib.BeanTilingNoise()
            if noise.get("record"):
                self.eps_used = torch.zeros((2, self.E), device=self.device, dtype=self.dtype)
                self.pi_used = torch.zeros((self.R, self.G, self.A), device=self.device, dtype=torch.float64)
                n.eps_out, n.pi_out = self.eps_used.data_ptr(), self.pi_used.data_ptr()
            if "eps_mu" in noise:
                self._put(keep, n, "eps_mu", noise["eps_mu"].reshape(-1), (self.E,))
                self._put(keep, n, "eps_sd", noise["eps_sd"].reshape(-1), (self.E,))
            if "pi" in noise:
                pi = noise["pi"]
                if pi.dim() == 4:  # reference layout (R, 1, G, A)
                    pi = pi[:, 0]
                self._put(keep, n, "pi", pi, (self.R, self.G, self.A), dtype=torch.float64)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        run = getattr(self.lib, _RUN[self.dtype])
        if not self.sharded:
            _lib.check(run(self.screen.c, self.state, self.cfg, n, first, n_steps, stream), _RUN[self.dtype])
        else:
            # per step: this shard's guides -> per-edit gradient sums; one all-reduce of 2 E numbers (edits are shared between
            # guides of different shards); then every rank updates every edit from the same sums
            import torch.distributed as dist

            for t in range(first, first + n_steps):
                self.cfg.phases = 1
                _lib.check(run(self.screen.c, self.state, self.cfg, n, t, 1, stream), _RUN[self.dtype])
                dist.all_reduce(self.edit_sum, group=self.group)
                self.cfg.phases = 2
                _lib.check(run(self.screen.c, self.state, self.cfg, n, t, 1, stream), _RUN[self.dtype])
            self.cfg.phases = 0
        return keep

    def _snapshot_tensors(self):
        return [self.edit_params, self.edit_m, self.edit_v, self.alpha_u, self.alpha_m, self.alpha_v]

    def _grads(self):
        return {"alpha_pi": self.alpha_grad, **dict(zip(("mu_loc", "mu_scale", "sd_loc", "sd_scale"), self.edit_grad))}

    def params(self) -> Dict[str, torch.Tensor]:
        """Constrained parameter values under the reference's names and shapes."""
        ep = self.edit_params
        alpha = torch.where(self.allele_mask, self.alpha_u.exp(), torch.full_like(self.alpha_u, float(self.state.epsilon)))
        return {"mu_loc": ep[0].clone(), "mu_scale": ep[1].exp(), "sd_loc": ep[2].clone(), "sd_scale": ep[3].exp(), "alpha_pi": alpha}
