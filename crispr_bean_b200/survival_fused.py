"""Device-resident SVI engine of the survival (proliferation) MixtureNormal program: host side of `bean_svi_survival_run_*`.

One step = `svi.step` of bean/model/run.py:376-380 for bean/model/survival_model.py:215-424 / :651-739 in three kernel
launches (per-guide, alpha_pi, per-variant; include/bean_b200.h), no torch op and no host round trip per step.  Parameter
names, shapes and initial values follow the pyro guide (survival_model.py:651-698): mu_loc = 0, mu_scale = 1 (T, 1),
alpha_pi = alpha_prior (G, 2), q0 = 1 / G (G,).

Sharding (SURVEY section 8e): guides may be split over the ranks of a torch.distributed group in contiguous variant blocks
(`dist.shard_data`).  The program's Dirichlet over ALL guides then needs R + 1 library-wide sums per step -- sum_g gamma[r][g]
and sum_g q0[g] -- the path's only data-path collective.  Where the ranks are the GPUs of one box they trade these numbers
INSIDE the kernels through CUDA-IPC-mapped peer memory (the per-variant kernel's last CTA stores its partial sums into every
rank's buffer over NVLink and raises a flag, the next step's guide kernel waits for the flags; csrc/bean_peer.cu), so that N
steps are one C call as on a single GPU and the host all-reduces only the sums the next call starts from.  Otherwise (peer
mapping unavailable, a single step, a kernel timed alone) this engine launches step by step and all-reduces the buffer with
NCCL between consecutive steps.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Dict, Optional

import torch

from . import _lib
from .device_pack import DeviceScreen, row_constants
from .halt import NonfiniteWatch

_RUN = {torch.float32: "bean_svi_survival_run_f32", torch.float64: "bean_svi_survival_run_f64"}


def _dist_active(group) -> bool:
    import torch.distributed as dist

    return dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1


class SurvivalFusedEngine(NonfiniteWatch):
    def __init__(self, data, device="cuda", dtype=torch.float32, use_bcmatch: bool = True, num_steps: int = 2000,
                 initial_lr: float = 0.01, gamma: float = 0.1, seed: int = 101, alpha_prior: float = 1.0, mask_thres: int = 10,
                 prior_params: Optional[dict] = None, mu_negctrl=(0.0, 0.1), group=None, guide_offset: int = 0,
                 variant_offset: int = 0, screen: Optional[DeviceScreen] = None):
        if not getattr(data, "is_survival", False):
            raise ValueError("SurvivalFusedEngine needs a *SurvivalScreenData object")
        if not torch.cuda.is_available():
            raise _lib.BeanError("SurvivalFusedEngine needs a CUDA device: there is no CPU fallback")
        self.lib = _lib.lib()
        self.model, self.dtype, self.device, self.group = "MixtureNormal", dtype, torch.device(device), group
        self.num_steps = int(num_steps)
        self.sharded = _dist_active(group)
        use_bcmatch = bool(use_bcmatch) and getattr(data, "X_bcmatch_masked", None) is not None
        self.screen = screen or DeviceScreen(data, self.device, dtype=dtype, use_bcmatch=use_bcmatch, mask_thres=mask_thres)
        G, R, T = self.screen.n_guides, self.screen.n_reps, int(data.n_targets)
        self.G, self.R, self.T = G, R, T
        dev, kw = self.device, dict(device=self.device, dtype=dtype)
        g_total = torch.tensor([float(G)], device=dev, dtype=torch.float64)
        self._all_reduce(g_total)
        self.G_total = int(g_total.item())
        self.guide_variant = data.guide_variant.to(dev).contiguous()
        self.variant_ptr = data.variant_ptr.to(dev).contiguous()
        # variant parameters in the layout of the shared per-variant kernel: rows (mu_loc, log mu_scale, -, -)
        self.var_params = torch.zeros((4, T), **kw)
        self.var_m, self.var_v, self.var_grad = torch.zeros((4, T), **kw), torch.zeros((4, T), **kw), torch.zeros((4, T), **kw)
        self.d_guide = torch.zeros((2, G), **kw)
        self.alpha_u = torch.full((G, 2), float(alpha_prior), **kw).log()
        self.alpha_m, self.alpha_v, self.alpha_grad = torch.zeros((G, 2), **kw), torch.zeros((G, 2), **kw), torch.zeros((G, 2), **kw)
        self.q0_u = torch.full((G,), 1.0 / self.G_total, **kw).log()
        self.q0_m, self.q0_v, self.q0_grad = torch.zeros(G, **kw), torch.zeros(G, **kw), torch.zeros(G, **kw)
        ac = data.allele_counts_control  # (R, C, G, 2): the reference's own layout
        self.C = int(ac.shape[1])
        self.allele_counts = ac.to(dev).to(dtype).contiguous()
        self.pi_a0 = torch.as_tensor(data.pi_a0).to(**kw).contiguous()
        self._tc = (C.c_double * self.C)(*[float(t) for t in data.control_timepoint.double().reshape(-1)])
        # observed initial abundance (survival_model.py:306-311): (X[:, 0] + 1) / its sum over ALL guides
        x0 = data.X[:, 0, :].to(dev).double() + 1.0
        tot = x0.sum(-1, keepdim=True)
        self._all_reduce(tot)
        self.log_obs = (x0 / tot).log().to(dtype).contiguous()  # (R, G)
        self.gamma = [torch.zeros((R, G), **kw), torch.zeros((R, G), **kw)]
        self.sums = [torch.zeros(R + 1, dtype=torch.float64, device=dev), torch.zeros(R + 1, dtype=torch.float64, device=dev)]
        n_partial = self.lib.bean_svi_num_partials(G, T)
        self.partial = torch.zeros(n_partial, dtype=torch.float64, device=dev)
        self.abund_partial = torch.zeros(((G + 127) // 128 * 4 + _lib.SURV_FOLD_ROWS, R + 1), dtype=torch.float64, device=dev)
        self.counter = torch.zeros(1, dtype=torch.int32, device=dev)
        self.loss = torch.zeros(max(self.num_steps, 1) + 1, dtype=torch.float64, device=dev)
        self.pw, self.dconc = torch.empty((R, G, 4), **kw), torch.empty((G, 4), **kw)
        self.step, self._primed = 0, False
        # data-only parts of the ELBO: Dirichlet-Multinomial rows (DeviceScreen) + the reporter Multinomial's coefficient
        mconst, _ = row_constants(self.allele_counts, with_xlogx=False)  # (R, C, G)
        ll_const = self.screen.ll_const + float((mconst * (self.screen.row_mask != 0).unsqueeze(1)).sum())

        c = _lib.BeanSviConfig()
        c.model, c.sd_is_sqrt, c.apply_update, c.fit_noise = _lib.MODEL_MIXTURE_NORMAL, 0, 1, 0
        c.mu_prior_normal, c.mu_prior_loc, c.mu_prior_scale = 0, 0.0, 1.0
        self._prior_v = {}
        if prior_params and ("mu_loc" in prior_params or "mu_scale" in prior_params):
            c.mu_prior_normal = 1
            for key in ("mu_loc", "mu_scale"):
                if key in prior_params:
                    val = prior_params[key]
                    if torch.is_tensor(val) and val.numel() > 1:
                        if val.numel() != T:
                            raise ValueError(f"prior_params[{key!r}] has {val.numel()} entries for {T} variants")
                        self._prior_v[key] = val.detach().reshape(-1).to(**kw).contiguous()
                    else:
                        setattr(c, f"mu_prior_{key[3:]}", float(val))
        c.sd_prior_loc, c.sd_prior_scale = 0.0, 1.0
        c.lr0, c.lrd = float(initial_lr), float(gamma) ** (1.0 / max(self.num_steps, 1))
        c.beta1, c.beta2, c.adam_eps, c.clip = 0.9, 0.999, 1e-8, 10.0
        c.ll_const, c.seed = ll_const, int(seed)
        # the reference evaluates pi exp(mu t_c) in the promoted dtype of (pi_a0, control_timepoint): float64 out of its data
        # class even on the float32 path, and torch's Multinomial clamps probabilities at the eps of THAT dtype
        pa0 = getattr(data, "pi_a0", None)
        ref_dtype = dtype
        for t in (pa0, data.control_timepoint):
            if torch.is_tensor(t):
                ref_dtype = torch.promote_types(ref_dtype, t.dtype)
        c.prob_clamp_eps = float(torch.finfo(ref_dtype).eps)
        c.guide_offset, c.variant_offset = int(guide_offset), int(variant_offset)
        self.cfg = c

        s = _lib.BeanSviState()
        s.n_variants, s.loss_capacity = T, self.loss.numel()
        s.guide_variant, s.variant_ptr = self.guide_variant.data_ptr(), self.variant_ptr.data_ptr()
        s.allele_counts, s.pi_a0 = self.allele_counts.data_ptr(), self.pi_a0.data_ptr()
        s.alpha_u, s.alpha_m, s.alpha_v, s.alpha_grad = (t.data_ptr() for t in (self.alpha_u, self.alpha_m, self.alpha_v, self.alpha_grad))
        s.var_params, s.var_m, s.var_v, s.var_grad = (t.data_ptr() for t in (self.var_params, self.var_m, self.var_v, self.var_grad))
        s.d_guide = self.d_guide.data_ptr()
        s.partial, s.counter, s.loss = self.partial.data_ptr(), self.counter.data_ptr(), self.loss.data_ptr()
        s.pw, s.dconc = self.pw.data_ptr(), self.dconc.data_ptr()
        if "mu_loc" in self._prior_v:
            s.mu_prior_loc_v = self._prior_v["mu_loc"].data_ptr()
        if "mu_scale" in self._prior_v:
            s.mu_prior_scale_v = self._prior_v["mu_scale"].data_ptr()
        s.nonfinite_step = self._init_nonfinite()
        self.state = s

        v = _lib.BeanSurvivalState()
        v.n_controls, v.n_guides_total = self.C, self.G_total
        v.control_time = self._tc
        v.negctrl_loc, v.negctrl_scale = float(mu_negctrl[0]), float(mu_negctrl[1])
        v.log_obs = self.log_obs.data_ptr()
        v.q0_u, v.q0_m, v.q0_v, v.q0_grad = (t.data_ptr() for t in (self.q0_u, self.q0_m, self.q0_v, self.q0_grad))
        v.gamma[0], v.gamma[1] = self.gamma[0].data_ptr(), self.gamma[1].data_ptr()
        v.sums[0], v.sums[1] = self.sums[0].data_ptr(), self.sums[1].data_ptr()
        v.abund_partial = self.abund_partial.data_ptr()
        v.nonfinite_step = s.nonfinite_step
        self.surv = v
        self.peers, self._peers_tried = None, False  # opened by the first multi-step call of a sharded run (_open_peer_exchange)

    # ---------------------------------------------------------------------------------------------
    def _open_peer_exchange(self):
        """The device-side exchange of the library-wide sums (include/bean_b200.h: BeanPeerBuffer): this rank's buffer, the
        other ranks' mapped through CUDA IPC.  Returns None (the host all-reduces between the steps instead) where peer
        mapping is not available -- a group that is not the GPUs of one box, or IPC refused by the driver."""
        import torch.distributed as dist

        world, rank = dist.get_world_size(self.group), dist.get_rank(self.group)
        if world > _lib.MAX_PEERS or self.R + 1 > _lib.PEER_MAX_VALS or os.environ.get("BEAN_NO_PEER_EXCHANGE"):
            return None
        own, handle = C.c_void_p(), (C.c_ubyte * 64)()
        ok = self.lib.bean_peer_alloc(C.byref(own), handle) == 0
        mine = torch.tensor(list(handle) + [1 if ok else 0], dtype=torch.uint8, device=self.device)
        everyone = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(everyone, mine, group=self.group)
        ex = _lib.BeanPeerExchange()
        ex.world, ex.rank = world, rank
        opened, good = [], ok and all(int(h[64]) == 1 for h in everyone)
        if good:
            for k, h in enumerate(everyone):
                if k == rank:
                    ex.buf[k] = own.value
                    continue
                ptr, raw = C.c_void_p(), (C.c_ubyte * 64)(*h[:64].tolist())
                if self.lib.bean_peer_open(raw, C.byref(ptr)) != 0:
                    good = False
                    break
                ex.buf[k] = ptr.value
                opened.append(ptr.value)
        # every rank must take the same path: one that cannot map its peers sends everybody back to the host exchange
        flag = torch.tensor([1 if good else 0], dtype=torch.int32, device=self.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=self.group)
        if int(flag.item()) == 0:
            for ptr in opened:
                self.lib.bean_peer_close(ptr)
            if ok:
                self.lib.bean_peer_free(own)
            return None
        self._peer_own, self._peer_opened = own.value, opened
        return ex

    def _peer_exchange(self):
        if not self._peers_tried:  # a collective of the group: every rank gets here in the same call
            self._peers_tried = True
            self.peers = self._open_peer_exchange()
        return self.peers

    def peer_timeouts(self) -> int:
        """Waits of the device-side exchange that gave up (0 on a healthy run); synchronises."""
        if self.peers is None:
            return 0
        out = C.c_uint64()
        _lib.check(self.lib.bean_peer_timeouts(self._peer_own, C.byref(out)), "bean_peer_timeouts")
        return int(out.value)

    def __del__(self):
        try:
            if getattr(self, "peers", None) is not None:
                torch.cuda.synchronize(self.device)
                for ptr in self._peer_opened:
                    self.lib.bean_peer_close(ptr)
                self.lib.bean_peer_free(self._peer_own)
                self.peers = None
        except Exception:  # pragma: no cover  (interpreter shutdown)
            pass

    def _snapshot_tensors(self):
        # the abundance draws and library-wide sums of the next step are written by the step before it
        return [self.var_params, self.var_m, self.var_v, self.alpha_u, self.alpha_m, self.alpha_v, self.q0_u, self.q0_m, self.q0_v,
                *self.gamma, *self.sums]

    def _snapshot_extra(self):
        return {"primed": self._primed}

    def _restore_extra(self, snap):
        self._primed = snap["primed"]
        if self.peers is not None:
            # the exchange flags hold the step each rank last published and only grow: steps run again would not wait for
            # their peers.  Every rank stops writing, then zeroes its own flags before any rank runs again.
            import torch.distributed as dist

            torch.cuda.synchronize(self.device)
            dist.barrier(group=self.group)
            _lib.check(self.lib.bean_peer_reset_flags(self._peer_own), "bean_peer_reset_flags")
            dist.barrier(group=self.group)

    def _all_reduce(self, t):
        if _dist_active(self.group):
            import torch.distributed as dist

            dist.all_reduce(t, group=self.group)
        return t

    def _noise_structs(self, noise):
        if noise is None:
            return None, None, ()
        kw = dict(device=self.device, dtype=self.dtype)
        n, sn, keep = _lib.BeanSviNoise(), _lib.BeanSurvivalNoise(), []

        def put(struct, field, tensor, shape):
            t = tensor.to(**kw).contiguous()
            assert tuple(t.shape) == shape, (field, tuple(t.shape), shape)
            setattr(struct, field, t.data_ptr())
            keep.append(t)

        if "eps_mu" in noise:
            put(n, "eps_mu", noise["eps_mu"].reshape(-1), (self.T,))
        if "pi" in noise:
            pi = noise["pi"]
            if pi.dim() == 4:  # reference layout (R, 1, G, 2) -> kernel layout (G, R, 2)
                pi = pi[:, 0].permute(1, 0, 2)
            put(n, "pi", pi, (self.G, self.R, 2))
        if "eps_negctrl" in noise:
            put(sn, "eps_negctrl", noise["eps_negctrl"].reshape(-1), (self.G,))
        if "q0" in noise:
            put(sn, "q0", noise["q0"], (self.R, self.G))
        return n, sn, keep

    def _launch(self, first, n, noise_structs, prime):
        n_struct, sn_struct, keep = noise_structs
        self.surv.prime = prime
        stream = torch.cuda.current_stream(self.device).cuda_stream
        rc = getattr(self.lib, _RUN[self.dtype])(self.screen.c, self.state, self.surv, self.cfg, n_struct, sn_struct, first, n, stream)
        _lib.check(rc, _RUN[self.dtype])
        self._keep = keep

    def run(self, n_steps: int, noise: Optional[Dict[str, torch.Tensor]] = None, apply_update: bool = True):
        """Advance `n_steps` SVI steps (asynchronously); injected `noise` applies to every one of them."""
        if self.step + n_steps > self.loss.numel() - (1 if apply_update else 0):
            raise ValueError("loss buffer exhausted: construct the engine with a larger num_steps")
        ns = self._noise_structs(noise)
        self.cfg.apply_update = 1 if apply_update else 0
        first = self.step
        self.surv.peers = None
        if not self.sharded:
            self._launch(first, n_steps, ns, _lib.SURV_PRIME_NONE if self._primed else _lib.SURV_PRIME_AND_RUN)
        elif apply_update and self.cfg.phases == 0 and n_steps > 1 and self._peer_exchange() is not None:
            # device-side exchange: the ranks trade their R + 1 partial sums through peer memory inside the kernels, the host
            # all-reduces only the sums the NEXT call starts from
            if not self._primed:
                self._launch(first, 1, ns, _lib.SURV_PRIME_ONLY)
                self._all_reduce(self.sums[first & 1])
                self._primed = True
            self.surv.peers = C.pointer(self.peers)
            self._launch(first, n_steps, ns, _lib.SURV_PRIME_NONE)
            self.surv.peers = None
            self._all_reduce(self.sums[(first + n_steps) & 1])
        else:
            for t in range(first, first + n_steps):
                if not self._primed:
                    self._launch(t, 1, ns, _lib.SURV_PRIME_ONLY)
                    self._all_reduce(self.sums[t & 1])
                    self._primed = True
                self._launch(t, 1, ns, _lib.SURV_PRIME_NONE)
                if apply_update:
                    self._all_reduce(self.sums[(t + 1) & 1])  # the exchange step: R + 1 doubles per SVI step
        self._primed = True
        if apply_update:
            self.step += n_steps
        return self.loss[first:first + n_steps]

    def gradients(self, noise=None) -> Dict[str, torch.Tensor]:
        """Loss and its gradient w.r.t. the unconstrained parameters at the current point (no update)."""
        loss = self.run(1, noise=noise, apply_update=False)
        return {"loss": loss[0].clone(), "mu_loc": self.var_grad[0].clone(), "mu_scale": self.var_grad[1].clone(),
                "alpha_pi": self.alpha_grad.clone(), "q0": self.q0_grad.clone()}

    def params(self) -> Dict[str, torch.Tensor]:
        """Constrained parameter values under the reference's names and shapes."""
        T = self.T
        return {"mu_loc": self.var_params[0].reshape(T, 1).clone(), "mu_scale": self.var_params[1].exp().reshape(T, 1),
                "alpha_pi": self.alpha_u.exp(), "q0": self.q0_u.exp()}

    def losses(self):
        return self.loss[: self.step].cpu()
