"""SVI engine for the tiling model (`MultiMixtureNormal`): torch autograd around the CUDA kernels.

The hot parts -- Normal-CDF bin masses, allele mixture, get_alpha and the Dirichlet-Multinomial rows with
their backward (`bean_ll_*`), and the allele <- edit contraction (`bean_allele_gather/scatter_*`) -- are the
C-ABI kernels; the O(G A) Dirichlet / Multinomial editing-rate sites, the priors and ClippedAdam are
ordinary torch CUDA ops (plumbing).  Mirrors bean/model/model.py:550-751 (model) and :878-962 (guide);
one `step()` = one `svi.step` of bean/model/run.py:376-380 with the loss kept on the device.

A step is ~200 small kernels (forward, backward, Adam); launched one by one from Python it is launch-bound (4.5 ms at
c3 / c4 size), so `run()` captures ONE step into a CUDA graph and replays it: the step counter, the ClippedAdam step
size of every step and the loss log live on the device, the generator is registered with the graph.
"""
from __future__ import annotations

import math
from typing import Dict, Optional

import torch
import torch.distributions as tdist

from . import _lib
from ._lib import BeanError
from .device_pack import DeviceScreen
from .halt import NonfiniteWatch
from .dirichlet import DirichletStream, dirichlet_rsample
from .ll_function import count_log_likelihood
from .latent_sites import LatentPrior, latent_sites
from .pi_sites import PiSiteData, pi_sites
from .tiling import AlleleMap, allele_gather

EPS = 1e-5
PI_NOISE_SD = 0.655


def _multinomial_log_prob(probs, value):
    """torch.distributions.Multinomial(probs=probs).log_prob(value) (probs normalised over the last axis and clamped to
    [eps, 1 - eps] of their dtype, then logged), written out because the distribution's constructor builds a Binomial
    from the python scalar total_count -- a host-to-device copy, which cannot be captured into a CUDA graph."""
    eps = torch.finfo(probs.dtype).eps
    logits = (probs / probs.sum(-1, keepdim=True)).clamp(min=eps, max=1 - eps).log()
    value = value.to(logits.dtype)
    return torch.lgamma(value.sum(-1) + 1) - torch.lgamma(value + 1).sum(-1) + (logits * value).sum(-1)


def _masked_sum(mask, lp):
    return torch.where(mask, lp, torch.zeros_like(lp)).sum()


class AutogradSviEngine(NonfiniteWatch):
    """Shared SVI plumbing of the models whose ELBO is assembled from torch CUDA ops around the C-ABI kernels:
    unconstrained parameters (positive ones as log), ClippedAdam (SURVEY App. A.6), device-side loss log."""

    def _init_optim(self, theta, positive, num_steps, initial_lr, gamma, seed):
        self.theta, self.positive = theta, set(positive)
        for p in self.theta.values():
            p.requires_grad_(True)
        self.m = {k: torch.zeros_like(v) for k, v in self.theta.items()}
        self.v = {k: torch.zeros_like(v) for k, v in self.theta.items()}
        self.lr0, self.lrd, self.num_steps = float(initial_lr), float(gamma) ** (1.0 / max(num_steps, 1)), int(num_steps)
        self.step = 0
        self.loss = torch.zeros(max(num_steps, 1), dtype=torch.float64, device=self.device)
        # draws of different shards must be independent (a Dirichlet over all guides is assembled from the shards' gammas):
        # the generator stream is keyed by (seed, rank of this shard)
        rank = 0
        import torch.distributed as dist

        if dist.is_available() and dist.is_initialized():
            rank = dist.get_rank(getattr(self, "group", None))
        self.gen = torch.Generator(device=self.device).manual_seed(int(seed) + 1_000_003 * rank)
        # device-side step counter and the ClippedAdam step size of every step (SURVEY App. A.6): a captured step reads
        # step_sizes[t] and writes loss[t], then increments t -- nothing about a step depends on the host
        t = torch.arange(1, max(num_steps, 1) + 1, dtype=torch.float64)
        self._step_sizes = (self.lr0 * self.lrd ** t * torch.sqrt(1 - 0.999 ** t) / (1 - 0.9 ** t)).to(self.device)
        self._t = torch.zeros(1, dtype=torch.int64, device=self.device)
        self._nonfinite_ptr = self._init_nonfinite()
        # the `pi` draws: counter-based, keyed by (seed, global guide id, replicate, allele, device step counter)
        self.pi_stream = DirichletStream(seed, self._t, guide_offset=getattr(self, "guide_offset", 0), site=0)
        self._graph, self._graph_noise, self.use_graph = None, None, True
        self._const = {}

    def _prior_t(self, value):
        """A prior hyper-parameter (python scalar or tensor) as a device tensor, converted once."""
        if not torch.is_tensor(value):
            return self._c(value)
        key = ("t", id(value))
        if key not in self._const:
            self._const[key] = value.detach().to(device=self.device, dtype=self.dtype)
        return self._const[key]

    def _c(self, value):
        """A python scalar as a cached 0-dim device tensor (no host-to-device copy inside a step: not capturable)."""
        key = float(value)
        if key not in self._const:
            self._const[key] = torch.full((), key, device=self.device, dtype=self.dtype)
        return self._const[key]

    def _draw(self, noise, key, shape):
        if noise is not None and key in noise:
            return noise[key].to(device=self.device, dtype=self.dtype).reshape(shape)
        return torch.randn(shape, generator=self.gen, device=self.device, dtype=self.dtype)

    # -- --scale-by-acc (bean/model/utils.py:79-178) ---------------------------------------------------
    def _acc_init(self, data, theta, positive, fit_noise):
        """Accessibility factor exp(b) acc^a (a = 0.2513, b = -1.9458) and, with fit_noise, the guide's
        (noise_loc, noise_scale) parameters of the logit-space noise site (initial values utils.py:146-151)."""
        if getattr(data, "guide_accessibility", None) is None:
            raise ValueError("scale_by_accessibility needs data.guide_accessibility (accessibility_col)")
        acc = torch.as_tensor(data.guide_accessibility).double()
        self.acc_k = (math.exp(-1.9458) * acc.pow(0.2513)).to(device=self.device, dtype=self.dtype)
        self.fit_noise = bool(fit_noise)
        if self.fit_noise:
            G = acc.numel()
            theta["noise_loc"] = torch.zeros(G, device=self.device, dtype=self.dtype)
            theta["noise_scale"] = torch.full((G,), PI_NOISE_SD, dtype=torch.float64).log().to(device=self.device, dtype=self.dtype)
            positive.add("noise_scale")

    def _acc_apply(self, pi, noise):
        """pi (R, 1, G, A) -> accessibility-scaled, logit-noised pi; returns (pi, model_lp, guide_lp) of the
        `logit_pi_noise` site.  The model never receives fit_noise (SURVEY App. B3): its density is the prior."""
        kw = dict(device=self.device, dtype=self.dtype)
        G = pi.shape[2]
        eps = self._draw(noise, "eps_noise", (G,))
        prior = tdist.Normal(self._c(0.0), self._c(PI_NOISE_SD))
        if self.fit_noise:
            loc, scale = self.theta["noise_loc"], self.theta["noise_scale"].exp()
            val = loc + scale * eps
            guide_lp = tdist.Normal(loc, scale).log_prob(val).sum()
        else:
            val = PI_NOISE_SD * eps
            guide_lp = prior.log_prob(val).sum()
        model_lp = prior.log_prob(val).sum()
        scaled = pi[..., 1:] * self.acc_k.reshape(1, 1, G, 1)                       # _scale_edited_pi
        full = torch.cat([(1 - scaled.sum(-1)).unsqueeze(-1), scaled], dim=-1)
        full = full / full.sum(-1).clamp(min=1.0).unsqueeze(-1)                      # only if the edited rates exceed 1
        logit = torch.logit(full[..., 1:].clamp(min=1e-3, max=1 - 1e-3)) + val.reshape(1, 1, G, 1)   # add_noise_to_pi
        ex = torch.exp(logit)
        noised = (ex / (1 + ex)).clamp(min=1e-3, max=1 - 1e-3)
        out = torch.cat([(1 - noised.sum(-1)).unsqueeze(-1), noised], dim=-1)       # WT may go negative (App. B10)
        return out, model_lp, guide_lp

    def _adam(self):
        """pyro.optim.ClippedAdam on the unconstrained tensors (SURVEY App. A.6): one `bean_clipped_adam` launch for all
        tensors of a dtype, step index and step size read from the device (capturable)."""
        stream = torch.cuda.current_stream(self.device).cuda_stream
        self._adam_keep = []  # gradient buffers stay referenced until the next step
        for dtype, name in ((torch.float32, "bean_clipped_adam_f32"), (torch.float64, "bean_clipped_adam_f64")):
            args, n = _lib.BeanAdamArgs(), 0
            for k, p in self.theta.items():
                if p.grad is None or p.dtype != dtype:
                    continue
                if n == _lib.ADAM_MAX_TENSORS:
                    raise BeanError(f"more than {_lib.ADAM_MAX_TENSORS} parameter tensors")
                g = p.grad.contiguous()
                if not (p.is_contiguous() and p.is_cuda and g.dtype == dtype and self.m[k].dtype == dtype and self.v[k].dtype == dtype):
                    raise BeanError(f"parameter {k}: the optimiser kernel needs contiguous CUDA tensors of one dtype")
                self._adam_keep.append(g)
                t = args.tensors[n]
                t.theta, t.grad, t.m, t.v, t.n = p.data_ptr(), g.data_ptr(), self.m[k].data_ptr(), self.v[k].data_ptr(), p.numel()
                n += 1
            if n == 0:
                continue
            args.n_tensors = n
            args.step_sizes, args.step, args.n_steps = self._step_sizes.data_ptr(), self._t.data_ptr(), self._step_sizes.numel()
            args.beta1, args.beta2, args.eps, args.clip = 0.9, 0.999, 1e-8, 10.0
            args.loss, args.nonfinite_step = self.loss.data_ptr(), self._nonfinite_ptr  # loss[t] is written before this launch
            _lib.check(getattr(_lib.lib(), name)(args, stream), name)

    def _step_once(self, noise):
        """One SVI step, entirely on the device (capturable)."""
        prev = tdist.Distribution._validate_args
        tdist.Distribution.set_default_validate_args(False)  # argument validation synchronises with the host
        try:
            loss = self.elbo_loss(noise)
            loss.backward()
        finally:
            tdist.Distribution.set_default_validate_args(prev)
        with torch.no_grad():
            self.loss.index_copy_(0, self._t.clamp(max=self.loss.numel() - 1), loss.detach().double().reshape(1))
        self._adam()
        self._t.add_(1)

    def _capture(self, noise):
        """Capture one step into a CUDA graph (torch.cuda.graph: side-stream warm-up, private memory pool, generator
        registered).  Warm-up steps run for real, so the optimiser state is snapshotted and restored around them."""
        keep = [(t, t.detach().clone()) for t in list(self.theta.values()) + list(self.m.values()) + list(self.v.values())
                + [self._t, self.loss]]
        gen_state = self.gen.get_state()  # the warm-up draws must not advance the run's noise stream
        side = torch.cuda.Stream(self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(side):
            for _ in range(2):
                for p in self.theta.values():
                    p.grad = None
                self._step_once(noise)
        torch.cuda.current_stream(self.device).wait_stream(side)
        for p in self.theta.values():
            p.grad = None  # the captured backward allocates the gradients inside the graph's pool
        self.gen.set_state(gen_state)
        graph = torch.cuda.CUDAGraph()
        graph.register_generator_state(self.gen)
        with torch.cuda.graph(graph):
            self._step_once(noise)
        with torch.no_grad():
            for t, saved in keep:
                t.copy_(saved)
        self._graph, self._graph_noise = graph, noise

    def _graph_ok(self, n_steps):
        if not (self.use_graph and self.device.type == "cuda" and n_steps >= 4):
            return False
        import torch.distributed as dist

        return not (dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1)  # collectives stay eager

    def run(self, n_steps: int, noise=None, use_graph: Optional[bool] = None):
        """Advance `n_steps` SVI steps; `noise` (parity runs) is injected into every one of them."""
        if self.step + n_steps > self.loss.numel():
            raise ValueError("loss buffer exhausted: construct the engine with a larger num_steps")
        if noise is not None:
            noise = {k: (v.to(self.device) if torch.is_tensor(v) else v) for k, v in noise.items()}
        graph = self._graph_ok(n_steps) if use_graph is None else use_graph
        if graph:
            if self._graph is None or self._graph_noise is not noise:
                if noise is not None and self._graph is not None and self._graph_noise is not None \
                        and set(noise) == set(self._graph_noise):
                    for k, v in noise.items():  # same keys: refill the captured buffers instead of re-capturing
                        self._graph_noise[k].copy_(v)
                else:
                    self._capture(noise)
            for _ in range(n_steps):
                self._graph.replay()
        else:
            for _ in range(n_steps):
                for p in self.theta.values():
                    p.grad = None
                self._step_once(noise)
        self.step += n_steps
        return self.loss[self.step - n_steps:self.step]

    def _snapshot_tensors(self):
        return [*self.theta.values(), *self.m.values(), *self.v.values(), self._t]

    def _snapshot_extra(self):
        return {"gen": self.gen.get_state()}  # the captured step replays from the registered generator

    def _restore_extra(self, snap):
        self.gen.set_state(snap["gen"])

    def gradients(self, noise=None):
        for p in self.theta.values():
            p.grad = None
        loss = self.elbo_loss(noise)
        loss.backward()
        out = {"loss": loss.detach().clone()}
        for k, p in self.theta.items():
            out[k] = (p.grad if p.grad is not None else torch.zeros_like(p)).detach().clone()
            p.grad = None
        return out

    def params(self):
        """Constrained values under the reference's parameter names."""
        return {k: (v.detach().exp() if k in self.positive else v.detach().clone()) for k, v in self.theta.items()}

    def losses(self):
        return self.loss[: self.step].cpu()


class TilingSviEngine(AutogradSviEngine):
    """MultiMixtureNormal on one GPU.  Parameter names / shapes follow the pyro guide (model.py:893-937)."""

    def __init__(self, data, device="cuda", dtype=torch.float32, use_bcmatch=True, num_steps=2000, initial_lr=0.01,
                 gamma=0.1, seed=101, alpha_prior=1.0, sd_scale=0.01, epsilon=EPS, prior_params: Optional[dict] = None,
                 scale_by_accessibility: bool = False, fit_noise: bool = False):
        if not torch.cuda.is_available():
            raise BeanError("TilingSviEngine needs a CUDA device: there is no CPU fallback")
        self.device, self.dtype = torch.device(device), dtype
        kw = dict(device=self.device, dtype=dtype)
        self.screen = DeviceScreen(data, self.device, dtype=dtype, use_bcmatch=use_bcmatch, mask_thres=10)
        self.G, self.R, self.A, self.E = data.n_guides, data.n_reps, data.n_max_alleles, data.n_edits
        self.amap = AlleleMap(data.allele_ptr.numpy(), data.allele_edit.numpy(), self.G, self.A, self.E, self.device)
        self.allele_mask = data.allele_mask.to(self.device)
        self.allele_mask_u8 = self.allele_mask.to(torch.uint8).contiguous()
        # pi_a0 keeps its own dtype (float64 out of the a0 fit): as in the reference, the editing-rate concentrations and
        # the pi draws are then float64 even on the float32 path (draws of non-existent alleles underflow float32)
        self.pi_a0 = torch.as_tensor(data.pi_a0).to(self.device)
        self.allele_counts_control = data.allele_counts_control.to(**kw)  # (R, C, G, A)
        self.rg_mask = data.repguide_mask.to(self.device).unsqueeze(1)  # (R, 1, G)
        self.pi_data = PiSiteData(self.allele_counts_control, self.rg_mask, None, mask_guide_site=True)
        self.epsilon, self.sd_scale, self.prior_params = epsilon, sd_scale, prior_params
        a0 = torch.full((self.G, self.A), float(alpha_prior), **kw)
        a0[~self.allele_mask] = epsilon
        z = lambda *s: torch.zeros(s, **kw)
        # unconstrained parameters (positive ones as log), initial values of model.py:893-937
        theta = {"mu_loc": z(self.E), "mu_scale": z(self.E), "sd_loc": z(self.E), "sd_scale": z(self.E), "alpha_pi": a0.log()}
        positive = {"mu_scale", "sd_scale", "alpha_pi"}
        self.acc = bool(scale_by_accessibility)
        if self.acc:
            self._acc_init(data, theta, positive, fit_noise)
        self.latent_prior = LatentPrior(self.E, prior_params, sd_scale, self.device, dtype)
        self._init_optim(theta, positive, num_steps, initial_lr, gamma, seed)

    # ---------------------------------------------------------------------------------------------
    def elbo_loss(self, noise: Optional[Dict[str, torch.Tensor]] = None):
        """-ELBO of one particle (SURVEY App. A.5 site list for MultiMixtureNormal)."""
        kw = dict(device=self.device, dtype=self.dtype)
        E, G, A, R = self.E, self.G, self.A, self.R
        eps = self.epsilon
        P = self.theta
        alpha_pi = P["alpha_pi"].exp()
        alpha_pi = torch.where(self.allele_mask, alpha_pi, torch.full_like(alpha_pi, eps))  # model.py:645 / :937
        # `mu_alleles` / `sd_alleles` per edit: draws, Laplace | Normal and LogNormal priors, guide densities (one kernel)
        mu_e, sd_e, model_lp = latent_sites(P["mu_loc"], P["mu_scale"], self._draw(noise, "eps_mu", (E,)), self.latent_prior,
                                            P["sd_loc"], P["sd_scale"], self._draw(noise, "eps_sd", (E,)))
        guide_lp = self._c(0.0)

        # allele <- edit contraction (CUDA CSR gather / CSC scatter), WT column (0, 1)
        mu_a, sd_a = allele_gather(mu_e, sd_e, self.amap)

        # editing-rate sites (model.py:632-670 model, :938-950 guide: masked, not clamped)
        conc_g = alpha_pi / alpha_pi.sum(-1, keepdim=True) * self.pi_a0[:, None]  # (G, A)
        conc_m = (alpha_pi + eps / A) / (alpha_pi.sum(-1, keepdim=True) + eps) * self.pi_a0[:, None]
        conc_m = torch.where(conc_m < eps, torch.full_like(conc_m, eps), conc_m)
        injected = noise["pi"].to(self.device) if (noise is not None and "pi" in noise) else None  # cast to the concentration's dtype
        pi = dirichlet_rsample(conc_g, R, self.pi_stream, injected).unsqueeze(1)  # (R, 1, G, A): bean_dirichlet_rsample_*
        # model `pi` Dirichlet + reporter Multinomial - guide `pi` Dirichlet, all under repguide_mask: one kernel
        model_lp = model_lp + pi_sites(conc_g, conc_m, pi, self.pi_data)

        if self.acc:
            pi, m_lp, g_lp = self._acc_apply(pi, noise)
            model_lp, guide_lp = model_lp + m_lp, guide_lp + g_lp
        # count likelihood of both layers (CUDA): bin masses, mixture, get_alpha, Dirichlet-Multinomial
        pi_g = pi[:, 0].permute(1, 0, 2).contiguous()  # (G, R, A)
        model_lp = model_lp + count_log_likelihood(self.screen, mu_a, sd_a, pi_g, self.allele_mask_u8)
        return -(model_lp - guide_lp)


class CovariateNormalEngine(AutogradSviEngine):
    """Sorting `Normal` model with sample covariates (`screen.uns["sample_covariates"]`; model.py:73-91, guide :771-782).

    The covariate shifts the phenotype mean per REPLICATE, mu[r, g] = mu_targets[v(g)] + rep_by_cov[r, 0] * mu_cov[0]
    (only the first column of rep_by_cov * mu_cov is used, as in the reference).  The likelihood kernel takes one mean
    per (guide, allele), so the R replicate-specific means are passed as R "alleles" with a one-hot pi[g, r, :] = e_r:
    e[r, b, g] = sum_a pi[g, r, a] P[b, g, a] = P[b, g, r] -- one `bean_ll` launch, gradients per replicate come back in
    d_mu / d_sd.  sigma = sqrt(sd_targets) (SURVEY App. B4)."""

    def __init__(self, data, device="cuda", dtype=torch.float32, use_bcmatch=True, num_steps=2000, initial_lr=0.01,
                 gamma=0.1, seed=101, sd_scale=0.01, mask_thres=10, prior_params: Optional[dict] = None):
        if not torch.cuda.is_available():
            raise BeanError("CovariateNormalEngine needs a CUDA device: there is no CPU fallback")
        self.device, self.dtype = torch.device(device), dtype
        kw = dict(device=self.device, dtype=dtype)
        use_bcmatch = bool(use_bcmatch) and getattr(data, "X_bcmatch_masked", None) is not None
        self.screen = DeviceScreen(data, self.device, dtype=dtype, use_bcmatch=use_bcmatch, mask_thres=mask_thres)
        self.G, self.R, self.T, self.C = data.n_guides, data.n_reps, int(data.n_targets), int(data.n_sample_covariates)
        self.target_lengths = data.target_lengths.to(self.device)
        self.rep_by_cov = data.rep_by_cov.to(**kw)  # (R, C)
        self.onehot = torch.eye(self.R, **kw).unsqueeze(0).expand(self.G, -1, -1).contiguous()  # pi[g, r, a] = [a == r]
        self.sd_scale, self.prior_params = sd_scale, prior_params
        z = lambda *s: torch.zeros(s, **kw)
        theta = {"mu_loc": z(self.T, 1), "mu_scale": z(self.T, 1), "sd_loc": z(self.T, 1), "sd_scale": z(self.T, 1),
                 "mu_cov_loc": z(self.C), "mu_cov_scale": z(self.C)}
        self._init_optim(theta, {"mu_scale", "sd_scale", "mu_cov_scale"}, num_steps, initial_lr, gamma, seed)

    def elbo_loss(self, noise: Optional[Dict[str, torch.Tensor]] = None):
        T, G, R = self.T, self.G, self.R
        P = self.theta
        mu_loc, sd_loc, cov_loc = P["mu_loc"], P["sd_loc"], P["mu_cov_loc"]
        mu_scale, sd_scale_q, cov_scale = P["mu_scale"].exp(), P["sd_scale"].exp(), P["mu_cov_scale"].exp()
        mu_t = mu_loc + mu_scale * self._draw(noise, "eps_mu", (T, 1))
        sd_t = torch.exp(sd_loc + sd_scale_q * self._draw(noise, "eps_sd", (T, 1)))
        mu_cov = cov_loc + cov_scale * self._draw(noise, "eps_cov", (self.C,))
        guide_lp = (tdist.Normal(mu_loc, mu_scale).log_prob(mu_t).sum() + tdist.LogNormal(sd_loc, sd_scale_q).log_prob(sd_t).sum()
                    + tdist.Normal(cov_loc, cov_scale).log_prob(mu_cov).sum())
        pp = self.prior_params or {}
        mu_prior = (tdist.Normal(self._prior_t(pp.get("mu_loc", 0.0)), self._prior_t(pp.get("mu_scale", 1.0)))
                    if ("mu_loc" in pp or "mu_scale" in pp) else tdist.Laplace(self._c(0.0), self._c(1.0)))
        sd_prior = tdist.LogNormal(self._prior_t(pp.get("sd_loc", 0.0)), self._prior_t(pp.get("sd_scale", self.sd_scale)))
        model_lp = (mu_prior.log_prob(mu_t).sum() + sd_prior.log_prob(sd_t).sum()
                    + tdist.Normal(self._c(0.0), self._c(1.0)).log_prob(mu_cov).sum())
        mu_g = torch.repeat_interleave(mu_t, self.target_lengths, dim=0, output_size=G)  # (G, 1)
        sd_g = torch.repeat_interleave(sd_t, self.target_lengths, dim=0, output_size=G)
        shift = (self.rep_by_cov * mu_cov)[:, 0]  # (R,)
        mu_a = mu_g + shift.unsqueeze(0)  # (G, R): replicate-specific means as "alleles"
        sd_a = torch.sqrt(sd_g).expand(G, R)
        ll = count_log_likelihood(self.screen, mu_a, sd_a, self.onehot, None)
        return -(model_lp + ll - guide_lp)
