"""CPU oracle: plain-torch restatement of the `bean run` SVI ELBO (sorting + survival).

TEST INFRASTRUCTURE ONLY -- never imported by `crispr_bean_b200/` (the product).

What it restates (all `file:line` relative to the original project's root):
  * `get_std_normal_prob`            bean/model/utils.py:34-76
  * `get_alpha`                      bean/model/utils.py:10-31
  * `scale_pi_by_accessibility`      bean/model/utils.py:79-178
  * `DirichletMultinomial.log_prob`  pyro.distributions.conjugate (pyro-ppl>=1.8.5, setup.py:42;
                                     NOT vendored in the reference -> formula restated, SURVEY App. A.3)
  * model/guide pairs                bean/model/model.py:19-962, bean/model/survival_model.py:15-833
  * `Trace_ELBO` (1 particle)        pyro.infer (restated: loss = -(sum model log p - sum guide log q),
                                     poutine.mask == where(mask, log_prob, 0); SURVEY App. A.5)
  * `ClippedAdam`                    pyro.optim.clipped_adam (restated; SURVEY App. A.6)
  * `run_inference`                  bean/model/run.py:347-396

PARITY PIN STATUS: pinned against the reference's own source files executed in the build container
(tests/refharness + tests/golden/make_reference_golden.py -> tests/golden/ref_*.npz, checked by
tests/test_reference_golden.py): every model/guide pair below reproduces the loss, per-parameter gradients and
6-step run_inference trajectories the reference's unmodified model.py / survival_model.py / run.py compute on the
same tensors and the same recorded draws (float64: <= 1e-11 loss, <= 1e-9 gradients).  What is NOT executed but
restated is pyro itself: pyro-ppl is not installable here, so those programs run on tests/refharness/pyro, a
restatement of the primitives they call (param / sample / plate / poutine.mask / Trace_ELBO / ClippedAdam).
Independent known answers (tests/test_oracle_known_answers.py):
  - torch.distributions (Normal, LogNormal, Laplace, Dirichlet, Multinomial) and
    torch._dirichlet_grad are the reference's REAL dependencies and are used directly here;
  - the Dirichlet-Multinomial log-pmf against scipy.stats.dirichlet_multinomial;
  - the Normal-CDF bin probabilities against scipy.stats.norm;
  - closed-form local gradients against torch.autograd in float64 + gradcheck.

Everything is written against the reference's `(R, B, G)` tensors with the reference attribute
names, so `data` may be any object exposing those attributes.
"""
from __future__ import annotations

import math
from types import SimpleNamespace
from typing import Dict, Optional

import torch
import torch.distributions as tdist

EPS = 1e-5
PI_NOISE_SD = 0.655


# ----------------------------------------------------------------------------------------------
# Elementary pieces
# ----------------------------------------------------------------------------------------------
def get_std_normal_prob(upper_quantile, lower_quantile, mu, sd, mask=None):
    """P(bin) = Phi((t_u - mu)/sd) - Phi((t_l - mu)/sd), t = Phi^-1(quantile).

    Restates bean/model/utils.py:34-76.  The reference writes through boolean masks
    (`x[~inf_mask] = ...`); `torch.where` yields the same values.  uq == 1 -> cdf 1, lq == 0 -> cdf 0.
    Dtype promotion follows torch: quantile tensors are float64 in the reference
    (`torch.as_tensor(pandas float64)`, data_class.py:963-964), so the CDF is evaluated in float64
    even when mu/sd are float32.
    """
    inf_mask = upper_quantile == 1.0
    ninf_mask = lower_quantile == 0.0
    std = tdist.Normal(0, 1)
    # icdf(1) = +inf / icdf(0) = -inf are never used: masked entries keep thres 1 / 0 (utils.py:51-54)
    uq_safe = torch.where(inf_mask, torch.full_like(upper_quantile, 0.5), upper_quantile)
    lq_safe = torch.where(ninf_mask, torch.full_like(lower_quantile, 0.5), lower_quantile)
    upper_thres = torch.where(inf_mask, torch.ones_like(upper_quantile), std.icdf(uq_safe))
    lower_thres = torch.where(ninf_mask, torch.zeros_like(lower_quantile), std.icdf(lq_safe))
    if mask is not None:
        sd = sd + (~mask).long() * 100  # utils.py:56-58
    nrm = tdist.Normal(mu, sd, validate_args=False)
    cdf_upper = torch.where(inf_mask, torch.ones_like(upper_quantile), nrm.cdf(upper_thres))
    cdf_lower = torch.where(ninf_mask, torch.zeros_like(lower_quantile), nrm.cdf(lower_thres))
    res = cdf_upper - cdf_lower
    if mask is not None:
        res = torch.where(mask, res, torch.zeros_like(res))  # utils.py:73-74
    return res


def get_alpha(expected_guide_p, size_factor, sample_mask, a0, epsilon=EPS):
    """bean/model/utils.py:10-25 (normalize_by_a0=True branch, the only one the models use)."""
    p = expected_guide_p.permute(0, 2, 1) * size_factor[:, None, :]  # (R, G, B)
    a = (p + epsilon / p.shape[-1]) / (p.sum(axis=-1)[:, :, None] + epsilon) * a0[None, :, None]
    a = (a * sample_mask[:, None, :]).clamp(min=epsilon)
    return a


def dm_log_prob(alpha, value):
    """pyro.distributions.DirichletMultinomial(alpha, validate_args=False).log_prob(value), dense.

    _log_beta_1(a, v) = lgamma(1+v) + lgamma(a) - lgamma(v+a);
    log_prob = _log_beta_1(a.sum(-1), v.sum(-1)) - _log_beta_1(a, v).sum(-1).   (SURVEY App. A.3)
    """

    def _log_beta_1(a, v):
        return torch.lgamma(1 + v) + torch.lgamma(a) - torch.lgamma(v + a)

    return _log_beta_1(alpha.sum(-1), value.sum(-1)) - _log_beta_1(alpha, value).sum(-1)


class InjectedDirichlet(torch.autograd.Function):
    """`Dirichlet(conc).rsample()` with the drawn value fixed from outside.

    forward returns the injected sample; backward is torch's own pathwise derivative
    (torch/distributions/dirichlet.py `_Dirichlet_backward`, built on `torch._dirichlet_grad`),
    i.e. exactly what autograd applies to a real `rsample()` draw in the reference.
    """

    @staticmethod
    def forward(ctx, concentration, x):
        ctx.save_for_backward(x, concentration)
        return x.clone()

    @staticmethod
    def backward(ctx, grad_output):
        x, concentration = ctx.saved_tensors
        total = concentration.sum(-1, True).expand_as(concentration)
        grad = torch._dirichlet_grad(x, concentration, total)
        return grad * (grad_output - (x * grad_output).sum(-1, True)), None


def dirichlet_rsample(concentration, injected=None):
    conc = concentration
    if injected is None:
        return tdist.Dirichlet(conc, validate_args=False).rsample()
    return InjectedDirichlet.apply(conc, injected.to(conc.dtype))


def scale_pi_by_accessibility(pi, guide_accessibility, logit_pi_noise, a=0.2513, b=-1.9458):
    """bean/model/utils.py:79-178 with the `logit_pi_noise` sample passed in (pyro replays it)."""
    scaled_pi = pi[..., 1:] * torch.exp(torch.tensor(b)) * torch.pow(guide_accessibility, a).unsqueeze(-1)
    ctrl_pi = torch.ones(pi[..., 0].shape) - scaled_pi.sum(axis=-1)
    pi = torch.concat([ctrl_pi.unsqueeze(-1), scaled_pi], axis=-1)
    pi = pi / pi.sum(axis=-1).clamp(min=1.0)[..., None]
    # add_noise_to_pi
    n_reps, _, n_guides, n_alleles = pi.shape
    logit_pi = torch.logit(pi[..., 1:].clamp(min=1e-3, max=1 - 1e-3))
    logit_pi = logit_pi + logit_pi_noise.unsqueeze(0).unsqueeze(0).unsqueeze(-1).expand(
        (n_reps, 1, -1, n_alleles - 1)
    )
    exp_pi_noised = torch.exp(logit_pi)
    pi_noised = (exp_pi_noised / (1 + exp_pi_noised)).clamp(min=1e-3, max=1 - 1e-3)
    pi = torch.concat(
        [(torch.ones(pi[:, :, :, 0].shape) - pi_noised.sum(axis=-1)).unsqueeze(-1), pi_noised], axis=-1
    )
    return pi


def _masked_sum(mask, lp):
    """poutine.mask + log_prob_sum: masked-out batch elements contribute exactly 0."""
    return torch.where(mask, lp, torch.zeros_like(lp)).sum()


# ----------------------------------------------------------------------------------------------
# Parameter store (pyro.param semantics: positive-constrained params live as log(value))
# ----------------------------------------------------------------------------------------------
class ParamStore:
    """Minimal pyro param-store: unconstrained leaves + `constraint=positive -> exp`."""

    def __init__(self):
        self.unconstrained: Dict[str, torch.Tensor] = {}
        self.positive: Dict[str, bool] = {}

    def param(self, name, init=None, positive=False):
        if name not in self.unconstrained:
            v = init.detach().clone()
            if positive:
                v = v.log()
            self.unconstrained[name] = v.requires_grad_(True)
            self.positive[name] = positive
        u = self.unconstrained[name]
        return u.exp() if self.positive[name] else u

    def constrained(self):
        return {k: (v.detach().exp() if self.positive[k] else v.detach().clone()) for k, v in self.unconstrained.items()}

    def zero_grad(self):
        for v in self.unconstrained.values():
            v.grad = None


class ClippedAdam:
    """pyro.optim.ClippedAdam restated (SURVEY App. A.6): one state per parameter tensor."""

    def __init__(self, lr=0.01, lrd=1.0, betas=(0.9, 0.999), eps=1e-8, clip_norm=10.0):
        self.lr0, self.lrd, self.betas, self.eps, self.clip = lr, lrd, betas, eps, clip_norm
        self.state = {}

    def step(self, named_params: Dict[str, torch.Tensor]):
        b1, b2 = self.betas
        for name, p in named_params.items():
            if p.grad is None:
                continue
            st = self.state.setdefault(
                name, {"step": 0, "lr": self.lr0, "m": torch.zeros_like(p), "v": torch.zeros_like(p)}
            )
            st["lr"] *= self.lrd
            g = p.grad.detach().clamp(-self.clip, self.clip)
            st["step"] += 1
            st["m"].mul_(b1).add_(g, alpha=1 - b1)
            st["v"].mul_(b2).addcmul_(g, g, value=1 - b2)
            denom = st["v"].sqrt().add_(self.eps)
            step_size = st["lr"] * math.sqrt(1 - b2 ** st["step"]) / (1 - b1 ** st["step"])
            with torch.no_grad():
                p.addcdiv_(st["m"], denom, value=-step_size)


# ----------------------------------------------------------------------------------------------
# Shared likelihood tail: get_alpha + Dirichlet-Multinomial observation sites
# ----------------------------------------------------------------------------------------------
def _count_sites(data, expected_guide_p, use_bcmatch, mask_thres, out):
    """model.py:123-165 / :506-547: `guide_counts` and `guide_bcmatch_counts` DM sites."""
    a = get_alpha(expected_guide_p, data.size_factor, data.sample_mask, data.a0)
    x = data.X_masked.permute(0, 2, 1)
    w = torch.logical_and(x.sum(axis=-1) > mask_thres, data.repguide_mask)
    ll = dm_log_prob(a, x)
    out["ll_guide_counts"] = ll
    out["w_guide_counts"] = w
    total = _masked_sum(w, ll)
    if use_bcmatch:
        a_bc = get_alpha(expected_guide_p, data.size_factor_bcmatch, data.sample_mask, data.a0_bcmatch)
        xb = data.X_bcmatch_masked.permute(0, 2, 1)
        wb = torch.logical_and(xb.sum(axis=-1) > mask_thres, data.repguide_mask)
        llb = dm_log_prob(a_bc, xb)
        out["ll_guide_bcmatch_counts"] = llb
        out["w_guide_bcmatch_counts"] = wb
        total = total + _masked_sum(wb, llb)
    return total


def _mu_sd_priors(shape, sd_scale, prior_params):
    """model.py:41-57 / :405-421 / :579-603: prior on mu (Laplace or user Normal) and LogNormal on sd."""
    sd_loc0 = torch.zeros(shape)
    sd_scale0 = torch.ones(shape) * sd_scale
    mu_dist = tdist.Laplace(0.0, 1.0)
    if prior_params is not None:
        sd_loc0 = prior_params.get("sd_loc", sd_loc0)
        sd_scale0 = prior_params.get("sd_scale", sd_scale0)
        if "mu_loc" in prior_params or "mu_scale" in prior_params:
            mu_dist = tdist.Normal(prior_params.get("mu_loc", 0.0), prior_params.get("mu_scale", 1.0))
    return mu_dist, tdist.LogNormal(sd_loc0, sd_scale0)


def _draw(noise, key, shape):
    if noise is not None and key in noise:
        return noise[key]
    return torch.randn(shape)


# ----------------------------------------------------------------------------------------------
# Sorting models: -ELBO for one particle.  `noise=None` draws fresh noise from torch's RNG.
# ----------------------------------------------------------------------------------------------
def elbo_normal(data, ps: ParamStore, noise=None, mask_thres=10, use_bcmatch=True, sd_scale=0.01,
                prior_params=None):
    """NormalModel / NormalGuide (model.py:19-165, :754-782).  A=1, sd = sqrt(sd_targets)."""
    T, G = data.n_targets, data.n_guides
    out = {}
    mu_loc = ps.param("mu_loc", torch.zeros((T, 1)))
    mu_scale = ps.param("mu_scale", torch.ones((T, 1)), positive=True)
    sd_loc = ps.param("sd_loc", torch.zeros((T, 1)))
    sd_scale_q = ps.param("sd_scale", torch.ones((T, 1)), positive=True)
    mu_t = mu_loc + mu_scale * _draw(noise, "eps_mu", (T, 1))
    sd_t = torch.exp(sd_loc + sd_scale_q * _draw(noise, "eps_sd", (T, 1)))
    guide_lp = tdist.Normal(mu_loc, mu_scale).log_prob(mu_t).sum() + tdist.LogNormal(sd_loc, sd_scale_q).log_prob(sd_t).sum()

    mu_dist, sd_dist = _mu_sd_priors((T, 1), sd_scale, prior_params)
    model_lp = mu_dist.log_prob(mu_t).sum() + sd_dist.log_prob(sd_t).sum()
    mu = torch.repeat_interleave(mu_t, data.target_lengths, dim=0)
    sd = torch.repeat_interleave(sd_t, data.target_lengths, dim=0)
    R, B = data.n_reps, data.n_condits
    uq = data.upper_bounds.unsqueeze(0).unsqueeze(-1).unsqueeze(-1).expand((R, -1, G, 1))
    lq = data.lower_bounds.unsqueeze(0).unsqueeze(-1).unsqueeze(-1).expand((R, -1, G, 1))
    mu4 = mu.unsqueeze(0).unsqueeze(0).expand((R, B, -1, -1))
    if hasattr(data, "sample_covariates"):
        # model.py:73-91 / guide :771-782: mu_cov ~ Normal(mu_cov_loc, mu_cov_scale) vs prior Normal(0, 1); only the FIRST
        # column of rep_by_cov * mu_cov shifts the replicate's mean (`[:, 0]`, as the reference does)
        C = data.n_sample_covariates
        cov_loc = ps.param("mu_cov_loc", torch.zeros((C,)))
        cov_scale = ps.param("mu_cov_scale", torch.ones((C,)), positive=True)
        mu_cov = cov_loc + cov_scale * _draw(noise, "eps_cov", (C,))
        guide_lp = guide_lp + tdist.Normal(cov_loc, cov_scale).log_prob(mu_cov).sum()
        model_lp = model_lp + tdist.Normal(0.0, 1.0).log_prob(mu_cov).sum()
        mu4 = mu4 + (data.rep_by_cov * mu_cov)[:, 0].unsqueeze(-1).unsqueeze(-1).unsqueeze(-1).expand((-1, B, G, 1))
    sd4 = torch.sqrt(sd.unsqueeze(0).unsqueeze(0).expand((R, B, -1, -1)))  # model.py:92-98
    alleles_p_bin = get_std_normal_prob(uq, lq, mu4, sd4)
    expected_guide_p = alleles_p_bin.sum(axis=-1)
    model_lp = model_lp + _count_sites(data, expected_guide_p, use_bcmatch, mask_thres, out)
    out["model_lp"], out["guide_lp"] = model_lp, guide_lp
    return -(model_lp - guide_lp), out


def elbo_control_normal(data, ps: ParamStore, noise=None, mask_thres=10, use_bcmatch=True):
    """ControlNormalModel / ControlNormalGuide (model.py:168-252, :861-875): one global (mu, sd)."""
    G = data.n_guides
    out = {}
    mu_loc = ps.param("mu_loc", torch.tensor(0.0))
    mu_scale = ps.param("mu_scale", torch.tensor(1.0), positive=True)
    sd_loc = ps.param("sd_loc", torch.tensor(0.0))
    sd_scale_q = ps.param("sd_scale", torch.tensor(1.0), positive=True)
    mu_t = mu_loc + mu_scale * _draw(noise, "eps_mu", ())
    sd_t = torch.exp(sd_loc + sd_scale_q * _draw(noise, "eps_sd", ()))
    guide_lp = tdist.Normal(mu_loc, mu_scale).log_prob(mu_t).sum() + tdist.LogNormal(sd_loc, sd_scale_q).log_prob(sd_t).sum()
    model_lp = tdist.Laplace(0.0, 1.0).log_prob(mu_t).sum() + tdist.LogNormal(0.0, 1.0).log_prob(sd_t).sum()
    mu = mu_t.repeat(G).unsqueeze(-1)
    sd = sd_t.repeat(G).unsqueeze(-1)
    B = data.n_condits
    uq = data.upper_bounds.unsqueeze(-1).unsqueeze(-1).expand((-1, G, 1))
    lq = data.lower_bounds.unsqueeze(-1).unsqueeze(-1).expand((-1, G, 1))
    alleles_p_bin = get_std_normal_prob(uq, lq, mu.unsqueeze(0).expand((B, -1, -1)), sd.unsqueeze(0).expand((B, -1, -1)))
    expected_guide_p = alleles_p_bin.unsqueeze(0).expand(data.n_reps, -1, -1, -1).sum(axis=-1)
    model_lp = model_lp + _count_sites(data, expected_guide_p, use_bcmatch, mask_thres, out)
    out["model_lp"], out["guide_lp"] = model_lp, guide_lp
    return -(model_lp - guide_lp), out


def _pi_sites(data, pi_a_scaled_model, conc_guide, guide_pi_masked, noise, out, allele_counts):
    """`pi` (Dirichlet) + control allele-count (Multinomial) sites.

    model.py:454-474 (model: both masked by repguide_mask), :837-847 (guide: unmasked, clamped) and
    :942-950 (tiling guide: masked, not clamped).
    """
    R, G = data.n_reps, data.n_guides
    rg_mask = data.repguide_mask.unsqueeze(1)  # (R, 1, G)
    conc_g = conc_guide.unsqueeze(0).unsqueeze(0).expand(R, 1, -1, -1)
    injected = noise.get("pi") if noise is not None else None
    pi = dirichlet_rsample(conc_g, injected)
    lq = tdist.Dirichlet(conc_g, validate_args=False).log_prob(pi)
    guide_lp = _masked_sum(rg_mask, lq) if guide_pi_masked else lq.sum()
    conc_m = pi_a_scaled_model.unsqueeze(0).unsqueeze(0).expand(R, 1, -1, -1)
    lp_pi = tdist.Dirichlet(conc_m, validate_args=False).log_prob(pi)
    lp_mult = tdist.Multinomial(probs=pi, validate_args=False).log_prob(allele_counts)
    out["lp_pi_model"], out["lp_bulk_allele"], out["lq_pi_guide"] = lp_pi, lp_mult, lq
    mult_mask = rg_mask if lp_mult.shape[1] == 1 else rg_mask.expand(lp_mult.shape)
    model_lp = _masked_sum(rg_mask, lp_pi) + _masked_sum(mult_mask, lp_mult)
    return pi, model_lp, guide_lp


def _noise_sites(data, ps, noise, fit_noise_guide):
    """`logit_pi_noise` site: guide Normal(noise_loc, noise_scale) when fit_noise else the prior;
    model always the prior Normal(0, 0.655) (utils.py:145-161; model never gets fit_noise, SURVEY B3)."""
    G = data.n_guides
    eps = _draw(noise, "eps_noise", (G,))
    prior = tdist.Normal(torch.tensor(0.0), torch.tensor(PI_NOISE_SD))
    if fit_noise_guide:
        noise_loc = ps.param("noise_loc", torch.zeros((G,)))
        noise_scale = ps.param("noise_scale", torch.ones((G,)) * PI_NOISE_SD, positive=True)
        val = noise_loc + noise_scale * eps
        guide_lp = tdist.Normal(noise_loc, noise_scale).log_prob(val).sum()
    else:
        val = PI_NOISE_SD * eps
        guide_lp = prior.log_prob(val).sum()
    model_lp = prior.log_prob(val).sum()
    return val, model_lp, guide_lp


def elbo_mixture_normal(data, ps: ParamStore, noise=None, alpha_prior=1.0, use_bcmatch=True, sd_scale=0.01,
                        scale_by_accessibility=False, fit_noise=False, prior_params=None):
    """MixtureNormalModel / MixtureNormalGuide (model.py:378-547, :785-858).  A = 2 (WT, edited)."""
    T, G = data.n_targets, data.n_guides
    out = {}
    mu_loc = ps.param("mu_loc", torch.zeros((T, 1)))
    mu_scale = ps.param("mu_scale", torch.ones((T, 1)), positive=True)
    sd_loc = ps.param("sd_loc", torch.zeros((T, 1)))
    sd_scale_q = ps.param("sd_scale", torch.ones((T, 1)), positive=True)
    alpha_pi = ps.param("alpha_pi", torch.ones((G, 2)) * alpha_prior, positive=True)
    mu_t = mu_loc + mu_scale * _draw(noise, "eps_mu", (T, 1))
    sd_t = torch.exp(sd_loc + sd_scale_q * _draw(noise, "eps_sd", (T, 1)))
    guide_lp = tdist.Normal(mu_loc, mu_scale).log_prob(mu_t).sum() + tdist.LogNormal(sd_loc, sd_scale_q).log_prob(sd_t).sum()
    mu_dist, sd_dist = _mu_sd_priors((T, 1), sd_scale, prior_params)
    model_lp = mu_dist.log_prob(mu_t).sum() + sd_dist.log_prob(sd_t).sum()

    pi_a_scaled = alpha_pi / alpha_pi.sum(axis=-1)[:, None] * data.pi_a0[:, None]
    pi, m_lp, g_lp = _pi_sites(data, pi_a_scaled, pi_a_scaled.clamp(1e-5), False, noise, out,
                               data.allele_counts_control)
    model_lp, guide_lp = model_lp + m_lp, guide_lp + g_lp
    if scale_by_accessibility:
        val, m_lp, g_lp = _noise_sites(data, ps, noise, fit_noise)
        model_lp, guide_lp = model_lp + m_lp, guide_lp + g_lp
        pi = scale_pi_by_accessibility(pi, data.guide_accessibility, val)

    mu_center = torch.cat([torch.zeros((T, 1)), mu_t], axis=-1)
    mu = torch.repeat_interleave(mu_center, data.target_lengths, dim=0)
    sd = torch.repeat_interleave(torch.cat([torch.ones((T, 1)), sd_t], axis=-1), data.target_lengths, dim=0)
    B = data.n_condits
    uq = data.upper_bounds.unsqueeze(-1).unsqueeze(-1).expand((-1, G, 2))
    lq = data.lower_bounds.unsqueeze(-1).unsqueeze(-1).expand((-1, G, 2))
    alleles_p_bin = get_std_normal_prob(uq, lq, mu.unsqueeze(0).expand((B, -1, -1)), sd.unsqueeze(0).expand((B, -1, -1)))
    expected_allele_p = pi.expand(data.n_reps, B, -1, -1) * alleles_p_bin[None, :, :, :]
    expected_guide_p = expected_allele_p.sum(axis=-1)
    out["pi_used"], out["alleles_p_bin"] = pi, alleles_p_bin
    # model.py:526-547 hard-codes the threshold 10
    model_lp = model_lp + _count_sites(data, expected_guide_p, use_bcmatch, 10, out)
    out["model_lp"], out["guide_lp"] = model_lp, guide_lp
    return -(model_lp - guide_lp), out


def elbo_multi_mixture_normal(data, ps: ParamStore, noise=None, alpha_prior=1.0, use_bcmatch=True, sd_scale=0.01,
                              scale_by_accessibility=False, fit_noise=True, prior_params=None, epsilon=EPS):
    """MultiMixtureNormalModel / Guide (model.py:550-751, :878-962): tiling screens, A = n_max_alleles."""
    E, G, A = data.n_edits, data.n_guides, data.n_max_alleles
    out = {}
    mu_loc = ps.param("mu_loc", torch.zeros((E,)))
    mu_scale = ps.param("mu_scale", torch.ones((E,)), positive=True)
    sd_loc = ps.param("sd_loc", torch.zeros((E,)))
    sd_scale_q = ps.param("sd_scale", torch.ones((E,)), positive=True)
    alpha_pi0 = torch.ones((G, A)) * alpha_prior
    alpha_pi0[~data.allele_mask] = epsilon
    alpha_pi = ps.param("alpha_pi", alpha_pi0, positive=True)
    # model.py:645 / :937 overwrite the constrained view in place -> no gradient to masked entries
    alpha_pi = torch.where(data.allele_mask, alpha_pi, torch.full_like(alpha_pi, epsilon))
    mu_e = mu_loc + mu_scale * _draw(noise, "eps_mu", (E,))
    sd_e = torch.exp(sd_loc + sd_scale_q * _draw(noise, "eps_sd", (E,)))
    guide_lp = tdist.Normal(mu_loc, mu_scale).log_prob(mu_e).sum() + tdist.LogNormal(sd_loc, sd_scale_q).log_prob(sd_e).sum()
    mu_dist, sd_dist = _mu_sd_priors((E,), sd_scale, prior_params)
    model_lp = mu_dist.log_prob(mu_e).sum() + sd_dist.log_prob(sd_e).sum()

    mu_targets = torch.matmul(data.allele_to_edit, mu_e)
    sd_targets = torch.linalg.norm(data.allele_to_edit * sd_e[None, None, :], dim=-1)
    mu = torch.cat([torch.zeros((G, 1)), mu_targets], axis=-1)
    sd = torch.cat([torch.ones((G, 1)), sd_targets], axis=-1)

    pi_a_scaled_guide = alpha_pi / alpha_pi.sum(axis=-1)[:, None] * data.pi_a0[:, None]  # :938, no clamp
    pi_a_scaled = (alpha_pi + epsilon / A) / (alpha_pi.sum(axis=-1)[:, None] + epsilon) * data.pi_a0[:, None]
    pi_a_scaled = torch.where(pi_a_scaled < epsilon, torch.full_like(pi_a_scaled, epsilon), pi_a_scaled)  # :651
    pi, m_lp, g_lp = _pi_sites(data, pi_a_scaled, pi_a_scaled_guide, True, noise, out, data.allele_counts_control)
    model_lp, guide_lp = model_lp + m_lp, guide_lp + g_lp
    if scale_by_accessibility:
        val, m_lp, g_lp = _noise_sites(data, ps, noise, fit_noise)
        model_lp, guide_lp = model_lp + m_lp, guide_lp + g_lp
        pi = scale_pi_by_accessibility(pi, data.guide_accessibility, val)

    B = data.n_condits
    uq = data.upper_bounds.unsqueeze(-1).unsqueeze(-1).expand((-1, G, A))
    lq = data.lower_bounds.unsqueeze(-1).unsqueeze(-1).expand((-1, G, A))
    alleles_p_bin = get_std_normal_prob(
        uq, lq, mu.unsqueeze(0).expand((B, -1, -1)), sd.unsqueeze(0).expand((B, -1, -1)),
        mask=data.allele_mask.unsqueeze(0).expand((B, -1, -1)),
    )
    expected_guide_p = (pi.expand(data.n_reps, B, -1, -1) * alleles_p_bin[None, :, :, :]).sum(axis=-1)
    out["pi_used"], out["alleles_p_bin"] = pi, alleles_p_bin
    model_lp = model_lp + _count_sites(data, expected_guide_p, use_bcmatch, 10, out)
    out["model_lp"], out["guide_lp"] = model_lp, guide_lp
    return -(model_lp - guide_lp), out


SORTING_ELBOS = {
    "Normal": elbo_normal,
    "ControlNormal": elbo_control_normal,
    "MixtureNormal": elbo_mixture_normal,
    "MultiMixtureNormal": elbo_multi_mixture_normal,
}


# ----------------------------------------------------------------------------------------------
# The likelihood core alone (the autograd.Function seam of the product): P -> e -> alpha -> DM
# ----------------------------------------------------------------------------------------------
def sorting_ll_core(data, mu_alleles, sd_alleles, pi, use_bcmatch=True, mask_thres=10, allele_mask=None):
    """log-likelihood of both count layers given per-guide allele (mu, sd) `(G, A)` and `pi (R,1,G,A)`.

    Same op chain as model.py:484-547; returns (masked total, per-row ll dict)."""
    G, A = mu_alleles.shape
    B = data.n_condits
    out = {}
    uq = data.upper_bounds.unsqueeze(-1).unsqueeze(-1).expand((-1, G, A))
    lq = data.lower_bounds.unsqueeze(-1).unsqueeze(-1).expand((-1, G, A))
    m = None if allele_mask is None else allele_mask.unsqueeze(0).expand((B, -1, -1))
    P = get_std_normal_prob(uq, lq, mu_alleles.unsqueeze(0).expand((B, -1, -1)),
                            sd_alleles.unsqueeze(0).expand((B, -1, -1)), mask=m)
    e = (pi.expand(data.n_reps, B, -1, -1) * P[None]).sum(axis=-1)
    total = _count_sites(data, e, use_bcmatch, mask_thres, out)
    out["alleles_p_bin"] = P
    return total, out


def survival_ll_core(data, mu_alleles, pi, use_bcmatch=True, mask_thres=10, allele_mask=None):
    """Survival counterpart of `sorting_ll_core`: exp(mu * t) replaces the Normal-CDF bin masses
    (bean/model/survival_model.py:352-424; masked alleles are multiplied by 0, :566-567)."""
    G, A = mu_alleles.shape
    B = data.n_condits
    out = {}
    time = data.timepoints
    P = torch.exp(mu_alleles.unsqueeze(0).expand((B, -1, -1)) * time.unsqueeze(-1).unsqueeze(-1).expand((-1, G, 1)))
    if allele_mask is not None:
        P = P * allele_mask.unsqueeze(0)
    e = (pi.expand(data.n_reps, B, -1, -1) * P[None]).sum(axis=-1)
    total = _count_sites(data, e, use_bcmatch, mask_thres, out)
    out["alleles_p_time"] = P
    return total, out


# ----------------------------------------------------------------------------------------------
# run_inference restated (bean/model/run.py:347-396)
# ----------------------------------------------------------------------------------------------
def run_inference(elbo_fn, data, initial_lr=0.01, gamma=0.1, num_steps=2000, noise_fn=None, **model_kwargs):
    """SVI loop: one-particle Trace_ELBO + ClippedAdam(lr, lrd = gamma ** (1/num_steps)).

    `noise_fn(t)` may inject the step's reparameterisation noise (parity runs); None = torch RNG.
    Returns (ParamStore, {"loss": [...], "params": {...}}) like the reference.
    """
    ps = ParamStore()
    opt = ClippedAdam(lr=initial_lr, lrd=gamma ** (1 / num_steps))
    losses = []
    for t in range(num_steps):
        noise = noise_fn(t) if noise_fn is not None else None
        loss, _ = elbo_fn(data, ps, noise=noise, **model_kwargs)
        ps.zero_grad()
        loss.backward()
        opt.step(ps.unconstrained)
        losses.append(float(loss.detach()))
    return ps, {"loss": losses, "params": {k: v.cpu() for k, v in ps.constrained().items()}}


def as_namespace(**kw):
    return SimpleNamespace(**kw)


# ----------------------------------------------------------------------------------------------
# Survival models (bean/model/survival_model.py).  exp(mu * t) replaces the Normal-CDF bin masses; the
# quirks of SURVEY App. B8 are reproduced: the guide samples `initial_abundance` although the model observes
# it, `q0` is the guide's (G,) parameter, `mu_negctrl` is a model-only latent drawn from its prior.
# ----------------------------------------------------------------------------------------------
def _survival_p(mu_alleles, timepoints):
    B = timepoints.shape[0]
    G = mu_alleles.shape[0]
    return torch.exp(mu_alleles.unsqueeze(0).expand((B, -1, -1)) * timepoints.unsqueeze(-1).unsqueeze(-1).expand((-1, G, 1)))


def elbo_survival_normal(data, ps: ParamStore, noise=None, mask_thres=10, use_bcmatch=True, prior_params=None):
    """survival NormalModel / NormalGuide (survival_model.py:15-130, :629-650): A = 1, e = exp(mu t) q_0[r, g]."""
    T, G, R = data.n_targets, data.n_guides, data.n_reps
    out = {}
    init_ab = ps.param("initial_abundance", torch.ones(G) / G, positive=True)
    mu_loc = ps.param("mu_loc", torch.zeros((T, 1)))
    mu_scale = ps.param("mu_scale", torch.ones((T, 1)), positive=True)
    conc_q = init_ab.unsqueeze(0).expand(R, -1)
    q_0 = dirichlet_rsample(conc_q, noise.get("q0") if noise is not None else None)
    mu_t = mu_loc + mu_scale * _draw(noise, "eps_mu", (T, 1))
    guide_lp = tdist.Dirichlet(conc_q, validate_args=False).log_prob(q_0).sum() + tdist.Normal(mu_loc, mu_scale).log_prob(mu_t).sum()
    mu_dist = tdist.Laplace(0.0, 1.0)
    prior_ab = torch.ones(G) / G
    if prior_params is not None:
        if "mu_loc" in prior_params or "mu_scale" in prior_params:
            mu_dist = tdist.Normal(prior_params.get("mu_loc", 0.0), prior_params.get("mu_scale", 1.0))
        prior_ab = prior_params.get("initial_abundance", prior_ab)
    model_lp = mu_dist.log_prob(mu_t).sum()
    mu = torch.repeat_interleave(mu_t, data.target_lengths, dim=0)
    if hasattr(data, "negctrl_guide_idx"):  # survival_model.py:59-60 (None indexes EVERY guide, as in the reference)
        keep = torch.ones((G, 1))
        if data.negctrl_guide_idx is None:
            keep = torch.zeros((G, 1))
        else:
            keep[torch.as_tensor(data.negctrl_guide_idx).long()] = 0.0
        mu = mu * keep
    model_lp = model_lp + tdist.Dirichlet(prior_ab.unsqueeze(0).expand(R, -1), validate_args=False).log_prob(q_0).sum()
    P = _survival_p(mu, data.timepoints)  # (B, G, 1)
    e = (P.unsqueeze(0).expand(R, -1, -1, -1) * q_0.unsqueeze(1).unsqueeze(-1)).sum(axis=-1)
    model_lp = model_lp + _count_sites(data, e, use_bcmatch, mask_thres, out)
    out["model_lp"], out["guide_lp"] = model_lp, guide_lp
    return -(model_lp - guide_lp), out


def elbo_survival_control_normal(data, ps: ParamStore, noise=None, mask_thres=10, use_bcmatch=True):
    """survival ControlNormalModel / Guide (survival_model.py:133-213, :742-757): one shared growth rate."""
    G = data.n_guides
    out = {}
    mu_loc = ps.param("mu_loc", torch.tensor(0.0))
    mu_scale = ps.param("mu_scale", torch.tensor(1.0), positive=True)
    mu_t = mu_loc + mu_scale * _draw(noise, "eps_mu", ())
    guide_lp = tdist.Normal(mu_loc, mu_scale).log_prob(mu_t).sum()
    model_lp = tdist.Normal(0.0, 1.0).log_prob(mu_t).sum()
    mu = mu_t.repeat(G)
    B = data.n_condits
    P = torch.exp(mu.unsqueeze(0).expand((B, -1)) * data.timepoints.unsqueeze(-1).expand((-1, G)))
    e = P.unsqueeze(0).expand(data.n_reps, -1, -1)
    model_lp = model_lp + _count_sites(data, e, use_bcmatch, mask_thres, out)
    out["model_lp"], out["guide_lp"] = model_lp, guide_lp
    return -(model_lp - guide_lp), out


def elbo_survival_mixture_normal(data, ps: ParamStore, noise=None, alpha_prior=1.0, use_bcmatch=True, mask_thres=10,
                                 prior_params=None, mu_negctrl=(0.0, 0.1), scale_by_accessibility=False, fit_noise=False):
    """survival MixtureNormalModel / Guide (survival_model.py:215-424, :651-739)."""
    T, G, R = data.n_targets, data.n_guides, data.n_reps
    out = {}
    q0 = ps.param("q0", torch.ones(G) / G, positive=True)
    mu_loc = ps.param("mu_loc", torch.zeros((T, 1)))
    mu_scale = ps.param("mu_scale", torch.ones((T, 1)), positive=True)
    alpha_pi = ps.param("alpha_pi", torch.ones((G, 2)) * alpha_prior, positive=True)
    conc_q = q0.unsqueeze(0).expand(R, -1)
    ia_sample = dirichlet_rsample(conc_q, noise.get("q0") if noise is not None else None)  # guide-only draw (App. B8)
    mu_t = mu_loc + mu_scale * _draw(noise, "eps_mu", (T, 1))
    guide_lp = tdist.Dirichlet(conc_q, validate_args=False).log_prob(ia_sample).sum() + tdist.Normal(mu_loc, mu_scale).log_prob(mu_t).sum()
    mu_dist = tdist.Laplace(0.0, 1.0)
    if prior_params is not None and ("mu_loc" in prior_params or "mu_scale" in prior_params):
        mu_dist = tdist.Normal(prior_params.get("mu_loc", 0.0), prior_params.get("mu_scale", 1.0))
    model_lp = mu_dist.log_prob(mu_t).sum()
    u = mu_negctrl[0] + mu_negctrl[1] * _draw(noise, "eps_negctrl", (G,))  # model-only latent, prior draw
    model_lp = model_lp + tdist.Normal(mu_negctrl[0], mu_negctrl[1]).log_prob(u).sum()
    mu_edit = torch.repeat_interleave(mu_t, data.target_lengths, dim=0)
    mu = torch.cat([u.unsqueeze(-1), mu_edit + u.unsqueeze(-1)], axis=-1)
    obs_ab = (data.X[:, 0, :] + 1) / (data.X[:, 0, :] + 1).sum(-1, keepdims=True)
    model_lp = model_lp + tdist.Dirichlet(conc_q, validate_args=False).log_prob(obs_ab).sum()
    pi_a_scaled = alpha_pi / alpha_pi.sum(axis=-1)[:, None] * data.pi_a0[:, None]
    rg_mask = data.repguide_mask.unsqueeze(1)
    conc_g = pi_a_scaled.clamp(1e-5).unsqueeze(0).unsqueeze(0).expand(R, 1, -1, -1)
    pi = dirichlet_rsample(conc_g, noise.get("pi") if noise is not None else None)
    guide_lp = guide_lp + tdist.Dirichlet(conc_g, validate_args=False).log_prob(pi).sum()
    conc_m = pi_a_scaled.unsqueeze(0).unsqueeze(0).expand(R, 1, -1, -1)
    model_lp = model_lp + _masked_sum(rg_mask, tdist.Dirichlet(conc_m, validate_args=False).log_prob(pi))
    tc = data.control_timepoint
    C = tc.shape[0]
    expanded = pi.expand(-1, C, -1, -1) * torch.exp(
        mu.unsqueeze(0).unsqueeze(0).expand(R, C, -1, -1) * tc.unsqueeze(0).unsqueeze(-1).unsqueeze(-1).expand(R, -1, G, 2))
    lp_mult = tdist.Multinomial(probs=expanded, validate_args=False).log_prob(data.allele_counts_control)
    model_lp = model_lp + _masked_sum(rg_mask.expand(lp_mult.shape), lp_mult)
    if scale_by_accessibility:  # survival_model.py:347-351
        val, m_lp, g_lp = _noise_sites(data, ps, noise, fit_noise)
        model_lp, guide_lp = model_lp + m_lp, guide_lp + g_lp
        pi = scale_pi_by_accessibility(pi, data.guide_accessibility, val)
    P = _survival_p(mu, data.timepoints)  # (B, G, 2)
    e = (pi.expand(-1, data.n_condits, -1, -1) * P[None]).sum(axis=-1)
    model_lp = model_lp + _count_sites(data, e, use_bcmatch, mask_thres, out)
    out["model_lp"], out["guide_lp"] = model_lp, guide_lp
    return -(model_lp - guide_lp), out


def elbo_survival_multi_mixture_normal(data, ps: ParamStore, noise=None, alpha_prior=1.0, use_bcmatch=True, prior_params=None,
                                       epsilon=EPS, mu_negctrl=(0.0, 0.1), scale_by_accessibility=False, fit_noise=False):
    """survival MultiMixtureNormalModel / Guide (survival_model.py:427-626, :759-833): tiling proliferation screens.

    Guide: mu_targets (E,), pi ~ Dirichlet(clamp(alpha/sum * pi_a0, 1e-5)) masked by repguide_mask; its
    `initial_abundance` parameter is declared but unused.  Model: mu_negctrl (G,) model-only latent; pi concentration
    epsilon-regularised as in the sorting tiling model; control allele counts ~ Multinomial(pi exp(mu t_control))."""
    E, G, A, R = data.n_edits, data.n_guides, data.n_max_alleles, data.n_reps
    out = {}
    ps.param("initial_abundance", torch.ones(G) / G, positive=True)  # declared by the guide, never used (no gradient)
    mu_loc = ps.param("mu_loc", torch.zeros((E,)))
    mu_scale = ps.param("mu_scale", torch.ones((E,)), positive=True)
    alpha_pi0 = torch.ones((G, A)) * alpha_prior
    alpha_pi0[~data.allele_mask] = epsilon
    alpha_pi = ps.param("alpha_pi", alpha_pi0, positive=True)
    alpha_pi = torch.where(data.allele_mask, alpha_pi, torch.full_like(alpha_pi, epsilon))
    mu_e = mu_loc + mu_scale * _draw(noise, "eps_mu", (E,))
    guide_lp = tdist.Normal(mu_loc, mu_scale).log_prob(mu_e).sum()
    mu_dist = tdist.Laplace(0.0, 1.0)
    if prior_params is not None and ("mu_loc" in prior_params or "mu_scale" in prior_params):
        mu_dist = tdist.Normal(prior_params.get("mu_loc", 0.0), prior_params.get("mu_scale", 1.0))
    model_lp = mu_dist.log_prob(mu_e).sum()
    mu_targets = torch.matmul(data.allele_to_edit, mu_e)  # (G, A-1)
    u = mu_negctrl[0] + mu_negctrl[1] * _draw(noise, "eps_negctrl", (G,))
    model_lp = model_lp + tdist.Normal(mu_negctrl[0], mu_negctrl[1]).log_prob(u).sum()
    mu = torch.cat([u.unsqueeze(-1), u.unsqueeze(-1) + mu_targets], axis=1)  # (G, A)
    conc_guide = (alpha_pi / alpha_pi.sum(axis=-1)[:, None] * data.pi_a0[:, None]).clamp(1e-5)
    pi_a_scaled = (alpha_pi + epsilon / A) / (alpha_pi.sum(axis=-1)[:, None] + epsilon) * data.pi_a0[:, None]
    pi_a_scaled = torch.where(pi_a_scaled < epsilon, torch.full_like(pi_a_scaled, epsilon), pi_a_scaled)
    rg_mask = data.repguide_mask.unsqueeze(1)
    conc_g = conc_guide.unsqueeze(0).unsqueeze(0).expand(R, 1, -1, -1)
    pi = dirichlet_rsample(conc_g, noise.get("pi") if noise is not None else None)
    guide_lp = guide_lp + _masked_sum(rg_mask, tdist.Dirichlet(conc_g, validate_args=False).log_prob(pi))
    conc_m = pi_a_scaled.unsqueeze(0).unsqueeze(0).expand(R, 1, -1, -1)
    model_lp = model_lp + _masked_sum(rg_mask, tdist.Dirichlet(conc_m, validate_args=False).log_prob(pi))
    tc = data.control_timepoint
    C = tc.shape[0]
    expanded = pi * torch.exp(mu.unsqueeze(0).unsqueeze(0).expand(R, C, -1, -1)
                              * tc.unsqueeze(0).unsqueeze(-1).unsqueeze(-1).expand(R, -1, G, A))
    lp_mult = tdist.Multinomial(probs=expanded, validate_args=False).log_prob(data.allele_counts_control)
    model_lp = model_lp + _masked_sum(rg_mask.expand(lp_mult.shape), lp_mult)
    if scale_by_accessibility:
        val, m_lp, g_lp = _noise_sites(data, ps, noise, fit_noise)
        model_lp, guide_lp = model_lp + m_lp, guide_lp + g_lp
        pi = scale_pi_by_accessibility(pi, data.guide_accessibility, val)
    B = data.n_condits
    P = torch.exp(data.timepoints.unsqueeze(-1).unsqueeze(-1).expand((-1, G, 1)) * mu.unsqueeze(0).expand((B, -1, -1)))
    P = P * data.allele_mask.unsqueeze(0).expand((B, -1, -1))  # survival_model.py:566-567
    e = (pi.expand(R, B, -1, -1) * P[None]).sum(axis=-1)
    model_lp = model_lp + _count_sites(data, e, use_bcmatch, 10, out)
    out["model_lp"], out["guide_lp"] = model_lp, guide_lp
    return -(model_lp - guide_lp), out


SURVIVAL_ELBOS = {
    "Normal": elbo_survival_normal,
    "ControlNormal": elbo_survival_control_normal,
    "MixtureNormal": elbo_survival_mixture_normal,
    "MultiMixtureNormal": elbo_survival_multi_mixture_normal,
}
