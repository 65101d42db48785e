"""Parity of the fused SVI step (`bean_svi_run_*`) against the CPU oracle's ELBO / autograd / ClippedAdam.

Noise is either injected identically into both sides, or drawn by the kernels (Philox) and replayed
into the oracle, so the comparison is deterministic.  Tolerances: 1e-9 (fp64) / 1e-5 (fp32) relative
for the loss and the (mu, sd) gradients (north_star); the alpha_pi gradient goes through
torch._dirichlet_grad, itself a ~1e-4-accurate approximation evaluated in float on the fp32 path, so
its fp32 tolerance is 2e-4 relative to the gradient's scale (stated here, tight in fp64).
"""
import math

import numpy as np

import pytest
import torch

from crispr_bean_b200.svi import SviEngine, VAR_PARAM_NAMES
from oracle import bean_oracle as O
from tests import helpers as H

pytestmark = pytest.mark.gpu


def rel_err(got, ref):
    got, ref = got.detach().double().cpu().reshape(-1), ref.detach().double().cpu().reshape(-1)
    return ((got - ref).abs() / (ref.abs() + ref.abs().mean() + 1e-300)).max().item()


def oracle_at(model, data, noise, unconstrained=None, **kw):
    """Oracle loss/grads, optionally at given unconstrained parameter values."""
    with H.default_dtype(torch.float64):
        d = H.cast_data(data, torch.float64)
        n = {k: v.double() for k, v in noise.items()}
        ps = O.ParamStore()
        fn = O.SORTING_ELBOS[model]
        if unconstrained is not None:
            fn(d, ps, noise=n, **kw)  # creates the parameters
            for k, v in unconstrained.items():
                ps.unconstrained[k].data.copy_(v.double().reshape(ps.unconstrained[k].shape))
        loss, aux = fn(d, ps, noise=n, **kw)
        ps.zero_grad()
        loss.backward()
    return float(loss.detach()), {k: v.grad.clone() for k, v in ps.unconstrained.items()}


def check_grads(model, data, cuda_device, dtype, tol, tol_alpha, perturb_seed=None, use_bcmatch=True, oracle_kw=None):
    oracle_kw = dict(oracle_kw or {})
    noise = H.fixed_noise(model, data, seed=21)
    eng = SviEngine(data, model, cuda_device, dtype=dtype, use_bcmatch=use_bcmatch, num_steps=10,
                    scale_by_accessibility=oracle_kw.get("scale_by_accessibility", False),
                    fit_noise=oracle_kw.get("fit_noise", False))
    unconstrained = None
    if perturb_seed is not None:
        g = torch.Generator().manual_seed(perturb_seed)
        vp = 0.3 * torch.randn(eng.var_params.shape, generator=g, dtype=torch.float64)
        eng.var_params.copy_(vp)
        unconstrained = {k: vp[i] for i, k in enumerate(VAR_PARAM_NAMES)}
        if eng.mixture:
            au = 0.5 * torch.randn(eng.alpha_u.shape, generator=g, dtype=torch.float64)
            eng.alpha_u.copy_(au)
            unconstrained["alpha_pi"] = au
        if eng.fit_noise:
            nu = 0.4 * torch.randn(eng.noise_u.shape, generator=g, dtype=torch.float64)
            nu[1] += math.log(0.655)
            eng.noise_u.copy_(nu)
            unconstrained["noise_loc"], unconstrained["noise_scale"] = nu[0], nu[1]
    got = eng.gradients(noise)
    if model != "MixtureNormal":
        oracle_kw["use_bcmatch"] = use_bcmatch and getattr(data, "X_bcmatch_masked", None) is not None
    ref_loss, ref = oracle_at(model, data, noise, unconstrained, **oracle_kw)
    errs = {"loss": abs(got["loss"].item() - ref_loss) / abs(ref_loss)}
    assert errs["loss"] <= tol, f"loss {got['loss'].item()} vs {ref_loss}"
    for k in VAR_PARAM_NAMES:
        errs[k] = rel_err(got[k], ref[k])
        assert errs[k] <= tol, f"{k}: {errs[k]:.3e}"
    if eng.mixture:
        errs["alpha_pi"] = rel_err(got["alpha_pi"], ref["alpha_pi"])
        assert errs["alpha_pi"] <= tol_alpha, f"alpha_pi: {errs['alpha_pi']:.3e}"
    if eng.fit_noise:
        for k in ("noise_loc", "noise_scale"):
            errs[k] = rel_err(got[k], ref[k])
            assert errs[k] <= tol, f"{k}: {errs[k]:.3e}"
    print(model, dtype, errs)
    return errs


CASES = [(torch.float64, 1e-9, 1e-9), (torch.float32, 1e-5, 2e-4)]


@pytest.mark.parametrize("dtype,tol,tol_alpha", CASES)
@pytest.mark.parametrize("perturb", [None, 5])
def test_mixture_normal_gradients(cuda_device, dtype, tol, tol_alpha, perturb):
    data = H.make_small_mixture_data(n_variants=40, n_reps=3)
    data.repguide_mask[1, ::4] = False
    check_grads("MixtureNormal", data, cuda_device, dtype, tol, tol_alpha, perturb_seed=perturb)


@pytest.mark.parametrize("dtype,tol,tol_alpha", CASES)
def test_mixture_normal_gradients_c5_shape(cuda_device, dtype, tol, tol_alpha):
    data = H.make_small_mixture_data(n_variants=200, n_reps=8, with_bulk_bin=False, seed=4)
    check_grads("MixtureNormal", data, cuda_device, dtype, tol, tol_alpha, perturb_seed=2)


@pytest.mark.parametrize("dtype,tol,tol_alpha", CASES)
@pytest.mark.parametrize("model", ["Normal", "ControlNormal"])
def test_normal_models_on_reference_fixture(cuda_device, dtype, tol, tol_alpha, model):
    data = H.load_var_mini()  # c1: tests/data/var_mini_*.csv of the reference
    if model == "ControlNormal" and dtype == torch.float32:
        # the single global (mu, sd) gradient is a sum of mixed-sign per-guide terms ~40x larger than the
        # sum itself: float rounding of the terms (1e-6 each) is amplified by that condition number
        tol = 2e-4
    check_grads(model, data, cuda_device, dtype, tol, tol_alpha, perturb_seed=3, use_bcmatch=False)


@pytest.mark.parametrize("dtype,tol,tol_alpha", CASES)
def test_normal_model_with_bcmatch_layer(cuda_device, dtype, tol, tol_alpha):
    data = H.make_small_mixture_data(n_variants=30, n_reps=4)
    check_grads("Normal", data, cuda_device, dtype, tol, tol_alpha, perturb_seed=1, use_bcmatch=True)


@pytest.mark.parametrize("dtype,tol,tol_alpha", CASES)
@pytest.mark.parametrize("fit_noise", [True, False])
def test_mixture_normal_scale_by_accessibility(cuda_device, dtype, tol, tol_alpha, fit_noise):
    """--scale-by-acc: pi scaled by accessibility + logit-space noise site (bean/model/utils.py:79-178)."""
    data = H.make_small_mixture_data(n_variants=30, n_reps=3, accessibility=True)
    check_grads("MixtureNormal", data, cuda_device, dtype, tol, tol_alpha, perturb_seed=8,
                oracle_kw=dict(scale_by_accessibility=True, fit_noise=fit_noise))


def test_steps_follow_oracle_clipped_adam(cuda_device):
    """k full steps with per-step injected noise: parameters track the oracle's SVI loop (fp64)."""
    data = H.make_small_mixture_data(n_variants=25, n_reps=3)
    k, num_steps = 6, 50
    noises = [H.fixed_noise("MixtureNormal", data, seed=100 + t) for t in range(k)]
    eng = SviEngine(data, "MixtureNormal", cuda_device, dtype=torch.float64, num_steps=num_steps)
    for t in range(k):
        eng.run(1, noise=noises[t])
    with H.default_dtype(torch.float64):
        d = H.cast_data(data, torch.float64)
        ps = O.ParamStore()
        opt = O.ClippedAdam(lr=0.01, lrd=0.1 ** (1 / num_steps))
        ref_losses = []
        for t in range(k):
            loss, _ = O.elbo_mixture_normal(d, ps, noise=noises[t])
            ps.zero_grad()
            loss.backward()
            opt.step(ps.unconstrained)
            ref_losses.append(float(loss.detach()))
    got = eng.params()
    ref = ps.constrained()
    for name in ("mu_loc", "mu_scale", "sd_loc", "sd_scale", "alpha_pi"):
        assert rel_err(got[name], ref[name]) <= 1e-9, name
    assert max(abs(a - b) / abs(b) for a, b in zip(eng.losses().tolist(), ref_losses)) <= 1e-10


@pytest.mark.parametrize("dtype,tol,tol_alpha", CASES)
def test_philox_draws_replayed_into_oracle(cuda_device, dtype, tol, tol_alpha):
    """Let the kernels draw their own noise, record it, and check the oracle agrees on that very noise."""
    data = H.make_small_mixture_data(n_variants=30, n_reps=4)
    eng = SviEngine(data, "MixtureNormal", cuda_device, dtype=dtype, num_steps=4, seed=7)
    got = eng.gradients({"record": True})
    eps, pi = eng.eps_used.double().cpu(), eng.pi_used.double().cpu()
    assert torch.isfinite(pi).all() and (pi > 0).all() and ((pi.sum(-1) - 1).abs() < 1e-6).all()
    noise = {"eps_mu": eps[0].reshape(-1, 1), "eps_sd": eps[1].reshape(-1, 1), "pi": pi.permute(1, 0, 2).unsqueeze(1)}
    ref_loss, ref = oracle_at("MixtureNormal", data, noise)
    assert abs(got["loss"].item() - ref_loss) / abs(ref_loss) <= tol
    for k in VAR_PARAM_NAMES:
        assert rel_err(got[k], ref[k]) <= tol, k
    assert rel_err(got["alpha_pi"], ref["alpha_pi"]) <= tol_alpha


def test_sampler_statistics(cuda_device):
    """Philox Normal and Marsaglia-Tsang Beta draws have the right moments (the CPU and CUDA RNG streams of
    the reference differ too -- SURVEY App. B11 -- so sampling parity is distributional)."""
    data = H.make_small_mixture_data(n_variants=1500, n_reps=8, with_bulk_bin=False, seed=9)
    eng = SviEngine(data, "MixtureNormal", cuda_device, dtype=torch.float32, num_steps=2, seed=3)
    g = torch.Generator().manual_seed(0)
    eng.alpha_u.copy_((torch.rand(eng.alpha_u.shape, generator=g) * 4 - 2))
    eng.gradients({"record": True})
    eps = eng.eps_used.double().cpu()
    n = eps.numel()
    assert abs(eps.mean().item()) < 4 / math.sqrt(n) and abs(eps.var().item() - 1) < 0.1
    al = eng.alpha_u.double().exp().cpu()
    conc = (al / al.sum(-1, keepdim=True) * eng.pi_a0.double().cpu()[:, None]).clamp(min=1e-5)  # (G, 2)
    pi1 = eng.pi_used.double().cpu()[:, :, 1]  # (G, R)
    mean = conc[:, 1] / conc.sum(-1)
    var = conc[:, 0] * conc[:, 1] / (conc.sum(-1) ** 2 * (conc.sum(-1) + 1))
    z = ((pi1.mean(1) - mean) / (var / pi1.shape[1]).sqrt())
    assert abs(z.mean().item()) < 0.15 and abs(z.std().item() - 1) < 0.15, (z.mean().item(), z.std().item())
    # second moment of the standardised draws
    s2 = (((pi1 - mean[:, None]) ** 2) / var[:, None]).mean().item()
    assert abs(s2 - 1) < 0.1, s2
    # a different seed gives different draws, the same seed the same draws
    eng2 = SviEngine(data, "MixtureNormal", cuda_device, dtype=torch.float32, num_steps=2, seed=3)
    eng2.alpha_u.copy_(eng.alpha_u)
    eng2.gradients({"record": True})
    assert torch.equal(eng2.pi_used, eng.pi_used)


def test_svi_improves_elbo_and_recovers_effects(cuda_device):
    """End-to-end run on a synthetic screen: the loss falls and strong true effects are ranked on top."""
    from crispr_bean_b200.data_class import VariantSortingReporterScreenData
    from crispr_bean_b200.synth import make_sorting_screen

    scr = make_sorting_screen(300, 5, n_reps=4, seed=12, frac_effect=0.1)
    data = VariantSortingReporterScreenData(scr, control_can_be_selected=True)
    eng = SviEngine(data, "MixtureNormal", cuda_device, dtype=torch.float32, num_steps=600, seed=1)
    eng.run(600)
    losses = eng.losses()
    assert torch.isfinite(losses).all()
    assert losses[-50:].mean() < losses[:20].mean()
    mu = eng.params()["mu_loc"].reshape(-1).cpu()
    true = torch.as_tensor(scr.guides.groupby("target", sort=False)["true_mu"].first().to_numpy()).float()
    strong = true.abs() > 1.0
    assert strong.sum() >= 5
    corr = torch.corrcoef(torch.stack([mu[strong], true[strong]]))[0, 1].item()
    assert corr > 0.8, corr


def test_sharded_run_reproduces_unsharded_run(cuda_device):
    """Variant shards with global Philox ids: 2 shards (run one after the other on this GPU) give exactly
    the parameters of the unsharded run -- the path needs no data-path collective (SURVEY 8e)."""
    from crispr_bean_b200.dist import shard_data

    data = H.make_small_mixture_data(n_variants=60, n_reps=4, seed=13)
    steps = 20
    full = SviEngine(data, "MixtureNormal", cuda_device, dtype=torch.float32, num_steps=steps, seed=5)
    full.run(steps)
    mu, alpha, loss = [], [], 0
    for rank in range(2):
        sub, off = shard_data(data, rank, 2)
        eng = SviEngine(sub, "MixtureNormal", cuda_device, dtype=torch.float32, num_steps=steps, seed=5,
                        guide_offset=off["guide_offset"], variant_offset=off["variant_offset"])
        eng.run(steps)
        mu.append(eng.params()["mu_loc"])
        alpha.append(eng.params()["alpha_pi"])
        loss = loss + eng.losses()
    assert torch.equal(torch.cat(mu), full.params()["mu_loc"])
    assert torch.equal(torch.cat(alpha), full.params()["alpha_pi"])
    torch.testing.assert_close(loss, full.losses(), rtol=1e-12, atol=0)


def test_end_to_end_result_table_equals_oracle_run(cuda_device):
    """North-star end-to-end check: `run_inference`-style run on the GPU with its OWN Philox draws (recorded per step),
    replayed into the oracle's SVI loop -> posterior mu / sd within 1e-8 (fp64), and the `bean_element_result` table
    built from both has the identical variant ranking and z-scores."""
    import pandas as pd

    from crispr_bean_b200.readwrite import write_result_table

    data = H.make_small_mixture_data(n_variants=40, n_reps=3, seed=12)
    steps = 60
    eng = SviEngine(data, "MixtureNormal", cuda_device, dtype=torch.float64, num_steps=steps, seed=5)
    draws = []
    for _ in range(steps):
        eng.run(1, noise={"record": True})
        eps, pi = eng.eps_used.double().cpu(), eng.pi_used.double().cpu()
        draws.append({"eps_mu": eps[0].reshape(-1, 1), "eps_sd": eps[1].reshape(-1, 1), "pi": pi.permute(1, 0, 2).unsqueeze(1)})
    with H.default_dtype(torch.float64):
        ps, hist = O.run_inference(O.elbo_mixture_normal, H.cast_data(data, torch.float64), num_steps=steps,
                                   noise_fn=lambda t: draws[t])
    got = {k: v.detach().cpu() for k, v in eng.params().items()}
    assert max(abs(a - b) / abs(b) for a, b in zip(eng.losses().tolist(), hist["loss"])) <= 1e-9
    for k, v in hist["params"].items():
        assert rel_err(got[k], v) <= 1e-8, k
    T = data.n_targets
    info = pd.DataFrame({"n": range(T)}, index=pd.Index([f"v{i}" for i in range(T)], name="target"))
    ginfo = pd.DataFrame({"x": range(data.n_guides)})
    import tempfile

    with tempfile.TemporaryDirectory() as tmp:
        kw = dict(model_label="MixtureNormal", prefix=f"{tmp}/", adjust_confidence_by_negative_control=True,
                  adjust_confidence_negatives=list(range(10)), return_result=True)
        tab_gpu = write_result_table(info.copy(), ginfo.copy(), got, **kw)
        tab_ref = write_result_table(info.copy(), ginfo.copy(), hist["params"], **kw)
    assert list(tab_gpu["target"]) == list(tab_ref["target"])  # identical ranking
    for c in ("mu", "mu_sd", "mu_z", "sd", "mu_z_adj"):
        assert (tab_gpu[c] - tab_ref[c]).abs().max() <= 1e-7 * tab_ref[c].abs().max(), c


def test_sampler_distribution_probability_integral_transform(cuda_device):
    """Every recorded pi draw pushed through ITS OWN Beta CDF must be uniform (Kolmogorov-Smirnov), across concentrations
    from 1e-2 (Marsaglia-Tsang boost path, draws piling up at the clamps) to 1e3; and the Normal draws must be normal."""
    from scipy import stats

    data = H.make_small_mixture_data(n_variants=2500, n_reps=8, with_bulk_bin=False, seed=19)
    eng = SviEngine(data, "MixtureNormal", cuda_device, dtype=torch.float32, num_steps=2, seed=11)
    g = torch.Generator().manual_seed(1)
    eng.alpha_u.copy_(torch.rand(eng.alpha_u.shape, generator=g) * 10 - 5)  # alpha_pi in e^-5 .. e^5
    eng.gradients({"record": True})
    al = eng.alpha_u.double().exp().cpu()
    conc = (al / al.sum(-1, keepdim=True) * eng.pi_a0.double().cpu()[:, None]).clamp(min=1e-5).numpy()  # (G, 2)
    pi1 = eng.pi_used.double().cpu()[:, :, 1].numpy()  # (G, R)
    # float32 draws are clamped to [FLT_MIN, 1 - 2^-24] (like torch._sample_dirichlet): for a concentration c the clamp holds
    # a point mass of ~ (1e-38)^c, so the KS test is run where that is negligible (c > 0.5) ...
    keep = conc.min(-1) > 0.5
    u = stats.beta.cdf(pi1[keep], conc[keep, 1:2], conc[keep, 0:1]).reshape(-1)
    assert u.size > 30_000
    ks = stats.kstest(u, "uniform")
    assert ks.statistic < 1.63 / np.sqrt(u.size) * 1.5, ks  # 1 % critical value, with 50 % slack for float32 rounding of the draws
    for lo, hi in ((0.5, 1.0), (1.0, 30.0), (30.0, 1e4)):  # within concentration bands (boost path / plain / large)
        band = (conc.min(-1) >= lo) & (conc.min(-1) < hi)
        if band.sum() * pi1.shape[1] > 3000:
            ub = stats.beta.cdf(pi1[band], conc[band, 1:2], conc[band, 0:1]).reshape(-1)
            assert stats.kstest(ub, "uniform").statistic < 1.63 / np.sqrt(ub.size) * 1.5, (lo, hi)
    # ... and for small concentrations (most draws near 0 or 1, Marsaglia-Tsang boost U^(1/c)) the mass below fixed
    # thresholds is compared with the Beta CDF (binomial 4-sigma bands)
    small = (conc[:, 1] > 1e-2) & (conc[:, 1] < 0.5) & (conc[:, 0] > 1.0)
    assert small.sum() > 100
    for thr in (1e-30, 1e-12, 1e-4, 1e-1):
        p_theory = stats.beta.cdf(thr, conc[small, 1:2], conc[small, 0:1])  # (n, 1) per guide
        expect = (p_theory * pi1.shape[1]).sum()
        var = (p_theory * (1 - p_theory) * pi1.shape[1]).sum()
        got = (pi1[small] <= thr).sum()
        assert abs(got - expect) <= 4 * np.sqrt(var) + 2, (thr, got, expect)
    eps = eng.eps_used.double().cpu().numpy().reshape(-1)
    assert stats.kstest(eps, "norm").statistic < 0.02


@pytest.mark.parametrize("dtype", [torch.float64, torch.float32])
@pytest.mark.parametrize("bulk_bin", [True, False])
def test_specialised_and_generic_guide_kernels_agree(cuda_device, dtype, bulk_bin):
    """Screens with exactly 4 / 5 bins and no masked sample run the specialised guide kernel (no bin predicates, size factors
    from shared memory, no sample-mask multiplies); `force_generic` sends the same screen through the generic one.  The two
    differ only by multiplications with 1.0 and by where constants are read from: same losses, same parameters."""
    data = H.make_small_mixture_data(n_variants=60, n_reps=4, seed=23, with_bulk_bin=bulk_bin)
    assert data.n_condits == (5 if bulk_bin else 4) and bool((data.sample_mask == 1).all())
    runs = []
    for generic in (0, 1):
        eng = SviEngine(data, "MixtureNormal", cuda_device, dtype=dtype, num_steps=10, seed=3)
        eng.cfg.force_generic = generic
        eng.run(6)
        runs.append((eng.losses(), {k: v.cpu() for k, v in eng.params().items()}))
    tol = 1e-12 if dtype == torch.float64 else 1e-6
    torch.testing.assert_close(runs[0][0], runs[1][0], rtol=tol, atol=0)
    for k, v in runs[0][1].items():
        torch.testing.assert_close(v, runs[1][1][k], rtol=tol * 10, atol=tol * 1e-2)
