"""Program options the golden fixtures do not exercise (`alpha_prior`, `sd_scale`, `mask_thres`, `use_bcmatch` off / on,
`mu_negctrl` fed from the negative-control fit, tiling `epsilon`): the CPU oracle against the reference's own model / guide
programs, evaluated live through tests/refharness on the same screen and draws (float64; skipped without BEAN_REFERENCE_ROOT)."""
import copy
from functools import partial

import numpy as np
import pytest
import torch

from crispr_bean_b200 import data_class as dc
from crispr_bean_b200.synth import make_sorting_screen, make_survival_screen, make_tiling_screen
from oracle import bean_oracle as O
from tests.helpers import cast_data, default_dtype
from tests.refharness import available, load_reference
from tests.refharness import golden as G

pytestmark = pytest.mark.skipif(not available(), reason="reference sources not mounted")

SORT = dict(control_can_be_selected=True)
SURV = dict(condition_column="condition", time_column="time", control_condition="D7")


def cases(ns):
    m, sm = ns.model, ns.survival_model
    sort_scr = make_sorting_screen(12, 4, n_reps=3, seed=31, n_negctrl_guides=5, depth=60.0)  # low depth: some rows near mask_thres
    surv_scr = make_survival_screen(10, 4, n_reps=3, seed=32, n_negctrl_guides=5, depth=150.0)
    til_scr = make_tiling_screen(n_guides=30, n_reps=3, seed=33)
    til_kw = dict(SORT, allele_df_key="allele_counts")
    return [
        ("mixture alpha_prior sd_scale", sort_scr, "VariantSortingReporterScreenData", SORT,
         partial(m.MixtureNormalModel, alpha_prior=3.0, sd_scale=0.05), partial(m.MixtureNormalGuide, alpha_prior=3.0),
         O.elbo_mixture_normal, dict(alpha_prior=3.0, sd_scale=0.05)),
        ("mixture without bcmatch", sort_scr, "VariantSortingReporterScreenData", SORT,
         partial(m.MixtureNormalModel, use_bcmatch=False), m.MixtureNormalGuide, O.elbo_mixture_normal, dict(use_bcmatch=False)),
        ("normal mask_thres sd_scale", sort_scr, "VariantSortingScreenData", SORT,
         partial(m.NormalModel, mask_thres=40, use_bcmatch=False, sd_scale=0.1), m.NormalGuide, O.elbo_normal,
         dict(mask_thres=40, use_bcmatch=False, sd_scale=0.1)),
        ("control normal with bcmatch", sort_scr, "VariantSortingScreenData", dict(SORT, use_bcmatch=True),
         partial(m.ControlNormalModel, use_bcmatch=True, mask_thres=25), partial(m.ControlNormalGuide, use_bcmatch=True),
         O.elbo_control_normal, dict(use_bcmatch=True, mask_thres=25)),
        ("tiling alpha_prior epsilon", til_scr, "TilingSortingReporterScreenData", til_kw,
         partial(m.MultiMixtureNormalModel, alpha_prior=2.0, epsilon=1e-4, use_bcmatch=(True,)),
         partial(m.MultiMixtureNormalGuide, alpha_prior=2.0, epsilon=1e-4), O.elbo_multi_mixture_normal, dict(alpha_prior=2.0, epsilon=1e-4)),
        ("survival mixture mu_negctrl alpha_prior", surv_scr, "VariantSurvivalReporterScreenData", SURV,
         partial(sm.MixtureNormalModel, mu_negctrl=(0.03, 0.2), alpha_prior=2.0), partial(sm.MixtureNormalGuide, alpha_prior=2.0),
         O.elbo_survival_mixture_normal, dict(mu_negctrl=(0.03, 0.2), alpha_prior=2.0)),
        ("survival normal mask_thres", surv_scr, "VariantSurvivalScreenData", dict(SURV, negctrl_guide_idx=[0, 1, 2, 3, 4]),
         partial(sm.NormalModel, mask_thres=60, use_bcmatch=False), sm.NormalGuide, O.elbo_survival_normal, dict(mask_thres=60, use_bcmatch=False)),
    ]


def ids():
    return ["mixture-alpha_prior-sd_scale", "mixture-no-bcmatch", "normal-mask_thres", "control-normal-bcmatch", "tiling-alpha_prior-epsilon",
            "survival-mixture-mu_negctrl", "survival-normal-mask_thres"]


@pytest.mark.parametrize("i", range(7), ids=ids())
def test_oracle_equals_reference_program_with_options(i):
    ns = load_reference()
    name, scr, cls, data_kw, model, guide, elbo, okw = cases(ns)[i]
    ref_scr = copy.deepcopy(scr)
    if cls.startswith("Tiling"):
        import sys

        from tests.helpers import GOLDEN

        sys.path.insert(0, GOLDEN)
        from make_reference_golden import with_allele_objects

        ref_scr = with_allele_objects(ns, scr)
    ref_data = getattr(ns.data_class, cls)(ref_scr, **data_kw)
    out, noise = G.reference_loss_and_grads(ns.pyro, model, guide, ref_data, seed=5, dtype=torch.float64)
    data = getattr(dc, cls)(copy.deepcopy(scr), **data_kw)
    for k in ("a0", "a0_bcmatch", "pi_a0"):  # the reference's curve_fit products (scipy's 1.5e-8 stopping tolerance)
        if hasattr(ref_data, k) and getattr(ref_data, k) is not None and hasattr(data, k):
            setattr(data, k, torch.as_tensor(getattr(ref_data, k)).clone())
    perm = None
    if hasattr(ref_data, "edit_index"):
        keys = sorted(ref_data.edit_index, key=ref_data.edit_index.get)
        perm = np.asarray([data.edit_index[str(k)] for k in keys])

    def ours(arr, key):  # (E,)-shaped reference arrays -> our edit order
        if perm is None or key.split("/")[-1] not in ("mu_loc", "mu_scale", "sd_loc", "sd_scale", "eps_mu", "eps_sd"):
            return arr
        o = np.empty_like(arr)
        o[..., perm] = arr
        return o

    inj = {k[len("noise/"):]: torch.as_tensor(ours(v, k)) for k, v in noise.items() if "/" not in k[len("noise/"):]}
    with default_dtype(torch.float64):
        ps = O.ParamStore()
        loss, _ = elbo(cast_data(data, torch.float64), ps, noise=inj, **okw)
        loss.backward()
    assert abs(float(loss.detach()) - float(out["loss"])) <= 1e-11 * abs(float(out["loss"])), name
    n = 0
    for k, v in out.items():
        if not k.startswith("grad/"):
            continue
        g = ps.unconstrained[k[5:]].grad
        g = (g if g is not None else torch.zeros_like(ps.unconstrained[k[5:]])).detach().double().numpy().reshape(v.shape)
        ref = ours(v, k)
        assert np.abs(g - ref).max() <= 1e-9 * max(np.abs(ref).max(), 1e-300), (name, k)
        n += 1
    assert n >= 2
