"""Tensoriser options the golden fixtures do not exercise (`shrink_alpha`, pre-fitted `popt` / `pi_popt`, `impute_pi_popt`,
a replicate x guide outlier mask, masked samples, `use_const_pi`-free variants): the mirror's data classes against the
reference's, built live through tests/refharness from the same screen (skipped without BEAN_REFERENCE_ROOT)."""
import copy

import numpy as np
import pandas as pd
import pytest
import torch

from crispr_bean_b200 import data_class as dc
from crispr_bean_b200.synth import make_sorting_screen, make_survival_screen, make_tiling_screen
from tests.refharness import available, load_reference
from tests.refharness.golden import data_tensors

pytestmark = pytest.mark.skipif(not available(), reason="reference sources not mounted")


def with_masks(scr, seed=0):
    """A replicate x guide outlier mask with some zeros and one masked sample (what `bean qc` writes)."""
    rng = np.random.default_rng(seed)
    reps = list(pd.unique(scr.samples["replicate"]))
    mask = pd.DataFrame(1, index=scr.guides.index, columns=reps)
    for r in reps:
        mask.loc[rng.choice(scr.guides.index, size=3, replace=False), r] = 0
    scr.uns["repguide_mask"] = mask
    scr.samples["mask"] = 1
    scr.samples.loc[scr.samples.index[1], "mask"] = 0
    return scr


def as_float64(scr):
    """`shrink_alpha` in the reference needs float64 counts (its masked assignment mixes the float32 moment estimate with the
    float64 fit and torch refuses: get_alpha0.py:115); screens written by `bean count` are float64 when they get there."""
    from crispr_bean_b200.screen import MiniScreen

    return MiniScreen(scr.X.astype(np.float64), scr.guides, scr.samples, {k: v.astype(np.float64) for k, v in scr.layers.items()}, scr.uns)


def compare(cls, scr, kw, fit_tol=1e-7):
    ns = load_reference()
    if kw.get("shrink_alpha"):
        scr = as_float64(scr)
    ref_scr = copy.deepcopy(scr)
    if cls.startswith("Tiling"):
        import sys

        from tests.helpers import GOLDEN

        sys.path.insert(0, GOLDEN)
        from make_reference_golden import with_allele_objects

        ref_scr = with_allele_objects(ns, scr)
    ref = data_tensors(getattr(ns.data_class, cls)(ref_scr, **kw))
    mine = getattr(dc, cls)(copy.deepcopy(scr), **kw)
    perm = None
    checked = 0
    for k, v in ref.items():
        if not hasattr(mine, k):
            assert v.ndim == 0, f"tensor {k} of the reference data class is absent from the mirror"
            continue
        m = getattr(mine, k)
        if not torch.is_tensor(m):
            assert m == v.item(), k
            continue
        m = m.numpy()
        if k == "allele_to_edit":
            continue  # edit numbering is a labelling (set order); covered by tests/test_reference_golden.py
        assert m.shape == v.shape and str(m.dtype) == str(v.dtype), (k, m.shape, v.shape, m.dtype, v.dtype)
        if k in ("a0", "a0_bcmatch", "pi_a0"):
            assert np.abs(m - v).max() <= fit_tol * np.abs(v).max(), (k, np.abs(m - v).max() / np.abs(v).max())
        else:
            assert np.array_equal(m, v, equal_nan=True), k
        checked += 1
    assert checked >= 12
    return mine


SORT = dict(control_can_be_selected=True)
CASES = [
    ("shrink_alpha", "VariantSortingReporterScreenData", lambda: make_sorting_screen(14, 4, n_reps=3, seed=1), dict(SORT, shrink_alpha=True)),
    ("popt", "VariantSortingReporterScreenData", lambda: make_sorting_screen(14, 4, n_reps=3, seed=2), dict(SORT, popt=(-1.2, 0.7))),
    ("pi_popt", "VariantSortingReporterScreenData", lambda: make_sorting_screen(14, 4, n_reps=3, seed=3), dict(SORT, pi_popt=(-2.0, 0.9))),
    ("impute_pi_popt", "VariantSortingReporterScreenData", lambda: make_sorting_screen(14, 4, n_reps=3, seed=4),
     dict(SORT, popt=(-1.2, 0.7), impute_pi_popt=True)),
    ("masks", "VariantSortingReporterScreenData", lambda: with_masks(make_sorting_screen(14, 4, n_reps=3, seed=5)),
     dict(SORT, repguide_mask="repguide_mask", sample_mask_column="mask")),
    ("masks-normal", "VariantSortingScreenData", lambda: with_masks(make_sorting_screen(14, 4, n_reps=3, seed=6)),
     dict(SORT, repguide_mask="repguide_mask", sample_mask_column="mask", use_bcmatch=True)),
    ("too-few-guides-fallback", "VariantSortingReporterScreenData", lambda: make_sorting_screen(1, 3, n_reps=2, seed=7), dict(SORT)),
    ("survival-shrink-masks", "VariantSurvivalReporterScreenData", lambda: with_masks(make_survival_screen(12, 4, n_reps=3, seed=8)),
     dict(condition_column="condition", time_column="time", control_condition="D7", shrink_alpha=True, repguide_mask="repguide_mask",
          sample_mask_column="mask")),
    ("tiling-shrink-masks", "TilingSortingReporterScreenData", lambda: with_masks(make_tiling_screen(n_guides=30, n_reps=3, seed=9)),
     dict(SORT, allele_df_key="allele_counts", shrink_alpha=True, repguide_mask="repguide_mask", sample_mask_column="mask")),
]


@pytest.mark.parametrize("name,cls,make,kw", CASES, ids=[c[0] for c in CASES])
def test_option_equals_reference(name, cls, make, kw):
    compare(cls, make(), kw)


def test_negctrl_subset_equals_reference():
    """`ndata[negctrl_idx]` (cli/run.py:247): the guide subset the negative-control fit runs on."""
    ns = load_reference()
    scr = make_sorting_screen(14, 4, n_reps=3, seed=11, n_negctrl_guides=8)
    idx = np.where(scr.guides["target_group"].to_numpy() == "NegCtrl")[0]
    ref = ns.data_class.VariantSortingReporterScreenData(copy.deepcopy(scr), **SORT)[idx]
    mine = dc.VariantSortingReporterScreenData(copy.deepcopy(scr), **SORT)[idx]
    r = data_tensors(ref)
    unsliced_there = {"X_control_masked", "X_bcmatch_control_masked", "allele_counts_control"}
    n = 0
    for k, v in r.items():
        if hasattr(mine, k) and torch.is_tensor(getattr(mine, k)):
            m = getattr(mine, k).numpy()
            if m.shape != v.shape:
                # the reference leaves some control-sample tensors unsliced (X_control_masked, allele_counts_control, ...:
                # data_class.py:207-218, :399-414 list what it slices); the mirror slices every guide-axis tensor
                assert k in unsliced_there and len(idx) in m.shape, k
                continue
            if k in ("a0", "a0_bcmatch", "pi_a0"):
                assert np.abs(m - v).max() <= 1e-7 * np.abs(v).max(), k
            else:
                assert np.array_equal(m, v, equal_nan=True), k
            n += 1
    assert n >= 12 and mine.n_guides == len(idx)
