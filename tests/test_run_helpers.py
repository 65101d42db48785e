"""Caller-side helpers of `bean run` mirrored in crispr_bean_b200/run.py (`check_args`, `_get_guide_target_info`,
`_get_guide_to_variant_df`, `_check_prior_params`) against the reference's own functions (bean/model/run.py:39-344,
:479-542, executed in place through tests/refharness where BEAN_REFERENCE_ROOT is set)."""
import copy
import pickle
from types import SimpleNamespace

import numpy as np
import pandas as pd
import pytest
import torch

from tests.support import run_helpers as mine
from crispr_bean_b200.synth import make_sorting_screen, make_survival_screen, make_tiling_screen
from tests.refharness import available, load_reference

needs_reference = pytest.mark.skipif(not available(), reason="reference sources not mounted")


def cli(**kw):
    base = dict(scale_by_acc=False, acc_col=None, acc_bw_path=None, outdir=None, bdata_path="/tmp/x/screen.h5ad", fit_negctrl=False,
                negctrl_col="target_group", negctrl_col_value="NegCtrl", selection="sorting", sorting_bin_upper_quantile_col="upper_quantile",
                sorting_bin_lower_quantile_col="lower_quantile", time_col="time", library_design="variant",
                dont_adjust_confidence_by_negative_control=False, allele_df_key=None, repguide_mask="repguide_mask", replicate_col="replicate",
                sample_mask_col="mask", condition_col="bin", control_condition="bulk", control_guide_tag=None,
                alpha_if_overdispersion_fitting_fails=None, target_col="target")
    base.update(kw)
    return SimpleNamespace(**base)


def screens():
    var = make_sorting_screen(14, 4, n_reps=3, seed=2, n_negctrl_guides=12)
    til = make_tiling_screen(n_guides=20, n_reps=2, seed=3)
    til.uns["allele_counts_filtered"] = til.uns["allele_counts"].iloc[::2].copy()
    til.uns["sample_covariates_note"] = "not a table"
    sur = make_survival_screen(12, 4, n_reps=3, seed=4, n_negctrl_guides=12)
    return var, til, sur


GOOD = [("variant", 0, dict()),
        ("variant-fit-negctrl", 0, dict(fit_negctrl=True)),
        ("variant-acc-both", 0, dict(scale_by_acc=True, acc_col="target_group", acc_bw_path="x.bw")),
        ("variant-popt", 0, dict(alpha_if_overdispersion_fitting_fails="-1.5,0.8", sample_mask_col="")),
        ("tiling-picks-most-filtered", 1, dict(library_design="tiling")),
        ("tiling-key-given", 1, dict(library_design="tiling", allele_df_key="allele_counts", dont_adjust_confidence_by_negative_control=True)),
        ("survival", 2, dict(selection="survival", condition_col="condition", control_condition="D7,D0"))]
BAD = [("acc-without-source", 0, dict(scale_by_acc=True)),
       ("negctrl-col-missing", 0, dict(fit_negctrl=True, negctrl_col="nope")),
       ("too-few-negctrl", 0, dict(fit_negctrl=True, negctrl_col_value="PosCtrl")),
       ("quantile-col-missing", 0, dict(sorting_bin_upper_quantile_col="uq")),
       ("time-col-missing", 2, dict(selection="survival", condition_col="condition", control_condition="D7", time_col="t")),
       ("condition-equals-time", 2, dict(selection="survival", condition_col="time", control_condition="7")),
       ("bad-design", 0, dict(library_design="other")),
       ("allele-key-missing", 1, dict(library_design="tiling", allele_df_key="nope")),
       ("mask-col-missing", 0, dict(sample_mask_col="nope")),
       ("condition-col-missing", 0, dict(condition_col="nope")),
       ("control-label-missing", 0, dict(control_condition="bulk,other")),
       ("replicate-col-missing", 0, dict(replicate_col="nope")),
       ("control-tag-in-variant-mode", 0, dict(control_guide_tag="CONTROL")),
       ("control-tag-absent", 1, dict(library_design="tiling", allele_df_key="allele_counts", control_guide_tag="zzz"))]


@needs_reference
@pytest.mark.parametrize("name,which,kw", GOOD, ids=[c[0] for c in GOOD])
def test_check_args_fills_the_same_derived_arguments(name, which, kw):
    ref_fn = load_reference().run.check_args
    scr = screens()[which]
    a_ref, a_mine = cli(**kw), cli(**kw)
    s_ref, s_mine = copy.deepcopy(scr), copy.deepcopy(scr)
    ref_fn(a_ref, s_ref)
    warned = []
    mine.check_args(a_mine, s_mine, warn=warned.append)
    assert vars(a_mine) == vars(a_ref)
    assert set(s_mine.uns) == set(s_ref.uns)
    if "repguide_mask" in s_ref.uns and "repguide_mask" not in scr.uns:
        m, r = s_mine.uns["repguide_mask"], s_ref.uns["repguide_mask"]
        assert list(m.index) == list(r.index) and list(m.columns) == list(r.columns) and (m.to_numpy() == 1).all() and (r.to_numpy() == 1).all()
        assert any("outlier mask" in w for w in warned)


@needs_reference
@pytest.mark.parametrize("name,which,kw", BAD, ids=[c[0] for c in BAD])
def test_check_args_rejects_what_the_reference_rejects(name, which, kw):
    ref_fn = load_reference().run.check_args
    scr = screens()[which]
    with pytest.raises((ValueError, KeyError)) as ref_exc:  # (a missing replicate column surfaces as pandas' KeyError there)
        ref_fn(cli(**kw), copy.deepcopy(scr))
    with pytest.raises(ref_exc.type):
        mine.check_args(cli(**kw), copy.deepcopy(scr), warn=lambda m: None)


@needs_reference
def test_guide_target_info_equals_reference():
    ref_fn = load_reference().run._get_guide_target_info
    scr = make_sorting_screen(14, "lognormal", n_reps=2, seed=5, n_negctrl_guides=6)
    rng = np.random.default_rng(1)
    scr.guides["edit_rate"] = rng.random(len(scr.guides))
    scr.guides["target_pos"] = scr.guides["target"].map(lambda t: hash(t) % 97)    # constant within a target: kept
    scr.guides["target_varies"] = np.arange(len(scr.guides))                        # not constant: dropped
    args = cli()
    a = mine._get_guide_target_info(scr, args, cols_include=["target_group"])
    b = ref_fn(scr, args, cols_include=["target_group"])
    pd.testing.assert_frame_equal(a, b)
    assert {"target_group", "target_pos", "n_guides", "edit_rate_mean", "edit_rate_std"} <= set(a.columns) and "target_varies" not in a.columns


@needs_reference
def test_guide_to_variant_df_equals_reference():
    ref_fn = load_reference().run._get_guide_to_variant_df
    t = pd.DataFrame({"edit": ["e1", "e2", "e3", "e4"], "editing_guides": ["g1,g2", "g2", "", np.nan],
                      "per_guide_editing_rates": ["0.1,0.25", "0.5", "", np.nan]})
    a, b = mine._get_guide_to_variant_df(t), ref_fn(t)
    assert list(a.index) == list(b.index) and list(a.columns) == list(b.columns)
    for col in a.columns:
        for x, y in zip(a[col], b[col]):
            assert len(x) == len(y) and all((p == q) or (p != p and q != q) for p, q in zip(x, y)), col


@needs_reference
@pytest.mark.parametrize("survival", [False, True])
def test_check_prior_params_equals_reference(tmp_path, survival):
    ns = load_reference()
    T = 9
    ours = SimpleNamespace(n_targets=T, n_guides=30, is_sorting=not survival)
    base = ns.data_class.ScreenData if survival else ns.data_class.SortingScreenData
    theirs = base.__new__(base)
    theirs.n_targets, theirs.n_guides = T, 30
    cases = [{"mu_loc": torch.zeros(T), "sd_loc": torch.zeros(T)},                 # 1-D: reshaped (sorting) / rejected (survival mu_loc)
             {"mu_loc": torch.zeros(T, 1), "mu_scale": torch.ones(T, 1), "sd_loc": torch.zeros(T, 1), "sd_scale": torch.ones(T, 1)},
             {"mu_loc": 0.1, "mu_scale": 2.0},                                      # scalars pass through
             {"sd_scale": torch.ones(T)},                                           # the int-vs-tuple comparison: rejected
             {"mu_scale": torch.ones(T)},
             {"mu_loc": torch.zeros(T + 1, 1)},
             {"initial_abundance": torch.ones(T)}, {"initial_abundance": torch.ones(T, 1)}]
    for i, prior in enumerate(cases):
        path = tmp_path / f"p{i}.pkl"
        with open(path, "wb") as f:
            pickle.dump(prior, f)
        outcome = []
        for fn, nd in ((ns.run._check_prior_params, theirs), (mine._check_prior_params, ours)):
            try:
                out = fn(str(path), nd)
                outcome.append({k: (tuple(v.shape) if torch.is_tensor(v) else v) for k, v in out.items()})
            except ValueError:
                outcome.append("ValueError")
        assert outcome[0] == outcome[1], (i, prior.keys(), outcome)
    with pytest.raises(ValueError, match="not found"):
        mine._check_prior_params(str(tmp_path / "absent.pkl"), ours)


def test_portable_expectations(tmp_path):
    """The same behaviour stated without the reference (runs anywhere)."""
    var, til, _ = screens()
    args, scr = mine.check_args(cli(library_design="tiling"), til, warn=lambda m: None)
    assert args.allele_df_key == "allele_counts_filtered" and args.adjust_confidence_by_negative_control is True and args.popt is None
    assert args.outdir == "/tmp/x" and "repguide_mask" in scr.uns
    with pytest.raises(ValueError, match="Not enough negative control"):
        mine.check_args(cli(fit_negctrl=True, negctrl_col_value="PosCtrl"), var, warn=lambda m: None)
    info = mine._get_guide_target_info(var, cli(), cols_include=["target_group"])
    assert info.index.name == "target" and info["n_guides"].sum() == len(var.guides)
