"""`prepare_bdata` (tests/support/prepare.py) against the reference's own function (bean/preprocessing/utils.py:24-67 +
bean/qc/guide_qc.py:49-75, executed in place through tests/refharness where BEAN_REFERENCE_ROOT is set) and against the
behaviour it documents (portable checks)."""
import os
from types import SimpleNamespace

import numpy as np
import pandas as pd
import pytest

from tests.support.prepare import filter_no_info_target, prepare_bdata
from crispr_bean_b200.screen import MiniScreen
from crispr_bean_b200.synth import make_sorting_screen, make_survival_screen
from tests.refharness import available, load_reference


def cli(**kw):
    base = dict(replicate_col="replicate", selection="sorting", exclude_control_condition_for_inference=False, condition_col="bin",
                control_condition="bulk", library_design="variant", target_col="target")
    base.update(kw)
    return SimpleNamespace(**base)


def shuffled_with_holes(scr, seed=0):
    """Guides in random order, some without counts, one whole target without counts."""
    rng = np.random.default_rng(seed)
    scr = scr[rng.permutation(len(scr.guides)), :]
    X = scr.X.copy()
    X[[2, 9], :] = 0                                                   # two empty guides
    X[(scr.guides["target"] == scr.guides["target"].iloc[5]).to_numpy(), :] = 0  # an empty target
    return MiniScreen(X, scr.guides, scr.samples, scr.layers, scr.uns)


def same_screen(a, b):
    assert list(a.guides.index) == list(b.guides.index) and list(a.samples.index) == list(b.samples.index)
    assert np.array_equal(a.X, b.X)
    for k in a.layers:
        assert np.array_equal(a.layers[k], b.layers[k]), k
    assert list(a.guides.columns) == list(b.guides.columns) and list(a.samples.columns) == list(b.samples.columns)
    assert str(a.samples["replicate"].dtype) == str(b.samples["replicate"].dtype) == "category"


CASES = [("sorting-variant", lambda: make_sorting_screen(14, 4, n_reps=3, seed=2, n_negctrl_guides=4), cli()),
         ("sorting-tiling", lambda: make_sorting_screen(10, 3, n_reps=2, seed=3), cli(library_design="tiling")),
         ("survival-variant", lambda: make_survival_screen(12, 4, n_reps=3, seed=4, n_negctrl_guides=4),
          cli(selection="survival", condition_col="condition", control_condition="D7")),
         ("survival-exclude-control", lambda: make_survival_screen(12, 4, n_reps=3, seed=5, n_negctrl_guides=4),
          cli(selection="survival", condition_col="condition", control_condition="D7", exclude_control_condition_for_inference=True))]


@pytest.mark.skipif(not available(), reason="reference sources not mounted")
@pytest.mark.parametrize("name,make,args", CASES, ids=[c[0] for c in CASES])
def test_equals_reference_prepare_bdata(tmp_path, name, make, args):
    ref_fn = load_reference().prep_utils.prepare_bdata
    scr = shuffled_with_holes(make())
    scr.guides["dup"] = 1
    scr.guides = pd.concat([scr.guides, scr.guides[["dup"]]], axis=1)  # a duplicated column name: dropped by both
    ref_dir, my_dir = tmp_path / "ref", tmp_path / "mine"
    ref_dir.mkdir(), my_dir.mkdir()
    ref_warn, my_warn = [], []
    ref = ref_fn(scr.copy(), args, ref_warn.append, str(ref_dir))
    mine = prepare_bdata(scr.copy(), args, my_warn.append, str(my_dir))
    same_screen(mine, ref)
    assert my_warn == ref_warn and len(my_warn) >= 1
    assert sorted(os.listdir(my_dir)) == sorted(os.listdir(ref_dir))
    for f in os.listdir(ref_dir):
        assert (my_dir / f).read_text() == (ref_dir / f).read_text(), f
    assert len(scr.guides) > len(mine.guides) and "replicate" in scr.samples.columns  # the input screen is left alone


def test_documented_behaviour(tmp_path):
    scr = shuffled_with_holes(make_sorting_screen(14, 4, n_reps=3, seed=2, n_negctrl_guides=4))
    warned = []
    out = prepare_bdata(scr, cli(), warned.append, str(tmp_path))
    assert (out.X.sum(axis=1) > 0).all()
    t = out.guides["target"].to_numpy()
    assert list(t) == sorted(t)  # guides of a variant contiguous (data_class.py:511-532 relies on it)
    assert "Filtering out" in warned[0]
    # the empty target's guides already went with the empty guides, so the side file exists and lists nothing
    assert list(pd.read_csv(tmp_path / "no_support_targets.csv").columns) == ["target"]
    assert scr.guides["target"].iloc[5] not in set(t)


def test_unmasked_sample_without_counts_is_an_error(tmp_path):
    scr = make_sorting_screen(8, 3, n_reps=2, seed=1)
    X = scr.X.copy()
    X[:, 3] = 0
    bad = MiniScreen(X, scr.guides, scr.samples, scr.layers, scr.uns)
    with pytest.raises(ValueError, match="has 0 counts"):
        prepare_bdata(bad, cli(), lambda m: None, str(tmp_path))
    bad.samples.loc[bad.samples.index[3], "mask"] = 0  # masking the sample is the documented way out
    assert prepare_bdata(bad, cli(), lambda m: None, str(tmp_path)).X.shape[1] == scr.X.shape[1]


def test_null_target_is_an_error(tmp_path):
    scr = make_sorting_screen(8, 3, n_reps=2, seed=1)
    scr.guides.loc[scr.guides.index[0], "target"] = None
    with pytest.raises(ValueError, match="value is null"):
        prepare_bdata(scr, cli(), lambda m: None, str(tmp_path))


def test_filter_no_info_target_counts_all_samples(tmp_path):
    scr = shuffled_with_holes(make_sorting_screen(10, 3, n_reps=2, seed=7))
    n, out = filter_no_info_target(scr, "bin", "bulk", write_no_support_targets=True, no_support_target_write_path=str(tmp_path / "t.csv"))
    assert n == 1 and len(out.guides) == len(scr.guides) - 3
