"""`read_h5ad` (crispr_bean_b200/screen.py) + the HDF5 subset reader (crispr_bean_b200/h5lite.py) on the reference's own
`.h5ad` test screens (reference: bean/framework/ReporterScreen.py:read_h5ad, used by cli/run.py:62).

The files are written by anndata/h5py and live under tests/data of the original project (a checkout of it named by
BEAN_REFERENCE_ROOT, tests/refharness): those tests skip without it.  The screens they decode to are ALSO committed inside
tests/golden/ref_*real*.npz (with everything the reference computed from them), so the rest of the suite -- CPU and
GPU -- exercises the decoded data without the files.
"""
import os

import numpy as np
import pandas as pd
import pytest

from crispr_bean_b200 import h5lite
from crispr_bean_b200.screen import MiniScreen, read_h5ad
from tests.helpers import GOLDEN
from tests.refharness import REFERENCE_ROOT
from tests.refharness.golden import screen_from_arrays

REF_DATA = os.path.join(REFERENCE_ROOT, "tests", "data")
needs_reference = pytest.mark.skipif(not (REFERENCE_ROOT and os.path.isdir(REF_DATA)), reason="reference test data not mounted")

SHAPES = {  # file -> (guides, samples, rows of uns['allele_counts'])
    "var_mini_screen": (30, 10, 4926),
    "var_mini_screen_dual": (30, 10, 4926),
    "var_mini_screen_missing": (30, 8, 4926),
    "tiling_mini_screen": (30, 10, 3853),
    "tiling_mini_screen_missing": (30, 8, 3853),
    "survival_var_mini_screen": (25, 9, 573),
    "survival_tiling_mini_screen": (30, 6, 3853),
    "bean_count_test_screen": (3455, 12, None),
}


def test_not_an_hdf5_file(tmp_path):
    p = tmp_path / "x.h5ad"
    p.write_bytes(b"guide,count\n" * 64)
    with pytest.raises(h5lite.H5Error, match="not an HDF5 file"):
        read_h5ad(str(p))


def test_unsupported_superblock_is_reported(tmp_path):
    p = tmp_path / "v3.h5ad"
    p.write_bytes(b"\x89HDF\r\n\x1a\n" + bytes([3]) + bytes(200))  # libver='latest' superblock
    with pytest.raises(h5lite.H5Error, match="superblock version 3"):
        h5lite.File(str(p))


@needs_reference
@pytest.mark.parametrize("name", sorted(SHAPES))
def test_reference_fixture_decodes(name):
    scr = read_h5ad(f"{REF_DATA}/{name}.h5ad")
    G, S, n_alleles = SHAPES[name]
    assert isinstance(scr, MiniScreen) and scr.X.shape == (G, S)
    assert scr.guides.index.is_unique and scr.samples.index.is_unique
    assert {"X_bcmatch", "edits"} <= set(scr.layers)
    assert (scr.X >= 0).all() and (scr.layers["X_bcmatch"] <= scr.X).all()  # barcode-matched reads are a subset
    if n_alleles is not None:
        tbl = scr.uns["allele_counts"]
        assert len(tbl) == n_alleles and list(tbl.columns[:2]) == ["guide", "allele"]
        assert list(tbl.columns[2:]) == list(scr.samples.index)
        assert set(tbl["guide"]) <= set(scr.guides.index)
    assert isinstance(scr.uns["tiling"], (bool, np.bool_))


@needs_reference
def test_var_mini_equals_the_csv_export():
    """var_mini_{counts,guides,samples}.csv are the reference's CSV export of var_mini_screen.h5ad."""
    scr = read_h5ad(f"{REF_DATA}/var_mini_screen.h5ad")
    counts = pd.read_csv(f"{REF_DATA}/var_mini_counts.csv", index_col=0)
    guides = pd.read_csv(f"{REF_DATA}/var_mini_guides.csv", index_col=0)
    samples = pd.read_csv(f"{REF_DATA}/var_mini_samples.csv", index_col=0)
    assert list(scr.guides.index) == list(counts.index) and list(scr.samples.index) == list(counts.columns)
    assert np.array_equal(scr.X, counts.to_numpy())
    for c in samples.columns:
        assert list(scr.samples[c]) == list(samples[c]), c
    for c in ("target_group", "sequence"):  # (`target` was relabelled after the CSV export)
        if c in guides.columns:
            assert list(scr.guides[c].astype(str)) == list(guides[c].astype(str)), c


REAL = {"real_var_mini_mixture": "var_mini_screen", "tiling_real_mini": "tiling_mini_screen",
        "survival_real_var_mixture": "survival_var_mini_screen", "survival_tiling_real_mini": "survival_tiling_mini_screen"}


@needs_reference
@pytest.mark.parametrize("case", sorted(REAL))
def test_committed_screens_are_what_the_reader_decodes(case):
    """The screens stored in the real-data golden fixtures == the .h5ad files decoded now (guards the fixtures
    against drifting from the reader)."""
    z = np.load(os.path.join(GOLDEN, f"ref_{case}.npz"))
    stored = screen_from_arrays(z)
    scr = read_h5ad(f"{REF_DATA}/{REAL[case]}.h5ad")
    if "target" in scr.guides.columns:
        scr = scr[np.argsort(scr.guides["target"].to_numpy(), kind="stable"), :]
    assert list(stored.guides.index) == list(scr.guides.index)
    assert list(stored.samples.index) == list(scr.samples.index)
    assert np.array_equal(stored.X, scr.X) and stored.X.dtype == scr.X.dtype
    for k in scr.layers:
        assert np.array_equal(stored.layers[k], scr.layers[k]), k
    a, b = stored.uns["allele_counts"], scr.uns["allele_counts"]
    assert list(a["allele"].astype(str)) == list(b["allele"].astype(str))
    assert np.array_equal(a.iloc[:, 2:].to_numpy(), b.iloc[:, 2:].to_numpy())


@needs_reference
def test_group_tree_and_attributes():
    """anndata's on-disk schema as the reader sees it: encoding attributes, categorical columns, nested groups."""
    f = h5lite.File(f"{REF_DATA}/var_mini_screen.h5ad")
    assert {"X", "layers", "obs", "var", "uns"} <= set(f.keys())
    assert f["obs"].attrs["encoding-type"] == "dataframe"
    assert f["X"].read().shape == (30, 10)
    listing = "\n".join(h5lite.tree(f))
    assert "layers" in listing and "allele_counts" in listing
    with pytest.raises(KeyError):
        f["no_such_member"]
