"""`--acc-bw-path`: the pure-Python bigWig reader (tests/support/bigwig.py) and the guide-accessibility lookup
(tests/support/accessibility.py, mirror of bean/preprocessing/utils.py:70-146).

The reader is checked against what each bigWig says about itself (the header's total summary: covered bases, min, max, sum
of the full-resolution data) on the reference's two tracks, and on a bigWig written here byte by byte; the lookup is
checked against the reference's own `get_accessibility_guides` (real code through tests/refharness) handed this reader in
place of pyBigWig."""
import os
import struct
import sys
import zlib

import numpy as np
import pandas as pd
import pytest
import torch

from tests.support import bigwig
from tests.support.accessibility import _get_accessibility_single, get_accessibility_guides
from tests.refharness import REFERENCE_ROOT, available, load_reference

REF_DATA = os.path.join(REFERENCE_ROOT, "tests", "data")
needs_data = pytest.mark.skipif(not (REFERENCE_ROOT and os.path.isdir(REF_DATA)), reason="reference test data not mounted")


def write_bigwig(path, chroms, sections, compress=True):
    """Minimal bigWig writer (one R-tree leaf node, one chromosome-tree leaf): `sections` = [(chrom id, kind, start, step,
    span, items)], items = (start, end, value) | (start, value) | value for kind 1 | 2 | 3."""
    key_size = max(len(c) for c in chroms)
    blocks, leaves = [], []
    for cid, kind, c_start, step, span, items in sections:
        if kind == 1:
            body = b"".join(struct.pack("<IIf", *it) for it in items)
            lo, hi = items[0][0], items[-1][1]
        elif kind == 2:
            body = b"".join(struct.pack("<If", *it) for it in items)
            lo, hi = items[0][0], items[-1][0] + span
        else:
            body = b"".join(struct.pack("<f", it) for it in items)
            lo, hi = c_start, c_start + step * (len(items) - 1) + span
        raw = struct.pack("<IIIIIBBH", cid, lo, hi, step, span, kind, 0, len(items)) + body
        blocks.append(zlib.compress(raw) if compress else raw)
        leaves.append((cid, lo, cid, hi))
    header_size, summary_off = 64, 64
    chrom_off = summary_off + 40
    chrom_tree = struct.pack("<IIIIQQ", bigwig.CHROM_TREE_MAGIC, len(chroms), key_size, 8, len(chroms), 0) + struct.pack("<BBH", 1, 0, len(chroms))
    for i, (name, size) in enumerate(chroms.items()):
        chrom_tree += name.encode().ljust(key_size, b"\0") + struct.pack("<II", i, size)
    data_off = chrom_off + len(chrom_tree)
    data = struct.pack("<Q", len(blocks))
    offsets, p = [], data_off + 8
    for b in blocks:
        offsets.append(p)
        p += len(b)
    data += b"".join(blocks)
    index_off = data_off + len(data)
    index = struct.pack("<IIQIIIIQII", bigwig.RTREE_MAGIC, 256, len(blocks), 0, 0, len(chroms) - 1, max(chroms.values()), index_off, 1, 0)
    index += struct.pack("<BBH", 1, 0, len(blocks))
    for (c0, b0, c1, b1), off, b in zip(leaves, offsets, blocks):
        index += struct.pack("<IIIIQQ", c0, b0, c1, b1, off, len(b))
    head = struct.pack("<IHHQQQHHQQIQ", bigwig.BIGWIG_MAGIC, 4, 0, chrom_off, data_off, index_off, 0, 0, 0, summary_off, 32768 if compress else 0, 0)
    assert len(head) == header_size
    with open(path, "wb") as f:
        f.write(head + struct.pack("<Qdddd", 0, 0, 0, 0, 0) + chrom_tree + data + index)


@pytest.mark.parametrize("compress", [True, False])
def test_values_of_a_handwritten_bigwig(tmp_path, compress):
    path = str(tmp_path / "t.bw")
    write_bigwig(path, {"chr1": 1000, "chrX": 500}, [
        (0, 1, 0, 0, 0, [(10, 20, 1.5), (20, 25, 2.5), (40, 41, 7.0)]),      # bedGraph
        (0, 2, 0, 0, 3, [(100, 4.0), (110, 5.0)]),                            # variableStep, span 3
        (1, 3, 50, 10, 2, [1.0, 2.0, 3.0]),                                    # fixedStep on chrX: 50-52, 60-62, 70-72
    ], compress=compress)
    bw = bigwig.open(path)
    assert bw.chroms() == {"chr1": 1000, "chrX": 500}
    v = bw.values("chr1", 5, 45)
    want = np.full(40, np.nan)
    want[5:15], want[15:20], want[35] = 1.5, 2.5, 7.0
    assert np.array_equal(v, want, equal_nan=True) and v.dtype == np.float64
    assert np.array_equal(bw.values("chr1", 99, 114), [np.nan, 4, 4, 4] + [np.nan] * 7 + [5, 5, 5, np.nan], equal_nan=True)
    assert np.array_equal(bw.values("chrX", 49, 63), [np.nan, 1, 1] + [np.nan] * 8 + [2, 2, np.nan], equal_nan=True)
    assert np.isnan(bw.values("chrX", 0, 40)).all()  # no block overlaps: all NaN, as pyBigWig
    for bad in (("chr2", 0, 10), ("chr1", -5, 10), ("chr1", 990, 1001), ("chr1", 10, 10)):
        with pytest.raises(bigwig.BigWigError):
            bw.values(*bad)
    assert bw.coverage_summary()["nBasesCovered"] == 10 + 5 + 1 + 6 + 6


def test_not_a_bigwig(tmp_path):
    p = tmp_path / "x.bw"
    p.write_bytes(b"track type=wiggle_0\n" * 10)
    with pytest.raises(bigwig.BigWigError, match="not a bigWig"):
        bigwig.open(str(p))


@needs_data
@pytest.mark.parametrize("name", ["accessibility_signal_chr6.bw", "accessibility_signal.bw"])
def test_reference_tracks_agree_with_their_own_total_summary(name):
    bw = bigwig.open(f"{REF_DATA}/{name}")
    got, want = bw.coverage_summary(), bw.summary
    assert got["nBasesCovered"] == want["nBasesCovered"] > 10_000
    assert got["minVal"] == want["minVal"] and got["maxVal"] == want["maxVal"]
    assert abs(got["sumData"] - want["sumData"]) <= 1e-8 * want["sumData"]


def guides_on_track(bw, chrom, n=12):
    """Guide positions inside, at the edge of and outside the covered part of the track."""
    cid, size = bw._chroms[chrom]
    starts = np.sort(np.concatenate([bw._intervals(off, nb)[1] for off, nb in bw._blocks(cid, 0, size)]))
    picks = starts[np.linspace(0, len(starts) - 1, n - 4).astype(int)]
    pos = [float(s) for s in picks] + [float(starts[0] - 50), 50.0, float(size - 10), np.nan]
    return pd.DataFrame({"genomic_pos": pos, "chrom": chrom}, index=[f"g{i}" for i in range(len(pos))])


@needs_data
@pytest.mark.skipif(not available(), reason="reference sources not mounted")
@pytest.mark.parametrize("name,chrom", [("accessibility_signal_chr6.bw", "chr6"), ("accessibility_signal.bw", "chr19")])
def test_lookup_equals_reference_function_on_this_reader(name, chrom, capsys):
    """The reference's `_get_accessibility_single` (real code) with this repo's reader as the track, guide by guide; its
    `get_accessibility_guides` wrapper cannot run here (`torch.as_tensor(pandas Series)` fails with pandas 3), so the
    median fill is checked against its definition."""
    ns = load_reference()
    path = f"{REF_DATA}/{name}"
    track = bigwig.open(path)
    info = guides_on_track(track, chrom)
    ref = np.asarray([ns.prep_utils._get_accessibility_single(p, track, chrom=chrom, guide_start_pos=0, half_window_size=100)
                      for p in info["genomic_pos"]])
    assert np.isnan(ref).sum() >= 2 and np.isfinite(ref).sum() >= 6  # outside the covered region / NaN position vs inside
    want = torch.as_tensor(ref.copy())
    want[torch.isnan(want)] = torch.nanmedian(want)  # utils.py:143-145
    for frame in (info, info.rename(columns={"chrom": "chr"})):
        mine = get_accessibility_guides(path, frame)
        assert mine.dtype == torch.float64 and torch.equal(mine, want)
    assert (want >= 1.0).all() and want.max() > 1.5
    with pytest.raises(ValueError, match="Cannot retrieve"):
        get_accessibility_guides(path, pd.DataFrame({"genomic_pos": [np.nan, 10.0], "chrom": chrom}))


@needs_data
def test_tiling_data_class_takes_the_track(tmp_path):
    """`bean run sorting tiling ... --scale-by-acc --acc-bw-path tests/data/accessibility_signal.bw` (tests/test_run.py:85):
    the tensoriser fills guide_accessibility from the track for the reference's tiling screen."""
    import ast

    from crispr_bean_b200 import data_class as dc
    from tests.helpers import GOLDEN
    from tests.refharness.golden import screen_from_arrays

    z = np.load(os.path.join(GOLDEN, "ref_tiling_real_mini.npz"))
    kw = ast.literal_eval(str(z["meta/data_kwargs"]))
    dc.ACCESSIBILITY_LOOKUP = get_accessibility_guides
    data = dc.TilingSortingReporterScreenData(screen_from_arrays(z), accessibility_bw_path=f"{REF_DATA}/accessibility_signal.bw", **kw)
    acc = data.guide_accessibility
    assert acc.shape == (data.n_guides,) and torch.isfinite(acc).all() and (acc >= 1).all() and acc.std() > 0


def test_single_position_rules():
    class Track:
        def values(self, chrom, s, e):
            if s < 0:
                raise RuntimeError("Invalid interval bounds!")
            return [0.0, np.nan, 3.0, 8.0][: e - s]

    assert np.isnan(_get_accessibility_single("control", Track())) and np.isnan(_get_accessibility_single(np.nan, Track()))
    assert np.isclose(_get_accessibility_single(2, Track(), half_window_size=2), np.exp(np.mean(np.log([1.0, 4.0, 9.0]))))
    assert np.isnan(_get_accessibility_single(1, Track(), half_window_size=2))  # window starts before the chromosome
    with pytest.raises(ValueError):
        _get_accessibility_single(5, Track(), half_window_size=-1)
