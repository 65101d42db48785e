"""Time-to-first-step on the host (SURVEY section 8 row f2): building the `*ScreenData` tensors from a screen.

    python profiles/tensoriser_timings.py            # one JSON line per shape

Mirror (crispr_bean_b200/data_class.py, vectorised, CSR tiling maps) beside the reference's own data classes
(bean/preprocessing/data_class.py: per-guide Python loops, dense allele_to_edit), the latter executed in place
through tests/refharness where BEAN_REFERENCE_ROOT names a checkout of the original.  Equality of the two outputs is
what tests/test_reference_golden.py checks; this script only reports wall-clock seconds on the host CPU.
"""
import copy
import json
import os
import sys
import time
import warnings

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
warnings.filterwarnings("ignore")
import logging  # noqa: E402

logging.disable(logging.CRITICAL)

from crispr_bean_b200 import data_class as dc  # noqa: E402
from crispr_bean_b200.synth import make_sorting_screen, make_tiling_screen  # noqa: E402
from tests.refharness import available, load_reference  # noqa: E402


def timed(fn):
    t0 = time.perf_counter()
    out = fn()
    return out, time.perf_counter() - t0


def main():
    ns = load_reference() if available() else None
    if ns is not None:
        sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "tests", "golden"))
        from make_reference_golden import with_allele_objects
    devnull = open(os.devnull, "w")
    shapes = [("variant sorting, reporter", "sorting", n) for n in (700, 10_000, 200_000)]
    shapes += [("tiling sorting, reporter", "tiling", n) for n in (200, 800, 3000)]
    for label, kind, n in shapes:
        if kind == "sorting":
            scr = make_sorting_screen(n, 5, n_reps=4, seed=1)
            cls, kw = "VariantSortingReporterScreenData", dict(control_can_be_selected=True)
        else:
            scr = make_tiling_screen(n_guides=n, max_alleles=7, n_reps=4, seed=1)
            cls, kw = "TilingSortingReporterScreenData", dict(control_can_be_selected=True, allele_df_key="allele_counts")
        data, t_mine = timed(lambda: getattr(dc, cls)(copy.deepcopy(scr), **kw))
        rec = {"shape": label, "n_guides": int(data.n_guides), "mirror_s": round(t_mine, 3)}
        # (tiling: per-guide Python loops + dense allele_to_edit in the reference)
        if ns is not None and (kind == "sorting" or (kind == "tiling" and n <= 3000)):
            ref_scr = with_allele_objects(ns, scr) if kind == "tiling" else copy.deepcopy(scr)
            stdout, sys.stdout = sys.stdout, devnull  # the reference prints its fits
            try:
                _, t_ref = timed(lambda: getattr(ns.data_class, cls)(ref_scr, **kw))
            finally:
                sys.stdout = stdout
            rec.update(reference_s=round(t_ref, 3), speedup=round(t_ref / t_mine, 1))
        print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
