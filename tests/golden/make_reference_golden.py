"""Golden vectors computed by the REFERENCE's own source (run in the build container only).

    python tests/golden/make_reference_golden.py          # writes tests/golden/ref_*.npz

The reference's unmodified files are imported in place from BEAN_REFERENCE_ROOT through tests/refharness
(bean/preprocessing/data_class.py + get_alpha0.py + get_pi_alpha0.py for the tensors; bean/model/model.py,
survival_model.py, utils.py, run.py for the programs).  pyro-ppl cannot be installed here, so the programs
run on tests/refharness/pyro -- a restatement of the handful of pyro primitives they call (see its
docstring).  What the vectors therefore pin: the tensoriser, the site lists / masks / shapes / formulas of every
model-guide pair, torch's distributions and `_dirichlet_grad`, and the ClippedAdam trajectory of
`run_inference` -- against the reference's CODE; pyro's own handler semantics stay restated.
"""
import copy
import os
import sys
import warnings
from functools import partial

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
warnings.filterwarnings("ignore")

from tests.refharness import REFERENCE_ROOT, load_reference  # noqa: E402
from tests.refharness import golden as G  # noqa: E402


def sorting_cases(ns):
    from crispr_bean_b200.synth import make_sorting_screen
    from tests.helpers import var_mini_screen

    m, dc = ns.model, ns.data_class
    c1 = var_mini_screen()
    c1 = c1[np.argsort(c1.guides["target"].to_numpy(), kind="stable"), :]  # prepare_bdata sorts guides by target
    c1.samples["mask"] = 1
    c1_kw = dict(condition_column="condition", control_condition="bulk", control_can_be_selected=True)
    small = make_sorting_screen(12, 4, n_reps=3, seed=3, n_negctrl_guides=6, depth=120.0, accessibility=True)
    wide = make_sorting_screen(10, 5, n_reps=8, seed=5, depth=300.0)  # c5 row shape (8 replicates) + bulk pseudo-bin
    ragged = make_sorting_screen(9, "lognormal", n_reps=2, seed=8, depth=25.0, n_negctrl_guides=3)  # low depth: masked rows
    rep_kw = dict(control_can_be_selected=True)
    cov = make_sorting_screen(10, 4, n_reps=4, seed=14, depth=150.0)  # two 0/1 sample covariates over 4 replicates
    cov.samples["cell_line"] = [str(int(r[3:]) % 2) for r in cov.samples["replicate"]]
    cov.samples["batch"] = [str(int(int(r[3:]) >= 2)) for r in cov.samples["replicate"]]
    cov.uns["sample_covariates"] = ["cell_line", "batch"]
    return [
        ("normal_covariates", cov, dc.VariantSortingScreenData, rep_kw, partial(m.NormalModel, use_bcmatch=False), m.NormalGuide,
         "Normal", dict(use_bcmatch=False)),
        # name, screen, data class, data kwargs, model, guide, oracle model name, oracle kwargs
        ("normal_c1", c1, dc.VariantSortingScreenData, c1_kw, partial(m.NormalModel, use_bcmatch=False), m.NormalGuide,
         "Normal", dict(use_bcmatch=False)),
        ("control_normal_c1", c1, dc.VariantSortingScreenData, c1_kw, partial(m.ControlNormalModel, use_bcmatch=False),
         partial(m.ControlNormalGuide, use_bcmatch=False), "ControlNormal", dict(use_bcmatch=False)),
        ("mixture_small", small, dc.VariantSortingReporterScreenData, rep_kw, m.MixtureNormalModel, m.MixtureNormalGuide,
         "MixtureNormal", {}),
        ("mixture_wide8", wide, dc.VariantSortingReporterScreenData, rep_kw, m.MixtureNormalModel, m.MixtureNormalGuide,
         "MixtureNormal", {}),
        ("mixture_ragged_lowdepth", ragged, dc.VariantSortingReporterScreenData, rep_kw, m.MixtureNormalModel,
         m.MixtureNormalGuide, "MixtureNormal", {}),
        ("mixture_acc_fitnoise", small, dc.VariantSortingReporterScreenData, dict(rep_kw, accessibility_col="accessibility"),
         partial(m.MixtureNormalModel, scale_by_accessibility=True),
         partial(m.MixtureNormalGuide, scale_by_accessibility=True, fit_noise=True), "MixtureNormal",
         dict(scale_by_accessibility=True, fit_noise=True)),
        ("mixture_acc_priornoise", small, dc.VariantSortingReporterScreenData, dict(rep_kw, accessibility_col="accessibility"),
         partial(m.MixtureNormalModel, scale_by_accessibility=True),
         partial(m.MixtureNormalGuide, scale_by_accessibility=True, fit_noise=False), "MixtureNormal",
         dict(scale_by_accessibility=True, fit_noise=False)),
        ("mixture_prior_params", small, dc.VariantSortingReporterScreenData, rep_kw,
         partial(m.MixtureNormalModel, prior_params={"mu_loc": 0.1, "mu_scale": 2.0}), m.MixtureNormalGuide,
         "MixtureNormal", dict(prior_params={"mu_loc": 0.1, "mu_scale": 2.0})),
        ("mixture_prior_tensors", small, dc.VariantSortingReporterScreenData, rep_kw, "PRIOR_TENSORS", m.MixtureNormalGuide,
         "MixtureNormal", "PRIOR_TENSORS"),
        ("normal_bcmatch", small, dc.VariantSortingScreenData, dict(rep_kw, use_bcmatch=True),
         partial(m.NormalModel, use_bcmatch=True), m.NormalGuide, "Normal", dict(use_bcmatch=True)),
    ]


def survival_cases(ns):
    from crispr_bean_b200.synth import make_survival_screen

    m, dc = ns.survival_model, ns.data_class
    scr = make_survival_screen(10, 4, n_reps=3, seed=4, n_negctrl_guides=5, depth=150.0)
    kw = dict(condition_column="condition", time_column="time", control_condition="D7")
    negctrl = [0, 1, 2, 3, 4]  # what cli/run.py:98-101 passes as negctrl_guide_idx
    return [
        ("survival_normal", scr, dc.VariantSurvivalScreenData, dict(kw, negctrl_guide_idx=negctrl),
         partial(m.NormalModel, use_bcmatch=False), m.NormalGuide, "Normal", dict(use_bcmatch=False)),
        # without negctrl_guide_idx the reference's `mu[None, :] = 0.0` zeroes EVERY guide's growth rate (survival_model.py:59-60)
        ("survival_normal_no_negctrl_idx", scr, dc.VariantSurvivalScreenData, kw,
         partial(m.NormalModel, use_bcmatch=False), m.NormalGuide, "Normal", dict(use_bcmatch=False)),
        ("survival_normal_bcmatch", scr, dc.VariantSurvivalScreenData, dict(kw, negctrl_guide_idx=negctrl, use_bcmatch=True),
         partial(m.NormalModel, use_bcmatch=True), m.NormalGuide, "Normal", dict(use_bcmatch=True)),
        ("survival_control_normal", scr, dc.VariantSurvivalScreenData, kw, partial(m.ControlNormalModel, use_bcmatch=False),
         partial(m.ControlNormalGuide, use_bcmatch=False), "ControlNormal", dict(use_bcmatch=False)),
        ("survival_mixture", scr, dc.VariantSurvivalReporterScreenData, kw, m.MixtureNormalModel, m.MixtureNormalGuide,
         "MixtureNormal", {}),
        ("survival_mixture_control_d0", scr, dc.VariantSurvivalReporterScreenData, dict(kw, control_condition="D0"),
         m.MixtureNormalModel, m.MixtureNormalGuide, "MixtureNormal", {}),
        ("survival_mixture_acc", make_survival_screen(10, 4, n_reps=3, seed=4, n_negctrl_guides=5, depth=150.0, accessibility=True),
         dc.VariantSurvivalReporterScreenData, dict(kw, accessibility_col="accessibility"),
         partial(m.MixtureNormalModel, scale_by_accessibility=True), partial(m.MixtureNormalGuide, scale_by_accessibility=True, fit_noise=True),
         "MixtureNormal", dict(scale_by_accessibility=True, fit_noise=True)),
    ]


def tiling_cases(ns):
    from crispr_bean_b200.synth import make_tiling_screen

    m, dc = ns.model, ns.data_class
    out = []
    for name, kw in (("tiling_small", dict(n_guides=40, n_reps=3, seed=2)), ("tiling_wide", dict(n_guides=30, n_reps=4, max_alleles=7, seed=6))):
        scr = make_tiling_screen(**kw)
        out.append((name, scr, dc.TilingSortingReporterScreenData, dict(control_can_be_selected=True, allele_df_key="allele_counts"),
                    partial(m.MultiMixtureNormalModel, scale_by_accessibility=False, use_bcmatch=(True,)),
                    partial(m.MultiMixtureNormalGuide, scale_by_accessibility=False, fit_noise=True), "MultiMixtureNormal", {}))
    acc = make_tiling_screen(n_guides=36, n_reps=3, seed=9, accessibility=True)
    out.append(("tiling_acc", acc, dc.TilingSortingReporterScreenData,
                dict(control_can_be_selected=True, allele_df_key="allele_counts", accessibility_col="accessibility"),
                partial(m.MultiMixtureNormalModel, scale_by_accessibility=True, use_bcmatch=(True,)),
                partial(m.MultiMixtureNormalGuide, scale_by_accessibility=True, fit_noise=True), "MultiMixtureNormal",
                dict(scale_by_accessibility=True, fit_noise=True)))
    # survival tiling (survival_model.py:427-626 / :759-833)
    sm = ns.survival_model
    surv = make_tiling_screen(n_guides=36, n_reps=3, seed=10, accessibility=True, as_survival=True)
    skw = dict(condition_column="condition", time_column="time", control_condition="D0", allele_df_key="allele_counts")
    out.append(("survival_tiling", surv, dc.TilingSurvivalReporterScreenData, skw,
                partial(sm.MultiMixtureNormalModel, use_bcmatch=(True,)), partial(sm.MultiMixtureNormalGuide, fit_noise=True),
                "MultiMixtureNormal", {}))
    out.append(("survival_tiling_acc", surv, dc.TilingSurvivalReporterScreenData, dict(skw, accessibility_col="accessibility"),
                partial(sm.MultiMixtureNormalModel, scale_by_accessibility=True, use_bcmatch=(True,)),
                partial(sm.MultiMixtureNormalGuide, scale_by_accessibility=True, fit_noise=True), "MultiMixtureNormal",
                dict(scale_by_accessibility=True, fit_noise=True)))
    return out


def real_cases(ns):
    """The reference's own test screens (tests/data/*.h5ad, the inputs of its tests/test_run.py), read with the
    repo's HDF5 reader and prepared as cli/run.py does (guides sorted by target, negative controls from
    `target_group`).  The screens travel inside the fixtures, so the tests never open the original project."""
    from crispr_bean_b200.screen import read_h5ad

    ref_data = os.path.join(REFERENCE_ROOT, "tests", "data") + os.sep
    m, sm, dc = ns.model, ns.survival_model, ns.data_class

    def load(name):
        scr = read_h5ad(ref_data + name + ".h5ad")
        if "target" in scr.guides.columns:
            scr = scr[np.argsort(scr.guides["target"].to_numpy(), kind="stable"), :]
        scr.samples["mask"] = 1
        for key in ("edit_counts",):  # not read by `bean run`; keeps the fixtures small
            scr.uns.pop(key, None)
        return scr

    var, til = load("var_mini_screen"), load("tiling_mini_screen")
    # `--scale-by-acc --acc-bw-path tests/data/accessibility_signal.bw` (tests/test_run.py:85): the signal is looked up with
    # this repo's bigWig reader and handed to BOTH tensorisers as a guide column (the reference's own pyBigWig wrapper cannot
    # run here); tests/test_bigwig_accessibility.py ties that lookup to the reference's per-guide function
    from tests.support.accessibility import get_accessibility_guides

    til_acc = til.copy()
    til_acc.guides["accessibility"] = get_accessibility_guides(ref_data + "accessibility_signal.bw", til_acc.guides).numpy()
    svar, stil = load("survival_var_mini_screen"), load("survival_tiling_mini_screen")
    sort_kw = dict(condition_column="condition", control_condition="bulk", control_can_be_selected=True)
    surv_kw = dict(condition_column="condition", time_column="time", control_condition="D7", control_can_be_selected=True)
    negctrl = np.where(svar.guides["target_group"].map(lambda s: s.lower()) == "negctrl")[0].tolist()
    til_kw = dict(allele_df_key="allele_counts", control_guide_tag=None)
    return [
        # tests/test_run.py: `bean run sorting variant ... --uniform-edit` / default / `--fit-negctrl`
        ("real_var_mini_normal", var, dc.VariantSortingScreenData, sort_kw, partial(m.NormalModel, use_bcmatch=False), m.NormalGuide,
         "Normal", dict(use_bcmatch=False)),
        ("real_var_mini_mixture", var, dc.VariantSortingReporterScreenData, sort_kw, m.MixtureNormalModel, m.MixtureNormalGuide,
         "MixtureNormal", {}),
        ("real_var_mini_control_normal", var, dc.VariantSortingScreenData, sort_kw, partial(m.ControlNormalModel, use_bcmatch=False),
         partial(m.ControlNormalGuide, use_bcmatch=False), "ControlNormal", dict(use_bcmatch=False)),
        # `bean run sorting tiling ... --allele-df-key allele_counts --control-guide-tag None`
        ("tiling_real_mini", til, dc.TilingSortingReporterScreenData, dict(sort_kw, **til_kw),
         partial(m.MultiMixtureNormalModel, scale_by_accessibility=False, use_bcmatch=(True,)),
         partial(m.MultiMixtureNormalGuide, scale_by_accessibility=False, fit_noise=True), "MultiMixtureNormal", {}),
        ("tiling_real_mini_acc", til_acc, dc.TilingSortingReporterScreenData, dict(sort_kw, accessibility_col="accessibility", **til_kw),
         partial(m.MultiMixtureNormalModel, scale_by_accessibility=True, use_bcmatch=(True,)),
         partial(m.MultiMixtureNormalGuide, scale_by_accessibility=True, fit_noise=True), "MultiMixtureNormal",
         dict(scale_by_accessibility=True, fit_noise=True)),
        # `bean run survival variant ... --control-condition=D7` (+ --uniform-edit)
        ("survival_real_var_normal", svar, dc.VariantSurvivalScreenData, dict(surv_kw, negctrl_guide_idx=negctrl),
         partial(sm.NormalModel, use_bcmatch=False), sm.NormalGuide, "Normal", dict(use_bcmatch=False)),
        ("survival_real_var_mixture", svar, dc.VariantSurvivalReporterScreenData, dict(surv_kw, negctrl_guide_idx=negctrl),
         sm.MixtureNormalModel, sm.MixtureNormalGuide, "MixtureNormal", {}),
        ("survival_tiling_real_mini", stil, dc.TilingSurvivalReporterScreenData, dict(surv_kw, control_condition="D0", **til_kw),
         partial(sm.MultiMixtureNormalModel, use_bcmatch=(True,)), partial(sm.MultiMixtureNormalGuide, fit_noise=True),
         "MultiMixtureNormal", {}),
    ]


def with_allele_objects(ns, screen):
    """The reference's tiling tensoriser works on `Allele` objects (bean/framework/Edit.py); the stored screen and
    our tensoriser hold their string form."""
    scr = copy.deepcopy(screen)
    for key, tbl in scr.uns.items():
        if hasattr(tbl, "columns") and "allele" in tbl.columns:
            tbl = tbl.copy()
            tbl["allele"] = tbl["allele"].map(ns.edit.Allele.from_str)
            scr.uns[key] = tbl
    return scr


def write_case(ns, name, screen, cls, data_kw, model, guide, oracle_model, oracle_kw, n_traj=0):
    data = cls(with_allele_objects(ns, screen), **data_kw)
    arrays = dict(G.screen_to_arrays(screen))
    if isinstance(model, str) and model == "PRIOR_TENSORS":
        # per-variant priors as `bean build-prior` writes them and run.py:_check_prior_params reshapes them: (T, 1) tensors
        g = torch.Generator().manual_seed(77)
        T = data.n_targets
        prior = {"mu_loc": 0.3 * torch.randn((T, 1), generator=g, dtype=torch.float64),
                 "mu_scale": 0.5 + torch.rand((T, 1), generator=g, dtype=torch.float64),
                 "sd_loc": 0.05 * torch.randn((T, 1), generator=g, dtype=torch.float64),
                 "sd_scale": 0.01 + 0.05 * torch.rand((T, 1), generator=g, dtype=torch.float64)}
        model = partial(ns.model.MixtureNormalModel, prior_params=prior)
        oracle_kw = {"prior_params": "FROM_FIXTURE"}
        arrays.update({f"prior/{k}": v.numpy() for k, v in prior.items()})
    if hasattr(data, "edit_index"):  # set-iteration order of the reference: a labelling, stored so tests can align to it
        keys = sorted(data.edit_index, key=data.edit_index.get)
        arrays["meta/edit_index_keys"] = np.asarray(keys).astype(str)
    arrays.update({f"data/{k}": v for k, v in G.data_tensors(data).items()})
    arrays["meta/data_class"] = np.asarray(cls.__name__)
    arrays["meta/data_kwargs"] = np.asarray(repr(data_kw))
    arrays["meta/oracle_model"] = np.asarray(oracle_model)
    arrays["meta/oracle_kwargs"] = np.asarray(repr(oracle_kw))
    for tag, dtype in (("f64", torch.float64), ("native", torch.float32)):
        out, noise = G.reference_loss_and_grads(ns.pyro, model, guide, data, seed=11, dtype=dtype)
        arrays.update({f"{tag}/{k}": v for k, v in out.items()})
        arrays.update({f"{tag}/{k}": v for k, v in noise.items()})
    if n_traj:
        arrays.update(trajectory(ns, model, guide, data, n_traj))
    path = os.path.join(HERE, f"ref_{name}.npz")
    np.savez_compressed(path, **arrays)
    print(f"{name:28s} f64 loss {float(arrays['f64/loss']):.10g}  native loss {float(arrays['native/loss']):.10g}  "
          f"{os.path.getsize(path) / 1024:.1f} KiB")


def trajectory(ns, model, guide, data, n_steps):
    """`run_inference` of the reference (bean/model/run.py:347-396), float64, recording every step's guide draws."""
    pyro = ns.pyro
    rec = []

    def recording_guide(d):
        tr = pyro.poutine.trace(guide).get_trace(d)  # inner trace: sees the same messages as SVI's own
        rec.append({k: v.double().numpy() for k, v in G.noise_from_guide_trace(pyro, tr).items()})

    def recording_model(d):
        tr = pyro.poutine.trace(model).get_trace(d)
        site = tr.nodes.get("mu_negctrl")  # survival MixtureNormal: model-only latent, fresh prior draw every step
        if site is not None and not site["is_observed"]:
            rec[-1]["eps_negctrl"] = ((site["value"] - site["fn"].loc) / site["fn"].scale).detach().double().numpy()

    old = torch.get_default_dtype()
    torch.set_default_dtype(torch.float64)
    try:
        torch.manual_seed(23)
        store, hist = ns.run.run_inference(recording_model, recording_guide, G.cast_floats(data, torch.float64), num_steps=n_steps)
    finally:
        torch.set_default_dtype(old)
        torch.autograd.set_detect_anomaly(False)
    out = {"traj/loss": np.asarray(hist["loss"], dtype=np.float64), "traj/n_steps": np.asarray(n_steps)}
    for k, v in hist["params"].items():
        out[f"traj/param/{k}"] = v.double().numpy()
    for k in rec[0]:
        out[f"traj/noise/{k}"] = np.stack([r[k] for r in rec])
    return out


def result_table_golden(ns):
    """The reference's `write_result_table` (bean/model/readwrite.py, real code) on fixed synthetic parameters."""
    import tempfile

    from tests.test_result_table import CASES, run

    with tempfile.TemporaryDirectory() as tmp:
        table, _ = run(ns.readwrite.write_result_table, CASES[0], tmp)
    table.to_csv(os.path.join(HERE, "ref_result_table.csv"), float_format="%.17g")
    print("ref_result_table.csv", table.shape)


def main():
    if os.environ.get("PYTHONHASHSEED") != "0":
        # the reference numbers tiling edits in set-iteration order (string hashes): pin it so the vectors are reproducible
        os.environ["PYTHONHASHSEED"] = "0"
        os.execv(sys.executable, [sys.executable] + sys.argv)
    ns = load_reference()
    if not sys.argv[1:]:
        result_table_golden(ns)
    traj = ("mixture_small", "normal_c1", "control_normal_c1", "mixture_acc_fitnoise", "survival_normal", "survival_mixture",
            "tiling_small", "survival_tiling_acc", "normal_covariates",
            "real_var_mini_mixture", "tiling_real_mini", "survival_real_var_mixture")
    only = sys.argv[1:]  # optional: case-name prefixes to regenerate
    for case in sorting_cases(ns) + survival_cases(ns) + tiling_cases(ns) + real_cases(ns):
        if only and not case[0].startswith(tuple(only)):
            continue
        write_case(ns, *case, n_traj=6 if case[0] in traj else 0)


if __name__ == "__main__":
    main()
