"""Loader that executes the reference's OWN source files (read in place from a checkout of the original project named by
the environment variable BEAN_REFERENCE_ROOT, never copied) for golden-vector generation and cross-checks.  TEST
INFRASTRUCTURE ONLY; the tests that need it skip without that checkout, the rest of the suite uses the committed vectors.

What is real and what is shimmed:
  real  (unmodified reference code): bean/model/{model,survival_model,utils,run,readwrite}.py,
        bean/preprocessing/{data_class,get_alpha0,get_pi_alpha0,utils}.py, bean/framework/Edit.py, bean/qc/guide_qc.py
  shim  pyro (tests/refharness/pyro: restated effect handlers, Trace_ELBO, ClippedAdam), `bean` top-level
        package (its __init__ imports anndata / perturb_tools, absent here), pyBigWig, perturb_tools (empty)
"""
from __future__ import annotations

import importlib
import os
import sys
import types

REFERENCE_ROOT = os.environ.get("BEAN_REFERENCE_ROOT", "")
_HERE = os.path.dirname(os.path.abspath(__file__))


def available() -> bool:
    return bool(REFERENCE_ROOT) and os.path.isdir(os.path.join(REFERENCE_ROOT, "bean", "model"))


def load_reference():
    """Returns a namespace with the reference modules: .model, .survival_model, .utils, .run, .readwrite,
    .data_class, .get_alpha0, .get_pi_alpha0, and the shim `pyro`."""
    if not available():
        raise RuntimeError(f"reference sources not found under {REFERENCE_ROOT}")
    if "bean" in sys.modules and getattr(sys.modules["bean"], "__refharness__", False):
        return sys.modules["bean"].__refharness_ns__
    if _HERE not in sys.path:
        sys.path.insert(0, _HERE)  # makes `import pyro` resolve to the shim
    import pyro  # noqa: F401

    assert os.path.dirname(os.path.abspath(pyro.__file__)).startswith(_HERE), "a real pyro is importable: use it instead"

    def pkg(name, path):
        m = types.ModuleType(name)
        m.__path__ = [path]
        m.__package__ = name
        sys.modules[name] = m
        return m

    bean = pkg("bean", os.path.join(REFERENCE_ROOT, "bean"))
    bean.__refharness__ = True
    bean.ReporterScreen = object  # only used in annotations (data_class.py:38)
    for sub in ("model", "preprocessing", "framework", "utils"):
        setattr(bean, sub, pkg(f"bean.{sub}", os.path.join(REFERENCE_ROOT, "bean", sub)))
    # bean/qc/guide_qc.py is real code too (prepare_bdata calls its filter_no_info_target); only its perturb_tools import
    # (the outlier-guide QC, out of scope) is given an empty stand-in
    for name in ("perturb_tools", "perturb_tools._qc", "perturb_tools._qc.qc"):
        if name not in sys.modules:
            stub = types.ModuleType(name)
            stub.__path__ = []
            sys.modules[name] = stub
    if not hasattr(sys.modules["perturb_tools._qc.qc"], "get_outlier_guides"):
        sys.modules["perturb_tools._qc.qc"].get_outlier_guides = None
    bean.qc = pkg("bean.qc", os.path.join(REFERENCE_ROOT, "bean", "qc"))
    sys.modules.setdefault("pyBigWig", types.ModuleType("pyBigWig"))

    ns = types.SimpleNamespace(pyro=pyro)
    for attr, mod in [("utils", "bean.model.utils"), ("data_class", "bean.preprocessing.data_class"),
                      ("get_alpha0", "bean.preprocessing.get_alpha0"), ("get_pi_alpha0", "bean.preprocessing.get_pi_alpha0"),
                      ("model", "bean.model.model"), ("survival_model", "bean.model.survival_model"),
                      ("run", "bean.model.run"), ("readwrite", "bean.model.readwrite"), ("edit", "bean.framework.Edit"),
                      ("prep_utils", "bean.preprocessing.utils"), ("guide_qc", "bean.qc.guide_qc")]:
        setattr(ns, attr, importlib.import_module(mod))
    bean.__refharness_ns__ = ns
    return ns
