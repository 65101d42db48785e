"""INTEGRATION.md section A, executed: the reference's OWN `MixtureNormalModel` with its count-likelihood block replaced by one
`pyro.factor` over a `count_log_likelihood(data, mu, sd, pi)` callable -- the `torch.autograd.Function` seam of the north_star.

The reference source is read in place (never copied into the repo): the function's text is taken with `inspect`, everything
from the first `with replicate_plate:` / `with bin_plate as b:` pair (bean/model/model.py:480-547: get_std_normal_prob ->
mixture -> get_alpha x 2 -> DirichletMultinomial x 2) to the end of the function is cut, the two seam lines are appended, and the
result is executed in the reference module's own namespace.  TEST INFRASTRUCTURE; needs BEAN_REFERENCE_ROOT.
"""
from __future__ import annotations

import inspect
import textwrap

SEAM_LINES = '''
    ll = _B200_COUNT_LL(data, mu, sd, pi)
    pyro.factor("guide_counts", ll)
'''


def patched_mixture_normal_model(ns, count_ll):
    """-> the reference's MixtureNormalModel with the DM block swapped for pyro.factor(count_ll(data, mu, sd, pi))."""
    src = textwrap.dedent(inspect.getsource(ns.model.MixtureNormalModel))
    marker = "    with replicate_plate:\n        with bin_plate as b:"
    assert src.count(marker) == 1, "reference layout changed: the likelihood block is no longer where INTEGRATION.md says"
    head = src[: src.index(marker)]
    assert "get_alpha" not in head and "DirichletMultinomial" not in head  # the whole likelihood is in the part cut away
    scope = dict(vars(ns.model))
    scope["_B200_COUNT_LL"] = count_ll
    exec(compile(head + SEAM_LINES, "<MixtureNormalModel + B200 seam>", "exec"), scope)
    return scope["MixtureNormalModel"]
