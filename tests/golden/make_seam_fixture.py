"""tests/golden/seam_mixture_small.npz: what the reference's own MixtureNormalModel hands to the B200 likelihood seam.

    python tests/golden/make_seam_fixture.py

Runs the reference program (read in place from BEAN_REFERENCE_ROOT, tests/refharness) with its count-likelihood block replaced by
`pyro.factor("guide_counts", count_ll(data, mu, sd, pi))` (INTEGRATION.md section A; tests/refharness/seam.py) on the screen of
ref_mixture_small.npz with the same seed as that golden case, and records the seam's inputs (mu, sd (G, 2); pi (R, 1, G, 2)),
the value the CPU oracle returns for them and its gradient w.r.t. the three inputs.  tests/test_integration_seam.py checks
(here) that the patched program reproduces the golden loss and gradients and (on the GPU) that the CUDA seam returns the
recorded value and gradients for the recorded inputs.
"""
import ast
import copy
import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
warnings.filterwarnings("ignore")


def run(write=True):
    from oracle import bean_oracle as O
    from tests.refharness import golden as G
    from tests.refharness import load_reference
    from tests.refharness.golden import screen_from_arrays
    from tests.refharness.seam import patched_mixture_normal_model

    ns = load_reference()
    z = np.load(os.path.join(HERE, "ref_mixture_small.npz"))
    data = ns.data_class.VariantSortingReporterScreenData(copy.deepcopy(screen_from_arrays(z)), **ast.literal_eval(str(z["meta/data_kwargs"])))
    rec = {}

    def count_ll(d, mu, sd, pi):
        m, s, p = (t.detach().clone().requires_grad_(True) for t in (mu, sd, pi))
        total, _ = O.sorting_ll_core(d, m, s, p)
        gm, gs, gp = torch.autograd.grad(total, (m, s, p))
        rec.update(mu=mu.detach().numpy().copy(), sd=sd.detach().numpy().copy(), pi=pi.detach().numpy().copy(),
                   ll=np.asarray(float(total)), d_mu=gm.numpy(), d_sd=gs.numpy(), d_pi=gp.numpy())
        return O.sorting_ll_core(d, mu, sd, pi)[0]  # differentiable: the program's own parameters get their gradients

    model = patched_mixture_normal_model(ns, count_ll)
    out, _ = G.reference_loss_and_grads(ns.pyro, model, ns.model.MixtureNormalGuide, data, seed=11, dtype=torch.float64)
    torch.autograd.set_detect_anomaly(False)
    if write:
        np.savez_compressed(os.path.join(HERE, "seam_mixture_small.npz"), **rec, loss=out["loss"])
        print("seam_mixture_small.npz: loss", float(out["loss"]), "golden", float(z["f64/loss"]))
    return z, out, rec


if __name__ == "__main__":
    run()
