"""Regenerate tests/golden/* (needs a checkout of the original project named by BEAN_REFERENCE_ROOT, tests/refharness).

1. `var_mini.npz`: the only count fixture of the reference that is readable without anndata/h5py --
   tests/data/var_mini_{guides,samples,counts}.csv (30 guides x 2 replicates x 5 conditions) -- stored as
   plain arrays (fixture DATA, no reference source code).
2. `var_mini_oracle.json`: frozen oracle outputs on that fixture with fixed injected noise
   (Normal model, the `--uniform-edit` path tests/test_create.py:29 runs on exactly these CSVs, and the
   ControlNormal model).  The reference asserts no numbers for this path ("parity unpinned"), so these
   values pin the ORACLE against silent drift, not against pyro.
3. `synthetic_oracle.json`: frozen oracle ELBO / site values for a small seeded synthetic MixtureNormal
   screen (reporter layers), same purpose.

    python tests/golden/make_golden.py
"""
import json
import os
import sys

import numpy as np
import pandas as pd
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from tests.refharness import REFERENCE_ROOT  # noqa: E402

REF = os.path.join(REFERENCE_ROOT, "tests", "data")


def main():
    from tests.helpers import (load_var_mini, fixed_noise, oracle_loss_and_grads, make_small_mixture_data)

    guides = pd.read_csv(f"{REF}/var_mini_guides.csv", index_col=0)
    guides = guides.loc[:, ~guides.columns.duplicated()]
    samples = pd.read_csv(f"{REF}/var_mini_samples.csv", index_col=0)
    counts = pd.read_csv(f"{REF}/var_mini_counts.csv", index_col=0).loc[guides.index, samples.index]
    np.savez_compressed(
        f"{HERE}/var_mini.npz",
        counts=counts.to_numpy().astype(np.float32),
        guide_names=guides.index.to_numpy().astype(str),
        target=guides["target"].to_numpy().astype(str),
        target_group=guides["target_group"].to_numpy().astype(str),
        sample_names=samples.index.to_numpy().astype(str),
        condition=samples["condition"].to_numpy().astype(str),
        replicate=samples["replicate"].to_numpy().astype(str),
        lower_quantile=samples["lower_quantile"].to_numpy().astype(np.float64),
        upper_quantile=samples["upper_quantile"].to_numpy().astype(np.float64),
    )
    out = {}
    data = load_var_mini()
    for model in ("Normal", "ControlNormal"):
        noise = fixed_noise(model, data, seed=7)
        res = oracle_loss_and_grads(model, data, noise, dtype=torch.float64, use_bcmatch=False)
        out[model] = {"loss": res["loss"], "grad_abs_sum": {k: float(v.abs().sum()) for k, v in res["grads"].items()},
                      "ll_guide_counts_sum": float(res["aux"]["ll_guide_counts"].sum())}
    json.dump(out, open(f"{HERE}/var_mini_oracle.json", "w"), indent=1, sort_keys=True)

    data = make_small_mixture_data()
    noise = fixed_noise("MixtureNormal", data, seed=11)
    res = oracle_loss_and_grads("MixtureNormal", data, noise, dtype=torch.float64)
    syn = {"loss": res["loss"], "grad_abs_sum": {k: float(v.abs().sum()) for k, v in res["grads"].items()},
           "ll_guide_counts_sum": float(res["aux"]["ll_guide_counts"].sum()),
           "ll_guide_bcmatch_counts_sum": float(res["aux"]["ll_guide_bcmatch_counts"].sum())}
    json.dump({"MixtureNormal": syn}, open(f"{HERE}/synthetic_oracle.json", "w"), indent=1, sort_keys=True)
    print("wrote", os.listdir(HERE))


if __name__ == "__main__":
    main()
