"""Where the fp32 alpha_pi error of the reference's var_mini screen comes from: the fused step in float32 and
float64, worst elements with their concentrations and draws.  GPU diagnostic; prints JSON lines."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from crispr_bean_b200.svi import SviEngine  # noqa: E402
from tests.fp32_floor import reference_fp32_floor  # noqa: E402
from tests.test_reference_golden import edit_perm, group, load_case, to_ours  # noqa: E402

dev = torch.device("cuda:0")
name = sys.argv[1] if len(sys.argv) > 1 else "real_var_mini_mixture"
z, data = load_case(name)
truth, floor = reference_fp32_floor(name)
perm = edit_perm(z, data)
noise = {k: torch.as_tensor(to_ours(v, perm, k)) for k, v in group(z, "native/noise/").items() if "/" not in k}
ref = np.asarray(truth["grads"]["alpha_pi"]).reshape(-1, 2)
scale = np.maximum(np.abs(ref), 1e-3 * np.abs(ref).max())
for label, dtype in (("f32", torch.float32), ("f64", torch.float64)):
    eng = SviEngine(data, "MixtureNormal", dev, dtype=dtype, num_steps=4)
    got = eng.gradients(noise)["alpha_pi"].detach().double().cpu().numpy().reshape(-1, 2)
    err = np.abs(got - ref) / scale
    order = np.argsort(-err.max(1))[:4]
    rows = []
    for g in order:
        al = eng.alpha_u[g].exp().double().cpu().numpy() if eng.alpha_u.dim() == 2 else eng.alpha_u.view(-1, 2)[g].exp().double().cpu().numpy()
        pa0 = float(torch.as_tensor(data.pi_a0)[g])
        pi = noise["pi"].reshape(-1, data.n_guides, 2)[:, g].double().numpy()
        rows.append({"g": int(g), "err": err[g].tolist(), "ref": ref[g].tolist(), "got": got[g].tolist(), "alpha": al.tolist(), "pi_a0": pa0,
                     "conc": (al / al.sum() * pa0).tolist(), "pi": pi.tolist(), "mask": data.repguide_mask[:, g].tolist()})
    print(json.dumps({"engine": label, "max_err": float(err.max()), "worst": rows}))
