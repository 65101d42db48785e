"""Per-kernel times of the fused sorting step at c5 (or a smaller workload), early and in steady state.

    python tools/quick_phase.py [--variants 200000] [--burn-in 300] [--steps 20] [--tag name]
Prints one JSON line; CUDA events on the launching stream, each phase timed alone (BeanSviConfig.phases).
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from bench import build_data, time_steps, WORKLOADS  # noqa: E402
from crispr_bean_b200.svi import SviEngine  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", default="c5_genome_scale")
    ap.add_argument("--burn-in", type=int, default=300)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--tag", default="")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    data = build_data(args.workload, seed=101)
    eng = SviEngine(data, "MixtureNormal", dev, dtype=torch.float32, num_steps=args.burn_in + 20 * args.steps + 64, seed=101)
    out = {"tag": args.tag, "workload": args.workload, "guides": data.n_guides}
    for label, burn in (("early", 5), ("steady", args.burn_in)):
        eng.run(max(burn - eng.step, 0))
        eng.run(3)
        full = time_steps(eng, args.steps) / args.steps
        g = time_steps(eng, args.steps, phases=1) / args.steps
        a = time_steps(eng, args.steps, phases=4) / args.steps
        v = time_steps(eng, args.steps, phases=2) / args.steps
        out[label] = {"step_ms": round(full, 4), "guide_ms": round(g, 4), "alpha_ms": round(a, 4), "variant_ms": round(v, 4)}
    out["loss"] = float(eng.loss[eng.step - 1])
    print(json.dumps(out))


if __name__ == "__main__":
    main()
