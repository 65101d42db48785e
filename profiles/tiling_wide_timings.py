"""The fused tiling step against the site-kernel engine (`generic.TilingSviEngine`) on screens with more than 32 alleles per
guide: ms per SVI step of each, and ms per launch of `tiling_wide_kernel` alone, on
  - tiling_real_mini: the reference's raw tiling screen (30 guides x 231 alleles, 2 replicates, 5 bins; tests/golden);
  - a user-sized synthetic screen: about 2,000 guides x 200 alleles x 4 replicates.

    python profiles/tiling_wide_timings.py [--steps 200] [--warmup 50] [--guides 2000] [--out profiles/tiling_wide_timings.json]

Step times: CUDA events around `steps` steps after `warmup` steps (float32, both engines in the same process, alternating).
Kernel time: torch.profiler's device time of `tiling_wide_kernel` over `steps` fused steps, in a separate pass.  The card's
name and power limit are read in the same run and written beside the numbers.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from crispr_bean_b200.data_class import TilingSortingReporterScreenData  # noqa: E402
from crispr_bean_b200.generic import TilingSviEngine  # noqa: E402
from crispr_bean_b200.synth import make_tiling_screen  # noqa: E402
from crispr_bean_b200.tiling_fused import TilingFusedEngine  # noqa: E402


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                         capture_output=True, text=True)
    return out.stdout.strip() or torch.cuda.get_device_name(0)


def screens(guides):
    from tests.test_reference_golden import load_case

    _, real = load_case("tiling_real_mini")
    yield "tiling_real_mini", real
    for g in guides:  # about 200 alleles per guide (at most 290; 205 at 2,000 guides), 4 replicates
        scr = make_tiling_screen(n_guides=g, window=48, max_alleles=290, n_reps=4, seed=7)
        yield f"synthetic_{g}g", TilingSortingReporterScreenData(scr, control_can_be_selected=True, allele_df_key="allele_counts")


def ms_per_step(eng, steps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    eng.run(steps)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / steps


def kernel_ms(eng, steps, name="tiling_wide_kernel"):
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eng.run(steps)
        torch.cuda.synchronize()
    times = [e.device_time_total for e in prof.events() if name in e.name and e.device_time_total > 0]
    return (sum(times) / len(times) / 1000.0, len(times)) if times else (None, 0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--guides", default="2000", help="comma-separated guide counts of the synthetic screens")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "tiling_wide_timings.json"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "timings need a CUDA device"
    dev = torch.device("cuda:0")
    res = {"card": card(), "dtype": "float32", "steps": args.steps, "warmup": args.warmup, "screens": {}}
    n = args.warmup + args.repeats * args.steps + args.steps
    for label, data in screens([int(g) for g in args.guides.split(",")]):
        fused = TilingFusedEngine(data, dev, dtype=torch.float32, num_steps=n)
        sites = TilingSviEngine(data, dev, dtype=torch.float32, num_steps=n)
        fused.run(args.warmup)
        sites.run(args.warmup)
        torch.cuda.synchronize()
        t_f, t_s = [], []
        for _ in range(args.repeats):  # alternating, so that both see the same machine
            t_s.append(ms_per_step(sites, args.steps))
            t_f.append(ms_per_step(fused, args.steps))
        k_ms, k_n = kernel_ms(fused, args.steps)
        row = {"guides": data.n_guides, "alleles": int(data.n_max_alleles), "reps": data.n_reps, "edits": int(data.n_edits),
               "site_kernel_ms_per_step": t_s, "fused_ms_per_step": t_f, "speedup_median": sorted(t_s)[len(t_s) // 2] / sorted(t_f)[len(t_f) // 2],
               "tiling_wide_kernel_ms_per_launch": k_ms, "kernel_launches_profiled": k_n,
               "fused_last_loss": float(fused.loss[fused.step - 1]), "site_kernel_last_loss": float(sites.losses()[-1])}
        res["screens"][label] = row
        print(label, json.dumps(row), flush=True)
        del fused, sites
        torch.cuda.empty_cache()
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
