#!/usr/bin/env python
"""bench.py -- SVI throughput of the `bean run` hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--scaling strong|weak] [--workload c5_genome_scale] [--impl reference]
                    [--dump-outputs DIR]

One "step" = one complete SVI step (guide sampling + ELBO forward/backward + ClippedAdam) of the MixtureNormal sorting
model over one synthetic screen.  Workload: the configuration BASELINE.json's target is quoted on, c5 = 1M guides x 8
replicates x 4 bins (+ barcode-matched layer, reporter edits).

N > 1 (torchrun, one rank per GPU).  Default `--scaling strong`, the north_star's own configuration: the ONE 1M-guide
screen is split into contiguous variant blocks (`dist.shard_variants`), every rank runs its block, and the per-step
ELBO scalars -- the only quantity of this model that crosses ranks (SURVEY section 8e) -- are all-reduced over NCCL in
batches of <= 100 steps INSIDE the timed region (the reference prints the loss every 100 steps, run.py:378).
`--scaling weak` gives every rank its own 1M-guide screen instead.

`--dump-outputs DIR` (one GPU) writes what the timed steps hand a caller, taken right after the last timed step: the ELBO
loss of every timed step (`DIR/loss.npy`, float64) and the fitted parameters under the reference's names
(`DIR/<name>.npy`, in the engine's dtype).  The screen and the engine's draws are seeded, so two builds run with the
same arguments can be compared array for array.

Prints ONE JSON line (rank 0).  `--impl reference` times the CPU oracle port of the reference path on the box's host
cores at the FULL workload size (pyro is not installable here, so the reference itself cannot run; SURVEY 8c).
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOADS = {
    # name: (n_variants, guides_per_variant, n_reps); sorting: 4 sort bins, bulk used for the reporter only
    "c5_genome_scale": (200_000, 5, 8),
    "c2_ldlc_variant": (690, 5, 4),
    "tiny": (2_000, 5, 8),
    "c5_quarter": (50_000, 5, 8),  # the shard one of four GPUs holds under strong scaling (kernel A/B at that size)
    # BASELINE.json config 4: proliferation / survival variant screen (MixtureNormal survival program), 3 replicates x
    # 3 timepoints (D0, D7, D14; control D7 stays selected), at the c5 guide count so that 1/2/4/8 GPUs have work to split
    "c4_survival": (200_000, 5, 3),
    "c4_survival_small": (690, 5, 3),
}
SURVIVAL = ("c4_survival", "c4_survival_small")
BASELINE_MD_PUBLISHED = None  # BASELINE.md holds no published number for this metric -> vs_baseline null
LOSS_BATCH = 100              # steps per ELBO all-reduce (reference print cadence, bean/model/run.py:378)
GUIDE_PROFILE = os.path.join(ROOT, "profiles", "r2_guide_metrics.txt")  # ncu --set full capture of the dominant kernel
DUMP_LIMIT = 64 << 20         # bytes --dump-outputs may write in all


def algorithmic_bytes_per_guide(R, B, L, guides_per_variant, itemsize=4):
    """HBM bytes the guide kernel must move per guide with every input read once and every output written once
    (SURVEY 8d): counts L*R*B + a0 L + row mask R (u8) + CSR id 4 B + reporter allele counts 2R + pi_a0 1 + alpha_pi 2
    (read) + per-guide (d_mu, d_sd) out 2 + variant params 4/guides-per-variant.  The hand-over to `svi_alpha_kernel`
    is NOT algorithmic (it exists because the step is split in two kernels); it is reported separately."""
    w = itemsize
    return L * R * B * w + L * w + R + 4 + 2 * R * w + w + 2 * w + 2 * w + 4.0 * w / guides_per_variant


def handover_bytes_per_guide(R, itemsize=4):
    """(pi0, pi1, w0, w1) per replicate + 4 concentration gradients, written by the guide kernel, read by the alpha kernel."""
    return (4 * R + 4) * itemsize


def alpha_kernel_bytes_per_guide(R, itemsize=4):
    """`svi_alpha_kernel`: the hand-over records 4R + 4, pi_a0 1, alpha_pi (param, m, v) read + written 12."""
    return (4 * R + 4 + 1 + 12) * itemsize


def build_data(workload, seed):
    from crispr_bean_b200.data_class import VariantSortingReporterScreenData, VariantSurvivalReporterScreenData
    from crispr_bean_b200.synth import make_sorting_screen, make_survival_screen

    nv, gpv, nr = WORKLOADS[workload]
    if workload in SURVIVAL:
        return VariantSurvivalReporterScreenData(make_survival_screen(nv, gpv, n_reps=nr, seed=seed), control_condition="D7")
    scr = make_sorting_screen(nv, gpv, n_reps=nr, seed=seed)
    # 4 sort bins; the bulk sample only feeds the reporter editing-rate sites (see DESIGN.md, "c5")
    return VariantSortingReporterScreenData(scr, control_can_be_selected=False)


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons of one GPU through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:  # pragma: no cover
            self.nv = None

    NAMES = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def run(self):
        if self.nv is None:
            return
        while not self.stop_flag:
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.NAMES.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def time_steps(engine, steps, phases=0):
    """CUDA-event time of `steps` steps on the launching (current) stream, in ms."""
    engine.cfg.phases = phases
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    start.record()
    engine.run(steps)
    stop.record()
    torch.cuda.synchronize()
    engine.cfg.phases = 0
    return start.elapsed_time(stop)


def run_with_loss_exchange(engine, steps, world):
    """`steps` SVI steps; the per-step ELBO scalars are summed over ranks in batches of LOSS_BATCH (one NCCL all-reduce
    of <= 100 doubles per batch, asynchronous, ordered after the batch on the launching stream)."""
    done = 0
    while done < steps:
        n = min(LOSS_BATCH, steps - done)
        losses = engine.run(n)
        if world > 1:
            import torch.distributed as dist

            dist.all_reduce(losses)  # a view of the engine's loss buffer: reduced in place
        done += n


def make_bench_engine(workload, data, dev, dtype, num_steps, seed, off):
    if workload in SURVIVAL:
        from crispr_bean_b200.survival_fused import SurvivalFusedEngine

        return SurvivalFusedEngine(data, dev, dtype=dtype, num_steps=num_steps, seed=seed, guide_offset=off["guide_offset"],
                                   variant_offset=off["variant_offset"])
    from crispr_bean_b200.svi import SviEngine

    return SviEngine(data, "MixtureNormal", dev, dtype=dtype, num_steps=num_steps, seed=seed, guide_offset=off["guide_offset"],
                     variant_offset=off["variant_offset"])


def dump_outputs(path, arrays):
    """Writes every array as `path/<name>.npy`; refuses to write more than DUMP_LIMIT bytes in all."""
    import numpy as np

    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise RuntimeError(f"--dump-outputs: {total} bytes of outputs exceed the {DUMP_LIMIT}-byte limit")
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(path, f"{name}.npy"), a)


def oracle_step_time(data, steps, warmup=1, anomaly=True, max_seconds=240.0):
    """Seconds per SVI step of the CPU oracle (plain-torch restatement of the reference's MixtureNormal program); stops early
    (after at least one timed step) once `max_seconds` have gone by; `max_seconds=None` times exactly `steps` steps."""
    from oracle import bean_oracle as O

    elbo_fn = O.elbo_survival_mixture_normal if getattr(data, "is_survival", False) else O.elbo_mixture_normal
    ps = O.ParamStore()
    opt = O.ClippedAdam(lr=0.01, lrd=0.1 ** (1 / 2000))
    times = []
    torch.autograd.set_detect_anomaly(anomaly)  # the reference switches it on for good (model.py:399; SURVEY App. B6)
    began = time.perf_counter()
    try:
        for t in range(warmup + steps):
            if max_seconds is not None and times and time.perf_counter() - began > max_seconds:
                break
            t0 = time.perf_counter()
            loss, _ = elbo_fn(data, ps)
            ps.zero_grad()
            loss.backward()
            opt.step(ps.unconstrained)
            float(loss.detach())  # the reference syncs the loss every step (run.py:377-380)
            if t >= warmup:
                times.append(time.perf_counter() - t0)
    finally:
        torch.autograd.set_detect_anomaly(False)
    return sum(times) / len(times)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None,
                    help="timed steps (default 100; the reference arm by default stops at --cpu-max-steps steps or after 240 s)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c5_genome_scale", choices=sorted(WORKLOADS))
    ap.add_argument("--scaling", default="strong", choices=["strong", "weak"])
    ap.add_argument("--dtype", default="f32", choices=["f32", "f64"])
    ap.add_argument("--cpu-sample-guides", type=int, default=0, help="0 = the full workload (default)")
    ap.add_argument("--cpu-max-steps", type=int, default=25, help="upper bound on the reference arm's timed steps when --steps is not given")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--full-run-steps", type=int, default=4000, help="length of the complete run timed after the K steps (0 = skip)")
    ap.add_argument("--burn-in", type=int, default=300,
                    help="untimed SVI steps before the timed region: a step gets slower over the first ~300 steps of a run "
                         "(alpha_pi fits the low editing rates, more Dirichlet draws leave the saddle-point regime), so the "
                         "timed steps are taken where a real 2000-step run spends its time")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the losses of the timed steps and the parameters after the last one as DIR/<name>.npy")
    args = ap.parse_args()
    steps_given = args.steps is not None
    args.steps = args.steps if steps_given else 100
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.dump_outputs and (args.impl != "ours" or world > 1):
        ap.error("--dump-outputs needs --impl ours on one GPU")
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    nv, gpv, nr = WORKLOADS[args.workload]
    survival = args.workload in SURVIVAL
    R, B, L = nr, (3 if survival else 4), 2
    program = "MixtureNormal survival (3 timepoints, control D7)" if survival else "MixtureNormal sorting"
    G_total = nv * gpv * (world if args.scaling == "weak" else 1)
    cells_per_step = G_total * R * B
    scaling = args.scaling if world > 1 else "strong"  # at N = 1 both are the same workload
    if args.scaling == "strong":
        shard_txt = f"ONE screen of {nv * gpv} guides / {nv} variants split into {world} contiguous variant block(s) (strong scaling)"
    else:
        shard_txt = f"{world} independent screen(s) of {nv * gpv} guides, one per GPU (weak scaling)"
    # L2 rule: where a rank's step footprint is below twice the L2 (strong scaling at N >= 4) the timed steps are separated by
    # an untimed overwrite of a 256 MB buffer, so that every timed step reads its inputs from HBM
    footprint = 700.0 * nv * gpv / (world if args.scaling == "strong" else 1)
    flush = footprint < 2 * 126e6
    exchange = (f"per-step ELBO scalars all-reduced over NCCL every {LOSS_BATCH} steps" +
                (f" + the {R + 1} library-wide sums of the abundance Dirichlet exchanged EVERY step (through CUDA-IPC peer memory inside "
                 f"the kernels where the steps run many per call; an NCCL all-reduce between the launches where every step is "
                 f"timed on its own)" if survival else "") +
                ", inside the timed region")
    config = {"workload": f"{args.workload}: {program}, {G_total} guides x {R} reps x {B} bins in total, "
                          f"bcmatch layer + reporter edits",
              "l2": (f"per-rank step footprint ~{footprint / 1e6:.0f} MB (~0.7 KB per guide: inputs + parameter state + hand-over scratch); " +
                     ("below 2x the 126 MB L2: a 256 MB buffer is overwritten between timed steps (untimed), every step timed by its own "
                      "CUDA events" if flush else "more than 2x the 126 MB L2: nothing of a previous step survives in cache, no flush")),
              "sharding": shard_txt,
              "exchange": exchange if world > 1 else "none (one GPU)"}

    # ------------------------------------------------------------------------------------------
    if args.impl == "reference":
        if rank != 0:
            return 0
        torch.set_num_threads(os.cpu_count() or 1)
        data = build_data(args.workload, seed=101)
        if args.cpu_sample_guides and args.cpu_sample_guides < data.n_guides:
            data = data[torch.arange(args.cpu_sample_guides)]
        # an explicit --steps is timed in full; by default the arm is capped, as one step of the full workload takes seconds
        steps = args.steps if steps_given else max(1, min(args.steps, args.cpu_max_steps))
        sec = oracle_step_time(data, steps, warmup=max(min(args.warmup, 2), 1), anomaly=True,
                               max_seconds=None if steps_given else 240.0)
        sec_off = oracle_step_time(data, min(steps, 3), warmup=1, anomaly=False)
        cells = data.n_guides * R * B
        value = cells / sec
        sample = (f"{'all' if data.n_guides == nv * gpv else 'first'} {data.n_guides} guides of the workload, {steps if steps_given else f'<= {steps}'} timed SVI steps{'' if steps_given else ' (240 s cap)'} of the "
                  f"plain-torch oracle port on {torch.get_num_threads()} threads, torch anomaly mode ON as the reference leaves it "
                  f"(model.py:399): {sec * 1e3:.0f} ms/step; anomaly mode off: {sec_off * 1e3:.0f} ms/step; pyro itself is not "
                  "installable (no poutine overhead in this number)")
        line = {
            "impl": "reference", "metric": "guide_rep_bin_cells_per_sec", "value": value, "unit": "cells/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3,
            "higher_is_better": True, "scaling": scaling, "vs_baseline": None, "dtype": "f32/f64 mixed (as the reference)",
            "data": "synthetic", "config": config,
            "svi_steps_per_sec": 1.0 / sec, "timed_steps": steps,
            "anomaly_mode_off": {"value": cells / sec_off, "ms_per_step": sec_off * 1e3},
            "cpu_baseline": {"value": value, "unit": "cells/s", "cores": torch.get_num_threads(), "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "cells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
        }
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------------------------------
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=dev)
    from crispr_bean_b200.dist import shard_data

    dtype = torch.float32 if args.dtype == "f32" else torch.float64
    if args.scaling == "strong":
        full = build_data(args.workload, seed=101)  # a0 / pi_a0 / size factors are fitted on the WHOLE screen, then sliced
        data, off = shard_data(full, rank, world)
        del full
    else:
        data = build_data(args.workload, seed=101 + rank)
        off = {"guide_offset": rank * nv * gpv, "variant_offset": rank * nv, "n_guides": nv * gpv, "n_variants": nv}
    G_rank = data.n_guides
    total_steps = args.warmup + args.steps
    burn_in = max(args.burn_in, 0)
    eng = make_bench_engine(args.workload, data, dev, dtype, max(2000, burn_in + 4 * total_steps + 64), 101, off)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return t.item()
        return ms

    # --- device-resident throughput: inputs already in HBM --------------------------------------
    run_with_loss_exchange(eng, burn_in, world)  # untimed: reach the steady-state regime of a long run (see --burn-in)
    run_with_loss_exchange(eng, args.warmup, world)
    scrub = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev) if flush else None
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    if not flush:
        start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        start.record()
        run_with_loss_exchange(eng, args.steps, world)
        stop.record()
        barrier()
        ms_local = start.elapsed_time(stop)
    else:
        evs = []
        for t in range(args.steps):
            scrub.fill_(t & 0xFF)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            losses = eng.run(1)
            if world > 1 and ((t + 1) % LOSS_BATCH == 0 or t + 1 == args.steps):
                lo = eng.step - 1 - (t % LOSS_BATCH)
                dist.all_reduce(eng.loss[lo:eng.step])
            e1.record()
            evs.append((e0, e1))
        barrier()
        ms_local = sum(a.elapsed_time(b) for a, b in evs)
    sampler.stop_flag = True
    sampler.join()
    if args.dump_outputs:  # before the per-kernel timings below advance the engine further
        outputs = {"loss": eng.loss[eng.step - args.steps:eng.step], **eng.params()}
        dump_outputs(args.dump_outputs, {k: v.detach().cpu().numpy() for k, v in outputs.items()})
    ms = max_over_ranks(ms_local)
    steps_per_sec = args.steps / (ms * 1e-3)
    value = cells_per_step * steps_per_sec
    final_loss = float(eng.loss[eng.step - 1].item())

    # --- per-kernel timing for the roofline: each kernel alone, same launches, CUDA events --------
    # sharded survival: whether the library-wide sums travelled through peer memory inside the kernels, and waits that gave up
    peer_exchange = None
    if survival and world > 1:
        peer_exchange = {"used": getattr(eng, "peers", None) is not None, "timeouts": eng.peer_timeouts()}
    ms_guide = max_over_ranks(time_steps(eng, args.steps, phases=1) / args.steps)
    split = getattr(eng, "split", True)
    ms_alpha = max_over_ranks(time_steps(eng, args.steps, phases=4) / args.steps) if split else 0.0
    ms_var = max_over_ranks(time_steps(eng, args.steps, phases=2) / args.steps)
    itemsize = 4 if dtype == torch.float32 else 8
    # survival: + log obs R + gamma R in, gamma R out, q0 (param, m, v) read + written 6, control allele counts as the reporter's
    bytes_launch = (algorithmic_bytes_per_guide(R, B, L, gpv, itemsize) + (3 * R + 6) * itemsize * survival) * G_rank
    handover = handover_bytes_per_guide(R, itemsize) * G_rank if split else 0.0
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "MEASURED_PEAKS.json hbm_gbs (measured copy bandwidth)"
    else:
        peak, peak_src = 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"
    # empirical FP32/SFU ceiling (SURVEY 8d): the Dirichlet-Multinomial row maths alone, operands in registers
    from crispr_bean_b200 import _lib as L_

    sink = torch.empty((G_rank + 127) // 128, device=dev, dtype=torch.float32)
    st = torch.cuda.current_stream(dev).cuda_stream
    for _ in range(3):
        L_.check(L_.lib().bean_row_ceiling_f32(G_rank, R * L, B, sink.data_ptr(), st), "bean_row_ceiling_f32")
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    c0.record()
    for _ in range(20):
        L_.check(L_.lib().bean_row_ceiling_f32(G_rank, R * L, B, sink.data_ptr(), st), "bean_row_ceiling_f32")
    c1.record()
    torch.cuda.synchronize()
    ms_ceiling = c0.elapsed_time(c1) / 20
    # the same maths in the north_star's lane = (row, bin) mapping (4 bins only): the A/B of the two mappings at the maths level
    ms_ceiling_lanes = None
    if B == 4:
        sink2 = torch.empty(4 * torch.cuda.get_device_properties(dev).multi_processor_count, device=dev, dtype=torch.float32)
        for _ in range(3):
            L_.check(L_.lib().bean_row_ceiling_lanes_f32(G_rank, R * L, sink2.data_ptr(), st), "bean_row_ceiling_lanes_f32")
        c0.record()
        for _ in range(20):
            L_.check(L_.lib().bean_row_ceiling_lanes_f32(G_rank, R * L, sink2.data_ptr(), st), "bean_row_ceiling_lanes_f32")
        c1.record()
        torch.cuda.synchronize()
        ms_ceiling_lanes = c0.elapsed_time(c1) / 20
    achieved = bytes_launch / (ms_guide * 1e-3) / 1e9
    # DRAM traffic, instruction count and pipe utilisation of one launch, from the committed ncu --set full capture
    traffic = warp_inst = None
    note = "no ncu capture of this configuration committed"
    if os.path.exists(GUIDE_PROFILE) and args.workload == "c5_genome_scale" and dtype == torch.float32 and world == 1:  # noqa: E501
        m = {}
        for ln in open(GUIDE_PROFILE):
            if " = " in ln:
                key, val = ln.rsplit(" = ", 1)
                try:
                    m[key.split(" [")[0].strip()] = float(val)
                except ValueError:
                    pass
        if "dram__bytes_read.sum" in m:
            traffic = (m["dram__bytes_read.sum"] + m["dram__bytes_write.sum"]) * m.get("_dram_unit_bytes", 1e6)
            warp_inst = m.get("smsp__inst_executed.sum")
            note = ("from " + os.path.relpath(GUIDE_PROFILE, ROOT) + ": issue slots "
                    f"{m.get('smsp__issue_active.avg.pct_of_peak_sustained_active', float('nan')):.1f} % busy, FMA pipe "
                    f"{m.get('sm__inst_executed_pipe_fma.avg.pct_of_peak_sustained_active', float('nan')):.1f} %, ALU "
                    f"{m.get('sm__inst_executed_pipe_alu.avg.pct_of_peak_sustained_active', float('nan')):.1f} %, XU "
                    f"{m.get('sm__inst_executed_pipe_xu.avg.pct_of_peak_sustained_active', float('nan')):.1f} %, DRAM "
                    f"{m.get('gpu__dram_throughput.avg.pct_of_peak_sustained_elapsed', float('nan')):.1f} % of peak")
    clk = (sampler.summary()["sm_mhz"] or 1965) * 1e6
    n_sm = torch.cuda.get_device_properties(dev).multi_processor_count
    roofline = {"bound": "hbm", "kernel": "surv_guide_kernel" if survival else "svi_guide_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic,
                "traffic_source": os.path.relpath(GUIDE_PROFILE, ROOT) + " (ncu --set full, one launch)" if traffic else None,
                "peak_source": peak_src,
                "algorithmic_bytes_per_launch": bytes_launch, "handover_bytes_per_launch": handover,
                "ms_per_launch": ms_guide, "ms_per_launch_how": "the guide kernel launched alone (BeanSviConfig.phases = 1), CUDA events",
                "ms_per_launch_variant_kernel": ms_var, "ms_per_launch_alpha_kernel": ms_alpha,
                "alpha_kernel_gbs": alpha_kernel_bytes_per_guide(R, itemsize) * G_rank / (ms_alpha * 1e-3) / 1e9 if ms_alpha else None,
                "whole_step_frac": (bytes_launch + (12 * itemsize + 24.0 * itemsize / gpv) * G_rank) / (ms / args.steps * 1e-3) / 1e9 / peak,
                "compute_roofline": {
                    "what": "register-only kernel evaluating the same Dirichlet-Multinomial row maths "
                            f"({R * L} rows x {B} bins per guide: {2 * B + 2} lgamma/digamma corrections + {2 * B} log1p per row) with "
                            "no memory traffic at the same launch geometry: the measured FP32/SFU floor of the step's row work",
                    "row_math_ceiling_ms": ms_ceiling, "frac": ms_ceiling / ms_guide,
                    "row_math_ceiling_lane_per_cell_ms": ms_ceiling_lanes,
                    "mapping_note": "thread per guide (rows and bins in registers) against lane per (row, bin) cell with 4-lane shuffle "
                                    "reductions (the north_star's mapping): same maths, the second spends its issue slots on the row-level "
                                    "terms four times over",
                    "warp_instructions_per_launch": warp_inst,
                    "issue_floor_ms": (warp_inst / (4 * n_sm * clk) * 1e3) if warp_inst else None},
                "note": note}

    # --- e2e: host-resident screen -> public API -> host-resident results ------------------------
    data.pin_memory()  # the contract's e2e starts from PINNED host memory; pinning itself is not timed
    del eng  # its device buffers go back to torch's caching allocator: the e2e engine below reuses them instead of cudaMalloc
    e2e_steps = args.steps
    loss_host = torch.zeros(e2e_steps, dtype=torch.float64).pin_memory()

    def e2e_once():
        barrier()
        t0, t1, t_up = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        t0.record()
        eng2 = make_bench_engine(args.workload, data, dev, dtype, e2e_steps, 7, off)  # H2D of the whole shard
        t_up.record()
        for t in range(e2e_steps):
            eng2.run(1)
            if world == 1:
                loss_host[t].copy_(eng2.loss[t], non_blocking=True)  # the step's result back on the host, every step
            elif (t + 1) % LOSS_BATCH == 0 or t + 1 == e2e_steps:
                lo = (t // LOSS_BATCH) * LOSS_BATCH
                dist.all_reduce(eng2.loss[lo:t + 1])
                loss_host[lo:t + 1].copy_(eng2.loss[lo:t + 1], non_blocking=True)
        params_host = {k: v.cpu() for k, v in eng2.params().items()}
        t1.record()
        barrier()
        return max_over_ranks(t0.elapsed_time(t1)), t0.elapsed_time(t_up), eng2, params_host

    # the whole region twice, the faster one reported (both listed): 100 steps are ~70 ms, and one scheduling hiccup of the
    # host thread that issues a launch per step was seen to double that (profiles/r2t_bench_c5.json)
    runs = []
    for _ in range(2):
        ms_e2e_i, ms_setup_i, eng2, params_host = e2e_once()
        runs.append((ms_e2e_i, ms_setup_i))
        if len(runs) < 2:
            del eng2, params_host
    ms_e2e, ms_e2e_setup = min(runs)
    scr = eng2.screen
    h2d = (scr.x.numel() + scr.a0.numel()) * itemsize + scr.row_mask.numel() + (eng2.allele_counts.numel() + eng2.pi_a0.numel()) * itemsize \
        + eng2.guide_variant.numel() * 4 + eng2.variant_ptr.numel() * 4 + (eng2.log_obs.numel() * itemsize if survival else 0)
    d2h = 8 * e2e_steps + sum(v.numel() * v.element_size() for v in params_host.values())
    e2e_value = cells_per_step * e2e_steps / (ms_e2e * 1e-3)
    assert torch.isfinite(loss_host).all()
    del eng2

    # --- the north_star's run: a complete SVI fit of `--full-run-steps` steps from step 0 --------
    full_run = None
    if args.full_run_steps > 0:
        eng3 = make_bench_engine(args.workload, data, dev, dtype, args.full_run_steps, 101, off)
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        run_with_loss_exchange(eng3, args.full_run_steps, world)
        f1.record()
        barrier()
        ms_full = max_over_ranks(f0.elapsed_time(f1))
        full_run = {"steps": args.full_run_steps, "seconds": ms_full * 1e-3, "svi_steps_per_sec": args.full_run_steps / (ms_full * 1e-3),
                    "value": cells_per_step * args.full_run_steps / (ms_full * 1e-3), "unit": "cells/s",
                    "loss_first": float(eng3.loss[0].item()), "loss_last": float(eng3.loss[args.full_run_steps - 1].item()),
                    "what": "fresh engine, steps 0..N-1 with lr decay over the run, ELBO exchange included; device-resident screen"}
        del eng3

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    line = {
        "metric": "guide_rep_bin_cells_per_sec", "value": value, "unit": "cells/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": scaling,
        "vs_baseline": BASELINE_MD_PUBLISHED, "dtype": args.dtype, "data": "synthetic", "config": config,
        "burn_in_steps": burn_in, "guides_per_gpu": G_rank,
        "svi_steps_per_sec": steps_per_sec,
        "clocks": sampler.summary(),
        "e2e": {"value": e2e_value, "unit": "cells/s", "h2d_bytes_per_step": h2d / e2e_steps, "d2h_bytes_per_step": d2h / e2e_steps,
                "ms_total": ms_e2e, "ms_upload_and_setup": ms_e2e_setup, "ms_total_of_each_run": [r[0] for r in runs],
                "what": f"SviEngine built from PINNED HOST tensors (this rank's shard: upload + re-tiling + data-only constants inside the "
                        f"timed region), {e2e_steps} steps from step 0, losses copied to pinned host memory (every step at N = 1, per "
                        f"{LOSS_BATCH}-step all-reduce batch at N > 1), final parameters copied to host; per-rank bytes"},
        "gpu_launches": (3 if split else 2) * args.steps,
        "roofline": roofline,
        "final_loss": final_loss,
    }
    if peer_exchange is not None:
        line["peer_exchange"] = peer_exchange
    if full_run:
        line["full_run"] = full_run
    if world == 1 and not args.no_cpu_baseline:
        torch.set_num_threads(os.cpu_count() or 1)
        sub = data if not args.cpu_sample_guides or args.cpu_sample_guides >= data.n_guides else data[torch.arange(args.cpu_sample_guides)]
        sec = oracle_step_time(sub, steps=3, warmup=1, anomaly=True)
        line["cpu_baseline"] = {"value": sub.n_guides * R * B / sec, "unit": "cells/s", "cores": torch.get_num_threads(), "kind": "port",
                                "sample": f"{'all' if sub.n_guides == data.n_guides else 'first'} {sub.n_guides} guides of the workload, 3 timed SVI "
                                          f"steps of the plain-torch oracle port ({sec * 1e3:.0f} ms/step, torch anomaly mode on as in the "
                                          "reference); pyro itself is not installable here"}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
