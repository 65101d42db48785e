"""Per-step time of the c5 workload over a long run, in blocks of 100 steps (CUDA events).

    python profiles/steady_state.py [n_steps]

A step gets slower over the first ~300 steps (alpha_pi fits the low editing rates and more Dirichlet draws leave the
saddle-point regime); bench.py therefore burns in before timing.  Also the target of the steady-state ncu capture
(profiles/capture.sh).
"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from bench import build_data
from crispr_bean_b200.svi import SviEngine
data = build_data("c5_genome_scale", 101)
dev = torch.device("cuda")
N = int(sys.argv[1]) if len(sys.argv) > 1 else 2000
eng = SviEngine(data, "MixtureNormal", dev, num_steps=N)
for blk in range(N // 100):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record(); eng.run(100); b.record(); torch.cuda.synchronize()
    al = eng.alpha_u.exp(); conc = al / al.sum(-1, keepdim=True) * eng.pi_a0[:, None]
    print(f"steps {blk*100:5d}-{blk*100+99:5d}: {a.elapsed_time(b)/100:.3f} ms/step  loss {eng.loss[eng.step-1].item():.6g}  conc<1: {(conc<1).float().mean().item():.3f} conc>6 both: {((conc>6).all(-1)).float().mean().item():.3f} min conc med {conc.min(-1).values.median().item():.3f}", flush=True)
