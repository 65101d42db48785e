"""The fused tiling step on raw allele tables: 33..1024 alleles per guide (`tiling_wide_kernel`, lane l walking the alleles
l, l + 32, ...), against the reference's own vectors of its 231-allele tiling_mini screen, the CPU oracle on synthetic wide
screens, and the routing of `run_inference`."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from crispr_bean_b200 import model as sm
from crispr_bean_b200.data_class import TilingSortingReporterScreenData
from crispr_bean_b200.generic import TilingSviEngine
from crispr_bean_b200.run import make_engine, run_inference
from crispr_bean_b200.synth import make_tiling_screen
from crispr_bean_b200.tiling_fused import TilingFusedEngine, serves, supports
from oracle import bean_oracle as O
from tests import helpers as H
from tests.fp32_floor import DTYPE_DEPENDENT, elem_rel
from tests.test_gpu_golden import KNOWN_EXCESS, rel
from tests.test_gpu_svi import rel_err
from tests.test_reference_golden import edit_perm, group, load_case, to_ours

pytestmark = pytest.mark.gpu
BEAN_EINVAL = -1
BINS5 = ((0.0, 0.2), (0.2, 0.4), (0.4, 0.6), (0.6, 0.8), (0.8, 1.0))

# synthetic wide screens: (make_tiling_screen arguments, realised n_max_alleles).  Every guide has its own number of alleles,
# so allele_mask is ragged in all of them.
SCREENS = {
    "a35": (dict(n_guides=40, window=48, max_alleles=36, n_reps=2, seed=1), 35),
    "a34_b5": (dict(n_guides=40, window=48, max_alleles=40, n_reps=3, seed=2, bins=BINS5), 34),
    "a63": (dict(n_guides=50, window=48, max_alleles=72, n_reps=2, seed=5), 63),
    "a81_b5": (dict(n_guides=60, window=48, max_alleles=100, n_reps=4, seed=4, bins=BINS5), 81),
    "a977": (dict(n_guides=4, window=300, max_alleles=1500, n_reps=2, seed=2), 977),
}


def wide_data(name):
    kw, width = SCREENS[name]
    data = TilingSortingReporterScreenData(make_tiling_screen(**kw), control_can_be_selected=True, allele_df_key="allele_counts")
    assert data.n_max_alleles == width, (name, data.n_max_alleles)
    return data


def widen(data, A):
    """The same screen with A alleles per guide: the extra columns are alleles no guide has (allele_mask 0, no edits, no
    counts).  They are still drawn and enter every sum, so the values change, but the screen stays consistent."""
    G, A0 = data.n_guides, data.n_max_alleles
    assert A >= A0
    ptr = data.allele_ptr.numpy().astype(np.int64)
    n_per_slot = np.zeros((G, A - 1), dtype=np.int64)
    n_per_slot[:, : A0 - 1] = np.diff(ptr).reshape(G, A0 - 1)
    data.allele_ptr = torch.as_tensor(np.concatenate([[0], np.cumsum(n_per_slot.reshape(-1))]).astype(np.int32))
    mask = torch.zeros((G, A), dtype=torch.bool)
    mask[:, :A0] = data.allele_mask
    data.allele_mask = mask
    ac = data.allele_counts_control
    data.allele_counts_control = torch.cat([ac, ac.new_zeros(ac.shape[:-1] + (A - A0,))], dim=-1)
    data.n_max_alleles = A
    return data


def _oracle_grads(data, eng, noise, use_bcmatch):
    """Loss and gradients of the oracle at the engine's parameters, and the float64 floor of alpha_pi's gradient (the same
    formula evaluated a second time in another order, oracle/tiling_closed_form.py; tests/test_gpu_tiling_fused.py)."""
    from oracle import tiling_closed_form as TC

    with H.default_dtype(torch.float64):
        ps = O.ParamStore()
        d = H.cast_data(data, torch.float64)
        O.elbo_multi_mixture_normal(d, ps, noise=noise, use_bcmatch=use_bcmatch)
        for i, k in enumerate(("mu_loc", "mu_scale", "sd_loc", "sd_scale")):
            ps.unconstrained[k].data.copy_(eng.edit_params[i].double().cpu().reshape(ps.unconstrained[k].shape))
        ps.unconstrained["alpha_pi"].data.copy_(eng.alpha_u.double().cpu())
        loss, _ = O.elbo_multi_mixture_normal(d, ps, noise=noise, use_bcmatch=use_bcmatch)
        ps.zero_grad()
        loss.backward()
        floor = None
        if use_bcmatch:  # the closed form restates the default program (bcmatch layer on)
            _, closed = TC.tiling_step(d, {k: v.detach() for k, v in ps.unconstrained.items()}, noise)
            floor = rel_err(torch.as_tensor(closed["alpha_pi"]).reshape(ps.unconstrained["alpha_pi"].shape),
                            ps.unconstrained["alpha_pi"].grad)
    return float(loss.detach()), {k: v.grad for k, v in ps.unconstrained.items()}, floor


def _check_against_oracle(data, cuda_device, dtype, tol, use_bcmatch=True, label=""):
    noise = H.fixed_noise("MultiMixtureNormal", data, seed=5)
    eng = TilingFusedEngine(data, cuda_device, dtype=dtype, num_steps=8, use_bcmatch=use_bcmatch)
    g = torch.Generator().manual_seed(7)  # away from the initial point
    eng.edit_params.copy_(0.3 * torch.randn((4, eng.E), generator=g, dtype=torch.float64))
    eng.alpha_u.copy_(torch.where(data.allele_mask, 0.5 * torch.randn(eng.alpha_u.shape, generator=g, dtype=torch.float64),
                                  eng.alpha_u.double().cpu()))
    got = eng.gradients(noise)
    ref, grads, floor = _oracle_grads(data, eng, noise, use_bcmatch)
    errs = {"loss": abs(got["loss"].item() - ref) / abs(ref)}
    for k, v in grads.items():
        errs[k] = rel_err(got[k], v)
    print(label, dtype, "A", data.n_max_alleles, errs, "float64 floor of alpha_pi", floor)
    assert errs["loss"] <= tol
    for k, e in errs.items():
        bound = 10 * tol if dtype == torch.float32 else tol
        if k == "alpha_pi" and floor is not None:
            bound = max(bound, 5 * floor)
        assert e <= bound, (k, e, bound)


# ---- the reference's own vectors: tiling_real_mini (231 alleles per guide, 5 bins), today served by the site-kernel engine

REAL = "tiling_real_mini"


def _real():
    z, data = load_case(REAL)
    assert data.n_max_alleles == 231 and serves(data) and not supports(data)
    return z, data, edit_perm(z, data)


def test_fp64_step_equals_reference_on_the_raw_tiling_screen(cuda_device):
    z, data, perm = _real()
    eng = TilingFusedEngine(data, cuda_device, dtype=torch.float64, num_steps=4)
    noise = {k: torch.as_tensor(to_ours(v, perm, k)) for k, v in group(z, "f64/noise/").items() if "/" not in k}
    got = eng.gradients(noise)
    ref_loss = float(z["f64/loss"])
    err = {"loss": abs(got["loss"].item() - ref_loss) / abs(ref_loss)}
    err.update({k: rel(got[k], to_ours(g, perm, k)) for k, g in group(z, "f64/grad/").items()})
    print(REAL, "fp64", err)
    for k, e in err.items():
        assert e <= 1e-9, (k, e)


def test_fused_run_follows_reference_run_inference_on_the_raw_tiling_screen(cuda_device):
    z, data, perm = _real()
    n = int(z["traj/n_steps"])
    eng = TilingFusedEngine(data, cuda_device, dtype=torch.float64, num_steps=n)
    tn = {k: to_ours(v, perm, k) for k, v in group(z, "traj/noise/").items()}
    for t in range(n):
        eng.run(1, noise={k: torch.as_tensor(v[t]) for k, v in tn.items()})
    loss = eng.losses().numpy()
    err = np.abs(loss - z["traj/loss"]).max() / np.abs(z["traj/loss"]).max()
    params = eng.params()
    perr = {k: rel(params[k], to_ours(v, perm, k)) for k, v in group(z, "traj/param/").items()}
    print(REAL, "traj loss", err, perr)
    assert err <= 1e-9
    for k, e in perr.items():
        assert e <= 1e-8, (k, e)


def test_fp32_step_on_the_raw_tiling_screen(cuda_device):
    """Draws on the sampler's float32 clamps (fp32_floor.DTYPE_DEPENDENT): compared with the reference's float32 results, each
    parameter no worse than max(1e-5, 2 x the error measured for the site-kernel engine that served this screen before)."""
    assert REAL in DTYPE_DEPENDENT
    z, data, perm = _real()
    eng = TilingFusedEngine(data, cuda_device, dtype=torch.float32, num_steps=4)
    noise = {k: torch.as_tensor(to_ours(v, perm, k)) for k, v in group(z, "native/noise/").items() if "/" not in k}
    got = eng.gradients(noise)
    ref_loss = float(z["native/loss"])
    err_loss = abs(got["loss"].item() - ref_loss) / abs(ref_loss)
    native = {k: to_ours(g, perm, k) for k, g in group(z, "native/grad/").items()}
    errs = {k: elem_rel(got[k].detach().double().cpu().numpy(), np.asarray(g).reshape(-1)) for k, g in native.items()}
    print(REAL, "fp32 loss", err_loss, errs)
    assert err_loss <= 1e-5
    for k, e in errs.items():
        tol = max(1e-5, 2.0 * KNOWN_EXCESS.get((REAL, k), 0.0))
        assert e <= tol, (k, e, tol)


def test_500_step_fp32_fit_on_the_raw_tiling_screen(cuda_device, monkeypatch):
    """tests/test_gpu_e2e_reference_screens.py's fit of tiling_real_mini (500 steps against the float32 oracle on the same
    injected draws; mu / mu_sd / mu_z / ranking tolerances) with the fused step serving it."""
    from tests import test_gpu_e2e_reference_screens as E2E

    def fused(z, data, dev, dtype, num_steps):
        return TilingFusedEngine(data, dev, dtype=dtype, num_steps=num_steps)

    monkeypatch.setattr(E2E, "make_engine", fused)
    assert E2E.N_STEPS[REAL] == 500
    E2E.test_2000_step_fp32_fit_matches_the_float64_reference_programs(cuda_device, REAL)


# ---- the CPU oracle on synthetic wide screens


@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-9), (torch.float32, 1e-5)])
@pytest.mark.parametrize("name", list(SCREENS))
def test_wide_step_equals_oracle(cuda_device, dtype, tol, name):
    data = wide_data(name)
    data.repguide_mask[1, ::6] = False
    _check_against_oracle(data, cuda_device, dtype, tol, label=name)


@pytest.mark.parametrize("dtype,tol", [(torch.float64, 1e-9), (torch.float32, 1e-5)])
def test_wide_step_without_bcmatch_equals_oracle(cuda_device, dtype, tol):
    data = wide_data("a63")
    data.repguide_mask[0, ::5] = False
    _check_against_oracle(data, cuda_device, dtype, tol, use_bcmatch=False, label="a63 no bcmatch")


@pytest.mark.parametrize("bins", [None, BINS5])
def test_1024_alleles_launch_and_equal_oracle(cuda_device, bins):
    """The widest table the fused step takes, in float64 with 4 and 5 bins (the most shared memory per guide)."""
    kw = dict(SCREENS["a977"][0])
    if bins is not None:
        kw["bins"] = bins
    data = widen(TilingSortingReporterScreenData(make_tiling_screen(**kw), control_can_be_selected=True,
                                                 allele_df_key="allele_counts"), 1024)
    _check_against_oracle(data, cuda_device, torch.float64, 1e-9, label="a1024")


# ---- free-running steps, recorded draws, non-finite flag


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_free_running_wide_steps_are_deterministic_and_improve_the_elbo(cuda_device, dtype):
    data = wide_data("a81_b5")
    runs = []
    for _ in range(2):
        eng = TilingFusedEngine(data, cuda_device, dtype=dtype, num_steps=300, seed=9)
        eng.run(150)
        eng.run(150)
        runs.append((eng.losses(), eng.params()))
    assert torch.equal(runs[0][0], runs[1][0])
    for k, v in runs[0][1].items():
        assert torch.equal(v, runs[1][1][k]), k
    loss = runs[0][0]
    assert torch.isfinite(loss).all()
    assert loss[-50:].mean() < loss[:50].mean()


def test_recorded_wide_draws_replay_into_the_oracle(cuda_device):
    """One free-running fp64 step: the kernel's own Philox draws, recorded, give the same loss and gradients in the oracle."""
    data = wide_data("a63")
    eng = TilingFusedEngine(data, cuda_device, dtype=torch.float64, num_steps=4, seed=3)
    loss = eng.run(1, noise={"record": True}, apply_update=False)
    noise = {"eps_mu": eng.eps_used[0].cpu(), "eps_sd": eng.eps_used[1].cpu(), "pi": eng.pi_used.cpu().unsqueeze(1)}
    assert torch.allclose(noise["pi"].sum(-1), torch.ones_like(noise["pi"].sum(-1)), atol=1e-12)
    with H.default_dtype(torch.float64):
        ps = O.ParamStore()
        ref, _ = O.elbo_multi_mixture_normal(H.cast_data(data, torch.float64), ps, noise=noise)
        ref.backward()
    assert abs(loss[0].item() - float(ref.detach())) <= 1e-9 * abs(float(ref.detach()))
    assert rel_err(eng.alpha_grad, ps.unconstrained["alpha_pi"].grad) <= 1e-9
    for i, k in enumerate(("mu_loc", "mu_scale", "sd_loc", "sd_scale")):
        assert rel_err(eng.edit_grad[i], ps.unconstrained[k].grad) <= 1e-9, k


def test_nan_parameter_is_recorded_at_its_step(cuda_device):
    k = 6
    eng = TilingFusedEngine(wide_data("a35"), cuda_device, dtype=torch.float32, num_steps=20)
    eng.run(k)
    assert eng.nonfinite_step() is None
    with torch.no_grad():
        eng.edit_params[0, 0] = float("nan")
    eng.run(5)
    assert eng.nonfinite_step() == k
    eng.gradients()  # apply_update = 0 never records
    assert eng.nonfinite_step() == k


# ---- routing


def test_run_inference_routes_wide_tiling_designs_to_the_fused_engine(cuda_device):
    M, Gd = sm.MultiMixtureNormalModel, sm.MultiMixtureNormalGuide
    data = wide_data("a34_b5")
    eng = make_engine(M, Gd, data, num_steps=10, device=cuda_device)
    assert isinstance(eng, TilingFusedEngine) and not eng.sharded
    eng.run(10)
    assert torch.isfinite(eng.losses()).all()
    assert isinstance(make_engine(M, Gd, widen(wide_data("a977"), 1024), num_steps=4, device=cuda_device), TilingFusedEngine)
    assert isinstance(make_engine(M, Gd, widen(wide_data("a977"), 1025), num_steps=4, device=cuda_device), TilingSviEngine)
    acc = TilingSortingReporterScreenData(make_tiling_screen(**SCREENS["a35"][0], accessibility=True), control_can_be_selected=True,
                                          allele_df_key="allele_counts", accessibility_col="accessibility")
    assert serves(acc) and not serves(acc, scale_by_accessibility=True)
    from functools import partial

    eng = make_engine(partial(M, scale_by_accessibility=True), partial(Gd, scale_by_accessibility=True), acc, num_steps=4,
                      device=cuda_device)
    assert isinstance(eng, TilingSviEngine)


def test_c_entry_point_rejects_1025_alleles(cuda_device):
    eng = TilingFusedEngine(widen(wide_data("a35"), 1024), cuda_device, dtype=torch.float32, num_steps=4)
    eng.amap.c.n_alleles = 1025  # the map of a 1025-allele design (the kernel is never reached)
    stream = torch.cuda.current_stream(eng.device).cuda_stream
    assert eng.lib.bean_svi_tiling_run_f32(eng.screen.c, eng.state, eng.cfg, None, 0, 1, stream) == BEAN_EINVAL
    eng.amap.c.n_alleles = 1024
    assert eng.lib.bean_svi_tiling_run_f32(eng.screen.c, eng.state, eng.cfg, None, 0, 1, stream) == 0


# ---- replicas: a wide screen is not sharded, so under a process group every rank fits it on its own


REPLICA_STEPS = 40


def _replica_fit(device):
    params, out = run_inference(sm.MultiMixtureNormalModel, sm.MultiMixtureNormalGuide, wide_data("a63"),
                                num_steps=REPLICA_STEPS, device=device, log_every=15)
    return {k: v.detach().cpu() for k, v in params.items()}, torch.tensor(out["loss"], dtype=torch.float64)


def _replica_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        torch.save(_replica_fit("cuda:0"), f"{out_dir}/r{rank}.pt")
    finally:
        dist.destroy_process_group()


def test_wide_screen_under_two_ranks_equals_one_process(cuda_device, tmp_path):
    """Two ranks on one GPU over gloo: an engine that took itself for a shard would all-reduce its whole-screen edit sums and
    double every per-edit gradient."""
    port = 29730 + os.getpid() % 100
    mp.spawn(_replica_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    params, loss = _replica_fit(cuda_device)
    for r in range(2):
        p, lo = torch.load(f"{tmp_path}/r{r}.pt")
        assert torch.equal(lo, loss), r
        assert set(p) == set(params)
        for k, v in params.items():
            assert torch.equal(p[k], v), (r, k)
