"""Halting a fit at its first non-finite SVI step on the GPU: the device word every engine keeps (include/bean_b200.h:
nonfinite_step), `snapshot` / `restore`, and `run_inference` raising FitHalted with the exact parameters of the bad step."""
import os
import pickle

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from crispr_bean_b200 import model as sorting_model
from crispr_bean_b200 import survival_model
from crispr_bean_b200.data_class import (TilingSortingReporterScreenData, VariantSurvivalReporterScreenData,
                                         VariantSurvivalScreenData)
from crispr_bean_b200.run import DUMP_PATH, FitHalted, make_engine, run_inference
from crispr_bean_b200.synth import make_survival_screen, make_tiling_screen
from tests import helpers as H

pytestmark = pytest.mark.gpu

ENGINES = ["Normal", "ControlNormal", "MixtureNormal", "MixtureNormal+Acc", "survival_fused", "tiling_fused", "tiling_sites",
           "survival_sites"]


def _sorting():
    return H.make_small_mixture_data(n_variants=30, n_reps=3, seed=4)


def _survival(reporter=True):
    scr = make_survival_screen(40, "lognormal", n_reps=3, seed=11, n_negctrl_guides=7)
    if reporter:
        return VariantSurvivalReporterScreenData(scr, control_condition="D7")
    return VariantSurvivalScreenData(scr, control_condition="D7", negctrl_guide_idx=list(range(7)))


def _tiling():
    return TilingSortingReporterScreenData(make_tiling_screen(n_guides=60, max_alleles=8, n_reps=3, seed=3), control_can_be_selected=True,
                                           allele_df_key="allele_counts")


def _engine(name, dev, num_steps):
    from crispr_bean_b200.generic import TilingSviEngine
    from crispr_bean_b200.survival import SurvivalSviEngine
    from crispr_bean_b200.survival_fused import SurvivalFusedEngine
    from crispr_bean_b200.svi import SviEngine
    from crispr_bean_b200.tiling_fused import TilingFusedEngine

    kw = dict(dtype=torch.float32, num_steps=num_steps)
    if name in ("Normal", "ControlNormal", "MixtureNormal"):
        return SviEngine(_sorting(), name, dev, **kw)
    if name == "MixtureNormal+Acc":
        data = H.make_small_mixture_data(n_variants=30, n_reps=3, seed=4, accessibility=True)
        return SviEngine(data, "MixtureNormal", dev, scale_by_accessibility=True, fit_noise=True, **kw)
    if name == "survival_fused":
        return SurvivalFusedEngine(_survival(), dev, **kw)
    if name == "tiling_fused":
        return TilingFusedEngine(_tiling(), dev, **kw)
    if name == "tiling_sites":
        return TilingSviEngine(_tiling(), dev, **kw)
    return SurvivalSviEngine(_survival(reporter=False), "Normal", dev, **kw)


def _poison(eng):
    """NaN into the first mu_loc of the engine, between two run() calls."""
    with torch.no_grad():
        if hasattr(eng, "theta"):
            eng.theta["mu_loc"].view(-1)[0] = float("nan")
        elif hasattr(eng, "edit_params"):
            eng.edit_params[0, 0] = float("nan")
        else:
            eng.var_params[0, 0] = float("nan")


def _state(eng):
    return {k: v.detach().clone() for k, v in eng.params().items()}


@pytest.mark.parametrize("name", ENGINES)
def test_finite_run_records_nothing(cuda_device, name):
    eng = _engine(name, cuda_device, 100)
    eng.run(100)
    assert torch.isfinite(eng.losses()).all()
    assert eng.nonfinite_step() is None


@pytest.mark.parametrize("name", ENGINES)
def test_nan_parameter_is_recorded_at_its_step(cuda_device, name):
    k = 6
    eng = _engine(name, cuda_device, 20)
    eng.run(k)
    assert eng.nonfinite_step() is None
    _poison(eng)
    eng.run(5)
    assert eng.nonfinite_step() == k
    eng.gradients()  # apply_update = 0 never records
    assert eng.nonfinite_step() == k


@pytest.mark.parametrize("name", ENGINES)
def test_snapshot_restore_replays_bit_for_bit(cuda_device, name):
    eng = _engine(name, cuda_device, 30)
    eng.run(5)
    snap = eng.snapshot()
    first = eng.run(9).clone()
    p1 = _state(eng)
    eng.restore(snap)
    assert eng.step == 5 and eng.nonfinite_step() is None
    second = eng.run(9).clone()
    assert torch.equal(first, second)
    for key, v in _state(eng).items():
        assert torch.equal(v, p1[key]), key


RUNS = {
    "sorting MixtureNormal": (sorting_model.MixtureNormalModel, sorting_model.MixtureNormalGuide, _sorting),
    "sorting Normal": (sorting_model.NormalModel, sorting_model.NormalGuide, _sorting),
    "survival fused": (survival_model.MixtureNormalModel, survival_model.MixtureNormalGuide, _survival),
    "survival sites": (survival_model.NormalModel, survival_model.NormalGuide, lambda: _survival(reporter=False)),
    "tiling fused": (sorting_model.MultiMixtureNormalModel, sorting_model.MultiMixtureNormalGuide, _tiling),
}


@pytest.mark.parametrize("case", list(RUNS))
def test_run_inference_halts_with_the_parameters_of_the_bad_step(cuda_device, tmp_path, monkeypatch, case):
    model, guide, make_data = RUNS[case]
    monkeypatch.chdir(tmp_path)
    steps, every, lr = 60, 25, 1e3
    with pytest.raises(FitHalted) as exc:
        run_inference(model, guide, make_data(), initial_lr=lr, num_steps=steps, device=cuda_device, log_every=every)
    err = exc.value
    t = err.step
    assert isinstance(err, ValueError) and 1 <= t < steps
    assert err.losses.numel() == t and torch.isfinite(err.losses).all()
    assert err.nonfinite
    # a fresh engine of the same run (same num_steps: the lr decay depends on it), driven in the same calls, t steps
    eng = make_engine(model, guide, make_data(), lr, 0.1, steps, cuda_device)
    start = t // every * every
    for _ in range(start // every):
        eng.run(every)
    if t > start:
        eng.run(t - start)
    want = {k: v.detach().cpu() for k, v in eng.params().items()}
    assert set(want) == set(err.params)
    for k, v in want.items():
        assert torch.equal(err.params[k], v), k
    with open(tmp_path / DUMP_PATH, "rb") as f:
        dump = pickle.load(f)
    for k, v in want.items():
        assert torch.equal(dump["param"][k], v), k


# ---- two GPUs: every rank halts at the same step, the gathered parameters are those of a sharded run of that many steps


def _sharded_worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from crispr_bean_b200.dist import run_sharded

    os.chdir(out_dir)
    res = {}
    for case in ("sorting MixtureNormal", "survival fused"):
        model, guide, make_data = RUNS[case]
        steps, every, lr = 60, 25, 1e3
        engines = []

        def make(sub, guide_offset, variant_offset):
            engines.append(make_engine(model, guide, sub, lr, 0.1, steps, f"cuda:{rank}", torch.float32, 101, guide_offset, variant_offset))
            return engines[-1]

        try:
            run_inference(model, guide, make_data(), initial_lr=lr, num_steps=steps, device=f"cuda:{rank}", log_every=every)
            res[case] = {"step": None}
            continue
        except FitHalted as err:
            got = {"step": err.step, "params": err.params}
        t = got["step"]
        # reference: the same sharded run for exactly t steps, in the same calls
        start = t // every * every

        def make_short(sub, guide_offset, variant_offset):
            eng = make(sub, guide_offset, variant_offset)

            class Capped:  # runs the batches the halted fit ran, then the steps before t
                device = eng.device
                replicated_params = getattr(eng, "replicated_params", ())

                def run(self, n):
                    return eng.run(n)

                def losses(self):
                    return eng.losses()

                def params(self):
                    return eng.params()

            return Capped()

        sizes = [every] * (start // every) + ([t - start] if t > start else [])
        ref = None
        if sizes:
            # run_sharded runs min(log_every, left) per batch: log_every = every, num_steps = t gives exactly `sizes`
            ref, _ = run_sharded(make_short, make_data(), t, rank, world, log_every=every)
        got["ref"] = {k: v.detach().cpu() for k, v in ref.items()} if ref is not None else None
        got["timeouts"] = sum(getattr(e, "peer_timeouts", lambda: 0)() for e in engines)
        res[case] = got
    torch.save(res, f"{out_dir}/h{rank}.pt")
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sharded_fit_halts_on_every_rank_at_the_same_step(tmp_path):
    port = 29630 + os.getpid() % 100
    mp.spawn(_sharded_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = (torch.load(f"{tmp_path}/h{r}.pt") for r in range(2))
    for case in r0:
        assert r0[case]["step"] is not None and r0[case]["step"] == r1[case]["step"], case
        assert r0[case]["timeouts"] == 0 and r1[case]["timeouts"] == 0, case
        if r0[case]["ref"] is None:
            continue
        for r in (r0, r1):
            for k, v in r[case]["ref"].items():
                assert torch.equal(r[case]["params"][k], v), (case, k)
