"""Halting a fit at its first non-finite SVI step, host logic on CPU: `run.run_batches` with a deterministic stand-in engine that
records its first bad step the way the kernels do (the smallest step in one int32 word), and a 2-rank gloo run through
`dist.run_sharded` in which the ranks go bad at different steps."""
import os
import pickle

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from crispr_bean_b200.dist import run_sharded
from crispr_bean_b200.halt import INT32_MAX, NonfiniteWatch
from crispr_bean_b200.run import DUMP_PATH, FitHalted, run_batches


class StepEngine(NonfiniteWatch):
    """theta[i] += 1 per step; from step `bad_at` on, the step's gradient of theta[0] is NaN (the update still applies, as in
    the kernels, and poisons theta[0]); loss[t] = t + 0.5 while finite."""

    def __init__(self, n, num_steps, bad_at=None, offset=0):
        self.device = torch.device("cpu")
        self.theta = torch.arange(n, dtype=torch.float64) + offset
        self.m = torch.zeros(n, dtype=torch.float64)
        self.loss = torch.zeros(num_steps + 1, dtype=torch.float64)
        self.bad_at, self.step, self.steps_run = bad_at, 0, 0
        self._init_nonfinite()

    def _grad(self, t):
        g = torch.ones_like(self.theta)
        if self.bad_at is not None and t >= self.bad_at:
            g[0] = float("nan")
        return g

    def run(self, n):
        for t in range(self.step, self.step + n):
            g = self._grad(t)
            self.loss[t] = t + 0.5 if torch.isfinite(g).all() else float("nan")
            if not torch.isfinite(g).all() or not torch.isfinite(self.loss[t]):
                self.nonfinite[0] = min(int(self.nonfinite[0]), t)
            self.m += g
            self.theta += g
            self.steps_run += 1
        self.step += n
        return self.loss[self.step - n:self.step]

    def gradients(self):
        return {"loss": self.loss[self.step].clone() if self.bad_at is None or self.step < self.bad_at else torch.tensor(float("nan")),
                "theta": self._grad(self.step)}

    def params(self):
        return {"theta": self.theta.clone()}

    def losses(self):
        return self.loss[: self.step].clone()

    def _snapshot_tensors(self):
        return [self.theta, self.m]


def test_finite_fit_runs_through(tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)
    eng = StepEngine(4, 25)
    params, losses = run_batches(eng, 25, log_every=10)
    assert eng.steps_run == 25 and eng.nonfinite_step() is None
    assert torch.equal(params["theta"], torch.arange(4, dtype=torch.float64) + 25)
    assert losses.numel() == 25 and not os.path.exists(DUMP_PATH)


@pytest.mark.parametrize("bad_at", [0, 10, 13, 29])
def test_halt_restores_and_replays_to_the_bad_step(tmp_path, monkeypatch, bad_at):
    monkeypatch.chdir(tmp_path)
    eng = StepEngine(3, 30, bad_at=bad_at)
    with pytest.raises(FitHalted) as exc:
        run_batches(eng, 30, log_every=10)
    err = exc.value
    assert isinstance(err, ValueError)
    assert err.step == bad_at
    start = bad_at // 10 * 10  # the batch the bad step falls in
    # every batch up to the bad one, then the steps of that batch before the bad step once more
    assert eng.steps_run == min(start + 10, 30) + (bad_at - start)
    assert eng.step == bad_at
    assert torch.equal(err.params["theta"], torch.arange(3, dtype=torch.float64) + bad_at)  # theta_t exactly
    assert torch.equal(err.losses, torch.arange(bad_at, dtype=torch.float64) + 0.5)
    assert err.nonfinite == ["loss", "theta"]
    with open(tmp_path / DUMP_PATH, "rb") as f:
        dump = pickle.load(f)
    assert set(dump) == {"param"} and torch.equal(dump["param"]["theta"], err.params["theta"])
    assert eng.nonfinite_step() is None  # restore cleared the word; the replayed steps were finite


def test_restore_resets_the_word():
    eng = StepEngine(2, 10, bad_at=1)
    snap = eng.snapshot()
    eng.run(3)
    assert eng.nonfinite_step() == 1
    eng.restore(snap)
    assert int(eng.nonfinite[0]) == INT32_MAX and eng.step == 0 and torch.equal(eng.theta, torch.arange(2, dtype=torch.float64))


BAD_AT = {0: 17, 1: 12}  # rank -> its first bad step


def _worker(rank, world, port, out_dir):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    torch.set_num_threads(1)
    os.chdir(out_dir)
    data = type("Guides", (), {"is_tiling": True, "n_guides": 4, "n_edits": 1, "__getitem__": lambda self, idx: self})()
    res = {}
    try:
        run_sharded(lambda sub, guide_offset, variant_offset: StepEngine(3, 40, BAD_AT[rank], offset=10 * rank),
                    data, 40, rank, world, log_every=10)
    except FitHalted as err:
        res = {"step": err.step, "params": err.params, "losses": err.losses}
    finally:
        dist.destroy_process_group()
    torch.save(res, f"{out_dir}/r{rank}.pt")


def test_two_ranks_halt_at_the_smallest_bad_step(tmp_path):
    port = 29950 + os.getpid() % 40
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    t = min(BAD_AT.values())
    # gathered: each rank's 3 parameters after t steps, rank blocks in order
    want = torch.cat([torch.arange(3, dtype=torch.float64) + t, torch.arange(3, dtype=torch.float64) + 10 + t])
    for rank in range(2):
        got = torch.load(f"{tmp_path}/r{rank}.pt")
        assert got["step"] == t
        assert torch.equal(got["params"]["theta"], want)
        assert torch.equal(got["losses"], 2 * (torch.arange(t, dtype=torch.float64) + 0.5))  # summed over the ranks
    with open(tmp_path / DUMP_PATH, "rb") as f:  # rank 0 writes the dump
        assert torch.equal(pickle.load(f)["param"]["theta"], want)
