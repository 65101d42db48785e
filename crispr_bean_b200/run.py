"""`run_inference` / `identify_model_guide` with the reference's signatures (bean/model/run.py:347-474).

`run_inference(model, guide, data, initial_lr=0.01, gamma=0.1, num_steps=2000)` returns
`(param_store_like, {"loss": [float per step], "params": {name: cpu tensor}})` exactly like
bean/model/run.py:391-396, but the loop runs on the GPU with no host sync per step.
"""
from __future__ import annotations

import pickle
from functools import partial
from logging import info
from typing import Callable, Dict, List, Optional

import torch

from . import model as sorting_model
from . import survival_model
from ._lib import BeanError
from .model import resolve, selection_of
from .svi import SviEngine

FUSED_MODELS = ("Normal", "ControlNormal", "MixtureNormal")
DUMP_PATH = "tmp_result.pkl"  # where the reference's run_inference pickles the parameter store of a failed fit (run.py:381-390)


class FitHalted(ValueError):
    """SVI step `step` produced a NaN / inf loss or gradient, so the fit stopped before applying it, as the reference's fit does
    under torch's anomaly mode.

    step: the first non-finite step (0-based).
    params: the parameters that step started from, {name: cpu tensor} -- exact, not the last batch boundary.
    losses: the (finite) losses of steps 0 .. step - 1.
    nonfinite: names among "loss" and the parameters whose value or gradient is non-finite at `params`.
    The same parameters are pickled to ./tmp_result.pkl as {"param": params} (rank 0 only when sharded)."""

    def __init__(self, step: int, params: Dict[str, torch.Tensor], losses: torch.Tensor, nonfinite: List[str]):
        super().__init__(f"SVI step {step} is not finite ({', '.join(nonfinite) or 'no term isolated'}); "
                         f"parameters of step {step} written to {DUMP_PATH}")
        self.step, self.params, self.losses, self.nonfinite = step, params, losses, nonfinite


def run_batches(eng, num_steps: int, log_every: int = 100, collect: Optional[Callable] = None,
                agree: Optional[Callable] = None, rank: int = 0, log: bool = True):
    """`num_steps` SVI steps of `eng` in batches of `log_every`; returns `collect(eng)` -> (params, losses).

    After every batch the engine's first non-finite step is read (`agree` makes the ranks of a sharded fit agree on it: MIN).
    Where there is one, the engine is set back to the start of the batch and re-runs the steps before it, and FitHalted is
    raised with the parameters that step started from.  `collect` defaults to this engine's own (params, losses).  An engine
    without `nonfinite_step` / `snapshot` / `restore` (a test double) is run without the check."""
    if collect is None:
        def collect(e):
            return e.params(), e.losses()
    watch = all(hasattr(eng, k) for k in ("nonfinite_step", "snapshot", "restore"))
    done = 0
    while done < num_steps:
        n = min(log_every, num_steps - done)
        snap = eng.snapshot() if watch else None
        losses = eng.run(n)
        if watch:
            t = eng.nonfinite_step()
            if agree is not None:
                t = agree(t)
            if t is not None:
                _halt(eng, snap, t, done, collect, rank)
        if log:
            info(f"loss {losses[0].item()} @ iter {done}")  # reference prints every 100 steps (run.py:378-379)
        done += n
    return collect(eng)


def _halt(eng, snap, t: int, batch_start: int, collect: Callable, rank: int):
    eng.restore(snap)
    if t > batch_start:
        eng.run(t - batch_start)
    grads = eng.gradients()  # step t's loss and gradient at theta_t (same counters as step t)
    params, losses = collect(eng)
    params = {k: v.detach().cpu() for k, v in params.items()}
    own = eng.params()

    def bad(x):
        return x is not None and not bool(torch.isfinite(x).all())

    nonfinite = ["loss"] if bad(grads["loss"]) else []
    nonfinite += [k for k in own if bad(own[k]) or bad(grads.get(k))]
    if rank == 0:
        with open(DUMP_PATH, "wb") as f:
            pickle.dump({"param": params}, f)
    raise FitHalted(t, params, losses.detach().cpu()[:t], nonfinite)


def make_engine(model, guide, data, initial_lr=0.01, gamma=0.1, num_steps=2000, device="cuda", dtype=torch.float32,
                seed=101, guide_offset=0, variant_offset=0, replica=False):
    """The device-resident SVI engine of a (model, guide) pair.  `guide_offset` / `variant_offset`: global index of the first
    guide / variant of `data` when it is one shard of a larger screen (the noise counters use global ids).  `replica`: `data` is
    the whole screen, fitted by this process alone even when torch.distributed has more than one rank (no collectives)."""
    name, mkw = resolve(model)
    gname, gkw = resolve(guide)
    if name != gname:
        raise ValueError(f"model {name} and guide {gname} do not belong together")
    if not torch.cuda.is_available():
        raise BeanError("run_inference needs a CUDA device: crispr_bean_b200 has no CPU fallback")
    if selection_of(model) != selection_of(guide):
        raise ValueError("model and guide belong to different selections (sorting vs survival)")
    use_bcmatch = mkw.get("use_bcmatch", True)
    use_bcmatch = True if isinstance(use_bcmatch, tuple) else bool(use_bcmatch)  # the reference passes a 1-tuple (App. B2)
    kw = dict(device=device, dtype=dtype, num_steps=num_steps, initial_lr=initial_lr, gamma=gamma, seed=seed,
              prior_params=mkw.get("prior_params"))
    alpha_prior, sd_scale = float(mkw.get("alpha_prior", 1.0)), float(mkw.get("sd_scale", 0.01))
    mask_thres, epsilon = int(mkw.get("mask_thres", 10)), float(mkw.get("epsilon", 1e-5))
    scale_by_acc = bool(mkw.get("scale_by_accessibility", False))
    fit_noise = bool(gkw.get("fit_noise", False))  # only the GUIDE's fit_noise matters: the model is never given it (App. B3)
    if selection_of(model) == "survival":
        from .survival import SurvivalSviEngine

        extra = {}
        if name in ("MixtureNormal", "MultiMixtureNormal"):
            extra = dict(mu_negctrl=mkw["mu_negctrl"], scale_by_accessibility=scale_by_acc, fit_noise=fit_noise)
        if name == "MultiMixtureNormal":
            extra["epsilon"] = epsilon
        if name == "MixtureNormal" and not scale_by_acc:
            from .survival_fused import SurvivalFusedEngine  # the whole step as three CUDA kernels

            return SurvivalFusedEngine(data, use_bcmatch=use_bcmatch, alpha_prior=alpha_prior, mask_thres=mask_thres,
                                       mu_negctrl=mkw["mu_negctrl"], guide_offset=guide_offset, variant_offset=variant_offset, **kw)
        return SurvivalSviEngine(data, name, use_bcmatch=use_bcmatch, alpha_prior=alpha_prior, mask_thres=mask_thres,
                                 guide_offset=guide_offset, **extra, **kw)
    if name == "MultiMixtureNormal":
        from .generic import TilingSviEngine
        from . import tiling_fused

        # 2..1024 alleles per guide, no --scale-by-acc, and (above 32 alleles) small enough for the fused step to be faster
        if tiling_fused.serves(data, scale_by_acc) and tiling_fused.faster_than_site_kernels(data):
            return tiling_fused.TilingFusedEngine(data, use_bcmatch=True, alpha_prior=alpha_prior, sd_scale=sd_scale, epsilon=epsilon,
                                                  guide_offset=guide_offset, sharded=False if replica else None, **kw)
        return TilingSviEngine(data, use_bcmatch=True, alpha_prior=alpha_prior, sd_scale=sd_scale, epsilon=epsilon,
                               scale_by_accessibility=scale_by_acc, fit_noise=fit_noise, **kw)
    if name == "Normal" and getattr(data, "sample_covariates", None) is not None:
        from .generic import CovariateNormalEngine  # replicate-specific means: not in the fused kernel

        return CovariateNormalEngine(data, use_bcmatch=use_bcmatch, sd_scale=sd_scale, mask_thres=mask_thres, **kw)
    if name not in FUSED_MODELS:
        raise NotImplementedError(f"model {name} is not built yet")
    return SviEngine(data, name, use_bcmatch=use_bcmatch, alpha_prior=alpha_prior, sd_scale=sd_scale, mask_thres=mask_thres,
                     scale_by_accessibility=scale_by_acc, fit_noise=fit_noise, guide_offset=guide_offset,
                     variant_offset=variant_offset, **kw)


def shards_over_ranks(model, data) -> bool:
    """Whether a (model, screen) pair is split over the ranks of torch.distributed (SURVEY section 8e): the variant designs
    shard by contiguous variant blocks; ControlNormal (a handful of global scalars over ~100 control guides), the covariate
    Normal model (replicate-level parameters) and the tiling designs (edits shared between overlapping guides) run as
    replicas -- every rank fits the whole screen and returns the same result.  The tiling sorting design shards by guide blocks
    where the fused step serves it (every rank keeps all edits and the per-edit gradient sums are all-reduced each step)."""
    name, mkw = resolve(model)
    scale_by_acc = bool(mkw.get("scale_by_accessibility", False))
    if name == "MultiMixtureNormal":  # guide blocks, the per-edit gradients all-reduced every step: the fused tiling step only
        from . import tiling_fused

        return (not getattr(data, "is_survival", False)) and tiling_fused.supports(data, scale_by_acc) and int(data.n_guides) >= 2
    if name == "ControlNormal":
        return False
    if getattr(data, "sample_covariates", None) is not None or not hasattr(data, "target_lengths"):
        return False
    return int(data.n_targets) >= 2


def run_inference(model, guide, data, initial_lr=0.01, gamma=0.1, num_steps=2000, autoguide=False, device="cuda",
                  dtype=torch.float32, seed=101, log_every=100):
    """Run SVI (one-particle Trace_ELBO + ClippedAdam, lr decaying by `gamma` over the run).

    Raises FitHalted (a ValueError) at the first step whose loss or gradient is NaN / inf, with the parameters that step
    started from, which are also pickled to ./tmp_result.pkl -- as the reference does (run.py:381-390).

    Same signature and return value as bean/model/run.py:347-396.  When torch.distributed is initialised with more than one
    rank (one process per GPU, e.g. under torchrun), every rank passes the SAME tensorised screen: the variants -- with all
    their guides -- are split over the ranks (`dist.shard_data`), each rank fits its block on its own GPU, the per-step ELBO
    scalars are summed and the parameters gathered, so that every rank returns the result of the whole screen."""
    import torch.distributed as tdist

    from .dist import run_sharded

    world = tdist.get_world_size() if (tdist.is_available() and tdist.is_initialized()) else 1
    if world > 1 and shards_over_ranks(model, data):
        def make(sub, guide_offset, variant_offset):
            return make_engine(model, guide, sub, initial_lr, gamma, num_steps, device, dtype, seed, guide_offset, variant_offset)

        params, loss = run_sharded(make, data, num_steps, tdist.get_rank(), world, log_every=log_every)
        return params, {"loss": loss.tolist(), "params": {k: v.detach().cpu() for k, v in params.items()}}
    # every rank fits the whole screen (a replica): its engine must not all-reduce with the other ranks
    eng = make_engine(model, guide, data, initial_lr, gamma, num_steps, device, dtype, seed, replica=True)
    params, losses = run_batches(eng, num_steps, log_every)
    return params, {"loss": losses.tolist(), "params": {k: v.detach().cpu() for k, v in params.items()}}


def identify_model_guide(args):
    """bean/model/run.py:399-457."""
    m = sorting_model if args.selection == "sorting" else survival_model
    if args.library_design == "tiling":
        return (
            f"MultiMixtureNormal{'+Acc' if args.scale_by_acc else ''}",
            partial(m.MultiMixtureNormalModel, scale_by_accessibility=args.scale_by_acc, use_bcmatch=(not args.ignore_bcmatch,)),
            partial(m.MultiMixtureNormalGuide, scale_by_accessibility=args.scale_by_acc, fit_noise=True),
        )
    if args.uniform_edit:
        if args.guide_activity_col is not None:
            raise ValueError("Can't use the guide activity column while constraining uniform edit.")
        return "Normal", partial(m.NormalModel, use_bcmatch=(not args.ignore_bcmatch)), m.NormalGuide
    return (
        f"{'_' if args.dont_fit_noise else ''}MixtureNormal{'+Acc' if args.scale_by_acc else ''}",
        partial(m.MixtureNormalModel, scale_by_accessibility=args.scale_by_acc, use_bcmatch=(not args.ignore_bcmatch,)),
        partial(m.MixtureNormalGuide, scale_by_accessibility=args.scale_by_acc, fit_noise=(not args.dont_fit_noise)),
    )


def identify_negctrl_model_guide(args, data_has_bcmatch):
    """bean/model/run.py:460-474."""
    use = (not args.ignore_bcmatch) and data_has_bcmatch
    m = sorting_model if getattr(args, "selection", "sorting") == "sorting" else survival_model
    return partial(m.ControlNormalModel, use_bcmatch=use), partial(m.ControlNormalGuide, use_bcmatch=use)
