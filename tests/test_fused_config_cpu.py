"""`fused.svi_config`: the BeanSviConfig the three fused engines pass to their C entry point, built without a GPU."""
import numpy as np
import pytest
import torch

from crispr_bean_b200 import _lib
from crispr_bean_b200.fused import set_prior_pointers, svi_config

EPS32, EPS64 = float(torch.finfo(torch.float32).eps), float(torch.finfo(torch.float64).eps)


def _cfg(**kw):
    args = dict(lr=0.01, gamma=0.1, num_steps=2000, seed=101, ll_const=-12.5)
    args.update(kw)
    return svi_config(**args)


def test_optimiser_counters_and_offsets():
    c, prior_v = _cfg(lr=0.02, gamma=0.25, num_steps=400, seed=7, guide_offset=1000, variant_offset=200)
    assert c.lr0 == 0.02 and c.lrd == 0.25 ** (1.0 / 400)
    assert (c.beta1, c.beta2, c.adam_eps, c.clip) == (0.9, 0.999, 1e-8, 10.0)
    assert c.seed == 7 and c.ll_const == -12.5
    assert (c.guide_offset, c.variant_offset) == (1000, 200)
    assert c.apply_update == 1 and c.model == _lib.MODEL_MIXTURE_NORMAL
    assert prior_v == {}
    assert _cfg(num_steps=0)[0].lrd == 0.1  # gamma ** (1 / max(num_steps, 1))


def test_default_priors():
    c, _ = _cfg(sd_scale=0.01)
    assert (c.mu_prior_normal, c.mu_prior_loc, c.mu_prior_scale) == (0, 0.0, 1.0)  # Laplace(0, 1)
    assert (c.sd_prior_loc, c.sd_prior_scale) == (0.0, 0.01)


def test_scalar_prior_params():
    c, prior_v = _cfg(sd_scale=0.01, prior_params={"mu_loc": 0.5, "sd_scale": torch.tensor([0.3])}, n_variants=4)
    assert (c.mu_prior_normal, c.mu_prior_loc, c.mu_prior_scale) == (1, 0.5, 1.0)
    assert (c.sd_prior_loc, c.sd_prior_scale) == (0.0, pytest.approx(0.3))
    assert prior_v == {}
    c, _ = _cfg(prior_params={"sd_loc": -1.0}, n_variants=4)
    assert c.mu_prior_normal == 0 and c.sd_prior_loc == -1.0


def test_per_variant_prior_params():
    T = 5
    pp = {"mu_loc": torch.arange(T, dtype=torch.float64), "mu_scale": torch.full((T, 1), 2.0),
          "sd_loc": torch.linspace(-1, 1, T), "sd_scale": 0.2}
    c, prior_v = _cfg(prior_params=pp, n_variants=T, dtype=torch.float32)
    assert c.mu_prior_normal == 1 and c.sd_prior_scale == 0.2
    assert sorted(prior_v) == ["mu_loc", "mu_scale", "sd_loc"]
    for key, t in prior_v.items():
        assert t.shape == (T,) and t.dtype == torch.float32 and t.is_contiguous()
        torch.testing.assert_close(t, pp[key].reshape(-1).float())
    state = _lib.BeanSviState()
    set_prior_pointers(state, prior_v)
    assert state.mu_prior_loc_v == prior_v["mu_loc"].data_ptr()
    assert state.sd_prior_loc_v == prior_v["sd_loc"].data_ptr()
    assert not state.sd_prior_scale_v


def test_prior_params_without_sd_site():
    """Survival has no sd site: sd keys are ignored and the sd prior stays (0, 1)."""
    c, prior_v = _cfg(sd_priors=False, prior_params={"mu_scale": torch.ones(3), "sd_loc": torch.zeros(3), "sd_scale": 5.0},
                      n_variants=3)
    assert c.mu_prior_normal == 1 and (c.sd_prior_loc, c.sd_prior_scale) == (0.0, 1.0)
    assert sorted(prior_v) == ["mu_scale"]


@pytest.mark.parametrize("unit", ["variants", "edits"])
def test_prior_params_length_mismatch(unit):
    with pytest.raises(ValueError, match=f"3 entries for 4 {unit}"):
        _cfg(prior_params={"mu_loc": torch.zeros(3)}, n_variants=4, unit=unit)


F32, F64 = torch.float32, torch.float64
NP = np.full(3, 0.5)


# (compute dtype, pi_a0, control_timepoint, promote) -> eps.  promote=False is the sorting / tiling rule: pi_a0's dtype, float64
# when computing in float64 or when pi_a0 is not a floating tensor; promote=True the survival rule: dtype promoted with the
# dtypes of pi_a0 and control_timepoint where they are tensors.
@pytest.mark.parametrize("dtype,pi_a0,ctp,promote,eps", [
    (F32, torch.full((3,), 0.5, dtype=F32), None, False, EPS32),
    (F32, torch.full((3,), 0.5, dtype=F64), None, False, EPS64),
    (F32, NP, None, False, EPS64),
    (F32, None, None, False, EPS64),
    (F64, torch.full((3,), 0.5, dtype=F32), None, False, EPS64),
    (F64, None, None, False, EPS64),
    (F32, torch.full((3,), 0.5, dtype=F32), torch.tensor([0.5], dtype=F32), True, EPS32),
    (F32, torch.full((3,), 0.5, dtype=F32), torch.tensor([0.5], dtype=F64), True, EPS64),
    (F32, torch.full((3,), 0.5, dtype=F64), torch.tensor([0.5], dtype=F32), True, EPS64),
    (F32, NP, torch.tensor([0.5], dtype=F32), True, EPS32),
    (F32, NP, torch.tensor([1]), True, EPS32),
    (F32, None, np.array([0.5]), True, EPS32),
    (F64, torch.full((3,), 0.5, dtype=F32), torch.tensor([0.5], dtype=F32), True, EPS64),
])
def test_prob_clamp_eps(dtype, pi_a0, ctp, promote, eps):
    c, _ = _cfg(dtype=dtype, pi_a0=pi_a0, control_timepoint=ctp, promote=promote)
    assert c.prob_clamp_eps == eps
