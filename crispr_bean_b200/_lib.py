"""ctypes binding of `libbean_b200.so` (declared in include/bean_b200.h).

There is no CPU fallback: if the library is missing or a call fails, this raises.
"""
from __future__ import annotations

import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
# BEAN_B200_LIB: an A/B build of the same library (tools/build_variants.sh), for kernel experiments on the GPU box only
LIB_PATH = os.environ.get("BEAN_B200_LIB") or os.path.join(_PKG, "libbean_b200.so")

BEAN_OK = 0
MODE_SORTING, MODE_SURVIVAL = 0, 1
MAX_BINS, MAX_RB, MAX_ALLELES, MAX_LAYERS = 8, 64, 4096, 2
SURV_FOLD_ROWS = 1024  # BEAN_SURV_FOLD_ROWS
MAX_PEERS, PEER_MAX_VALS = 8, 72  # BEAN_MAX_PEERS, BEAN_PEER_MAX_VALS


class BeanError(RuntimeError):
    pass


class BeanScreen(C.Structure):
    _fields_ = [
        ("n_guides", C.c_int32), ("n_reps", C.c_int32), ("n_bins", C.c_int32), ("n_layers", C.c_int32),
        ("mode", C.c_int32), ("mask_thres", C.c_int32),
        ("x", C.c_void_p), ("a0", C.c_void_p), ("row_mask", C.c_void_p), ("row_const", C.c_void_p),
        ("size_factor", C.POINTER(C.c_double)), ("sample_mask", C.POINTER(C.c_double)),
        ("upper_thres", C.POINTER(C.c_double)), ("lower_thres", C.POINTER(C.c_double)),
        ("timepoints", C.POINTER(C.c_double)),
    ]


class BeanLLArgs(C.Structure):
    _fields_ = [
        ("n_alleles", C.c_int32),
        ("mu_allele", C.c_void_p), ("sd_allele", C.c_void_p), ("pi", C.c_void_p), ("allele_mask", C.c_void_p),
        ("ll_row", C.c_void_p), ("ll_partial", C.c_void_p),
        ("d_mu", C.c_void_p), ("d_sd", C.c_void_p), ("d_pi", C.c_void_p),
    ]


class BeanSviConfig(C.Structure):
    _fields_ = [
        ("model", C.c_int32), ("sd_is_sqrt", C.c_int32), ("mu_prior_normal", C.c_int32), ("apply_update", C.c_int32),
        ("phases", C.c_int32), ("fit_noise", C.c_int32), ("force_generic", C.c_int32), ("reserved_", C.c_int32),
        ("mu_prior_loc", C.c_double), ("mu_prior_scale", C.c_double),
        ("sd_prior_loc", C.c_double), ("sd_prior_scale", C.c_double),
        ("lr0", C.c_double), ("lrd", C.c_double),
        ("beta1", C.c_double), ("beta2", C.c_double), ("adam_eps", C.c_double), ("clip", C.c_double),
        ("ll_const", C.c_double), ("prob_clamp_eps", C.c_double), ("seed", C.c_uint64),
        ("guide_offset", C.c_uint32), ("variant_offset", C.c_uint32),
    ]


class BeanSviState(C.Structure):
    _fields_ = [
        ("n_variants", C.c_int32), ("loss_capacity", C.c_int32),
        ("guide_variant", C.c_void_p), ("variant_ptr", C.c_void_p),
        ("allele_counts", C.c_void_p), ("pi_a0", C.c_void_p),
        ("var_params", C.c_void_p), ("var_m", C.c_void_p), ("var_v", C.c_void_p),
        ("alpha_u", C.c_void_p), ("alpha_m", C.c_void_p), ("alpha_v", C.c_void_p),
        ("d_guide", C.c_void_p), ("var_grad", C.c_void_p), ("alpha_grad", C.c_void_p),
        ("partial", C.c_void_p), ("counter", C.c_void_p), ("loss", C.c_void_p),
        ("acc_k", C.c_void_p), ("noise_u", C.c_void_p), ("noise_m", C.c_void_p), ("noise_v", C.c_void_p),
        ("noise_grad", C.c_void_p),
        ("mu_prior_loc_v", C.c_void_p), ("mu_prior_scale_v", C.c_void_p), ("sd_prior_loc_v", C.c_void_p), ("sd_prior_scale_v", C.c_void_p),
        ("pw", C.c_void_p), ("dconc", C.c_void_p), ("nonfinite_step", C.c_void_p),
    ]


class BeanSviNoise(C.Structure):
    _fields_ = [("eps_mu", C.c_void_p), ("eps_sd", C.c_void_p), ("pi", C.c_void_p), ("eps_noise", C.c_void_p),
                ("eps_out", C.c_void_p), ("pi_out", C.c_void_p)]


class BeanAlleleMap(C.Structure):
    _fields_ = [("n_guides", C.c_int32), ("n_alleles", C.c_int32), ("n_edits", C.c_int32), ("nnz", C.c_int32),
                ("allele_ptr", C.c_void_p), ("allele_edit", C.c_void_p), ("edit_ptr", C.c_void_p), ("edit_slot", C.c_void_p)]


ADAM_MAX_TENSORS = 16


class BeanAdamTensor(C.Structure):
    _fields_ = [("theta", C.c_void_p), ("grad", C.c_void_p), ("m", C.c_void_p), ("v", C.c_void_p), ("n", C.c_int64)]


class BeanAdamArgs(C.Structure):
    _fields_ = [("n_tensors", C.c_int32), ("tensors", BeanAdamTensor * ADAM_MAX_TENSORS),
                ("step_sizes", C.c_void_p), ("step", C.c_void_p), ("n_steps", C.c_int64),
                ("beta1", C.c_double), ("beta2", C.c_double), ("eps", C.c_double), ("clip", C.c_double),
                ("loss", C.c_void_p), ("nonfinite_step", C.c_void_p)]


class BeanPiSitesArgs(C.Structure):
    _fields_ = [("n_guides", C.c_int32), ("n_reps", C.c_int32), ("n_alleles", C.c_int32), ("n_controls", C.c_int32),
                ("mask_guide_site", C.c_int32),
                ("conc_guide", C.c_void_p), ("conc_model", C.c_void_p), ("pi", C.c_void_p), ("counts", C.c_void_p),
                ("rep_guide_mask", C.c_void_p), ("growth", C.c_void_p), ("control_time", C.POINTER(C.c_double)),
                ("prob_eps", C.c_double), ("partial", C.c_void_p),
                ("d_conc_guide", C.c_void_p), ("d_conc_model", C.c_void_p), ("d_pi", C.c_void_p), ("d_growth", C.c_void_p)]


class BeanLatentSitesArgs(C.Structure):
    _fields_ = [("n", C.c_int64), ("has_sd", C.c_int32), ("mu_prior_normal", C.c_int32),
                ("mu_loc", C.c_void_p), ("mu_log_scale", C.c_void_p), ("sd_loc", C.c_void_p), ("sd_log_scale", C.c_void_p),
                ("eps_mu", C.c_void_p), ("eps_sd", C.c_void_p),
                ("mu_prior_loc", C.c_double), ("mu_prior_scale", C.c_double), ("sd_prior_loc", C.c_double), ("sd_prior_scale", C.c_double),
                ("mu_prior_loc_v", C.c_void_p), ("mu_prior_scale_v", C.c_void_p), ("sd_prior_loc_v", C.c_void_p), ("sd_prior_scale_v", C.c_void_p),
                ("mu", C.c_void_p), ("sd", C.c_void_p), ("partial", C.c_void_p), ("dv", C.c_void_p)]


class BeanLatentSitesGradArgs(C.Structure):
    _fields_ = [("n", C.c_int64), ("has_sd", C.c_int32),
                ("mu_log_scale", C.c_void_p), ("sd_log_scale", C.c_void_p), ("eps_mu", C.c_void_p), ("eps_sd", C.c_void_p),
                ("sd", C.c_void_p), ("dv", C.c_void_p), ("g_mu", C.c_void_p), ("g_sd", C.c_void_p), ("g_v", C.c_void_p),
                ("grad", C.c_void_p)]


class BeanDirichletArgs(C.Structure):
    _fields_ = [("n_guides", C.c_int32), ("n_reps", C.c_int32), ("n_alleles", C.c_int32), ("site", C.c_uint32),
                ("conc", C.c_void_p), ("x", C.c_void_p), ("grad_x", C.c_void_p), ("d_conc", C.c_void_p),
                ("seed", C.c_uint64), ("guide_offset", C.c_uint32), ("step", C.c_void_p), ("step_value", C.c_int64)]


class BeanPeerBuffer(C.Structure):  # lives in device memory; mirrored for its size and layout only
    _fields_ = [("vals", C.c_double * PEER_MAX_VALS * MAX_PEERS * 2), ("flag", C.c_uint64 * MAX_PEERS * 2), ("timeouts", C.c_uint64)]


class BeanPeerExchange(C.Structure):
    _fields_ = [("world", C.c_int32), ("rank", C.c_int32), ("buf", C.c_void_p * MAX_PEERS)]


class BeanSurvivalState(C.Structure):
    _fields_ = [("n_controls", C.c_int32), ("prime", C.c_int32), ("n_guides_total", C.c_int64),
                ("control_time", C.POINTER(C.c_double)), ("negctrl_loc", C.c_double), ("negctrl_scale", C.c_double),
                ("log_obs", C.c_void_p), ("q0_u", C.c_void_p), ("q0_m", C.c_void_p), ("q0_v", C.c_void_p), ("q0_grad", C.c_void_p),
                ("gamma", C.c_void_p * 2), ("sums", C.c_void_p * 2), ("abund_partial", C.c_void_p),
                ("peers", C.POINTER(BeanPeerExchange)), ("nonfinite_step", C.c_void_p)]


class BeanSurvivalNoise(C.Structure):
    _fields_ = [("eps_negctrl", C.c_void_p), ("q0", C.c_void_p)]


class BeanTilingState(C.Structure):
    _fields_ = [("map", C.POINTER(BeanAlleleMap)), ("n_controls", C.c_int32), ("loss_capacity", C.c_int32),
                ("allele_mask", C.c_void_p), ("pi_a0", C.c_void_p), ("counts", C.c_void_p),
                ("edit_params", C.c_void_p), ("edit_m", C.c_void_p), ("edit_v", C.c_void_p), ("edit_grad", C.c_void_p),
                ("alpha_u", C.c_void_p), ("alpha_m", C.c_void_p), ("alpha_v", C.c_void_p), ("alpha_grad", C.c_void_p),
                ("mu_e", C.c_void_p), ("sd_e", C.c_void_p), ("d_slot", C.c_void_p),
                ("partial", C.c_void_p), ("counter", C.c_void_p), ("loss", C.c_void_p),
                ("mu_prior_loc_v", C.c_void_p), ("mu_prior_scale_v", C.c_void_p), ("sd_prior_loc_v", C.c_void_p), ("sd_prior_scale_v", C.c_void_p),
                ("epsilon", C.c_double), ("pi_tiny", C.c_double),
                ("edit_sum", C.c_void_p), ("edit_iota", C.c_void_p), ("edit_term_weight", C.c_double),
                ("nonfinite_step", C.c_void_p)]


class BeanTilingNoise(C.Structure):
    _fields_ = [("eps_mu", C.c_void_p), ("eps_sd", C.c_void_p), ("pi", C.c_void_p), ("eps_out", C.c_void_p), ("pi_out", C.c_void_p)]


SURV_PRIME_NONE, SURV_PRIME_AND_RUN, SURV_PRIME_ONLY = 0, 1, 2
MODEL_NORMAL, MODEL_MIXTURE_NORMAL = 0, 1
ABI_VERSION = 16  # include/bean_b200.h: BEAN_ABI_VERSION
_GATHER = [C.POINTER(BeanAlleleMap), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
_SCATTER = [C.POINTER(BeanAlleleMap), C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]

# every symbol include/bean_b200.h declares: name -> (restype, argtypes)
_PROTOTYPES = {
    "bean_abi_version": (C.c_int, []),
    "bean_last_error": (C.c_char_p, []),
    "bean_device_sm_count": (C.c_int, []),
    "bean_ll_num_partials": (C.c_int, [C.c_int32, C.c_int32]),
    "bean_ll_f32": (C.c_int, [C.POINTER(BeanScreen), C.POINTER(BeanLLArgs), C.c_void_p]),
    "bean_ll_f64": (C.c_int, [C.POINTER(BeanScreen), C.POINTER(BeanLLArgs), C.c_void_p]),
    "bean_allele_gather_f32": (C.c_int, _GATHER), "bean_allele_gather_f64": (C.c_int, _GATHER),
    "bean_allele_scatter_f32": (C.c_int, _SCATTER), "bean_allele_scatter_f64": (C.c_int, _SCATTER),
    "bean_svi_num_partials": (C.c_int, [C.c_int32, C.c_int32]),
    "bean_svi_run_f32": (C.c_int, [C.POINTER(BeanScreen), C.POINTER(BeanSviState), C.POINTER(BeanSviConfig),
                                   C.POINTER(BeanSviNoise), C.c_int32, C.c_int32, C.c_void_p]),
    "bean_svi_run_f64": (C.c_int, [C.POINTER(BeanScreen), C.POINTER(BeanSviState), C.POINTER(BeanSviConfig),
                                   C.POINTER(BeanSviNoise), C.c_int32, C.c_int32, C.c_void_p]),
    "bean_svi_survival_run_f32": (C.c_int, [C.POINTER(BeanScreen), C.POINTER(BeanSviState), C.POINTER(BeanSurvivalState),
                                            C.POINTER(BeanSviConfig), C.POINTER(BeanSviNoise), C.POINTER(BeanSurvivalNoise),
                                            C.c_int32, C.c_int32, C.c_void_p]),
    "bean_svi_survival_run_f64": (C.c_int, [C.POINTER(BeanScreen), C.POINTER(BeanSviState), C.POINTER(BeanSurvivalState),
                                            C.POINTER(BeanSviConfig), C.POINTER(BeanSviNoise), C.POINTER(BeanSurvivalNoise),
                                            C.c_int32, C.c_int32, C.c_void_p]),
    "bean_row_const_f32": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bean_row_const_f64": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p]),
    "bean_peer_exchange_bytes": (C.c_int, []),
    "bean_peer_alloc": (C.c_int, [C.POINTER(C.c_void_p), C.POINTER(C.c_ubyte)]),
    "bean_peer_open": (C.c_int, [C.POINTER(C.c_ubyte), C.POINTER(C.c_void_p)]),
    "bean_peer_close": (C.c_int, [C.c_void_p]),
    "bean_peer_free": (C.c_int, [C.c_void_p]),
    "bean_peer_timeouts": (C.c_int, [C.c_void_p, C.POINTER(C.c_uint64)]),
    "bean_peer_reset_flags": (C.c_int, [C.c_void_p]),
    "bean_svi_tiling_num_partials": (C.c_int, [C.c_int32, C.c_int32]),
    "bean_svi_tiling_run_f32": (C.c_int, [C.POINTER(BeanScreen), C.POINTER(BeanTilingState), C.POINTER(BeanSviConfig),
                                          C.POINTER(BeanTilingNoise), C.c_int32, C.c_int32, C.c_void_p]),
    "bean_svi_tiling_run_f64": (C.c_int, [C.POINTER(BeanScreen), C.POINTER(BeanTilingState), C.POINTER(BeanSviConfig),
                                          C.POINTER(BeanTilingNoise), C.c_int32, C.c_int32, C.c_void_p]),
    "bean_pi_sites_f32": (C.c_int, [C.POINTER(BeanPiSitesArgs), C.c_void_p]),
    "bean_pi_sites_f64": (C.c_int, [C.POINTER(BeanPiSitesArgs), C.c_void_p]),
    "bean_latent_sites_num_partials": (C.c_int, [C.c_int64]),
    "bean_latent_sites_f32": (C.c_int, [C.POINTER(BeanLatentSitesArgs), C.c_void_p]),
    "bean_latent_sites_f64": (C.c_int, [C.POINTER(BeanLatentSitesArgs), C.c_void_p]),
    "bean_latent_sites_grad_f32": (C.c_int, [C.POINTER(BeanLatentSitesGradArgs), C.c_void_p]),
    "bean_latent_sites_grad_f64": (C.c_int, [C.POINTER(BeanLatentSitesGradArgs), C.c_void_p]),
    "bean_clipped_adam_f32": (C.c_int, [C.POINTER(BeanAdamArgs), C.c_void_p]),
    "bean_clipped_adam_f64": (C.c_int, [C.POINTER(BeanAdamArgs), C.c_void_p]),
    "bean_dirichlet_rsample_f32": (C.c_int, [C.POINTER(BeanDirichletArgs), C.c_void_p]),
    "bean_dirichlet_rsample_f64": (C.c_int, [C.POINTER(BeanDirichletArgs), C.c_void_p]),
    "bean_dirichlet_rsample_grad_f32": (C.c_int, [C.POINTER(BeanDirichletArgs), C.c_void_p]),
    "bean_dirichlet_rsample_grad_f64": (C.c_int, [C.POINTER(BeanDirichletArgs), C.c_void_p]),
    "bean_row_ceiling_f32": (C.c_int, [C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "bean_row_ceiling_lanes_f32": (C.c_int, [C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
}

_lib = None


def exported_symbols():
    return sorted(_PROTOTYPES)


def lib() -> C.CDLL:
    """Load the library (building it if nvcc is around and it is missing); raise if impossible."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            from .build import build
            build()
        try:
            handle = C.CDLL(LIB_PATH)
        except OSError as exc:  # pragma: no cover
            raise BeanError(f"cannot load {LIB_PATH}: {exc} (the CUDA extension is required; no CPU fallback)") from exc
        for name, (res, args) in _PROTOTYPES.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        if handle.bean_abi_version() != ABI_VERSION:
            raise BeanError(f"{LIB_PATH} has ABI version {handle.bean_abi_version()}, expected {ABI_VERSION}: rebuild it "
                            "(python -m crispr_bean_b200.build --force)")
        _lib = handle
    return _lib


def check(rc: int, what: str):
    if rc != BEAN_OK:
        msg = lib().bean_last_error().decode(errors="replace")
        raise BeanError(f"{what} failed (code {rc}): {msg}")
