"""ctypes binding of libd3p_b200.so — the C ABI declared in include/d3p_b200.h.

There is NO fallback: if the shared library is missing or a call fails, this raises.
"""
import ctypes as C
import os

import numpy as np

from . import _build

MAX_LEAVES = 16

OK = 0
ERR_PEER_TIMEOUT = -5
FAMILY_LOGREG, FAMILY_GAUSS = 0, 1
LINK_EXP, LINK_SOFTPLUS = 0, 1
OPT_NONE, OPT_SGD, OPT_ADAM, OPT_ADADP = 0, 1, 2, 3
OPT_MOMENTUM, OPT_ADAGRAD, OPT_RMSPROP, OPT_RMSPROP_MOMENTUM, OPT_CLIPPED_ADAM = 4, 5, 6, 7, 8
OPT_SCHEDULED = 0x100
SCHED_CONSTANT, SCHED_EXPONENTIAL, SCHED_INVERSE_TIME, SCHED_POLYNOMIAL, SCHED_PIECEWISE = 0, 1, 2, 3, 4
MAX_BOUNDARIES = 16


class MeanfieldDesc(C.Structure):
    _fields_ = [("family", C.c_int32), ("link", C.c_int32), ("joint_site", C.c_int32), ("d", C.c_uint32),
                ("n_params", C.c_uint32), ("loc_off", C.c_uint32), ("rho_off", C.c_uint32),
                ("b_loc_off", C.c_uint32), ("b_rho_off", C.c_uint32), ("num_obs_total", C.c_float),
                ("lik_scale", C.c_float)]


class VaeDesc(C.Structure):
    _fields_ = [("out_dim", C.c_uint32), ("hidden_dim", C.c_uint32), ("z_dim", C.c_uint32), ("n_params", C.c_uint32),
                ("off_w4", C.c_uint32), ("off_b4", C.c_uint32), ("off_w5", C.c_uint32), ("off_b5", C.c_uint32),
                ("off_w1", C.c_uint32), ("off_b1", C.c_uint32), ("off_w2", C.c_uint32), ("off_b2", C.c_uint32),
                ("off_w3", C.c_uint32), ("off_b3", C.c_uint32), ("site_scale", C.c_float)]


class GmmDesc(C.Structure):
    _fields_ = [("K", C.c_uint32), ("d", C.c_uint32), ("n_params", C.c_uint32), ("alpha_off", C.c_uint32),
                ("mus_off", C.c_uint32), ("num_obs_total", C.c_float)]


class AutodiagDesc(C.Structure):
    _fields_ = [("latent_dim", C.c_uint32), ("n_params", C.c_uint32), ("loc_off", C.c_uint32),
                ("scale_off", C.c_uint32), ("num_obs_total", C.c_float)]


class LeafTable(C.Structure):
    _fields_ = [("n_leaves", C.c_uint32), ("leaf_off", C.c_uint32 * MAX_LEAVES),
                ("leaf_len", C.c_uint32 * MAX_LEAVES), ("site_state", (C.c_uint32 * 16) * MAX_LEAVES)]


class OptimDesc(C.Structure):
    _fields_ = [("kind", C.c_int32), ("step_size", C.c_float), ("b1", C.c_float), ("b2", C.c_float),
                ("eps", C.c_float), ("step", C.c_int32), ("tol", C.c_float), ("stability_check", C.c_int32),
                ("lr_d", C.c_void_p), ("err_ws_d", C.c_void_p),
                # appended: read only for kinds OPT_MOMENTUM .. OPT_CLIPPED_ADAM or with OPT_SCHEDULED
                ("momentum", C.c_float), ("gamma", C.c_float), ("clip_norm", C.c_float), ("schedule", C.c_int32),
                ("decay_steps", C.c_float), ("decay_rate", C.c_float), ("staircase", C.c_int32),
                ("final_step_size", C.c_float), ("power", C.c_float), ("n_boundaries", C.c_uint32),
                ("boundaries", C.c_float * MAX_BOUNDARIES), ("values", C.c_float * (MAX_BOUNDARIES + 1))]


class SamplerDesc(C.Structure):
    _fields_ = [("kind", C.c_int32), ("q", C.c_float), ("n_records", C.c_uint32), ("batch", C.c_uint32),
                ("suppress", C.c_int32), ("perm_d", C.c_void_p)]


SAMPLER_POISSON, SAMPLER_SUBSAMPLE, SAMPLER_SPLIT, SAMPLER_SUBSAMPLE_REPLACE = 0, 1, 2, 3

_u32p = C.POINTER(C.c_uint32)
_vp = C.c_void_p

_SIGNATURES = {
    "d3p_abi_version": (C.c_int32, []),
    "d3p_error_string": (C.c_char_p, [C.c_int32]),
    "d3p_event_create": (C.c_int32, [C.POINTER(C.c_void_p)]),
    "d3p_event_record": (C.c_int32, [_vp, _vp]),
    "d3p_event_elapsed_ms": (C.c_int32, [_vp, _vp, C.POINTER(C.c_float)]),
    "d3p_event_destroy": (C.c_int32, [_vp]),
    "d3p_chacha_key_from_seed_h": (C.c_int32, [_vp, C.c_size_t, _u32p]),
    "d3p_chacha_fold_in_h": (C.c_int32, [_u32p, C.c_uint32, _u32p]),
    "d3p_chacha_split_h": (C.c_int32, [_u32p, C.c_int32, _u32p]),
    "d3p_chacha_random_bits_h": (C.c_int32, [_u32p, C.c_uint64, _u32p, C.c_size_t]),
    "d3p_chacha_random_bits": (C.c_int32, [_u32p, C.c_uint64, _vp, C.c_size_t, _vp]),
    "d3p_chacha_uniform_f32": (C.c_int32, [_u32p, C.c_uint64, C.c_float, C.c_float, _vp, C.c_size_t, _vp]),
    "d3p_chacha_normal_f32": (C.c_int32, [_u32p, C.c_uint64, _vp, C.c_size_t, _vp]),
    "d3p_chacha_randint_round_u32": (C.c_int32, [_u32p, C.c_uint32, C.c_uint32, C.c_int32, _vp, C.c_size_t, _vp, _vp]),
    "d3p_randint_finish_i32": (C.c_int32, [_vp, C.c_int32, _vp, C.c_size_t, _vp]),
    "d3p_chacha_randint_round": (C.c_int32, [_u32p, C.c_uint32, C.c_uint32, C.c_uint32, C.c_int32, _vp, C.c_size_t, _vp, _vp]),
    "d3p_randint_finish": (C.c_int32, [_vp, C.c_int32, C.c_uint32, _vp, C.c_size_t, _vp]),
    "d3p_chacha_randint": (C.c_int32, [_u32p, C.c_uint32, C.c_int64, C.c_int64, _vp, C.c_size_t, _vp]),
    "d3p_randint_bitmask": (C.c_uint32, [C.c_uint32, C.c_uint32]),
    "d3p_feistel_round_constants_h": (C.c_int32, [_u32p, _u32p]),
    "d3p_feistel_sample": (C.c_int32, [_u32p, C.c_uint32, C.c_uint32, C.c_uint32, _vp, _vp]),
    "d3p_poisson_workspace_bytes": (C.c_size_t, [C.c_uint32]),
    "d3p_poisson_sample": (C.c_int32, [_u32p, C.c_float, C.c_uint32, C.c_uint32, C.c_int32, _vp, _vp, _vp, _vp,
                                       C.c_size_t, _vp]),
    "d3p_gather_rows_masked": (C.c_int32, [_vp, C.c_size_t, _vp, _vp, C.c_uint32, _vp, _vp]),
    "d3p_clip_rows_f32": (C.c_int32, [_vp, C.c_uint32, C.c_uint32, C.c_float, _vp, _vp]),
    "d3p_vector_norm_f32": (C.c_int32, [_vp, C.c_size_t, C.c_float, _vp, _vp]),
    "d3p_clip_and_sum_workspace_bytes": (C.c_size_t, [C.c_uint32, C.c_uint32]),
    "d3p_clip_and_sum_f32": (C.c_int32, [_vp, _vp, _vp, C.c_uint32, C.c_uint32, C.c_float, _vp, _vp, C.c_size_t, _vp]),
    "d3p_meanfield_workspace_bytes": (C.c_size_t, [C.POINTER(MeanfieldDesc), _u32p]),
    "d3p_dpsvi_step_meanfield": (C.c_int32, [C.POINTER(MeanfieldDesc), _vp, _vp, C.c_size_t, _vp, _vp, _vp, _vp,
                                             C.c_uint32, C.c_uint32, C.c_uint32, _u32p, C.c_float, C.c_float,
                                             _vp, _vp, _vp, _vp, C.c_size_t, _vp]),  # norms, grads, loss, ws
    "d3p_autodiag_draw_f32": (C.c_int32, [C.POINTER(AutodiagDesc), _vp, _u32p, C.c_uint32, C.c_uint32, C.c_uint32,
                                          _vp, _vp, C.c_size_t, _vp]),
    "d3p_autodiag_workspace_bytes": (C.c_size_t, [C.POINTER(AutodiagDesc), C.c_uint32, _u32p]),
    "d3p_dpsvi_step_autodiag": (C.c_int32, [C.POINTER(AutodiagDesc), _vp, _vp, _vp, C.c_size_t, _vp, _vp, _vp,
                                            C.c_uint32, C.c_uint32, C.c_uint32, C.c_float, C.c_float,
                                            _vp, _vp, _vp, _vp, C.c_size_t, _vp]),  # norms, grads, loss, ws
    "d3p_perturb_finalize_f32": (C.c_int32, [_vp, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(LeafTable),
                                             C.c_float, C.c_float, C.c_float, C.c_int32, _vp,
                                             C.POINTER(OptimDesc), _vp, _vp, _vp, _vp,
                                             C.POINTER(C.c_float), _vp]),
    "d3p_optim_step_size": (C.c_int32, [C.POINTER(OptimDesc), C.c_int32, C.POINTER(C.c_float)]),
    "d3p_adadp_workspace_floats": (C.c_size_t, [C.c_uint32]),
    "d3p_adadp_finish_f32": (C.c_int32, [C.POINTER(OptimDesc), C.c_uint32, _vp, _vp, _vp]),
    "d3p_dpsvi_epoch_workspace_bytes": (C.c_size_t, [C.POINTER(MeanfieldDesc), C.POINTER(SamplerDesc)]),
    "d3p_dpsvi_run_epoch_meanfield": (C.c_int32, [C.POINTER(MeanfieldDesc), C.POINTER(SamplerDesc), _vp, C.c_size_t,
                                                  _vp, _u32p, _u32p, C.c_uint32, C.c_uint32, C.c_float, C.c_float,
                                                  C.c_float, C.POINTER(LeafTable), C.POINTER(OptimDesc), _vp, _vp,
                                                  _vp, _vp, _vp, _vp, C.c_size_t, _vp, _vp]),
    "d3p_dpsvi_epoch_gmm_workspace_bytes": (C.c_size_t, [C.POINTER(GmmDesc), C.POINTER(SamplerDesc)]),
    "d3p_dpsvi_run_epoch_gmm": (C.c_int32, [C.POINTER(GmmDesc), C.POINTER(SamplerDesc), _vp, C.c_size_t,
                                            _u32p, _u32p, C.c_uint32, C.c_uint32, C.c_float, C.c_float,
                                            C.c_float, C.POINTER(LeafTable), C.POINTER(OptimDesc), _vp, _vp,
                                            _vp, _vp, _vp, _vp, C.c_size_t, _vp, _vp]),
    "d3p_dpsvi_epoch_vae_workspace_bytes": (C.c_size_t, [C.POINTER(VaeDesc), C.POINTER(SamplerDesc), C.c_int32]),
    "d3p_dpsvi_run_epoch_vae": (C.c_int32, [C.POINTER(VaeDesc), C.POINTER(SamplerDesc), _vp, C.c_size_t,
                                            _u32p, _u32p, C.c_uint32, C.c_uint32, C.c_float, C.c_float,
                                            C.c_float, C.POINTER(LeafTable), C.POINTER(OptimDesc), _vp, _vp,
                                            _vp, _vp, _vp, _vp, C.c_size_t, _vp, _vp]),
    "d3p_comm_create": (C.c_int32, [C.c_int32, C.c_int32, C.c_uint32, C.c_uint32, C.POINTER(C.c_void_p),
                                    C.POINTER(C.c_uint8)]),
    "d3p_poisson_sample_sharded": (C.c_int32, [_vp, _u32p, C.c_float, C.c_uint32, C.c_uint32, C.c_int32, C.c_uint32,
                                               C.c_uint32, _vp, _vp, _vp, _vp, C.c_size_t, _vp]),
    "d3p_comm_connect": (C.c_int32, [_vp, C.POINTER(C.c_uint8)]),
    "d3p_comm_timeouts": (C.c_int32, [_vp, _u32p]),
    "d3p_comm_window": (C.c_int32, [_vp, C.POINTER(C.c_void_p), C.POINTER(C.c_size_t)]),
    "d3p_comm_connect_local": (C.c_int32, [_vp, C.POINTER(C.c_void_p)]),
    "d3p_comm_timeout_detail": (C.c_int32, [_vp, _u32p]),
    "d3p_comm_set_timeout_ms": (C.c_int32, [_vp, C.c_uint32]),
    "d3p_comm_set_sampler_margin": (C.c_int32, [_vp, C.c_uint32]),
    "d3p_comm_destroy": (C.c_int32, [_vp]),
    "d3p_perturb_finalize_p2p_f32": (C.c_int32, [_vp, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(LeafTable),
                                                 C.c_float, C.c_float, C.c_float, C.c_int32, _vp,
                                                 C.POINTER(OptimDesc), _vp, _vp, _vp, _vp,
                                                 C.POINTER(C.c_float), _vp, _vp]),
    "d3p_reduce_partials_f32": (C.c_int32, [_vp, C.c_uint32, C.c_uint32, _vp, _vp]),
    "d3p_vae_workspace_bytes": (C.c_size_t, [C.POINTER(VaeDesc), C.c_uint32, _u32p]),
    "d3p_vae_ctx_create": (C.c_int32, [C.POINTER(C.c_void_p)]),
    "d3p_epoch_ctx_create": (C.c_int32, [C.POINTER(C.c_void_p)]),
    "d3p_epoch_ctx_destroy": (C.c_int32, [_vp]),
    "d3p_vae_ctx_destroy": (C.c_int32, [_vp]),
    "d3p_dpsvi_step_vae": (C.c_int32, [C.POINTER(VaeDesc), _vp, _vp, C.c_size_t, _vp, _vp, _vp, C.c_uint32, C.c_uint32,
                                       C.c_uint32, _u32p, C.c_float, C.c_float, _vp, _vp, _vp, C.c_size_t,
                                       C.POINTER(C.c_void_p), _vp, _vp]),
    # ---- device-key forms: every key argument is a device pointer (c_void_p) ----
    "d3p_chacha_split_dk": (C.c_int32, [_vp, C.c_int32, _vp, _vp]),
    "d3p_chacha_fold_in_dk": (C.c_int32, [_vp, _vp, C.c_uint32, _vp, _vp]),
    "d3p_chacha_random_bits_dk": (C.c_int32, [_vp, C.c_uint64, _vp, C.c_size_t, _vp]),
    "d3p_chacha_uniform_f32_dk": (C.c_int32, [_vp, C.c_uint64, C.c_float, C.c_float, _vp, C.c_size_t, _vp]),
    "d3p_chacha_normal_f32_dk": (C.c_int32, [_vp, C.c_uint64, _vp, C.c_size_t, _vp]),
    "d3p_chacha_randint_dk": (C.c_int32, [_vp, C.c_uint32, C.c_int64, C.c_int64, _vp, C.c_size_t, _vp]),
    "d3p_dpsvi_keys_dk": (C.c_int32, [_vp, C.c_uint32, _vp, _vp, _vp]),
    "d3p_feistel_round_constants_dk": (C.c_int32, [_vp, _vp, _vp]),
    "d3p_feistel_sample_dk": (C.c_int32, [_vp, C.c_uint32, C.c_uint32, C.c_uint32, _vp, _vp]),
    "d3p_poisson_sample_dk": (C.c_int32, [_vp, C.c_float, C.c_uint32, C.c_uint32, C.c_int32, _vp, _vp, _vp, _vp,
                                          C.c_size_t, _vp]),
    "d3p_poisson_sample_sharded_dk": (C.c_int32, [_vp, _vp, C.c_float, C.c_uint32, C.c_uint32, C.c_int32, C.c_uint32,
                                                  C.c_uint32, _vp, _vp, _vp, _vp, C.c_size_t, _vp]),
    "d3p_dpsvi_step_meanfield_dk": (C.c_int32, [C.POINTER(MeanfieldDesc), _vp, _vp, C.c_size_t, _vp, _vp, _vp, _vp,
                                                C.c_uint32, C.c_uint32, C.c_uint32, _vp, C.c_float, C.c_float,
                                                _vp, _vp, _vp, _vp, C.c_size_t, _vp]),
    "d3p_autodiag_draw_f32_dk": (C.c_int32, [C.POINTER(AutodiagDesc), _vp, _vp, C.c_uint32, C.c_uint32, C.c_uint32,
                                             _vp, _vp, C.c_size_t, _vp]),
    "d3p_dpsvi_step_vae_dk": (C.c_int32, [C.POINTER(VaeDesc), _vp, _vp, C.c_size_t, _vp, _vp, _vp, C.c_uint32, C.c_uint32,
                                          C.c_uint32, _vp, C.c_float, C.c_float, _vp, _vp, _vp, C.c_size_t,
                                          C.POINTER(C.c_void_p), _vp, _vp]),
    "d3p_dpsvi_step_gmm_dk": (C.c_int32, [C.POINTER(GmmDesc), _vp, _vp, C.c_size_t, _vp, _vp, _vp, C.c_uint32, C.c_uint32,
                                          C.c_uint32, _vp, C.c_float, C.c_float, _vp, _vp, _vp, _vp, C.c_size_t, _vp]),
    "d3p_perturb_finalize_dk_f32": (C.c_int32, [_vp, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(LeafTable), _vp,
                                                C.c_float, C.c_float, C.c_float, _vp, C.POINTER(OptimDesc), _vp, _vp,
                                                _vp, _vp, _vp, _vp]),
    "d3p_dpsvi_run_epoch_meanfield_dk": (C.c_int32, [C.POINTER(MeanfieldDesc), C.POINTER(SamplerDesc), _vp, C.c_size_t,
                                                     _vp, _vp, _vp, C.c_uint32, C.c_uint32, C.c_float, C.c_float,
                                                     C.c_float, C.POINTER(LeafTable), C.POINTER(OptimDesc), _vp, _vp,
                                                     _vp, _vp, _vp, _vp, C.c_size_t, _vp, _vp]),
    "d3p_dpsvi_run_epoch_vae_dk": (C.c_int32, [C.POINTER(VaeDesc), C.POINTER(SamplerDesc), _vp, C.c_size_t,
                                               _vp, _vp, C.c_uint32, C.c_uint32, C.c_float, C.c_float,
                                               C.c_float, C.POINTER(LeafTable), C.POINTER(OptimDesc), _vp, _vp,
                                               _vp, _vp, _vp, _vp, C.c_size_t, _vp, _vp]),
    "d3p_gmm_log_prob_f32": (C.c_int32, [_vp, C.c_size_t, _vp, _vp, _vp, C.c_uint32, C.c_uint32, C.c_uint32, _vp, _vp]),
    "d3p_gmm_workspace_bytes": (C.c_size_t, [C.POINTER(GmmDesc), _u32p]),
    "d3p_dpsvi_step_gmm": (C.c_int32, [C.POINTER(GmmDesc), _vp, _vp, C.c_size_t, _vp, _vp, _vp, C.c_uint32, C.c_uint32,
                                       C.c_uint32, _u32p, C.c_float, C.c_float, _vp, _vp, _vp, _vp, C.c_size_t, _vp]),
    "d3p_elbo_evaluate_workspace_bytes": (C.c_size_t, []),
    "d3p_elbo_evaluate_meanfield": (C.c_int32, [C.POINTER(MeanfieldDesc), _vp, _vp, C.c_size_t, _vp, _vp, C.c_uint32,
                                                _u32p, _vp, _vp, C.c_size_t, _vp]),
    "d3p_elbo_evaluate_vae": (C.c_int32, [C.POINTER(VaeDesc), _vp, _vp, C.c_size_t, _vp, C.c_uint32, _u32p, _vp, _vp,
                                          C.c_size_t, _vp, _vp]),
    "d3p_elbo_evaluate_gmm_workspace_bytes": (C.c_size_t, [C.POINTER(GmmDesc)]),
    "d3p_elbo_evaluate_gmm": (C.c_int32, [C.POINTER(GmmDesc), _vp, _vp, C.c_size_t, _vp, C.c_uint32, _u32p, _vp, _vp,
                                          C.c_size_t, _vp]),
    "d3p_threefry_random_bits": (C.c_int32, [_u32p, _vp, C.c_size_t, _vp]),
    "d3p_threefry_uniform_f32": (C.c_int32, [_u32p, C.c_float, C.c_float, _vp, C.c_size_t, _vp]),
    "d3p_threefry_normal_f32": (C.c_int32, [_u32p, _vp, C.c_size_t, _vp]),
    "d3p_threefry_gamma_f32": (C.c_int32, [_u32p, _vp, C.c_uint32, C.c_uint32, C.c_int32, _vp, _vp]),
    "d3p_split_tf32": (C.c_int32, [_vp, _vp, C.c_uint32, _vp, _vp, C.c_size_t, _vp]),
    "d3p_gemm_f32x3": (C.c_int32, [_vp, C.c_int32, C.c_size_t, _vp, C.c_int32, C.c_size_t, C.c_uint32, C.c_uint32,
                                   C.c_uint32, C.c_uint32, C.c_int32, _vp, C.c_size_t, C.c_size_t, C.c_int32, _vp]),
    "d3p_gemm_tf32x3": (C.c_int32, [_vp, _vp, C.c_int32, C.c_size_t, _vp, _vp, C.c_int32, C.c_size_t, C.c_uint32,
                                    C.c_uint32, C.c_uint32, C.c_uint32, C.c_int32, _vp, C.c_size_t, C.c_size_t,
                                    C.c_int32, _vp]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)
_lib = None


class D3PNativeError(RuntimeError):
    pass


def lib():
    """Load libd3p_b200.so (once).  Raises if it has not been built — there is no CPU fallback."""
    global _lib
    if _lib is None:
        path = _build.lib_path()
        if not os.path.exists(path):
            raise D3PNativeError(
                f"{path} is missing: build it with `python -m d3p_b200._build` "
                "(d3p_b200 has no CPU fallback; the CUDA library is the product).")
        handle = C.CDLL(path)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, args
        _lib = handle
    return _lib


def check(rc, what=""):
    if rc != OK:
        msg = lib().d3p_error_string(rc).decode()
        raise D3PNativeError(f"{what or 'd3p_b200 call'} failed: {msg} (code {rc})")


def u32(arr):
    """numpy uint32 array (contiguous) -> ctypes pointer; keeps `arr` alive via the return pair."""
    a = np.ascontiguousarray(arr, dtype=np.uint32)
    return a, a.ctypes.data_as(_u32p)


def ptr(t):
    """device pointer of a torch CUDA tensor (or None)."""
    if t is None:
        return None
    return C.c_void_p(t.data_ptr())


def stream_ptr():
    import torch
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)
