"""ctypes binding of libpbx (include/pbx.h).  The library is mandatory: there is
no CPU fallback -- ``load()`` raises if the shared object is missing, and every
device entry point raises ``PbxError`` on a non-zero status."""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "csrc", "libpbx.so")

PBX_MAX_DIMS = 8
PBX_MAX_PARAMS = 3
ACCEPT_REFERENCE, ACCEPT_LOG = 0, 1
PROP_NORMAL, PROP_UNIFORM, PROP_SPHERICAL = 0, 1, 2
LIK_NORMAL, LIK_STUDENT_T, LIK_STUDENT_T_NU = 0, 1, 2

c_double_p = C.POINTER(C.c_double)


class PbxError(RuntimeError):
    pass


class DevInfo(C.Structure):
    _fields_ = [("device", C.c_int32), ("cc_major", C.c_int32), ("cc_minor", C.c_int32),
                ("sm_count", C.c_int32), ("l2_bytes_mb", C.c_int32),
                ("smem_per_block_optin", C.c_int32), ("global_mem_bytes", C.c_int64),
                ("name", C.c_char * 64)]


class MhMvnParams(C.Structure):
    _fields_ = [
        ("n_chains", C.c_int32), ("n_dims", C.c_int32), ("n_steps", C.c_int32),
        ("thin", C.c_int32), ("step0", C.c_int64), ("chain0", C.c_int64),
        ("seed", C.c_uint64), ("log_pscale", C.c_int32), ("accept_mode", C.c_int32),
        ("prop_kind", C.c_int32), ("has_prop_mat", C.c_int32),
        ("kernel_variant", C.c_int32), ("reserved0", C.c_int32),
        ("mean", C.c_double * PBX_MAX_DIMS),
        ("whiten", C.c_double * (PBX_MAX_DIMS * PBX_MAX_DIMS)),
        ("norm_c", C.c_double),
        ("prop_scale", C.c_double * PBX_MAX_DIMS),
        ("prop_mat", C.c_double * (PBX_MAX_DIMS * PBX_MAX_DIMS)),
        ("prop_radius", C.c_double),
        ("state", C.c_void_p), ("state_lp", C.c_void_p),
        ("inj_delta", C.c_void_p), ("inj_thresh", C.c_void_p),
        ("out_x", C.c_void_p), ("out_prob", C.c_void_p),
        ("out_accept", C.c_void_p), ("out_score", C.c_void_p),
        ("accept_count", C.c_void_p), ("stat_sum", C.c_void_p), ("stat_sumsq", C.c_void_p),
        ("out_xprop", C.c_void_p), ("out_pprop", C.c_void_p),
        ("prop_bound", C.c_int32), ("reserved1", C.c_int32),
        ("lims", (C.c_double * 2) * PBX_MAX_DIMS),
        ("open_end", (C.c_int32 * 2) * PBX_MAX_DIMS),
    ]


class RejectionParams(C.Structure):
    _fields_ = [
        ("n_params", C.c_int32), ("target_kind", C.c_int32), ("prop_kind", C.c_int32),
        ("score_mode", C.c_int32), ("n_samples", C.c_int64), ("sample0", C.c_int64),
        ("seed", C.c_uint64), ("lims", (C.c_double * 2) * 8), ("log_ufun", C.c_int32 * 8),
        ("target_centre", C.c_double * 8), ("target_radius", C.c_double),
        ("prop_loc", C.c_double * 8), ("prop_scale", C.c_double * 8),
        ("thresh_lo", C.c_double), ("thresh_hi", C.c_double),
        ("inj_unif", C.c_void_p), ("out_theta", C.c_void_p), ("out_p", C.c_void_p),
        ("out_q", C.c_void_p), ("out_s", C.c_void_p), ("out_t", C.c_void_p),
        ("out_u", C.c_void_p),
    ]


class MhNormregParams(C.Structure):
    _fields_ = [
        ("n_chains", C.c_int32), ("n_params", C.c_int32), ("n_steps", C.c_int32),
        ("thin", C.c_int32), ("step0", C.c_int64), ("chain0", C.c_int64),
        ("seed", C.c_uint64), ("has_slope", C.c_int32), ("accept_mode", C.c_int32),
        ("accept_coef", C.c_double), ("prop_kind", C.c_int32), ("variant", C.c_int32),
        ("n_obs", C.c_int64), ("x_obs", C.c_void_p), ("y_obs", C.c_void_p),
        ("lims", (C.c_double * 2) * PBX_MAX_PARAMS),
        ("open_end", (C.c_int32 * 2) * PBX_MAX_PARAMS),
        ("log_ufun", C.c_int32 * PBX_MAX_PARAMS), ("prop_bound", C.c_int32),
        ("prop_scale", C.c_double * PBX_MAX_PARAMS),
        ("prop_radius", C.c_double),
        ("state", C.c_void_p), ("state_lp", C.c_void_p),
        ("inj_delta", C.c_void_p), ("inj_thresh", C.c_void_p),
        ("out_x", C.c_void_p), ("out_prob", C.c_void_p),
        ("out_accept", C.c_void_p), ("out_score", C.c_void_p),
        ("accept_count", C.c_void_p), ("stat_sum", C.c_void_p), ("stat_sumsq", C.c_void_p),
        ("out_xprop", C.c_void_p), ("out_pprop", C.c_void_p),
        ("has_prop_mat", C.c_int32), ("reserved0", C.c_int32),
        ("prop_mat", C.c_double * (PBX_MAX_PARAMS * PBX_MAX_PARAMS)),
        ("lik_kind", C.c_int32), ("reserved1", C.c_int32),
        ("lik_df", C.c_double), ("lik_logc", C.c_double),
    ]


class GibbsMvnParams(C.Structure):
    _fields_ = [
        ("n_chains", C.c_int32), ("n_dims", C.c_int32), ("n_steps", C.c_int32),
        ("thin", C.c_int32), ("step0", C.c_int64), ("chain0", C.c_int64),
        ("seed", C.c_uint64), ("log_pscale", C.c_int32), ("want_prob", C.c_int32),
        ("mean", C.c_void_p), ("coef", C.c_void_p), ("stdv", C.c_void_p),
        ("cdf_lo", C.c_void_p), ("cdf_hi", C.c_void_p), ("whiten", C.c_void_p),
        ("dens_mean", C.c_void_p), ("norm_c", C.c_double),
        ("state", C.c_void_p), ("inj_runif", C.c_void_p),
        ("out_x", C.c_void_p), ("out_prob", C.c_void_p),
        ("stat_sum", C.c_void_p), ("stat_sumsq", C.c_void_p),
    ]


# name -> (restype, argtypes); every symbol include/pbx.h declares
SIGNATURES = {
    "pbx_version": (C.c_int, []),
    "pbx_last_error": (C.c_char_p, []),
    "pbx_device_count": (C.c_int, [C.POINTER(C.c_int)]),
    "pbx_device_info": (C.c_int, [C.c_int, C.POINTER(DevInfo)]),
    "pbx_ctx_create": (C.c_int, [C.c_int, C.c_void_p, C.c_int32, C.POINTER(C.c_void_p)]),
    "pbx_ctx_destroy": (C.c_int, [C.c_void_p]),
    "pbx_ctx_sync": (C.c_int, [C.c_void_p]),
    "pbx_ctx_launch_count": (C.c_int64, [C.c_void_p]),
    "pbx_ctx_last_kernel_ms": (C.c_int, [C.c_void_p, C.POINTER(C.c_float)]),
    "pbx_host_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "pbx_host_free": (C.c_int, [C.c_void_p]),
    "pbx_mh_mvn_run": (C.c_int, [C.c_void_p, C.POINTER(MhMvnParams)]),
    "pbx_mh_mvn_walk_host": (C.c_int, [C.c_void_p, C.POINTER(MhMvnParams), C.c_int32]),
    "pbx_mh_normreg_run": (C.c_int, [C.c_void_p, C.POINTER(MhNormregParams)]),
    "pbx_normreg_logjoint": (C.c_int, [C.c_void_p, C.POINTER(MhNormregParams),
                                       C.c_void_p, C.c_void_p]),
    "pbx_grid_norm_logjoint": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p,
                                         C.c_int32, C.c_void_p, C.c_int32, C.c_void_p,
                                         C.c_void_p, C.c_void_p]),
    "pbx_grid_t_logjoint": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p,
                                      C.c_int32, C.c_void_p, C.c_int32, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_double, C.c_double]),
    "pbx_grid_norm_logjoint_ss": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p,
                                            C.c_int32, C.c_void_p, C.c_int32, C.c_void_p,
                                            C.c_void_p, C.c_void_p]),
    "pbx_grid_max_sumexp": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]),
    "pbx_grid_rescale_sumexp": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "pbx_grid_posterior2": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32,
                                      C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_int32]),
    "pbx_rejection_sample": (C.c_int, [C.c_void_p, C.POINTER(RejectionParams)]),
    "pbx_log_prob_inplace": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
    "pbx_exp_logp_inplace": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64]),
    "pbx_gibbs_mvn_run": (C.c_int, [C.c_void_p, C.POINTER(GibbsMvnParams)]),
    "pbx_mvn_logpdf": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_void_p,
                                 C.c_void_p, C.c_double, C.c_int32, C.c_void_p]),
    "pbx_ndtri": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "pbx_ndtri_host": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p]),
    "pbx_reduce_chain_stats": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                         C.c_int64, C.c_int64, C.c_void_p]),
    "pbx_argsort_workspace_bytes": (C.c_int, [C.c_int64, C.POINTER(C.c_size_t)]),
    "pbx_argsort_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_size_t]),
    "pbx_gather_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    "pbx_take_axis_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int32,
                                    C.c_void_p, C.c_void_p]),
    "pbx_scan_workspace_bytes": (C.c_int, [C.c_int64, C.POINTER(C.c_size_t)]),
    "pbx_cumprob_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p,
                                  C.c_void_p, C.c_void_p, C.c_size_t]),
    "pbx_digitize_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64,
                                   C.POINTER(C.c_double), C.c_int32, C.c_void_p]),
    "pbx_expectation_f64": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_int32,
                                      C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p,
                                      C.c_void_p, C.c_size_t]),
    "pbx_pd_binary_f64": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_int64,
                                    C.c_int32, C.c_void_p, C.c_int64, C.c_int64, C.c_int32,
                                    C.c_int64, C.c_int64, C.c_int32, C.c_void_p]),
    "pbx_box_sample": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.POINTER(C.c_double),
                                 C.POINTER(C.c_int32), C.c_uint64, C.c_int64, C.c_void_p,
                                 C.c_void_p]),
    "pbx_selftest_fastmath": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64,
                                        C.c_void_p]),
    "pbx_fp64_peak": (C.c_int, [C.c_void_p, C.POINTER(C.c_double)]),
    "pbx_fp64_dep_latency": (C.c_int, [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double)]),
}

_lib = None


def load():
    """Loads libpbx.so (building nothing: run ``python -m probayes_b200.build`` or
    ``__graft_entry__.build()`` first).  Raises if the library is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise PbxError(
            "probayes_b200: CUDA library %s not built -- run `python -m probayes_b200.build`. "
            "There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is missing
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc, what=""):
    if rc != 0:
        msg = load().pbx_last_error().decode("utf-8", "replace")
        raise PbxError("%s failed (status %d): %s" % (what or "libpbx call", rc, msg))
