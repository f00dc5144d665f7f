"""ctypes binding of libelfi_b200.so (the C ABI declared in include/elfi_b200.h).

There is no CPU fallback: if the shared library is missing or a call fails, an exception is
raised.  Build it with ``python -c "import __graft_entry__ as g; g.build()"`` (nvcc, sm_100a).
"""
import ctypes
import os

LIB_PATH = os.environ.get(
    'ELFI_B200_LIB',
    os.path.join(os.path.dirname(os.path.abspath(__file__)), 'lib', 'libelfi_b200.so'))

c_i64 = ctypes.c_int64
c_u64 = ctypes.c_uint64
c_int = ctypes.c_int
c_dbl = ctypes.c_double
c_ptr = ctypes.c_void_p

# name -> (argtypes); every function returns int (0 = ok) unless listed in _SPECIAL_RESTYPE
SIGNATURES = {
    'elfi_b200_version': [],
    'elfi_b200_last_error': [],
    'elfi_b200_ctx_create': [c_int, ctypes.POINTER(c_ptr)],
    'elfi_b200_ctx_destroy': [c_ptr],
    'elfi_b200_ctx_sm_count': [c_ptr],
    'elfi_b200_allgather_particles': [c_ptr, c_i64, c_ptr, c_i64, c_i64, c_ptr, c_ptr],
    'elfi_b200_dist_euclid_thr_f64': [c_ptr, c_ptr, c_i64, c_i64, c_i64, c_ptr, c_ptr, c_i64,
                                      c_ptr, c_ptr, c_ptr, c_ptr, c_ptr],
    'elfi_b200_dist_euclid_thr_dev_f64': [c_ptr, c_ptr, c_i64, c_i64, c_i64, c_ptr, c_ptr, c_i64,
                                          c_ptr, c_ptr, c_ptr, c_ptr, c_ptr],
    'elfi_b200_dist_euclid_mom_f64': [c_ptr, c_ptr, c_i64, c_i64, c_i64, c_ptr, c_ptr, c_i64,
                                      c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr],
    'elfi_b200_dist_euclid_thr_f64_host': [c_ptr, c_ptr, c_i64, c_i64, c_i64, c_ptr, c_ptr, c_i64,
                                           c_ptr, c_ptr, c_ptr, c_ptr],
    'elfi_b200_dist_metric_thr_f64': [c_ptr, ctypes.c_int32, c_dbl, c_ptr, c_i64, c_i64, c_i64, c_ptr,
                                      c_ptr, c_ptr, c_ptr, c_ptr, c_ptr],
    'elfi_b200_dist_seuclidean_thr_f64': [c_ptr, c_ptr, c_i64, c_i64, c_i64, c_ptr, c_ptr, c_ptr,
                                          c_ptr, c_ptr, c_ptr, c_ptr],
    'elfi_b200_topn_merge_f64': [c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_i64,
                                 c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_ptr],
    'elfi_b200_summary_autocov_f64': [c_ptr, c_ptr, c_i64, c_i64, c_i64, c_ptr, c_i64, c_ptr, c_i64,
                                      c_ptr],
    'elfi_b200_summary_meanvar_f64': [c_ptr, c_ptr, c_i64, c_i64, c_i64, c_ptr, c_i64,
                                      ctypes.c_int32, ctypes.c_int32, c_ptr],
    'elfi_b200_sort_pairs_f64': [c_ptr, c_ptr, c_i64, c_ptr, c_ptr, c_ptr],
    'elfi_b200_gather_rows_f64': [c_ptr, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_ptr],
    'elfi_b200_gather2_rows_f64': [c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_ptr, c_ptr, c_i64,
                                   c_i64, c_ptr, c_i64, c_ptr],
    'elfi_b200_accept_append_f64': [c_ptr, c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_i64,
                                    c_i64, c_ptr, c_ptr, c_ptr],
    'elfi_b200_rejection_batch_f64': [c_ptr, c_ptr, c_i64, c_i64, c_i64, c_ptr, c_ptr, c_i64, c_ptr, c_ptr,
                                      c_ptr, c_ptr, c_ptr, c_i64, c_ptr, c_ptr, c_ptr, c_ptr, c_i64,
                                      c_i64, c_ptr, c_ptr, c_ptr],
    'elfi_b200_wquantile_f64': [c_ptr, c_ptr, c_ptr, c_i64, c_dbl, c_ptr, c_ptr],
    'elfi_b200_colmoments_f64': [c_ptr, c_ptr, c_i64, c_i64, c_i64, c_ptr, c_ptr],
    'elfi_b200_weighted_stats_f64': [c_ptr, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_ptr, c_ptr],
    'elfi_b200_gm_logpdf_f64': [c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_ptr, c_i64, c_i64,
                                c_ptr, c_dbl, c_ptr, c_ptr],
    'elfi_b200_gm_logpdf_mixed_f64': [c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_ptr, c_i64, c_i64,
                                      c_ptr, c_dbl, c_ptr, c_ptr],
    'elfi_b200_smc_weights_f64': [c_ptr, c_ptr, c_ptr, c_i64, c_ptr, c_ptr],
    'elfi_b200_probe_fp64_f64': [c_ptr, c_ptr],
    'elfi_b200_rowsort_f64': [c_ptr, c_ptr, c_i64, c_i64, c_i64, c_ptr, c_i64, c_ptr],
    'elfi_b200_kliep_fit_f64': [c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_i64, c_i64, c_ptr, c_ptr,
                                c_dbl, c_i64, c_dbl, c_i64, c_dbl, c_i64, c_ptr, c_ptr],
    'elfi_b200_prior_ma2_f64': [c_ptr, c_i64, c_u64, c_u64, ctypes.c_int32, c_ptr, c_ptr, c_ptr],
    'elfi_b200_logprior_ma2_f64': [c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_ptr],
    'elfi_b200_sim_ma2_f64': [c_ptr, c_ptr, c_ptr, c_i64, c_i64, c_u64, c_u64, c_ptr, c_i64, c_ptr,
                              c_i64, c_ptr],
    'elfi_b200_gm_rvs_f64': [c_ptr, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_u64, c_u64,
                             ctypes.c_int32, c_ptr, c_ptr, c_i64, c_ptr],
    'elfi_b200_gm_cdf_f64': [c_ptr, c_ptr, c_i64, c_ptr, c_ptr],
    'elfi_b200_gm_rvs_cdf_f64': [c_ptr, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_u64, c_u64,
                                 ctypes.c_int32, c_ptr, c_ptr, c_i64, c_ptr],
    'elfi_b200_prior_gauss_f64': [c_ptr, c_i64, c_u64, c_u64, c_ptr, c_ptr, c_ptr, c_ptr],
    'elfi_b200_logprior_gauss_f64': [c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_ptr, c_ptr],
    'elfi_b200_sim_gauss_f64': [c_ptr, c_ptr, c_ptr, c_i64, c_i64, c_u64, c_u64, c_ptr, c_i64, c_ptr,
                                c_i64, c_ptr],
    'elfi_b200_sim_gnk_f64': [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_dbl, c_i64, c_i64, c_u64, c_u64,
                              c_ptr, c_i64, c_ptr],
    'elfi_b200_logprior_box_f64': [c_ptr, c_ptr, c_i64, c_i64, c_i64, c_ptr, c_ptr, c_ptr],
    'elfi_b200_gp_padded_size': [c_i64],
    'elfi_b200_gp_fit_f64': [c_ptr, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_dbl, c_dbl, c_dbl, c_dbl,
                             c_ptr, c_ptr, c_ptr, c_i64, c_ptr, c_ptr, c_ptr],
    'elfi_b200_gp_predict_f64': [c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_i64, c_i64, c_ptr,
                                 c_i64, c_ptr, c_dbl, c_dbl, c_dbl, c_dbl, c_dbl, c_ptr, c_ptr,
                                 c_ptr, c_ptr],
    'elfi_b200_gp_predict_grad_f64': [c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_i64, c_i64, c_ptr,
                                      c_ptr, c_i64, c_ptr, c_dbl, c_dbl, c_dbl, c_ptr, c_ptr, c_ptr,
                                      c_ptr, c_ptr],
    'elfi_b200_gp_whiten_f64': [c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_i64, c_i64, c_ptr, c_i64,
                                c_dbl, c_dbl, c_dbl, c_ptr, c_i64, c_ptr],
    'elfi_b200_gp_apply_wt_f64': [c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_ptr],
    'elfi_b200_gp_cross_cov_f64': [c_ptr, c_ptr, c_i64, c_i64, c_ptr, c_i64, c_ptr, c_i64, c_i64, c_ptr,
                                   c_i64, c_i64, c_i64, c_dbl, c_dbl, c_dbl, c_ptr, c_ptr],
    'elfi_b200_lcbsc_f64': [c_ptr, c_ptr, c_ptr, c_ptr, c_ptr, c_i64, c_i64, c_dbl, c_ptr, c_ptr,
                            c_ptr],
    'elfi_b200_synlik_f64': [c_ptr, ctypes.c_int32, c_ptr, c_i64, c_i64, c_i64, c_i64, c_i64, c_ptr,
                             c_ptr, c_ptr, c_i64, c_ptr, c_ptr],
}
_SPECIAL_RESTYPE = {'elfi_b200_last_error': ctypes.c_char_p, 'elfi_b200_gp_padded_size': c_i64}
_NO_STATUS = {'elfi_b200_version', 'elfi_b200_last_error', 'elfi_b200_ctx_sm_count',
              'elfi_b200_gp_padded_size'}


class ElfiB200Error(RuntimeError):
    """A call into libelfi_b200.so failed."""


_lib = None


def load():
    """Load the shared library (once) and declare all signatures."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ElfiB200Error(
            "libelfi_b200.so not found at {}. The CUDA extension must be built "
            "(__graft_entry__.build()); elfi_b200 has no CPU fallback.".format(LIB_PATH))
    lib = ctypes.CDLL(LIB_PATH)
    for name, argtypes in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the header and the library disagree
        fn.argtypes = argtypes
        fn.restype = _SPECIAL_RESTYPE.get(name, c_int)
    _lib = lib
    return lib


def last_error():
    msg = load().elfi_b200_last_error()
    return msg.decode('utf-8', 'replace') if msg else ''


def call(name, *args):
    """Call a status-returning entry point; raise ElfiB200Error on a non-zero code."""
    lib = load()
    rc = getattr(lib, name)(*args)
    if name in _NO_STATUS:
        return rc
    if rc != 0:
        raise ElfiB200Error('{} failed ({}): {}'.format(name, rc, last_error()))
    return rc
