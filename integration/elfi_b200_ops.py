"""Reference-side binding of libelfi_b200.so: the module a maintainer of elfi-dev/elfi would add
(e.g. as ``elfi/b200_ops.py``) to run the hot path of an UNMODIFIED ELFI installation on a B200.

It uses nothing but ctypes + the C ABI of include/elfi_b200.h (torch only allocates the device
buffers and supplies the stream) and plugs into the reference through its own extension points:

    elfi.Distance(device_cdist_euclidean, *summaries)      # elfi/model/elfi_model.py:1016-1019
    elfi.Summary(partial(device_autocov, lag=1), sim)      # elfi/model/elfi_model.py:922-937
    elfi.BSL(m, n_sim, likelihood=partial(device_gaussian_syn_likelihood, ...))   # bsl.py:35-53

``tests/test_reference_plugin.py`` runs the reference's own Rejection sampler on a model built
this way and reproduces the reference's golden result bit for bit.
"""
import ctypes
import os

import numpy as np
import torch

_LIB_PATH = os.environ.get('ELFI_B200_LIB') or os.path.join(
    os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'elfi_b200', 'lib',
    'libelfi_b200.so')
_lib = ctypes.CDLL(_LIB_PATH)
_lib.elfi_b200_last_error.restype = ctypes.c_char_p
_ctx = ctypes.c_void_p()
_P, _I64 = ctypes.c_void_p, ctypes.c_int64


def _check(rc):
    if rc != 0:
        raise RuntimeError(_lib.elfi_b200_last_error().decode())


def _context():
    if not _ctx.value:
        _check(_lib.elfi_b200_ctx_create(ctypes.c_int(torch.cuda.current_device()),
                                         ctypes.byref(_ctx)))
    return _ctx


def _stream():
    return _P(torch.cuda.current_stream().cuda_stream)


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float64)).cuda()


def device_cdist_euclidean(XA, XB, w=None):
    """Drop-in for ``partial(scipy.spatial.distance.cdist, metric='euclidean')`` as used by
    elfi.Distance (elfi_model.py:1037): XA (B, D), XB (1, D) -> (B, 1), bit-identical."""
    X = _dev(np.atleast_2d(XA))
    obs = _dev(np.ravel(XB))
    W = None if w is None else _dev(np.ravel(w))
    B, D = X.shape
    d = torch.empty(B, dtype=torch.float64, device='cuda')
    _check(_lib.elfi_b200_dist_euclid_thr_f64(
        _context(), _P(X.data_ptr()), _I64(D), _I64(B), _I64(D), _P(obs.data_ptr()),
        _P(W.data_ptr() if W is not None else 0), _I64(1), None, _P(d.data_ptr()), None, None,
        _stream()))
    return d.cpu().numpy()[:, None]


def device_autocov(x, lag=1):
    """Drop-in for elfi.examples.ma2.autocov (ma2.py:40-59): x (B, n_obs) -> (B,),
    ``np.mean(x[:, lag:] * x[:, :-lag], axis=1)`` bit for bit (NumPy's pairwise order)."""
    X = _dev(np.atleast_2d(x))
    B, n = X.shape
    lags = (ctypes.c_int32 * 1)(int(lag))
    out = torch.empty((B, 1), dtype=torch.float64, device='cuda')
    _check(_lib.elfi_b200_summary_autocov_f64(
        _context(), _P(X.data_ptr()), _I64(n), _I64(B), _I64(n), lags, _I64(1),
        _P(out.data_ptr()), _I64(1), _stream()))
    return out.cpu().numpy()[:, 0]


def device_gaussian_syn_likelihood(ssx, ssy, shrinkage=None, penalty=None, whitening=None,
                                   standardise=False):
    """Drop-in for elfi.methods.bsl.pdf_methods.gaussian_syn_likelihood (pdf_methods.py:77-135)
    with shrinkage None or 'warton': ssx (n, d), ssy (d,) or (1, d) -> array([loglik]) from one
    call of elfi_b200_synlik_f64 (-inf for a singular covariance, like the reference)."""
    if shrinkage not in (None, 'warton'):
        raise NotImplementedError('only shrinkage=None or \'warton\' runs on the device')
    X = _dev(np.atleast_2d(ssx))
    n, d = X.shape
    obs = _dev(np.ravel(ssy))
    Wh = None if whitening is None else _dev(whitening)
    gam = None
    if shrinkage == 'warton':
        gam = (ctypes.c_double * 1)(1 - penalty)
    out = torch.empty(1, dtype=torch.float64, device='cuda')
    _check(_lib.elfi_b200_synlik_f64(
        _context(), ctypes.c_int32(0), _P(X.data_ptr()), _I64(d), _I64(1), _I64(n), _I64(n),
        _I64(d), _P(obs.data_ptr()), _P(Wh.data_ptr() if Wh is not None else 0), gam, _I64(1),
        _P(out.data_ptr()), _stream()))
    return out.cpu().numpy()
