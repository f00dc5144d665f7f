"""Array-level operators of the hot path: thin Python wrappers over the C ABI.

Each wrapper accepts CUDA tensors (or host arrays, which are uploaded) and returns CUDA
tensors.  Reference call sites are cited per function (paths relative to the reference repo).
"""
import ctypes

import numpy as np
import torch

from . import _lib
from . import device as dev

MAX_NESTED = 32


def _matrix(S):
    if dev.is_device_array(S) and S.dtype == torch.float64 and S.dim() == 2 \
            and S.stride(1) == 1 and S.stride(0) >= S.shape[1]:
        return S  # row-strided views are consumed in place (leading dimension = stride(0))
    S = dev.to_device(S)
    if S.dim() == 1:
        S = S[:, None]
    if S.dim() != 2:
        raise ValueError('expected a 2-d (batch, dim) array, got shape {}'.format(tuple(S.shape)))
    if S.stride(1) != 1:
        S = S.contiguous()
    return S


def dist_euclid(S, obs, w=None, thresholds=None, want_indices=True, sync=True, moments=False):
    """Euclidean / nested weighted distances of the rows of S to ``obs`` + acceptance.

    Replaces ``cdist(S, obs, 'euclidean'[, w=w])`` reached through
    elfi/model/utils.py:37-52 and elfi/model/elfi_model.py:1037, 1135-1151, and the mask of
    elfi/methods/inference/samplers.py:223-225.

    Parameters
    ----------
    S : (B, D) array
    obs : (D,) or (1, D) array
    w : None, (D,) or (K, D) -- cdist's ``w`` per nested column (a row of ones == unweighted)
    thresholds : None, float, (K,) host values, or a (K,) DEVICE array (no host round trip)
        -- accept rows with all_k(d[:, k] <= thresholds[k])
    sync : False leaves the accepted count on the device: acc_idx is then the pair
        (int32 buffer of B indices of which the first n_acc are valid, n_acc device int64[1])
    moments : True also returns the (2, D) device array [column means; column M2] of S, computed
        from the same read of S (AdaptiveDistance.add_data, elfi_model.py:1104-1125)

    Returns
    -------
    d : (B,) tensor if K == 1 and w was not 2-d, else (B, K)
    acc_idx : int32 tensor of accepted row indices, ascending (None without thresholds)
    """
    S = _matrix(S)
    B, D = S.shape
    obs_t = dev.to_device(obs).reshape(-1)
    if obs_t.numel() != D:
        raise ValueError('XA and XB must have the same number of columns '
                         '(i.e. feature dimension.)')
    squeeze = True
    W = None
    K = 1
    if w is not None:
        W = dev.to_device(w)
        if W.dim() == 1:
            W = W[None, :]
        else:
            squeeze = False
        K = W.shape[0]
        if W.shape[1] != D:
            raise ValueError('weights must have {} columns'.format(D))
        if K > MAX_NESTED:
            raise ValueError('at most {} nested distances are supported'.format(MAX_NESTED))
    thr = None
    thr_on_device = dev.is_device_array(thresholds)
    if thr_on_device:
        thr = thresholds.reshape(-1)
        if thr.dtype != torch.float64 or not thr.is_contiguous():
            thr = thr.to(torch.float64).contiguous()
    elif thresholds is not None:
        thr = np.ascontiguousarray(np.atleast_1d(thresholds), dtype=np.float64)
    if thr is not None and thr.shape[0] != K:
        raise ValueError('need one threshold per distance column ({} != {})'.format(
            thr.shape[0], K))
    d = dev.empty((B, K))
    acc_idx = n_acc = None
    if thr is not None:
        n_acc = dev.zeros((1,), dtype=torch.int64)
        if want_indices:
            acc_idx = dev.empty((max(B, 1),), dtype=torch.int32)
    mom = None
    if moments:
        mom = dev.empty((2, D))
        _lib.call('elfi_b200_dist_euclid_mom_f64', dev.context(), dev.ptr(S),
                  S.stride(0) if B > 1 else D, B, D, dev.ptr(obs_t), dev.ptr(W), K,
                  None if thr_on_device else dev.ptr(thr), dev.ptr(thr) if thr_on_device else None,
                  dev.ptr(d), dev.ptr(acc_idx), dev.ptr(n_acc), dev.ptr(mom), dev.stream_ptr())
    else:
        _lib.call('elfi_b200_dist_euclid_thr_dev_f64' if thr_on_device else
                  'elfi_b200_dist_euclid_thr_f64', dev.context(), dev.ptr(S),
                  S.stride(0) if B > 1 else D, B, D, dev.ptr(obs_t), dev.ptr(W), K, dev.ptr(thr),
                  dev.ptr(d), dev.ptr(acc_idx), dev.ptr(n_acc), dev.stream_ptr())
    if thr is not None:
        if not sync:
            acc_idx = (acc_idx, n_acc)
        else:
            n = int(n_acc.item())
            acc_idx = acc_idx[:n] if want_indices else n
    if squeeze:
        d = d.reshape(B)
    return (d, acc_idx, mom) if moments else (d, acc_idx)


METRIC_CODES = {'sqeuclidean': 1, 'cityblock': 2, 'chebyshev': 3, 'minkowski': 4}


def dist_metric(S, obs, metric, p=2.0, threshold=None, want_indices=True):
    """cdist(S, obs, metric) for 'sqeuclidean', 'cityblock', 'chebyshev' and 'minkowski' (p)
    + acceptance, on the device (elfi/model/elfi_model.py:1016-1037 passes these metric strings to
    SciPy).  Minkowski with p = 1, 2, inf is routed to cityblock / euclidean / chebyshev as SciPy
    does.  Returns (d (B,), acc_idx or None)."""
    if metric == 'minkowski':
        if p == 1:
            metric = 'cityblock'
        elif p == 2:
            return dist_euclid(S, obs, thresholds=threshold, want_indices=want_indices)
        elif np.isinf(p):
            metric = 'chebyshev'
        elif not p > 0:
            raise ValueError('p must be greater than 0')
    if metric not in METRIC_CODES:
        raise ValueError('Unknown Distance Metric: {}'.format(metric))
    S = _matrix(S)
    B, D = S.shape
    obs_t = dev.to_device(obs).reshape(-1)
    if obs_t.numel() != D:
        raise ValueError('XA and XB must have the same number of columns '
                         '(i.e. feature dimension.)')
    thr = None
    if threshold is not None:
        thr = np.ascontiguousarray(np.atleast_1d(threshold), dtype=np.float64)
        if thr.shape[0] != 1:
            raise ValueError('need one threshold per distance column ({} != 1)'.format(thr.shape[0]))
    d = dev.empty((B,))
    acc_idx = n_acc = None
    if thr is not None:
        n_acc = dev.zeros((1,), dtype=torch.int64)
        if want_indices:
            acc_idx = dev.empty((max(B, 1),), dtype=torch.int32)
    _lib.call('elfi_b200_dist_metric_thr_f64', dev.context(), METRIC_CODES[metric], float(p),
              dev.ptr(S), S.stride(0) if B > 1 else D, B, D, dev.ptr(obs_t), dev.ptr(thr),
              dev.ptr(d), dev.ptr(acc_idx), dev.ptr(n_acc), dev.stream_ptr())
    if thr is not None:
        n = int(n_acc.item())
        acc_idx = acc_idx[:n] if want_indices else n
    return d, acc_idx


def dist_seuclidean(S, obs, V, threshold=None, want_indices=True):
    """cdist(S, obs, 'seuclidean', V=V) + acceptance on the device, bit-identical to SciPy (two
    running sums and an IEEE division per term; elfi/model/elfi_model.py:1016-1037 forwards the
    metric string and V to cdist).  Returns (d (B,), acc_idx or None)."""
    S = _matrix(S)
    B, D = S.shape
    obs_t = dev.to_device(obs).reshape(-1)
    if obs_t.numel() != D:
        raise ValueError('XA and XB must have the same number of columns '
                         '(i.e. feature dimension.)')
    V_t = dev.to_device(V)
    if V_t.dim() != 1 or V_t.shape[0] != D:
        raise ValueError('Variance vector V must be of the same dimension as the vectors on '
                         'which the distances are computed.')
    thr = None
    if threshold is not None:
        thr = np.ascontiguousarray(np.atleast_1d(threshold), dtype=np.float64)
        if thr.shape[0] != 1:
            raise ValueError('need one threshold per distance column ({} != 1)'.format(thr.shape[0]))
    d = dev.empty((B,))
    acc_idx = n_acc = None
    if thr is not None:
        n_acc = dev.zeros((1,), dtype=torch.int64)
        if want_indices:
            acc_idx = dev.empty((max(B, 1),), dtype=torch.int32)
    _lib.call('elfi_b200_dist_seuclidean_thr_f64', dev.context(), dev.ptr(S),
              S.stride(0) if B > 1 else D, B, D, dev.ptr(obs_t), dev.ptr(V_t), dev.ptr(thr),
              dev.ptr(d), dev.ptr(acc_idx), dev.ptr(n_acc), dev.stream_ptr())
    if thr is not None:
        n = int(n_acc.item())
        acc_idx = acc_idx[:n] if want_indices else n
    return d, acc_idx


def dist_euclid_host(S, obs, w=None, thresholds=None, return_distances=True):
    """Host-buffer variant (elfi_b200_dist_euclid_thr_f64_host): numpy in, numpy out."""
    S = np.asarray(S, dtype=np.float64)
    if S.ndim == 1:
        S = S[:, None]
    if S.strides[1] != 8:
        S = np.ascontiguousarray(S)
    B, D = S.shape
    ld = S.strides[0] // 8 if B > 1 else D
    obs = np.ascontiguousarray(obs, dtype=np.float64).reshape(-1)
    K = 1
    W = None
    if w is not None:
        W = np.ascontiguousarray(np.atleast_2d(w), dtype=np.float64)
        K = W.shape[0]
    thr = None if thresholds is None else np.ascontiguousarray(np.atleast_1d(thresholds),
                                                               dtype=np.float64)
    d = np.empty((B, K)) if return_distances else None
    idx = np.empty(max(B, 1), dtype=np.int32) if thr is not None else None
    n = ctypes.c_int64(0)
    _lib.call('elfi_b200_dist_euclid_thr_f64_host', dev.context(), dev.ptr(S), ld, B, D,
              dev.ptr(obs), dev.ptr(W), K, dev.ptr(thr), dev.ptr(d), dev.ptr(idx),
              ctypes.byref(n) if thr is not None else None)
    if d is not None and K == 1 and (w is None or np.ndim(w) == 1):
        d = d.reshape(B)
    return d, (idx[:n.value] if idx is not None else None)


def _ld(t):
    return t.stride(0) if t.shape[0] > 1 else t.shape[1]


def autocov(x, lags=(1,), out=None):
    """MA2 autocovariance summaries (elfi/examples/ma2.py:40-59) for one or more lags.

    Returns a (B, len(lags)) tensor: column l is ``np.mean(x[:, lag:] * x[:, :-lag], axis=1)``
    bit for bit.  This is already the column-stacked summary matrix of
    elfi/model/utils.py:39, so it can be handed to :func:`dist_euclid` directly."""
    x = _matrix(x)
    B, n = x.shape
    lags_arr = np.ascontiguousarray(np.atleast_1d(lags), dtype=np.int32)
    for lag in lags_arr:
        if not 1 <= lag < n:
            raise ValueError('lag {} outside [1, {})'.format(lag, n))
    if out is None:
        out = dev.empty((B, len(lags_arr)))
    _lib.call('elfi_b200_summary_autocov_f64', dev.context(), dev.ptr(x), _ld(x), B, n,
              dev.ptr(lags_arr), len(lags_arr), dev.ptr(out), out.stride(0) if B > 1 else
              out.shape[1], dev.stream_ptr())
    return out


def meanvar(y, out=None):
    """Gaussian-model summaries ss_mean / ss_var (elfi/examples/gauss.py:142-173).

    Returns a (B, 2) tensor [np.mean(y, axis=1), np.var(y, axis=1)], bit for bit."""
    y = _matrix(y)
    B, n = y.shape
    if out is None:
        out = dev.empty((B, 2))
    _lib.call('elfi_b200_summary_meanvar_f64', dev.context(), dev.ptr(y), _ld(y), B, n,
              dev.ptr(out), out.stride(0) if B > 1 else out.shape[1], 0, 1, dev.stream_ptr())
    return out


def argsort(keys, return_keys=False):
    """Stable ascending argsort of a 1-d fp64 array (NaN last) -> int32 permutation.

    np.argsort of elfi/methods/inference/samplers.py:235 and elfi/methods/utils.py:397."""
    keys = dev.to_device(keys).reshape(-1)
    n = keys.numel()
    perm = dev.empty((n,), dtype=torch.int32)
    ks = dev.empty((n,)) if return_keys else None
    _lib.call('elfi_b200_sort_pairs_f64', dev.context(), dev.ptr(keys), n, dev.ptr(ks),
              dev.ptr(perm), dev.stream_ptr())
    return (perm, ks) if return_keys else perm


def _as_2d(t):
    if t.dim() == 2:
        return t
    width = 1
    for extent in t.shape[1:]:
        width *= int(extent)
    return t.reshape(t.shape[0], width)


def take_rows(src, idx):
    """src[idx] for an fp64 array with the batch on axis 0 (samplers.py:230, 237)."""
    src = dev.to_device(src)
    shape = src.shape
    s2 = _as_2d(src)
    if s2.stride(-1) != 1 and s2.shape[1] > 0:
        s2 = s2.contiguous()
    idx = dev.to_device(idx, dtype=torch.int32)
    n = idx.numel()
    width = s2.shape[1]
    dst = dev.empty((n, width))
    if n and width:
        _lib.call('elfi_b200_gather_rows_f64', dev.context(), dev.ptr(s2), _ld(s2), dev.ptr(idx),
                  n, width, dev.ptr(dst), width, dev.stream_ptr())
    return dst.reshape((n,) + tuple(shape[1:]))


def take_rows2(a, b, perm, n_out, map_b=None):
    """Rows perm[:n_out] of the virtual concatenation [a; b[map_b]] (top-n merge gather)."""
    shape = a.shape if a is not None else b.shape
    a2 = _as_2d(a) if a is not None else None
    b2 = _as_2d(b) if b is not None else None
    width = (a2 if a2 is not None else b2).shape[1]
    n_a = a2.shape[0] if a2 is not None else 0
    dst = dev.empty((n_out, width))
    if n_out and width:
        _lib.call('elfi_b200_gather2_rows_f64', dev.context(), dev.ptr(a2),
                  _ld(a2) if a2 is not None else width, n_a, dev.ptr(b2),
                  _ld(b2) if b2 is not None else width, dev.ptr(map_b), dev.ptr(perm), n_out,
                  width, dev.ptr(dst), width, dev.stream_ptr())
    return dst.reshape((n_out,) + tuple(shape[1:]))


def merge_topn(state, batch, key_state, key_batch, map_b, n_keep):
    """Rejection._merge_batch (samplers.py:226-237) as one library call: the virtual concatenation
    [state[k]; batch[k][map_b]] is ranked by [key_state; key_batch[map_b]] (1-d views, possibly a
    strided column of a (rows, K) distance matrix) and the n_keep smallest rows of every output k
    come back as new device arrays.  map_b None: every batch row is a candidate."""
    if map_b is not None and map_b.dtype != torch.int32:
        raise TypeError('map_b must be an int32 device array of batch row indices')
    n_a = int(key_state.shape[0])
    n_b = int(map_b.numel()) if map_b is not None else int(key_batch.shape[0])
    a2 = [_as_2d(t) for t in state]
    b2 = [_as_2d(dev.to_device(t)) for t in batch]
    widths = [t.shape[1] for t in b2]
    outs = [dev.empty((n_keep, w)) for w in widths]
    n = len(outs)
    if n_keep and n:
        arr_p, arr_i = ctypes.c_void_p * n, ctypes.c_int64 * n
        pa = arr_p(*[t.data_ptr() if n_a else 0 for t in a2])
        la = arr_i(*[_ld(t) if n_a else w for t, w in zip(a2, widths)])
        pb = arr_p(*[t.data_ptr() for t in b2])
        lb = arr_i(*[_ld(t) for t in b2])
        wd = arr_i(*widths)
        pd = arr_p(*[t.data_ptr() for t in outs])
        ld = arr_i(*widths)
        cast = lambda a: ctypes.cast(a, ctypes.c_void_p)   # noqa: E731
        _lib.call('elfi_b200_topn_merge_f64', dev.context(), dev.ptr(key_state) if n_a else None,
                  key_state.stride(0) if n_a > 1 else 1, n_a, dev.ptr(key_batch),
                  key_batch.stride(0) if key_batch.shape[0] > 1 else 1, dev.ptr(map_b), n_b,
                  n_keep, n, cast(pa), cast(la), cast(pb), cast(lb), cast(wd), cast(pd), cast(ld),
                  dev.stream_ptr())
    return [o.reshape((n_keep,) + tuple(t.shape[1:])) for o, t in zip(outs, batch)]


class CandidateBuffer:
    """Packed (capacity, width) device buffer of accepted rows + device-side row count: the tail
    of the reference's sample buffers (samplers.py:196-230) filled without host round trips."""

    def __init__(self, capacity, widths):
        self.widths = [int(w) for w in widths]
        self.width = sum(self.widths)
        self.capacity = int(capacity)
        self.rows = dev.empty((self.capacity, self.width))
        self._counters = dev.zeros((2,), dtype=torch.int64)      # [count, dropped]: one D2H reads both
        self.count = self._counters[0:1]
        self.dropped = self._counters[1:2]

    def reset(self):
        self._counters.zero_()

    def _descriptors(self, sources):
        """ctypes descriptor arrays of a source list, cached while the same buffers come back
        (a sampler appends from the same output tensors batch after batch)."""
        key = tuple((t.data_ptr(), tuple(t.shape), t.stride(0)) for t in sources)
        cached = getattr(self, '_desc', None)
        if cached is not None and cached[0] == key:
            return cached[1]
        srcs = [_as_2d(t) for t in sources]
        if [t.shape[1] for t in srcs] != self.widths:
            raise ValueError('source widths do not match the buffer layout')
        n = len(srcs)
        ptrs = (ctypes.c_void_p * n)(*[t.data_ptr() for t in srcs])
        lds = (ctypes.c_int64 * n)(*[_ld(t) for t in srcs])
        wid = (ctypes.c_int64 * n)(*self.widths)
        desc = (n, ptrs, lds, wid, ctypes.cast(ptrs, ctypes.c_void_p),
                ctypes.cast(lds, ctypes.c_void_p), ctypes.cast(wid, ctypes.c_void_p),
                dev.ptr(self.rows), dev.ptr(self.count), dev.ptr(self.dropped))
        self._desc = (key, desc)
        return desc

    def append(self, sources, acc_idx, n_acc, max_rows):
        """Append rows acc_idx[:n_acc] (device int32 / device int64 count) of `sources`."""
        n, _, _, _, pp, pl, pw, prow, pcount, pdrop = self._descriptors(sources)
        _lib.call('elfi_b200_accept_append_f64', dev.context(), dev.ptr(acc_idx), dev.ptr(n_acc),
                  int(max_rows), n, pp, pl, pw, prow, self.width, self.capacity, pcount, pdrop,
                  dev.stream_ptr())

    def bind_batch(self, S, obs, thresholds, d_out, acc_idx, n_acc, extras, w=None):
        """A zero-argument callable running ONE threshold-mode batch -- distances of S + acceptance
        + append of the accepted rows [d | extras] to this buffer -- as a single library call
        (elfi_b200_rejection_batch_f64) with every argument marshalled once: ~10 us of host time
        per batch, so that a busy host cannot starve a 0.17 ms kernel.  All tensors are device
        tensors the caller keeps alive; `thresholds` is a host sequence or a device tensor."""
        S = _matrix(S)
        B, D = S.shape
        W = None if w is None else dev.to_device(w).reshape(-1, D)
        K = 1 if W is None else W.shape[0]
        extras = [_as_2d(t) for t in extras]
        if [K] + [t.shape[1] for t in extras] != self.widths:
            raise ValueError('d / extra widths do not match the buffer layout')
        thr_dev = thresholds if dev.is_device_array(thresholds) else None
        thr_host = None if thr_dev is not None else np.ascontiguousarray(
            np.atleast_1d(thresholds), dtype=np.float64)
        n = len(extras)
        ptrs = (ctypes.c_void_p * max(n, 1))(*[t.data_ptr() for t in extras])
        lds = (ctypes.c_int64 * max(n, 1))(*[_ld(t) for t in extras])
        wid = (ctypes.c_int64 * max(n, 1))(*[t.shape[1] for t in extras])
        keep = (S, obs, W, thr_dev, thr_host, d_out, acc_idx, n_acc, extras, ptrs, lds, wid)
        args = (dev.context(), dev.ptr(S), S.stride(0) if B > 1 else D, B, D, dev.ptr(obs),
                dev.ptr(W), K, dev.ptr(thr_host), dev.ptr(thr_dev), dev.ptr(d_out),
                dev.ptr(acc_idx), dev.ptr(n_acc), n, ctypes.cast(ptrs, ctypes.c_void_p),
                ctypes.cast(lds, ctypes.c_void_p), ctypes.cast(wid, ctypes.c_void_p),
                dev.ptr(self.rows), self.width, self.capacity, dev.ptr(self.count),
                dev.ptr(self.dropped))

        def run(_keep=keep):
            _lib.call('elfi_b200_rejection_batch_f64', *args, dev.stream_ptr())
        return run

    def best(self, n, key_col=0):
        """(rows sorted by column key_col, first n; count, dropped) -- one D2H of the counters."""
        count, dropped = (int(v) for v in self._counters.cpu().tolist())
        keys = self.rows[:count, key_col].contiguous()
        perm = argsort(keys)
        return take_rows(self.rows, perm[:min(n, count)]), count, dropped


def allgather_particles(blocks):
    """Single-process multi-GPU all-gather (elfi_b200_allgather_particles): `blocks` = one
    (rows, width) fp64 CUDA tensor per GPU (equal shapes, each on its own device); returns one
    (len(blocks) * rows, width) tensor per GPU holding the blocks in list order.  The copies are
    enqueued on each device's current stream."""
    n = len(blocks)
    blocks = [b.contiguous() for b in blocks]
    rows = blocks[0].shape[0]
    width = int(np.prod(blocks[0].shape[1:])) if blocks[0].dim() > 1 else 1
    if any(tuple(b.shape) != tuple(blocks[0].shape) or b.dtype != torch.float64 for b in blocks):
        raise ValueError('blocks must be fp64 tensors of equal shape')
    outs, streams, ctxs = [], [], []
    for b in blocks:
        with torch.cuda.device(b.device):
            outs.append(torch.empty((n * rows,) + tuple(b.shape[1:]), dtype=torch.float64,
                                    device=b.device))
            streams.append(torch.cuda.current_stream(b.device).cuda_stream)
            ctxs.append(dev.context(b.device).value)
    arr = ctypes.c_void_p * n
    _lib.call('elfi_b200_allgather_particles', ctypes.cast(arr(*ctxs), ctypes.c_void_p), n,
              ctypes.cast(arr(*[b.data_ptr() for b in blocks]), ctypes.c_void_p), rows, width,
              ctypes.cast(arr(*[o.data_ptr() for o in outs]), ctypes.c_void_p),
              ctypes.cast(arr(*streams), ctypes.c_void_p))
    return outs


def weighted_sample_quantile(x, alpha, weights=None):
    """elfi/methods/utils.py:379-411 on the device; returns a Python float."""
    x = dev.to_device(x).reshape(-1)
    w = None if weights is None else dev.to_device(weights).reshape(-1)
    if w is not None and w.numel() != x.numel():
        raise ValueError('x and weights must have the same length')
    out = dev.empty((2,))
    _lib.call('elfi_b200_wquantile_f64', dev.context(), dev.ptr(x), dev.ptr(w), x.numel(),
              float(alpha), dev.ptr(out), dev.stream_ptr())
    return float(out[0].item())


def colmoments(S):
    """(mean, M2) per column of one batch (AdaptiveDistance.add_data's per-batch ingredients,
    elfi/model/elfi_model.py:1104-1125).  Returns two host arrays of length D."""
    S = _matrix(S)
    B, D = S.shape
    out = dev.empty((2, D))
    _lib.call('elfi_b200_colmoments_f64', dev.context(), dev.ptr(S), _ld(S), B, D, dev.ptr(out),
              dev.stream_ptr())
    out = out.cpu().numpy()
    return out[0], out[1]


def weighted_stats(x, weights=None):
    """V1, V2, weighted mean and unbiased weighted variance (elfi/methods/utils.py:108-139).

    Returns (V1, V2, xbar (p,), s2 (p,)) as host values."""
    x = _matrix(x)
    N, p = x.shape
    w = None if weights is None else dev.to_device(weights).reshape(-1)
    stats = dev.empty((2 + 2 * p,))
    _lib.call('elfi_b200_weighted_stats_f64', dev.context(), dev.ptr(x), _ld(x), dev.ptr(w), N, p,
              dev.ptr(stats), dev.stream_ptr())
    s = stats.cpu().numpy()
    return s[0], s[1], s[2:2 + p].copy(), s[2 + p:2 + 2 * p].copy()


def weighted_var(x, weights=None):
    """elfi/methods/utils.py:108-139."""
    return weighted_stats(x, weights)[3]


def gm_logpdf(x, means, cov=1, weights=None, validate=True, mixed=False):
    """GMDistribution.logpdf (elfi/methods/utils.py:174-197) on the device.

    x (N, p) and means (M, p) may be host or device arrays; returns a device tensor (N,).
    ``validate=False`` skips the two synchronising weight checks of normalize_weights
    (utils.py:80-88) for weights the caller produced itself.  ``mixed=True`` takes 2^f from the
    fp32 special-function unit (term error <= 2e-7 instead of 2e-9, 1.3x faster): the throughput
    mode's choice, where parity with the reference is statistical."""
    means = _matrix(means)
    M, p = means.shape
    x = dev.to_device(x)
    x = x.reshape(-1, p) if x.dim() != 2 else x
    x = _matrix(x)
    N = x.shape[0]
    cov = np.atleast_2d(np.asarray(cov, dtype=np.float64))
    if cov.shape == (1, 1) and p > 1:
        cov = np.eye(p) * cov[0, 0]
    L = np.linalg.cholesky(cov)
    Linv = np.ascontiguousarray(np.linalg.inv(L))
    logdet = 2.0 * float(np.sum(np.log(np.diag(L))))
    w = None if weights is None else dev.to_device(weights).reshape(-1)
    if w is not None and validate:
        if bool((w < 0).any()):
            raise ValueError("Weights must be positive")
        if float(w.sum()) == 0:
            raise ValueError("All weights are zero")
    logq = dev.empty((N,))
    _lib.call('elfi_b200_gm_logpdf_mixed_f64' if mixed else 'elfi_b200_gm_logpdf_f64',
              dev.context(), dev.ptr(x), _ld(x), N, dev.ptr(means),
              _ld(means), dev.ptr(w), M, p, dev.ptr(Linv), logdet, dev.ptr(logq), dev.stream_ptr())
    return logq


def smc_weights(logprior, logq):
    """w = exp(logprior - logq) (elfi/methods/inference/samplers.py:514)."""
    lp = dev.to_device(logprior).reshape(-1)
    lq = dev.to_device(logq).reshape(-1)
    w = dev.empty((lp.numel(),))
    _lib.call('elfi_b200_smc_weights_f64', dev.context(), dev.ptr(lp), dev.ptr(lq), lp.numel(),
              dev.ptr(w), dev.stream_ptr())
    return w


# ------------------------------------------------------------------ throughput mode (device RNG)
def prior_ma2(batch_size, seed, offset=0, t1=None, which='both'):
    """MA2 prior draws on the device (elfi/examples/ma2.py:96-186).

    which='both' -> (t1, t2); 't1' -> t1; 't2' -> t2 conditional on the given t1."""
    mode = {'both': 0, 't1': 1, 't2': 2}[which]
    if mode == 2:
        t1 = dev.to_device(t1).reshape(-1).contiguous()
        batch_size = t1.numel()
    else:
        t1 = dev.empty((batch_size,))
    t2 = dev.empty((batch_size,)) if mode != 1 else None
    _lib.call('elfi_b200_prior_ma2_f64', dev.context(), batch_size, int(seed), int(offset), mode,
              dev.ptr(t1), dev.ptr(t2), dev.stream_ptr())
    return (t1, t2) if mode == 0 else (t1 if mode == 1 else t2)


def logprior_ma2(params):
    """Joint log prior density of MA2's (t1, t2); -inf outside the support."""
    x = _matrix(params)
    out = dev.empty((x.shape[0],))
    _lib.call('elfi_b200_logprior_ma2_f64', dev.context(), dev.ptr(x), _ld(x), x.shape[0],
              dev.ptr(out), dev.stream_ptr())
    return out


def sim_ma2(t1, t2, n_obs=100, seed=0, offset=0, want_data=False, want_summaries=True):
    """MA2 simulator on the device; returns (X or None, S or None) with S = autocov lags (1, 2)
    computed in the same kernel (X never touches HBM unless asked for)."""
    t1 = dev.to_device(t1).reshape(-1)
    t2 = dev.to_device(t2).reshape(-1)
    B = t1.numel()
    X = dev.empty((B, n_obs)) if want_data else None
    S = dev.empty((B, 2)) if want_summaries else None
    _lib.call('elfi_b200_sim_ma2_f64', dev.context(), dev.ptr(t1), dev.ptr(t2), B, n_obs,
              int(seed), int(offset), dev.ptr(X), n_obs, dev.ptr(S), 2, dev.stream_ptr())
    return X, S


def gm_cdf(weights, n=None):
    """Inclusive running sum of the mixture weights (None -> n equal weights): the lookup table of
    the component draw in GMDistribution.rvs (elfi/methods/utils.py:239), built once per population
    and handed to every :func:`gm_rvs` call of that population."""
    w = None if weights is None else dev.to_device(weights).reshape(-1)
    n = int(w.numel()) if w is not None else int(n)
    cumw = dev.empty((n,))
    _lib.call('elfi_b200_gm_cdf_f64', dev.context(), dev.ptr(w), n, dev.ptr(cumw), dev.stream_ptr())
    return cumw


def gm_rvs(means, cov, weights, size, seed, offset=0, support=0, box=None, cdf=None):
    """GMDistribution.rvs on the device (elfi/methods/utils.py:200-261); support=1 keeps only
    draws inside the MA2 prior support, support=2 inside ``box`` = (lo (p,), hi (p,)) (redrawn per
    particle).  ``cdf`` = :func:`gm_cdf` of the weights (then ``weights`` is not read)."""
    means = _matrix(means)
    N, p = means.shape
    cov = np.atleast_2d(np.asarray(cov, dtype=np.float64))
    if cov.shape == (1, 1) and p > 1:
        cov = np.eye(p) * cov[0, 0]
    L = np.ascontiguousarray(np.linalg.cholesky(cov))
    boxarr = None
    if support == 2:
        boxarr = np.ascontiguousarray(np.concatenate([np.asarray(box[0], dtype=np.float64),
                                                      np.asarray(box[1], dtype=np.float64)]))
    out = dev.empty((size, p))
    if cdf is None:
        cdf = gm_cdf(weights, N)
    elif cdf.numel() != N:
        raise ValueError('cdf must have one entry per mixture component')
    _lib.call('elfi_b200_gm_rvs_cdf_f64', dev.context(), dev.ptr(means), _ld(means), dev.ptr(cdf), N,
              p, dev.ptr(L), size, int(seed), int(offset), int(support), dev.ptr(boxarr),
              dev.ptr(out), p, dev.stream_ptr())
    return out


def _gauss_prm(prm):
    return np.ascontiguousarray(prm, dtype=np.float64)


def prior_gauss(batch_size, seed, prm, offset=0):
    """Gaussian-model prior draws (elfi/examples/gauss.py:118-126): prm = [mu_lo, mu_width, a, b]."""
    mu, sigma = dev.empty((batch_size,)), dev.empty((batch_size,))
    _lib.call('elfi_b200_prior_gauss_f64', dev.context(), batch_size, int(seed), int(offset),
              dev.ptr(_gauss_prm(prm)), dev.ptr(mu), dev.ptr(sigma), dev.stream_ptr())
    return mu, sigma


def logprior_gauss(params, prm):
    x = _matrix(params)
    out = dev.empty((x.shape[0],))
    _lib.call('elfi_b200_logprior_gauss_f64', dev.context(), dev.ptr(x), _ld(x), x.shape[0],
              dev.ptr(_gauss_prm(prm)), dev.ptr(out), dev.stream_ptr())
    return out


def sim_gauss(mu, sigma, n_obs=50, seed=0, offset=0, want_data=False, want_summaries=True):
    """Gaussian simulator on the device -> (Y or None, S or None), S = [mean, var] fused."""
    mu = dev.to_device(mu).reshape(-1).contiguous()
    sigma = dev.to_device(sigma).reshape(-1).contiguous()
    B = mu.numel()
    Y = dev.empty((B, n_obs)) if want_data else None
    S = dev.empty((B, 2)) if want_summaries else None
    _lib.call('elfi_b200_sim_gauss_f64', dev.context(), dev.ptr(mu), dev.ptr(sigma), B, n_obs,
              int(seed), int(offset), dev.ptr(Y), n_obs, dev.ptr(S), 2, dev.stream_ptr())
    return Y, S


def sim_gnk(A, B, g, k, n_obs=50, seed=0, offset=0, c=0.8):
    """g-and-k simulator on the device (elfi/examples/gnk.py:11-68) -> Y (batch, n_obs)."""
    cols = [dev.to_device(v).reshape(-1).contiguous() for v in (A, B, g, k)]
    n = cols[0].numel()
    if any(col.numel() != n for col in cols):
        raise ValueError('A, B, g and k must have the same number of elements')
    Y = dev.empty((n, n_obs))
    _lib.call('elfi_b200_sim_gnk_f64', dev.context(), dev.ptr(cols[0]), dev.ptr(cols[1]),
              dev.ptr(cols[2]), dev.ptr(cols[3]), float(c), n, n_obs, int(seed), int(offset),
              dev.ptr(Y), n_obs, dev.stream_ptr())
    return Y


def logprior_box(params, lo, width):
    """Sum of independent uniform(lo, width) log densities per row (scipy convention: -inf
    outside); the joint prior of the g-and-k example (elfi/examples/gnk.py:99-103)."""
    x = _matrix(params)
    p = x.shape[1]
    box = np.ascontiguousarray(np.concatenate([np.broadcast_to(np.asarray(lo, dtype=np.float64), (p,)),
                                               np.broadcast_to(np.asarray(width, dtype=np.float64), (p,))]))
    out = dev.empty((x.shape[0],))
    _lib.call('elfi_b200_logprior_box_f64', dev.context(), dev.ptr(x), _ld(x), x.shape[0], p,
              dev.ptr(box), dev.ptr(out), dev.stream_ptr())
    return out


def kliep_fit(x, y, weights_x=None, weights_y=None, sigma=1.0, n_basis=100, epsilon=0.001,
              max_iter=200, abs_tol=0.01, conv_check_interval=20):
    """KLIEP fit on the device (elfi/methods/density_ratio_estimation.py:71-207).

    Returns (alpha device tensor (n_basis,), max_ratio float, steps int)."""
    x = _matrix(x)
    y = _matrix(y)
    if x.shape[0] < n_basis:
        raise ValueError("Number of RBFs ({}) can't be larger than number of samples ({}).".format(
            n_basis, x.shape[0]))
    wx = None if weights_x is None else dev.to_device(weights_x).reshape(-1)
    wy = None if weights_y is None else dev.to_device(weights_y).reshape(-1)
    alpha = dev.empty((n_basis,))
    res = (ctypes.c_double * 2)()
    dev.synchronize()   # this entry point runs on its own stream order: inputs must be complete
    _lib.call('elfi_b200_kliep_fit_f64', dev.context(), dev.ptr(x), _ld(x), x.shape[0], dev.ptr(y),
              _ld(y), y.shape[0], x.shape[1], dev.ptr(wx), dev.ptr(wy), float(sigma), int(n_basis),
              float(epsilon), int(max_iter), float(abs_tol), int(conv_check_interval),
              dev.ptr(alpha), res)
    return alpha, float(res[0]), int(res[1])


SYNLIK_ESTIMATORS = {'gaussian': 0, 'ghurye_olkin': 1}


def synlik(S, obs, n, *, group_stride=None, estimator='gaussian', whitening=None, gammas=None):
    """Gaussian synthetic log-likelihoods of groups of n simulated summary rows
    (elfi/methods/bsl/pdf_methods.py:77-176) in one call of elfi_b200_synlik_f64.

    S : (rows, d) array, group g = rows g * group_stride .. g * group_stride + n - 1 (group_stride
        defaults to n; a row-strided view is read in place), or (P, n_rows, d) with group_stride
        n_rows.
    estimator : 'gaussian' or 'ghurye_olkin' (the unbiased estimator; no whitening / gammas).
    whitening : (d, d) matrix Wh or None.
    gammas : None (no shrinkage) or the L Warton parameters gamma = 1 - penalty (host values).

    Returns a (P, L) device tensor; -inf for a group with non-finite values or a singular
    covariance."""
    if estimator not in SYNLIK_ESTIMATORS:
        raise ValueError('unknown synthetic likelihood estimator {!r}'.format(estimator))
    if dev.is_device_array(S) and S.dim() == 3 or not dev.is_device_array(S) and np.ndim(S) == 3:
        S = dev.to_device(S)
        if group_stride is None:
            group_stride = S.shape[1]
        S = S.reshape(-1, S.shape[2])
    S = _matrix(S)
    rows, d = S.shape
    n = int(n)
    gs = n if group_stride is None else int(group_stride)
    P = (rows - n) // gs + 1 if rows >= n and gs > 0 else 0
    obs_t = dev.to_device(obs).reshape(-1)
    if obs_t.numel() != d:
        raise ValueError('obs has {} entries, the summaries {} columns'.format(obs_t.numel(), d))
    W = None
    if whitening is not None:
        W = dev.to_device(whitening).contiguous()
        if tuple(W.shape) != (d, d):
            raise ValueError('whitening must be a ({0}, {0}) matrix'.format(d))
    g = None if gammas is None else np.ascontiguousarray(np.atleast_1d(gammas), dtype=np.float64)
    L = 1 if g is None else len(g)
    out = dev.empty((P, L))
    _lib.call('elfi_b200_synlik_f64', dev.context(), SYNLIK_ESTIMATORS[estimator], dev.ptr(S),
              S.stride(0) if rows > 1 else d, P, n, gs, d, dev.ptr(obs_t), dev.ptr(W), dev.ptr(g),
              L, dev.ptr(out), dev.stream_ptr())
    return out


def rowsort(x):
    """np.sort(x, axis=1) on the device (ascending, NaN last); order-statistic summaries."""
    x = _matrix(x)
    B, n = x.shape
    out = dev.empty((B, n))
    _lib.call('elfi_b200_rowsort_f64', dev.context(), dev.ptr(x), _ld(x), B, n, dev.ptr(out), n,
              dev.stream_ptr())
    return out
