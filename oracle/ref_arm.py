"""CPU arm of bench.py (`--impl reference`): the UNMODIFIED reference's own code, timed on the host.

BASELINE INFRASTRUCTURE ONLY (like the rest of oracle/): imported by bench.py's reference arm and
by tests; never by the product.  The reference package is imported through ref_shim (from the
checkout that ELFI_REFERENCE points to).

Config #2 step = one 1e6 x 128 batch through the reference's distance node and its rejection
merge, i.e. exactly what `elfi.Rejection(d, batch_size=1e6)` does per batch:
  * `distance_as_discrepancy(partial(cdist, metric='euclidean'), S, observed=(obs,))`
        (elfi/model/utils.py:37-52, the operation of elfi.Distance, elfi_model.py:1037)
  * `Rejection.update(batch, batch_index)` -> `_merge_batch` (mask, copy to the buffer tail,
        argsort over n + batch_size rows, permutation of every output), `_update_state_meta`,
        `_update_objective_n_batches`                     (elfi/methods/inference/samplers.py:140-277)
All host cores: the reference parallelises over batches in worker processes and merges in the
master (elfi/clients/multiprocessing.py, parameter_inference.py:270-305).  Here the rows of ONE
batch are spread over `processes` forked workers (more favourable to the reference than its own
batch-per-process client: no idle cores for a single batch) and, as in the reference's pipeline,
the master merges batch k while the workers compute batch k + 1.
"""
import multiprocessing as mp
import os
import time
from functools import partial

import numpy as np

from ref_shim import import_reference

_G = {}


def _worker_distance(bounds):
    lo, hi = bounds
    from scipy.spatial.distance import cdist
    dad = _G['distance_as_discrepancy']
    return dad(partial(cdist, metric='euclidean'), _G['S'][lo:hi], observed=(_G['obs'],))


class ReferenceRejectionStep:
    """Drives the reference's own Distance operation and Rejection.update on synthetic batches."""

    def __init__(self, S, obs, params, threshold, n_samples, processes=None):
        elfi = import_reference()
        from elfi.examples import ma2
        from elfi.model.utils import distance_as_discrepancy
        self.elfi = elfi
        self.S, self.obs = S, np.atleast_2d(obs)
        self.t1, self.t2 = params
        self.B = len(S)
        self.processes = processes or os.cpu_count() or 1
        _G.update(S=self.S, obs=self.obs, distance_as_discrepancy=distance_as_discrepancy)
        m = ma2.get_model(seed_obs=4)
        self.rej = elfi.Rejection(m['d'], batch_size=self.B, seed=1)
        self.rej.set_objective(n_samples, threshold=threshold)
        self.pool = None
        if self.processes > 1:
            # fork: the workers see S without a copy (as the reference's workers hold their own
            # simulator output); must be created after _G is filled
            self.pool = mp.get_context('fork').Pool(self.processes)
            per = -(-self.B // self.processes)
            self.bounds = [(lo, min(self.B, lo + per)) for lo in range(0, self.B, per)]
        self._pending = None
        self._index = 0

    def _submit(self):
        if self.pool is None:
            return None
        return self.pool.map_async(_worker_distance, self.bounds)

    def _collect(self, pending):
        if self.pool is None:
            return _worker_distance((0, self.B))
        return np.concatenate(pending.get())

    def distances(self):
        return self._collect(self._submit())

    def step(self):
        """One batch; with workers the next batch's distances are computed during the merge."""
        if self._pending is None:
            self._pending = self._submit()
        d = self._collect(self._pending)
        self._pending = self._submit()
        self.rej.update({'d': d, 't1': self.t1, 't2': self.t2}, self._index)
        self._index += 1
        return d

    def accepted_now(self):
        st = self.rej.state['samples']
        n = self.rej.objective['n_samples']
        return st['d'][:n], st['t1'][:n], st['t2'][:n]

    def close(self):
        if self.pool is not None:
            if self._pending is not None:
                try:
                    self._pending.get(timeout=60)
                except Exception:
                    pass
            self.pool.terminate()
            self.pool.join()
            self.pool = None


def time_ma2_rejection(n_sim, batch_size, processes, quantile=0.01, seed=1):
    """(ii) the reference end to end: elfi.Rejection(MA2, batch_size).sample(n_sim=...) with its
    own multiprocessing client on `processes` workers (native client when processes == 1)."""
    elfi = import_reference()
    from elfi.examples import ma2
    old = elfi.client.get_client()
    client = None
    try:
        if processes > 1:
            from elfi.clients import multiprocessing as emp
            client = emp.Client(num_processes=processes)
            elfi.set_client(client)
        else:
            elfi.set_client('native')
        m = ma2.get_model(seed_obs=4)
        rej = elfi.Rejection(m['d'], batch_size=batch_size, seed=seed)
        n_samples = int(n_sim * quantile)
        rej.sample(max(1, n_samples // 100), n_sim=batch_size * min(2, processes), bar=False)
        t0 = time.perf_counter()
        res = rej.sample(n_samples, n_sim=n_sim, bar=False)
        dt = time.perf_counter() - t0
    finally:
        if client is not None:
            client.reset()
        elfi.set_client(old)
    return {'seconds': dt, 'n_sim': int(res.n_sim), 'simulated_per_s': res.n_sim / dt,
            'accepted_per_s': n_samples / dt, 'batch_size': batch_size, 'processes': processes,
            'threshold': float(res.threshold),
            'posterior_mean_t1': float(res.sample_means['t1'])}
