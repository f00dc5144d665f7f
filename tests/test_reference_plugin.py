"""Plugin boundaries of SURVEY.md section 8b, driven by the UNMODIFIED reference (its copy
in oracle/_ref/ that build() makes from a checkout, or ELFI_REFERENCE; they skip without it):
  * #2 the client: elfi_b200.client.Client under the reference's BatchHandler / samplers
    (CPU: the node operations are the reference's host ones);
  * #1 the operators: the reference's own Rejection on a model whose Distance and Summary
    operations are the ctypes stubs of integration/elfi_b200_ops.py (INTEGRATION.md section B),
    i.e. the CUDA kernels inside an unmodified ELFI -- GPU test, bit-equal to the golden.
The same operator model under elfi_b200's own samplers, the stubs against SciPy / NumPy and the
client under the BatchHandler's task protocol are checked against the committed goldens without
the reference."""
import os
import sys
from functools import partial

import numpy as np
import pytest

from conftest import load_golden

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, 'oracle'))
import ref_shim  # noqa: E402

needs_reference = pytest.mark.skipif(
    not ref_shim.reference_available(),
    reason='the reference ELFI package is not present (build with a checkout of it, or set '
           'ELFI_REFERENCE)')


def _operator_model(elfi, ma2, b200, distance):
    """MA2 with host priors / simulator and the device stubs as its Summary and Distance."""
    y = ma2.MA2(.6, .2, random_state=np.random.RandomState(4))
    m = elfi.ElfiModel()
    elfi.Prior(ma2.CustomPrior1, 2, model=m, name='t1')
    elfi.Prior(ma2.CustomPrior2, m['t1'], 1, name='t2')
    elfi.Simulator(partial(ma2.MA2, n_obs=100), m['t1'], m['t2'], observed=y, name='MA2')
    elfi.Summary(b200.device_autocov, m['MA2'], name='S1')
    elfi.Summary(partial(b200.device_autocov, lag=2), m['MA2'], name='S2')
    elfi.Distance(distance, m['S1'], m['S2'], name='d')
    return m


def _ops_module():
    sys.path.insert(0, os.path.join(ROOT, 'integration'))
    import elfi_b200_ops
    return elfi_b200_ops


@needs_reference
@pytest.mark.gpu
def test_reference_rejection_with_device_operators():
    """elfi.Rejection (reference code, reference client loop) + device Distance / Summary."""
    elfi = ref_shim.import_reference()
    from elfi.examples import ma2
    b200 = _ops_module()
    import importlib
    import elfi_b200.client as bc
    importlib.reload(bc)
    g = load_golden('ma2_rejection_quantile')
    old = elfi.client.get_client()
    try:
        elfi.set_client(bc.Client(devices=[0]))
        m = _operator_model(elfi, ma2, b200, b200.device_cdist_euclidean)
        res = elfi.Rejection(m['d'], batch_size=1000, seed=123).sample(100, quantile=0.01,
                                                                       bar=False)
    finally:
        elfi.set_client(old)
    assert res.n_sim == int(g['n_sim']) and res.threshold == float(g['threshold'])
    assert np.array_equal(res.discrepancies, g['out_d'])
    assert np.array_equal(res.samples['t1'], g['out_t1'])
    assert np.array_equal(res.samples['t2'], g['out_t2'])
    # the reference's own SMC (proposals, importance weights, weighted quantile: all reference
    # host code) on the same device-operator model: every population equals the golden of the
    # all-host reference run bit for bit
    gs = load_golden('ma2_smc_thresholds')
    try:
        elfi.set_client(bc.Client(devices=[0]))
        smc = elfi.SMC(m['d'], batch_size=1000, seed=20).sample(150, thresholds=[.6, .3, .15],
                                                                bar=False)
    finally:
        elfi.set_client(old)
    assert len(smc.populations) == int(gs['n_pops']) and smc.n_sim == int(gs['n_sim'])
    for i, pop in enumerate(smc.populations):
        assert np.array_equal(pop.discrepancies, gs['pop{}_out_d'.format(i)])
        assert np.array_equal(pop.samples['t1'], gs['pop{}_out_t1'.format(i)])
        assert np.array_equal(pop.weights, gs['pop{}_weights'.format(i)])


@pytest.mark.gpu
def test_device_operators_under_own_samplers():
    """The operator model of the test above under elfi_b200's Rejection and SMC: the rejection
    sample equals the golden of the all-host reference run bit for bit, the SMC populations
    within the tolerances of test_samplers_gpu."""
    import elfi_b200 as elfi
    from elfi_b200.examples import ma2
    from test_samplers_gpu import _check_smc
    b200 = _ops_module()
    # elfi_b200 hands a callable distance the stacked summaries as one device matrix
    m = _operator_model(elfi, ma2, b200,
                        lambda XA, XB: b200.device_cdist_euclidean(XA.cpu().numpy(), XB))
    g = load_golden('ma2_rejection_quantile')
    res = elfi.Rejection(m['d'], batch_size=1000, seed=123).sample(100, quantile=0.01, bar=False)
    assert res.n_sim == int(g['n_sim']) and res.threshold == float(g['threshold'])
    assert np.array_equal(res.discrepancies, g['out_d'])
    assert np.array_equal(res.samples['t1'], g['out_t1'])
    assert np.array_equal(res.samples['t2'], g['out_t2'])
    smc = elfi.SMC(m['d'], batch_size=1000, seed=20).sample(150, thresholds=[.6, .3, .15],
                                                           bar=False)
    _check_smc(smc, load_golden('ma2_smc_thresholds'))


@pytest.mark.gpu
def test_device_operator_stubs_match_scipy():
    """The stubs alone against SciPy / NumPy."""
    b200 = _ops_module()
    from scipy.spatial.distance import cdist
    rs = np.random.RandomState(5)
    S, obs, w = rs.randn(3000, 128), rs.randn(1, 128), rs.rand(128)
    assert np.array_equal(b200.device_cdist_euclidean(S, obs), cdist(S, obs, 'euclidean'))
    assert np.array_equal(b200.device_cdist_euclidean(S, obs, w=w), cdist(S, obs, 'euclidean', w=w))
    x = rs.randn(500, 100)
    assert np.array_equal(b200.device_autocov(x, 2), np.mean(x[:, 2:] * x[:, :-2], axis=1))


def test_client_runs_reference_rejection(cpu_double):
    """Config #1 (MA2, batch 1000, seed 123, quantile 0.01) with elfi_b200's Client as the batch
    client, equal to the reference's golden.  Without the reference, the client is driven the way
    the reference's BatchHandler drives it (elfi/client.py:129-182: at most num_cores batches in
    flight, results taken by task id in batch order) over elfi_b200's MA2 batches on the host
    double of the library; with the reference present, its own Rejection drives it too."""
    import elfi_b200.model as em
    from elfi_b200 import device as dev
    from elfi_b200.client import Client
    from elfi_b200.examples import ma2 as b200_ma2
    g = load_golden('ma2_rejection_quantile')
    client = Client(devices=[0])
    assert client.num_cores == 1
    m = b200_ma2.get_model(seed_obs=4)
    context = em.ComputationContext(batch_size=1000, seed=123)
    n_batches = int(np.ceil(100 / 0.01 / 1000))        # quantile mode: n_sim = n / quantile
    pending, batches = [], []
    for i in range(n_batches):
        while len(pending) >= client.num_cores:
            batches.append(client.get_result(pending.pop(0)))
        pending.append(client.apply(em.execute_batch, m, ['t1', 't2', 'd'], context, i))
    batches += [client.get_result(t) for t in pending]
    assert not client.tasks
    out = {k: np.concatenate([dev.to_host(b[k]).reshape(-1) for b in batches])
           for k in ('t1', 't2', 'd')}
    best = np.argsort(out['d'], kind='mergesort')[:100]
    assert len(out['d']) == int(g['n_sim'])
    assert out['d'][best[-1]] == float(g['threshold'])
    assert np.array_equal(out['d'][best], g['out_d'])
    assert np.array_equal(out['t1'][best], g['out_t1'])
    assert np.array_equal(out['t2'][best], g['out_t2'])
    if not ref_shim.reference_available():
        return
    elfi = ref_shim.import_reference()
    from elfi.examples import ma2
    import importlib
    import elfi_b200.client as bc
    importlib.reload(bc)                       # pick up elfi.client.ClientBase as the base class
    assert issubclass(bc.Client, elfi.client.ClientBase)
    old = elfi.client.get_client()
    try:
        elfi.set_client(bc.Client(devices=[0]))
        assert elfi.client.get_client().num_cores == 1
        m = ma2.get_model(seed_obs=4)
        res = elfi.Rejection(m['d'], batch_size=1000, seed=123).sample(100, quantile=0.01,
                                                                       bar=False)
    finally:
        elfi.set_client(old)
    g = load_golden('ma2_rejection_quantile')
    assert res.n_sim == int(g['n_sim'])
    assert np.array_equal(res.discrepancies, g['out_d'])


def test_client_task_api():
    from elfi_b200.client import Client
    c = Client(devices=[0])
    a = c.apply(lambda x, y=1: x + y, 2, y=3)
    b = c.apply(lambda: 7)
    assert c.is_ready(a) and c.num_cores == 1
    c.remove_task(b)
    assert c.get_result(a) == 5
    with pytest.raises(KeyError):
        c.get_result(b)
    assert c.apply_sync(lambda: 'ok') == 'ok'
    c.reset()
    assert not c.tasks


@pytest.mark.gpu
def test_client_spreads_batches_over_devices():
    """Two worker threads (both on GPU 0 here, any two GPUs on a bigger box): tasks land on
    devices round-robin, run concurrently and come back by id."""
    import threading
    import torch
    from elfi_b200.client import Client
    n = min(2, torch.cuda.device_count())
    c = Client(devices=list(range(n)) if n == 2 else [0, 0])
    assert c.num_cores == 2
    seen = []

    def task(i):
        seen.append((i, torch.cuda.current_device(), threading.get_ident()))
        return torch.full((4,), float(i), device='cuda').sum().item()
    ids = [c.apply(task, i) for i in range(6)]
    assert [c.get_result(t) for t in ids] == [4.0 * i for i in range(6)]
    assert len({ident for _, _, ident in seen}) == 2
    for i, device, _ in seen:
        assert device == c.devices[i % 2]
