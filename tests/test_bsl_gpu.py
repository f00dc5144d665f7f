"""BSL on the device: elfi_b200_synlik_f64 against the fp64 NumPy restatement of tests/bsl_cases.py
(itself pinned against the reference's values), the golden chains and pre-sampling results, the
device MA2 model at the reference's own BSL bound, and the unmodified reference's BSL with the
ctypes likelihood stub."""
import os
import sys
from functools import partial

import numpy as np
import pytest

import bsl_cases as cases

pytestmark = [pytest.mark.gpu, pytest.mark.first_device_run]

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _groups(rs, P, n, d, stride, ld):
    """P well-conditioned groups of n rows in a (P * stride, ld) buffer; returns (view, host)."""
    import torch
    buf = np.full((P * stride, ld), 7.0)
    for g in range(P):
        A = np.eye(d) + 0.1 * rs.randn(d, d) / np.sqrt(d)
        buf[g * stride:g * stride + n, :d] = rs.randn(n, d) @ A.T + rs.randn(d)
    t = torch.from_numpy(buf).cuda()
    return t[:, :d], buf[:, :d]


def _tol(S, n, stride, P):
    """1e-8 on covariances with condition number <= 1e4; the n = d + 2 groups are worse
    conditioned, and the bound grows with their condition number (rounding of the factor)."""
    conds = [np.linalg.cond(np.atleast_2d(np.cov(S[g * stride:g * stride + n], rowvar=False)))
             for g in range(P)]
    return 1e-8 * max(1.0, max(c for c in conds if np.isfinite(c)) / 1e4)


@pytest.mark.parametrize('n_kind', ['d+2', 100, 500, 5000])
@pytest.mark.parametrize('d', [1, 2, 8, 50, 127, 128])
def test_kernel_matches_restatement(d, n_kind):
    from elfi_b200 import ops
    rs = np.random.RandomState(d * 7919 + (n_kind if isinstance(n_kind, int) else 1))
    n = d + 2 if n_kind == 'd+2' else n_kind
    P, stride, ld = 3, n + 3, d + 5          # group_stride > n and a strided leading dimension
    S, host = _groups(rs, P, n, d, stride, ld)
    obs = host[:n].mean(0) + 0.3 * rs.randn(d)
    tol = _tol(host, n, stride, P)
    got = ops.synlik(S, obs, n, group_stride=stride).cpu().numpy()
    cases._close(got, cases.synlik_reference(host, obs, n, stride), tol)
    got = ops.synlik(S, obs, n, group_stride=stride, estimator='ghurye_olkin').cpu().numpy()
    cases._close(got, cases.synlik_reference(host, obs, n, stride, 'ghurye_olkin'), tol)
    Wh = np.eye(d) + 0.1 * rs.randn(d, d) / np.sqrt(d)
    gam = np.linspace(0.2, 1.0, 31)
    got = ops.synlik(S, obs, n, group_stride=stride, whitening=Wh, gammas=gam).cpu().numpy()
    cases._close(got, cases.synlik_reference(host, obs, n, stride, whitening=Wh, gammas=gam),
                 tol * 10)
    # a NaN group and a singular group next to a normal one: the neighbour is unaffected.  The
    # Warton penalties add (1 - gamma) 1e-5 to the diagonal, so only gamma = 1 leaves the singular
    # group singular.  The singular group repeats one row of integers: its mean is then exact in
    # np.cov's two-pass arithmetic too, so the covariance is exactly zero in both implementations
    # (a row of arbitrary doubles leaves a rounding-level variance, ~1e-32, in np.cov's mean).
    host2 = host.copy()
    host2[stride + n // 2, d - 1] = np.nan
    host2[2 * stride:2 * stride + n] = np.round(host2[2 * stride])
    import torch
    S2 = torch.from_numpy(np.ascontiguousarray(host2)).cuda()
    got = ops.synlik(S2, obs, n, group_stride=stride).cpu().numpy()
    assert np.isneginf(got[1:]).all()
    cases._close(got, cases.synlik_reference(host2, obs, n, stride), tol)
    got = ops.synlik(S2, obs, n, group_stride=stride, gammas=gam).cpu().numpy()
    want = cases.synlik_reference(host2, obs, n, stride, gammas=gam)
    assert np.isneginf(got[1]).all() and np.isneginf(got[2, -1])
    cases._close(got[0], want[0], tol)


@pytest.mark.parametrize('P,n,d,L', [(1024, 500, 50, 1), (1024, 100, 2, 1), (1024, 130, 128, 1),
                                     (10, 100, 50, 31)])
def test_kernel_many_groups(P, n, d, L):
    from elfi_b200 import ops
    rs = np.random.RandomState(P + n + d + L)
    S, host = _groups(rs, P, n, d, n, d)
    obs = host[:n].mean(0) + 0.3 * rs.randn(d)
    gam = None if L == 1 else np.linspace(0.1, 1.0, L)
    got = ops.synlik(S, obs, n, gammas=gam).cpu().numpy()
    cases._close(got, cases.synlik_reference(host, obs, n, gammas=gam), _tol(host, n, n, 3))


def test_kernel_argument_errors():
    from elfi_b200 import ops
    from elfi_b200._lib import ElfiB200Error
    rs = np.random.RandomState(0)
    with pytest.raises(ElfiB200Error, match='d = 129'):
        ops.synlik(rs.randn(40, 129), rs.randn(129), 20)
    with pytest.raises(ElfiB200Error, match='at least 2 rows'):
        ops.synlik(rs.randn(40, 3), rs.randn(3), 1)
    with pytest.raises(ElfiB200Error, match='group_stride'):
        ops.synlik(rs.randn(40, 3), rs.randn(3), 20, group_stride=10)
    with pytest.raises(ElfiB200Error, match='Ghurye-Olkin'):
        ops.synlik(rs.randn(40, 3), rs.randn(3), 20, estimator='ghurye_olkin', gammas=[0.5])


def test_factories_match_golden():
    cases.case_factories_match_golden()


@pytest.mark.parametrize('name', sorted(cases.CHAINS))
def test_chain_matches_golden(name):
    cases.case_chain_matches_golden(name)


def test_pre_sampling_match_golden():
    cases.case_pre_sampling_match_golden()


@pytest.mark.parametrize('features', [['S1', 'S2'], ['MA2']])
def test_device_model_posterior(features):
    """The reference's check_bsl (tests/functional/test_inference.py:251-265) on the device model:
    2000 iterations at n_sim_round = 500, posterior mean within 0.15 of the true (0.6, 0.2)."""
    import elfi_b200 as elfi
    from elfi_b200.examples import ma2
    m = ma2.get_device_model(n_obs=50, true_params=cases.THETA, seed_obs=4)
    res = elfi.BSL(m, 500, features, seed=123).sample(2000, sigma_proposals=cases.SIGMA,
                                                      params0=np.array(cases.THETA))
    means = np.array([np.mean(res.samples[p]) for p in ('t1', 't2')])
    assert np.all(np.abs(means - np.array(cases.THETA)) < 0.15), means
    # proposals outside the prior support are rejected without simulating
    assert 0 < res.acc_rate < 1 and res.n_sim <= 2000 * 500 and res.n_sim % 500 == 0


def test_reference_bsl_with_device_likelihood():
    """The UNMODIFIED reference's BSL with the ctypes stub as its likelihood reproduces the
    golden standard chain."""
    sys.path.insert(0, os.path.join(ROOT, 'oracle'))
    import ref_shim
    if not ref_shim.reference_available():
        pytest.skip('the reference ELFI package is not present')
    elfi = ref_shim.import_reference()
    if not hasattr(np, 'NINF'):
        np.NINF = -np.inf
    from elfi.examples import ma2
    sys.path.insert(0, os.path.join(ROOT, 'integration'))
    import elfi_b200_ops as b200
    g = cases.load_golden('bsl')
    cfg = cases.CHAINS['standard']
    m = cases.ma2_model(ma2)
    bsl = elfi.BSL(m, cfg['n_sim_round'], cfg['features'],
                   likelihood=partial(b200.device_gaussian_syn_likelihood), seed=cases.SEED)
    res = bsl.sample(cfg['n_samples'], sigma_proposals=cases.SIGMA, params0=cfg['params0'])
    got = np.column_stack([res.samples_all[p] for p in m.parameter_names])
    assert np.array_equal(got, g['chain_standard_samples_all'])
    np.testing.assert_allclose(bsl.state['logposterior'], g['chain_standard_logposterior'],
                               rtol=1e-9)
