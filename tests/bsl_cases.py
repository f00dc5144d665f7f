"""BSL test bodies shared by the CPU-double and GPU collections, the configuration of the golden
fixture (tests/golden/bsl.npz, generator tests/golden/gen_golden_bsl.py) and a NumPy restatement of
elfi_b200_synlik_f64 pinned against the reference's values."""
import numpy as np
from scipy import linalg

from conftest import load_golden

# ------------------------------------------------------------------------- golden configuration
SEED = 123
THETA = [0.6, 0.2]
SIGMA = np.array([[0.02, 0.01], [0.01, 0.02]])
WH_N, WH_SEED = 200, 1
WARTON_PENALTY = 0.3
PRE_N_SIM, PRE_M, PRE_SEED = [50, 100], 10, 7
CHAINS = {
    'standard': dict(features=['MA2'], n_sim_round=100, n_samples=300, params0=THETA),
    'unbiased': dict(features=['MA2'], n_sim_round=100, n_samples=200, params0=THETA),
    'wwarton': dict(features=['MA2'], n_sim_round=100, n_samples=300, params0=THETA, burn_in=50,
                    logit_transform_bound=[[-2, 2], [-1, 1]]),
    'summaries': dict(features=['S1', 'S2'], n_sim_round=100, batch_size=25, n_samples=300,
                      params0=THETA),
    'params0none': dict(features=['MA2'], n_sim_round=100, n_samples=100),
}


def ma2_model(ma2):
    return ma2.get_model(n_obs=50, true_params=THETA, seed_obs=4)


def _lik_cases():
    rs = np.random.RandomState(2024)
    cases = []
    for d, n in [(1, 40), (2, 60), (7, 80), (50, 300)]:
        A = rs.randn(d, d) / np.sqrt(d) + np.eye(d)
        ssx = rs.randn(n, d) @ A.T + rs.randn(d)
        ssy = ssx.mean(0) + 0.5 * rs.randn(d)
        # the reference's unbiased estimator returns -inf for every 1-column input: np.cov gives a
        # 0-d covariance there and slogdet raises; this package computes the value
        cases.append(dict(name='d{}'.format(d), data='d{}'.format(d), ssx=ssx, ssy=ssy, go=d > 1))
        Wh = np.eye(d) + 0.1 * rs.randn(d, d)
        if d > 1:   # the reference squeezes a 1-d observation to a scalar it cannot whiten
            cases.append(dict(name='d{}w'.format(d), data='d{}'.format(d), ssx=ssx, ssy=ssy,
                              whitening=Wh, penalties=[0.0, 0.3, 0.8]))
        cases.append(dict(name='d{}p'.format(d), data='d{}'.format(d), ssx=ssx, ssy=ssy,
                          penalties=[0.05, 0.5, 0.95]))
    ssx = rs.randn(5, 7)
    cases.append(dict(name='singular', data='singular', ssx=ssx, ssy=rs.randn(7)))
    ssx = rs.randn(30, 3)
    ssx[4, 1] = np.nan
    cases.append(dict(name='nan', data='nan', ssx=ssx, ssy=rs.randn(3), nan=True))
    return cases


LIK_CASES = _lik_cases()


# ---------------------------------------------------------------------------- NumPy restatement
def synlik_reference(S, obs, n, group_stride=None, estimator='gaussian', whitening=None,
                     gammas=None):
    """elfi_b200_synlik_f64 in NumPy: (P, L) log-likelihoods of the groups of S (rows, d)."""
    S = np.asarray(S, dtype=np.float64)
    gs = n if group_stride is None else group_stride
    P = (S.shape[0] - n) // gs + 1
    d = S.shape[1]
    gam = [None] if gammas is None else list(gammas)
    out = np.full((P, len(gam)), -np.inf)
    for g in range(P):
        X = S[g * gs:g * gs + n]
        if not np.all(np.isfinite(X)):
            continue
        mu = X.mean(0)
        Sigma = np.atleast_2d(np.cov(X, rowvar=False))
        r = np.asarray(obs, dtype=np.float64).reshape(-1) - mu
        if whitening is not None:
            Sigma = whitening @ Sigma @ whitening.T
            r = whitening @ r
        for l, gamma in enumerate(gam):
            A = Sigma if gamma is None else \
                gamma * Sigma + (1 - gamma) * np.diag(np.diag(Sigma) + 1e-5)
            tol = 1e6 * np.finfo(np.float64).eps * np.max(np.diag(A))
            try:
                Lf = linalg.cholesky(A, lower=True)
            except linalg.LinAlgError:
                continue
            if np.any(np.diag(Lf) ** 2 <= tol):
                continue
            z = linalg.solve_triangular(Lf, r, lower=True)
            q = float(z @ z)
            logdet = 2.0 * float(np.sum(np.log(np.diag(Lf))))
            if estimator == 'gaussian':
                out[g, l] = -0.5 * (q + logdet + d * np.log(2 * np.pi))
            else:
                from scipy.special import gammaln
                wcon = lambda k, nu: (-k * nu / 2 * np.log(2) - k * (k - 1) / 4 * np.log(np.pi)  # noqa: E731
                                      - np.sum(gammaln([0.5 * (nu - x) for x in range(k)])))
                logdet_psi = d * np.log(n - 1) + logdet + np.log(abs(1 - q * n / (n - 1) ** 2))
                A_ = wcon(d, n - 2) - wcon(d, n - 1) - 0.5 * d * np.log(1 - 1 / n)
                B_ = -0.5 * (n - d - 2) * (np.log(n - 1) + logdet)
                C_ = 0.5 * (n - d - 3) * logdet_psi
                out[g, l] = -0.5 * d * np.log(2 * np.pi) + A_ + B_ + C_
    return out


def install_restatement(monkeypatch):
    """Put the restatement behind the CPU double's elfi_b200_synlik_f64."""
    import abi_double as ad
    from elfi_b200 import _lib

    def synlik_f64(ctx, estimator, S, ldS, P, n, group_stride, d, obs, Wh, gamma_host, L, loglik,
                   stream):
        ad._require(1 <= d <= 128 and n >= 2 and group_stride >= n and L >= 1,
                    'synlik: argument out of range')
        ad._require(ad._addr(gamma_host) or L == 1, 'synlik: L > 1 needs gammas')
        ad._require(estimator == 0 or not (ad._addr(Wh) or ad._addr(gamma_host)),
                    'synlik: Ghurye-Olkin takes neither whitening nor shrinkage')
        if P == 0:
            return
        rows = (P - 1) * group_stride + n
        g = ad._vec(gamma_host, L)
        if g is not None:
            ad._require(np.all((g >= 0) & (g <= 1)), 'synlik: gamma outside [0, 1]')
        res = synlik_reference(ad._mat(S, rows, d, ldS), ad._vec(obs, d), int(n), int(group_stride),
                               'gaussian' if estimator == 0 else 'ghurye_olkin',
                               ad._mat(Wh, d, d), None if g is None else g.copy())
        ad._mat(loglik, P, L)[:] = res

    monkeypatch.setitem(ad._TABLE, 'elfi_b200_synlik_f64', synlik_f64)
    assert 'elfi_b200_synlik_f64' in _lib.SIGNATURES


# ---------------------------------------------------------------------------------------- cases
def _lik_values(case, g):
    name = case['name']
    ssx, ssy = g['lik_{}_ssx'.format(case['data'])], g['lik_{}_ssy'.format(case['data'])]
    wh = g.get('lik_{}_wh'.format(name))
    pens = g.get('lik_{}_pen'.format(name))
    return ssx, ssy, wh, pens


def _close(got, want, tol=1e-8):
    got, want = np.asarray(got, dtype=float), np.asarray(want, dtype=float)
    assert got.shape == want.shape, (got.shape, want.shape)
    fin = np.isfinite(want)
    assert np.array_equal(fin, np.isfinite(got)), (got, want)
    assert np.array_equal(got[~fin], want[~fin])
    assert np.all(np.abs(got[fin] - want[fin]) <= tol * np.maximum(1, np.abs(want[fin]))), \
        np.max(np.abs(got[fin] - want[fin]))


def case_restatement_matches_golden():
    g = load_golden('bsl')
    for case in LIK_CASES:
        name = case['name']
        ssx, ssy, wh, pens = _lik_values(case, g)
        gam = None if pens is None else 1 - pens
        got = synlik_reference(ssx, ssy, len(ssx), whitening=wh, gammas=gam)[0]
        _close(got, g['lik_{}_gauss'.format(name)], 1e-9)
        if 'lik_{}_go'.format(name) in g:
            _close(synlik_reference(ssx, ssy, len(ssx), estimator='ghurye_olkin')[0],
                   g['lik_{}_go'.format(name)], 1e-9)


def case_factories_match_golden():
    from elfi_b200 import bsl
    g = load_golden('bsl')
    for case in LIK_CASES:
        name = case['name']
        ssx, ssy, wh, pens = _lik_values(case, g)
        if pens is None:
            got = bsl.gaussian_syn_likelihood(ssx, ssy, whitening=wh)
        else:
            got = np.concatenate([bsl.standard_likelihood('warton', p, wh)(ssx, ssy) for p in pens])
        _close(got, g['lik_{}_gauss'.format(name)])
        if 'lik_{}_go'.format(name) in g:
            _close(bsl.unbiased_likelihood()(ssx, ssy), g['lik_{}_go'.format(name)])


def run_chain(name, model=None):
    import elfi_b200 as elfi
    from elfi_b200 import bsl
    from elfi_b200.examples import ma2
    g = load_golden('bsl')
    cfg = CHAINS[name]
    m = model if model is not None else ma2_model(ma2)
    lik = {'unbiased': bsl.unbiased_likelihood(),
           'wwarton': bsl.standard_likelihood(shrinkage='warton', penalty=WARTON_PENALTY,
                                              whitening=g['pre_whitening'])}.get(name)
    sampler = elfi.BSL(m, cfg['n_sim_round'], cfg['features'], likelihood=lik,
                       batch_size=cfg.get('batch_size'), seed=SEED)
    res = sampler.sample(cfg['n_samples'], sigma_proposals=SIGMA, params0=cfg.get('params0'),
                         burn_in=cfg.get('burn_in', 0),
                         logit_transform_bound=cfg.get('logit_transform_bound'))
    return g, sampler, res


def case_chain_matches_golden(name):
    g, sampler, res = run_chain(name)
    key = 'chain_{}_'.format(name)
    got = np.column_stack([res.samples_all[p] for p in res.parameter_names])
    assert np.array_equal(got, g[key + 'samples_all'])
    np.testing.assert_allclose(sampler.state['logposterior'], g[key + 'logposterior'], rtol=1e-9)
    assert res.acc_rate == float(g[key + 'acc_rate'])
    assert res.n_sim == int(g[key + 'n_sim'])
    burn = CHAINS[name].get('burn_in', 0)
    assert np.array_equal(res.samples['t1'], res.samples_all['t1'][burn:])
    ess = res.compute_ess()
    assert set(ess) == {'t1', 't2'} and all(v > 0 for v in ess.values())


def case_pre_sampling_match_golden():
    from elfi_b200 import bsl
    from elfi_b200.examples import ma2
    g = load_golden('bsl')
    W = bsl.estimate_whitening_matrix(ma2_model(ma2), WH_N, THETA, ['MA2'], seed=WH_SEED)
    assert np.array_equal(W, g['pre_whitening'])
    sd = bsl.log_SL_stdev(ma2_model(ma2), THETA, PRE_N_SIM, ['MA2'], M=PRE_M, seed=PRE_SEED)
    np.testing.assert_allclose(sd, g['pre_log_sl_stdev'], rtol=1e-8)
    lmdas, stds = bsl.select_penalty(ma2_model(ma2), PRE_N_SIM, THETA, ['MA2'], M=PRE_M, sigma=1.5,
                                     shrinkage='warton', whitening=g['pre_whitening'],
                                     seed=PRE_SEED)
    assert np.array_equal(lmdas, g['pre_select_lmdas'])
    np.testing.assert_allclose(stds, g['pre_select_stds'], rtol=1e-8)


def case_unsupported_raise():
    import pytest
    from elfi_b200 import bsl
    for call in (lambda: bsl.standard_likelihood(shrinkage='glasso', penalty=0.1),
                 lambda: bsl.semiparametric_likelihood(),
                 lambda: bsl.robust_likelihood('mean'),
                 lambda: bsl.gaussian_syn_likelihood(np.ones((5, 2)), np.ones(2), 'glasso', 0.1)):
        with pytest.raises(NotImplementedError):
            call()


def case_argument_errors():
    import pytest
    import elfi_b200 as elfi
    from elfi_b200.examples import ma2
    m = ma2_model(ma2)
    with pytest.raises(ValueError, match='n_sim_round must be a multiple of batch_size'):
        elfi.BSL(m, 100, ['MA2'], batch_size=30)
    with pytest.raises(ValueError, match='Node nope not found in the model'):
        elfi.BSL(m, 100, ['nope'])
    sampler = elfi.BSL(m, 100, ['MA2'], seed=1)
    with pytest.raises(ValueError, match='outside prior support'):
        sampler.sample(10, sigma_proposals=SIGMA, params0=[3.0, 0.0])
    with pytest.raises(ValueError, match='Gamma must be between 0 and 1'):
        elfi.bsl.standard_likelihood(shrinkage='warton', penalty=1.5)
    # default features: every public Summary node
    assert elfi.BSL(m, 100, seed=1).feature_names == ['S1', 'S2']


def case_first_round_not_finite():
    import pytest
    import elfi_b200 as elfi
    from elfi_b200.examples import ma2
    sampler = elfi.BSL(ma2_model(ma2), 20, ['MA2'], likelihood=lambda x, y: -np.inf, seed=1)
    with pytest.raises(RuntimeError, match='not finite on initialisation round'):
        sampler.sample(5, sigma_proposals=SIGMA, params0=THETA)
