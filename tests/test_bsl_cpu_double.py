"""BSL on the CPU test double (bodies in tests/bsl_cases.py; reference goldens in
tests/golden/bsl.npz): the synthetic-likelihood entry point is the NumPy restatement."""
import pytest

import bsl_cases as cases


@pytest.fixture(autouse=True)
def bsl_double(cpu_double, monkeypatch):
    cases.install_restatement(monkeypatch)
    return cpu_double


def test_restatement_matches_golden():
    cases.case_restatement_matches_golden()


def test_factories_match_golden():
    cases.case_factories_match_golden()


@pytest.mark.parametrize('name', sorted(cases.CHAINS))
def test_chain_matches_golden(name):
    cases.case_chain_matches_golden(name)


def test_pre_sampling_match_golden():
    cases.case_pre_sampling_match_golden()


def test_unsupported_raise():
    cases.case_unsupported_raise()


def test_argument_errors():
    cases.case_argument_errors()


def test_first_round_not_finite():
    cases.case_first_round_not_finite()


def test_one_synlik_call_per_round(bsl_double):
    """A round is one synthetic-likelihood call; a user's callable gets host arrays instead."""
    import numpy as np
    import elfi_b200 as elfi
    from elfi_b200.examples import ma2
    m = cases.ma2_model(ma2)
    del bsl_double.CALLS[:]
    res = elfi.BSL(m, 60, ["MA2"], seed=3).sample(20, sigma_proposals=cases.SIGMA,
                                                   params0=cases.THETA)
    rounds = res.n_sim // 60
    assert bsl_double.CALLS.count('elfi_b200_synlik_f64') == rounds
    seen = []

    def host_lik(ssx, ssy):
        seen.append((type(ssx), ssx.shape, ssy.shape))
        return cases.synlik_reference(ssx, ssy, len(ssx))[0]
    elfi.BSL(m, 60, ["MA2"], likelihood=host_lik, seed=3).sample(
        5, sigma_proposals=cases.SIGMA, params0=cases.THETA)
    assert seen and all(t is np.ndarray and s == (60, 50) and o == (1, 50) for t, s, o in seen)


def test_synlik_operator_layouts(bsl_double):
    """ops.synlik: strided groups, (P, n, d) input, L penalties, the restatement's -inf cases."""
    import numpy as np
    from elfi_b200 import ops
    rs = np.random.RandomState(5)
    S = rs.randn(3 * 40, 4)
    S[45, 2] = np.nan
    obs = rs.randn(4)
    got = ops.synlik(S, obs, 30, group_stride=40, gammas=[1.0, 0.5]).cpu().numpy()
    want = cases.synlik_reference(S, obs, 30, 40, gammas=[1.0, 0.5])
    assert got.shape == (3, 2) and np.isneginf(got[1]).all()
    np.testing.assert_allclose(got, want)
    got3 = ops.synlik(S.reshape(3, 40, 4), obs, 40).cpu().numpy()
    np.testing.assert_allclose(got3, cases.synlik_reference(S, obs, 40))
    with pytest.raises(elfi_err()):
        ops.synlik(S, obs, 1)


def elfi_err():
    from elfi_b200._lib import ElfiB200Error
    return ElfiB200Error
