"""Golden fixtures for the BOLFI sampling path, from the UNMODIFIED reference (elfi-dev/elfi).

    ELFI_REFERENCE=<checkout of elfi-dev/elfi> python tests/golden/gen_golden_bolfi.py

* mcmc.npz            -- elfi.methods.mcmc.nuts / metropolis chains on analytic targets and the
                         ESS / R-hat of those chains (mcmc.py is pure NumPy).
* bolfi_posterior.npz -- elfi.methods.posteriors.BolfiPosterior (logpdf, gradient_logpdf),
                         elfi.model.extensions.ModelPrior.gradient_logpdf and
                         elfi.methods.bo.acquisition.MaxVar (evaluate, evaluate_gradient) evaluated on
                         a duck-typed GP whose predict / predictive_gradients are the oracle's
                         restatement of gpy_regression.py:127-160, 206-218 (GPy itself is not
                         installable here, DESIGN.md section 2).
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, 'oracle'))

from ref_shim import REFERENCE_ROOT, import_reference  # noqa: E402

elfi = import_reference()
import elfi_oracle as o  # noqa: E402
from elfi.examples import ma2  # noqa: E402
from elfi.methods import mcmc  # noqa: E402
from elfi.methods.bo.acquisition import LCBSC, ExpIntVar, MaxVar  # noqa: E402
from elfi.methods.bo.utils import minimize as ref_minimize  # noqa: E402
from elfi.methods.posteriors import BolfiPosterior  # noqa: E402
from elfi.model.extensions import ModelPrior  # noqa: E402


def save(name, **arrays):
    np.savez(os.path.join(HERE, name + '.npz'), **arrays)
    print('wrote', name, {k: np.shape(v) for k, v in arrays.items()})


# ----------------------------------------------------------------------------- analytic targets
PREC = np.linalg.inv(np.array([[1.0, 0.6], [0.6, 0.8]]))
MEAN = np.array([0.5, -0.3])


def gauss_logpdf(x):
    d = np.asarray(x) - MEAN
    return -0.5 * d @ PREC @ d


def gauss_grad(x):
    return -PREC @ (np.asarray(x) - MEAN)


BOX = (np.array([-1.0, -1.0]), np.array([2.0, 1.0]))


def boxed_logpdf(x):
    x = np.asarray(x)
    if np.any(x < BOX[0]) or np.any(x > BOX[1]):
        return -np.inf
    return gauss_logpdf(x)


def boxed_grad(x):
    x = np.asarray(x)
    if np.any(x < BOX[0]) or np.any(x > BOX[1]):
        return np.zeros(2)
    return gauss_grad(x)


class DuckGP:
    """What BolfiPosterior / MaxVar touch of GPyRegression, backed by the oracle's GP."""

    def __init__(self, X, y, hyper, bounds, parameter_names):
        self.X, self.Y = X, y.reshape(-1, 1)
        self.h = hyper
        self.bounds = bounds
        self.parameter_names = parameter_names
        self.input_dim = X.shape[1]
        self.L, self.alpha = o.gp_fit(X, y, hyper['kernel_var'], hyper['lengthscale'],
                                      hyper['bias_var'], hyper['noise_var'], jitter=1e-8)

        # ExpIntVar reaches into GPy for the prior covariance function (acquisition.py:754)
        from types import SimpleNamespace
        self._gp = SimpleNamespace(kern=SimpleNamespace(K=self._prior_cov))

    def _prior_cov(self, a, b):
        a, b = np.atleast_2d(a), np.atleast_2d(b)
        r2 = np.sum(a ** 2., 1)[:, None] + np.sum(b ** 2., 1)[None, :] - 2. * a.dot(b.T)
        return self.h['kernel_var'] * np.exp(np.maximum(r2, 0.) * (-0.5 / self.h['lengthscale'] ** 2)) \
            + self.h['bias_var']

    @property
    def noise(self):
        return self.h['noise_var']

    def predict(self, x, noiseless=False):
        x = np.asanyarray(x).reshape((-1, self.input_dim))
        mu, var = o.gp_predict(x, self.X, self.L, self.alpha, self.h['kernel_var'],
                               self.h['lengthscale'], self.h['bias_var'],
                               None if noiseless else self.h['noise_var'])
        return mu, var

    def predict_mean(self, x):
        return self.predict(x)[0]

    def predictive_gradients(self, x):
        x = np.asanyarray(x).reshape((-1, self.input_dim))
        return o.gp_predictive_gradients(x, self.X, self.L, self.alpha, self.h['kernel_var'],
                                         self.h['lengthscale'], self.h['bias_var'])

    def predictive_gradient_mean(self, x):
        return self.predictive_gradients(x)[0]


def main():
    # ---- MCMC
    out = {}
    out['nuts_gauss'] = mcmc.nuts(300, np.array([1.5, 0.5]), gauss_logpdf, gauss_grad, n_adapt=100,
                                  seed=11)
    out['nuts_gauss_depth3'] = mcmc.nuts(200, np.array([-1.0, 0.2]), gauss_logpdf, gauss_grad,
                                         n_adapt=50, max_depth=3, target_prob=0.8, seed=5)
    out['nuts_boxed'] = mcmc.nuts(300, np.array([1.8, 0.9]), boxed_logpdf, boxed_grad, n_adapt=100,
                                  seed=3)
    out['nuts_fixed_step'] = mcmc.nuts(100, np.array([0.0, 0.0]), gauss_logpdf, gauss_grad,
                                       n_adapt=0, stepsize=0.4, seed=7)
    out['metropolis'] = mcmc.metropolis(400, np.array([1.5, 0.5]), boxed_logpdf,
                                        np.array([0.4, 0.3]), warmup=50, seed=9)
    chains = np.stack([mcmc.nuts(200, np.array([0.1 * i, -0.1 * i]), gauss_logpdf, gauss_grad,
                                 n_adapt=100, seed=20 + i) for i in range(4)])
    out['chains'] = chains
    out['ess'] = np.array([mcmc.eff_sample_size(chains[:, :, k]) for k in range(2)])
    out['ess_single'] = np.float64(mcmc.eff_sample_size(chains[0, :, 0]))
    out['rhat'] = np.array([mcmc.gelman_rubin_statistic(chains[:, :, k]) for k in range(2)])
    # known-answer values held by the reference's own test (tests/unit/test_mcmc.py: chains
    # generated in PyStan with Stan's ESS and split R-hat)
    import importlib.util
    spec = importlib.util.spec_from_file_location(
        'ref_test_mcmc', os.path.join(REFERENCE_ROOT, 'tests', 'unit', 'test_mcmc.py'))
    ref_test = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ref_test)
    out['stan_chains'] = np.asarray(ref_test.chains_Stan)
    out['stan_ess'] = np.float64(ref_test.ess_Stan)
    out['stan_rhat'] = np.float64(ref_test.Rhat_Stan)
    save('mcmc', **out)

    # ---- BolfiPosterior / ModelPrior gradient / MaxVar on the duck GP, MA2 priors
    m = ma2.get_model(seed_obs=4)
    prior = ModelPrior(m)
    rs = np.random.RandomState(2)
    X = np.column_stack([rs.uniform(-2, 2, 80), rs.uniform(-1, 1, 80)])
    y = np.log(0.05 + (X[:, 0] - 0.6) ** 2 + 2 * (X[:, 1] - 0.2) ** 2) + 0.1 * rs.randn(80)
    hyper = dict(kernel_var=1.3, lengthscale=0.7, bias_var=0.4, noise_var=0.05)
    bounds = [(-2, 2), (-1, 1)]
    gp = DuckGP(X, y, hyper, bounds, ['t1', 't2'])
    thr = -1.0
    post = BolfiPosterior(gp, threshold=thr, prior=prior)
    # points inside the prior support, outside it but inside the bounds, and outside the bounds
    pts = np.array([[0.6, 0.2], [0.1, 0.5], [-0.8, 0.3], [1.2, -0.1], [0.0, -0.9], [1.9, 0.9],
                    [-1.9, -0.9], [2.5, 0.0], [0.0, 1.5], [0.3, 0.31], [-0.3, 0.9]])
    with np.errstate(all='ignore'):
        logpdf = post.logpdf(pts)
        grad = post.gradient_logpdf(pts)
        loglik = post._unnormalized_loglikelihood(pts)
        gradlik = post._gradient_unnormalized_loglikelihood(pts)
        prior_grad = prior.gradient_logpdf(pts)
        prior_logpdf = prior.logpdf(pts)
        single_logpdf = post.logpdf(pts[1])
        single_grad = post.gradient_logpdf(pts[1])
    # default threshold = minimum of the GP mean found by the multi-start minimiser
    post_default = BolfiPosterior(gp, prior=prior, seed=0)

    acq = MaxVar(model=gp, prior=prior, quantile_eps=0.05, noise_var=0.1, seed=1)
    acq.eps = np.percentile(gp.Y, 5.0)
    inside = pts[[0, 1, 2, 3, 4, 9]]
    with np.errstate(all='ignore'):
        mv = acq.evaluate(inside)
        mv_grad = acq.evaluate_gradient(inside)
    eiv = ExpIntVar(model=gp, prior=prior, quantile_eps=0.05, integration='grid', d_grid=0.4,
                    noise_var=0.1, seed=1, n_inits=5, max_opt_iters=100)
    with np.errstate(all='ignore'):
        eiv_x = eiv.acquire(1, t=0)
        eiv_pts = np.vstack([inside, eiv_x])
        eiv_loss = eiv.evaluate(eiv_pts)
        eiv_single = eiv.evaluate(inside[1])
    save('expintvar', X=X, y=y, hyper=np.array([hyper[k] for k in
                                                ('kernel_var', 'lengthscale', 'bias_var',
                                                 'noise_var')]),
         grid=eiv.points_int, eps=np.float64(eiv.eps), pts=eiv_pts, loss=eiv_loss,
         single=eiv_single, acquired=eiv_x, omegas=eiv.omegas_int, phi_int=eiv.phi_int)

    # ---- LCBSC.evaluate / evaluate_gradient / acquire / _add_noise (acquisition.py:129-301) and
    # bo.utils.minimize (utils.py:40-111) of the reference classes on the same duck GP
    lc = LCBSC(model=gp, prior=prior, noise_var=0.1, exploration_rate=10, seed=1, n_inits=10,
               max_opt_iters=1000)
    lc_pts = pts[[0, 1, 2, 3, 4, 5, 9]]
    lc_out = {'pts': lc_pts}
    for t in (0, 4, 40):
        lc_out['value_t{}'.format(t)] = lc.evaluate(lc_pts, t)
        lc_out['grad_t{}'.format(t)] = lc.evaluate_gradient(lc_pts, t)
        lc_out['beta_t{}'.format(t)] = np.float64(lc._beta(t))
    lc_out['acquired_t4'] = lc.acquire(3, t=4)              # consumes lc.random_state
    lc_out['acquired_t5'] = lc.acquire(2, t=5)              # ... further
    lc_quiet = LCBSC(model=gp, prior=prior, noise_var=0, exploration_rate=10, seed=3, n_inits=6)
    lc_out['acquired_quiet'] = lc_quiet.acquire(2, t=2)     # no noise: the minimiser itself
    lc_dict = LCBSC(model=gp, prior=None, noise_var={'t1': 0.2, 't2': 0.0}, delta=0.2, seed=5)
    lc_out['acquired_dict'] = lc_dict.acquire(4, t=1)       # uniform starts, per-parameter noise
    lc_noise = LCBSC(model=gp, prior=prior, noise_var=0.5, seed=9)
    edge = np.array([[1.99, -0.99], [-1.99, 0.99], [0.0, 0.0], [0.6, 0.2]])
    lc_out['noise_in'] = edge.copy()
    lc_out['noise_out'] = lc_noise._add_noise(edge.copy())

    def quad(x):
        x = np.atleast_2d(x)
        return (x[:, 0] - 0.3) ** 2 + 3 * (x[:, 1] + 0.4) ** 2 + 0.5 * np.sin(5 * x[:, 0])

    def quad_grad(x):
        x = np.atleast_2d(x)
        return np.column_stack([2 * (x[:, 0] - 0.3) + 2.5 * np.cos(5 * x[:, 0]), 6 * (x[:, 1] + 0.4)])
    loc, val = ref_minimize(quad, bounds, grad=quad_grad, prior=prior, n_start_points=7,
                            random_state=np.random.RandomState(4))
    loc_u, val_u = ref_minimize(quad, bounds, grad=quad_grad, prior=None, n_start_points=5,
                                random_state=np.random.RandomState(6))
    lc_out.update(min_loc=loc, min_val=np.float64(val), min_loc_uniform=loc_u,
                  min_val_uniform=np.float64(val_u))
    save('lcbsc_acquire', X=X, y=y, hyper=np.array([hyper[k] for k in
                                                    ('kernel_var', 'lengthscale', 'bias_var',
                                                     'noise_var')]), **lc_out)

    save('bolfi_posterior', X=X, y=y, hyper=np.array([hyper[k] for k in
                                                      ('kernel_var', 'lengthscale', 'bias_var',
                                                       'noise_var')]),
         threshold=np.float64(thr), pts=pts, logpdf=logpdf, grad=grad, loglik=loglik,
         gradlik=gradlik, prior_grad=prior_grad, prior_logpdf=prior_logpdf,
         single_logpdf=np.float64(single_logpdf), single_grad=single_grad,
         default_threshold=np.float64(post_default.threshold),
         maxvar_eps=np.float64(acq.eps), maxvar_pts=inside, maxvar=mv, maxvar_grad=mv_grad)


if __name__ == '__main__':
    main()
