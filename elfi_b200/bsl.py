"""Bayesian synthetic likelihood (BSL) with the likelihood estimate on the device.

Host control flow mirrors the reference (file:line in elfi-dev/elfi v0.8.7):
  ModelBased                        elfi/methods/inference/parameter_inference.py:374-545
  BSL                               elfi/methods/inference/bsl.py:21-442
  likelihood factories              elfi/methods/bsl/pdf_methods.py:19-176
  log_SL_stdev, select_penalty,     elfi/methods/bsl/pre_sample_methods.py:102-318
  estimate_whitening_matrix
What runs on the GPU: the features of a round are written into one (n_sim_round, d) device buffer
and reduced by ONE call of elfi_b200_synlik_f64 (mean, covariance, optional whitening and Warton
shrinkage, Cholesky factor, Gaussian log density); the Metropolis-Hastings test then reads a single
double back.  The pre-sampling tools evaluate all M x len(n_sim) x L log-likelihoods of a given n
in one call.  A likelihood that is a user's own Python callable runs on the host with host arrays.

Out of scope: semiBSL, robust BSL, graphical-lasso shrinkage and its `standardise` flag (they
raise NotImplementedError), the plotting pre-sample methods, several chains, multi-GPU BSL.
"""
import logging
from functools import partial

import numpy as np
from scipy import linalg

from . import device as dev
from . import model as em
from . import ops
from .results import BslSample
from .samplers import ModelPrior, ParameterInference

logger = logging.getLogger(__name__)

__all__ = ['BSL', 'ModelBased', 'standard_likelihood', 'unbiased_likelihood',
           'semiparametric_likelihood', 'robust_likelihood', 'gaussian_syn_likelihood',
           'gaussian_syn_likelihood_ghurye_olkin', 'log_SL_stdev', 'select_penalty',
           'estimate_whitening_matrix']


def _out_of_scope(what):
    raise NotImplementedError(
        '{} is not implemented in elfi_b200: only the Gaussian synthetic likelihood (standard, '
        'with whitening and Warton shrinkage, or the unbiased estimator) runs on the device; '
        'semiBSL, robust BSL and graphical-lasso shrinkage are out of scope'.format(what))


def _warton_gammas(shrinkage, penalty):
    """Warton parameters gamma = 1 - penalty (cov_warton(S, 1 - penalty), pdf_methods.py:122-123),
    or None without shrinkage.  Other strings are ignored, as in the reference."""
    if shrinkage == 'glasso':
        _out_of_scope("shrinkage='glasso'")
    if shrinkage != 'warton':
        return None
    gammas = 1 - np.atleast_1d(np.asarray(penalty, dtype=np.float64))
    if np.any(gammas < 0) or np.any(gammas > 1):
        raise ValueError("Gamma must be between 0 and 1")
    return gammas


class SynLikelihood:
    """A Gaussian synthetic likelihood evaluated by elfi_b200_synlik_f64: the callable the factories
    return.  ``self(ssx, ssy)`` takes ssx as (n, d) or (P, n, d), host or device, and returns the
    host log-likelihoods ((1,) or (P,)); ``device(ssx, ssy)`` returns the (P,) device tensor."""

    def __init__(self, estimator='gaussian', shrinkage=None, penalty=None, whitening=None):
        self.estimator = estimator
        self.gammas = _warton_gammas(shrinkage, penalty)
        if self.gammas is not None and len(self.gammas) != 1:
            raise ValueError('penalty must be a single value')
        self.whitening = None if whitening is None else np.asarray(whitening, dtype=np.float64)
        self._wh_dev = None

    def _wh(self):
        if self.whitening is not None and self._wh_dev is None:
            self._wh_dev = dev.to_device(self.whitening)
        return self._wh_dev

    def device(self, ssx, ssy, n=None, group_stride=None):
        obs = ssy if dev.is_device_array(ssy) else np.asarray(ssy, dtype=np.float64)
        if n is None:
            n = ssx.shape[-2] if len(ssx.shape) == 3 else ssx.shape[0]
        return ops.synlik(ssx, obs, n, group_stride=group_stride, estimator=self.estimator,
                          whitening=self._wh(), gammas=self.gammas)[:, 0]

    def __call__(self, ssx, ssy):
        return dev.to_host(self.device(ssx, ssy))


def gaussian_syn_likelihood(ssx, ssy, shrinkage=None, penalty=None, whitening=None,
                            standardise=False):
    """Standard synthetic log-likelihood (pdf_methods.py:77-135); `standardise` only matters for
    the graphical lasso, which is out of scope."""
    return SynLikelihood('gaussian', shrinkage, penalty, whitening)(ssx, ssy)


def gaussian_syn_likelihood_ghurye_olkin(ssx, ssy):
    """Unbiased synthetic log-likelihood of Ghurye & Olkin (pdf_methods.py:138-176)."""
    return SynLikelihood('ghurye_olkin')(ssx, ssy)


def standard_likelihood(shrinkage=None, penalty=None, whitening=None, standardise=False):
    if shrinkage == 'glasso':
        _out_of_scope("shrinkage='glasso'")
    return SynLikelihood('gaussian', shrinkage, penalty, whitening)


def unbiased_likelihood():
    return SynLikelihood('ghurye_olkin')


def semiparametric_likelihood(shrinkage=None, penalty=None, whitening=None):
    _out_of_scope('semiparametric_likelihood (semiBSL)')


def robust_likelihood(adjustment):
    _out_of_scope('robust_likelihood (R-BSL)')


def _device_form(likelihood):
    """The SynLikelihood behind `likelihood`, or None for a user's host callable."""
    if isinstance(likelihood, SynLikelihood):
        return likelihood
    if likelihood is gaussian_syn_likelihood:
        return SynLikelihood('gaussian')
    if likelihood is gaussian_syn_likelihood_ghurye_olkin:
        return SynLikelihood('ghurye_olkin')
    if isinstance(likelihood, partial) and likelihood.func is gaussian_syn_likelihood \
            and not likelihood.args:
        kw = dict(likelihood.keywords)
        kw.pop('standardise', None)
        return SynLikelihood('gaussian', **kw)
    return None


# ------------------------------------------------------------------------------------ features
def _columns(value, rows):
    """One feature of a batch as a (rows, width) device matrix: host arrays are uploaded, device
    tensors used as they are, lazily simulated outputs (LazyMA2Data) materialised."""
    if hasattr(value, 'materialize'):
        value = value.materialize()
    t = value if dev.is_device_array(value) else dev.to_device(np.asarray(value, dtype=np.float64))
    return t.reshape(rows, -1)


def _feature_width(model, names):
    return int(sum(np.size(dev.to_host(model[name].observed)) for name in names))


def _observed(model, names):
    return np.column_stack([dev.to_host(model[name].observed) for name in names])


def _write_features(batch, names, out, row0, rows):
    col = 0
    for name in names:
        t = _columns(batch[name], rows)
        out[row0:row0 + rows, col:col + t.shape[1]] = t
        col += t.shape[1]


def _simulate_features(model, names, params, counts_seeds, width):
    """model.generate(n_i, outputs=names, with_values=params, seed=s_i) for every (n_i, s_i),
    stacked into one (sum n_i, width) device buffer in that order."""
    total = sum(n for n, _ in counts_seeds)
    out = dev.empty((total, width))
    row = 0
    for n, seed in counts_seeds:
        batch = model.generate(int(n), outputs=list(names), with_values=params, seed=seed)
        _write_features(batch, names, out, row, int(n))
        row += int(n)
    return out


def _resolve_theta(model, theta, feature_names):
    params = theta if isinstance(theta, dict) else dict(zip(model.parameter_names, theta))
    feature_names = [feature_names] if isinstance(feature_names, str) else list(feature_names)
    return params, feature_names


# ----------------------------------------------------------------------------------- inference
class ModelBased(ParameterInference):
    """Inference that runs n_sim_round simulations at one parameter value per round
    (parameter_inference.py:374-545).  The features of a round go into one device buffer
    `simulated` of shape (n_sim_round, d)."""

    def __init__(self, model, n_sim_round, feature_names=None, batch_size=None, **kwargs):
        self.n_sim_round = n_sim_round
        batch_size = batch_size or self.n_sim_round
        if n_sim_round % batch_size != 0:
            raise ValueError('n_sim_round must be a multiple of batch_size.')
        model = model.model if isinstance(model, em.NodeReference) else model
        feature_names = [feature_names] if isinstance(feature_names, str) else feature_names
        self.feature_names = feature_names or self._get_summary_names(model)
        if len(self.feature_names) == 0:
            raise ValueError('feature_names must include at least one item.')
        for node in self.feature_names:
            if node not in model.nodes:
                raise ValueError('Node {} not found in the model'.format(node))
        output_names = model.parameter_names + self.feature_names
        super().__init__(model, output_names, batch_size=batch_size, distributed=False, **kwargs)
        self.observed = _observed(self.model, self.feature_names)
        self.state['round'] = 0
        self.state['n_sim_round'] = 0
        self.simulated = dev.zeros((self.n_sim_round, self.observed.size))

    @staticmethod
    def _get_summary_names(model):
        return [node for node in model.nodes if isinstance(model[node], em.Summary)
                and not node.startswith('_')]

    def _init_state(self):
        self.state['n_batches'] = 0
        self.state['n_sim'] = 0
        self.state['round'] = 0
        self.state['n_sim_round'] = 0

    def set_objective(self, rounds):
        self.objective['round'] = rounds
        self.objective['n_batches'] = rounds * int(self.n_sim_round / self.batch_size)

    def update(self, batch, batch_index):
        super().update(batch, batch_index)
        self._merge_batch(batch)
        if self.state['n_sim_round'] == self.n_sim_round:
            self._process_simulated()
            self.state['round'] += 1
            if self.state['round'] < self.objective['round']:
                self._init_round()

    def _init_round(self):
        self.state['n_sim_round'] = 0

    def _process_simulated(self):
        raise NotImplementedError

    def prepare_new_batch(self, batch_index):
        params = np.atleast_2d(self.current_params)
        batch_params = np.repeat(params, self.batch_size, axis=0)
        return {name: batch_params[:, i] for i, name in enumerate(self.parameter_names)}

    @property
    def current_params(self):
        raise NotImplementedError

    def infer(self, *args, **kwargs):
        if self.state['round'] > 0:
            self._init_round()
        return super().infer(*args, **kwargs)

    def _merge_batch(self, batch):
        _write_features(batch, self.feature_names, self.simulated, self.state['n_sim_round'],
                        self.batch_size)
        self.state['n_sim_round'] += self.batch_size


class BSL(ModelBased):
    """Bayesian synthetic likelihood with a random-walk Metropolis-Hastings sampler
    (bsl.py:21-442; Price et al. 2018).  Each round makes one device call and reads one double."""

    def __init__(self, model, n_sim_round, feature_names=None, likelihood=None, **kwargs):
        super().__init__(model, n_sim_round, feature_names=feature_names, **kwargs)
        self.random_state = np.random.RandomState(self.seed)
        self.likelihood = likelihood or gaussian_syn_likelihood
        self._synlik = _device_form(self.likelihood)
        self._obs_dev = dev.to_device(self.observed.reshape(-1))
        self.param_names = None
        self.prior = None
        self.sigma_proposals = None
        self.burn_in = 0
        self.logit_transform_bound = None

    @property
    def parameter_names(self):
        return self.param_names or self.model.parameter_names

    def sample(self, n_samples, sigma_proposals, params0=None, param_names=None, burn_in=0,
               logit_transform_bound=None, **kwargs):
        """Run n_samples Metropolis-Hastings iterations (burn-in included); returns BslSample."""
        self.sigma_proposals = sigma_proposals
        self.param_names = param_names
        self.prior = ModelPrior(self.model, parameter_names=self.parameter_names)
        self.burn_in = burn_in
        self.logit_transform_bound = None if logit_transform_bound is None \
            else np.array(logit_transform_bound)
        self._init_state(n_samples, params0)
        return self.infer(n_samples, **kwargs)

    def _init_state(self, n_samples, params0=None):
        super()._init_state()
        if params0 is None:
            params0 = self.model.generate(1, self.parameter_names, seed=self.seed)
            params0 = np.column_stack([dev.to_host(params0[p]) for p in self.parameter_names])
        else:
            params0 = np.array(params0)
            if not np.isfinite(self.prior.logpdf(params0)):
                raise ValueError('Initial point {} is outside prior support.'.format(params0))
        self.state['n_samples'] = 0
        self.num_accepted = 0
        self.state['params'] = np.zeros((n_samples, len(self.parameter_names)))
        self.state['params'][0] = params0
        self.state['logprior'] = np.zeros(n_samples)
        self.state['logprior'][0] = np.squeeze(self.prior.logpdf(params0))
        self.state['logposterior'] = np.zeros(n_samples)

    def extract_result(self):
        samples_all = {p: np.array(self.state['params'][:, i])
                       for i, p in enumerate(self.parameter_names)}
        acc_rate = self.num_accepted / (self.state['n_samples'] - self.burn_in)
        logger.info("MCMC acceptance rate: {}".format(acc_rate))
        return BslSample(method_name='BSL', samples_all=samples_all, acc_rate=acc_rate,
                         burn_in=self.burn_in, n_sim=self.state['n_sim'],
                         parameter_names=self.parameter_names)

    @property
    def current_params(self):
        return self.state['params'][self.state['n_samples']]

    def _init_round(self):
        """Draw proposals until one lies inside the prior support; each rejected proposal is a
        chain step without simulations and drops the objective by one round."""
        while self.state['n_samples'] < len(self.state['params']):
            n = self.state['n_samples']
            prop = self._propagate_state()
            logprior = self.prior.logpdf(prop)
            if np.isfinite(logprior):
                self.state['logprior'][n] = np.squeeze(logprior)
                self.state['params'][n] = prop
                self.state['n_sim_round'] = 0
                break
            self.state['logprior'][n] = self.state['logprior'][n - 1]
            self.state['params'][n] = self.state['params'][n - 1]
            self.state['logposterior'][n] = self.state['logposterior'][n - 1]
            self.state['n_samples'] += 1
            self.set_objective(self.objective['round'] - 1)

    def _loglikelihood(self):
        if self._synlik is not None:
            return float(self._synlik.device(self.simulated, self._obs_dev)[0].item())
        simulated = dev.to_host(self.simulated)
        if not np.all(np.isfinite(simulated)):
            return -np.inf
        return float(np.squeeze(self.likelihood(simulated, self.observed)))

    def _process_simulated(self):
        loglikelihood = self._loglikelihood()
        n = self.state['n_samples']
        if not np.isfinite(loglikelihood):
            if n == 0:
                raise RuntimeError('Estimated likelihood not finite on initialisation round.')
            logger.warning('Estimated likelihood not finite.')
        self.state['logposterior'][n] = loglikelihood + self.state['logprior'][n]
        if n == 0:
            accept_candidate = True
        else:
            prob = np.minimum(1.0, self._get_mh_ratio())
            accept_candidate = self.random_state.uniform() < prob
        if accept_candidate:
            if n >= self.burn_in:
                self.num_accepted += 1
        else:
            self.state['logprior'][n] = self.state['logprior'][n - 1]
            self.state['params'][n] = self.state['params'][n - 1]
            self.state['logposterior'][n] = self.state['logposterior'][n - 1]
        self.state['n_samples'] += 1

    def _propagate_state(self):
        mean = self.state['params'][self.state['n_samples'] - 1]
        if self.logit_transform_bound is not None:
            mean_tilde = self._para_logit_transform(mean, self.logit_transform_bound)
            sample = self.random_state.multivariate_normal(mean_tilde, self.sigma_proposals)
            prop = self._para_logit_back_transform(sample, self.logit_transform_bound)
        else:
            prop = self.random_state.multivariate_normal(mean, self.sigma_proposals)
        return np.atleast_2d(prop)

    def _get_mh_ratio(self):
        n = self.state['n_samples']
        logp2 = 0
        if self.logit_transform_bound is not None:
            logp2 = self._jacobian_logit_transform(self.state['params'][n],
                                                   self.logit_transform_bound) - \
                self._jacobian_logit_transform(self.state['params'][n - 1],
                                               self.logit_transform_bound)
        res = logp2 + self.state['logposterior'][n] - self.state['logposterior'][n - 1]
        res = 700 if res > 700 else res          # the reference's overflow guard
        res = -700 if res < -700 else res
        return np.exp(res)

    # Bounds per parameter: both finite -> logit, only the upper -> log(1 / (b - x)), only the
    # lower -> log(x - a), none -> identity (bsl.py:322-442).
    @staticmethod
    def _bound_types(bound):
        return np.matmul(np.isinf(bound), [1, 2])

    @classmethod
    def _para_logit_transform(cls, theta, bound):
        theta = theta.flatten()
        out = np.zeros(len(theta))
        for i, kind in enumerate(cls._bound_types(bound)):
            a, b, x = bound[i, 0], bound[i, 1], theta[i]
            if kind == 0:
                out[i] = np.log((x - a) / (b - x))
            elif kind == 1:
                out[i] = np.log(1 / (b - x))
            elif kind == 2:
                out[i] = np.log(x - a)
            else:
                out[i] = x
        return out

    @classmethod
    def _para_logit_back_transform(cls, theta_tilde, bound):
        theta_tilde = theta_tilde.flatten()
        out = np.zeros(len(theta_tilde))
        for i, kind in enumerate(cls._bound_types(bound)):
            a, b, y = bound[i, 0], bound[i, 1], theta_tilde[i]
            ey = np.exp(y)
            if kind == 0:
                out[i] = a / (1 + ey) + b / (1 + (1 / ey))
            elif kind == 1:
                out[i] = b - (1 / ey)
            elif kind == 2:
                out[i] = a + ey
            else:
                out[i] = y
        return out

    @classmethod
    def _jacobian_logit_transform(cls, theta_tilde, bound):
        theta_tilde = theta_tilde.flatten()
        logJ = np.zeros(len(theta_tilde))
        for i, kind in enumerate(cls._bound_types(bound)):
            y = theta_tilde[i]
            if kind == 0:
                ey = np.exp(y)
                logJ[i] = np.log(bound[i, 1] - bound[i, 0]) - np.log((1 / ey) + 2 + ey)
            elif kind in (1, 2):
                logJ[i] = y
        return np.sum(logJ)


# ------------------------------------------------------------------------- pre-sampling tools
def log_SL_stdev(model, theta, n_sim, feature_names, likelihood=None, M=20, seed=None):
    """Standard deviation of the log synthetic likelihood over M data sets for each n in n_sim
    (pre_sample_methods.py:102-143): the reference's child seeds and model.generate calls, then
    one synthetic-likelihood call per n over all M data sets."""
    params, feature_names = _resolve_theta(model, theta, feature_names)
    observed = _observed(model, feature_names)
    likelihood = likelihood or gaussian_syn_likelihood
    n_sim = np.atleast_1d(n_sim)
    max_sim = int(max(n_sim))
    child_seeds = np.random.SeedSequence(seed).generate_state(M)
    ssx = _simulate_features(model, feature_names, params, [(max_sim, s) for s in child_seeds],
                             observed.size)
    ll = np.zeros((len(n_sim), M))
    synlik = _device_form(likelihood)
    for n_i, n in enumerate(n_sim):
        if synlik is not None:
            ll[n_i] = dev.to_host(synlik.device(ssx, observed, n=int(n), group_stride=max_sim))
        else:
            host = dev.to_host(ssx)
            for i in range(M):
                ll[n_i, i] = np.squeeze(likelihood(host[i * max_sim:i * max_sim + n], observed))
    return np.std(ll, axis=1)


def estimate_whitening_matrix(model, n_sim, theta, feature_names, likelihood_type="standard",
                              seed=None):
    """Whitening matrix of Priddle et al. 2021 for the standard likelihood
    (pre_sample_methods.py:146-212); the d x d eigendecomposition is host work."""
    if likelihood_type not in ["standard", "semiparametric"]:
        raise ValueError("Unsupported likelihood type \'{}\'.".format(likelihood_type))
    if likelihood_type == "semiparametric":
        _out_of_scope('the semiparametric whitening matrix')
    params, feature_names = _resolve_theta(model, theta, feature_names)
    width = _feature_width(model, feature_names)
    ssx = dev.to_host(_simulate_features(model, feature_names, params, [(n_sim, seed)], width))
    ns = ssx.shape[0]
    mu = np.mean(ssx, axis=0)
    std = np.std(ssx, axis=0)
    ssx_std = (ssx - np.tile(np.array([mu]), (ns, 1))) / np.tile(np.array([std]), (ns, 1))
    cov_mat = np.cov(np.transpose(ssx_std))
    w, v = linalg.eig(cov_mat)
    diag_w = np.diag(np.power(w, -0.5)).real.round(8)
    return np.dot(diag_w, v.T).real.round(8)


def select_penalty(model, n_sim, theta, feature_names, likelihood=None, lmdas=None, M=20,
                   sigma=1.5, shrinkage="glasso", whitening=None, seed=None, verbose=False):
    """Warton penalty whose log-likelihood standard deviation is closest to sigma, per n in n_sim
    (pre_sample_methods.py:215-318).  All M x len(lmdas) log-likelihoods of one n come from one
    synthetic-likelihood call."""
    if shrinkage != 'warton':
        _out_of_scope("select_penalty with shrinkage={!r}".format(shrinkage))
    params, feature_names = _resolve_theta(model, theta, feature_names)
    ssy = _observed(model, feature_names)
    likelihood = likelihood or gaussian_syn_likelihood
    if lmdas is None:
        lmdas = list(np.arange(0.2, 0.8, 0.02))
    n_lambda = len(lmdas)
    batch_size = np.array([n_sim]).flatten()
    ns = len(batch_size)
    max_sim = int(max(batch_size))
    child_seeds = np.random.SeedSequence(seed).generate_state(M)
    ssx = _simulate_features(model, feature_names, params, [(max_sim, s) for s in child_seeds],
                             ssy.size)
    logliks = np.zeros((M, ns, n_lambda))
    if likelihood is gaussian_syn_likelihood:
        gammas = _warton_gammas('warton', lmdas)
        wh = None if whitening is None else np.asarray(whitening, dtype=np.float64)
        for n_i, n in enumerate(batch_size):
            logliks[:, n_i, :] = dev.to_host(ops.synlik(ssx, ssy, int(n), group_stride=max_sim,
                                                        whitening=wh, gammas=gammas))
    else:
        host = dev.to_host(ssx)
        for m in range(M):
            for n_i, n in enumerate(batch_size):
                ssx_n = host[m * max_sim:m * max_sim + n]
                for j in range(n_lambda):
                    logliks[m, n_i, j] = np.squeeze(likelihood(ssx_n, ssy, shrinkage=shrinkage,
                                                               penalty=lmdas[j],
                                                               whitening=whitening))
    closest_lmdas = np.zeros(ns)
    closest_std_devs = np.zeros(ns)
    for i in range(ns):
        std_devs = np.array([np.std(logliks[:, i, j]) for j in range(n_lambda)])
        closest_arg = np.argmin(np.abs(std_devs - sigma))
        closest_lmdas[i] = lmdas[closest_arg]
        closest_std_devs[i] = std_devs[closest_arg]
    if verbose:
        print('logliks: ', logliks)
        print('std_devs: ', std_devs)
    return closest_lmdas, closest_std_devs
