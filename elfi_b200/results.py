"""Result containers with the attribute surface of elfi/methods/results.py (Sample at 73-108,
SmcSample at 387-413, OptimizationResult at 55-70): host arrays in `outputs`, parameter draws in
`samples`, optional `weights`, and every extra keyword (threshold, n_sim, accept_rate, seed, cov,
means, adaptive_distance_w, ...) readable as an attribute.  Plotting / saving are out of scope.
"""
from collections import OrderedDict
from collections.abc import Mapping

import numpy as np


def _host(v):
    """Device array -> host ndarray (one synchronising D2H copy); host values pass through."""
    return v.detach().cpu().numpy() if hasattr(v, 'is_cuda') else v


class DeviceOutputs(Mapping):
    """`outputs` of a sample whose arrays still live on the device: name -> host ndarray, copied
    to the host the first time a name is read.  The samplers hand populations from one
    generation to the next on the device, so an SMC run only pays the D2H copies of what the user
    actually looks at (the reference's Sample holds host arrays, results.py:73-108)."""

    def __init__(self, device_arrays):
        self.device = dict(device_arrays)
        self._host = {}

    def __getitem__(self, name):
        if name not in self._host:
            self._host[name] = _host(self.device[name])
        return self._host[name]

    def __iter__(self):
        return iter(self.device)

    def __len__(self):
        return len(self.device)

    def rows(self, name):
        return int(self.device[name].shape[0])


class _Result:
    """Common part: method name, node outputs, parameter names and free-form meta data."""

    def __init__(self, method_name, outputs, parameter_names, **meta):
        self.method_name = method_name
        self.outputs = outputs if isinstance(outputs, DeviceOutputs) else dict(outputs)
        self.parameter_names = parameter_names
        self.meta = meta

    def __getattr__(self, name):
        # only reached when normal lookup fails: expose the meta entries as attributes
        meta = self.__dict__.get('meta')
        if meta is not None and name in meta:
            return meta[name]
        raise AttributeError("No attribute '{}' in this sample".format(name))

    @property
    def is_multivariate(self):
        return any(np.ndim(self.outputs[p]) > 1 for p in self.parameter_names)


ParameterInferenceResult = _Result


class OptimizationResult(_Result):
    """Result of an optimisation: `x_min` holds the minimiser per parameter."""

    def __init__(self, x_min, **kwargs):
        super().__init__(**kwargs)
        self.x_min = x_min


class Sample(_Result):
    """Draws from an (approximate) posterior."""

    def __init__(self, method_name, outputs, parameter_names, discrepancy_name=None, weights=None,
                 **meta):
        super().__init__(method_name, outputs, parameter_names, **meta)
        self.discrepancy_name = discrepancy_name
        self.weights = weights

    # `samples`, `weights` and `means` may be backed by device arrays; they become host arrays
    # on first access and stay so
    @property
    def samples(self):
        cached = self.__dict__.get('_samples')
        if cached is None:
            cached = OrderedDict((name, self.outputs[name]) for name in self.parameter_names)
            self.__dict__['_samples'] = cached
        return cached

    @property
    def weights(self):
        w = self.__dict__.get('_weights')
        if hasattr(w, 'is_cuda'):
            w = self.__dict__['_weights'] = _host(w)
        return w

    @weights.setter
    def weights(self, value):
        self.__dict__['_weights'] = value

    @property
    def means(self):
        m = self.__dict__.get('_means')
        if m is None:
            raise AttributeError("No attribute 'means' in this sample")
        if hasattr(m, 'is_cuda'):
            m = self.__dict__['_means'] = _host(m)
        return m

    @means.setter
    def means(self, value):
        self.__dict__['_means'] = value

    @property
    def n_samples(self):
        first = self.parameter_names[0]
        if isinstance(self.outputs, DeviceOutputs):
            return self.outputs.rows(first)
        return len(self.outputs[first])

    @property
    def dim(self):
        return len(self.parameter_names)

    @property
    def discrepancies(self):
        if self.discrepancy_name is None:
            return None
        return self.outputs[self.discrepancy_name]

    @property
    def samples_array(self):
        return np.column_stack([self.samples[name] for name in self.parameter_names])

    @property
    def sample_means(self):
        means = OrderedDict()
        for name, draws in self.samples.items():
            means[name] = np.average(draws, axis=0, weights=self.weights)
        return means

    @property
    def sample_means_array(self):
        return np.array([v for v in self.sample_means.values()])

    def __repr__(self):
        return '{}(method={!r}, n_samples={}, parameters={})'.format(
            type(self).__name__, self.method_name, self.n_samples, list(self.parameter_names))


class SmcSample(Sample):
    """Final population of an SMC run plus the list of all populations."""

    def __init__(self, method_name, outputs, parameter_names, populations, *args, **kwargs):
        super().__init__(method_name, outputs, parameter_names, *args, **kwargs)
        if self.__dict__.get('_weights') is None:
            raise ValueError("No weights provided for the sample")
        self.populations = populations

    @property
    def n_populations(self):
        return len(self.populations)


class BolfiSample(Sample):
    """Posterior draws of BOLFI.sample: `chains` is (n_chains, n_samples, n_parameters) with the
    warm-up iterations included; `samples` holds the post-warm-up draws of all chains
    (elfi/methods/results.py:507-543)."""

    def __init__(self, method_name, chains, parameter_names, warmup, **meta):
        chains = np.array(chains, copy=True)
        kept = chains[:, warmup:, :].reshape((-1,) + chains.shape[2:])
        outputs = {name: kept[:, i] for i, name in enumerate(parameter_names)}
        super().__init__(method_name=method_name, outputs=outputs, parameter_names=parameter_names,
                         chains=chains, n_chains=chains.shape[0], warmup=warmup, **meta)


class BslSample(Sample):
    """Result of BSL.sample (elfi/methods/results.py:546-605): `samples_all` holds the whole chain
    (burn-in included), `samples` / `outputs` the draws after burn-in; `acc_rate`, `burn_in` and
    `n_sim` are attributes."""

    def __init__(self, method_name, samples_all, parameter_names, burn_in=0, acc_rate=None, **meta):
        outputs = {k: samples_all[k][burn_in:] for k in samples_all}
        super().__init__(method_name=method_name, outputs=outputs, parameter_names=parameter_names,
                         samples_all=samples_all, burn_in=burn_in, acc_rate=acc_rate, **meta)

    def compute_ess(self):
        """Effective sample size of the post-burn-in chain of each parameter."""
        from .mcmc import eff_sample_size
        return {p: eff_sample_size(self.samples[p]) for p in self.parameter_names}
