"""Generate the golden fixtures from the UNMODIFIED reference (elfi-dev/elfi v0.8.7).

Needs a checkout of the reference, which the tests themselves never do:

    ELFI_REFERENCE=<checkout of elfi-dev/elfi> python tests/golden/gen_golden.py

Writes tests/golden/*.npz / *.json.  The reference is imported through oracle/ref_shim.py
(stubs for packages that are absent here and that the sampler path never touches).
"""
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, 'oracle'))

from ref_shim import import_reference  # noqa: E402

elfi = import_reference()
from elfi.examples import gauss, ma2  # noqa: E402
from elfi.methods.utils import (GMDistribution, weighted_sample_quantile,  # noqa: E402
                                weighted_var)
from elfi.model.extensions import ModelPrior  # noqa: E402
from elfi.utils import get_sub_seed  # noqa: E402


def save(name, **arrays):
    np.savez(os.path.join(HERE, name + '.npz'), **arrays)
    print('wrote', name, {k: np.shape(v) for k, v in arrays.items()})


def sample_arrays(res, prefix=''):
    out = {prefix + 'threshold': np.float64(res.threshold), prefix + 'n_sim': np.int64(res.n_sim),
           prefix + 'n_batches': np.int64(res.n_batches)}
    for k, v in res.outputs.items():
        out[prefix + 'out_' + k] = np.asarray(v)
    if getattr(res, 'weights', None) is not None:
        out[prefix + 'weights'] = np.asarray(res.weights)
    return out


def main():
    meta = {'numpy': np.__version__}
    import scipy
    meta['scipy'] = scipy.__version__

    # --- sub seeds (elfi/utils.py:71-127)
    meta['sub_seeds_123'] = [int(get_sub_seed(123, i)) for i in range(8)]
    meta['sub_seeds_1_hi'] = [int(get_sub_seed(1, i)) for i in (10, 100, 1000)]

    # --- MA2 forward pass (elfi_model.py:265-299 generate)
    m = ma2.get_model(seed_obs=4)
    gen = m.generate(1000, ['t1', 't2', 'MA2', 'S1', 'S2', 'd'], seed=123)
    save('ma2_generate', observed_MA2=np.asarray(m.observed['MA2']),
         obs_S1=np.asarray(m['S1'].observed), obs_S2=np.asarray(m['S2'].observed),
         **{k: np.asarray(v) for k, v in gen.items()})

    # --- config #1: Rejection quantile / threshold / n_sim modes
    r = elfi.Rejection(m['d'], batch_size=1000, seed=123).sample(100, quantile=0.01, bar=False)
    save('ma2_rejection_quantile', **sample_arrays(r))
    r = elfi.Rejection(m['d'], batch_size=1000, seed=123).sample(150, threshold=0.2, bar=False)
    save('ma2_rejection_threshold', **sample_arrays(r))
    r = elfi.Rejection(m['d'], batch_size=500, seed=7, output_names=['S1', 'S2']).sample(
        64, n_sim=3000, bar=False)
    save('ma2_rejection_nsim', **sample_arrays(r))

    # --- SMC with quantiles and thresholds
    s = elfi.SMC(m['d'], batch_size=1000, seed=123).sample(200, quantiles=[.5, .5, .5], bar=False)
    arrs = sample_arrays(s)
    for i, pop in enumerate(s.populations):
        arrs.update(sample_arrays(pop, 'pop{}_'.format(i)))
        arrs['pop{}_cov'.format(i)] = np.asarray(pop.cov)
    arrs['n_pops'] = np.int64(len(s.populations))
    save('ma2_smc_quantiles', **arrs)
    s = elfi.SMC(m['d'], batch_size=1000, seed=20).sample(150, thresholds=[.6, .3, .15], bar=False)
    arrs = sample_arrays(s)
    for i, pop in enumerate(s.populations):
        arrs.update(sample_arrays(pop, 'pop{}_'.format(i)))
        arrs['pop{}_cov'.format(i)] = np.asarray(pop.cov)
    arrs['n_pops'] = np.int64(len(s.populations))
    save('ma2_smc_thresholds', **arrs)

    # --- AdaptiveDistanceSMC on MA2
    m2 = ma2.get_model(seed_obs=4)
    m2['d'].become(elfi.AdaptiveDistance(m2['S1'], m2['S2']))
    ad = elfi.AdaptiveDistanceSMC(m2['d'], batch_size=500, seed=11)
    s = ad.sample(100, rounds=3, quantile=0.5, bar=False)
    arrs = sample_arrays(s)
    for i, pop in enumerate(s.populations):
        arrs.update(sample_arrays(pop, 'pop{}_'.format(i)))
        arrs['pop{}_cov'.format(i)] = np.asarray(pop.cov)
        arrs['pop{}_w'.format(i)] = np.asarray(
            pop.adaptive_distance_w if pop.adaptive_distance_w is not None else np.nan)
    arrs['n_pops'] = np.int64(len(s.populations))
    save('ma2_adaptive_distance_smc', **arrs)

    # --- Gaussian model forward pass + SMC
    g = gauss.get_model(n_obs=50, seed_obs=3)
    gen = g.generate(500, ['mu', 'sigma', 'gauss', 'ss_mean', 'ss_var', 'd'], seed=5)
    save('gauss_generate', observed_gauss=np.asarray(g.observed['gauss']),
         obs_ss_mean=np.asarray(g['ss_mean'].observed), obs_ss_var=np.asarray(g['ss_var'].observed),
         **{k: np.asarray(v) for k, v in gen.items()})
    s = elfi.SMC(g['d'], batch_size=1000, seed=9).sample(300, quantiles=[.3, .3, .3], bar=False)
    arrs = sample_arrays(s)
    for i, pop in enumerate(s.populations):
        arrs.update(sample_arrays(pop, 'pop{}_'.format(i)))
        arrs['pop{}_cov'.format(i)] = np.asarray(pop.cov)
    arrs['n_pops'] = np.int64(len(s.populations))
    save('gauss_smc_quantiles', **arrs)

    # --- utilities: known-answer vectors (tests/unit/test_utils.py:64-121 in the reference)
    rs = np.random.RandomState(42)
    x = rs.randn(5000)
    w = rs.rand(5000)
    qs = np.array([0.0, 0.01, 0.25, 0.5, 0.9, 1.0])
    save('weighted_quantile', x=x, w=w, alphas=qs,
         q_w=np.array([weighted_sample_quantile(x, a, w) for a in qs]),
         q_unw=np.array([weighted_sample_quantile(x, a) for a in qs]))
    x2 = rs.randn(4000, 3) * np.array([1., 5., .1]) + np.array([0., 3., -2.])
    w2 = rs.rand(4000)
    save('weighted_var', x=x2, w=w2, var_w=weighted_var(x2, w2), var_unw=weighted_var(x2))

    means = rs.randn(300, 2) * .5
    wts = rs.rand(300)
    cov = np.diag([0.3, 0.05])
    pts = rs.randn(400, 2)
    save('gm_logpdf', means=means, weights=wts, cov=cov, x=pts,
         logpdf=GMDistribution.logpdf(pts, means, cov, wts),
         pdf=GMDistribution.pdf(pts, means, cov, wts))
    cov_full = np.array([[0.3, 0.1], [0.1, 0.2]])
    save('gm_logpdf_fullcov', means=means, weights=wts, cov=cov_full, x=pts,
         logpdf=GMDistribution.logpdf(pts, means, cov_full, wts))

    # ModelPrior.logpdf on MA2 (extensions.py:180-211)
    prior = ModelPrior(m)
    theta = np.column_stack([rs.uniform(-2.5, 2.5, 500), rs.uniform(-1.5, 1.5, 500)])
    with np.errstate(divide='ignore'):
        lp = prior.logpdf(theta)
    save('ma2_prior_logpdf', theta=theta, logpdf=lp)
    gprior = ModelPrior(g)
    theta = np.column_stack([rs.uniform(-3, 11, 500), rs.uniform(-1, 12, 500)])
    with np.errstate(divide='ignore'):
        lp = gprior.logpdf(theta)
    save('gauss_prior_logpdf', theta=theta, logpdf=lp)


    # --- deterministic topological order (elfi/executor.py:162-246) on random DAGs
    import networkx as nx
    from elfi.executor import nx_constant_topological_sort
    cases = []
    rs2 = np.random.RandomState(5)
    names = ['a', 'B', '_c', 'd1', 'd10', 'd2', 'E', '_f_observed', 'g', 'h', '_i', 'J', 'k', 'l0']
    for trial in range(12):
        n = rs2.randint(4, len(names) + 1)
        nodes = list(rs2.permutation(names)[:n])
        edges = [(nodes[i], nodes[j]) for i in range(n) for j in range(i + 1, n)
                 if rs2.rand() < 0.3]
        G = nx.DiGraph()
        G.add_nodes_from(nodes)
        G.add_edges_from(edges)
        cases.append({'nodes': [str(x) for x in nodes], 'edges': [[str(a), str(b)] for a, b in edges],
                      'order': [str(x) for x in nx_constant_topological_sort(G)]})
    mc = elfi.get_client().compile(m.source_net, ['d'])
    named = {n: ('c%d' % i if n.startswith('_t') else n) for i, n in enumerate(sorted(mc.nodes()))}
    cases.append({'nodes': [named[n] for n in mc.nodes()],
                  'edges': [[named[a], named[b]] for a, b in mc.edges()],
                  'order': None})
    H = nx.DiGraph()
    H.add_nodes_from(cases[-1]['nodes'])
    H.add_edges_from(cases[-1]['edges'])
    cases[-1]['order'] = [str(x) for x in nx_constant_topological_sort(H)]
    with open(os.path.join(HERE, 'topo_orders.json'), 'w') as f:
        json.dump(cases, f)

    # --- GMDistribution.rvs host RNG stream (elfi/methods/utils.py:200-261)
    gm_means = rs.randn(50, 2) * 0.3 + [0.5, 0.1]
    gm_w = rs.rand(50)
    gm_cov = np.array([[0.02, 0.004], [0.004, 0.01]])
    gm_cov_wide = np.array([[1.5, 0.0], [0.0, 0.8]])
    draws = GMDistribution.rvs(gm_means, gm_cov, gm_w, size=333, random_state=np.random.RandomState(7))
    draws2 = GMDistribution.rvs(gm_means, gm_cov_wide, gm_w, size=333, prior_logpdf=prior.logpdf,
                                random_state=np.random.RandomState(8))
    save('gm_rvs', means=gm_means, weights=gm_w, cov=gm_cov, cov_wide=gm_cov_wide, size=np.int64(333),
         draws=draws, draws_with_prior=draws2)



    # --- AdaptiveThresholdSMC on MA2 (samplers.py:662-840)
    ats = elfi.AdaptiveThresholdSMC(m['d'], batch_size=500, seed=2)
    s = ats.sample(200, max_iter=4, bar=False)
    arrs = sample_arrays(s)
    for i, pop in enumerate(s.populations):
        arrs.update(sample_arrays(pop, 'pop{}_'.format(i)))
        arrs['pop{}_cov'.format(i)] = np.asarray(pop.cov)
    arrs['n_pops'] = np.int64(len(s.populations))
    arrs['quantiles'] = np.array([np.nan if q is None else q for q in ats._quantiles], dtype=float)
    save('ma2_adaptive_threshold_smc', **arrs)


    # --- g-and-k: stock model forward pass + the 2-d order-statistic / AdaptiveDistance variant
    from elfi.examples import gnk
    gk = gnk.get_model(n_obs=50, seed=7)
    gen = gk.generate(300, ['A', 'B', 'g', 'k', 'GNK', 'd'], seed=3)
    save('gnk_generate', observed_GNK=np.asarray(gk.observed['GNK']),
         **{k: np.asarray(v) for k, v in gen.items()})
    gk2 = gnk.get_model(n_obs=64, seed=7)
    elfi.Summary(lambda y: np.sort(y[:, :, 0], axis=1), gk2['GNK'], name='ss_sorted')
    gk2['d'].become(elfi.AdaptiveDistance(gk2['ss_sorted']))
    s = elfi.AdaptiveDistanceSMC(gk2['d'], batch_size=400, seed=13).sample(100, rounds=2,
                                                                           quantile=0.5, bar=False)
    arrs = sample_arrays(s)
    for i, pop in enumerate(s.populations):
        arrs.update(sample_arrays(pop, 'pop{}_'.format(i)))
        arrs['pop{}_w'.format(i)] = np.asarray(
            pop.adaptive_distance_w if pop.adaptive_distance_w is not None else np.nan)
    arrs['n_pops'] = np.int64(len(s.populations))
    save('gnk_adaptive_distance_smc', **arrs)

    # --- KLIEP (elfi/methods/density_ratio_estimation.py) at a size the Python loops can do
    from elfi.methods.density_ratio_estimation import DensityRatioEstimation
    kx = rs.randn(400, 2) * 0.5
    ky = rs.randn(500, 2) * 0.8 + 0.1
    kwx = rs.rand(400) + 0.5
    kwy = rs.rand(500) + 0.5
    dre = DensityRatioEstimation(n=100, epsilon=0.001, max_iter=200, abs_tol=0.01, fold=5,
                                 optimize=False)
    dre.fit(x=kx, y=ky, weights_x=kwx, weights_y=kwy, sigma=0.7)
    ratios = dre.w(kx)
    save('kliep', x=kx, y=ky, wx=kwx, wy=kwy, sigma=np.float64(0.7), ratios=ratios,
         max_ratio=np.float64(dre.max_ratio()))

    with open(os.path.join(HERE, 'meta.json'), 'w') as f:
        json.dump(meta, f, indent=1)
    print(meta)


if __name__ == '__main__':
    main()
