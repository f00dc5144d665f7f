"""Golden fixtures for BSL, from the UNMODIFIED reference (elfi-dev/elfi).

    ELFI_REFERENCE=<checkout of elfi-dev/elfi> python tests/golden/gen_golden_bsl.py

bsl.npz holds
* lik_*      -- gaussian_syn_likelihood / gaussian_syn_likelihood_ghurye_olkin on seeded inputs
                (d = 1, 2, 7, 50; whitening; Warton penalties; a singular n < d group).  The NaN
                group's value is what BSL does with it (bsl.py:242-243: -inf without calling the
                likelihood), not a likelihood call;
* chain_*    -- elfi.BSL on ma2.get_model(n_obs=50, true_params=[.6, .2], seed_obs=4), seed 123:
                samples_all, logposterior, acc_rate, n_sim;
* pre_*      -- log_SL_stdev, select_penalty(shrinkage='warton') and estimate_whitening_matrix.
"""
import os
import sys
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, os.path.join(ROOT, 'oracle'))
sys.path.insert(0, os.path.join(ROOT, 'tests'))

from ref_shim import import_reference  # noqa: E402

elfi = import_reference()
if not hasattr(np, 'NINF'):
    np.NINF = -np.inf          # NumPy 2 dropped the alias that bsl.py and select_penalty use
from elfi.examples import ma2  # noqa: E402
from elfi.methods.bsl import pdf_methods as pdf  # noqa: E402
from elfi.methods.bsl import pre_sample_methods as pre  # noqa: E402

import bsl_cases as spec  # noqa: E402

out = {}

# ----------------------------------------------------------------------------- likelihood values
for case in spec.LIK_CASES:
    name, ssx, ssy = case['name'], case['ssx'], case['ssy']
    out['lik_{}_ssx'.format(case['data'])] = ssx     # shared by the cases of one data set
    out['lik_{}_ssy'.format(case['data'])] = ssy
    if case.get('nan'):
        out['lik_{}_gauss'.format(name)] = np.array([-np.inf])
        continue
    kw = {}
    if case.get('whitening') is not None:
        kw['whitening'] = case['whitening']
        out['lik_{}_wh'.format(name)] = case['whitening']
    pens = case.get('penalties')
    if pens is None:
        out['lik_{}_gauss'.format(name)] = pdf.gaussian_syn_likelihood(ssx, ssy, **kw)
    else:
        out['lik_{}_pen'.format(name)] = np.asarray(pens)
        out['lik_{}_gauss'.format(name)] = np.concatenate([
            pdf.gaussian_syn_likelihood(ssx, ssy, shrinkage='warton', penalty=p, **kw) for p in pens])
    if case.get('go'):
        out['lik_{}_go'.format(name)] = pdf.gaussian_syn_likelihood_ghurye_olkin(ssx, ssy)

# ---------------------------------------------------------------------------------------- chains
W = pre.estimate_whitening_matrix(spec.ma2_model(ma2), spec.WH_N, spec.THETA, ['MA2'],
                                  seed=spec.WH_SEED)
out['pre_whitening'] = W

likelihoods = {
    'standard': lambda: None,
    'unbiased': pdf.unbiased_likelihood,
    'wwarton': lambda: pdf.standard_likelihood(shrinkage='warton', penalty=spec.WARTON_PENALTY,
                                               whitening=W),
    'summaries': lambda: None,
    'params0none': lambda: None,
}
for name, cfg in spec.CHAINS.items():
    m = spec.ma2_model(ma2)
    bsl = elfi.BSL(m, cfg['n_sim_round'], cfg['features'], likelihood=likelihoods[name](),
                   batch_size=cfg.get('batch_size'), seed=spec.SEED)
    res = bsl.sample(cfg['n_samples'], sigma_proposals=spec.SIGMA, params0=cfg.get('params0'),
                     burn_in=cfg.get('burn_in', 0),
                     logit_transform_bound=cfg.get('logit_transform_bound'))
    out['chain_{}_samples_all'.format(name)] = np.column_stack(
        [res.samples_all[p] for p in m.parameter_names])
    out['chain_{}_logposterior'.format(name)] = bsl.state['logposterior']
    out['chain_{}_acc_rate'.format(name)] = np.array(res.acc_rate)
    out['chain_{}_n_sim'.format(name)] = np.array(res.n_sim)
    print(name, 'acc_rate', res.acc_rate, 'n_sim', res.n_sim)

# ---------------------------------------------------------------------------- pre-sampling tools
out['pre_log_sl_stdev'] = pre.log_SL_stdev(spec.ma2_model(ma2), spec.THETA, spec.PRE_N_SIM, ['MA2'],
                                           M=spec.PRE_M, seed=spec.PRE_SEED)
lmdas, stds = pre.select_penalty(spec.ma2_model(ma2), spec.PRE_N_SIM, spec.THETA, ['MA2'],
                                 M=spec.PRE_M, sigma=1.5, shrinkage='warton', whitening=W,
                                 seed=spec.PRE_SEED)
out['pre_select_lmdas'] = lmdas
out['pre_select_stds'] = stds

np.savez(os.path.join(HERE, 'bsl.npz'), **out)
print('wrote bsl', {k: np.shape(v) for k, v in out.items()})
