"""Times elfi_b200_synlik_f64 and BSL chains on the GPU; prints one JSON line.

    python scripts/time_bsl.py [--out profiles/bsl_time.json] [--iters 2000]

1. Kernel time (CUDA events, after warm-up) at (P, n, d, L) = (1, 500, 50, 1), (1024, 500, 50, 1),
   (4096, 100, 2, 1), (10, 100, 50, 31), (256, 1000, 128, 1), each against its two bounds: HBM
   bytes P n d 8 at 7.7 TB/s and FMAs P n d (d + 1) / 2 + P L d^3 / 6 at the DMMA rate measured by
   elfi_b200_probe_fp64_f64.  The outputs are checked against the NumPy restatement.  The larger
   inputs exceed the 126 MB L2 only at (1024, 500, 50) (205 MB); the others are re-read from L2.
2. BSL wall clock for `--iters` iterations on MA2 (n_obs 50, features ['MA2'], n_sim_round 500):
   the parity model (host simulator), the device model, and the reference when oracle/_ref holds a
   copy of it ("not run" otherwise).
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))
sys.path.insert(0, os.path.join(ROOT, 'oracle'))

SIZES = [(1, 500, 50, 1), (1024, 500, 50, 1), (4096, 100, 2, 1), (10, 100, 50, 31),
         (256, 1000, 128, 1)]
HBM_TBPS = 7.7


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm',
                            '--format=csv,noheader'], capture_output=True, text=True, timeout=30)
        return q.stdout.strip().splitlines()[0]
    except Exception as e:   # noqa: BLE001
        return 'unknown ({})'.format(e)


def time_kernel(dmma_tflops, reps=50):
    import torch
    import bsl_cases as cases
    from elfi_b200 import ops
    rows = []
    for P, n, d, L in SIZES:
        rs = np.random.RandomState(P + n + d)
        host = rs.randn(P * n, d) @ (np.eye(d) + 0.1 * rs.randn(d, d) / np.sqrt(d)).T
        obs = host[:n].mean(0) + 0.3 * rs.randn(d)
        S = torch.from_numpy(host).cuda()
        gam = None if L == 1 else np.linspace(0.1, 1.0, L)
        for _ in range(3):
            out = ops.synlik(S, obs, n, gammas=gam)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            ops.synlik(S, obs, n, gammas=gam)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        got = out.cpu().numpy()
        want = cases.synlik_reference(host, obs, n, gammas=gam)
        err = float(np.max(np.abs(got - want) / np.maximum(1, np.abs(want))))
        nbytes = P * n * d * 8
        fmas = P * n * d * (d + 1) / 2 + P * L * d ** 3 / 6
        t_hbm = nbytes / (HBM_TBPS * 1e12) * 1e3
        t_dmma = 2 * fmas / (dmma_tflops * 1e12) * 1e3
        rows.append(dict(P=P, n=n, d=d, L=L, ms=round(ms, 5), bytes=nbytes, fmas=fmas,
                         hbm_bound_ms=t_hbm, dmma_bound_ms=t_dmma,
                         bound='hbm' if t_hbm > t_dmma else 'dmma',
                         frac_of_bound=round(max(t_hbm, t_dmma) / ms, 4), max_rel_err=err))
    return rows


def time_chain(model_fn, iters):
    import torch
    import elfi_b200 as elfi
    m = model_fn()
    bsl = elfi.BSL(m, 500, ['MA2'], seed=123)
    t0 = time.perf_counter()
    res = bsl.sample(iters, sigma_proposals=np.array([[0.02, 0.01], [0.01, 0.02]]),
                     params0=np.array([0.6, 0.2]))
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    return dict(seconds=round(dt, 3), us_per_iter=round(dt / iters * 1e6, 1),
                acc_rate=res.acc_rate, mean=[float(np.mean(res.samples[p])) for p in ('t1', 't2')])


def time_reference(iters):
    import ref_shim
    if not ref_shim.reference_available():
        return 'not run'
    elfi = ref_shim.import_reference()
    if not hasattr(np, 'NINF'):
        np.NINF = -np.inf
    from elfi.examples import ma2
    m = ma2.get_model(n_obs=50, true_params=[.6, .2], seed_obs=4)
    bsl = elfi.BSL(m, 500, ['MA2'], seed=123)
    t0 = time.perf_counter()
    res = bsl.sample(iters, sigma_proposals=np.array([[0.02, 0.01], [0.01, 0.02]]),
                     params0=np.array([0.6, 0.2]), bar=False)
    dt = time.perf_counter() - t0
    return dict(seconds=round(dt, 3), us_per_iter=round(dt / iters * 1e6, 1),
                acc_rate=res.acc_rate)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None)
    ap.add_argument('--iters', type=int, default=2000)
    args = ap.parse_args()
    import ctypes
    import torch
    if not torch.cuda.is_available():
        raise SystemExit('time_bsl.py measures on a GPU; none found')
    from elfi_b200 import _lib
    from elfi_b200 import device as dev
    from elfi_b200.examples import ma2
    peaks = (ctypes.c_double * 2)()
    _lib.call('elfi_b200_probe_fp64_f64', dev.context(), peaks)
    result = dict(card=card(), dfma_tflops=peaks[0], dmma_tflops=peaks[1])
    result['kernel'] = time_kernel(peaks[1])
    mk = lambda f: (lambda: f(n_obs=50, true_params=[.6, .2], seed_obs=4))  # noqa: E731
    time_chain(mk(ma2.get_device_model), 20)    # warm-up: module load, first allocations
    result['chain_parity_model'] = time_chain(mk(ma2.get_model), args.iters)
    result['chain_device_model'] = time_chain(mk(ma2.get_device_model), args.iters)
    result['chain_reference_host'] = time_reference(args.iters)
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(line + '\n')


if __name__ == '__main__':
    main()
