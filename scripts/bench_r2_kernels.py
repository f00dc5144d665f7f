#!/usr/bin/env python
"""Round-2 kernel timings (CUDA events around batches of back-to-back launches, so the per-call
Python overhead overlaps with the previous kernel; median of the batches).  One JSON line per
kernel + gpurun_out/r2_kernels[_TAG].json.  Variants selected by environment variables are
static per process: run the script once per variant (TAG names the output)."""
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from elfi_b200 import ops  # noqa: E402

HBM = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))['hbm_gbs'] \
    if os.path.exists(os.path.join(ROOT, 'MEASURED_PEAKS.json')) else 6650.0
TAG = os.environ.get('TAG', 'default')
out = []


def timeit(fn, per_batch=10, batches=7, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(batches):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(per_batch):
            fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b) / per_batch)
    return float(np.median(ts)), float(np.min(ts))


def rec(name, ms, best, nbytes, **kw):
    e = dict(name=name, tag=TAG, ms_median=ms, ms_min=best, algorithmic_GB=nbytes / 1e9,
             GBps=nbytes / (ms * 1e-3) / 1e9, frac_hbm_measured=nbytes / (ms * 1e-3) / 1e9 / HBM, **kw)
    out.append(e)
    print(json.dumps(e), flush=True)


gen = torch.Generator(device='cuda').manual_seed(0)


def randn(*shape):
    return torch.randn(*shape, dtype=torch.float64, device='cuda', generator=gen)


# headline distance kernel (must agree with bench.py's roofline.kernel_ms)
S, obs = randn(1_000_000, 128), randn(128)
ms, best = timeit(lambda: ops.dist_euclid(S, obs))
rec('dist_euclid_1e6x128', ms, best, S.numel() * 8 + S.shape[0] * 8)
del S

# K6 mean/var (Gaussian model summaries)
for B in (1_000_000, 2_000_000):
    y = randn(B, 50)
    ms, best = timeit(lambda: ops.meanvar(y))
    rec('meanvar_{}x50'.format(B), ms, best, y.numel() * 8 + B * 16)
    del y
y = randn(1_000_000, 64)
ms, best = timeit(lambda: ops.meanvar(y))
rec('meanvar_1e6x64', ms, best, y.numel() * 8 + y.shape[0] * 16)
del y

# K6 autocov, single leaf and tree
x = randn(1_000_000, 100)
ms, best = timeit(lambda: ops.autocov(x, lags=(1, 2)))
rec('autocov12_1e6x100', ms, best, x.numel() * 8 + x.shape[0] * 16)
del x
z = randn(400_000, 256)
ms, best = timeit(lambda: ops.autocov(z, lags=(1, 2)))
rec('autocov12_4e5x256', ms, best, z.numel() * 8 + z.shape[0] * 16)
ms, best = timeit(lambda: ops.meanvar(z))
rec('meanvar_4e5x256', ms, best, z.numel() * 8 + z.shape[0] * 16)
del z

# K4 nested distances (K = 5) with and without the fused column moments; K5 alone
Sg, og = randn(500_000, 256), randn(256)
W = torch.rand(5, 256, dtype=torch.float64, device='cuda', generator=gen) + 0.5
thr = np.full(5, 1e9)
nb = Sg.numel() * 8 + Sg.shape[0] * 5 * 8
ms, best = timeit(lambda: ops.dist_euclid(Sg, og, w=W, thresholds=thr, sync=False))
rec('nested_K5_5e5x256', ms, best, nb)
ms_f, best_f = timeit(lambda: ops.dist_euclid(Sg, og, w=W, thresholds=thr, sync=False, moments=True))
rec('nested_K5_plus_moments_fused_5e5x256', ms_f, best_f, nb + 2 * 256 * 8)
ms_c, best_c = timeit(lambda: ops.colmoments(Sg))
rec('colmoments_alone_5e5x256', ms_c, best_c, Sg.numel() * 8)
out.append(dict(name='fused_vs_two_passes', tag=TAG, fused_ms=ms_f, two_passes_ms=ms + ms_c,
                speedup=(ms + ms_c) / ms_f))
print(json.dumps(out[-1]), flush=True)
W1 = torch.ones(1, 256, dtype=torch.float64, device='cuda')
ms, best = timeit(lambda: ops.dist_euclid(Sg, og, w=W1, thresholds=thr[:1], sync=False, moments=True))
rec('nested_K1_plus_moments_fused_5e5x256', ms, best, Sg.numel() * 8 + Sg.shape[0] * 8)
del Sg

# sharded mixture density: one rank's share of N = 1e6 new particles against M = 1e6 components
M = 1_000_000
means = randn(M, 2) * 0.3
w = torch.rand(M, dtype=torch.float64, device='cuda', generator=gen) + 0.1
cov = np.array([[0.02, 0.004], [0.004, 0.01]])
for N in (125_000, 1_000_000):
    xs = randn(N, 2) * 0.3
    ms, best = timeit(lambda: ops.gm_logpdf(xs, means, cov, w, validate=False), per_batch=1,
                      batches=3, warm=1)
    e = dict(name='gm_logpdf_N{}_M1e6'.format(N), tag=TAG, ms_median=ms, ms_min=best,
             pairs_per_s=N * M / (ms * 1e-3), fp64_inst_per_pair=16,
             tflops_equiv=N * M * 16 / (ms * 1e-3) / 1e12)
    out.append(e)
    print(json.dumps(e), flush=True)
    if N == 125_000:
        np.save(os.path.join(ROOT, 'gpurun_out', 'gm_logq_{}.npy'.format(TAG)),
                ops.gm_logpdf(xs, means, cov, w, validate=False).cpu().numpy())

with open(os.path.join(ROOT, 'gpurun_out', 'r2_kernels_{}.json'.format(TAG)), 'w') as f:
    json.dump(out, f, indent=1)
