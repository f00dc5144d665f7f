#!/usr/bin/env python
"""mean/var timings for contiguous rows (n = 2 mod 4 takes the 1-D bulk row-group kernel, the
other widths the 2-D tensor-map row-stream path), checked bit for bit against NumPy.
--once: a single launch (for ncu)."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main(once):
    import numpy as np
    import torch
    from elfi_b200 import ops
    hbm = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))['hbm_gbs'] \
        if os.path.exists(os.path.join(ROOT, 'MEASURED_PEAKS.json')) else 6650.0
    gen = torch.Generator(device='cuda').manual_seed(0)
    shapes = [(1_000_000, 50)] if once else [(1_000_000, 50), (2_000_000, 50), (1_000_000, 62),
                                             (1_000_000, 34), (1_000_000, 18), (1_000_000, 64)]
    for B, n in shapes:
        y = torch.randn(B, n, dtype=torch.float64, device='cuda', generator=gen)
        if once:
            ops.meanvar(y)
            torch.cuda.synchronize()
            return
        for _ in range(3):
            ops.meanvar(y)
        torch.cuda.synchronize()
        ts = []
        for _ in range(7):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(10):
                ops.meanvar(y)
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b) / 10)
        ms = float(np.median(ts))
        nbytes = B * n * 8 + B * 16
        ref = y[:4096].cpu().numpy()
        got = ops.meanvar(y[:4096].contiguous()).cpu().numpy()
        exact = bool(np.array_equal(got[:, 0], ref.mean(axis=1)) and
                     np.array_equal(got[:, 1], ref.var(axis=1)))
        print(json.dumps(dict(name='meanvar_{}x{}'.format(B, n), ms_median=ms,
                              ms_min=float(min(ts)), GBps=nbytes / ms / 1e6,
                              frac_hbm_measured=nbytes / ms / 1e6 / hbm, bit_exact=exact)),
              flush=True)
        del y


if __name__ == '__main__':
    main('--once' in sys.argv)
