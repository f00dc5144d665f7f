#!/usr/bin/env python
"""GP grid prediction (m = 1e5 points, n = 2000, 2048 and 700 training points) and the n = 2000
fit, timed with CUDA events; the predictions are checked against a float64 NumPy evaluation on a
sub-grid."""
import ctypes
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    import torch
    from elfi_b200 import _lib, device as dev
    from elfi_b200.bo import GPyRegression
    peaks = (ctypes.c_double * 2)()
    _lib.call('elfi_b200_probe_fp64_f64', dev.context(), peaks)
    dmma = peaks[1]
    res = []
    for n in (2000, 2048, 700):
        rs = np.random.RandomState(0)
        Xe = rs.uniform([-2, -1], [2, 1], (n, 2))
        ye = np.log(0.05 + np.sum((Xe - 0.3) ** 2, axis=1)) + 0.1 * rs.randn(n)
        gp = GPyRegression(['t1', 't2'], bounds={'t1': (-2, 2), 't2': (-1, 1)})
        gp.update(Xe, ye)
        if n == 2000:      # the fit shares the GEMM kernel: it must not have become slower
            for _ in range(2):
                gp._fit()
            torch.cuda.synchronize()
            ft = []
            for _ in range(5):
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
                for _ in range(3):
                    gp._fit()
                b.record()
                torch.cuda.synchronize()
                ft.append(a.elapsed_time(b) / 3)
            print(json.dumps(dict(name='gp_fit_n2000', ms_median=float(np.median(ft)),
                                  ms_min=float(min(ft)))), flush=True)
        g1, g2 = np.meshgrid(np.linspace(-2, 2, 400), np.linspace(-1, 1, 250))
        grid_h = np.column_stack([g1.ravel(), g2.ravel()])
        grid = dev.to_device(grid_h)
        for _ in range(2):
            out = gp.predict_device(grid, noiseless=True, beta=20.0)
        torch.cuda.synchronize()
        ts = []
        for _ in range(5):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(3):
                out = gp.predict_device(grid, noiseless=True, beta=20.0)
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b) / 3)
        ms = float(np.median(ts))
        m = grid.shape[0]
        flops = (m * n * n / 2 + m * n) * 2.0
        mean, var = out[0].cpu().numpy(), out[1].cpu().numpy()
        # float64 host evaluation of 500 grid points with the GP's own hyper-parameters
        h = gp.hyperparameters
        sub = np.linspace(0, m - 1, 500).astype(int)

        def k(A, B):
            d2 = ((A[:, None, :] - B[None, :, :]) ** 2).sum(-1)
            return h['kernel_var'] * np.exp(-0.5 * d2 / h['lengthscale'] ** 2) + h['bias_var']
        Ky = k(Xe, Xe) + (h['noise_var'] + 1e-8) * np.eye(n)
        Ks = k(grid_h[sub], Xe)
        sol = np.linalg.solve(Ky, np.column_stack([ye, Ks.T]))
        mean_h = Ks @ sol[:, 0]
        var_h = h['kernel_var'] + h['bias_var'] - np.einsum('ij,ji->i', Ks, sol[:, 1:])
        res.append(dict(name='gp_predict_lcbsc_m1e5_n{}'.format(n), ms_median=ms,
                        ms_min=float(min(ts)), TFLOPs=flops / ms / 1e9,
                        frac_dmma_peak=flops / ms / 1e9 / dmma, dmma_peak_tflops=dmma,
                        max_rel_err_mean=float(np.max(np.abs(mean[sub] - mean_h) /
                                                      (np.abs(mean_h) + 1e-12))),
                        max_abs_err_var=float(np.max(np.abs(var[sub] - var_h)))))
        print(json.dumps(res[-1]), flush=True)


if __name__ == '__main__':
    main()
