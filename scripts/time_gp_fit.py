#!/usr/bin/env python
"""CUDA-event time of one GP fit at n = $N training points (default 2000)."""
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from elfi_b200.bo import GPyRegression  # noqa: E402

n = int(os.environ.get('N', 2000))
rs = np.random.RandomState(0)
X = rs.uniform([-2, -1], [2, 1], (n, 2))
y = np.log(0.05 + np.sum((X - 0.3) ** 2, axis=1)) + 0.1 * rs.randn(n)
gp = GPyRegression(['t1', 't2'], bounds={'t1': (-2, 2), 't2': (-1, 1)}, incremental=False)
gp.update(X, y)
ts = []
for _ in range(12):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    gp._fit()
    b.record()
    torch.cuda.synchronize()
    ts.append(a.elapsed_time(b))
print(os.environ.get('TAG', ''), 'fit ms median %.3f min %.3f' % (np.median(ts[2:]), np.min(ts[2:])))
