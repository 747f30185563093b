#!/usr/bin/env python
"""LAB: device time of the exact matcher (apap_match_nn), 4000 x 4000 x 128, L2 flushed."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np, torch
from cvx_proj_b200.utils import match_descriptors
from timing import l2_flush
dev = torch.device("cuda", 0)
rng = np.random.default_rng(0)
for nq, nt in ((4000, 4000), (500, 500), (20000, 20000)):
    t = torch.from_numpy(np.rint(rng.uniform(0, 255, (nt, 128))).astype(np.float32)).to(dev)
    q = torch.from_numpy(np.rint(rng.uniform(0, 255, (nq, 128))).astype(np.float32)).to(dev)
    flush = l2_flush(dev)
    ts = []
    for k in range(10):
        flush.add_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); match_descriptors(q, t); e1.record(); e1.synchronize()
        if k >= 3: ts.append(e0.elapsed_time(e1) * 1e3)
    print(f"{nq} x {nt}: {np.median(ts):.1f} us, {3.0 * nq * nt * 128 / (np.median(ts) * 1e-6) / 1e12:.1f} TFLOP/s")
