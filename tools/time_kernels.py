#!/usr/bin/env python
"""Quick device timing of the pass's kernels (CUDA events, L2 flushed before every launch):
python tools/time_kernels.py [workload] [iters] [what]
what = comma list of gram,eig,warp,fused,blend (default all).  Also checks the H grid against the
one the first run on this machine saved (max normalised error), so a change that breaks the
numbers shows up next to its time."""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402

name = sys.argv[1] if len(sys.argv) > 1 else "c2"
iters = int(sys.argv[2]) if len(sys.argv) > 2 else 10
what = (sys.argv[3] if len(sys.argv) > 3 else "gram,eig,warp,fused,blend").split(",")
torch.cuda.set_device(0)
dev = torch.device("cuda", 0)
p = bench.Pass(torch, dev, name)
flush = torch.zeros(256 << 20, dtype=torch.uint8, device=dev)
p.gram(); p.eig()
if any(w in what for w in ("warp", "fused", "blend")):
    p.prepare_warp()
def _gwarp_setup():
    from cvx_proj_b200 import utils as putils, synth as _synth
    sc = p.sc
    img = torch.from_numpy(sc.image(1)).to(dev)
    base = torch.from_numpy(_synth.make_image(sc.width, sc.height, seed=2)).to(dev)
    cw, ch, tx, ty, m = putils.warping_canvas(img.shape, img.shape, sc.h_gt)
    out = torch.empty((ch, cw, 3), dtype=torch.uint8, device=dev)
    return lambda mode: putils.warp_perspective(img, m, (cw, ch), base=base, offset=(tx, ty), mode=mode, out=out)


_gw = _gwarp_setup() if any(w.startswith("gwarp") for w in what) else None
ops = {"gwarp": lambda: _gw(0), "gwarp_paste": lambda: _gw(1), "gwarp_mean": lambda: _gw(2), "gram": p.gram, "eig": p.eig, "dlt": p.dlt, "warp": lambda: p.warp(False), "fused": lambda: p.warp(True), "blend": p.blend}
res = {}
for w in what:
    ts = []
    for k in range(iters + 3):
        if not os.environ.get('NOFLUSH'):
            flush.add_(1)
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); ops[w](); e1.record(); e1.synchronize()
        if k >= 3:
            ts.append(e0.elapsed_time(e1) * 1e3)
    res[w] = (float(np.median(ts)), float(np.min(ts)))
h = p.h_out.cpu().numpy().astype(np.float64)
ref_path = f"/tmp/h_ref_{name}.npy"
err = ""
if os.path.exists(ref_path):
    ref = np.load(ref_path)
    L = float(max(p.sc.width, p.sc.height))
    s = np.array([1 / L, 1 / L, 1.0])
    d = (h - ref).reshape(-1, 3, 3) * s[None, :, None] / s[None, None, :]
    r = ref.reshape(-1, 3, 3) * s[None, :, None] / s[None, None, :]
    err = f" | H vs first run: {np.abs(d).max(axis=(1, 2)).max() / 1.0:.2e} (norm by max|ref| per cell: {(np.abs(d).max(axis=(1, 2)) / np.abs(r).max(axis=(1, 2))).max():.2e})"
else:
    np.save(ref_path, h)
print(f"{name} " + " ".join(f"{w}={m:7.1f}us(min {mn:6.1f})" for w, (m, mn) in res.items()) + err, flush=True)
