#!/usr/bin/env python
"""Lab: time K1 (tensor-core Gram) alone for arbitrary (cells, keypoints) to separate per-CTA and
per-step costs:  python tools/gram_scan.py cells:n_kp [cells:n_kp ...]"""
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from cvx_proj_b200 import _runtime as rt, synth  # noqa: E402
from cvx_proj_b200.apap import APAP, scale_anchors, weight_scale  # noqa: E402

torch.cuda.set_device(0)
dev = torch.device("cuda", 0)
lib = rt.load_library()
flush = torch.zeros(256 << 20, dtype=torch.uint8, device=dev)
for spec in sys.argv[1:]:
    cells, n_kp = (int(v) for v in spec.split(":"))
    src, dst, _ = synth.make_keypoints(3840, 2160, n_kp, seed=0)
    st = APAP(0.5, 100, [4448, 2332], [0, 0], device=dev)  # tcgen05 engine
    table, tmats = st._prepare(src, dst)
    rng = np.random.default_rng(1)
    verts = rng.uniform([0, 0], [4448, 2332], size=(cells, 1, 2))
    n_pad = table.shape[0]
    t_dev = st.kp_table_device(torch.from_numpy(table[None]).to(dev))[0]
    a_dev = torch.from_numpy(scale_anchors(verts, weight_scale(100))).to(dev)
    ks, cp, nbytes = rt.gram_plan(cells, n_pad, rt.GRAM_TCGEN05)
    partials = torch.empty(nbytes // 4, dtype=torch.float32, device=dev)
    s = rt.stream_ptr(torch, dev)
    ts = []
    for k in range(13):
        flush.add_(1)
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        rt.check(lib.apap_gram_partials(t_dev.data_ptr(), a_dev.data_ptr(), 1, cells, n_pad, 0.25, rt.GRAM_TCGEN05,
                                        None, partials.data_ptr(), s), "gram")
        e1.record(); e1.synchronize()
        if k >= 3:
            ts.append(e0.elapsed_time(e1) * 1e3)
    ctas = ((cells + 127) // 128) * ks
    print(f"cells={cells:7d} n_kp={n_kp:6d} splits={ks:3d} ctas={ctas:6d} ({ctas / 592:6.2f} waves)  "
          f"{np.median(ts):8.1f} us (min {np.min(ts):8.1f})  {2.0 * cells * n_pad / np.median(ts) / 1e6:6.2f} T MUFU/s", flush=True)
