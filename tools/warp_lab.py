#!/usr/bin/env python
"""LAB: K3 timing, cold (L2 flushed) vs warm (source and canvas L2-resident, no launch gap): the plain warp on the
tile engine and on round 1's strip kernel, and the warp fused with the blend (strip kernel); checks both engines write
the same bytes."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import bench
name = sys.argv[1] if len(sys.argv) > 1 else "c2"
torch.cuda.set_device(0)
dev = torch.device("cuda", 0)
p = bench.Pass(torch, dev, name)
p.gram(); p.eig(); p.prepare_warp()
flush = torch.zeros(256 << 20, dtype=torch.uint8, device=dev)
def call(legacy, fused):
    p.st.warp_device(p.img, p.tables, p.sc.mesh_cells, out=p.canvas, legacy=legacy,
                     centre_dev=p.centre if fused else None)
def run(legacy, fused, warm, reps=20):
    ts = []
    for _ in range(reps + 3):
        flush.add_(1)
        if warm:
            call(legacy, fused)
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        call(legacy, fused)
        e1.record(); e1.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    ts = ts[3:]
    return sum(ts) / len(ts), min(ts)
outs = []
for legacy in (False, True):
    call(legacy, False); outs.append(p.canvas.clone())
print(f"{name} plain: engines agree = {bool(torch.equal(outs[0], outs[1]))}, "
      f"non-black {float((outs[0].amax(-1) > 0).float().mean()):.3f}")
for legacy, fused in ((False, False), (True, False), (True, True)):
    for warm in (False, True):
        avg, best = run(legacy, fused, warm)
        print(f"{name} {'fused' if fused else 'plain'} {'strip' if legacy else 'tile '} "
              f"{'warm L2' if warm else 'cold   '} avg {avg:7.2f} us  best {best:7.2f} us")
