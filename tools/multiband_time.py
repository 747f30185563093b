#!/usr/bin/env python
"""Cost of the multi-band blend (utils.multiband_blend, stitch_panorama(blend="multiband")).  One run prints:
  - the card's name, power limit and top SM clock (queries only);
  - on the layer sets of timing.LAYER_SETS (the c4-size case, centre + 16; the c2-size case, centre + 4; 64
    synthetic 1920 x 1080 layers), each call preceded by a 256 MiB write that flushes L2:
      apap_multiband_blend at 5 bands, without and with gains, by CUDA events (median), against its floor: the layer
      bytes in the canvas read once plus the canvas written, at 7.7 TB/s;
      per kernel (all k_mb_down launches of a call, all k_mb_band launches), by torch.profiler in a run of its own;
      cv.detail_MultiBandBlender(0, 5, CV_16S) on the host cores, fed as the contract says (sets of at most 20 layers);
      every output checked against oracle.multiband_oracle (the oracle's layers spread over host processes);
  - end to end on the c4 and c2 cases: stitch_panorama(blend="multiband") against "feather" and "mean".

    python tools/multiband_time.py [--reps 30] [--out FILE]
"""
import argparse
import ctypes
import json
import multiprocessing as mp
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import cv2 as cv  # noqa: E402
import numpy as np  # noqa: E402
import torch  # noqa: E402

from cvx_proj_b200 import _runtime as rt  # noqa: E402
from cvx_proj_b200 import synth  # noqa: E402
from cvx_proj_b200.driver import stitch_panorama  # noqa: E402
from cvx_proj_b200.utils import _gain_table, _layer_descs, exposure_gains, multiband_blend  # noqa: E402
from oracle import feather_oracle as fo  # noqa: E402
from oracle import multiband_oracle as mo  # noqa: E402
from timing import (HBM_TBS, LAYER_SETS, card, clipped_px, event_us, host_ms, kernel_times, l2_flush,  # noqa: E402
                    name_in, say, write_out)

BANDS = 5
KERNELS = ("k_mb_down", "k_mb_band")


def calls(lib, dev, layers, origins, size, gains):
    width, height = size
    n = len(layers)
    _, desc = _layer_descs(torch, dev, layers, origins, True)     # packed device layers: described in place
    ptr = desc.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong))
    ws_bytes = ctypes.c_size_t()
    rt.check(lib.apap_multiband_workspace_bytes(ptr, n, height, width, BANDS, ctypes.byref(ws_bytes)), "ws bytes")
    ws = torch.empty(max(ws_bytes.value, 16), dtype=torch.uint8, device=dev)
    lut = torch.from_numpy(_gain_table("multiband_time", gains, n)).to(dev)
    outs = {k: torch.empty((height, width, 3), dtype=torch.uint8, device=dev) for k in ("plain", "gain")}
    st = rt.stream_ptr(torch, dev)
    fns = {
        "plain": lambda: rt.check(lib.apap_multiband_blend(ptr, n, height, width, BANDS, ws.data_ptr(), ws.numel(),
                                                           outs["plain"].data_ptr(), outs["plain"].numel(), st),
                                  "multiband"),
        "gain": lambda: rt.check(lib.apap_multiband_blend_gain(ptr, n, height, width, BANDS, lut.data_ptr(),
                                                               ws.data_ptr(), ws.numel(), outs["gain"].data_ptr(),
                                                               outs["gain"].numel(), st), "multiband gain"),
    }
    return fns, outs, ws_bytes.value


def kernel_us(fn, reps, flush):
    """Per call, the summed device time of every launch of each kernel in KERNELS (mean over ``reps`` calls)."""
    fn()
    torch.cuda.synchronize()
    times = kernel_times([fn], name_in(KERNELS), reps, flush)
    return {k: float(np.sum(times[k])) / reps for k in KERNELS if k in times}


def _accumulate(args):
    layers, origins, size, gains = args
    return mo.accumulate(layers, origins, size, BANDS, gains)


def oracle(layers_np, origins, size, gains, procs):
    """mo.multiband_blend, with the layers' sums computed in ``procs`` host processes."""
    chunks = [list(range(i, len(layers_np), procs)) for i in range(min(procs, len(layers_np)))]
    jobs = [([layers_np[i] for i in c], [origins[i] for i in c], size,
             None if gains is None else [gains[i] for i in c]) for c in chunks]
    with mp.get_context("fork").Pool(len(jobs)) as pool:
        band, wsum = None, None
        for b, w in pool.imap_unordered(_accumulate, jobs):
            if band is None:
                band, wsum = b, w
            else:
                for i in range(len(band)):
                    band[i] += b[i]
                    wsum[i] += w[i]
    return mo.finish(band, wsum, size)


def opencv_ms(layers_np, origins, size, reps):
    def run():
        b = cv.detail_MultiBandBlender(0, BANDS, cv.CV_16S)
        b.prepare((0, 0, size[0], size[1]))
        for img, o in zip(layers_np, origins):
            p = fo.paste(img, o, size)
            b.feed(p.astype(np.int16), np.where(p.max(axis=-1) > 0, 255, 0).astype(np.uint8), (0, 0))
        return np.clip(b.blend(None, None)[0], 0, 255).astype(np.uint8)
    got = run()
    return host_ms(run, reps)[0], got


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--procs", type=int, default=8, help="host processes for the oracle check")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    _, dev = rt.torch_cuda()
    lib = rt.load_library()
    res = {**card(dev), "sets": [], "e2e": []}
    say(f"cv2 {cv.__version__}, {os.cpu_count()} host cores, bands {BANDS}")
    flush = l2_flush(dev)
    say(f"== every call after a 256 MiB L2-flushing write; CUDA events over {args.reps} calls (median); per kernel: "
        f"torch.profiler, summed over a call's launches; floor: 3 B per layer pixel in the canvas + 3 B per canvas "
        f"pixel at {HBM_TBS} TB/s")
    for name, make in LAYER_SETS:
        layers, origins, size = make(dev)
        px = clipped_px(layers, origins, size)
        g = exposure_gains(layers, origins, size)
        fns, outs, ws_bytes = calls(lib, dev, layers, origins, size, g)
        us = {k: event_us(fn, args.reps, flush) for k, fn in fns.items()}
        per = {k: kernel_us(fn, args.reps, flush) for k, fn in fns.items()}
        torch.cuda.synchronize()
        t_call = host_ms(lambda: (multiband_blend(layers, origins, size, BANDS), torch.cuda.synchronize()), 5)[0]
        for fn in fns.values():
            fn()
        got = {k: v.cpu().numpy() for k, v in outs.items()}
        layers_np = [t.cpu().numpy() for t in layers]
        ok = {k: bool(np.array_equal(got[k], oracle(layers_np, origins, size, None if k == "plain" else g, args.procs)))
              for k in got}
        if len(layers) <= 20:
            cv_ms, cv_out = opencv_ms(layers_np, origins, size, 3)
            ok_cv = bool(np.array_equal(cv_out, got["plain"]))
        else:   # not measured: the host blender builds every layer's pyramid over the whole 41.6 Mpix canvas
            cv_ms, ok_cv = float("nan"), None
        floor_us = 3 * (px + size[0] * size[1]) / (HBM_TBS * 1e12) * 1e6
        say(f"{name}: {len(layers)} layers, canvas {size[0]} x {size[1]}, {px / 1e6:.1f} Mpix of layers in the canvas, "
            f"nb {mo.num_bands(BANDS, *size)}, workspace {ws_bytes / 2**20:.0f} MiB")
        for k in ("plain", "gain"):
            kern = ", ".join(f"{n_} {v:.1f} us" for n_, v in per[k].items())
            say(f"  apap_multiband_blend{'_gain' if k == 'gain' else ''} {us[k][0]:.1f} us (min {us[k][1]:.1f}); "
                f"{kern}; floor {floor_us:.1f} us = {100 * floor_us / us[k][0]:.1f} % of the floor")
        cv_txt = f"{cv_ms:.1f} ms" if cv_ms == cv_ms else "not measured"
        say(f"  multiband_blend call on device tensors (host clock, to a synchronise) {t_call:.2f} ms; "
            f"OpenCV CV_16S blender on the host {cv_txt}")
        say(f"  equal: plain = oracle {ok['plain']}, with gains = oracle {ok['gain']}, plain = OpenCV "
            + ("not measured" if ok_cv is None else str(ok_cv)))
        res["sets"].append({"set": name, "layers": len(layers), "canvas": list(size), "layer_px": px,
                            "workspace_bytes": ws_bytes, "call_us": {k: v[0] for k, v in us.items()},
                            "kernel_us": per, "floor_us": floor_us, "multiband_blend_ms": t_call,
                            "opencv_ms": cv_ms, "equal_oracle": ok, "equal_opencv": ok_cv})
        del layers, fns, outs
    for name, k in (("c4", 16), ("c2", 4)):
        centre, others, raw_c, raw_os = synth.make_case(name, k)
        row = {"case": name, "k": k}
        for blend in ("mean", "feather", "multiband"):
            stitch_panorama(centre, others, raw_c, raw_os, ransac="gpu", blend=blend)
            row[f"{blend}_ms"] = host_ms(lambda: stitch_panorama(centre, others, raw_c, raw_os, ransac="gpu",
                                                                 blend=blend), 3)[0]
        say(f"== end to end {name}, centre + {k}, ransac='gpu' (3 reps, medians): mean {row['mean_ms']:.1f} ms, "
            f"feather {row['feather_ms']:.1f} ms, multiband {row['multiband_ms']:.1f} ms")
        res["e2e"].append(row)
    say(json.dumps(res))
    write_out(args.out)


if __name__ == "__main__":
    main()
