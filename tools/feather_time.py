#!/usr/bin/env python
"""Cost of the feather blend (utils.feather_blend, stitch_panorama(blend="feather")).  One run prints:
  - the card's name, power limit and top SM clock (queries only);
  - on the layer sets of tools/panorama_time.py (the c4-size case, centre + 16; the c2-size case, centre + 4; 64
    synthetic 1920 x 1080 layers), each call preceded by a 256 MiB write that flushes L2:
      the whole apap_feather_blend call by CUDA events, and each of its kernels (k_feather_rows, k_feather_cols,
      k_feather_blend) from torch.profiler in a separate pass, with the bytes each must move over its time against
      7.7 TB/s; k_blend_layers (apap_blend_layers) on the same layers for comparison;
      cv.detail.FeatherBlender on the host cores, fed as the contract says (every layer pasted into the canvas);
      every output checked against oracle.feather_oracle (the mean blend against oracle.panorama_oracle);
  - end to end on the c4 and c2 cases: stitch_panorama(blend="feather") against blend="mean".

    python tools/feather_time.py [--reps 100] [--out FILE]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import cv2 as cv  # noqa: E402
import numpy as np  # noqa: E402
import torch  # noqa: E402

from cvx_proj_b200 import _runtime as rt  # noqa: E402
from cvx_proj_b200.driver import stitch_panorama  # noqa: E402
from oracle import feather_oracle as fo  # noqa: E402
from oracle import panorama_oracle as po  # noqa: E402
from panorama_time import HBM_TBS, case_layers, synthetic_layers  # noqa: E402
from sift_time import host_ms  # noqa: E402
from tests.test_case import _scene  # noqa: E402

SHARPNESS = 0.02
KERNELS = ("k_feather_rows", "k_feather_cols", "k_feather_blend", "k_blend_layers")


def model_bytes(layers, origins, size):
    """Bytes each kernel must move at least: rows read the layer and write 2-byte distances, cols read and write
    them, the blend reads layer and distances and writes the canvas; the mean blend reads layers, writes the canvas."""
    width, height = size
    px = 0
    for t, (x0, y0) in zip(layers, origins):
        h, w = t.shape[:2]
        px += max(0, min(x0 + w, width) - max(x0, 0)) * max(0, min(y0 + h, height) - max(y0, 0))
    canvas = 3 * width * height
    return {"k_feather_rows": 5 * px, "k_feather_cols": 4 * px, "k_feather_blend": 5 * px + canvas,
            "k_blend_layers": 3 * px + canvas, "call": 14 * px + canvas}, px


def calls(lib, dev, layers, origins, size):
    width, height = size
    desc = np.array([[t.data_ptr(), t.shape[0], t.shape[1], t.stride(0), x0, y0]
                     for t, (x0, y0) in zip(layers, origins)], dtype=np.int64)
    ptr = desc.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong))
    ws_bytes = ctypes.c_size_t()
    rt.check(lib.apap_feather_workspace_bytes(ptr, len(layers), height, width, ctypes.byref(ws_bytes)), "ws bytes")
    ws = torch.empty(ws_bytes.value, dtype=torch.uint8, device=dev)
    out_f = torch.empty((height, width, 3), dtype=torch.uint8, device=dev)
    out_m = torch.empty((height, width, 3), dtype=torch.uint8, device=dev)
    st = rt.stream_ptr(torch, dev)

    def feather():
        rt.check(lib.apap_feather_blend(ptr, len(layers), height, width, SHARPNESS, ws.data_ptr(), ws.numel(),
                                        out_f.data_ptr(), out_f.numel(), st), "apap_feather_blend")

    def mean():
        rt.check(lib.apap_blend_layers(ptr, len(layers), height, width, out_m.data_ptr(), out_m.numel(), st),
                 "apap_blend_layers")
    return feather, mean, out_f, out_m, ws_bytes.value


def event_us(fn, reps, flush):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    return float(np.median(ts)), float(np.min(ts))


def profiled_us(fns, reps, flush):
    """Median device time of every kernel named in KERNELS over ``reps`` flushed calls of each fn."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            for fn in fns:
                flush.fill_(1)
                fn()
        torch.cuda.synchronize()
    per = {k: [] for k in KERNELS}
    for ev in prof.events():
        for k in KERNELS:
            if k in ev.name and ev.device_type.name == "CUDA":
                per[k].append(ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total)
    return {k: float(np.median(v)) for k, v in per.items() if v}


def opencv_ms(layers_np, origins, size, reps):
    def run():
        blender = cv.detail.FeatherBlender(SHARPNESS)
        blender.prepare((0, 0, size[0], size[1]))
        for img, o in zip(layers_np, origins):
            p = fo.paste(img, o, size)
            blender.feed(p.astype(np.int16), np.where(p.max(axis=-1) > 0, 255, 0).astype(np.uint8), (0, 0))
        return blender.blend(None, None)[0].astype(np.uint8)
    got = run()
    return host_ms(run, reps)[0], got


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=100)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    _, dev = rt.torch_cuda()
    lib = rt.load_library()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    say(f"card: {torch.cuda.get_device_name(dev)} | nvidia-smi: {q.stdout.strip() or q.stderr.strip()}")
    say(f"cv2 {cv.__version__}, {os.cpu_count()} host cores, sharpness {SHARPNESS}")
    res = {"card": torch.cuda.get_device_name(dev), "nvidia_smi": q.stdout.strip(), "sets": [], "e2e": []}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    say(f"== every call after a 256 MiB L2-flushing write; whole call by CUDA events over {args.reps} calls (median), "
        f"kernels by torch.profiler over {args.reps} calls (median); bytes: rows 5 B, cols 4 B, blend 5 B per layer "
        f"pixel in the canvas + 3 B per canvas pixel; share of {HBM_TBS} TB/s")
    sets = [("c4 centre + 16", lambda: case_layers(dev, "c4", 16)), ("c2 centre + 4", lambda: case_layers(dev, "c2", 4)),
            ("64 synthetic 1920 x 1080", lambda: synthetic_layers(dev))]
    for name, make in sets:
        layers, origins, size = make()
        nbytes, px = model_bytes(layers, origins, size)
        feather, mean, out_f, out_m, ws_bytes = calls(lib, dev, layers, origins, size)
        call_us = event_us(feather, args.reps, flush)
        mean_us = event_us(mean, args.reps, flush)
        kern = profiled_us([feather, mean], args.reps, flush)
        layers_np = [t.cpu().numpy() for t in layers]
        t0 = time.perf_counter()
        want = fo.feather_blend(layers_np, origins, size, SHARPNESS)
        oracle_s = time.perf_counter() - t0
        ok_f = bool(np.array_equal(out_f.cpu().numpy(), want))
        ok_m = bool(np.array_equal(out_m.cpu().numpy(), po.blend_layers(layers_np, origins, size)))
        cv_ms, cv_out = opencv_ms(layers_np, origins, size, 1 if len(layers) > 20 else 3)
        ok_cv = bool(np.array_equal(cv_out, want))
        say(f"{name}: {len(layers)} layers, canvas {size[0]} x {size[1]}, {px / 1e6:.1f} Mpix of layers in the canvas, "
            f"workspace {ws_bytes / 1e6:.1f} MB")

        def rate(k, us):
            tbs = nbytes[k] / (us * 1e-6) / 1e12
            return f"{us:.1f} us, {nbytes[k] / 1e6:.0f} MB, {tbs:.2f} TB/s = {100 * tbs / HBM_TBS:.0f} %"
        for k in KERNELS[:3]:
            say(f"  {k:16s} {rate(k, kern.get(k, float('nan')))}")
        say(f"  apap_feather_blend call {rate('call', call_us[0])} (min {call_us[1]:.1f} us; "
            f"floor {nbytes['call'] / (HBM_TBS * 1e12) * 1e6:.1f} us)")
        say(f"  k_blend_layers (mean) {rate('k_blend_layers', kern.get('k_blend_layers', float('nan')))}; "
            f"apap_blend_layers call {mean_us[0]:.1f} us")
        say(f"  cv.detail.FeatherBlender on the host: {cv_ms:.1f} ms; numpy oracle {oracle_s:.1f} s")
        say(f"  equal: feather = oracle {ok_f}, OpenCV = oracle {ok_cv}, mean = mean oracle {ok_m}")
        res["sets"].append({"set": name, "layers": len(layers), "canvas": list(size), "layer_px": px,
                            "kernels_us": kern, "call_us": call_us[0], "mean_call_us": mean_us[0], "bytes": nbytes,
                            "opencv_ms": cv_ms, "equal_oracle": ok_f, "opencv_equal_oracle": ok_cv,
                            "mean_equal_oracle": ok_m})
        del layers, out_f, out_m
    for name, k in (("c4", 16), ("c2", 4)):
        centre, others, raw_c, raw_os = _scene(name, k)
        fe = stitch_panorama(centre, others, raw_c, raw_os, ransac="gpu", blend="feather")
        me = stitch_panorama(centre, others, raw_c, raw_os, ransac="gpu")
        same = fe.final_size == me.final_size and np.array_equal(fe.origins, me.origins)
        t_f = host_ms(lambda: stitch_panorama(centre, others, raw_c, raw_os, ransac="gpu", blend="feather"), 3)
        t_m = host_ms(lambda: stitch_panorama(centre, others, raw_c, raw_os, ransac="gpu"), 3)
        say(f"== end to end {name}, centre + {k}, ransac='gpu': stitch_panorama blend='feather' {t_f[0]:.1f} ms vs "
            f"blend='mean' {t_m[0]:.1f} ms (3 reps, medians; same canvas and origins: {same})")
        res["e2e"].append({"case": name, "k": k, "feather_ms": t_f[0], "mean_ms": t_m[0], "same_layout": bool(same)})
    say(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
