#!/usr/bin/env python
"""Cost of exposure compensation (utils.exposure_gains, the blends with gains, stitch_panorama(exposure="gain")).
One run prints:
  - the card's name, power limit and top SM clock (queries only);
  - on the layer sets of tools/feather_time.py (the c4-size case, centre + 16; the c2-size case, centre + 4; 64
    synthetic 1920 x 1080 layers), each call preceded by a 256 MiB write that flushes L2, by CUDA events:
      apap_gain_stats (memset + k_gain_stats) against its floor of 3 B per layer pixel in the canvas at 7.7 TB/s;
      apap_blend_layers and apap_feather_blend with gains against without;
      the whole exposure_gains call (host clock, ends in its download and the host solve);
      cv.detail.GainCompensator.feed on the host cores, fed as the contract says (sets of at most 20 layers);
      the statistics checked against oracle.gain_oracle, the gains against OpenCV's;
  - end to end on the c4 and c2 cases: stitch_panorama(exposure="gain") against "none", for both blends.

    python tools/gain_time.py [--reps 50] [--out FILE]
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
from cvx_proj_b200.utils import _gain_table, exposure_gains, gain_stats_ints  # noqa: E402
from feather_time import event_us  # noqa: E402
from oracle import feather_oracle as fo  # noqa: E402
from oracle import gain_oracle as go  # noqa: E402
from panorama_time import HBM_TBS, case_layers, synthetic_layers  # noqa: E402
from sift_time import host_ms  # noqa: E402
from tests.test_case import _scene  # noqa: E402

SHARPNESS = 0.02


def layer_px(layers, origins, size):
    width, height = size
    px = 0
    for t, (x0, y0) in zip(layers, origins):
        h, w = t.shape[:2]
        px += max(0, min(x0 + w, width) - max(x0, 0)) * max(0, min(y0 + h, height) - max(y0, 0))
    return px


def calls(lib, dev, layers, origins, size, gains):
    width, height = size
    n = len(layers)
    desc = np.array([[t.data_ptr(), t.shape[0], t.shape[1], t.stride(0), x0, y0]
                     for t, (x0, y0) in zip(layers, origins)], dtype=np.int64)
    ptr = desc.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong))
    nb = ctypes.c_size_t()
    rt.check(lib.apap_gain_stats_bytes(n, ctypes.byref(nb)), "stats bytes")
    stats = torch.empty(nb.value // 8, dtype=torch.int64, device=dev)
    ws_bytes = ctypes.c_size_t()
    rt.check(lib.apap_feather_workspace_bytes(ptr, n, height, width, ctypes.byref(ws_bytes)), "ws bytes")
    ws = torch.empty(ws_bytes.value, dtype=torch.uint8, device=dev)
    lut = torch.from_numpy(_gain_table("gain_time", gains, n)).to(dev)
    out = torch.empty((height, width, 3), dtype=torch.uint8, device=dev)
    st = rt.stream_ptr(torch, dev)
    fns = {
        "stats": lambda: rt.check(lib.apap_gain_stats(ptr, n, height, width, stats.data_ptr(), nb.value, st), "stats"),
        "mean": lambda: rt.check(lib.apap_blend_layers(ptr, n, height, width, out.data_ptr(), out.numel(), st), "mean"),
        "mean_gain": lambda: rt.check(lib.apap_blend_layers_gain(ptr, n, height, width, lut.data_ptr(), out.data_ptr(),
                                                                 out.numel(), st), "mean gain"),
        "feather": lambda: rt.check(lib.apap_feather_blend(ptr, n, height, width, SHARPNESS, ws.data_ptr(), ws.numel(),
                                                           out.data_ptr(), out.numel(), st), "feather"),
        "feather_gain": lambda: rt.check(lib.apap_feather_blend_gain(ptr, n, height, width, SHARPNESS, lut.data_ptr(),
                                                                     ws.data_ptr(), ws.numel(), out.data_ptr(),
                                                                     out.numel(), st), "feather gain"),
    }
    return fns, stats


def opencv_feed_ms(layers_np, origins, size, reps):
    ps = [fo.paste(img, o, size) for img, o in zip(layers_np, origins)]
    ms = [np.where(p.max(axis=-1) > 0, 255, 0).astype(np.uint8) for p in ps]
    ups, ums = [cv.UMat(p) for p in ps], [cv.UMat(m) for m in ms]

    def run():
        comp = cv.detail.GainCompensator()
        comp.feed([(0, 0)] * len(ps), ups, ums)
        return np.asarray(comp.getMatGains(), dtype=np.float64).reshape(-1)
    got = run()
    return host_ms(run, reps)[0], got


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
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
    say(f"cv2 {cv.__version__}, {os.cpu_count()} host cores, feather sharpness {SHARPNESS}")
    res = {"card": torch.cuda.get_device_name(dev), "nvidia_smi": q.stdout.strip(), "sets": [], "e2e": []}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    say(f"== every kernel call after a 256 MiB L2-flushing write, CUDA events over {args.reps} calls (median); "
        f"stats floor: 3 B per layer pixel in the canvas at {HBM_TBS} TB/s")
    sets = [("c4 centre + 16", lambda: case_layers(dev, "c4", 16)), ("c2 centre + 4", lambda: case_layers(dev, "c2", 4)),
            ("64 synthetic 1920 x 1080", lambda: synthetic_layers(dev))]
    for name, make in sets:
        layers, origins, size = make()
        px = layer_px(layers, origins, size)
        g = exposure_gains(layers, origins, size)
        fns, stats = calls(lib, dev, layers, origins, size, g)
        us = {k: event_us(fn, args.reps, flush) for k, fn in fns.items()}
        torch.cuda.synchronize()
        t_call = host_ms(lambda: exposure_gains(layers, origins, size), 5)[0]
        fns["stats"]()
        got = gain_stats_ints(stats.cpu().numpy(), len(layers))
        layers_np = [t.cpu().numpy() for t in layers]
        want = go.stats(layers_np, origins, size)
        ok_stats = got == want
        ok_gains = bool(np.array_equal(g, go.gains_from_stats(*want)))
        if len(layers) <= 20:
            cv_ms, g_cv = opencv_feed_ms(layers_np, origins, size, 3)
            rel = float(np.max(np.abs(g - g_cv) / np.abs(g_cv)))
        else:   # not measured: feed walks each of the 2 016 pairs over the whole pasted canvas
            cv_ms, rel = float("nan"), float("nan")
        floor_us = 3 * px / (HBM_TBS * 1e12) * 1e6
        say(f"{name}: {len(layers)} layers, canvas {size[0]} x {size[1]}, {px / 1e6:.1f} Mpix of layers in the canvas; "
            f"gains {np.round(g, 4).tolist()}")
        say(f"  apap_gain_stats {us['stats'][0]:.1f} us (min {us['stats'][1]:.1f}); floor {floor_us:.1f} us "
            f"({3 * px / 1e6:.0f} MB) = {100 * floor_us / us['stats'][0]:.0f} % of the floor")
        say(f"  apap_blend_layers {us['mean'][0]:.1f} us, with gains {us['mean_gain'][0]:.1f} us; "
            f"apap_feather_blend {us['feather'][0]:.1f} us, with gains {us['feather_gain'][0]:.1f} us")
        cv_txt = f"{cv_ms:.1f} ms" if cv_ms == cv_ms else "not measured"
        say(f"  exposure_gains call {t_call:.2f} ms; GainCompensator.feed on the host {cv_txt}")
        say(f"  equal: stats = oracle {ok_stats}, gains = oracle {ok_gains}; max relative gap to OpenCV's gains "
            + (f"{rel:.1e}" if rel == rel else "not measured"))
        res["sets"].append({"set": name, "layers": len(layers), "canvas": list(size), "layer_px": px,
                            "call_us": {k: v[0] for k, v in us.items()}, "exposure_gains_ms": t_call,
                            "opencv_feed_ms": cv_ms, "stats_equal_oracle": ok_stats, "gains_equal_oracle": ok_gains,
                            "rel_gap_opencv": rel})
        del layers, stats
    for name, k in (("c4", 16), ("c2", 4)):
        centre, others, raw_c, raw_os = _scene(name, k)
        row = {"case": name, "k": k}
        for blend in ("mean", "feather"):
            for exposure in ("none", "gain"):
                stitch_panorama(centre, others, raw_c, raw_os, ransac="gpu", blend=blend, exposure=exposure)
                row[f"{blend}_{exposure}_ms"] = host_ms(lambda: stitch_panorama(
                    centre, others, raw_c, raw_os, ransac="gpu", blend=blend, exposure=exposure), 3)[0]
        say(f"== end to end {name}, centre + {k}, ransac='gpu' (3 reps, medians): mean {row['mean_none_ms']:.1f} ms, "
            f"with gains {row['mean_gain_ms']:.1f} ms; feather {row['feather_none_ms']:.1f} ms, "
            f"with gains {row['feather_gain_ms']:.1f} ms")
        res["e2e"].append(row)
    say(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
