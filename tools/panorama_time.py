#!/usr/bin/env python
"""Cost of the panorama of a case (driver.stitch_panorama) and of its blend kernel.  One run prints:
  - the card's name, power limit and top SM clock (queries only);
  - k_blend_layers (one apap_blend_layers call) by CUDA events on three layer sets, each call preceded by a 256 MiB
    write that flushes L2 (the c4 set is about L2-sized), and back to back without the flush:
      the c4-size case (centre + 16 others) and the c2-size case (centre + 4 others) of tests/test_case.py, layers =
      the pair canvases local_warp makes plus the centre, placed as stitch_panorama places them;
      64 synthetic 1920 x 1080 layers spread over a larger canvas;
    with the bytes the blend must move, 3 x sum |layer ∩ canvas| + 3 x W x H, over kernel time, against 7.7 TB/s, and
    the kernel's output checked against oracle.panorama_oracle.blend_layers;
  - end to end on the two cases: stitch_panorama against what a user had to do without it -- stitch_case(stitch=False),
    K local_warp calls with numpy out, then the numpy blend of the oracle -- with the outputs checked equal.

    python tools/panorama_time.py [--reps 200] [--out FILE]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from cvx_proj_b200 import _runtime as rt  # noqa: E402
from cvx_proj_b200.apap import APAP  # noqa: E402
from cvx_proj_b200.driver import panorama_size, stitch_case, stitch_panorama  # noqa: E402
from oracle import panorama_oracle as po  # noqa: E402
from sift_time import host_ms  # noqa: E402
from tests.test_case import _scene  # noqa: E402

HBM_TBS = 7.7           # B200 data sheet, one GPU


def case_layers(dev, name, k):
    """The layers stitch_panorama blends for the test scene ``name`` with ``k`` others, on the device."""
    centre, others, raw_c, raw_os = _scene(name, k)
    pairs = stitch_case(centre, others, raw_c, raw_os, stitch=False, ransac="gpu")
    layers = []
    for p, o in zip(pairs, others):
        w, h, ox, oy = p.final_size
        layers.append(APAP(0.5, 100, [w, h], [ox, oy], device=dev).local_warp(torch.from_numpy(o).to(dev),
                                                                               p.local_homography.copy(), p.mesh))
    (width, height, ox, oy), origins = panorama_size([p.final_size for p in pairs])
    layers.append(torch.from_numpy(centre).to(dev))
    return layers, [tuple(map(int, o)) for o in origins] + [(ox, oy)], (width, height)


def synthetic_layers(dev, n=64):
    r = np.random.default_rng(0)
    w, h = 1920, 1080
    layers, origins = [], []
    for j in range(n):
        img = r.integers(1, 256, (h, w, 3), dtype=np.uint8)
        img[: h // 8] = 0                                       # an empty band, as a warped canvas has
        layers.append(torch.from_numpy(img).to(dev))
        origins.append((int((j % 8) * 0.5 * w + r.integers(0, 50)), int((j // 8) * 0.5 * h + r.integers(0, 50))))
    width = max(x + w for x, _ in origins) - 100
    height = max(y + h for _, y in origins) - 60                # the last row and column stick out: clipped
    return layers, origins, (width, height)


def moved_bytes(layers, origins, size):
    width, height = size
    inside = 0
    for t, (x0, y0) in zip(layers, origins):
        h, w = t.shape[:2]
        inside += max(0, min(x0 + w, width) - max(x0, 0)) * max(0, min(y0 + h, height) - max(y0, 0))
    return 3 * inside + 3 * width * height


def kernel_us(lib, dev, layers, origins, size, reps, flush):
    width, height = size
    desc = np.array([[t.data_ptr(), t.shape[0], t.shape[1], t.stride(0), x0, y0]
                     for t, (x0, y0) in zip(layers, origins)], dtype=np.int64)
    out = torch.empty((height, width, 3), dtype=torch.uint8, device=dev)
    st = rt.stream_ptr(torch, dev)
    ptr = desc.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong))

    def call():
        rt.check(lib.apap_blend_layers(ptr, len(layers), height, width, out.data_ptr(), out.numel(), st),
                 "apap_blend_layers")
    for _ in range(3):
        call()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        if flush is not None:
            flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        call()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    return float(np.median(ts)), float(np.min(ts)), out.cpu().numpy()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=200)
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
    res = {"card": torch.cuda.get_device_name(dev), "nvidia_smi": q.stdout.strip(), "kernel": [], "e2e": []}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    say(f"== k_blend_layers, CUDA events over {args.reps} calls (median, min); bytes = 3 sum|layer ∩ canvas| + 3 W H; "
        f"share of {HBM_TBS} TB/s")
    sets = [("c4 centre + 16", *case_layers(dev, "c4", 16)), ("c2 centre + 4", *case_layers(dev, "c2", 4)),
            ("64 synthetic 1920 x 1080", *synthetic_layers(dev))]
    for name, layers, origins, size in sets:
        nbytes = moved_bytes(layers, origins, size)
        cold = kernel_us(lib, dev, layers, origins, size, args.reps, flush)
        warm = kernel_us(lib, dev, layers, origins, size, args.reps, None)
        want = po.blend_layers([t.cpu().numpy() for t in layers], origins, size)
        ok = bool(np.array_equal(cold[2], want) and np.array_equal(warm[2], want))
        bw = nbytes / (cold[0] * 1e-6) / 1e12
        say(f"{name}: {len(layers)} layers, canvas {size[0]} x {size[1]}, {nbytes / 1e6:.1f} MB moved "
            f"(floor {nbytes / (HBM_TBS * 1e12) * 1e6:.1f} us); L2 flushed {cold[0]:.1f} us (min {cold[1]:.1f}) = "
            f"{bw:.2f} TB/s = {100 * bw / HBM_TBS:.0f} % of HBM; back to back {warm[0]:.1f} us (min {warm[1]:.1f}) = "
            f"{nbytes / (warm[0] * 1e-6) / 1e12:.2f} TB/s; equals oracle: {ok}")
        res["kernel"].append({"set": name, "layers": len(layers), "canvas": list(size), "bytes": nbytes,
                              "flushed_us": cold[0], "flushed_min_us": cold[1], "warm_us": warm[0],
                              "warm_min_us": warm[1], "tbs": bw, "equal_oracle": ok})
    del sets
    for name, k in (("c4", 16), ("c2", 4)):
        centre, others, raw_c, raw_os = _scene(name, k)
        say(f"== end to end: {name} ({centre.shape[1]} x {centre.shape[0]}), centre + {k} others, mesh 100")
        for mode in ("opencv", "gpu"):
            def user_path():
                pairs = stitch_case(centre, others, raw_c, raw_os, stitch=False, ransac=mode)
                layers = []
                for p, o in zip(pairs, others):
                    w, h, ox, oy = p.final_size
                    layers.append(APAP(0.5, 100, [w, h], [ox, oy]).local_warp(o, p.local_homography.copy(), p.mesh))
                (width, height, ox, oy), origins = panorama_size([p.final_size for p in pairs])
                return po.blend_layers(layers + [centre], [tuple(o) for o in origins] + [(ox, oy)], (width, height))
            got = stitch_panorama(centre, others, raw_c, raw_os, ransac=mode)
            want = user_path()
            eq = bool(np.array_equal(got.panorama, want))
            reps = 3
            t_p = host_ms(lambda: stitch_panorama(centre, others, raw_c, raw_os, ransac=mode), reps)
            t_c = host_ms(lambda: stitch_case(centre, others, raw_c, raw_os, stitch=False, ransac=mode), reps)
            t_u = host_ms(user_path, reps)
            say(f"  ransac={mode!r}: panorama {got.final_size[0]} x {got.final_size[1]}; stitch_panorama {t_p[0]:.1f} ms "
                f"vs stitch_case(stitch=False) + {k} local_warp downloads + numpy blend {t_u[0]:.1f} ms "
                f"(of which stitch_case {t_c[0]:.1f} ms) (equal: {eq}) ({reps} reps, medians)")
            res["e2e"].append({"case": name, "k": k, "ransac": mode, "panorama": list(got.final_size),
                               "stitch_panorama_ms": t_p[0], "user_path_ms": t_u[0], "stitch_case_ms": t_c[0],
                               "equal": eq})
    say(json.dumps(res))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
