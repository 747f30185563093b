"""What the timing tools (tools/*_time.py) measure with: the report and the card query, the L2 flush, CUDA-event,
torch.profiler and host timing, and the placed-layer sets the blend tools time.  A module, not a tool."""
import os
import subprocess
import time

import numpy as np
import torch

from cvx_proj_b200 import synth
from cvx_proj_b200.apap import APAP
from cvx_proj_b200.driver import panorama_size, stitch_case

HBM_TBS = 7.7           # HGX B200 data sheet, one GPU

_lines = []


def say(s):
    """Print ``s`` now and keep it for ``write_out``."""
    print(s, flush=True)
    _lines.append(s)


def card(dev):
    """Say the card's name, power limit and top SM clock (queries only: nothing is set) and return them as the JSON
    result's ``card`` and ``nvidia_smi``."""
    name = torch.cuda.get_device_name(dev)
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    say(f"card: {name} | nvidia-smi: {q.stdout.strip() or q.stderr.strip()}")
    return {"card": name, "nvidia_smi": q.stdout.strip()}


def write_out(path):
    """Write every line said so far to ``path`` (a tool's ``--out``), creating its directory; nothing when None."""
    if path:
        os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
        with open(path, "w") as f:
            f.write("\n".join(_lines) + "\n")


def l2_flush(dev):
    """A 256 MiB buffer, twice the B200's L2: ``fill_(1)`` on it before a call evicts that call's inputs."""
    return torch.empty(256 << 20, dtype=torch.uint8, device=dev)


def event_us(fn, reps, flush=None, warmup=3):
    """(median, min) device time in us of ``reps`` calls of ``fn``, each between two CUDA events and followed by a
    synchronise, after ``flush.fill_(1)`` when a flush buffer is given; ``warmup`` untimed calls first."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        if flush is not None:
            flush.fill_(1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    return float(np.median(ts)), float(np.min(ts))


def host_ms(fn, reps):
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), float(np.min(ts))


def kernel_times(fns, name_of, reps, flush=None):
    """{name: [device us of each launch]} from one torch.profiler run of ``reps`` rounds over ``fns``, each call after
    ``flush.fill_(1)`` when a flush buffer is given.  ``name_of(kernel name)`` gives the name to file a launch under,
    or None to leave it out."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            for fn in fns:
                if flush is not None:
                    flush.fill_(1)
                fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.events():
        name = name_of(ev.name) if ev.device_type.name == "CUDA" else None
        if name:
            out.setdefault(name, []).append(ev.device_time_total)
    return out


def name_in(names):
    """A ``name_of`` for ``kernel_times``: the first of ``names`` that a kernel's name contains."""
    return lambda kernel: next((n for n in names if n in kernel), None)


def clipped_px(layers, origins, size):
    """Pixels of the layers (``[h, w, ...]``, top-left corner at ``origins``) that fall inside the ``size`` canvas."""
    width, height = size
    px = 0
    for t, (x0, y0) in zip(layers, origins):
        h, w = t.shape[:2]
        px += max(0, min(x0 + w, width) - max(x0, 0)) * max(0, min(y0 + h, height) - max(y0, 0))
    return px


def case_layers(dev, name, k):
    """The layers stitch_panorama blends for synth.make_case(``name``, ``k``), on the device: the pair canvases
    local_warp makes plus the centre, with their origins and the canvas size."""
    centre, others, raw_c, raw_os = synth.make_case(name, k)
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


# The sets the blend tools time, (name, make(dev) -> (layers, origins, size)): the c4-size case (about L2-sized), the
# c2-size case, and 64 synthetic layers over a larger canvas.
LAYER_SETS = (("c4 centre + 16", lambda dev: case_layers(dev, "c4", 16)),
              ("c2 centre + 4", lambda dev: case_layers(dev, "c2", 4)),
              ("64 synthetic 1920 x 1080", synthetic_layers))
