#!/usr/bin/env python
"""Cost of per-channel exposure compensation (utils.channel_gains, the blends with per-channel tables,
stitch_panorama(exposure="channels")).  One run prints:
  - the card's name, power limit and top SM clock (queries only);
  - on the layer sets of timing.LAYER_SETS, each call preceded by a 256 MiB write that flushes L2, by CUDA events:
      apap_channel_stats against apap_gain_stats (both memset + k_gain_stats);
      apap_blend_layers, apap_feather_blend and apap_multiband_blend with per-channel tables, against one table and
      against none;
      the whole channel_gains call (host clock, ends in its download and the three host solves);
      cv.detail.ChannelsCompensator.feed on the host cores, fed as the contract says (sets of at most 20 layers);
      the statistics checked against oracle.channels_oracle, the gains against it and against OpenCV's;
  - end to end on the c4 and c2 cases: stitch_panorama(exposure="channels" | "gain" | "none") for all three blends.

    python tools/channels_time.py [--reps 50] [--out FILE]
"""
import argparse
import ctypes
import json
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
from cvx_proj_b200.utils import _gain_table, _layer_descs, channel_gains, exposure_gains  # noqa: E402
from oracle import channels_oracle as co  # noqa: E402
from oracle import feather_oracle as fo  # noqa: E402
from timing import LAYER_SETS, card, clipped_px, event_us, host_ms, l2_flush, say, write_out  # noqa: E402

SHARPNESS = 0.02
BANDS = 5


def calls(lib, dev, layers, origins, size, gains, gains3):
    width, height = size
    n = len(layers)
    _, desc = _layer_descs(torch, dev, layers, origins, True)     # packed device layers: described in place
    ptr = desc.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong))
    nb = ctypes.c_size_t()
    rt.check(lib.apap_gain_stats_bytes(n, ctypes.byref(nb)), "stats bytes")
    stats = torch.empty(nb.value // 8, dtype=torch.int64, device=dev)
    fws, mws = ctypes.c_size_t(), ctypes.c_size_t()
    rt.check(lib.apap_feather_workspace_bytes(ptr, n, height, width, ctypes.byref(fws)), "feather ws bytes")
    ws_f = torch.empty(max(fws.value, 16), dtype=torch.uint8, device=dev)
    ws_m = None
    if n <= rt.MULTIBAND_MAX_LAYERS:
        rt.check(lib.apap_multiband_workspace_bytes(ptr, n, height, width, BANDS, ctypes.byref(mws)), "mb ws bytes")
        ws_m = torch.empty(max(mws.value, 16), dtype=torch.uint8, device=dev)
    lut1 = torch.from_numpy(_gain_table("channels_time", gains, n)).to(dev)
    lut3 = torch.from_numpy(_gain_table("channels_time", gains3, n)).to(dev)
    out = torch.empty((height, width, 3), dtype=torch.uint8, device=dev)
    st = rt.stream_ptr(torch, dev)
    o = (out.data_ptr(), out.numel(), st)
    fns = {
        "gain_stats": lambda: rt.check(lib.apap_gain_stats(ptr, n, height, width, stats.data_ptr(), nb.value, st), "g"),
        "channel_stats": lambda: rt.check(lib.apap_channel_stats(ptr, n, height, width, stats.data_ptr(), nb.value, st),
                                          "c"),
        "mean": lambda: rt.check(lib.apap_blend_layers(ptr, n, height, width, *o), "mean"),
        "mean_gain": lambda: rt.check(lib.apap_blend_layers_gain(ptr, n, height, width, lut1.data_ptr(), *o), "mg"),
        "mean_channels": lambda: rt.check(lib.apap_blend_layers_channels(ptr, n, height, width, lut3.data_ptr(), *o),
                                          "mc"),
    }
    if n <= rt.FEATHER_MAX_LAYERS:
        fw = (ws_f.data_ptr(), ws_f.numel(), *o)
        fns["feather"] = lambda: rt.check(lib.apap_feather_blend(ptr, n, height, width, SHARPNESS, *fw), "f")
        fns["feather_gain"] = lambda: rt.check(lib.apap_feather_blend_gain(ptr, n, height, width, SHARPNESS,
                                                                           lut1.data_ptr(), *fw), "fg")
        fns["feather_channels"] = lambda: rt.check(lib.apap_feather_blend_channels(ptr, n, height, width, SHARPNESS,
                                                                                   lut3.data_ptr(), *fw), "fc")
    if ws_m is not None:
        mw = (ws_m.data_ptr(), ws_m.numel(), *o)
        fns["multiband"] = lambda: rt.check(lib.apap_multiband_blend(ptr, n, height, width, BANDS, *mw), "m")
        fns["multiband_gain"] = lambda: rt.check(lib.apap_multiband_blend_gain(ptr, n, height, width, BANDS,
                                                                               lut1.data_ptr(), *mw), "mbg")
        fns["multiband_channels"] = lambda: rt.check(lib.apap_multiband_blend_channels(ptr, n, height, width, BANDS,
                                                                                       lut3.data_ptr(), *mw), "mbc")
    return fns, stats


def opencv_feed_ms(layers_np, origins, size, reps):
    ps = [fo.paste(img, o, size) for img, o in zip(layers_np, origins)]
    ms = [np.where(p.max(axis=-1) > 0, 255, 0).astype(np.uint8) for p in ps]
    ups, ums = [cv.UMat(p) for p in ps], [cv.UMat(m) for m in ms]

    def run():
        comp = cv.detail.ChannelsCompensator()
        comp.feed([(0, 0)] * len(ps), ups, ums)
        return np.array([np.asarray(v, np.float64).reshape(-1)[:3] for v in comp.getMatGains()])
    got = run()
    return host_ms(run, reps)[0], got


def fmt(us, k):
    return f"{us[k][0]:.1f}" if k in us else "not measured"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    _, dev = rt.torch_cuda()
    lib = rt.load_library()
    res = {**card(dev), "sets": [], "e2e": []}
    say(f"cv2 {cv.__version__}, {os.cpu_count()} host cores, feather sharpness {SHARPNESS}, multiband bands {BANDS}")
    flush = l2_flush(dev)
    say(f"== every kernel call after a 256 MiB L2-flushing write, CUDA events over {args.reps} calls (median, us)")
    for name, make in LAYER_SETS:
        layers, origins, size = make(dev)
        px = clipped_px(layers, origins, size)
        g1 = exposure_gains(layers, origins, size)
        g3 = channel_gains(layers, origins, size)
        fns, stats = calls(lib, dev, layers, origins, size, g1, g3)
        us = {k: event_us(fn, args.reps, flush) for k, fn in fns.items()}
        torch.cuda.synchronize()
        t_call = host_ms(lambda: channel_gains(layers, origins, size), 5)[0]
        fns["channel_stats"]()
        n = len(layers)
        w = stats.cpu().numpy().view(np.uint64).reshape(4, n, n)
        layers_np = [t.cpu().numpy() for t in layers]
        want = co.stats(layers_np, origins, size)
        got = ([[int(v) for v in row] for row in w[0]], [[[int(v) for v in row] for row in w[1 + c]] for c in range(3)])
        ok_stats = all(got[0][i][j] == (want[0][i][j] if i <= j else 0) for i in range(n) for j in range(n)) and \
            all(got[1][c][i][j] == (want[1][c][i][j] if i != j else 0) for c in range(3) for i in range(n)
                for j in range(n))
        ok_gains = bool(np.array_equal(g3, co.gains_from_stats(*want)))
        if n <= 20:
            cv_ms, g_cv = opencv_feed_ms(layers_np, origins, size, 3)
            ok_cv = bool(np.array_equal(g3, g_cv))
        else:   # not measured: feed walks each of the 2 016 pairs over the whole pasted canvas, per channel
            cv_ms, ok_cv = float("nan"), None
        say(f"{name}: {n} layers, canvas {size[0]} x {size[1]}, {px / 1e6:.1f} Mpix of layers in the canvas")
        say(f"  apap_channel_stats {fmt(us, 'channel_stats')} us, apap_gain_stats {fmt(us, 'gain_stats')} us")
        for b in ("mean", "feather", "multiband"):
            say(f"  {b}: per-channel tables {fmt(us, b + '_channels')} us, one table {fmt(us, b + '_gain')} us, "
                f"none {fmt(us, b)} us")
        cv_txt = f"{cv_ms:.1f} ms" if cv_ms == cv_ms else "not measured"
        say(f"  channel_gains call {t_call:.2f} ms; ChannelsCompensator.feed on the host {cv_txt}")
        say(f"  equal: stats = oracle {ok_stats}, gains = oracle {ok_gains}, gains = OpenCV "
            + ("not measured" if ok_cv is None else str(ok_cv)))
        res["sets"].append({"set": name, "layers": n, "canvas": list(size), "layer_px": px,
                            "call_us": {k: v[0] for k, v in us.items()}, "channel_gains_ms": t_call,
                            "opencv_feed_ms": cv_ms, "stats_equal_oracle": ok_stats, "gains_equal_oracle": ok_gains,
                            "gains_equal_opencv": ok_cv})
        del layers, stats
    for name, k in (("c4", 16), ("c2", 4)):
        centre, others, raw_c, raw_os = synth.make_case(name, k)
        row = {"case": name, "k": k}
        for blend in ("mean", "feather", "multiband"):
            for exposure in ("none", "gain", "channels"):
                stitch_panorama(centre, others, raw_c, raw_os, ransac="gpu", blend=blend, exposure=exposure)
                row[f"{blend}_{exposure}_ms"] = host_ms(lambda: stitch_panorama(
                    centre, others, raw_c, raw_os, ransac="gpu", blend=blend, exposure=exposure), 3)[0]
            say(f"== end to end {name}, centre + {k}, ransac='gpu', blend={blend!r} (3 reps, medians): "
                f"none {row[blend + '_none_ms']:.1f} ms, gain {row[blend + '_gain_ms']:.1f} ms, "
                f"channels {row[blend + '_channels_ms']:.1f} ms")
        res["e2e"].append(row)
    say(json.dumps(res))
    write_out(args.out)


if __name__ == "__main__":
    main()
