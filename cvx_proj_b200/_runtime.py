"""ctypes binding of libapap_b200.so + device-buffer plumbing (torch is used only for device
memory, pinned host memory and streams).  There is NO CPU fallback: a missing library or a
missing GPU raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_size_t, c_void_p

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libapap_b200.so")

GRAM_TERMS = 24
KP_ROW = 28
KP_CHUNK = 128
HINV_ROW = 12
WARP_BLOCK_ROWS = 4
ABI_VERSION = 23
KP_BLOCK = 8
KP_BLOCK_FLOATS = 528
GRAM_TCGEN05 = 0
GRAM_FFMA2 = 1
EIG_AUTO = 0
EIG_JACOBI = 1
WARP_FORCE_EXACT = 1
WARP_LEGACY = 2
RANSAC_MAX_ITERS = 1 << 20
BLEND_MAX_LAYERS = 256
FEATHER_MAX_LAYERS = 128
GAIN_MAX_LAYERS = 256
MULTIBAND_MAX_LAYERS = 127
MULTIBAND_MAX_HEIGHT = 524280  # 65535 tiles of 8 rows: apap_multiband_* return APAP_E_TOOBIG above
E_TOOBIG = -3           # APAP_E_TOOBIG

# symbol -> (restype, argtypes); tests check every symbol of include/apap_b200.h is exported
SIGNATURES = {
    "apap_abi_version": (c_int, []),
    "apap_last_error": (c_char_p, []),
    "apap_device_sm_count": (c_int, [POINTER(c_int)]),
    "apap_gram_plan": (c_int, [c_int, c_int, c_int, POINTER(c_int), POINTER(c_int), POINTER(c_size_t)]),
    "apap_gram_partials": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_int, c_void_p, c_void_p, c_void_p]),
    "apap_weight_bound": (c_int, [c_void_p, c_void_p, c_int, c_int, c_double, c_void_p, c_int, c_void_p, c_void_p]),
    "apap_eig_denorm": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "apap_local_homography": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_int, c_int,
                                      c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "apap_pass_workspace_bytes": (c_int, [c_int, c_int, c_int, c_int, POINTER(c_size_t)]),
    "apap_local_homography_points": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_int, c_double, c_float,
                                             c_int, c_int, c_void_p, c_size_t, c_void_p, c_void_p, c_void_p, c_void_p]),
    "apap_local_weight": (c_int, [c_void_p, c_void_p, c_int, c_int, c_double, c_double, c_void_p, c_void_p]),
    "apap_warp": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int,
                          c_int, c_int, c_int, c_int, c_int, c_void_p, c_int, c_int, c_void_p, c_size_t, c_int, c_int,
                          c_void_p, c_void_p]),
    "apap_warp_bilinear": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                   c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "apap_warp_tiles_bytes": (c_int, [c_int, c_int, POINTER(c_size_t)]),
    "apap_warp_tiles": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                                c_int, c_void_p, c_size_t, c_void_p]),
    "apap_blend": (c_int, [c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "apap_blend_layers": (c_int, [POINTER(ctypes.c_longlong), c_int, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "apap_feather_distance_cap": (c_int, [c_float, c_int, c_int, POINTER(c_int)]),
    "apap_feather_workspace_bytes": (c_int, [POINTER(ctypes.c_longlong), c_int, c_int, c_int, POINTER(c_size_t)]),
    "apap_feather_blend": (c_int, [POINTER(ctypes.c_longlong), c_int, c_int, c_int, c_float, c_void_p, c_size_t,
                                   c_void_p, c_size_t, c_void_p]),
    "apap_gain_stats_bytes": (c_int, [c_int, POINTER(c_size_t)]),
    "apap_gain_stats": (c_int, [POINTER(ctypes.c_longlong), c_int, c_int, c_int, c_void_p, c_size_t, c_void_p]),
    "apap_blend_layers_gain": (c_int, [POINTER(ctypes.c_longlong), c_int, c_int, c_int, c_void_p, c_void_p, c_size_t,
                                       c_void_p]),
    "apap_feather_blend_gain": (c_int, [POINTER(ctypes.c_longlong), c_int, c_int, c_int, c_float, c_void_p, c_void_p,
                                        c_size_t, c_void_p, c_size_t, c_void_p]),
    "apap_multiband_workspace_bytes": (c_int, [POINTER(ctypes.c_longlong), c_int, c_int, c_int, c_int,
                                               POINTER(c_size_t)]),
    "apap_multiband_blend": (c_int, [POINTER(ctypes.c_longlong), c_int, c_int, c_int, c_int, c_void_p, c_size_t,
                                     c_void_p, c_size_t, c_void_p]),
    "apap_multiband_blend_gain": (c_int, [POINTER(ctypes.c_longlong), c_int, c_int, c_int, c_int, c_void_p, c_void_p,
                                          c_size_t, c_void_p, c_size_t, c_void_p]),
    "apap_pipe_probe": (c_int, [c_int, c_int, c_void_p, POINTER(c_double), c_void_p]),
    "apap_warp_perspective": (c_int, [c_void_p, c_int, c_int, POINTER(c_double), c_void_p, c_int, c_int, c_void_p, c_int,
                                      c_int, c_int, c_int, c_int, c_void_p]),
    "apap_affinity_matrix": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_float, c_void_p, c_void_p]),
    "apap_power_iterate": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "apap_multicast_copy": (c_int, [c_void_p, c_void_p, c_size_t, c_void_p]),
    "apap_peer_copy": (c_int, [c_void_p, c_void_p, c_int, c_size_t, c_void_p]),
    "apap_match_nn": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "apap_sift_describe": (c_int, [c_void_p, c_int, c_int, c_void_p, c_int, c_void_p, c_int, c_float, c_void_p, c_void_p,
                                   c_void_p]),
    "apap_sift_describe_lut": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_int, c_float, c_void_p,
                                       c_void_p, c_void_p]),
    "apap_equalize_hist": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "apap_ransac_workspace_bytes": (c_int, [c_int, POINTER(c_size_t)]),
    "apap_ransac_homography": (c_int, [c_void_p, c_void_p, c_int, c_double, c_int, c_void_p, c_size_t, c_void_p, c_void_p,
                                       c_void_p, c_void_p, c_void_p]),
    "apap_ransac_batch_workspace_bytes": (c_int, [c_int, c_int, POINTER(c_size_t)]),
    "apap_ransac_homography_batch": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_double, c_int, c_void_p,
                                             c_size_t, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "apap_invert_grid": (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "apap_kp_rows": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_double, c_void_p, c_void_p]),
    "apap_condition": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "apap_kp_blocks": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "apap_warp_tables": (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p,
                                 c_void_p]),
}


class ApapError(RuntimeError):
    """A non-zero return from libapap_b200 (CUDA error or argument error)."""


_lib = None


def load_library():
    """Load libapap_b200.so (built in-tree by ``__graft_entry__.build()`` / ``csrc/Makefile``)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ApapError(
            f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C cvx_proj_b200/csrc`.  cvx_proj_b200 has no CPU fallback.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError here = the .so does not match the header
        fn.restype = res
        fn.argtypes = args
    if lib.apap_abi_version() != ABI_VERSION:
        raise ApapError(f"libapap_b200 ABI {lib.apap_abi_version()} != expected {ABI_VERSION}")
    _lib = lib
    return lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = load_library().apap_last_error().decode("utf-8", "replace")
        raise ApapError(f"libapap_b200 {what} failed (code {rc}): {msg}")


def gram_plan(cells: int, n_kp_padded: int, engine: int = GRAM_TCGEN05):
    """(k_splits, cells_padded, partial_bytes_per_scene) -- pure host arithmetic, no GPU needed."""
    lib = load_library()
    ks, cp, nb = c_int(), c_int(), c_size_t()
    check(lib.apap_gram_plan(int(cells), int(n_kp_padded), int(engine), ctypes.byref(ks), ctypes.byref(cp), ctypes.byref(nb)),
          "apap_gram_plan")
    return ks.value, cp.value, nb.value


# ------------------------------------------------------------------------------- device plumbing
def torch_cuda(device=None):
    """Return (torch, torch.device) or raise: the compute path needs a CUDA device."""
    import torch

    if not torch.cuda.is_available():
        raise ApapError("no CUDA device: cvx_proj_b200 runs its hot path only on the GPU (no CPU fallback)")
    if device is None:
        device = torch.device("cuda", torch.cuda.current_device())
    else:
        device = torch.device(device)
        if device.type != "cuda":
            raise ApapError(f"device must be a CUDA device, got {device}")
        if device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
    return torch, device


def stream_ptr(torch, device) -> int:
    return int(torch.cuda.current_stream(device).cuda_stream)


def to_device(torch, device, host_array: np.ndarray):
    """Async H2D of a contiguous numpy array (true async when the array's memory is pinned)."""
    t = torch.from_numpy(np.ascontiguousarray(host_array))
    return t.to(device, non_blocking=True)


def to_host(torch, dev_tensor) -> np.ndarray:
    """D2H into fresh pinned memory (torch's caching host allocator), synchronised."""
    out = torch.empty(dev_tensor.shape, dtype=dev_tensor.dtype, pin_memory=True)
    out.copy_(dev_tensor, non_blocking=True)
    torch.cuda.current_stream(dev_tensor.device).synchronize()
    return out.numpy()


def to_host_many(torch, dev_tensors) -> list:
    """D2H of several tensors of one device into fresh pinned memory with a single synchronise."""
    outs = []
    for t in dev_tensors:
        out = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
        out.copy_(t, non_blocking=True)
        outs.append(out)
    if dev_tensors:
        torch.cuda.current_stream(dev_tensors[0].device).synchronize()
    return [o.numpy() for o in outs]


def pinned_empty(shape, dtype=np.uint8) -> np.ndarray:
    """A numpy array backed by pinned host memory (for callers that want full-speed copies)."""
    import torch

    tdt = {np.dtype(np.uint8): torch.uint8, np.dtype(np.float32): torch.float32,
           np.dtype(np.float64): torch.float64, np.dtype(np.uint16): torch.uint16,
           np.dtype(np.int32): torch.int32}[np.dtype(dtype)]
    return torch.empty(tuple(shape), dtype=tdt, pin_memory=True).numpy()


# ------------------------------------------------------------------------------ thin op wrappers
def blend_device(torch, a, b, out=None):
    """uniform_blend on device tensors ``[H, W, 3]`` uint8 (contiguous)."""
    lib = load_library()
    if a.shape != b.shape or a.dtype != torch.uint8 or b.dtype != torch.uint8 or a.shape[-1] != 3:
        raise ValueError("uniform_blend expects two uint8 images of identical [H, W, 3] shape")
    a = a.contiguous()
    b = b.contiguous()
    if out is None:
        out = torch.empty_like(a)
    n_px = a.numel() // 3
    with torch.cuda.device(a.device):
        check(lib.apap_blend(a.data_ptr(), b.data_ptr(), out.data_ptr(), n_px, stream_ptr(torch, a.device)),
              "apap_blend")
    return out


def blend_host(img1, img2):
    """``uniform_blend`` with the reference's numpy-in / numpy-out contract (or device tensors)."""
    torch, device = torch_cuda(getattr(img1, "device", None) if not isinstance(img1, np.ndarray) else None)
    if not isinstance(img1, np.ndarray):
        return blend_device(torch, img1, img2)
    if img1.shape != img2.shape or img1.ndim != 3 or img1.shape[-1] != 3:
        raise ValueError("uniform_blend expects two images of identical [H, W, 3] shape")
    a = to_device(torch, device, img1.astype(np.uint8, copy=False))
    b = to_device(torch, device, img2.astype(np.uint8, copy=False))
    return to_host(torch, blend_device(torch, a, b))


PROBE_FFMA = 0
PROBE_MUFU = 1


def pipe_peak(kind: int, device=None, iters: int = 1 << 15, reps: int = 5) -> float:
    """Measured peak of a pipe in operations/s (FFMA: flop/s, MUFU: lane-ops/s): best of ``reps``
    timed launches of the probe kernel."""
    torch, device = torch_cuda(device)
    lib = load_library()
    sink = torch.zeros(1, dtype=torch.float32, device=device)
    ops = c_double()
    best = 0.0
    with torch.cuda.device(device):
        st = stream_ptr(torch, device)
        check(lib.apap_pipe_probe(kind, iters, sink.data_ptr(), ctypes.byref(ops), st), "apap_pipe_probe")
        for _ in range(reps):
            e0 = torch.cuda.Event(enable_timing=True)
            e1 = torch.cuda.Event(enable_timing=True)
            e0.record()
            check(lib.apap_pipe_probe(kind, iters, sink.data_ptr(), ctypes.byref(ops), st), "apap_pipe_probe")
            e1.record()
            e1.synchronize()
            best = max(best, ops.value / (e0.elapsed_time(e1) * 1e-3))
    return best


def fp32_peak_tflops(device=None) -> float:
    """Measured FP32 FMA-pipe peak (TFLOP/s)."""
    return pipe_peak(PROBE_FFMA, device, iters=1 << 16) / 1e12
