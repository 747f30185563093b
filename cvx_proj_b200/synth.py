"""Seeded synthetic image pairs and matched keypoints for the APAP path.

The reference's dataset (hazy image cases + ``keypoints.mat``) is not shipped
(``/root/reference/.gitignore:1-3``), so every test, golden vector and benchmark uses
this generator (SURVEY.md section 8d): matched keypoints from a known global homography
plus a smooth local distortion and pixel noise, and images whose values all lie in
[1, 255] (``uniform_blend`` treats black as "empty", reference pyviz/apap_utils.py:81).

Named configurations follow BASELINE.json ``configs``:
  c1  1024x768,  N=500,  100x100 grid   (the reference's own CPU-runnable case)
  c2  3840x2160, N=5k,   200x200 grid   (1 B200; the headline bench workload)
  c3  7680x4320, N=20k,  400x400 grid   (cells / row bands sharded over 2/4/8 B200)
  c4  1920x1080, N=2k,   100x100 grid   (x64 pairs, seeds 0..63)
  c5  1920x1080, N=1k..64k, 256x256 grid (keypoint sweep)
"""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from .apap_utils import final_size, get_mesh, get_vertice

CONFIGS = {
    "c1": dict(width=1024, height=768, n_kp=500, mesh=100),
    "c2": dict(width=3840, height=2160, n_kp=5000, mesh=200),
    "c3": dict(width=7680, height=4320, n_kp=20000, mesh=400),
    "c4": dict(width=1920, height=1080, n_kp=2000, mesh=100),
    "c5": dict(width=1920, height=1080, n_kp=4096, mesh=256),
    # small shapes for unit tests / golden vectors (not in BASELINE.json)
    "tiny": dict(width=160, height=120, n_kp=96, mesh=8),
    "mini": dict(width=256, height=192, n_kp=200, mesh=16),
}

GAMMA = 0.5   # reference pyviz/apap.py:222
SIGMA = 100   # reference pyviz/apap.py:223


def ground_truth_h(width: int, height: int) -> np.ndarray:
    """The known global homography of the generator (float64 3x3)."""
    k = 1024.0 / width
    return np.array(
        [[1.02, 0.03, 0.12 * width],
         [-0.02, 0.98, -0.045 * height],
         [1e-5 * k, -2e-5 * k, 1.0]], dtype=np.float64)


def make_keypoints(width: int, height: int, n_kp: int, seed: int = 0):
    """``(src[N,2] f32, dst[N,2] f32, H_gt)``: dst = proj(H_gt src) + smooth warp + noise."""
    rng = np.random.default_rng(seed)
    h_gt = ground_truth_h(width, height)
    src = rng.uniform([0.0, 0.0], [float(width), float(height)], size=(n_kp, 2))
    hom = np.concatenate([src, np.ones((n_kp, 1))], axis=1) @ h_gt.T
    proj = hom[:, :2] / hom[:, 2:3]
    wobble = 3.0 * (width / 1024.0) * np.sin(src / (0.15 * width))
    noise = rng.normal(0.0, 0.5, size=(n_kp, 2))
    dst = proj + wobble + noise
    return src.astype(np.float32), dst.astype(np.float32), h_gt


def make_image(width: int, height: int, seed: int = 1) -> np.ndarray:
    """``[height, width, 3]`` uint8 BGR-like image, every value in [1, 255].

    Low-frequency colour pattern plus per-pixel noise, so that neighbouring source
    pixels differ (a wrong nearest-pixel pick changes the value) and nothing is black.
    """
    rng = np.random.default_rng(seed)
    yy = np.arange(height, dtype=np.float32)[:, None]
    xx = np.arange(width, dtype=np.float32)[None, :]
    img = np.empty((height, width, 3), dtype=np.uint8)
    for ch, (fx, fy, ph) in enumerate(((3.0, 2.0, 0.0), (2.0, 5.0, 1.3), (7.0, 3.0, 2.1))):
        base = 128.0 + 90.0 * np.sin(2 * np.pi * fx * xx / width + ph) * np.cos(2 * np.pi * fy * yy / height)
        noise = rng.integers(-24, 25, size=(height, width), dtype=np.int16)
        img[..., ch] = np.clip(base.astype(np.int16) + noise, 1, 255).astype(np.uint8)
    return img


@dataclass
class Scene:
    """Everything one APAP pass needs, laid out as the reference driver builds it
    (pyviz/apap.py:238-241)."""
    name: str
    width: int
    height: int
    mesh_cells: int
    src: np.ndarray          # [N,2] f32 keypoints in the image to be warped
    dst: np.ndarray          # [N,2] f32 matched keypoints in the centre image
    h_gt: np.ndarray         # [3,3] f64
    final_w: int
    final_h: int
    offset_x: int
    offset_y: int
    mesh: np.ndarray         # [2, mesh_cells+1] f64 cell edges
    vertices: np.ndarray     # [mesh_cells, mesh_cells, 2] f64 anchors
    gamma: float = GAMMA
    sigma: float = SIGMA

    @property
    def n_cells(self) -> int:
        return self.mesh_cells * self.mesh_cells

    @property
    def canvas_px(self) -> int:
        return int(self.final_w) * int(self.final_h)

    def image(self, seed: int = 1) -> np.ndarray:
        return make_image(self.width, self.height, seed)


def make_scene(name: str = "c1", seed: int = 0, **override) -> Scene:
    """Build the scene for a named configuration (``override`` replaces width/height/n_kp/mesh)."""
    cfg = dict(CONFIGS[name])
    cfg.update(override)
    w, h, n, mesh = cfg["width"], cfg["height"], cfg["n_kp"], cfg["mesh"]
    src, dst, h_gt = make_keypoints(w, h, n, seed)

    class _Shape:  # final_size only reads .shape
        shape = (h, w, 3)

    fw, fh, ox, oy = (int(v) for v in final_size(_Shape, _Shape, h_gt))
    return Scene(name=name, width=w, height=h, mesh_cells=mesh, src=src, dst=dst, h_gt=h_gt,
                 final_w=fw, final_h=fh, offset_x=ox, offset_y=oy,
                 mesh=get_mesh((fw, fh), mesh + 1),
                 vertices=get_vertice((fw, fh), mesh, (ox, oy)))


def make_pair(name: str):
    """A synthetic pair of the bench shape ``name``: centre image, the other view warped by the scene's homography,
    centre keypoints and their (noisy) images in the other view."""
    import cv2 as cv

    sc = make_scene(name)
    rng = np.random.default_rng(1)
    img_c = make_image(sc.width, sc.height, seed=2)
    hinv = np.linalg.inv(sc.h_gt)
    img_o = cv.warpPerspective(img_c, hinv, (sc.width, sc.height))
    raw_c = sc.dst.astype(np.float32)
    raw_o = cv.perspectiveTransform(raw_c[None].astype(np.float64), hinv)[0].astype(np.float32)
    keep = np.all((raw_o > 8) & (raw_o < [sc.width - 8, sc.height - 8]) & (raw_c > 8) & (raw_c < [sc.width - 8, sc.height - 8]),
                  axis=1)
    raw_c, raw_o = raw_c[keep], raw_o[keep]
    raw_o = raw_o + rng.normal(0, 0.3, raw_o.shape).astype(np.float32)
    return img_c, img_o, raw_c, raw_o


def make_case(name: str, k: int):
    """A centre image of the bench shape ``name`` and ``k`` others warped from it by different homographies (rotation,
    shift, a little perspective), with the centre keypoints and their noisy images in each other view."""
    import cv2 as cv

    cfg = CONFIGS[name]
    w, h = cfg["width"], cfg["height"]
    centre = make_image(w, h, seed=2)
    r = np.random.default_rng(5)
    raw_c = (r.random((cfg["n_kp"], 2)) * [w - 48, h - 48] + 24).astype(np.float32)
    others, raw_os = [], []
    for j in range(k):
        a = 0.015 * (j + 1) * (-1) ** j
        hom = np.array([[np.cos(a), -np.sin(a), 0.02 * w * (j + 1)], [np.sin(a), np.cos(a), -0.015 * h * (j + 1)],
                        [2e-6 * (j + 1), -3e-6 * j, 1.0]])
        hinv = np.linalg.inv(hom)
        others.append(cv.warpPerspective(centre, hinv, (w, h)))
        raw_o = cv.perspectiveTransform(raw_c[None].astype(np.float64), hinv)[0].astype(np.float32)
        raw_os.append(raw_o + r.normal(0, 0.3, raw_o.shape).astype(np.float32))
    return centre, others, raw_c, raw_os
