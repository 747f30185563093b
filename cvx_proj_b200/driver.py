"""The reference's APAP driver (``pyviz/apap.py:220-265``, its ``__main__`` block) as functions.

The reference script has no function for what it does after ``local_homography``: the per-cell
inverse + ``/[2, 2]`` + column-major ``[cells, 9]`` float64 layout of the ``.mat`` product
(``:250-265``), and -- commented out -- the warp / paste / blend that makes the stitched image
(``:258-262``).  A caller that switches packages needs both, so they live here:

  ``mat_layout``      pyviz/apap.py:250-254,263-264   (in place on the caller's grid, like the script)
  ``save2mat``        pyviz/utils.py:68-70
  ``stitch_pair``     pyviz/apap.py:238-265           (grid, H field, ``.mat`` matrix, stitched image)
  ``stitch_case``     run_all.sh:15,29                (every image of a case against the centre, from raw keypoints)
  ``stitch_panorama`` (no reference counterpart)      (the same, blended into one panorama of the case)

The keypoint-pair producer (``visualize_feature_pairs``) and the dataset IO stay with the caller
(SURVEY.md section 8f, rows N3/N4): ``stitch_pair`` starts where the script has its matched
keypoints and its two images.
"""
from __future__ import annotations

from typing import NamedTuple, Optional

import numpy as np

from .apap_utils import final_size, get_mesh, get_vertice

__all__ = ["mat_layout", "save2mat", "stitch_pair", "stitch_case", "StitchResult", "panorama_size", "stitch_panorama",
           "PanoramaResult"]


def mat_layout(local_homography: np.ndarray, stitcher=None) -> np.ndarray:
    """``[mesh_y, mesh_x, 3, 3]`` float32 grid -> the ``[cells, 9]`` float64 matrix the script saves.

    Like the script (pyviz/apap.py:250-254) it first replaces every cell of ``local_homography``
    IN PLACE by its float32 inverse divided by its last entry; one stacked ``np.linalg.inv`` is the
    same LAPACK call per 3x3 block as the reference's loop (bit-identical, tests).  Then
    ``transpose(0, 1, 3, 2)`` (column-major 3x3, what the MATLAB evaluator reads), float64,
    ``reshape(-1, 9)`` (pyviz/apap.py:263-264).  With ``stitcher`` (an ``APAP``) the inverse runs on its GPU
    (``APAP.invert_grid``: same bits, 10 ms less at 40 000 cells).
    """
    if stitcher is not None:
        stitcher.invert_grid(local_homography)
    else:
        local_homography[...] = np.linalg.inv(local_homography)
    local_homography /= local_homography[..., -1:, -1:].copy()
    return local_homography.transpose(0, 1, 3, 2).astype(np.float64).reshape(-1, 9)


def save2mat(path: str, arr: np.ndarray, name: str = "sift_feature", prefix: str = "./output/") -> str:
    """``scipy.io.savemat(f"{prefix}{path}.mat", {name: arr})`` (pyviz/utils.py:68-70); returns the file name.
    The script calls it as ``save2mat(f"case{c}/H3{i}_apap", H, name='H', prefix="../diff_1/results/")``."""
    import scipy.io

    mat_file_path = f"{prefix}{path}.mat"
    scipy.io.savemat(mat_file_path, {name: arr})
    return mat_file_path


class StitchResult(NamedTuple):
    final_size: tuple            # (final_w, final_h, offset_x, offset_y)   pyviz/apap.py:238
    mesh: np.ndarray             # [2, mesh_size + 1] float64 cell edges      :239
    vertices: np.ndarray         # [mesh_size, mesh_size, 2] float64 anchors  :240
    local_homography: np.ndarray  # [mesh, mesh, 3, 3] float32 as returned by APAP.local_homography   :242
    mat: np.ndarray              # [cells, 9] float64, the matrix the script saves under 'H'        :263-265
    stitched: Optional[np.ndarray]  # [final_h, final_w, 3] uint8 blend of the warped and the centre image, or None


def stitch_pair(center_img, other_img, final_src, final_dst, project_h, *, mesh_size: int = 100, gamma=0.5,
                sigma=100, warp_img=None, blend_img=None, stitch: bool = True, device=None) -> StitchResult:
    """One pass of the script from its matched keypoints on (pyviz/apap.py:238-265).

    ``center_img`` / ``other_img`` size the canvas (``final_size``), ``final_src`` / ``final_dst`` are the
    matched keypoints (other image, centre image) and ``project_h`` the global homography, all as
    ``visualize_feature_pairs(..., swap=True)`` returns them.  ``warp_img`` / ``blend_img`` are the
    images that get warped and pasted (the script uses the de-hazed pair, ``:245``; default: the same
    two images).  With ``stitch`` the commented pipeline runs too: warp the other image through the
    per-cell homographies, paste the centre image at the offsets, ``uniform_blend`` -- one fused kernel.
    """
    from .apap import APAP

    final_w, final_h, offset_x, offset_y = final_size(center_img, other_img, project_h)
    mesh = get_mesh((final_w, final_h), mesh_size + 1)
    vertices = get_vertice((final_w, final_h), mesh_size, (offset_x, offset_y))
    stitcher = APAP(gamma, sigma, [final_w, final_h], [offset_x, offset_y], device=device)
    local_h, _ = stitcher.local_homography(final_src, final_dst, vertices)
    mat = mat_layout(local_h.copy(), stitcher)
    stitched = None
    if stitch:
        # The script's commented lines (:258-261) would hand local_warp the grid it has just inverted for the
        # .mat product, and local_warp inverts its argument again (:201-203).  Here the warp gets the grid as
        # local_homography returned it -- canvas pixel -> inv(H_cell) -> pixel of the other image -- which is
        # the call `stitcher.local_warp(other_img, local_homography, mesh)` made right after :242.
        warp_img = other_img if warp_img is None else warp_img
        blend_img = center_img if blend_img is None else blend_img
        stitched = stitcher.local_warp_blend(warp_img, local_h.copy(), mesh, blend_img)
    return StitchResult((final_w, final_h, offset_x, offset_y), mesh, vertices, local_h, mat, stitched)


def stitch_case(center_img, other_imgs, raw_kpts_cp, raw_kpts_ops, *, mesh_size: int = 100, gamma=0.5, sigma=100,
                warp_imgs=None, blend_img=None, stitch: bool = True, equalize: bool = True, ransac: str = "opencv",
                device=None) -> list:
    """The reference's multi-image mode for one centre: ``pyviz/apap.py <case> <img>`` for every other image of a case
    (run_all.sh:15,29), from the images and raw keypoints to one ``StitchResult`` per other image.  Element ``i`` is
    field for field, bit for bit ``stitch_pair(center_img, other_imgs[i], *keypoint_pairs(center_img, other_imgs[i],
    kc_i, raw_kpts_ops[i], equalize=equalize, ransac=ransac), ...)`` with ``warp_img=warp_imgs[i]``; ``raw_kpts_cp``
    is one array for all pairs or a list with one per pair (``utils.keypoint_pairs_batch``).

    The keypoint pairs come from ``keypoint_pairs_batch`` (the centre uploaded and described once, one RANSAC batch
    with ``ransac="gpu"``), and the warp and blend read the images the producer already holds on the device: without
    ``warp_imgs`` / ``blend_img`` each image crosses PCIe once.  The moving DLT runs per pair (``local_homography``):
    ``local_homography_batch`` pads every pair to the largest keypoint count, which changes the Gram kernel's split
    plan, so a smaller pair's grid could differ from ``stitch_pair``'s in the last bits.  ``warp_imgs`` (one per pair) and ``blend_img`` (one for all) are the de-hazed images the script warps
    and pastes (pyviz/apap.py:245); each is uploaded once.  ``stitched`` comes back as a numpy array.  The ``.mat`` and
    keypoint files stay with the caller, as for ``stitch_pair``."""
    from . import _runtime as rt
    from .utils import _device_image

    if warp_imgs is not None and len(warp_imgs) != len(other_imgs):
        raise ValueError(f"stitch_case: {len(other_imgs)} other images but {len(warp_imgs)} warp images")
    front = _case_front(center_img, other_imgs, raw_kpts_cp, raw_kpts_ops, mesh_size, gamma, sigma, equalize, ransac,
                        device)
    if front is None:
        return []
    centre_dev, other_devs, stitchers, meshes, vertices, grids = front
    torch, device = rt.torch_cuda(centre_dev.device)
    if stitch:
        warp_devs = other_devs if warp_imgs is None else [_device_image(torch, device, img) for img in warp_imgs]
        blend_dev = centre_dev if blend_img is None else _device_image(torch, device, blend_img)
    results = []
    for i, (st, local_h) in enumerate(zip(stitchers, grids)):
        mat = mat_layout(local_h.copy(), st)
        stitched = None
        if stitch:
            # the grid as local_homography returned it, as in stitch_pair
            stitched = rt.to_host(torch, st.local_warp_blend(warp_devs[i], local_h.copy(), meshes[i], blend_dev))
        results.append(StitchResult((st.final_width, st.final_height, st.offset_x, st.offset_y), meshes[i],
                                    vertices[i], local_h, mat, stitched))
    return results


def _case_front(center_img, other_imgs, raw_kpts_cp, raw_kpts_ops, mesh_size, gamma, sigma, equalize, ransac, device):
    """What ``stitch_case`` and ``stitch_panorama`` share: the keypoint pairs of every other image against the centre
    (``_keypoint_pairs_uploaded``), then per pair its canvas, mesh, anchors and grid.  ``None`` without other images,
    else ``(centre device tensor, [other device tensors], [APAP], [mesh], [vertices], [grid])``."""
    from . import _runtime as rt
    from .apap import APAP
    from .utils import _keypoint_pairs_uploaded

    pairs, centre_dev, other_devs = _keypoint_pairs_uploaded(center_img, other_imgs, raw_kpts_cp, raw_kpts_ops,
                                                              equalize, device, ransac)
    if not pairs:
        return None
    _, device = rt.torch_cuda(centre_dev.device)
    stitchers, meshes, vertices = [], [], []
    for other_img, (_, _, project_h) in zip(other_imgs, pairs):
        final_w, final_h, offset_x, offset_y = final_size(center_img, other_img, project_h)
        meshes.append(get_mesh((final_w, final_h), mesh_size + 1))
        vertices.append(get_vertice((final_w, final_h), mesh_size, (offset_x, offset_y)))
        stitchers.append(APAP(gamma, sigma, [final_w, final_h], [offset_x, offset_y], device=device))
    # per pair, not local_homography_batch: a batch pads every pair to the largest keypoint count, and the Gram
    # kernel's split plan follows that count, so a smaller pair's grid can differ from its single call in the last bits
    grids = [st.local_homography(p[0], p[1], v)[0] for st, p, v in zip(stitchers, pairs, vertices)]
    return centre_dev, other_devs, stitchers, meshes, vertices, grids


def panorama_size(final_sizes):
    """The panorama canvas of a case from its pairs' ``final_size`` tuples ``(W_k, H_k, ox_k, oy_k)``: pair k's canvas
    covers ``[-ox_k, W_k - ox_k) x [-oy_k, H_k - oy_k)`` in centre coordinates, and the panorama is the union of those
    rectangles.  Returns ``((W, H, OX, OY), origins)``: the centre lies at ``(OX, OY)`` of the panorama and pair k's
    canvas at ``origins[k] = (OX - ox_k, OY - oy_k)`` (int64 ``[K, 2]``).  For one pair this is its own ``final_size``
    with origin ``(0, 0)``.  Host arithmetic."""
    fs = np.asarray(final_sizes, dtype=np.int64).reshape(-1, 4)
    if len(fs) == 0:
        raise ValueError("panorama_size: at least one final_size")
    ox, oy = int(fs[:, 2].max()), int(fs[:, 3].max())
    width = int((fs[:, 0] - fs[:, 2]).max()) + ox
    height = int((fs[:, 1] - fs[:, 3]).max()) + oy
    origins = np.stack([ox - fs[:, 2], oy - fs[:, 3]], axis=1)
    return (width, height, ox, oy), origins


class PanoramaResult(NamedTuple):
    final_size: tuple        # (W, H, OX, OY): the panorama canvas, the centre at (OX, OY)
    origins: np.ndarray      # [K, 2] int64 top-left panorama position of each pair's canvas
    pairs: list              # one StitchResult per other image, stitched = None (stitch_case(..., stitch=False))
    panorama: np.ndarray     # [H, W, 3] uint8


def stitch_panorama(center_img, other_imgs, raw_kpts_cp, raw_kpts_ops, *, mesh_size: int = 100, gamma=0.5, sigma=100,
                    warp_imgs=None, blend_img=None, equalize: bool = True, ransac: str = "opencv",
                    device=None, blend: str = "mean", sharpness=0.02, exposure: str = "none",
                    bands: int = 5) -> PanoramaResult:
    """Every image of a case stitched against the centre into ONE panorama (the reference has no multi-image blend;
    ``stitch_case`` returns one two-image canvas per pair, each in a frame of its own).

    ``pairs[i]`` is ``stitch_case(..., stitch=False)[i]`` field for field.  Every pair's grid maps its canvas into the
    centre's frame, so the panorama is the union of the pair canvases (``panorama_size``) with
      - layer k: ``APAP.local_warp(warp_imgs[k], grid_k, mesh_k)`` on pair k's own canvas (nearest, as the reference),
        placed at ``origins[k]`` -- not re-warped on a union mesh, the cell lookup belongs to the pair canvas;
      - the centre layer: ``blend_img`` (default ``center_img``) at ``(OX, OY)``;
    blended by ``utils.blend_layers``: per pixel the floor mean of the non-empty layers.  With one other image the
    panorama is ``stitch_pair(...).stitched`` bit for bit; with none it is the centre image itself (``pairs == []``).

    ``blend="feather"`` blends the same layers in the same order (the others, then the centre) by
    ``utils.feather_blend(..., sharpness)``, OpenCV's ``FeatherBlender``: each layer's weight ramps up from its
    boundary over about ``1 / sharpness`` pixels, so the seams along the layers' edges fade.  Every field but
    ``panorama`` is the mean call's.  With no other image the panorama is ``feather_blend([centre])``, the centre less
    1 where it is non-empty (OpenCV's ``trunc(v / 1.00001)``).  ``sharpness`` is used by ``"feather"`` only.

    ``blend="multiband"`` blends the same layers in the same order by ``utils.multiband_blend(..., bands)``, OpenCV's
    ``MultiBandBlender`` with int16 weights (``cv.detail_MultiBandBlender(0, bands, cv.CV_16S)``), the blender
    OpenCV's stitcher runs by default: each Laplacian band is blended over a width matched to its scale, so low
    frequencies mix over a wide seam while edges switch over a few pixels.  Every field but ``panorama`` is the mean
    call's.  With no other image the panorama is ``multiband_blend([centre])``.  ``bands`` is used by
    ``"multiband"`` only.

    ``exposure="gain"`` evens out the brightness of the layers before any blend, as OpenCV's stitching pipeline
    runs ``cv.detail.GainCompensator`` in front of its blender: ``utils.exposure_gains`` over the same layers in the
    same order gives one gain per layer, and the blend gets them (``gains=``), compensating each layer's bytes while
    keeping its original mask.  With no other image it equals ``"none"``.  The gains are not part of the result; a
    caller who wants them calls ``exposure_gains`` on the layers.

    The layers are warped from the images the keypoint-pair producer already holds on the device and stay there; one
    blend call and one download make the panorama.  At most 255 other images (127 with ``"feather"``, 126 with
    ``"multiband"``); an unknown ``blend``, an unknown ``exposure``, too many images, a ``sharpness`` that
    ``feather_blend`` refuses for every canvas or (with ``"multiband"``) a ``bands`` that ``multiband_blend`` refuses
    raise ``ValueError`` before any keypoint work."""
    from . import _runtime as rt
    from .utils import (_device_image, _feather_sharpness, _multiband_bands, blend_layers, exposure_gains,
                        feather_blend, multiband_blend)

    if blend not in ("mean", "feather", "multiband"):
        raise ValueError(f"stitch_panorama: blend must be 'mean', 'feather' or 'multiband', got {blend!r}")
    if exposure not in ("none", "gain"):
        raise ValueError(f"stitch_panorama: exposure must be 'none' or 'gain', got {exposure!r}")
    if warp_imgs is not None and len(warp_imgs) != len(other_imgs):
        raise ValueError(f"stitch_panorama: {len(other_imgs)} other images but {len(warp_imgs)} warp images")
    max_layers = {"mean": rt.BLEND_MAX_LAYERS, "feather": rt.FEATHER_MAX_LAYERS,
                  "multiband": rt.MULTIBAND_MAX_LAYERS}[blend]
    if len(other_imgs) >= max_layers:
        raise ValueError(f"stitch_panorama: at most {max_layers - 1} other images with blend={blend!r}, "
                         f"got {len(other_imgs)}")
    if blend == "feather":
        sharpness = _feather_sharpness("stitch_panorama", sharpness)

        def blend_fn(layers, origins, size, device=None, gains=None):
            return feather_blend(layers, origins, size, sharpness, device=device, gains=gains)
    elif blend == "multiband":
        bands = _multiband_bands("stitch_panorama", bands)

        def blend_fn(layers, origins, size, device=None, gains=None):
            return multiband_blend(layers, origins, size, bands, device=device, gains=gains)
    else:
        blend_fn = blend_layers
    front = _case_front(center_img, other_imgs, raw_kpts_cp, raw_kpts_ops, mesh_size, gamma, sigma, equalize, ransac,
                        device)
    centre = center_img if blend_img is None else blend_img
    if front is None:
        h, w = centre.shape[0], centre.shape[1]
        pano = blend_fn([centre], [(0, 0)], (w, h), device=device)
        if not isinstance(pano, np.ndarray):
            pano = rt.to_host(rt.torch_cuda(pano.device)[0], pano)
        return PanoramaResult((int(w), int(h), 0, 0), np.zeros((0, 2), np.int64), [], pano)
    centre_dev, other_devs, stitchers, meshes, vertices, grids = front
    torch, device = rt.torch_cuda(centre_dev.device)
    warp_devs = other_devs if warp_imgs is None else [_device_image(torch, device, img) for img in warp_imgs]
    blend_dev = centre_dev if blend_img is None else _device_image(torch, device, blend_img)
    pairs, layers = [], []
    for i, (st, local_h) in enumerate(zip(stitchers, grids)):
        mat = mat_layout(local_h.copy(), st)
        pairs.append(StitchResult((st.final_width, st.final_height, st.offset_x, st.offset_y), meshes[i], vertices[i],
                                  local_h, mat, None))
        # the grid as local_homography returned it, as stitch_pair hands it to the fused warp
        layers.append(st.local_warp(warp_devs[i], local_h.copy(), meshes[i]))
    (width, height, ox, oy), origins = panorama_size([p.final_size for p in pairs])
    layers, places = layers + [blend_dev], [tuple(o) for o in origins] + [(ox, oy)]
    if exposure == "gain":
        pano = blend_fn(layers, places, (width, height), gains=exposure_gains(layers, places, (width, height)))
    else:
        pano = blend_fn(layers, places, (width, height))
    return PanoramaResult((width, height, ox, oy), origins, pairs, rt.to_host(torch, pano))
