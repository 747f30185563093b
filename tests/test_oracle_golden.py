"""The oracle (oracle/apap_oracle.py) against the golden vectors produced by the live
reference (oracle/gen_golden.py).  CPU only."""
import hashlib
import zlib

import numpy as np
import pytest

from cvx_proj_b200 import synth
from oracle import apap_oracle as orc


@pytest.mark.parametrize("name", ["tiny", "mini"])
def test_host_pieces_bit_exact(golden, name):
    g = golden(f"ref_{name}.npz")
    src, dst = g["src"], g["dst"]
    n1, nf1 = orc.normalize_2d_pts(src)
    n2, nf2 = orc.normalize_2d_pts(dst)
    c1, c2 = orc.conditioner_from_pts(nf1), orc.conditioner_from_pts(nf2)
    cf1, cf2 = orc.point_normalize(nf1, c1), orc.point_normalize(nf2, c2)
    aa = orc.matrix_generate(src.shape[0], cf1, cf2)
    for got, key in ((n1, "N1"), (n2, "N2"), (nf1, "nf1"), (nf2, "nf2"), (c1, "C1"), (c2, "C2"),
                     (cf1, "cf1"), (cf2, "cf2"), (aa, "A")):
        assert got.dtype == g[key].dtype, key
        assert np.array_equal(got, g[key]), key


@pytest.mark.parametrize("name", ["tiny", "mini"])
def test_canvas_helpers_bit_exact(golden, name):
    g = golden(f"ref_{name}.npz")
    sc = synth.make_scene(name)
    assert np.array_equal(sc.src, g["src"]) and np.array_equal(sc.dst, g["dst"])  # generator is pinned too
    fs = orc.final_size((sc.height, sc.width, 3), (sc.height, sc.width, 3), g["h_gt"])
    assert [int(v) for v in fs] == list(g["final_size"])
    fw, fh, ox, oy = (int(v) for v in fs)
    assert np.array_equal(orc.get_mesh((fw, fh), sc.mesh_cells + 1), g["mesh"])
    assert np.array_equal(orc.get_vertice((fw, fh), sc.mesh_cells, (ox, oy)), g["vertices"])


@pytest.mark.parametrize("name", ["tiny", "mini"])
def test_local_homography_svd_matches_reference(golden, name):
    g = golden(f"ref_{name}.npz")
    h = orc.local_homography_svd(g["src"], g["dst"], g["vertices"], float(g["gamma"]), float(g["sigma"]))
    assert h.dtype == np.float32
    assert np.array_equal(h, g["H"])          # same calls, same machine image: bit-exact
    w = orc.local_weight(g["src"], g["vertices"], float(g["gamma"]), float(g["sigma"]))
    assert np.array_equal(w, g["W"])


def test_clamped_weights_case(golden):
    g = golden("ref_tiny_sigma8.npz")
    t = golden("ref_tiny.npz")
    h = orc.local_homography_svd(t["src"], t["dst"], t["vertices"], 0.5, 8.0)
    assert np.array_equal(h, g["H"])
    w = orc.local_weight(t["src"], t["vertices"], 0.5, 8.0)
    assert np.array_equal(w, g["W"]) and (w == 0.5).mean() > 0.5


@pytest.mark.parametrize("name", ["tiny", "mini"])
def test_gram64_agrees_with_reference(golden, name):
    g = golden(f"ref_{name}.npz")
    h = orc.local_homography_gram64(g["src"], g["dst"], g["vertices"], float(g["gamma"]), float(g["sigma"]))
    fw = int(g["final_size"][0]); fh = int(g["final_size"][1])
    err = orc.h_error_normalised(h, g["H"], max(fw, fh))
    assert err.max() < 2e-6, err.max()


def test_gram64_c1_and_c2_spot(golden):
    g = golden("ref_c1.npz")
    sc = synth.make_scene("c1")
    assert hashlib.sha256(sc.src.tobytes() + sc.dst.tobytes()).hexdigest() == str(g["src_sha"])
    h = orc.local_homography_gram64(sc.src, sc.dst, sc.vertices, sc.gamma, sc.sigma)
    err = orc.h_error_normalised(h, g["H"], max(sc.final_w, sc.final_h))
    assert err.max() < 2e-6, err.max()
    s = golden("ref_c2_spot.npz")
    sc2 = synth.make_scene("c2")
    assert hashlib.sha256(sc2.src.tobytes() + sc2.dst.tobytes()).hexdigest() == str(s["src_sha"])
    sub = sc2.vertices[s["rows"]][:, s["cols"]]
    h2 = orc.local_homography_gram64(sc2.src, sc2.dst, sub, sc2.gamma, sc2.sigma)
    err2 = orc.h_error_normalised(h2, s["H"], max(sc2.final_w, sc2.final_h))
    assert err2.max() < 2e-6, err2.max()


@pytest.mark.parametrize("name", ["tiny", "mini"])
def test_warp_and_blend_bit_exact(golden, name):
    g = golden(f"ref_{name}.npz")
    sc = synth.make_scene(name)
    img = sc.image(1)
    inv = orc.invert_grid(g["H"])
    assert np.array_equal(inv, g["H_inverted_in_place"])      # stacked inv == the reference's loop
    fw, fh, ox, oy = (int(v) for v in g["final_size"])
    warped = orc.local_warp(img, inv, g["mesh"], (fw, fh), (ox, oy))
    assert np.array_equal(warped, g["warped"])
    centre = synth.make_image(sc.width, sc.height, seed=2)
    pasted = orc.paste_centre(warped, centre, (ox, oy))
    assert np.array_equal(orc.uniform_blend(warped, pasted), g["blended"])
    assert np.array_equal(orc.uniform_blend_float(warped, pasted), g["blended"])
    assert np.array_equal(orc.mat_layout(g["H"]), g["mat"])


def test_warp_loop_equals_vectorised(golden):
    g = golden("ref_tiny.npz")
    sc = synth.make_scene("tiny")
    img = sc.image(1)
    inv = orc.invert_grid(g["H"])
    fw, fh, ox, oy = (int(v) for v in g["final_size"])
    a = orc.local_warp_loop(img, inv, g["mesh"], (fw, fh), (ox, oy))
    assert np.array_equal(a, g["warped"])


def test_warp_c1_rows(golden):
    g = golden("ref_c1.npz")
    sc = synth.make_scene("c1")
    img = sc.image(1)
    assert hashlib.sha256(img.tobytes()).hexdigest() == str(g["img_sha"])
    inv = orc.invert_grid(g["H"])
    assert np.array_equal(inv, g["H_inverted_in_place"])
    warped = orc.local_warp(img, inv, sc.mesh, (sc.final_w, sc.final_h), (sc.offset_x, sc.offset_y))
    crc = np.array([zlib.crc32(np.ascontiguousarray(r).tobytes()) for r in warped], dtype=np.uint32)
    assert np.array_equal(crc, g["warped_row_crc"])
    assert hashlib.sha256(warped.tobytes()).hexdigest() == str(g["warped_sha"])


def test_blend_edge_cases(golden):
    g = golden("ref_blend.npz")
    assert np.array_equal(orc.uniform_blend(g["a"], g["b"]), g["out"])
    assert np.array_equal(orc.uniform_blend_float(g["a"], g["b"]), g["out"])


# ------------------------------------------------------------- global-homography warp (SURVEY 8f, N4)
def test_image_warping_oracle_reproduces_live_reference(golden):
    """oracle/warp_oracle.py (OpenCV's fixed-point bilinear warp restated) against outputs of the live reference's
    utils.image_warping (oracle/gen_golden_warping.py), both blend modes, odd sizes."""
    import hashlib
    from oracle import warp_oracle as wo
    from oracle.gen_golden_warping import CASES, FULL, warping_case
    g = golden("ref_image_warping.npz")
    for name in CASES:
        base, warp, hmat = warping_case(name)
        assert np.array_equal(hmat, g[name + "_H"])
        for db in (True, False):
            tag = f"{name}_{'paste' if db else 'mean'}"
            res = wo.image_warping(base, warp, hmat, direct_blend=db)
            assert tuple(g[tag + "_shape"]) == res.shape
            assert hashlib.sha256(res.tobytes()).hexdigest() == str(g[tag + "_sha"]), tag
            if name in FULL:
                assert np.array_equal(res, g[tag])


def test_spectral_oracle_reproduces_live_reference(golden):
    """oracle/spectral_oracle.py against outputs of the live reference's calculate_M (oracle/gen_golden_spectral.py).
    The segment is |U[:, 0]| of LAPACK's SVD, whose last bits depend on the CPU (OpenBLAS picks its kernels at run
    time) and on the thread count: it is held to 1e-12 of the reference's (the GPU path's gate is 1e-10), the ransac
    mask (float32 copies of segment entries) as in the GPU test, the original mask bit for bit."""
    from oracle import spectral_oracle as so
    from oracle.gen_golden_spectral import CASES, OPTS, spectral_case
    g = golden("ref_spectral.npz")
    for name in ("s40", "s300", "s1000"):
        c, o, cf, of, fmat, hg = spectral_case(name)
        seg, rmask, omask = so.calculate_m(c, o, cf, of, fmat, hg, **OPTS)
        err = np.abs(seg - g[name + "_segment"]).max()
        print(f"{name}: max |segment - reference| = {err:.2e}")
        assert seg.dtype == np.float64 and seg.shape == g[name + "_segment"].shape and err <= 1e-12
        assert np.allclose(rmask, g[name + "_ransac_mask"], rtol=0, atol=1e-7)
        assert np.array_equal(omask, g[name + "_original_mask"])
    assert set(CASES) == {"s40", "s300", "s1000", "s2500"}


def test_match_oracle_equals_live_bfmatcher():
    """oracle/match_oracle.exact_match is pinned against OpenCV's own exact matcher (the dependency the reference's
    matcher step lives in): same train index and distance bits on SIFT-like integer descriptors, ties included."""
    cv = pytest.importorskip("cv2")
    from oracle import match_oracle as mo
    rng = np.random.default_rng(5)
    for nq, nt in ((1, 1), (40, 17), (300, 900)):
        t = np.minimum(np.rint(rng.gamma(0.6, 40.0, size=(nt, 128))), 255).astype(np.float32)
        q = np.clip(t[rng.integers(0, nt, size=nq)] + rng.integers(-5, 6, size=(nq, 128)), 0, 255).astype(np.float32)
        if nt > 4:
            t[nt - 1] = t[2]; q[0] = t[2]
        idx, dist = mo.exact_match(q, t)
        bf = cv.BFMatcher(cv.NORM_L2).match(q, t)
        assert np.array_equal(idx, [m.trainIdx for m in bf])
        assert np.array_equal(dist.view(np.uint32), np.array([m.distance for m in bf], np.float32).view(np.uint32))
