"""CPU tests of the host layer: the numpy pieces kept bit-identical to the reference, the
kernel-input builders, the guard-band logic of the warp's float32 fast path (emulated in numpy),
the C-ABI library (loads, exports every declared symbol) and the no-fallback rule."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

from cvx_proj_b200 import _runtime as rt
from cvx_proj_b200 import apap as papap
from cvx_proj_b200 import apap_utils, sharding, synth
from cvx_proj_b200.apap import APAP
from oracle import apap_oracle as orc

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("name", ["tiny", "mini"])
def test_static_methods_bit_exact_vs_reference(golden, name):
    g = golden(f"ref_{name}.npz")
    n1, nf1 = APAP.getNormalize2DPts(g["src"])
    n2, nf2 = APAP.getNormalize2DPts(g["dst"])
    c1, c2 = APAP.getConditionerFromPts(nf1), APAP.getConditionerFromPts(nf2)
    cf1, cf2 = APAP.point_normalize(nf1, c1), APAP.point_normalize(nf2, c2)
    dlt = APAP.matrix_generate(g["src"].shape[0], cf1, cf2)
    for got, key in ((n1, "N1"), (n2, "N2"), (nf1, "nf1"), (nf2, "nf2"), (c1, "C1"), (c2, "C2"),
                     (cf1, "cf1"), (cf2, "cf2"), (dlt, "A")):
        assert got.dtype == g[key].dtype and np.array_equal(got, g[key]), key


@pytest.mark.parametrize("name", ["tiny", "mini"])
def test_utils_bit_exact_vs_reference(golden, name):
    g = golden(f"ref_{name}.npz")
    sc = synth.make_scene(name)
    img = np.zeros((sc.height, sc.width, 3), np.uint8)
    assert [int(v) for v in apap_utils.final_size(img, img, g["h_gt"])] == list(g["final_size"])
    fw, fh, ox, oy = (int(v) for v in g["final_size"])
    assert np.array_equal(apap_utils.get_mesh((fw, fh), sc.mesh_cells + 1), g["mesh"])
    assert np.array_equal(apap_utils.get_vertice((fw, fh), sc.mesh_cells, (ox, oy)), g["vertices"])


def test_warp_coordinate_estimate():
    h = np.array([[1.5, 0, 2], [0, 2, -1], [0, 0, 2]], dtype=np.float32)
    out = APAP.warp_coordinate_estimate(np.array([4, 6, 1]), h)
    assert out.dtype == np.float64 and np.array_equal(out, [4.0, 5.5, 1.0])


def test_kp_table_reproduces_weighted_gram(golden):
    g = golden("ref_mini.npz")
    src, dlt = g["src"], g["A"]
    scale = papap.weight_scale(100.0)
    tab = papap.build_kp_table(src, dlt, scale)
    n = src.shape[0]
    assert tab.shape == (256, rt.KP_ROW) and tab.dtype == np.float32
    assert not tab[n:].any()
    assert np.array_equal(tab[:n, 24], tab[:n, 25]) and np.array_equal(tab[:n, 26], tab[:n, 27])
    np.testing.assert_allclose(tab[:n, 24:28:2], src.astype(np.float64) * scale, rtol=6e-8)
    # the kernel's weight 2^-|s v - s x| is the reference's squared weight exp(-|v - x| / sigma^2)^2
    v = g["vertices"][3, 5]
    d = np.hypot(*(papap.scale_anchors(v, scale)[0].astype(np.float64)[:, None] - tab[:n, 24:28:2].T.astype(np.float64)))
    np.testing.assert_allclose(np.maximum(2.0 ** -d, 0.25), g["W"][3, 5] ** 2, rtol=2e-6)
    w = g["W"][3, 5]
    a64 = dlt.astype(np.float64) * np.repeat(w, 2)[:, None]
    want = a64.T @ a64
    got = papap.expand_gram((w[:, None] ** 2 * tab[:n, :24].astype(np.float64)).sum(0))
    assert np.abs(got - want).max() <= 2e-6 * np.abs(want).max()
    assert np.array_equal(got, got.T)


def test_kp_blocks_layout_and_split(golden):
    """Tensor-core table: P = Ph + Pl exactly, Ph is TF32, element (k, n) sits where the MMA's K-major
    core-matrix descriptor (LBO 512 B, SBO 128 B) expects it, coordinates follow."""
    g = golden("ref_mini.npz")
    tab = papap.build_kp_table(g["src"], g["A"], papap.weight_scale(100.0))
    blk = papap.build_kp_blocks(tab)
    n_kb = tab.shape[0] // rt.KP_BLOCK
    assert blk.shape == (n_kb, rt.KP_BLOCK_FLOATS) and blk.dtype == np.float32
    tile = blk[:, :512]
    at = lambda k, m: (k // 4) * 256 + (m // 8) * 32 + (m % 8) * 4 + k % 4        # noqa: E731
    hi_idx = [at(k, n) for k in range(8) for n in range(32)]
    lo_idx = [at(k, 32 + n) for k in range(8) for n in range(32)]
    assert sorted(hi_idx + lo_idx) == list(range(512))
    assert not (tile[:, hi_idx].view(np.uint32) & 0x1FFF).any()        # TF32: low 13 mantissa bits clear
    for kb, k, n in ((0, 0, 0), (3, 5, 17), (7, 7, 23), (11, 2, 8), (24, 4, 5)):
        p = tab[kb * 8 + k, n]
        h, l = tile[kb, at(k, n)], tile[kb, at(k, 32 + n)]
        assert h + l == p and abs(l) <= abs(p) * 2.0 ** -11
    # the 8 padding columns (terms 24..31) are zero in both halves
    pad = [at(k, m) for k in range(8) for m in list(range(24, 32)) + list(range(56, 64))]
    assert not tile[:, pad].any()
    total = tile.astype(np.float64).sum()
    assert total == tab[:, :24].astype(np.float64).sum()
    assert np.array_equal(blk[:, 512:520].ravel(), tab[:, 24]) and np.array_equal(blk[:, 520:528].ravel(), tab[:, 26])


def test_cell_lookup_matches_reference_rule(golden):
    g = golden("ref_mini.npz")
    fw, fh = int(g["final_size"][0]), int(g["final_size"][1])
    mesh = g["mesh"]
    col, row = papap.cell_lookup_tables(mesh, fw, fh, 16, 16)
    assert col.dtype == np.uint16 and row.dtype == np.uint16
    for j in range(fw):
        assert col[j] == np.where(j < mesh[0])[0][0] - 1
    for i in range(fh):
        assert row[i] == np.where(i < mesh[1])[0][0] - 1
    assert np.array_equal(col, orc.cell_lookup(mesh[0], fw)) and np.array_equal(row, orc.cell_lookup(mesh[1], fh))
    with pytest.raises(IndexError):            # canvas wider than the mesh: the reference's [0][0] fails
        papap.cell_lookup_tables(mesh, fw + 5, fh, 16, 16)
    with pytest.raises(IndexError):            # mesh finer than the homography grid
        papap.cell_lookup_tables(mesh, fw, fh, 8, 8)


def _rows_from_blocks(blocks, row_cell, row_first, row0=0):
    """Expand the kernel's row blocks to per-row (cell row, dy) the way the kernel walks them, and
    check the invariants: canvas order, no block crosses a cell row, blocks are full (4 rows) unless
    the whole run is shorter, overlapped rows get the same (cell row, dy) from both blocks."""
    fh = row_cell.shape[0]
    row_lut = np.zeros((fh, 2), dtype=np.uint32)
    seen = np.zeros(fh, dtype=np.int64)
    prev_end, prev_i0 = row0, -1
    for w0, w1 in blocks:
        i0, n, cr, dy0 = int(w0) & 0x0fffffff, int(w0) >> 28, int(w1) & 0xffff, int(w1) >> 16
        assert 1 <= n <= rt.WARP_BLOCK_ROWS and prev_i0 < i0 <= prev_end      # ordered, no gap
        rows = np.arange(i0, i0 + n)
        assert (row_cell[rows] == cr).all() and dy0 == i0 - row_first[cr]
        if n < rt.WARP_BLOCK_ROWS:            # partial only when the run itself is that short
            assert (i0 == 0 or row_cell[i0 - 1] != cr or i0 == row0) and (i0 + n == fh or row_cell[i0 + n] != cr or True)
        dy = np.float32(dy0) + np.arange(n, dtype=np.float32)        # the kernel's dy0 + (float)k
        new = np.stack([np.full(n, cr, np.uint32), dy.astype(np.float32).view(np.uint32)], 1)
        again = seen[rows] > 0
        assert np.array_equal(row_lut[rows][again], new[again])
        row_lut[rows] = new
        seen[rows] += 1
        prev_end, prev_i0 = max(prev_end, i0 + n), i0
    return row_lut, seen


def _emulate_fast_path(fast, col_lut, row_lut, gc, sw, sh, rng):
    """float32 fast path of k_warp (csrc/warp_blend.cu warp_row) in numpy: fma emulated through
    float64 (the product of two float32 is exact there; the double rounding is harmless at these
    magnitudes), rcp.approx emulated as the correctly rounded reciprocal perturbed by +-1 ulp."""
    f32 = np.float32
    cell = row_lut[:, 0].astype(np.int64)[:, None] * gc + col_lut[:, 0].astype(np.int64)[None, :]
    r = fast[cell]                                                            # [fh, fw, 12]
    dx = np.ascontiguousarray(col_lut[:, 1]).view(f32)[None, :]
    dy = np.ascontiguousarray(row_lut[:, 1]).view(f32)[:, None]
    dx, dy = np.broadcast_to(dx, cell.shape), np.broadcast_to(dy, cell.shape)
    fma = lambda a, b, c: (a.astype(np.float64) * b.astype(np.float64) + c.astype(np.float64)).astype(f32)  # noqa
    n0 = fma(r[..., 1], dy, fma(r[..., 0], dx, r[..., 2]))
    n1 = fma(r[..., 4], dy, fma(r[..., 3], dx, r[..., 5]))
    d = fma(r[..., 7], dy, fma(r[..., 6], dx, r[..., 8]))
    with np.errstate(all="ignore"):
        rc = (f32(1) / d).astype(f32)
        pick = rng.random(rc.shape)
        rc = np.where(pick < 0.4, np.nextafter(rc, f32(np.inf)), np.where(pick < 0.8, np.nextafter(rc, f32(-np.inf)), rc))
        qx, qy = (n0 * rc).astype(f32), (n1 * rc).astype(f32)
        flx, fly = np.floor(qx), np.floor(qy)
        fx, fy = (qx - flx).astype(f32), (qy - fly).astype(f32)
        clear = np.maximum(np.abs(fx - f32(0.5)), np.abs(fy - f32(0.5))) <= r[..., 11]
    bits = np.ascontiguousarray(r[..., 9:11]).view(np.int32).astype(np.int64) + 0x4B400000
    ix = np.where(clear, flx, 0).astype(np.int64) + bits[..., 0]
    iy = np.where(clear, fly, 0).astype(np.int64) + bits[..., 1]
    inb = (ix >= 0) & (ix < sw) & (iy >= 0) & (iy < sh)
    outside = r[..., 11] > 1.0                        # the kernel leaves these cells black without arithmetic
    return np.where(inb & ~outside, iy * sw + ix, -1), ~clear & ~outside


def _exact_path(inv_h, col, row, fw, fh, ox, oy, sw, sh):
    h = inv_h[row[:, None], col[None, :]].astype(np.float64)
    x = (np.arange(fw) - ox).astype(np.float64)[None, :]
    y = (np.arange(fh) - oy).astype(np.float64)[:, None]
    t0 = h[..., 0, 0] * x + h[..., 0, 1] * y + h[..., 0, 2]
    t1 = h[..., 1, 0] * x + h[..., 1, 1] * y + h[..., 1, 2]
    t2 = h[..., 2, 0] * x + h[..., 2, 1] * y + h[..., 2, 2]
    with np.errstate(all="ignore"):
        tx, ty = t0 / t2, t1 / t2
    ok = (0 < tx) & (tx < sw) & (0 < ty) & (ty < sh)
    return np.where(ok, np.where(ok, ty, 0).astype(np.int64) * sw + np.where(ok, tx, 0).astype(np.int64), -1)


@pytest.mark.parametrize("name,scale", [("mini", 1.0), ("c1", 1.0), ("mini", 40.0)])
def test_guard_band_makes_fast_path_exact(golden, name, scale):
    """Every pixel the float32 fast path does NOT flag must pick the reference's source pixel."""
    g = golden(f"ref_{name}.npz")
    sc = synth.make_scene(name)
    inv = g["H_inverted_in_place"].copy()
    fw, fh, ox, oy = sc.final_w, sc.final_h, sc.offset_x, sc.offset_y
    sw, sh = sc.width, sc.height
    if scale != 1.0:   # stress: 8K-like magnitudes (coordinates and offsets scaled up)
        s = np.diag([scale, scale, 1.0])
        inv = (s @ inv.astype(np.float64) @ np.linalg.inv(s)).astype(np.float32)
        fw, fh, ox, oy, sw, sh = (int(v * scale) for v in (fw, fh, ox, oy, sw, sh))
        fh = min(fh, 600)
    mesh = apap_utils.get_mesh((fw, fh), sc.mesh_cells + 1)
    col, row = papap.cell_lookup_tables(mesh, fw, fh, sc.mesh_cells, sc.mesh_cells)
    fast, col_lut, row_first = papap.build_warp_tables(inv, col, row, ox, oy, sw, sh)
    row_lut, seen = _rows_from_blocks(papap.build_row_blocks(row, row_first), row, row_first)
    assert (seen >= 1).all() and seen.mean() < 1.2
    assert fast.shape == (sc.mesh_cells ** 2, rt.HINV_ROW) and fast.dtype == np.float32
    assert np.array_equal(col_lut[:, 0], col) and np.array_equal(row_lut[:, 0], row)
    off, flagged = _emulate_fast_path(fast, col_lut, row_lut, sc.mesh_cells, sw, sh, np.random.default_rng(3))
    want = _exact_path(inv, col, row, fw, fh, ox, oy, sw, sh)
    assert np.array_equal(off[~flagged], want[~flagged])
    # cells of the stress case are ~750 px wide (quotients up to +-370), typical cells are 10-40 px
    assert flagged.mean() < (2e-4 if scale == 1.0 else 1e-2), flagged.mean()
    assert (want >= 0).mean() > 0.3        # the case does exercise in-bounds pixels
    outside = fast[:, 11] > 1.0            # ... and whole cells outside the source image
    assert 0.02 < outside.mean() < 0.6, outside.mean()


def test_guard_band_adversarial_integer_hits():
    """Homographies whose coordinates land exactly on (or within 1e-6 of) integers: the fast path
    must flag every such pixel (identity / integer translation / tiny perturbations of them)."""
    rng = np.random.default_rng(8)
    fw, fh, sw, sh = 640, 200, 600, 180
    mesh = apap_utils.get_mesh((fw, fh), 9)
    col, row = papap.cell_lookup_tables(mesh, fw, fh, 8, 8)
    for trial in range(6):
        inv = np.tile(np.eye(3, dtype=np.float32), (8, 8, 1, 1))
        inv[..., 0, 2] = rng.integers(-5, 6, size=(8, 8))
        inv[..., 1, 2] = rng.integers(-5, 6, size=(8, 8))
        if trial >= 2:
            inv += (rng.standard_normal(inv.shape) * 10.0 ** -(trial + 3)).astype(np.float32)
        fast, col_lut, row_first = papap.build_warp_tables(inv, col, row, 11, 7, sw, sh)
        row_lut, _ = _rows_from_blocks(papap.build_row_blocks(row, row_first), row, row_first)
        off, flagged = _emulate_fast_path(fast, col_lut, row_lut, 8, sw, sh, rng)
        want = _exact_path(inv, col, row, fw, fh, 11, 7, sw, sh)
        assert np.array_equal(off[~flagged], want[~flagged]), trial
        if trial < 2:
            assert flagged.all()


def test_row_blocks_bands_and_odd_luts():
    """Runs are covered by full blocks (overlapping where the run is not a multiple of 4), short runs
    by one partial block; bands of a sharded run get exactly their rows; a lookup table with
    non-monotone cell rows (mesh start > 0 wraps to the last cell) still tiles."""
    row = np.repeat(np.arange(7), [11, 12, 3, 8, 9, 17, 1]).astype(np.uint16)
    first = np.r_[0, np.cumsum([11, 12, 3, 8, 9, 17])]
    g = papap.build_row_blocks(row, first)
    _, seen = _rows_from_blocks(g, row, first)
    assert (seen >= 1).all()
    of = lambda cr: [(int(a) & 0x0fffffff, int(a) >> 28) for a, b in g if (int(b) & 0xffff) == cr]     # noqa: E731
    assert of(0) == [(0, 4), (4, 4), (7, 4)] and of(1) == [(11, 4), (15, 4), (19, 4)] and of(2) == [(23, 3)]
    assert of(3) == [(26, 4), (30, 4)] and of(4) == [(34, 4), (37, 4), (39, 4)] and of(6) == [(60, 1)]
    assert [n for _, n in of(5)] == [4] * 5 and of(5)[0][0] == 43 and of(5)[-1][0] == 56
    band = papap.build_row_blocks(row, first, 20, 45)
    _, seen = _rows_from_blocks(band, row, first, row0=20)
    assert seen[20:45].all() and not seen[:20].any() and not seen[45:].any()
    assert int(band[0, 1]) >> 16 == 20 - 11                            # dy of the band's first row inside cell row 1
    assert papap.build_row_blocks(row, first, 30, 30).shape == (0, 2)
    wrapped = np.r_[np.full(4, 6), row].astype(np.uint16)               # rows 0..3 wrap to the last cell row
    first_w = np.r_[4 + first[:6], 0]
    with pytest.raises(ValueError):                                     # rows before their cell row's origin
        papap.build_row_blocks(np.r_[row, np.full(3, 0)].astype(np.uint16), np.r_[60, first[1:]])
    _, seen = _rows_from_blocks(papap.build_row_blocks(wrapped, first_w), wrapped, first_w)
    assert (seen >= 1).all()


def test_guard_band_degenerate_cells_go_exact():
    inv = np.tile(np.eye(3, dtype=np.float32), (2, 2, 1, 1))
    inv[0, 0, 2] = [0.02, 0.0, -0.5]          # denominator crosses zero inside the cell
    inv[1, 1] = np.nan
    mesh = apap_utils.get_mesh((100, 80), 3)
    col, row = papap.cell_lookup_tables(mesh, 100, 80, 2, 2)
    fast, _, _ = papap.build_warp_tables(inv, col, row, 0, 0, 64, 64)
    fast = fast.reshape(2, 2, -1)
    assert fast[0, 0, 11] == -1.0 and fast[1, 1, 11] == -1.0
    assert np.isfinite(fast[..., :9]).all() and (fast[0, 0, 8] == 1.0) and (fast[1, 1, 8] == 1.0)
    assert 0.499 < fast[0, 1, 11] < 0.5 and 0.499 < fast[1, 0, 11] < 0.5


def test_gram_plan_depends_only_on_keypoints():
    seen = {}
    for engine, longest in ((rt.GRAM_FFMA2, 1024), (rt.GRAM_TCGEN05, 2048)):
        for cells in (64, 10_000, 40_000, 160_000):
            for n_pad in (128, 512, 2048, 5120, 20096, 65536):
                ks, cp, nb = rt.gram_plan(cells, n_pad, engine)
                assert seen.setdefault((engine, n_pad), ks) == ks   # same split structure however the grid is sharded
                assert cp >= cells and cp % 512 == 0 and nb == ks * 24 * cp * 4
                assert -(-n_pad // ks) <= longest + 128       # FFMA2: FP32 chains stay <= 1024 keypoints (+ chunk rounding)
    assert rt.gram_plan(160_000, 20096, rt.GRAM_TCGEN05)[0] < rt.gram_plan(160_000, 20096, rt.GRAM_FFMA2)[0]
    with pytest.raises(rt.ApapError):
        rt.gram_plan(10, 100)                                # not a multiple of the chunk
    with pytest.raises(rt.ApapError):
        rt.gram_plan(10, 128, 7)                             # unknown engine


def test_library_exports_every_declared_symbol():
    lib = rt.load_library()
    header = open(os.path.join(REPO, "include", "apap_b200.h")).read()
    declared = set(re.findall(r"\b(apap_[a-z0-9_]+)\s*\(", header))
    assert declared == set(rt.SIGNATURES), declared ^ set(rt.SIGNATURES)
    raw = ctypes.CDLL(rt.LIB_PATH)
    for name in declared:
        assert hasattr(raw, name), name
    assert lib.apap_abi_version() == rt.ABI_VERSION == 23
    # flag 4 (a fused tile-engine variant up to ABI 22) is refused before any pointer is used: dummy pointers are safe
    d = 256
    assert (lib.apap_warp(d, 1, 1, d, d, d, d, 1, 1, 1, 0, 0, 0, 1, None, 0, 0, d, 3, 4, 0, None, None) == -1   # APAP_E_BADARG
            and b"unknown flag" in lib.apap_last_error())
    m = re.search(r"#define\s+APAP_KP_ROW\s+(\d+)", header)
    assert int(m.group(1)) == rt.KP_ROW


def test_no_cpu_fallback_and_no_oracle_in_product():
    import torch
    if not torch.cuda.is_available():
        st = APAP(0.5, 100, [64, 48], [0, 0])
        sc = synth.make_scene("tiny")
        with pytest.raises(rt.ApapError):
            st.local_homography(sc.src, sc.dst, sc.vertices)
        with pytest.raises(rt.ApapError):
            apap_utils.uniform_blend(np.zeros((4, 4, 3), np.uint8), np.zeros((4, 4, 3), np.uint8))
    pkg = os.path.join(REPO, "cvx_proj_b200")
    for root, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh")):
                text = open(os.path.join(root, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", text, re.M), f
                assert not re.search(r"""["']/root/reference""", text), f     # citations in docstrings are fine


def test_shard_plan_tiles_canvas():
    sc = synth.make_scene("c1")
    col, row = papap.cell_lookup_tables(sc.mesh, sc.final_w, sc.final_h, sc.mesh_cells, sc.mesh_cells)
    for world in (1, 2, 3, 4, 8):
        shards = sharding.plan_shards(row, sc.mesh_cells, world)
        assert shards[0].cell_row0 == 0 and shards[-1].cell_row1 == sc.mesh_cells
        assert shards[0].px_row0 == 0 and shards[-1].px_row1 == sc.final_h
        for a, b in zip(shards, shards[1:]):
            assert a.cell_row1 == b.cell_row0 and a.px_row1 == b.px_row0
        for s in shards:
            assert set(np.unique(row[s.px_row0:s.px_row1])) <= set(range(s.cell_row0, s.cell_row1))
        sizes = [s.n_cell_rows for s in shards]
        assert max(sizes) - min(sizes) <= 1


_GLOO_WORKER = r"""
import os, sys
sys.path.insert(0, {repo!r})
import numpy as np, torch, torch.distributed as dist
from cvx_proj_b200 import sharding, synth
from cvx_proj_b200.apap import cell_lookup_tables
dist.init_process_group("gloo")
rank, world = dist.get_rank(), dist.get_world_size()
sc = synth.make_scene("mini")
col, row = cell_lookup_tables(sc.mesh, sc.final_w, sc.final_h, sc.mesh_cells, sc.mesh_cells)
shards = sharding.plan_shards(row, sc.mesh_cells, world)
rng = np.random.default_rng(5)
full = rng.integers(0, 256, size=(sc.final_h, sc.final_w, 3), dtype=np.uint8)     # same on every rank
me = shards[rank]
band = torch.from_numpy(full[me.px_row0:me.px_row1].copy())
pano = sharding.gather_bands(band, shards, sc.final_w)
assert pano.shape == (sc.final_h, sc.final_w, 3), pano.shape
assert np.array_equal(pano.numpy(), full)
dist.barrier()
dist.destroy_process_group()
print("rank", rank, "ok")
"""


def test_band_gather_gloo_world2(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_GLOO_WORKER.format(repo=REPO))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2",
           "--master-addr", "127.0.0.1", "--master-port", "29611", str(script)]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stdout + res.stderr
    assert res.stdout.count("ok") == 2


# ---------------------------------------------------------------------------- driver pieces (N1)
@pytest.mark.parametrize("name", ["tiny", "mini"])
def test_mat_layout_bit_exact_vs_reference_and_in_place(golden, name, tmp_path):
    """pyviz/apap.py:250-265: the reference's own post-processing output is in the golden file ('mat')."""
    import scipy.io
    from cvx_proj_b200 import driver
    g = golden(f"ref_{name}.npz")
    grid = g["H"].copy()
    mat = driver.mat_layout(grid)
    assert mat.dtype == np.float64 and mat.shape == (grid.shape[0] * grid.shape[1], 9)
    assert np.array_equal(mat, g["mat"])
    # the caller's grid now holds the normalised inverses, like the script's loop leaves it
    assert np.array_equal(grid.transpose(0, 1, 3, 2).astype(np.float64).reshape(-1, 9), mat)
    assert np.all(grid[..., 2, 2] == 1.0)
    path = driver.save2mat("H31_apap", mat, name="H", prefix=str(tmp_path) + "/")
    back = scipy.io.loadmat(path)
    assert np.array_equal(back["H"], mat)


def test_image_warping_host_arithmetic(golden):
    """Canvas size / offsets / composed matrix and the closed-form inverse of cvx_proj_b200.utils against the
    golden canvases' shapes (live reference) and the oracle."""
    from cvx_proj_b200 import utils as putils
    from oracle import warp_oracle as wo
    from oracle.gen_golden_warping import CASES, warping_case
    g = golden("ref_image_warping.npz")
    for name in CASES:
        base, warp, hmat = warping_case(name)
        cw, ch, tx, ty, m = putils.warping_canvas(base.shape, warp.shape, hmat)
        assert (ch, cw, 3) == tuple(g[name + "_paste_shape"])
        ow = wo.warping_canvas(base.shape, warp.shape, hmat)
        assert (cw, ch, tx, ty) == ow[:4] and np.array_equal(m, ow[4])
        assert np.array_equal(putils.invert3x3(m).view(np.uint64), wo.invert3x3(m).view(np.uint64))
    assert np.array_equal(putils.invert3x3(np.zeros((3, 3))), np.zeros((3, 3)))


def test_spectral_host_pieces_vs_oracle(golden):
    """cv_to_array / recompute_matching / affinity_diagonal of cvx_proj_b200.spectral_method (host, numpy) against the
    oracle and the live reference's masks; keypoints and matches are duck-typed stand-ins for cv2's objects."""
    from types import SimpleNamespace
    from cvx_proj_b200 import spectral_method as psm
    from oracle import spectral_oracle as so
    from oracle.gen_golden_spectral import OPTS, spectral_case
    g = golden("ref_spectral.npz")
    opts = SimpleNamespace(**OPTS)
    for name in ("s40", "s300", "s1000"):
        c, o, cf, of, fmat, hg = spectral_case(name)
        n = c.shape[0]
        perm = np.random.default_rng(1).permutation(n)
        kc = [SimpleNamespace(pt=(float(x), float(y))) for x, y in c[np.argsort(perm)]]     # stored shuffled ...
        fc = cf[np.argsort(perm)]
        ko = [SimpleNamespace(pt=(float(x), float(y))) for x, y in o]
        matches = [SimpleNamespace(queryIdx=int(perm[i]), trainIdx=i) for i in range(n)]       # ... matches undo it
        sp, dp = psm.cv_to_array(kc, ko, matches)
        assert np.array_equal(sp, c) and np.array_equal(dp, o)
        mask = psm.recompute_matching(kc, fc, ko, of, matches, hg, opts)
        assert np.array_equal(mask, g[name + "_original_mask"])
        diag = psm.affinity_diagonal(c, o, cf, of, fmat, OPTS["epi_weight"])
        want = np.diag(so.affinity_matrix(c, o, cf, of, fmat, OPTS["epi_weight"], OPTS["affinity_eps"]))
        assert np.array_equal(diag, want)


def _prmt(a, b, sel):
    """PTX ``prmt.b32 d, a, b, sel`` (default mode) on uint32 arrays: nibble i of ``sel`` picks byte (nibble & 7)
    of the pair (a = bytes 0-3, b = bytes 4-7); nibble bit 3 replicates the picked byte's sign bit over the byte."""
    a, b = np.asarray(a, dtype=np.uint64), np.asarray(b, dtype=np.uint64)
    pair = a | (b << np.uint64(32))
    out = np.zeros_like(a)
    for i in range(4):
        nib = (sel >> (4 * i)) & 0xF
        byte = (pair >> np.uint64(8 * (nib & 7))) & np.uint64(0xFF)
        if nib & 8:
            byte = np.where(byte & np.uint64(0x80), np.uint64(0xFF), np.uint64(0))
        out |= byte << np.uint64(8 * i)
    return out.astype(np.uint32)


def test_blend_simd_word_arithmetic_equals_uniform_blend():
    """The 32-bit SIMD formulation of ``k_blend`` (csrc/warp_blend.cu ``blend16``: PRMT gathers of the channel bytes,
    carry-trick non-zero test, sign-replicating PRMT to spread the pixel flag, per-byte floor average), restated in
    numpy on four pixels = three words, equals uniform_blend (pyviz/apap_utils.py:75-88) for every byte pattern class."""
    rng = np.random.default_rng(11)
    palette = np.array([0, 0, 0, 1, 0x7F, 0x80, 0xFE, 0xFF], dtype=np.uint8)
    a = np.concatenate([palette[rng.integers(0, 8, size=(20000, 4, 3))],
                        rng.integers(0, 256, size=(20000, 4, 3), dtype=np.uint8)])
    b = np.concatenate([palette[rng.integers(0, 8, size=(20000, 4, 3))],
                        rng.integers(0, 256, size=(20000, 4, 3), dtype=np.uint8)])
    b = b[rng.permutation(b.shape[0])]
    wa = np.ascontiguousarray(a).reshape(-1, 12).view("<u4")          # [n, 3] words of 4 pixels
    wb = np.ascontiguousarray(b).reshape(-1, 12).view("<u4")

    def pixel_or4(w):
        x = _prmt(_prmt(w[:, 0], w[:, 1], 0x0630), w[:, 2], 0x5210)
        y = _prmt(_prmt(w[:, 0], w[:, 1], 0x0741), w[:, 2], 0x6210)
        z = _prmt(_prmt(w[:, 0], w[:, 1], 0x0052), w[:, 2], 0x7410)
        return x | y | z

    def nonzero_msb(v):
        return (((v & np.uint32(0x7F7F7F7F)).astype(np.uint64) + 0x7F7F7F7F).astype(np.uint32)) | v

    both = nonzero_msb(pixel_or4(wa)) & nonzero_msb(pixel_or4(wb))
    out = np.empty_like(wa)
    for w, sel in enumerate((0x9888, 0xAA99, 0xBBBA)):
        m = _prmt(both, both, sel)
        x, y = wa[:, w], wb[:, w]
        avg = ((x & y).astype(np.uint64) + (((x ^ y) & np.uint32(0xFEFEFEFE)) >> np.uint32(1))).astype(np.uint32)
        out[:, w] = (avg & m) | ((x | y) & ~m)
    got = out.view(np.uint8).reshape(-1, 4, 3)
    assert np.array_equal(got, orc.uniform_blend(a, b))


def test_certified_inverse_restatement_has_numpys_bits():
    """``invert_grid_certified`` (numpy restatement of ``apap_invert_grid``): every cell it certifies carries exactly
    the float32 bits of ``np.linalg.inv`` (pyviz/apap.py:201-203); degenerate classes are never certified; on
    homography-like grids almost every cell is certified."""
    rng = np.random.default_rng(23)
    n = 200_000
    g = np.tile(np.eye(3), (n, 1, 1))
    g[:, :2, :2] += rng.normal(0, 0.2, (n, 2, 2))
    g[:, :2, 2] = rng.normal(0, 1, (n, 2)) * 10.0 ** rng.uniform(0, 3.7, (n, 1))
    g[:, 2, :2] = rng.normal(0, 1, (n, 2)) * 10.0 ** rng.uniform(-7, -3, (n, 1))
    g *= 10.0 ** rng.uniform(-2, 2, (n, 1, 1))
    g = g.astype(np.float32)
    g[::1000, 2, :2] = 0                                    # affine: exact zeros in the inverse
    g[7] = np.nan
    g[11] = 0                                               # singular
    g[13, 1] = g[13, 0]                                     # singular, rank 2
    g[17, 1, 0] = g[17, 0, 0]                               # tie in the first pivot search
    f, flag = papap.invert_grid_certified(g)
    assert flag[[0, 1000, 7, 11, 13, 17]].all()
    keep = ~flag
    want = np.linalg.inv(g[keep])
    assert np.array_equal(f[keep].view(np.uint32), want.view(np.uint32))
    assert flag.mean() < 0.005
    # an ill-conditioned family: the certificate gives up instead of guessing
    ill = np.tile(np.eye(3, dtype=np.float32), (1000, 1, 1))
    ill[:, 0, 1] = 1.0
    ill[:, 1, 1] = (1.0 + rng.uniform(1e-7, 1e-6, 1000)).astype(np.float32)
    ill[:, 1, 0] = 1.0
    f, flag = papap.invert_grid_certified(ill)
    want = np.linalg.inv(ill[~flag])
    assert np.array_equal(f[~flag].view(np.uint32), want.view(np.uint32))


@pytest.mark.parametrize("family", ["uniform", "row_scales", "col_scales", "near_rank1", "small_ints", "hilbert"])
def test_certified_inverse_never_certifies_a_different_rounding(family):
    """The certificate of ``invert_grid_certified`` over matrix families far from homographies: whatever it certifies
    has numpy's bits; what it cannot decide it flags (near-singular, exact zeros, pivot ties)."""
    rng = np.random.default_rng(31)
    n = 30000
    if family == "uniform":
        g = rng.uniform(-1, 1, (n, 3, 3))
    elif family == "row_scales":
        g = rng.normal(0, 1, (n, 3, 3)) * 10.0 ** rng.uniform(-6, 6, (n, 3, 1))
    elif family == "col_scales":
        g = rng.normal(0, 1, (n, 3, 3)) * 10.0 ** rng.uniform(-6, 6, (n, 1, 3))
    elif family == "near_rank1":
        g = rng.normal(0, 1, (n, 3, 1)) * rng.normal(0, 1, (n, 1, 3)) + 10.0 ** rng.uniform(-7, -3, (n, 1, 1)) * rng.normal(0, 1, (n, 3, 3))
    elif family == "small_ints":
        g = rng.integers(-3, 4, (n, 3, 3)).astype(np.float64)
    else:
        g = (1.0 / (np.arange(3)[:, None] + np.arange(3)[None, :] + 1.0))[None] * (1 + 1e-3 * rng.normal(0, 1, (n, 3, 3)))
    g = g.astype(np.float32)
    f, flag = papap.invert_grid_certified(g)
    keep = ~flag
    want = np.linalg.inv(g[keep])                            # numpy never raises on a certified cell
    assert np.array_equal(f[keep].view(np.uint32), want.view(np.uint32))
    if family in ("uniform", "row_scales", "col_scales", "hilbert"):
        assert flag.mean() < 0.01


def test_compat_modules_have_the_reference_module_names_and_signatures():
    """SURVEY 8(b): the reference's driver does ``from apap_utils import *`` and defines ``class APAP`` in module
    ``apap`` (pyviz/apap.py:15,21).  With ``compat/`` on sys.path the same imports resolve to this package, with the
    reference's parameter names (pyviz/apap.py:22,35,63,92,103,121,172,186; pyviz/apap_utils.py:10,23,40,75)."""
    import importlib
    import inspect
    compat = os.path.join(REPO, "compat")
    sys.path.insert(0, compat)
    try:
        for name in ("apap", "apap_utils"):
            sys.modules.pop(name, None)
        apap_mod = importlib.import_module("apap")
        utils_mod = importlib.import_module("apap_utils")
    finally:
        sys.path.remove(compat)
    assert sorted(utils_mod.__all__) == ["final_size", "get_mesh", "get_vertice", "uniform_blend"]
    for fn in utils_mod.__all__:                                   # star-imported into `apap`, like the reference
        assert getattr(apap_mod, fn) is getattr(utils_mod, fn)
    params = lambda f: list(inspect.signature(f).parameters)       # noqa: E731
    assert params(utils_mod.get_mesh) == ["size", "mesh_size", "start"]
    assert params(utils_mod.get_vertice) == ["size", "mesh_size", "offsets"]
    assert params(utils_mod.final_size) == ["src_img", "dst_img", "project_H"]
    assert params(utils_mod.uniform_blend) == ["img1", "img2"]
    cls = apap_mod.APAP
    assert params(cls.__init__)[:5] == ["self", "gamma", "sigma", "final_size", "offset"]
    assert params(cls.getNormalize2DPts) == ["point"] and params(cls.getConditionerFromPts) == ["point"]
    assert params(cls.point_normalize) == ["nf", "c"] and params(cls.matrix_generate) == ["sample_n", "cf1", "cf2"]
    assert params(cls.local_homography) == ["self", "src_point", "dst_point", "vertices"]
    assert params(cls.warp_coordinate_estimate) == ["pt", "homography"]
    assert params(cls.local_warp)[:5] == ["self", "ori_img", "local_homography", "mesh", "progress"]      # + interpolation= (extension)
    st = cls(0.5, 100, [64, 48], [3, 2])
    assert (st.gamma, st.sigma, st.final_width, st.final_height, st.offset_x, st.offset_y) == (0.5, 100, 64, 48, 3, 2)
    mesh = utils_mod.get_mesh((64, 48), 5)
    assert mesh.shape == (2, 5) and mesh.dtype == np.float64
    for name in ("apap", "apap_utils"):
        sys.modules.pop(name, None)


def test_cell_lookup_tables_refuse_grids_beyond_16_bit_cell_indices():
    """ADVICE round 1: the warp tables hold cell rows / columns in 16 bits; a larger grid must not wrap silently."""
    from cvx_proj_b200.apap import cell_lookup_tables
    mesh = (np.linspace(0, 100, 70001), np.linspace(0, 100, 11))
    with pytest.raises(ValueError, match="65535"):
        cell_lookup_tables(mesh, 100, 100, 10, 70000)


def test_pass_workspace_layout_is_host_side_and_consistent():
    """apap_pass_workspace_bytes (the scratch of the one-call apap_local_homography_points) is pure host arithmetic:
    it answers without a GPU, grows with every dimension, covers the partial planes of the gram plan, and rejects
    nonsense."""
    import ctypes
    lib = rt.load_library()

    def need(batch, n, cells, engine):
        out = ctypes.c_size_t()
        rc = lib.apap_pass_workspace_bytes(batch, n, cells, engine, ctypes.byref(out))
        return rc, int(out.value)

    for engine in (rt.GRAM_TCGEN05, rt.GRAM_FFMA2):
        rc, base = need(1, 5000, 40_000, engine)
        assert rc == 0 and base % 256 == 0
        n_pad = 5120
        _, _, partial = rt.gram_plan(40_000, n_pad, engine)
        rows = n_pad * 28 * 4
        blocks = (n_pad // 8) * 528 * 4 if engine == rt.GRAM_TCGEN05 else 0
        assert base >= partial + rows + blocks + 40_000 * 8 + 2 * 5000 * 8
        assert base < 1.05 * (partial + rows + blocks + 40_000 * 8 + 2 * 5000 * 8) + 8 * 256
        assert need(2, 5000, 40_000, engine)[1] > base
        assert need(1, 5200, 40_000, engine)[1] > base            # one more chunk of keypoints
        assert need(1, 5000, 41_000, engine)[1] > base
    assert need(0, 10, 10, 0)[0] != 0 and need(1, 0, 10, 0)[0] != 0 and need(1, 10, 10, 7)[0] != 0


def test_invert_grid_finish_writes_numpys_inverse_for_flagged_cells():
    """The host tail of the device inverse (APAP._invert_grid_finish): certified cells take the device's bits, flagged
    cells numpy's own inverse computed from the caller's values BEFORE anything is overwritten; a singular flagged cell
    raises like np.linalg.inv and leaves the array untouched."""
    import torch
    rng = np.random.default_rng(2)
    grid = (np.eye(3) + 0.1 * rng.standard_normal((6, 3, 3))).astype(np.float32)
    before = grid.copy()
    device_inverse = torch.from_numpy(np.linalg.inv(before).reshape(-1) + np.float32(1.0))     # recognisably "the GPU's"
    flags = torch.tensor([0, 1, 0, 0, 1, 0], dtype=torch.uint8)
    assert papap.APAP._invert_grid_finish(grid, device_inverse, flags) == 2
    want = device_inverse.numpy().reshape(6, 3, 3).copy()
    want[[1, 4]] = np.linalg.inv(before[[1, 4]])
    assert np.array_equal(grid, want)
    singular = before.copy()
    singular[4] = 0
    keep = singular.copy()
    with pytest.raises(np.linalg.LinAlgError):
        papap.APAP._invert_grid_finish(singular, device_inverse, flags)
    assert np.array_equal(singular, keep)
