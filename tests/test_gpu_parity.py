"""GPU parity tests: the CUDA path (through the C ABI, via the reference-shaped Python surface)
against the golden vectors of the live reference and against the oracle.

Tolerances (SURVEY.md section 8c / BASELINE.json north_star):
  per-cell H: max|S2 (H - Href) S1^-1| / max|S2 Href S1^-1| <= 1e-4, S = diag(1/L, 1/L, 1)
  warp, blend, lookup tables, in-place inverse: bit-exact
  local_weight (float64): relative 1e-13
"""
import hashlib
import os
import zlib

import numpy as np
import pytest

from cvx_proj_b200 import apap_utils, sharding, synth
from cvx_proj_b200 import _runtime as rt
from cvx_proj_b200.apap import APAP, cell_lookup_tables
from oracle import apap_oracle as orc

pytestmark = pytest.mark.gpu
H_GATE = 1e-4


ENGINES = ["tcgen05", "ffma2"]


def _stitcher(sc, **kw):
    return APAP(kw.get("gamma", sc.gamma), kw.get("sigma", sc.sigma), [sc.final_w, sc.final_h],
                [sc.offset_x, sc.offset_y], gram_engine=kw.get("engine", "tcgen05"))


def _herr(h, ref, sc):
    return orc.h_error_normalised(h, ref, max(sc.final_w, sc.final_h))


# ------------------------------------------------------------------------------- moving DLT
@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("name", ["tiny", "mini"])
def test_local_homography_vs_reference_golden(golden, name, engine):
    g = golden(f"ref_{name}.npz")
    sc = synth.make_scene(name)
    h, w = _stitcher(sc, engine=engine).local_homography(g["src"], g["dst"], g["vertices"])
    assert h.shape == g["H"].shape and h.dtype == np.float32
    assert _herr(h, g["H"], sc).max() <= H_GATE
    assert w.shape == g["W"].shape
    np.testing.assert_allclose(np.asarray(w), g["W"], rtol=1e-13, atol=0)
    np.testing.assert_allclose(w[2, 3], g["W"][2, 3], rtol=1e-13, atol=0)
    np.testing.assert_allclose(w[1], g["W"][1], rtol=1e-13, atol=0)


@pytest.mark.parametrize("engine", ENGINES)
def test_local_homography_c1_full_vs_reference(golden, engine):
    g = golden("ref_c1.npz")
    sc = synth.make_scene("c1")
    h, w = _stitcher(sc, engine=engine).local_homography(sc.src, sc.dst, sc.vertices)
    err = _herr(h, g["H"], sc)
    print(f"c1 [{engine}]: normalised H error max {err.max():.3e}, raw elementwise {orc.h_error_raw(h, g['H']):.3e}")
    assert err.max() <= H_GATE
    np.testing.assert_allclose(np.asarray(w)[::9, ::9, ::7], g["W_sample"], rtol=1e-13, atol=0)


@pytest.mark.parametrize("engine", ENGINES)
def test_clamped_weights(golden, engine):
    g = golden("ref_tiny_sigma8.npz")
    sc = synth.make_scene("tiny")
    h, w = _stitcher(sc, sigma=8.0, engine=engine).local_homography(sc.src, sc.dst, sc.vertices)
    assert _herr(h, g["H"], sc).max() <= H_GATE
    wa = np.asarray(w)
    np.testing.assert_allclose(wa, g["W"], rtol=1e-13, atol=0)
    assert np.array_equal(wa == 0.5, g["W"] == 0.5)


@pytest.mark.parametrize("engine", ENGINES)
def test_c2_spot_cells_vs_reference_and_full_grid_vs_oracle(golden, engine):
    s = golden("ref_c2_spot.npz")
    sc = synth.make_scene("c2")
    h, _ = _stitcher(sc, engine=engine).local_homography(sc.src, sc.dst, sc.vertices)
    got = h[s["rows"]][:, s["cols"]]
    err = _herr(got, s["H"], sc)
    print(f"c2 spot [{engine}]: normalised H error max {err.max():.3e}, raw {orc.h_error_raw(got, s['H']):.3e}")
    assert err.max() <= H_GATE
    # every 5th row and column of the full grid against the float64 Gram oracle
    sub = sc.vertices[::5, ::5]
    ref = orc.local_homography_gram64(sc.src, sc.dst, sub, sc.gamma, sc.sigma)
    full = _herr(h[::5, ::5], ref, sc)
    print(f"c2 grid [{engine}]: normalised H error vs float64 Gram oracle max {full.max():.3e} mean {full.mean():.3e}")
    assert full.max() <= H_GATE


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("n_kp", [4, 7, 128, 129, 1500, 9000])
def test_ragged_keypoint_counts(n_kp, engine):
    sc = synth.make_scene("mini", n_kp=n_kp, mesh=6)
    h, _ = _stitcher(sc, engine=engine).local_homography(sc.src, sc.dst, sc.vertices)
    if n_kp >= 7:        # fewer than ~5 pairs leave the DLT rank-deficient; the reference's answer is arbitrary there
        ref = orc.local_homography_gram64(sc.src, sc.dst, sc.vertices, sc.gamma, sc.sigma)
        assert _herr(h, ref, sc).max() <= H_GATE
    assert np.isfinite(h).all() or n_kp < 7


@pytest.mark.parametrize("engine", ENGINES)
@pytest.mark.parametrize("gamma,sigma", [(0.5, 100), (0.3, 100), (0.8, 100), (0.05, 20), (0.5, 8), (0.9999, 100),
                                         (1.0, 100), (1.7, 50)])
def test_clamp_and_falloff_sweep(gamma, sigma, engine):
    """gamma decides which weight path the tensor-core kernel takes (polynomial 2^-t for gamma >= 0.5,
    MUFU.EX2 below); sigma moves the weights between ~1 everywhere and clamped almost everywhere."""
    sc = synth.make_scene("mini", n_kp=700, mesh=12)
    h, _ = _stitcher(sc, engine=engine, gamma=gamma, sigma=sigma).local_homography(sc.src, sc.dst, sc.vertices)
    ref = orc.local_homography_gram64(sc.src, sc.dst, sc.vertices, gamma, sigma)
    err = _herr(h, ref, sc)
    print(f"gamma {gamma} sigma {sigma} [{engine}]: normalised H error max {err.max():.3e}")
    assert err.max() <= H_GATE


def test_exact_homography_gives_global_h_everywhere():
    sc = synth.make_scene("mini", n_kp=400)
    hom = np.concatenate([sc.src.astype(np.float64), np.ones((400, 1))], 1) @ sc.h_gt.T
    dst = (hom[:, :2] / hom[:, 2:3]).astype(np.float32)
    h, _ = _stitcher(sc).local_homography(sc.src, dst, sc.vertices)
    want = np.broadcast_to((sc.h_gt / sc.h_gt[2, 2]).astype(np.float32), h.shape)
    # inputs are float32-rounded, so the fit is exact only to ~1e-5 of a pixel scale
    assert _herr(h, want, sc).max() <= 2e-4


def test_all_weights_clamped_equals_unweighted_dlt():
    sc = synth.make_scene("mini")
    h, _ = _stitcher(sc, gamma=1.0).local_homography(sc.src, sc.dst, sc.vertices)   # max(w, 1) == 1
    ref = orc.local_homography_svd(sc.src, sc.dst, sc.vertices[:1, :1], 1.0, sc.sigma)[0, 0]
    assert _herr(h, np.broadcast_to(ref, h.shape), sc).max() <= H_GATE
    assert np.abs(h - h[0, 0]).max() <= 1e-6 * np.abs(h[0, 0]).max()


def test_keypoint_permutation_invariance():
    sc = synth.make_scene("mini", n_kp=700)
    st = _stitcher(sc)
    h0, _ = st.local_homography(sc.src, sc.dst, sc.vertices)
    perm = np.random.default_rng(11).permutation(700)
    h1, _ = st.local_homography(sc.src[perm], sc.dst[perm], sc.vertices)
    assert _herr(h1, h0, sc).max() <= H_GATE


@pytest.mark.parametrize("engine", ENGINES)
def test_batch_equals_single_pairs_bitwise(engine):
    scenes = [synth.make_scene("mini", seed=s, n_kp=n) for s, n in ((0, 200), (1, 333), (2, 120))]
    st = _stitcher(scenes[0], engine=engine)
    many = st.local_homography_batch([s.src for s in scenes], [s.dst for s in scenes], scenes[0].vertices)
    for sc, hb in zip(scenes, many):
        h1, _ = st.local_homography(sc.src, sc.dst, scenes[0].vertices)
        assert np.array_equal(hb, h1)


@pytest.mark.parametrize("engine", ENGINES)
def test_cell_row_sharding_is_bitwise_identical(engine):
    """Rows solved on their own (what a rank of the multi-GPU run does) equal the same rows of the
    full-grid solve bit for bit: the FP32 chain boundaries depend only on the keypoint count, and an
    accumulator row of the tensor-core tile depends only on its own cell."""
    sc = synth.make_scene("c1", mesh=40)
    st = _stitcher(sc, engine=engine)
    full, _ = st.local_homography(sc.src, sc.dst, sc.vertices)
    for r0, r1 in sharding.split_rows(40, 3):
        part, _ = st.local_homography(sc.src, sc.dst, sc.vertices[r0:r1])
        assert np.array_equal(part, full[r0:r1])


def test_overlapped_k2_launch_equals_plain_sequence():
    """K2 launched as a programmatic dependent of K1 (per-tile completion counters) gives the same bits as the
    plain K1 -> K2 sequence, call after call (the counters are zero again after every call), batches included."""
    import torch
    from cvx_proj_b200.apap import scale_anchors, weight_scale
    dev = torch.device("cuda", torch.cuda.current_device())
    for name, kw, batch in (("c1", {}, 1), ("mini", {"n_kp": 3000, "mesh": 50}, 3), ("c2", {}, 1)):
        sc = synth.make_scene(name, **kw)
        st = _stitcher(sc)
        table, tmats = st._prepare(sc.src, sc.dst)
        t = st.kp_table_device(torch.from_numpy(np.stack([table] * batch)).to(dev))
        a = torch.from_numpy(np.stack([scale_anchors(sc.vertices, weight_scale(sc.sigma))] * batch)).to(dev)
        m = torch.from_numpy(np.stack([tmats] * batch)).to(dev)
        plain = st.local_homography_device(t, a, m, batch, sc.n_cells, overlap=False).cpu().numpy()
        for _ in range(4):
            got = st.local_homography_device(t, a, m, batch, sc.n_cells, overlap=True).cpu().numpy()
            assert np.array_equal(got.view(np.uint32), plain.view(np.uint32))
        assert int(st._tile_counters(torch, dev, batch, sc.n_cells).abs().sum().item()) == 0


def test_clamp_free_k1_path_is_bit_identical_and_the_bound_is_an_upper_bound():
    """apap_weight_bound bounds the pre-scaled distance of every (cell, match) pair; with it K1 leaves the clamp
    max(w, gamma^2) out where no weight can reach it (reference defaults on c1 / c2) and keeps it where some do (small
    sigma) -- the H grid has the same bits as the always-clamping launch either way, and as a launch told +inf."""
    import torch
    from cvx_proj_b200.apap import scale_anchors, weight_scale
    dev = torch.device("cuda", torch.cuda.current_device())
    for name, kw, clamp_free in (("c1", {}, True), ("c2", {}, True), ("c1", {"sigma": 8.5}, False),
                                 ("mini", {"sigma": 30.0, "gamma": 0.1}, True), ("mini", {"sigma": 10.0, "gamma": 0.1}, False)):
        sc = synth.make_scene(name)
        st = _stitcher(sc, **kw)
        table, tmats = st._prepare(sc.src, sc.dst)
        s = weight_scale(st.sigma)
        t = st.kp_table_device(torch.from_numpy(table[None]).to(dev))
        anchors = scale_anchors(sc.vertices, s)
        a = torch.from_numpy(anchors[None]).to(dev)
        m = torch.from_numpy(tmats[None]).to(dev)
        raw = torch.from_numpy(np.ascontiguousarray(sc.src[None], dtype=np.float32)).to(dev)
        bound = st.weight_bound_device(raw, None, a)
        # the largest pre-scaled distance any pair really has (float64)
        flat = anchors.reshape(-1, 2).astype(np.float64)
        some = np.concatenate([flat[::97], flat[[0, sc.mesh_cells - 1, -sc.mesh_cells, -1]]])
        d = np.float64(s) * sc.src.astype(np.float64)[None] - some[:, None]
        true_max = np.sqrt((d ** 2).sum(-1)).max()
        k = np.float64(s) * sc.src.astype(np.float64)
        box = np.hypot(max(k[:, 0].max() - flat[:, 0].min(), flat[:, 0].max() - k[:, 0].min()),
                       max(k[:, 1].max() - flat[:, 1].min(), flat[:, 1].max() - k[:, 1].min()))
        got_bound = float(bound.item())
        assert true_max <= got_bound and box <= got_bound <= box * 1.0001 + 2e-6
        t_max = -np.log2(np.float32(st.gamma) ** 2)
        limit = min(t_max, 2.0) if np.float32(st.gamma) ** 2 >= 0.25 else t_max      # the polynomial 2^-t covers t <= 2
        assert (got_bound * 1.001 + 1e-3 < limit) == clamp_free
        plain = st.local_homography_device(t, a, m, 1, sc.n_cells).cpu().numpy()
        with_bound = st.local_homography_device(t, a, m, 1, sc.n_cells, t_bound=bound).cpu().numpy()
        inf = torch.full((1,), float("inf"), dtype=torch.float32, device=dev)
        with_inf = st.local_homography_device(t, a, m, 1, sc.n_cells, t_bound=inf).cpu().numpy()
        assert np.array_equal(plain.view(np.uint32), with_bound.view(np.uint32))
        assert np.array_equal(plain.view(np.uint32), with_inf.view(np.uint32))
    # counts: matches past a scene's count do not widen its box; a scene without matches gets +inf
    pts = torch.tensor([[[10.0, 20.0], [30.0, 5.0], [9000.0, 9000.0]], [[1.0, 1.0], [2.0, 2.0], [3.0, 3.0]]], device=dev)
    counts = torch.tensor([2, 0], dtype=torch.int32, device=dev)
    anch = torch.tensor([[[0.0, 0.0], [0.04, 0.02]]] * 2, device=dev)
    st = APAP(0.5, 100, [64, 64], [0, 0])
    b = st.weight_bound_device(pts, counts, anch).cpu().numpy()
    s = weight_scale(100)
    want = np.hypot(max(abs(30 * s - 0.0), abs(0.04 - 10 * s)), max(abs(20 * s - 0.0), abs(0.02 - 5 * s)))
    assert np.isinf(b[1]) and want <= b[0] <= want * 1.0001 + 2e-6


def test_gram_engines_agree_on_partial_sums():
    """The tensor-core (3xTF32, TMEM) and the FP32 SIMT Gram kernels produce the same partial sums to
    ~1e-6 of the largest sum of each term (tcgen05 accumulates per 256-keypoint segment)."""
    import torch
    from cvx_proj_b200.apap import build_kp_blocks, scale_anchors, weight_scale
    sc = synth.make_scene("c1", mesh=37, n_kp=3001)
    table, _ = _stitcher(sc, engine="ffma2")._prepare(sc.src, sc.dst)
    lib = rt.load_library()
    dev = torch.device("cuda", torch.cuda.current_device())
    cells, n_pad = 37 * 37, table.shape[0]
    a = torch.from_numpy(scale_anchors(sc.vertices, weight_scale(sc.sigma))).to(dev)
    out = {}
    for engine, tab in ((rt.GRAM_FFMA2, table), (rt.GRAM_TCGEN05, build_kp_blocks(table))):
        ks, cp, nbytes = rt.gram_plan(cells, n_pad, engine)
        t = torch.from_numpy(tab).to(dev)
        part = torch.zeros(nbytes // 4, dtype=torch.float32, device=dev)
        rt.check(lib.apap_gram_partials(t.data_ptr(), a.data_ptr(), 1, cells, n_pad, 0.25, engine, None, part.data_ptr(),
                                        rt.stream_ptr(torch, dev)), "gram")
        out[engine] = part.cpu().numpy().reshape(ks, 24, cp)[:, :, :cells].astype(np.float64).sum(0)
    ref, got = out[rt.GRAM_FFMA2], out[rt.GRAM_TCGEN05]
    scale = np.abs(ref).max(axis=1, keepdims=True)
    err = np.abs(got - ref) / scale
    print(f"gram engines: max |tcgen05 - ffma2| / max|sum| per term = {err.max():.3e}, mean {err.mean():.3e}")
    assert err.max() <= 2e-5


@pytest.mark.parametrize("name,n_kp", [("mini", None), ("c1", None), ("c2", None), ("mini", 3), ("mini", 1)])
def test_device_conditioning_agrees_with_the_reference_host_prologue(name, n_kp):
    """apap_condition (float64 reductions in a fixed order) against the reference's numpy prologue, which the class
    keeps on the host bit-exact (pyviz/apap.py:129-141): conditioned points and de-normalisation matrices to float32
    accuracy, and the H grid of the public call against the one computed from the HOST prologue far inside the gate."""
    import torch
    sc = synth.make_scene(name) if n_kp is None else synth.make_scene(name, n_kp=n_kp)
    st = _stitcher(sc)
    dev = torch.device("cuda", torch.cuda.current_device())
    with np.errstate(all="ignore"):
        cf1, cf2, tmats = st._condition(sc.src, sc.dst)
    raw = torch.from_numpy(np.stack([sc.src, sc.dst])[:, None].astype(np.float32)).to(dev)
    cond, tm = st.condition_device(raw)
    cond, tm = cond.cpu().numpy(), tm.cpu().numpy()[0]
    if sc.src.shape[0] == 1:                       # the reference divides by n - 1 = 0: NaN on both sides
        assert not np.isfinite(tm).all() and not np.isfinite(tmats).all()
        return
    assert np.allclose(cond[0, 0], cf1, rtol=0, atol=2e-5) and np.allclose(cond[1, 0], cf2, rtol=0, atol=2e-5)
    assert np.allclose(tm, tmats, rtol=2e-6, atol=1e-9 * np.abs(tmats).max())
    if sc.src.shape[0] >= 8:
        h_pub, _ = st.local_homography(sc.src, sc.dst, sc.vertices)
        table, tmats_h = st._prepare(sc.src, sc.dst)                      # host prologue -> device K1 + K2
        t_dev = st.kp_table_device(torch.from_numpy(table[None]).to(dev))
        from cvx_proj_b200.apap import scale_anchors, weight_scale
        a_dev = torch.from_numpy(scale_anchors(sc.vertices, weight_scale(sc.sigma))[None]).to(dev)
        h_host = st.local_homography_device(t_dev, a_dev, torch.from_numpy(tmats_h[None]).to(dev), 1, sc.n_cells)
        h_host = h_host.cpu().numpy().reshape(h_pub.shape)
        assert _herr(h_pub, h_host, sc).max() <= 2e-5


@pytest.mark.parametrize("n_kp", [5, 128, 1000, 2049])
def test_device_kp_blocks_equal_host_restatement(n_kp):
    """apap_kp_blocks packs the tensor-core block table on the device: same bits as build_kp_blocks."""
    import torch
    from cvx_proj_b200.apap import build_kp_blocks
    sc = synth.make_scene("mini", n_kp=n_kp, mesh=4)
    st = _stitcher(sc)
    table, _ = st._prepare(sc.src, sc.dst)
    dev = torch.device("cuda", torch.cuda.current_device())
    rows = torch.from_numpy(np.stack([table, table[::-1].copy()])).to(dev)          # batch of 2
    got = st.kp_table_device(rows).cpu().numpy()
    for b, tab in enumerate((table, table[::-1].copy())):
        want = build_kp_blocks(tab)
        assert got[b].shape == want.shape
        assert np.array_equal(got[b].view(np.uint32), want.view(np.uint32))


@pytest.mark.parametrize("n_kp", [1, 5, 128, 1000, 2049])
def test_device_kp_rows_equal_host_restatement(n_kp):
    """apap_kp_rows builds the keypoint row table on the device from the conditioned points: same bits as
    build_kp_table on the reference's DLT matrix, ragged batch (the second scene has fewer matches) included."""
    import torch
    sc = synth.make_scene("mini", n_kp=max(n_kp, 4), mesh=4)
    st = _stitcher(sc)
    src, dst = sc.src[:n_kp], sc.dst[:n_kp]
    short = max(1, n_kp // 3)
    dev = torch.device("cuda", torch.cuda.current_device())
    scenes = [(src, dst), (src[:short] * np.float32(0.75), dst[:short])]
    points = np.zeros((3, 2, n_kp, 2), dtype=np.float32)
    for b, (s_, d_) in enumerate(scenes):
        cf1, cf2, _ = st._condition(s_, d_)
        points[0, b, :len(s_)], points[1, b, :len(s_)], points[2, b, :len(s_)] = cf1, cf2, s_
    counts = torch.tensor([n_kp, short], dtype=torch.int32, device=dev)
    got = st.kp_rows_device(torch.from_numpy(points).to(dev), counts).cpu().numpy()
    for b, (s_, d_) in enumerate(scenes):
        want, _ = st._prepare(s_, d_)
        assert got.shape[1] >= want.shape[0]
        assert np.array_equal(got[b, :want.shape[0]].view(np.uint32), want.view(np.uint32))
        assert not got[b, want.shape[0]:].any()
    one = st.kp_rows_device(torch.from_numpy(points[:, :1].copy()).to(dev)).cpu().numpy()      # counts = NULL
    assert np.array_equal(one[0].view(np.uint32), got[0].view(np.uint32))


def test_device_warp_tables_equal_host_restatement():
    """apap_warp_tables builds the fast-path records on the device: same bits as build_warp_tables (whose
    guard-band logic the CPU tests check), on a real grid and on degenerate / adversarial cells."""
    import torch
    from cvx_proj_b200.apap import build_warp_tables
    for name, kw in (("mini", {}), ("c1", {}), ("mini", {"mesh": 300})):      # mesh 300 > canvas: unused cells
        sc = synth.make_scene(name, **kw)
        st = _stitcher(sc)
        m = sc.mesh_cells
        rng = np.random.default_rng(5)
        h = np.linalg.inv(sc.h_gt)[None, None].repeat(m, 0).repeat(m, 1)
        h = (h * (1 + 1e-3 * rng.standard_normal(h.shape))).astype(np.float32)
        h[0, 0] = 0                                   # degenerate cells
        h[1 % m, 2 % m] = np.nan
        h[2 % m, 1 % m, 2] = [1e-30, 1e-30, 1e-30]    # denominator ~ 0
        h[3 % m, 3 % m] *= -1                         # negative denominator
        h[4 % m, 0] = np.eye(3, dtype=np.float32)     # exact integer hits
        h[m - 1, m - 1, :, 2] += 1e9                  # far outside / beyond 2^30
        col, row = cell_lookup_tables(sc.mesh, sc.final_w, sc.final_h, m, m)
        want, _, _ = build_warp_tables(h, col, row, sc.offset_x, sc.offset_y, sc.width, sc.height)
        tabs = st.warp_tables_device(h, col, row, sc.width, sc.height)
        got = tabs.cell_fast.cpu().numpy().reshape(-1, 12)
        same = got.view(np.uint32) == want.view(np.uint32)
        assert same.all(), (name, kw, np.argwhere(~same)[:5], got[~same.all(1)][:2], want[~same.all(1)][:2])
        assert 0.0 <= tabs.exact_cells_frac() <= 1.0


def test_eig_solvers_agree_and_report():
    """AUTO (float64 LDL^T inverse iteration) and JACOBI (full FP32 diagonalisation) give the same
    grid; out_sweeps tells which one ran per cell."""
    import torch
    from cvx_proj_b200.apap import scale_anchors, weight_scale
    sc = synth.make_scene("c1", mesh=40)
    st = _stitcher(sc)
    table, tmats = st._prepare(sc.src, sc.dst)
    dev = torch.device("cuda", torch.cuda.current_device())
    t = st.kp_table_device(torch.from_numpy(table[None]).to(dev))
    a = torch.from_numpy(scale_anchors(sc.vertices, weight_scale(sc.sigma))[None]).to(dev)
    m = torch.from_numpy(tmats[None]).to(dev)
    cells = 40 * 40
    out = {}
    for solver in (rt.EIG_AUTO, rt.EIG_JACOBI):
        sw = torch.zeros((1, cells), dtype=torch.int32, device=dev)
        h = st.local_homography_device(t, a, m, 1, cells, sweeps=sw, solver=solver)
        out[solver] = (h.cpu().numpy().reshape(40, 40, 3, 3), sw.cpu().numpy().ravel())
    h_auto, sw_auto = out[rt.EIG_AUTO]
    h_jac, sw_jac = out[rt.EIG_JACOBI]
    assert (sw_auto < 0).all() and (sw_auto >= -6).all(), (sw_auto.min(), sw_auto.max())
    assert (sw_jac > 0).all() and (sw_jac <= 12).all()
    assert _herr(h_auto, h_jac, sc).max() <= 2e-5
    ref = orc.local_homography_gram64(sc.src, sc.dst, sc.vertices, sc.gamma, sc.sigma)
    print(f"eig: auto vs gram64 {_herr(h_auto, ref, sc).max():.2e}, jacobi vs gram64 {_herr(h_jac, ref, sc).max():.2e}, "
          f"inverse-iteration steps {-sw_auto.max()}..{-sw_auto.min()}, jacobi sweeps {sw_jac.min()}..{sw_jac.max()}")
    assert _herr(h_auto, ref, sc).max() <= H_GATE and _herr(h_jac, ref, sc).max() <= H_GATE


def test_degenerate_keypoints_fall_back_to_jacobi():
    """Collinear keypoints: the Gram matrix has a multi-dimensional null space, inverse iteration
    cannot settle on a direction-independent answer -> those cells take the Jacobi path (or settle
    on a null vector); the result must be finite either way, as it is for the reference's SVD."""
    import torch
    sc = synth.make_scene("mini", mesh=6)
    src = sc.src.copy()
    src[:, 1] = 0.5 * src[:, 0] + 3.0
    dst = src + np.float32(2.0)
    h, _ = _stitcher(sc).local_homography(src, dst, sc.vertices)
    assert h.shape == (6, 6, 3, 3)
    assert np.isfinite(h[..., 2, 2]).all()
    torch.cuda.synchronize()


# --------------------------------------------------------------------------------- mesh warp
@pytest.mark.parametrize("name", ["tiny", "mini"])
def test_local_warp_bit_exact_vs_reference_golden(golden, name):
    g = golden(f"ref_{name}.npz")
    sc = synth.make_scene(name)
    img = sc.image(1)
    h = g["H"].copy()
    warped = _stitcher(sc).local_warp(img, h, g["mesh"], progress=True)
    assert warped.dtype == np.uint8 and np.array_equal(warped, g["warped"])
    assert np.array_equal(h, g["H_inverted_in_place"])          # the in-place inversion side effect
    centre = synth.make_image(sc.width, sc.height, seed=2)
    pasted = orc.paste_centre(warped, centre, (sc.offset_x, sc.offset_y))
    assert np.array_equal(apap_utils.uniform_blend(warped, pasted), g["blended"])
    fused = _stitcher(sc).local_warp_blend(img, g["H"].copy(), g["mesh"], centre)
    assert np.array_equal(fused, g["blended"])


def test_local_warp_c1_rows_vs_reference(golden):
    g = golden("ref_c1.npz")
    sc = synth.make_scene("c1")
    img = sc.image(1)
    warped = _stitcher(sc).local_warp(img, g["H"].copy(), sc.mesh)
    crc = np.array([zlib.crc32(np.ascontiguousarray(r).tobytes()) for r in warped], dtype=np.uint32)
    bad = np.flatnonzero(crc != g["warped_row_crc"])
    assert bad.size == 0, f"rows differ: {bad[:10]}"
    assert hashlib.sha256(warped.tobytes()).hexdigest() == str(g["warped_sha"])


def test_fast_path_equals_forced_float64_path():
    sc = synth.make_scene("c1")
    img = sc.image(1)
    st = _stitcher(sc)
    h = orc.local_homography_gram64(sc.src, sc.dst, sc.vertices, sc.gamma, sc.sigma)
    a = st._warp(img, h.copy(), sc.mesh)
    b = st._warp(img, h.copy(), sc.mesh, force_exact=True)
    assert np.array_equal(a, b)
    assert (a.max(axis=-1) > 0).mean() > 0.3


def test_local_warp_c2_full_size_vs_oracle():
    sc = synth.make_scene("c2")
    img = sc.image(1)
    st = _stitcher(sc)
    h, _ = st.local_homography(sc.src, sc.dst, sc.vertices)
    want = orc.local_warp(img, orc.invert_grid(h), sc.mesh, (sc.final_w, sc.final_h), (sc.offset_x, sc.offset_y))
    got = st.local_warp(img, h, sc.mesh)
    diff = np.flatnonzero((got != want).any(axis=-1).ravel())
    assert diff.size == 0, f"{diff.size} pixels differ, first {diff[:5]}"


def _device_warp(st, sc, img, inv, centre=None, legacy=False, rows=None):
    """K3 through warp_tables_device + warp_device on cuda tensors (``legacy`` = round 1's strip kernel)."""
    import torch
    dev = torch.device("cuda", torch.cuda.current_device())
    gr, gc = inv.shape[0], inv.shape[1]
    col, row = cell_lookup_tables(sc.mesh, sc.final_w, sc.final_h, gr, gc)
    r0, r1 = rows if rows is not None else (0, sc.final_h)
    tabs = st.warp_tables_device(inv, col, row, img.shape[1], img.shape[0], dev, r0, r1)
    out = st.warp_device(torch.from_numpy(img).to(dev), tabs, gc, legacy=legacy,
                         centre_dev=torch.from_numpy(centre).to(dev) if centre is not None else None)
    return out.cpu().numpy()


def test_tile_engine_equals_legacy_strip_kernel_c2():
    """The tile engine (TMA-staged source boxes, LDS gathers, bulk row stores) and round 1's strip kernel pick the same
    bytes on the full c2 canvas and on a row band that starts mid-cell-row; fused with the blend (always the strip
    kernel) the default call and ``legacy`` agree."""
    sc = synth.make_scene("c2")
    img = sc.image(1)
    centre = synth.make_image(sc.width, sc.height, seed=2)
    st = _stitcher(sc)
    h, _ = st.local_homography(sc.src, sc.dst, sc.vertices)
    inv = orc.invert_grid(h)
    a = _device_warp(st, sc, img, inv)
    b = _device_warp(st, sc, img, inv, legacy=True)
    assert np.array_equal(a, b) and (a.max(axis=-1) > 0).mean() > 0.3
    fa = _device_warp(st, sc, img, inv, centre=centre)
    fb = _device_warp(st, sc, img, inv, centre=centre, legacy=True)
    assert np.array_equal(fa, fb)
    band = _device_warp(st, sc, img, inv, rows=(1001, 1777))
    assert np.array_equal(band, a[1001:1777])


@pytest.mark.parametrize("src_w,src_h,fw,fh,off", [(1000, 700, 1100, 800, (37, 21)),      # source rows not 16-byte aligned
                                                    (1024, 768, 1196, 822, (90, 30)),      # canvas rows 4- but not 16-byte aligned
                                                    (1024, 768, 1203, 811, (90, 30)),      # canvas rows not even 4-byte aligned
                                                    (640, 240, 2048, 352, (300, 60))])     # many tiles across, few down
def test_tile_engine_alignment_cases_vs_oracle(src_w, src_h, fw, fh, off):
    rng = np.random.default_rng(src_w + fw)
    img = rng.integers(1, 256, size=(src_h, src_w, 3), dtype=np.uint8)
    centre = rng.integers(0, 256, size=(src_h, src_w, 3), dtype=np.uint8)
    st = APAP(0.5, 100, [fw, fh], list(off))
    mesh = apap_utils.get_mesh((fw, fh), 24)
    yy, xx = np.meshgrid(np.arange(23), np.arange(23), indexing="ij")
    h = np.tile(np.array([[1.02, 0.03, 12.0], [-0.02, 0.98, -4.5], [1e-5, -2e-5, 1]], np.float32), (23, 23, 1, 1))
    h[..., 0, 2] += (3 * np.sin(xx / 4.0)).astype(np.float32)
    h[..., 1, 2] += (2 * np.cos(yy / 5.0)).astype(np.float32)
    want = orc.local_warp(img, orc.invert_grid(h), mesh, (fw, fh), off)
    got = st.local_warp(img, h.copy(), mesh)
    assert np.array_equal(got, want) and got.any()
    pasted = orc.paste_centre(want, centre, off)
    assert np.array_equal(st.local_warp_blend(img, h.copy(), mesh, centre), orc.uniform_blend(want, pasted))


@pytest.mark.parametrize("kind", ["rot90", "rot30", "minify3", "magnify4", "flip"])
def test_tile_engine_large_footprints_vs_oracle(kind):
    """Maps whose source box per tile is tall, wide or huge (rotation, minification: the box may not fit shared memory
    and the tile gathers from global memory), tiny (magnification) or mirrored."""
    rng = np.random.default_rng(11)
    sw, sh, fw, fh = 512, 384, 640, 416
    img = rng.integers(1, 256, size=(sh, sw, 3), dtype=np.uint8)
    c, s = np.cos(np.pi / 6), np.sin(np.pi / 6)
    fwd = {"rot90": [[0, -1, fw - 100.3], [1, 0, 10.2], [0, 0, 1]],
           "rot30": [[c, -s, 200.5], [s, c, -40.25], [1e-5, 0, 1]],
           "minify3": [[1 / 3, 0, 50.1], [0, 1 / 3, 60.7], [0, 1e-5, 1]],
           "magnify4": [[4, 0.1, -300.3], [0.05, 4, -200.9], [0, 0, 1]],
           "flip": [[-1, 0, fw - 70.4], [0.01, 1, 3.3], [0, 0, 1]]}[kind]
    h = np.tile(np.array(fwd, np.float32), (12, 12, 1, 1))
    h[..., 0, 2] += rng.uniform(-2, 2, size=(12, 12)).astype(np.float32)
    st = APAP(0.5, 100, [fw, fh], [0, 0])
    mesh = apap_utils.get_mesh((fw, fh), 13)
    want = orc.local_warp(img, orc.invert_grid(h), mesh, (fw, fh), (0, 0))
    got = st.local_warp(img, h.copy(), mesh)
    assert want.any() and np.array_equal(got, want)



def _sampled_cells_vs_oracle(sc, h, step):
    """H grid on every `step`-th cell row / column against the float64 Gram oracle (the full grid is too much
    float64 work for the CPU at the BASELINE sizes; the GPU computed every cell)."""
    ref = orc.local_homography_gram64(sc.src, sc.dst, np.ascontiguousarray(sc.vertices[::step, ::step]), sc.gamma,
                                      sc.sigma)
    return _herr(np.ascontiguousarray(h[::step, ::step]), ref, sc)


def test_c3_full_size_grid_and_warp():
    """BASELINE config c3 at full size on one GPU: 8K pair, 20 000 keypoints, 400 x 400 grid, 41.5 Mpix canvas."""
    sc = synth.make_scene("c3")
    st = _stitcher(sc)
    h, _ = st.local_homography(sc.src, sc.dst, sc.vertices)
    assert h.shape == (400, 400, 3, 3) and np.isfinite(h).all() and np.all(h[..., 2, 2] == 1.0)
    err = _sampled_cells_vs_oracle(sc, h, 40)
    print(f"c3 sampled cells: normalised H error max {err.max():.3e}")
    assert err.max() <= H_GATE
    img = sc.image(1)
    inv = orc.invert_grid(h)
    want = orc.local_warp(img, inv, sc.mesh, (sc.final_w, sc.final_h), (sc.offset_x, sc.offset_y))
    grid = h.copy()
    got = st.local_warp(img, grid, sc.mesh)
    assert np.array_equal(grid, inv)                                   # in-place inverse, the reference's bits
    diff = np.flatnonzero((got != want).any(axis=-1).ravel())
    assert diff.size == 0, f"{diff.size} pixels differ, first {diff[:5]}"
    # idempotence of the pipeline on its own output grid, and the row bands of a 4-way shard tile the canvas
    col, row = cell_lookup_tables(sc.mesh, sc.final_w, sc.final_h, 400, 400)
    shards = sharding.plan_shards(row, 400, 4)
    assert shards[0].px_row0 == 0 and shards[-1].px_row1 == sc.final_h
    import torch
    dev = torch.device("cuda", torch.cuda.current_device())
    src_dev = torch.from_numpy(img).to(dev)
    for s in shards:
        tabs = st.warp_tables_device(inv, col, row, sc.width, sc.height, dev, s.px_row0, s.px_row1)
        band = st.warp_device(src_dev, tabs, 400).cpu().numpy()
        assert np.array_equal(band, want[s.px_row0:s.px_row1])


def test_c5_keypoint_sweep_ends_vs_oracle():
    """BASELINE config c5 (256 x 256 grid) at both ends of the keypoint sweep, 1k and 64k."""
    for n_kp in (1000, 64000):
        sc = synth.make_scene("c5", n_kp=n_kp)
        h, _ = _stitcher(sc).local_homography(sc.src, sc.dst, sc.vertices)
        err = _sampled_cells_vs_oracle(sc, h, 32)
        print(f"c5 N={n_kp}: normalised H error max {err.max():.3e}")
        assert np.isfinite(h).all() and err.max() <= H_GATE


def test_c4_batch_of_64_pairs():
    """BASELINE config c4: 64 1080p pairs (2 000 keypoints, 100 x 100 grid) in one launch; every pair equals its
    single-pair call bit for bit, sampled cells match the oracle."""
    scs = [synth.make_scene("c4", seed=k) for k in range(64)]
    st = _stitcher(scs[0])
    hs = st.local_homography_batch([sc.src for sc in scs], [sc.dst for sc in scs], [sc.vertices for sc in scs])
    assert len(hs) == 64
    for k in (0, 17, 63):
        single, _ = st.local_homography(scs[k].src, scs[k].dst, scs[k].vertices)
        assert np.array_equal(hs[k].view(np.uint32), single.view(np.uint32))
        assert _sampled_cells_vs_oracle(scs[k], hs[k], 20).max() <= H_GATE
    assert all(np.isfinite(x).all() for x in hs)


def test_local_warp_batch_equals_single_calls():
    scs = [synth.make_scene("mini", seed=k) for k in range(3)]
    st = _stitcher(scs[0])
    hs = st.local_homography_batch([sc.src for sc in scs], [sc.dst for sc in scs], scs[0].vertices)
    imgs = [sc.image(10 + k) for k, sc in enumerate(scs)]
    centres = [synth.make_image(scs[0].width, scs[0].height, seed=20 + k) for k in range(3)]
    grids = [h.copy() for h in hs]
    out = st.local_warp_batch(imgs, grids, scs[0].mesh)
    fused = st.local_warp_batch(imgs, [h.copy() for h in hs], scs[0].mesh, centres)
    for k in range(3):
        g = hs[k].copy()
        assert np.array_equal(out[k], st.local_warp(imgs[k], g, scs[0].mesh)) and np.array_equal(grids[k], g)
        assert np.array_equal(fused[k], st.local_warp_blend(imgs[k], hs[k].copy(), scs[0].mesh, centres[k]))
    with pytest.raises(ValueError):
        st.local_warp_batch(imgs, grids[:2], scs[0].mesh)


def test_identity_and_translation_hit_exact_integers():
    """Integer-valued coordinates sit exactly on the truncation boundary: every pixel is decided
    by the float64 path and must match the reference rule (strict bounds drop row/column 0)."""
    rng = np.random.default_rng(4)
    img = rng.integers(1, 256, size=(90, 120, 3), dtype=np.uint8)
    st = APAP(0.5, 100, [150, 100], [7, 5])
    mesh = apap_utils.get_mesh((150, 100), 5)
    h = np.tile(np.eye(3, dtype=np.float32), (4, 4, 1, 1))
    h[..., 0, 2] = 3.0
    got = st.local_warp(img, h.copy(), mesh)
    want = orc.local_warp(img, orc.invert_grid(h), mesh, (150, 100), (7, 5))
    assert np.array_equal(got, want)
    assert got.any() and not got[:, :7 + 3 + 1].any()


def test_warp_degenerate_cells():
    """Singular-ish / sign-changing denominators inside a cell (whole cell takes the exact path)."""
    rng = np.random.default_rng(9)
    img = rng.integers(1, 256, size=(64, 64, 3), dtype=np.uint8)
    st = APAP(0.5, 100, [96, 80], [0, 0])
    mesh = apap_utils.get_mesh((96, 80), 4)
    inv = np.tile(np.eye(3, dtype=np.float32), (3, 3, 1, 1))
    inv[0, 0, 2] = [0.05, 0.0, -0.5]         # t2 crosses zero at x = 10
    inv[1, 1, 2] = [0.0, 0.0, 1e-30]         # enormous coordinates
    inv[2, 2] = [[1.3, 0.2, -4.1], [0.1, 0.9, 2.2], [1e-3, -2e-3, 1.0]]
    h = np.linalg.inv(inv.astype(np.float64)).astype(np.float32)
    got = st.local_warp(img, h.copy(), mesh)
    want = orc.local_warp(img, orc.invert_grid(h), mesh, (96, 80), (0, 0))
    assert np.array_equal(got, want)


@pytest.mark.parametrize("fw,fh", [(1, 1), (3, 2), (5, 7), (130, 3)])
def test_warp_tiny_and_ragged_canvases(fw, fh):
    rng = np.random.default_rng(fw * 10 + fh)
    img = rng.integers(1, 256, size=(9, 11, 3), dtype=np.uint8)
    st = APAP(0.5, 100, [fw, fh], [1, 1])
    mesh = apap_utils.get_mesh((fw, fh), 3)
    h = np.tile(np.array([[0.9, 0.05, 0.3], [0.02, 1.1, -0.2], [1e-3, 0, 1]], np.float32), (2, 2, 1, 1))
    got = st.local_warp(img, h.copy(), mesh)
    want = orc.local_warp(img, orc.invert_grid(h), mesh, (fw, fh), (1, 1))
    assert got.shape == (fh, fw, 3) and np.array_equal(got, want)


def test_row_bands_tile_the_full_warp():
    import torch
    sc = synth.make_scene("c1", mesh=30)
    img = sc.image(1)
    st = _stitcher(sc)
    h = orc.local_homography_gram64(sc.src, sc.dst, sc.vertices, sc.gamma, sc.sigma)
    full = st.local_warp(img, h.copy(), sc.mesh)
    col, row = cell_lookup_tables(sc.mesh, sc.final_w, sc.final_h, 30, 30)
    for world in (2, 3, 8):
        parts = []
        for rank in range(world):
            sh = sharding.ShardedAPAP(st, sc.mesh, 30, 30, rank, world)
            band = sh.local_warp_band(img, h[sh.me.cell_row0:sh.me.cell_row1].copy())
            assert band.shape[0] == sh.me.n_px_rows
            parts.append(band.cpu().numpy())
        assert np.array_equal(np.concatenate(parts, 0), full)
    torch.cuda.synchronize()


def test_device_tensor_input_stays_on_device():
    import torch
    sc = synth.make_scene("mini")
    img = sc.image(1)
    st = _stitcher(sc)
    h = orc.local_homography_gram64(sc.src, sc.dst, sc.vertices, sc.gamma, sc.sigma)
    host = st.local_warp(img, h.copy(), sc.mesh)
    dev = st.local_warp(torch.from_numpy(img).cuda(), h.copy(), sc.mesh)
    assert dev.is_cuda and np.array_equal(dev.cpu().numpy(), host)


# --------------------------------------------------------------------------------------- blend
def test_uniform_blend_golden_and_tails(golden):
    g = golden("ref_blend.npz")
    assert np.array_equal(apap_utils.uniform_blend(g["a"], g["b"]), g["out"])
    rng = np.random.default_rng(2)
    for hh, ww in ((1, 1), (1, 15), (1, 16), (1, 17), (5, 13), (64, 100)):
        a = rng.integers(0, 256, size=(hh, ww, 3), dtype=np.uint8)
        b = rng.integers(0, 256, size=(hh, ww, 3), dtype=np.uint8)
        a[rng.random((hh, ww)) < 0.3] = 0
        b[rng.random((hh, ww)) < 0.3] = 0
        assert np.array_equal(apap_utils.uniform_blend(a, b), orc.uniform_blend(a, b)), (hh, ww)
    # channel values from the corners of the byte arithmetic (pixels with some channels zero, carries, msb), and pixel
    # counts at and around whole CTAs of the kernel (256 units of 16 pixels)
    palette = np.array([0, 0, 1, 0x7f, 0x80, 0xfe, 0xff], dtype=np.uint8)
    for hh, ww in ((7, 33), (64, 64), (1, 4096 + 5), (3, 4096), (257, 16)):
        a = palette[rng.integers(0, palette.size, size=(hh, ww, 3))]
        b = palette[rng.integers(0, palette.size, size=(hh, ww, 3))]
        assert np.array_equal(apap_utils.uniform_blend(a, b), orc.uniform_blend(a, b)), (hh, ww)


def test_uniform_blend_full_size_properties():
    sc = synth.make_scene("c2")
    a = synth.make_image(sc.final_w, sc.final_h, seed=3)
    b = synth.make_image(sc.final_w, sc.final_h, seed=4)
    a[: sc.final_h // 3] = 0
    b[2 * sc.final_h // 3:] = 0
    out = apap_utils.uniform_blend(a, b)
    assert np.array_equal(out, orc.uniform_blend(a, b))
    assert np.array_equal(apap_utils.uniform_blend(b, a), out)                      # symmetric
    assert np.array_equal(apap_utils.uniform_blend(a, np.zeros_like(a)), a)        # black is neutral
    assert np.array_equal(apap_utils.uniform_blend(a, a), np.where(a.max(-1, keepdims=True) > 0, a, 0))


def test_stitch_pair_driver_vs_oracle_pipeline():
    """The script from its matched keypoints on (pyviz/apap.py:238-265): grid, .mat matrix, stitched image."""
    from cvx_proj_b200 import driver
    sc = synth.make_scene("mini")
    other, centre = sc.image(1), synth.make_image(sc.width, sc.height, seed=2)
    res = driver.stitch_pair(centre, other, sc.src, sc.dst, sc.h_gt, mesh_size=sc.mesh_cells, gamma=sc.gamma,
                             sigma=sc.sigma)
    assert res.final_size == (sc.final_w, sc.final_h, sc.offset_x, sc.offset_y)
    assert np.array_equal(res.mesh, sc.mesh) and np.array_equal(res.vertices, sc.vertices)
    ref = orc.local_homography_gram64(sc.src, sc.dst, sc.vertices, sc.gamma, sc.sigma)
    assert _herr(res.local_homography, ref, sc).max() <= H_GATE
    # the .mat matrix and the image are functions of the float32 grid we returned: bit-exact against the oracle
    assert np.array_equal(res.mat, orc.mat_layout(res.local_homography))
    inv = orc.invert_grid(res.local_homography)
    warped = orc.local_warp(other, inv, sc.mesh, (sc.final_w, sc.final_h), (sc.offset_x, sc.offset_y))
    want = orc.uniform_blend(warped, orc.paste_centre(warped, centre, (sc.offset_x, sc.offset_y)))
    assert np.array_equal(res.stitched, want)


# ------------------------------------------------------------- global-homography warp (SURVEY 8f, N4)
def test_image_warping_bit_exact_vs_reference_golden(golden):
    """cvx_proj_b200.utils.image_warping against the live reference's outputs (cv.warpPerspective + paste / mean
    blend, pyviz/utils.py:93-127): every case, both modes, bit-exact."""
    from cvx_proj_b200 import utils as putils
    from oracle.gen_golden_warping import CASES, FULL, warping_case
    g = golden("ref_image_warping.npz")
    for name in CASES:
        base, warp, hmat = warping_case(name)
        for db in (True, False):
            tag = f"{name}_{'paste' if db else 'mean'}"
            res = putils.image_warping(base, warp, hmat, direct_blend=db)
            assert res.dtype == np.uint8 and tuple(g[tag + "_shape"]) == res.shape
            crc = np.array([zlib.crc32(np.ascontiguousarray(r).tobytes()) for r in res], dtype=np.uint32)
            bad = np.flatnonzero(crc != g[tag + "_rowcrc"])
            assert bad.size == 0, (tag, bad[:8])
            if name in FULL:
                assert np.array_equal(res, g[tag])


def test_warp_perspective_4k_and_degenerate_maps_vs_oracle():
    from cvx_proj_b200 import utils as putils
    from oracle import warp_oracle as wo
    img = synth.make_image(3840, 2160, seed=1)
    hmat = synth.ground_truth_h(3840, 2160)
    cw, ch, tx, ty, m = putils.warping_canvas(img.shape, img.shape, hmat)
    got = putils.warp_perspective(img, m, (cw, ch))
    want = wo.warp_perspective(img, m, (cw, ch))
    diff = np.flatnonzero((got != want).any(axis=-1).ravel())
    assert diff.size == 0, f"{diff.size} pixels differ, first {diff[:5]}"
    small = synth.make_image(200, 100, seed=9)
    for mm in (np.eye(3), np.array([[1, 0, 0.5], [0, 1, 0.25], [0, 0, 1.0]]), np.array([[1, 0, 0], [0, 1, 0], [0.01, 0, 1.0]]),
               np.array([[0.5, 0.2, -300], [0.1, 2, 50], [-0.002, 0.001, 1.0]]), np.zeros((3, 3)),
               np.array([[1e-9, 0, 0], [0, 1e-9, 0], [0, 0, 1.0]])):
        assert np.array_equal(putils.warp_perspective(small, mm, (300, 200)), wo.warp_perspective(small, mm, (300, 200)))
    assert putils.warp_perspective(small, np.eye(3), (7, 3)).shape == (3, 7, 3)


# ------------------------------------------------------------- spectral match weighting (SURVEY 8f, N4)
def test_calculate_m_vs_reference_golden(golden):
    """cvx_proj_b200.spectral_method.calculate_M against the live reference's outputs: the affinity matrix is the
    reference's bit for bit (checked through the oracle), the leading singular vector within 1e-10 of numpy's SVD,
    the masks identical."""
    import torch
    from types import SimpleNamespace
    from cvx_proj_b200 import spectral_method as psm
    from oracle import spectral_oracle as so
    from oracle.gen_golden_spectral import CASES, OPTS, spectral_case
    g = golden("ref_spectral.npz")
    opts = SimpleNamespace(**OPTS)
    lib = rt.load_library()
    dev = torch.device("cuda", torch.cuda.current_device())
    for name in CASES:
        c, o, cf, of, fmat, hg = spectral_case(name)
        n = c.shape[0]
        kc = [SimpleNamespace(pt=(float(x), float(y))) for x, y in c]
        ko = [SimpleNamespace(pt=(float(x), float(y))) for x, y in o]
        matches = [SimpleNamespace(queryIdx=i, trainIdx=i) for i in range(n)]
        seg, h_ret, rmask, omask = psm.calculate_M(kc, cf.copy(), ko, of.copy(), fmat, matches, opts, Hg=hg)
        assert h_ret is hg and seg.dtype == np.float64 and rmask.dtype == np.float32
        err = np.abs(seg - g[name + "_segment"]).max()
        print(f"{name}: max |segment - reference| = {err:.2e}")
        assert err <= 1e-10
        assert np.array_equal(omask, g[name + "_original_mask"])
        assert np.allclose(rmask, g[name + "_ransac_mask"], rtol=0, atol=1e-7)
        if n <= 1000:                                  # the matrix itself, bit for bit
            diag = psm.affinity_diagonal(c, o, cf, of, fmat, OPTS["epi_weight"])
            m = torch.empty((n, n), dtype=torch.float64, device=dev)
            c_dev, o_dev, g_dev = (torch.from_numpy(v).to(dev) for v in (c, o, diag))       # keep them alive
            rt.check(lib.apap_affinity_matrix(c_dev.data_ptr(), o_dev.data_ptr(), g_dev.data_ptr(), n,
                                              float(np.float32(1 / 2 / OPTS["affinity_eps"] ** 2)), m.data_ptr(),
                                              rt.stream_ptr(torch, dev)), "affinity")
            want = so.affinity_matrix(c, o, cf, of, fmat, OPTS["epi_weight"], OPTS["affinity_eps"])
            assert np.array_equal(m.cpu().numpy(), want)


def test_errors_surface_as_exceptions():
    st = APAP(0.5, 100, [64, 48], [0, 0])
    with pytest.raises(ValueError):
        st.local_homography(np.zeros((10, 3), np.float32), np.zeros((10, 2), np.float32), np.zeros((2, 2, 2)))
    with pytest.raises(ValueError):
        apap_utils.uniform_blend(np.zeros((4, 4, 3), np.uint8), np.zeros((4, 5, 3), np.uint8))
    lib = rt.load_library()
    assert lib.apap_blend(None, None, None, 10, None) != 0
    assert b"null" in lib.apap_last_error()


def test_integration_md_ctypes_stub_runs_and_matches():
    """The ctypes stub INTEGRATION.md shows a reference maintainer (raw C ABI, no cvx_proj_b200 host layer) is executed
    as written and gives the same H grid as the package's own call, bit for bit."""
    import os
    import re
    import types
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    text = open(os.path.join(root, "INTEGRATION.md")).read()
    block = re.search(r"```python\n(import ctypes, math.*?)```", text, re.S).group(1)
    block = block.replace('ctypes.CDLL("libapap_b200.so")', f'ctypes.CDLL({rt.LIB_PATH!r})')
    ns = {}
    exec(compile(block, "INTEGRATION.md", "exec"), ns)
    sc = synth.make_scene("mini")
    st = _stitcher(sc)
    st.local_homography_stub = types.MethodType(ns["local_homography"], st)
    got, _ = st.local_homography_stub(sc.src, sc.dst, sc.vertices)
    want, _ = st.local_homography(sc.src, sc.dst, sc.vertices)
    assert got.shape == want.shape
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))


def test_device_invert_grid_has_numpys_bits():
    """APAP.invert_grid (GPU float64 inverse + certificate, numpy for the uncertified cells) leaves exactly the bits of
    the reference's per-cell np.linalg.inv (pyviz/apap.py:201-203) in the caller's array: a real grid, two million
    homography-like cells of mixed conditioning (a plain float64 LU rounds ~1 in 10^6 entries differently),
    affine cells (exact zeros), NaN cells, a float64 grid; singular cells raise like numpy."""
    sc = synth.make_scene("c2")
    st = _stitcher(sc)
    h, _ = st.local_homography(sc.src, sc.dst, sc.vertices)
    want = np.linalg.inv(h)
    redo = st.invert_grid(h)
    assert np.array_equal(h.view(np.uint32), want.view(np.uint32))
    print(f"invert_grid c2: {redo} of {h.size // 9} cells went through numpy")
    assert redo < 0.01 * h.size / 9

    rng = np.random.default_rng(17)
    n = 2_000_000
    g = np.tile(np.eye(3), (n, 1, 1))
    g[:, :2, :2] += rng.normal(0, 0.2, (n, 2, 2))
    g[:, :2, 2] = rng.normal(0, 1, (n, 2)) * 10.0 ** rng.uniform(0, 3.7, (n, 1))
    g[:, 2, :2] = rng.normal(0, 1, (n, 2)) * 10.0 ** rng.uniform(-7, -3, (n, 1))
    g *= 10.0 ** rng.uniform(-2, 2, (n, 1, 1))
    g = g.astype(np.float32)
    g[::1000, 2, :2] = 0                                    # affine cells: exact zeros in the inverse
    g[5] = np.nan
    want = np.linalg.inv(g)
    redo = st.invert_grid(g)
    same = g.view(np.uint32) == want.view(np.uint32)
    print(f"invert_grid stress: {redo} of {n} cells through numpy, {int((~same).sum())} differing entries")
    assert same.all()
    assert redo < 0.02 * n

    # families far from homographies: what the device certifies still has numpy's bits, the rest goes through numpy
    m = 200_000
    families = {
        "uniform": rng.uniform(-1, 1, (m, 3, 3)),
        "row scales": rng.normal(0, 1, (m, 3, 3)) * 10.0 ** rng.uniform(-6, 6, (m, 3, 1)),
        "near rank 1": rng.normal(0, 1, (m, 3, 1)) * rng.normal(0, 1, (m, 1, 3))
        + 10.0 ** rng.uniform(-7, -3, (m, 1, 1)) * rng.normal(0, 1, (m, 3, 3)),
        "small integers": rng.integers(-3, 4, (m, 3, 3)).astype(np.float64) + 4 * np.eye(3),
    }
    for name, fam in families.items():
        fam = fam.astype(np.float32)
        fam = fam[np.abs(np.linalg.det(fam.astype(np.float64))) > 1e-30]       # numpy itself raises on singular cells
        want_f = np.linalg.inv(fam)
        redo_f = st.invert_grid(fam)
        print(f"invert_grid {name}: {redo_f} of {len(fam)} cells through numpy")
        assert np.array_equal(fam.view(np.uint32), want_f.view(np.uint32)), name

    g64 = np.linalg.inv(want[100:200].astype(np.float64))
    want64 = np.linalg.inv(g64)
    assert st.invert_grid(g64) == 100 and np.array_equal(g64, want64)            # not float32: numpy throughout
    bad = np.tile(np.eye(3, dtype=np.float32), (4, 1, 1))
    bad[2] = 0
    with pytest.raises(np.linalg.LinAlgError):
        st.invert_grid(bad)


def test_sharded_pass_over_nccl_two_gpus_is_bit_identical():
    """Two ranks over NCCL (torchrun, one rank per GPU): the cell-row / row-band sharded pass equals the one-GPU pass
    bit for bit -- H grid, all-gathered panorama, and the panorama assembled through the NVLS multicast mapping
    (broadcast kernel and the warp kernel's own multimem stores).  tools/check_sharded_nccl.py is the rank program.
    Skips on a box with fewer than two GPUs."""
    import subprocess
    import sys
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    repo = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
           "--master-port", "29541", os.path.join(repo, "tools", "check_sharded_nccl.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=repo)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert "SHARDED NCCL CHECK PASSED" in res.stdout, res.stdout[-3000:]


@pytest.mark.parametrize("name", ["mini", "c1", "c2"])
def test_local_warp_bilinear_opt_in_within_one_lsb_of_float64_restatement(name):
    """BASELINE.json north_star: "bilinear sample ... warped pixels within +-1 LSB".  The opt-in mode writes exactly the
    pixels the reference's truncating mode writes and samples them bilinearly; gate: |GPU - float64 oracle| <= 1."""
    sc = synth.make_scene(name)
    img = sc.image(1)
    st = _stitcher(sc)
    h = orc.local_homography_gram64(sc.src, sc.dst, sc.vertices[::8, ::8], sc.gamma, sc.sigma) if name == "c2" else \
        orc.local_homography_gram64(sc.src, sc.dst, sc.vertices, sc.gamma, sc.sigma)
    if name == "c2":
        h = np.repeat(np.repeat(h, 8, 0), 8, 1).copy()
    inv = orc.invert_grid(h)
    want = orc.local_warp_bilinear(img, inv, sc.mesh, (sc.final_w, sc.final_h), (sc.offset_x, sc.offset_y))
    grid = h.copy()
    got = st.local_warp(img, grid, sc.mesh, interpolation="bilinear")
    assert np.array_equal(grid, inv)                                        # same in-place inverse as the parity mode
    diff = np.abs(got.astype(np.int16) - want.astype(np.int16))
    assert diff.max() <= 1, f"max |diff| {diff.max()}"
    assert (diff != 0).mean() < 0.02
    nearest = st.local_warp(img, h.copy(), sc.mesh)
    assert np.array_equal(got.any(axis=-1), nearest.any(axis=-1))           # the same pixels are written (images are >= 1)
    with pytest.raises(ValueError):
        st.local_warp(img, h.copy(), sc.mesh, interpolation="cubic")


def test_peer_copy_writes_every_listed_buffer():
    """apap_peer_copy (the unicast panorama assembly): every listed destination receives the band, bytes outside stay;
    argument checks fire before anything is launched.  (Peers are buffers of this GPU here; tools/assemble_lab.py and
    tools/check_sharded_nccl.py run it across GPUs.)"""
    import ctypes
    import torch
    dev = torch.device("cuda", torch.cuda.current_device())
    lib = rt.load_library()
    stream = rt.stream_ptr(torch, dev)
    for n_bytes, n_peers in ((16, 1), (4096 + 16, 3), (1 << 20, 15)):
        src = torch.randint(0, 256, (n_bytes,), dtype=torch.uint8, device=dev)
        dsts = [torch.full((n_bytes + 32,), 7, dtype=torch.uint8, device=dev) for _ in range(n_peers)]
        ptrs = (ctypes.c_void_p * n_peers)(*[d.data_ptr() + 16 for d in dsts])
        rt.check(lib.apap_peer_copy(src.data_ptr(), ptrs, n_peers, n_bytes, stream), "apap_peer_copy")
        torch.cuda.synchronize()
        for d in dsts:
            assert torch.equal(d[16:16 + n_bytes], src) and int(d[:16].min()) == 7 and int(d[-16:].max()) == 7
    bad = (ctypes.c_void_p * 1)(src.data_ptr() + 8)
    assert lib.apap_peer_copy(src.data_ptr(), bad, 1, 16, stream) != 0            # misaligned destination
    assert lib.apap_peer_copy(src.data_ptr(), ptrs, 16, 16, stream) != 0           # more than APAP_MAX_PEERS
    assert lib.apap_peer_copy(src.data_ptr(), ptrs, 1, 24, stream) != 0            # size not a multiple of 16


def test_spectral_power_iteration_reports_a_repeated_leading_eigenvalue(monkeypatch):
    """Two disjoint, identical clusters of consistent matches: the affinity matrix is block diagonal with two equal
    leading eigenvalues, the power iteration cannot settle on one vector -- it must say so (RuntimeWarning,
    info['converged'] False) instead of returning a mixture silently.  A single cluster converges and says that."""
    from cvx_proj_b200 import spectral_method as psm
    rng = np.random.default_rng(3)
    a = rng.uniform(0, 50, size=(24, 2)).astype(np.float32)
    src = np.concatenate([a, a + np.float32(4000.0)])
    dst = np.concatenate([a + np.float32(3.0), a + np.float32(9000.0)])      # second cluster far away in both images
    diag = np.full(48, 0.9)
    monkeypatch.setattr(psm, "POWER_MAX_ITER", 256)
    with pytest.warns(RuntimeWarning, match="repeated"):
        _, info = psm.spectral_segment_device(src, dst, diag, 30.0, return_info=True)
    assert info["converged"] is False and info["iterations"] == 256
    seg, info = psm.spectral_segment_device(src[:24], dst[:24], diag[:24], 30.0, return_info=True)
    assert info["converged"] is True and seg.max() == 1.0


def test_lazy_local_weight_behaves_like_the_reference_ndarray():
    """ADVICE round 1: the lazy second return value takes numpy arithmetic, reductions and boolean indexing, keeps
    float64 keypoints in float64 (the reference subtracts them from float64 vertices), and refuses to build tens of GB
    in one piece."""
    sc = synth.make_scene("mini")
    st = _stitcher(sc)
    src64 = sc.src.astype(np.float64) + 1e-7                      # not representable in float32
    _, w = st.local_homography(src64, sc.dst, sc.vertices)
    want = orc.local_weight(src64, sc.vertices, sc.gamma, sc.sigma)
    got = np.asarray(w)
    assert got.shape == want.shape and np.allclose(got, want, rtol=1e-13, atol=0)
    assert np.allclose(w * 2, want * 2, rtol=1e-13) and np.allclose(2 - w, 2 - want, rtol=1e-12)
    assert np.isclose(w.sum(), want.sum(), rtol=1e-12) and np.isclose(np.mean(w), want.mean(), rtol=1e-12)
    assert np.array_equal(w[w > 0.9], got[got > 0.9]) and (w >= sc.gamma).all()
    assert np.array_equal(np.concatenate([w, w], axis=0), np.concatenate([got, got], axis=0))
    big = type(w)(sc.src, sc.vertices, sc.gamma, sc.sigma)
    big.materialize_limit = 1 << 10
    with pytest.raises(MemoryError):
        np.asarray(big)
    assert big[0].shape == want[0].shape                          # slices still stream


# ------------------------------------------------------------- keypoint-pair producer: matcher (SURVEY 8f, N3)
def _sift_like(rng, n, dim=128):
    """Integer-valued float32 descriptors with SIFT's range and norm (0..255, L2 norm ~512)."""
    d = rng.gamma(0.6, 1.0, size=(n, dim))
    d = d / np.linalg.norm(d, axis=1, keepdims=True) * 512.0
    return np.minimum(np.rint(d), 255.0).astype(np.float32)


@pytest.mark.parametrize("nq,nt", [(1, 1), (5, 3), (64, 32), (65, 33), (381, 381), (3975, 4100), (300, 20000)])
def test_exact_matcher_equals_cv_bfmatcher(nq, nt):
    """apap_match_nn against the live cv.BFMatcher(NORM_L2).match and the numpy oracle on SIFT-like descriptors: same
    train index and the same float32 distance bits for every query, duplicates in the train set included (a tie
    falls to the lowest train index, as in OpenCV)."""
    import cv2 as cv
    from cvx_proj_b200.utils import match_descriptors
    from oracle import match_oracle as mo
    rng = np.random.default_rng(nq * 7 + nt)
    train = _sift_like(rng, nt)
    noise = rng.integers(-6, 7, size=(nq, 128)).astype(np.float32)
    query = np.clip(train[rng.integers(0, nt, size=nq)] + noise, 0, 255).astype(np.float32)
    if nt >= 8:
        train[nt // 2] = train[1]                                  # an exact duplicate: ties
        query[0] = train[1]
    idx, dist = match_descriptors(query, train)
    want_idx, want_dist = mo.exact_match(query, train)
    assert np.array_equal(idx, want_idx) and np.array_equal(dist.view(np.uint32), want_dist.view(np.uint32))
    bf = cv.BFMatcher(cv.NORM_L2).match(query, train)
    assert len(bf) == nq
    assert np.array_equal(idx, np.array([m.trainIdx for m in bf], dtype=np.int32))
    assert np.array_equal(dist.view(np.uint32), np.array([m.distance for m in bf], dtype=np.float32).view(np.uint32))
    if nt >= 8:
        assert idx[0] == 1 and dist[0] == 0.0


def test_exact_matcher_edge_cases_and_general_floats():
    """Empty sets, other descriptor widths, CUDA tensors in / out, and non-integer descriptors: the index is the exact
    nearest neighbour wherever the two smallest distances differ by more than float32 rounding."""
    import torch
    from cvx_proj_b200.utils import match_descriptors
    from oracle import match_oracle as mo
    rng = np.random.default_rng(0)
    idx, dist = match_descriptors(np.zeros((0, 128), np.float32), _sift_like(rng, 10))
    assert idx.shape == (0,) and dist.shape == (0,)
    idx, dist = match_descriptors(_sift_like(rng, 7), np.zeros((0, 128), np.float32))
    assert (idx == -1).all() and np.isinf(dist).all()
    for dim in (2, 64, 130, 256):
        q, t = rng.standard_normal((97, dim)).astype(np.float32), rng.standard_normal((211, dim)).astype(np.float32)
        idx, dist = match_descriptors(q, t)
        d2 = ((q[:, None, :].astype(np.float64) - t[None].astype(np.float64)) ** 2).sum(-1)
        order = np.sort(d2, axis=1)
        clear = order[:, 1] - order[:, 0] > 1e-5 * order[:, 1]
        assert clear.mean() > 0.9 and np.array_equal(idx[clear], d2.argmin(1)[clear])
        assert np.allclose(dist, np.sqrt(d2[np.arange(97), idx]), rtol=1e-5)
    dev = torch.device("cuda", torch.cuda.current_device())
    q, t = _sift_like(rng, 130), _sift_like(rng, 70)
    idx_d, dist_d = match_descriptors(torch.from_numpy(q).to(dev), torch.from_numpy(t).to(dev))
    assert idx_d.is_cuda and np.array_equal(idx_d.cpu().numpy(), mo.exact_match(q, t)[0])
    with pytest.raises(rt.ApapError):
        match_descriptors(np.zeros((3, 7), np.float32), np.zeros((3, 7), np.float32))       # odd width


def test_coarse_matching_mirror_on_a_synthetic_pair():
    """cvx_proj_b200.utils.coarse_matching (pyviz/utils.py:142-151): OpenCV's own SIFT descriptors at the given keypoints,
    matches = the exact nearest neighbours; on a pair related by a known homography nearly all of them are the true
    correspondences, and cv.findHomography on them (the reference's next call, baseline_stitch_test.py:40) recovers it."""
    import cv2 as cv
    from cvx_proj_b200.utils import coarse_matching
    sc = synth.make_scene("c1")
    img_c = synth.make_image(sc.width, sc.height, seed=2)
    hinv = np.linalg.inv(sc.h_gt)
    img_o = cv.warpPerspective(img_c, hinv, (sc.width, sc.height))
    raw_c = sc.dst.astype(np.float32)
    raw_o = cv.perspectiveTransform(raw_c[None].astype(np.float64), hinv)[0].astype(np.float32)
    keep = np.all((raw_o > 16) & (raw_o < [sc.width - 16, sc.height - 16]) & (raw_c > 16) & (raw_c < [sc.width - 16, sc.height - 16]), axis=1)
    raw_c, raw_o = raw_c[keep], raw_o[keep]
    kc, fc, ko, fo, matches = coarse_matching(img_c, img_o, raw_c, raw_o)
    assert len(matches) == len(kc) == fc.shape[0] and all(isinstance(m, cv.DMatch) for m in matches)
    bf = cv.BFMatcher(cv.NORM_L2).match(fc, fo)
    assert [m.trainIdx for m in matches] == [m.trainIdx for m in bf]
    assert np.mean([m.trainIdx == m.queryIdx for m in matches]) > 0.8
    src = np.float32([kc[m.queryIdx].pt for m in matches]); dst = np.float32([ko[m.trainIdx].pt for m in matches])
    h, mask = cv.findHomography(src, dst, cv.RANSAC, 5.0)
    assert mask.sum() > 0.8 * len(matches) and np.abs(h / h[2, 2] - hinv / hinv[2, 2]).max() < 0.05 * np.abs(hinv / hinv[2, 2]).max()


def test_one_call_pass_equals_the_separate_entry_points():
    """apap_local_homography_points (what APAP.local_homography calls: anchors scaled, conditioned, tabled, bounded and
    solved by ONE library call) gives the same H bits as the separate entry points driven from Python, for a single
    pair, a ragged batch, both engines, and with pinned or pageable vertices."""
    import torch
    from cvx_proj_b200.apap import scale_anchors, weight_scale
    dev = torch.device("cuda", torch.cuda.current_device())
    for engine in ENGINES:
        sc = synth.make_scene("c1")
        st = _stitcher(sc, engine=engine)
        h, _ = st.local_homography(sc.src, sc.dst, sc.vertices)
        vert_pin = rt.pinned_empty(sc.vertices.shape, np.float64); vert_pin[...] = sc.vertices
        h_pin, _ = st.local_homography(sc.src, sc.dst, vert_pin)
        raw = torch.from_numpy(np.stack([sc.src, sc.dst]).astype(np.float32)[:, None]).to(dev)
        cond, tmats = st.condition_device(raw)
        rows = st.kp_rows_device((cond[0], cond[1], raw[0]))
        a = torch.from_numpy(scale_anchors(sc.vertices, weight_scale(sc.sigma))[None]).to(dev)
        bound = st.weight_bound_device(raw[0], None, a)
        want = st.local_homography_device(st.kp_table_device(rows), a, tmats, 1, sc.n_cells, t_bound=bound).cpu().numpy()
        assert np.array_equal(h.reshape(-1, 9).view(np.uint32), want.reshape(-1, 9).view(np.uint32))
        assert np.array_equal(h.view(np.uint32), h_pin.view(np.uint32))
        # ragged batch: every item equals its single-pair call
        scs = [synth.make_scene("mini", seed=k, n_kp=n) for k, n in enumerate((200, 131, 77))]
        stb = _stitcher(scs[0], engine=engine)
        got = stb.local_homography_batch([s.src for s in scs], [s.dst for s in scs], [s.vertices for s in scs])
        for s_, g in zip(scs, got):
            one, _ = stb.local_homography(s_.src, s_.dst, s_.vertices)
            assert np.array_equal(g.view(np.uint32), one.view(np.uint32))
