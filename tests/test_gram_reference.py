"""The moving-DLT kernels one at a time against a float64 reference (oracle/gram_oracle.py).

K1 (``apap_gram_partials``, both engines) is compared split by split with ``partials64`` under the per-entry bound
``gate`` -- at every split, segment and cell-tile boundary of the plan, on both weight paths and both kinds of
keypoint table -- and must leave the padding columns of ``partials`` unwritten.  K2 (``apap_eig_denorm``) is fed
synthetic float32 planes and compared with ``eig64``.  The H-level tests (tests/test_gpu_parity.py) use the 1e-4
contract gate, which a K1 that lost a k-block still passes; these gates are far tighter, and the CPU tests below check
that a lost k-block exceeds them tenfold.
"""
import math

import numpy as np
import pytest

from cvx_proj_b200 import synth
from cvx_proj_b200 import _runtime as rt
from cvx_proj_b200.apap import APAP, build_kp_blocks, build_kp_table, scale_anchors, weight_scale
from oracle import apap_oracle as orc
from oracle import gram_oracle as go

ENGINES = {"tcgen05": go.GRAM_TCGEN05, "ffma2": go.GRAM_FFMA2}
# keypoint counts at the plan's boundaries: chunk (128), segment (256), one-chunk splits (384), a short last split
# (640), the FFMA2 split cap (1024 / 1025), the tensor-core cap (2048 / 2049), five tensor-core splits ending on a half
# segment (8320), c3 (20000)
COUNTS = [1, 7, 8, 9, 128, 129, 255, 256, 257, 384, 640, 1024, 1025, 2048, 2049, 8320, 20000]
# cell tiles are 128 cells; 513 leaves one cell in the last tile and cells_padded = 1024
CELLS = [1, 127, 128, 129, 513]
K2_SPLITS = [1, 2, 3, 10, 64]
H_TIGHT = 1e-6            # K2 against eig64, normalised H error (100x under the contract's 1e-4)
RESIDUAL = 1e-5           # K2 on degenerate sets: ||G h|| / (||G|| ||h||)


# ------------------------------------------------------------------------------------------- K1 cases
def _pad(n):
    return max(go.KP_CHUNK, -(-n // go.KP_CHUNK) * go.KP_CHUNK)


def _dlt_rows(n_kp, sigma=100.0, seed=0, name="c1"):
    """Real DLT rows (``APAP._prepare``) of the first n_kp matches of a synthetic scene, padded like the product pads
    them; the scene has at least 64 matches so that its conditioning is defined whatever n_kp."""
    sc = synth.make_scene(name, n_kp=max(n_kp, 64), seed=seed)
    full, _ = APAP(0.5, sigma, [sc.final_w, sc.final_h], [sc.offset_x, sc.offset_y])._prepare(sc.src, sc.dst)
    rows = np.zeros((_pad(n_kp), 28), dtype=np.float32)
    rows[:n_kp] = full[:n_kp]
    return rows, sc


def _synthetic_rows(rows, n_kp, seed):
    """The same keypoints with synthetic product terms: mixed signs, exact zeros and magnitudes 2^-30 .. 2^30 (every
    bit of the mantissa set at random), which stress the TF32 head / tail split of the tensor-core table."""
    rng = np.random.default_rng(seed)
    out = rows.copy()
    mag = np.ldexp(rng.uniform(1.0, 2.0, (n_kp, go.TERMS)), rng.integers(-30, 31, (n_kp, go.TERMS)))
    val = np.where(rng.random((n_kp, go.TERMS)) < 0.1, 0.0, mag * rng.choice([-1.0, 1.0], (n_kp, go.TERMS)))
    out[:n_kp, :go.TERMS] = val.astype(np.float32)
    return out


def _random_anchors(sc, cells, sigma, seed):
    rng = np.random.default_rng(seed)
    v = rng.uniform([-0.1 * sc.width, -0.1 * sc.height], [1.1 * sc.width, 1.1 * sc.height], size=(cells, 2))
    return scale_anchors(v, weight_scale(sigma))


class K1Case:
    """One launch of K1: per scene a row table and anchors, the clamp, and (optionally) the subset of cells the
    reference is computed on."""

    def __init__(self, name, rows, anchors, gamma, counts, raw_src=None, cell_idx=None, bound=False):
        self.name, self.rows, self.anchors = name, rows, anchors          # [B, n_pad, 28], [B, cells, 2]
        self.gamma_sq = np.float32(gamma * gamma)
        self.counts = counts                                              # real keypoints per scene
        self.raw_src = raw_src                                            # [B, n, 2] raw points (t_bound)
        self.cell_idx = cell_idx
        self.bound = bound

    @property
    def n_pad(self):
        return self.rows.shape[1]

    @property
    def cells(self):
        return self.anchors.shape[1]

    def reference(self, engine, b):
        a = self.anchors[b] if self.cell_idx is None else self.anchors[b][self.cell_idx]
        ref = go.partials64(self.rows[b], a, self.gamma_sq, self.n_pad, engine)
        A, T = go.abs_sums64(self.rows[b], a, self.gamma_sq, self.n_pad, engine)
        return ref, A, T


def _grid_case(n_kp, cells, table):
    rows, sc = _dlt_rows(n_kp)
    if table == "synthetic":
        rows = _synthetic_rows(rows, n_kp, seed=n_kp)
    return K1Case(f"n{n_kp}-c{cells}-{table}", rows[None], _random_anchors(sc, cells, 100.0, seed=cells)[None], 0.5,
                  [n_kp])


def _strided(cells, stride):
    return np.unique(np.concatenate([np.arange(128), np.arange(0, cells, stride), np.arange(cells - 128, cells)]))


def _full_grid_case(name, n_kp, stride):
    sc = synth.make_scene(name, n_kp=n_kp)
    rows, _ = APAP(sc.gamma, sc.sigma, [sc.final_w, sc.final_h], [sc.offset_x, sc.offset_y])._prepare(sc.src, sc.dst)
    a = scale_anchors(sc.vertices, weight_scale(sc.sigma))
    return K1Case(f"{name}-grid", rows[None], a[None], sc.gamma, [n_kp], cell_idx=_strided(a.shape[0], stride))


def _batch_case():
    """Three scenes of different tables, counts and anchors in one launch (cross-scene indexing)."""
    counts = [3001, 2000, 257]
    n_pad = _pad(max(counts))
    rows = np.zeros((3, n_pad, 28), dtype=np.float32)
    anchors = []
    for b, n in enumerate(counts):
        r, sc = _dlt_rows(n, seed=b + 1)
        rows[b, :r.shape[0]] = r
        anchors.append(_random_anchors(sc, 700, 100.0, seed=10 + b))
    return K1Case("batch3", rows, np.stack(anchors), 0.5, counts)


def _weight_case(kind):
    n_kp, cells = 2049, 513
    gamma, sigma = {"poly": (0.5, 100.0), "poly-bound": (0.5, 100.0), "mufu": (0.3, 100.0), "clamped": (1.0, 100.0),
                    "gamma-gt-1": (1.7, 50.0), "far": (0.05, 8.0), "exact-t": (0.5, 100.0)}[kind]
    rows, sc = _dlt_rows(n_kp, sigma=sigma)
    anchors = _random_anchors(sc, cells, sigma, seed=99)
    if kind == "exact-t":
        # keypoint coordinates moved onto multiples of 2^-20 so that an anchor 2 away (2^-t = gamma^2 = 1/4, the end
        # of the polynomial's range) is exact in float32; then anchors on keypoints (t = 0) and 2 to their right
        k = np.arange(0, n_kp, 32)[:64]
        rows[k, 24:28] = np.round(rows[k, 24:28] * 2.0 ** 20) * 2.0 ** -20
        anchors[0:64] = rows[k][:, [24, 26]]
        anchors[64:128] = rows[k][:, [24, 26]] + np.float32([2.0, 0.0])
        assert (np.hypot(anchors[64:128, 0].astype(np.float64) - rows[k, 24], anchors[64:128, 1].astype(np.float64)
                         - rows[k, 26]) == 2.0).all()
    return K1Case(f"weights-{kind}", rows[None], anchors[None], gamma, [n_kp], raw_src=sc.src[None, :n_kp],
                  bound=kind == "poly-bound")


GRID = [(n, c) for n in COUNTS for c in CELLS]
EXTRA = ["c2-grid", "c3-grid", "batch3"] + [f"weights-{k}" for k in
                                             ("poly", "poly-bound", "mufu", "clamped", "gamma-gt-1", "far", "exact-t")]
_CACHE = {}


def _case(key):
    if key not in _CACHE:
        if isinstance(key, tuple):
            c = _grid_case(*key)
        elif key == "c2-grid":
            c = _full_grid_case("c2", 5000, 97)
        elif key == "c3-grid":
            c = _full_grid_case("c3", 20000, 409)
        elif key == "batch3":
            c = _batch_case()
        else:
            c = _weight_case(key[len("weights-"):])
        _CACHE.clear()                     # one case at a time: the big ones hold hundreds of MB of reference
        _CACHE[key] = c
    return _CACHE[key]


ALL_CASES = [(n, c, t) for n, c in GRID for t in ("dlt", "synthetic")] + EXTRA


def _case_id(key):
    return "-".join(str(k) for k in key) if isinstance(key, tuple) else key


# ------------------------------------------------------------------------------------------------ CPU
def test_plan_restatement_equals_apap_gram_plan():
    for engine in ENGINES.values():
        for n_chunks in range(1, 601):
            n_pad = n_chunks * go.KP_CHUNK
            for cells in (1, 513):
                ks, cp, nbytes = rt.gram_plan(cells, n_pad, engine)
                assert (ks, cp) == (go.plan(n_pad, engine)[0], go.cells_padded(cells)), (engine, n_chunks)
                assert nbytes == ks * go.TERMS * cp * 4
            r = go.split_ranges(n_pad, engine)
            assert r[0][0] == 0 and r[-1][1] == n_pad and all(a[1] == b[0] for a, b in zip(r, r[1:]))
            cap = go.SPLIT_CAP[engine] * go.KP_CHUNK
            assert all(0 < k1 - k0 <= cap for k0, k1 in r)


def test_boundaries_of_the_plan_are_covered_by_the_counts():
    """Each boundary of the docstring of COUNTS has a count on both sides of it."""
    plans = {n: {e: go.split_ranges(_pad(n), e) for e in ENGINES.values()} for n in COUNTS}
    tc, ff = go.GRAM_TCGEN05, go.GRAM_FFMA2
    assert any(len(plans[n][ff]) == 3 and plans[n][ff][-1][1] - plans[n][ff][-1][0] == 128 for n in COUNTS)
    assert any(len({k1 - k0 for k0, k1 in plans[n][tc]}) == 2 for n in COUNTS)            # a shorter last split
    assert any(max(k1 - k0 for k0, k1 in plans[n][ff]) == 1024 for n in COUNTS)
    assert any(len(plans[n][tc]) == 5 and (plans[n][tc][-1][1] - plans[n][tc][-1][0]) % go.SEGMENT for n in COUNTS)
    for b in (128, 256, 1024, 2048):
        assert b in COUNTS and b + 1 in COUNTS
    assert any(c % 128 == 1 for c in CELLS) and any(c % 128 == 127 for c in CELLS) and 513 in CELLS


@pytest.mark.parametrize("name", ["mini", "c1"])
def test_partials64_and_eig64_reproduce_the_float64_gram_oracle(name):
    sc = synth.make_scene(name)
    st = APAP(sc.gamma, sc.sigma, [sc.final_w, sc.final_h], [sc.offset_x, sc.offset_y])
    rows, tmats = st._prepare(sc.src, sc.dst)
    a = scale_anchors(sc.vertices, weight_scale(sc.sigma))
    want = orc.local_homography_gram64(sc.src, sc.dst, sc.vertices, sc.gamma, sc.sigma, dtype=np.float64)
    for engine in ENGINES.values():
        h, _, _ = go.eig64(go.partials64(rows, a, np.float32(sc.gamma ** 2), rows.shape[0], engine), tmats,
                           dtype=np.float64)
        err = orc.h_error_normalised(h, want, max(sc.final_w, sc.final_h))
        assert err.max() <= 1e-7, err.max()


def _removal_positions(case, engine, b):
    """Keypoint index of the k-blocks whose loss must be visible: the first, the first of the second segment, the first
    of the last split, the last real one."""
    n = case.counts[b]
    last_split = go.split_ranges(case.n_pad, engine)[-1][0]
    pos = {0, go.SEGMENT, last_split, (n - 1) // go.KP_BLOCK * go.KP_BLOCK}
    return sorted(p for p in pos if p < n)


@pytest.mark.parametrize("key", ALL_CASES, ids=_case_id)
def test_a_lost_k_block_exceeds_the_gate_tenfold(key):
    """Sensitivity of the K1 gate: on every K1 case of the GPU tests, removing one 8-keypoint block at a split,
    segment or end boundary moves some partial entry by at least 10x its gate."""
    case = _case(key)
    for engine in ENGINES.values():
        for b in range(case.rows.shape[0]):
            _, A, T = case.reference(engine, b)
            g = go.gate(A, T, engine)
            a = case.anchors[b] if case.cell_idx is None else case.anchors[b][case.cell_idx]
            ranges = go.split_ranges(case.n_pad, engine)
            for p in _removal_positions(case, engine, b):
                s = max(i for i, (k0, _) in enumerate(ranges) if k0 <= p)
                _, w2 = go.weights64(case.rows[b], a, case.gamma_sq, p, p + go.KP_BLOCK)
                delta = np.abs(w2 @ case.rows[b, p:p + go.KP_BLOCK, :go.TERMS].astype(np.float64)).T     # [24, cells]
                worst = (delta / np.maximum(g[s], 1e-300)).max()
                assert worst >= 10.0, (key, engine, b, p, worst)


# ------------------------------------------------------------------------------------------------ GPU
@pytest.fixture(scope="module")
def cuda():
    import torch
    return torch, torch.device("cuda", torch.cuda.current_device())


def _upload_table(torch, dev, rows, engine):
    tab = rows if engine == go.GRAM_FFMA2 else np.stack([build_kp_blocks(r) for r in rows])
    return torch.from_numpy(np.ascontiguousarray(tab)).to(dev)


def _launch_k1(cuda, case, engine, table=None):
    """K1 on partials filled with NaN; returns [B, k_splits, 24, cells_padded] float32 on the host."""
    torch, dev = cuda
    lib = rt.load_library()
    batch = case.rows.shape[0]
    ks, cp, nbytes = rt.gram_plan(case.cells, case.n_pad, engine)
    t = _upload_table(torch, dev, case.rows, engine) if table is None else table
    a = torch.from_numpy(np.ascontiguousarray(case.anchors)).to(dev)
    bound = None
    if case.bound:
        st = APAP(math.sqrt(float(case.gamma_sq)), 100.0, [1, 1], [0, 0])
        raw = torch.from_numpy(np.ascontiguousarray(case.raw_src, dtype=np.float32)).to(dev)
        bound = st.weight_bound_device(raw, None, a)
        b = float(bound.cpu().numpy().max())
        assert b * 1.001 + 1e-3 < min(-math.log2(float(case.gamma_sq)), 2.0), "the case must take the clamp-free loop"
    part = torch.full((batch * nbytes // 4,), float("nan"), dtype=torch.float32, device=dev)
    rt.check(lib.apap_gram_partials(t.data_ptr(), a.data_ptr(), batch, case.cells, case.n_pad, float(case.gamma_sq),
                                    engine, bound.data_ptr() if bound is not None else None, part.data_ptr(),
                                    rt.stream_ptr(torch, dev)), "apap_gram_partials")
    return part.cpu().numpy().reshape(batch, ks, go.TERMS, cp)


def _compare(case, engine, got):
    """(max |err| / gate, max |err| / A, sum of |err| / A, entries) over the scenes of the case; asserts the NaN
    padding."""
    worst_gate = worst_a = 0.0
    sum_a, n_a = 0.0, 0
    for b in range(case.rows.shape[0]):
        assert np.isnan(got[b, :, :, case.cells:]).all(), "K1 wrote into the padding columns of partials"
        sub = got[b, :, :, :case.cells] if case.cell_idx is None else got[b][:, :, case.cell_idx]
        assert np.isfinite(sub).all(), "K1 left a partial entry unwritten or non-finite"
        ref, A, T = case.reference(engine, b)
        err = np.abs(sub.astype(np.float64) - ref)
        g = go.gate(A, T, engine)
        assert (err[g == 0] == 0).all()
        pos = A > 0
        r = err[pos] / A[pos]
        worst_gate = max(worst_gate, float((err[pos] / g[pos]).max()))
        worst_a = max(worst_a, float(r.max()))
        sum_a += float(r.sum())
        n_a += r.size
    return worst_gate, worst_a, sum_a, n_a


@pytest.fixture(scope="module")
def k1_stats():
    """Per engine [max |err| / gate, max |err| / A, sum of |err| / A, entries] over every K1 case; printed at the end
    (the accuracy figures of csrc/gram_tc.cu and DESIGN.md)."""
    stats = {}
    yield stats
    for name, (g, mx, total, n) in stats.items():
        print(f"\nK1 [{name}] over all cases: max |err|/gate {g:.3f}, |err|/A max {mx:.2e} mean {total / n:.2e}")


@pytest.mark.gpu
@pytest.mark.parametrize("key", ALL_CASES, ids=_case_id)
def test_k1_partials_within_gate_of_float64_reference(cuda, k1_stats, key):
    case = _case(key)
    bad = []
    for name, engine in ENGINES.items():
        if case.bound and engine == go.GRAM_FFMA2:
            continue                                   # t_bound only steers the tensor-core kernel
        got = _launch_k1(cuda, case, engine)
        worst_gate, worst_a, sum_a, n_a = _compare(case, engine, got)
        print(f"K1 {case.name} [{name}]: max |err|/gate {worst_gate:.3f}, max |err|/A {worst_a:.2e}, "
              f"mean |err|/A {sum_a / max(n_a, 1):.2e}")
        acc = k1_stats.setdefault(name, [0.0, 0.0, 0.0, 0])
        acc[0], acc[1] = max(acc[0], worst_gate), max(acc[1], worst_a)
        acc[2] += sum_a
        acc[3] += n_a
        if worst_gate > 1.0:
            bad.append((name, worst_gate))
    assert not bad, bad


@pytest.mark.gpu
@pytest.mark.parametrize("engine", list(ENGINES))
def test_k1_negative_control_a_zeroed_k_block_is_detected(cuda, engine):
    """The first k-block of the second segment zeroed in the uploaded table (a data change only): the comparison with
    the reference of the unmodified table must fail, so the gate sees a lost block on the real kernel."""
    torch, dev = cuda
    eng = ENGINES[engine]
    case = _case((8320, 129, "dlt"))
    t = _upload_table(torch, dev, case.rows, eng)
    if eng == go.GRAM_FFMA2:
        t[0, go.SEGMENT:go.SEGMENT + go.KP_BLOCK] = 0.0
    else:
        t[0, go.SEGMENT // go.KP_BLOCK] = 0.0
    worst_gate = _compare(case, eng, _launch_k1(cuda, case, eng, table=t))[0]
    print(f"K1 negative control [{engine}]: zeroed k-block at keypoint {go.SEGMENT} detected, "
          f"max |err|/gate {worst_gate:.1f}")
    assert worst_gate > 1.0


# ------------------------------------------------------------------------------------------------ K2
def _k2_scene(kind, b):
    """Per-keypoint product terms P [n, 24], per-cell weights w2 [513, n] and the de-normalisation tmats of one scene
    of the K2 tests.  Scene 0 is mini, scene 1 is c1 (another size, other tmats)."""
    name, seed = (("mini", 0), ("c1", 1))[b]
    sc = synth.make_scene(name, seed=seed, n_kp=500)
    src, dst = sc.src, sc.dst
    if kind == "exact":
        hom = np.concatenate([src.astype(np.float64), np.ones((src.shape[0], 1))], 1) @ sc.h_gt.T
        dst = (hom[:, :2] / hom[:, 2:3]).astype(np.float32)
    elif kind == "collinear":
        src = src.copy()
        src[:, 1] = 0.5 * src[:, 0] + 3.0
        dst = src + np.float32(2.0)
    elif kind == "three":
        src, dst = src[:3], dst[:3]
    sigma = 0.15 * sc.width
    st = APAP(0.5, sigma, [sc.final_w, sc.final_h], [sc.offset_x, sc.offset_y])
    rows, tmats = st._prepare(src, dst)
    n = src.shape[0]
    _, w2 = go.weights64(rows, _random_anchors(sc, 513, sigma, seed=7 + b), np.float32(0.01), 0, n)
    if kind in ("collinear", "three"):
        # well-conditioned general tmats: the residual is measured on h pulled back through them
        rng = np.random.default_rng(3 + b)
        tm = [np.eye(3) + 0.2 * rng.standard_normal((3, 3)) for _ in range(2)]
        tmats = np.concatenate([tm[0].reshape(9), tm[1].reshape(9)])
    return rows[:n, :go.TERMS].astype(np.float64), w2, tmats, max(sc.final_w, sc.final_h)


_K2_CACHE = {}


def _k2_planes(kind, k_splits, cells):
    """[2, k_splits, 24, cells_padded] float32 planes (NaN padding), tmats [2, 18], extents: per scene the keypoints
    dealt at random over the splits, each plane the float32 rounding of its float64 sum."""
    planes = np.full((2, k_splits, go.TERMS, go.cells_padded(cells)), np.nan, dtype=np.float32)
    tmats, ext = [], []
    for b in range(2):
        if (kind, b) not in _K2_CACHE:
            _K2_CACHE[(kind, b)] = _k2_scene(kind, b)
        p, w2, tm, e = _K2_CACHE[(kind, b)]
        split_of = np.random.default_rng(k_splits * 1000 + cells + b).integers(0, k_splits, p.shape[0])
        for s in range(k_splits):
            sel = split_of == s
            planes[b, s, :, :cells] = (w2[:cells, sel] @ p[sel]).T.astype(np.float32)
        tmats.append(tm)
        ext.append(e)
    return planes, np.stack(tmats), ext


def _launch_k2(cuda, planes, tmats, cells):
    torch, dev = cuda
    lib = rt.load_library()
    batch, ks = planes.shape[:2]
    p = torch.from_numpy(np.ascontiguousarray(planes)).to(dev)
    m = torch.from_numpy(np.ascontiguousarray(tmats)).to(dev)
    out = torch.full((batch, cells, 9), float("nan"), dtype=torch.float32, device=dev)
    sw = torch.zeros((batch, cells), dtype=torch.int32, device=dev)
    rt.check(lib.apap_eig_denorm(p.data_ptr(), m.data_ptr(), batch, cells, ks, rt.EIG_AUTO, out.data_ptr(),
                                 sw.data_ptr(), rt.stream_ptr(torch, dev)), "apap_eig_denorm")
    return out.cpu().numpy(), sw.cpu().numpy()


def _residual(h, g, tmats):
    """||G h^|| / (||G|| ||h^||) with h^ = the output H pulled back through tmats (float64)."""
    t2inv, t1 = tmats[:9].reshape(3, 3), tmats[9:].reshape(3, 3)
    hh = (np.linalg.inv(t2inv) @ h.reshape(-1, 3, 3).astype(np.float64) @ np.linalg.inv(t1)).reshape(-1, 9)
    num = np.linalg.norm(np.einsum("cij,cj->ci", g, hh), axis=1)
    return num / (np.linalg.norm(g, ord=2, axis=(1, 2)) * np.linalg.norm(hh, axis=1))


@pytest.mark.gpu
@pytest.mark.parametrize("cells", CELLS)
@pytest.mark.parametrize("k_splits", K2_SPLITS)
def test_k2_against_float64_eigensolve(cuda, k_splits, cells):
    for kind in ("healthy", "exact", "collinear", "three"):
        planes, tmats, ext = _k2_planes(kind, k_splits, cells)
        h, sweeps = _launch_k2(cuda, planes, tmats, cells)
        assert np.isfinite(h).all(), kind
        for b in range(2):
            want, gap, g = go.eig64(planes[b, :, :, :cells], tmats[b])
            if kind in ("healthy", "exact"):
                assert (gap >= 1e-6).all(), (kind, gap.min())           # the data: a healthy spectral gap
                err = orc.h_error_normalised(h[b], want, ext[b])
                print(f"K2 {kind} splits {k_splits} cells {cells} scene {b}: H err {err.max():.2e}, "
                      f"min gap {gap.min():.1e}, inverse-iteration steps {-sweeps[b].max()}..{-sweeps[b].min()}")
                assert (sweeps[b] < 0).all(), (kind, sweeps[b].max())
                assert err.max() <= H_TIGHT, (kind, b, err.max())
            else:
                res = _residual(h[b], g, tmats[b])
                print(f"K2 {kind} splits {k_splits} cells {cells} scene {b}: residual {res.max():.2e}, "
                      f"Jacobi cells {(sweeps[b] > 0).sum()}/{cells}")
                assert res.max() <= RESIDUAL, (kind, b, res.max())
        # power-of-two scaling of every plane is exact, and K2 divides by sum(w^2) first: the same bits
        for e in (-40, 40):
            hs, ss = _launch_k2(cuda, np.ldexp(planes, e), tmats, cells)
            assert np.array_equal(hs.view(np.uint32), h.view(np.uint32)) and np.array_equal(ss, sweeps), (kind, e)


@pytest.mark.gpu
def test_k2_degenerate_sets_take_the_jacobi_path(cuda):
    hits = {}
    for kind in ("collinear", "three"):
        planes, tmats, _ = _k2_planes(kind, 3, 513)
        _, sweeps = _launch_k2(cuda, planes, tmats, 513)
        hits[kind] = float((sweeps > 0).mean())
    print(f"K2 degenerate sets: share of cells on the Jacobi path {hits}")
    assert all(v > 0 for v in hits.values()), hits


@pytest.mark.gpu
def test_k2_all_zero_planes_are_pinned(cuda):
    """No weight anywhere: the Gram matrix is 0 / 0.  K2 runs 0 Jacobi sweeps, takes e0 as the eigenvector and stores
    T2inv e0 T1 divided by its [2][2] entry, which is 0 for affine tmats: NaN where T2inv[:, 0] T1[0, :] is 0, +-inf
    elsewhere (include/apap_b200.h, apap_eig_denorm)."""
    _, tmats, _ = _k2_planes("healthy", 2, 129)
    planes = np.zeros((2, 2, go.TERMS, go.cells_padded(129)), dtype=np.float32)
    planes[..., 129:] = np.nan
    h, sweeps = _launch_k2(cuda, planes, tmats, 129)
    assert (sweeps == 0).all()
    for b in range(2):
        outer = np.outer(tmats[b, :9].reshape(3, 3)[:, 0], tmats[b, 9:].reshape(3, 3)[0, :]).reshape(9)
        assert outer[8] == 0
        assert (np.isnan(h[b]) == (outer == 0)[None]).all() and (np.isinf(h[b]) == (outer != 0)[None]).all()


# ------------------------------------------------------------------------------------------ ragged batch
@pytest.mark.gpu
def test_ragged_batch_within_tight_gate_of_each_scenes_own_reference(cuda):
    """local_homography_batch plans K1 for the largest count, so the 300-match scene runs on the 8320-match plan; each
    scene's H is checked against the float64 reference of its own matches alone (its own plan, the product's
    conditioning) -- the bound on "may differ from its single call in the last bits"."""
    torch, dev = cuda
    scenes = [synth.make_scene("c1", n_kp=8320, seed=0), synth.make_scene("c1", n_kp=300, seed=1)]
    sc0 = scenes[0]
    st = APAP(sc0.gamma, sc0.sigma, [sc0.final_w, sc0.final_h], [sc0.offset_x, sc0.offset_y])
    got = st.local_homography_batch([s.src for s in scenes], [s.dst for s in scenes], sc0.vertices)
    counts = [s.src.shape[0] for s in scenes]
    raw = np.zeros((2, 2, max(counts), 2), dtype=np.float32)
    for b, s in enumerate(scenes):
        raw[0, b, :counts[b]], raw[1, b, :counts[b]] = s.src, s.dst
    cond, tmats = st.condition_device(torch.from_numpy(raw).to(dev),
                                      torch.tensor(counts, dtype=torch.int32, device=dev))
    cond, tmats = cond.cpu().numpy(), tmats.cpu().numpy()
    a = scale_anchors(sc0.vertices, weight_scale(sc0.sigma))
    for b, s in enumerate(scenes):
        n = counts[b]
        dlt = APAP.matrix_generate(n, cond[0, b, :n], cond[1, b, :n])
        rows = build_kp_table(s.src, dlt, weight_scale(sc0.sigma))
        want, _, _ = go.eig64(go.partials64(rows, a, np.float32(sc0.gamma ** 2), rows.shape[0], go.GRAM_TCGEN05),
                              tmats[b])
        err = orc.h_error_normalised(got[b], want, max(sc0.final_w, sc0.final_h))
        print(f"ragged batch scene {b} ({n} matches): H err vs its own float64 reference {err.max():.2e}")
        assert err.max() <= H_TIGHT, (b, err.max())
