"""CPU: the geometry-metric oracle (closest point, crop, integer CDF sampler, F1) on known answers and properties."""
import numpy as np
import pytest
from scipy import stats

from oracle import metrics3d_oracle as mo
from tests.golden.cases_metrics3d import METRICS3D_CASES, bumpy_sphere, on_bound_vertex

A, B, C = np.array([0.0, 0.0, 0.0]), np.array([1.0, 0.0, 0.0]), np.array([0.0, 1.0, 0.0])


def _closest(p, a=A, b=B, c=C):
    q, d2 = mo.closest_on_triangle(np.asarray(p, np.float64), a, b, c)
    return q, float(d2)


@pytest.mark.parametrize('p, q', [
    ((-1.0, -1.0, 0.5), (0.0, 0.0, 0.0)),        # vertex region A
    ((2.0, -0.5, 0.0), (1.0, 0.0, 0.0)),         # vertex region B
    ((-0.5, 2.0, -1.0), (0.0, 1.0, 0.0)),        # vertex region C
    ((0.25, -1.0, 2.0), (0.25, 0.0, 0.0)),       # edge AB
    ((-3.0, 0.75, 0.0), (0.0, 0.75, 0.0)),       # edge AC
    ((1.0, 1.0, 0.5), (0.5, 0.5, 0.0)),          # edge BC
    ((0.25, 0.25, -2.0), (0.25, 0.25, 0.0)),     # interior
])
def test_closest_point_in_each_voronoi_region(p, q):
    got, d2 = _closest(p)
    assert np.array_equal(got, q)
    assert d2 == float(np.sum((np.array(p) - np.array(q)) ** 2))


def test_degenerate_faces_fall_back_to_edges():
    # collinear: a, b, c on the x axis
    a, b, c = np.array([0.0, 0, 0]), np.array([1.0, 0, 0]), np.array([3.0, 0, 0])
    q, d2 = _closest((2.0, 1.0, 0.0), a, b, c)
    assert np.array_equal(q, [2.0, 0.0, 0.0]) and d2 == 1.0
    q, d2 = _closest((-1.0, 0.0, 2.0), a, b, c)
    assert np.array_equal(q, [0.0, 0.0, 0.0]) and d2 == 5.0
    # all three vertices equal
    v = np.array([0.5, -0.25, 2.0])
    q, d2 = _closest((1.5, -0.25, 2.0), v, v, v)
    assert np.array_equal(q, v) and d2 == 1.0
    # c equal to a: the segment ab
    q, d2 = _closest((0.5, 2.0, 0.0), A, B, A.copy())
    assert np.array_equal(q, [0.5, 0.0, 0.0]) and d2 == 4.0


def test_distance_against_dense_sampling():
    rng = np.random.default_rng(0)
    for _ in range(20):
        a, b, c = rng.normal(size=(3, 3))
        p = rng.normal(size=(64, 3)) * 2
        q, d2 = mo.closest_on_triangle(p, a, b, c)
        u = rng.random((20000, 2))
        u = np.where(u.sum(1, keepdims=True) > 1, 1 - u, u)
        s = a + u[:, :1] * (b - a) + u[:, 1:] * (c - a)
        dense = ((p[:, None, :] - s[None]) ** 2).sum(-1).min(1)
        assert (d2 <= dense * (1 + 1e-12) + 1e-15).all()             # never above any point of the triangle
        # and the closest point lies on the triangle (so no point of it is closer than d2, up to rounding)
        M = np.stack([b - a, c - a], 1)
        uv, *_ = np.linalg.lstsq(M, (q - a).T, rcond=None)
        assert np.abs(M @ uv - (q - a).T).max() <= 1e-12
        assert (uv >= -1e-12).all() and (uv.sum(0) <= 1 + 1e-12).all()
        assert np.allclose(d2, ((p - q) ** 2).sum(1), rtol=1e-14, atol=0)


def test_ties_go_to_the_smallest_face_id():
    V = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [1, 1, 0], [-1, 0, 0]], np.float64)
    F = np.array([[1, 3, 2], [0, 1, 2], [0, 2, 4], [0, 1, 2]])
    d2, face, q = mo.point_mesh_squared_distance(np.array([[0.5, 0.5, 1.0], [0.0, 0.0, 0.0], [0.25, 0.25, -1.0]]), V, F)
    assert face.tolist() == [0, 1, 1]          # on the shared edge / vertex: the smallest id among the faces touching it
    assert d2.tolist() == [1.0, 0.0, 1.0]
    assert np.array_equal(q[1], [0, 0, 0])


def test_exhaustive_search_chunks_agree():
    V, F = bumpy_sphere(1, 12, 16)
    P = np.random.default_rng(1).normal(size=(300, 3)) * 0.3
    a = mo.point_mesh_squared_distance(P, V, F, chunk=1 << 21)
    b = mo.point_mesh_squared_distance(P, V, F, chunk=len(F) * 7)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


# ---------------------------------------------------------------- crop
def test_filter_mesh_edges():
    roi, bw = ((0, 0), (256, 256)), 1.0               # x in (-0.5, 0.0), y in (0.0, 0.5)
    assert mo.roi_bounds(roi, bw) == (-0.5, 0.0, 0.0, 0.5)
    v = np.array([[-0.25, 0.25, 0], [-0.1, 0.1, 0], [-0.3, 0.4, 0],       # 0-2 inside
                  [0.0, 0.25, 0],                                         # 3 exactly on x_hi: dropped
                  [-0.2, 0.2, 0], [0.2, 0.2, 0],                          # 4 inside, 5 outside
                  [-0.4, 0.1, 5.0]], np.float64)                          # 6 inside, no face
    f = np.array([[0, 1, 2], [0, 1, 3], [1, 4, 5], [2, 4, 0]])
    out = mo.filter_mesh(v, f, roi, bw)
    assert np.array_equal(out['verts'], v[[0, 1, 2, 4, 6]])
    assert out['faces'].tolist() == [[0, 1, 2], [2, 3, 0]]
    assert out['faces'].dtype == np.int64


def test_filter_mesh_compares_in_the_vertex_dtype():
    case = METRICS3D_CASES['vol_crop_cull16_gt32']
    v, _ = bumpy_sphere(case['gt_seed'])
    v32, i = on_bound_vertex(v.astype(np.float32), case['roi'], case['bw'])
    assert not mo.filter_mask(v32, case['roi'], case['bw'])[i]                        # fp32 bounds: on the bound
    assert mo.filter_mask(v32.astype(np.float64), case['roi'], case['bw'])[i]         # float64 bounds: inside
    # numpy's own weak-scalar comparison (what the reference's expression does) agrees with the explicit cast
    x_lo, x_hi, y_lo, y_hi = mo.roi_bounds(case['roi'], case['bw'])
    raw = (x_lo < v32[:, 0]) & (v32[:, 0] < x_hi) & (y_lo < v32[:, 1]) & (v32[:, 1] < y_hi)
    assert np.array_equal(raw, mo.filter_mask(v32, case['roi'], case['bw']))


# ---------------------------------------------------------------- sampler
def test_integer_cdf_is_exact_and_skips_zero_weight_faces():
    V = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 0], [2, 0, 0], [0, 2, 0], [5, 5, 5]], np.float64)
    F = np.array([[0, 1, 2], [6, 6, 6], [3, 4, 5], [0, 1, 4]])       # areas 1, 0, 4, 0 (collinear)
    w = mo.face_weights(V, F)
    assert w.tolist() == [2 ** 30, 0, 2 ** 32, 0]
    cdf = mo.face_cdf(V, F)
    assert cdf.tolist() == [2 ** 30, 2 ** 30, 2 ** 30 + 2 ** 32, 2 ** 30 + 2 ** 32]
    total = int(cdf[-1])
    k = np.array([0, 2 ** 64 - 1, 2 ** 62, (2 ** 64 // total) * 2 ** 30, 3 << 62], np.uint64)
    assert mo.mulhi64(k, total).tolist() == [(int(x) * total) >> 64 for x in k]
    _, fi, _ = mo.sample_from_bits(V, F, k, np.full((len(k), 2), 0.25))
    assert set(fi.tolist()) <= {0, 2}
    rng = np.random.default_rng(2)
    kk = rng.integers(0, 2 ** 64, size=100000, dtype=np.uint64)
    _, fi, _ = mo.sample_from_bits(V, F, kk, rng.random((100000, 2)))
    assert set(np.unique(fi).tolist()) == {0, 2}


def test_sampler_distribution():
    V, F = bumpy_sphere(4, 8, 10)
    n = 100000
    rng = np.random.default_rng(3)
    Bc, fi, pts = mo.sample_from_bits(V, F, rng.integers(0, 2 ** 64, size=n, dtype=np.uint64), rng.random((n, 2)))
    area = mo.face_areas(V, F)
    expected = area / area.sum() * n
    chi2 = ((np.bincount(fi, minlength=len(F)) - expected) ** 2 / expected).sum()
    assert stats.chi2.sf(chi2, len(F) - 1) > 1e-3
    # barycentrics: on the simplex, (a, b) uniform over the triangle: a and b have density 2(1-x), a+b density 2x
    assert np.allclose(Bc.sum(1), 1.0) and (Bc >= 0).all()
    for x, cdf in ((Bc[:, 1], lambda t: 1 - (1 - t) ** 2), (Bc[:, 2], lambda t: 1 - (1 - t) ** 2),
                   (Bc[:, 1] + Bc[:, 2], lambda t: t ** 2)):
        assert stats.kstest(x, cdf).pvalue > 1e-3
    # bary2cart's order, in float64
    f = F[fi]
    want = (V[f[:, 0]] * Bc[:, :1] + V[f[:, 1]] * Bc[:, 1:2]) + V[f[:, 2]] * Bc[:, 2:]
    assert np.array_equal(pts, want)


def test_point_mesh_f1_zero_when_both_zero():
    r = mo.point_mesh_f1(np.array([1.0, 2.0]), np.array([3.0]), 0.5)
    assert r['precision'] == 0 and r['recall'] == 0 and r['f1'] == 0.0
    r = mo.point_mesh_f1(np.array([0.1, 2.0]), np.array([0.3]), 0.5)
    assert r['precision'] == 0.5 and r['recall'] == 1.0 and r['f1'] == 2 * 0.5 * 1.0 / 1.5
