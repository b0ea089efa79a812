"""GPU: surface sampling, BVH distances and the per-subject geometry metrics (panic3d_b200.metrics3d) against the
exhaustive-search oracle bit for bit, the reference fixtures, and whole-size properties."""
import os

import numpy as np
import pytest
import torch

from oracle import metrics3d_oracle as mo
from tests import mesh_checks as mc
from tests.golden.cases_metrics3d import METRICS3D_CASES, bumpy_sphere, gt_mesh, injected_bits, pred_mc

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def _mc_mesh(field):
    import panic3d_b200.mesh as pm
    m = pm.marching_cubes_device(torch.from_numpy(getattr(mc, field)()).to(DEV), 0.0)
    return m['verts'].double().cpu().numpy() / 64 - 0.5, m['faces'].cpu().numpy()


def _points_near(V, rng, n):
    lo, hi = V.min(0), V.max(0)
    near = V[rng.integers(0, len(V), n // 2)] + rng.normal(size=(n // 2, 3)) * 0.01
    far = lo - (hi - lo) + rng.random((n - n // 2, 3)) * 3 * (hi - lo)
    return np.concatenate([near, far])


def _assert_equals_exhaustive(P, V, F):
    import panic3d_b200.metrics3d as m3
    d2, face, q = m3.point_mesh_squared_distance(torch.from_numpy(P).to(DEV), torch.from_numpy(V).to(DEV), torch.from_numpy(F).to(DEV))
    w2, wf, wq = mo.point_mesh_squared_distance(P, V, F)
    assert np.array_equal(d2.cpu().numpy(), w2)
    assert np.array_equal(face.cpu().numpy(), wf)
    assert np.array_equal(q.cpu().numpy(), wq)
    return w2, wf


@pytest.mark.parametrize('field', ['sphere', 'torus'])
def test_distance_equals_exhaustive_on_closed_meshes(field):
    V, F = _mc_mesh(field)
    _assert_equals_exhaustive(_points_near(V, np.random.default_rng(0), 2000), V, F)


def test_distance_ties_on_vertices_and_edges():
    V, F = bumpy_sphere(2, 16, 24)
    rng = np.random.default_rng(1)
    e = F[rng.integers(0, len(F), 300)]
    t = rng.random((300, 1))
    P = np.concatenate([V, V[e[:, 0]] * (1 - t) + V[e[:, 1]] * t, V[e[:, 0]] + 0.5 * (V[e[:, 1]] - V[e[:, 0]])])
    d2, _ = _assert_equals_exhaustive(P, V, F)
    assert (d2[:len(V)] == 0).all()


def test_distance_degenerate_faces():
    V, F = bumpy_sphere(5, 10, 12)
    F = F.copy()
    F[::7, 2] = F[::7, 0]                                   # repeated vertex
    V = np.concatenate([V, [[0.1, 0.1, 0.1], [0.2, 0.2, 0.2], [0.4, 0.4, 0.4]]])
    n = len(V)
    F = np.concatenate([F, [[n - 3, n - 2, n - 1], [n - 1, n - 1, n - 1]]])   # collinear, all equal
    _assert_equals_exhaustive(_points_near(V, np.random.default_rng(2), 1000), V, F)


def test_distance_one_face_mesh():
    V = np.array([[0.0, 0.0, 0.0], [1.0, 0.0, 0.0], [0.0, 1.0, 0.5]])
    F = np.array([[0, 1, 2]])
    _assert_equals_exhaustive(np.random.default_rng(3).normal(size=(500, 3)), V, F)


def test_distance_many_identical_triangles():
    V, F = bumpy_sphere(6, 6, 8)
    F = np.concatenate([F] * 40 + [F[:5]] * 200)            # equal centroids: equal Morton codes, distinct keys
    _assert_equals_exhaustive(_points_near(V, np.random.default_rng(4), 500), V, F)


def test_distance_on_volume_query_256_mesh_subset():
    import panic3d_b200.mesh as pm
    from tests.test_mesh_gpu import _query
    vol, bw = _query(256, want_coordinates=False)
    m = pm.marching_cubes_device(vol['densities'][0, 0], 0.5)
    V = (m['verts'].double() / 256 * bw - 0.5 * bw).cpu().numpy()
    F = m['faces'].cpu().numpy()
    assert len(F) > 100000
    _assert_equals_exhaustive(_points_near(V, np.random.default_rng(5), 512), V, F)


# ---------------------------------------------------------------- sampler
def test_sampler_injected_bits_equal_oracle():
    import panic3d_b200.metrics3d as m3
    V, F = bumpy_sphere(7, 20, 30)
    rng = np.random.default_rng(6)
    fb, bu = rng.integers(0, 2 ** 64, size=5000, dtype=np.uint64), rng.random((5000, 2))
    B, FI = m3.random_points_on_mesh(5000, V, F, face_bits=fb, bary_u=bu)
    wB, wFI, _ = mo.sample_from_bits(V, F, fb, bu)
    assert np.array_equal(B, wB) and np.array_equal(FI, wFI)
    _, _, pts = m3._sample(torch.from_numpy(V).to(DEV), torch.from_numpy(F).to(DEV, torch.int32), 5000, 0, 0,
                           torch.from_numpy(fb).to(DEV), torch.from_numpy(bu).to(DEV), torch.zeros(1, dtype=torch.int32, device=DEV))
    assert np.array_equal(pts.cpu().numpy(), mo.sample_from_bits(V, F, fb, bu)[2])


def test_sampler_philox_properties():
    import panic3d_b200.metrics3d as m3
    from scipy import stats
    V, F = bumpy_sphere(8, 8, 10)
    Vd, Fd = torch.from_numpy(V).to(DEV), torch.from_numpy(F).to(DEV)
    n = 100000
    a = m3.random_points_on_mesh(n, Vd, Fd, seed='subject/0001')
    b = m3.random_points_on_mesh(n, Vd, Fd, seed='subject/0001')
    assert all(torch.equal(x, y) for x, y in zip(a, b))                 # bit-identical run to run
    c = m3.random_points_on_mesh(n, Vd, Fd, seed='subject/0002')
    d = m3.random_points_on_mesh(n, Vd, Fd, seed='subject/0001', stream=1)
    assert not torch.equal(a[0], c[0]) and not torch.equal(a[0], d[0])
    area = mo.face_areas(V, F)
    expected = area / area.sum() * n
    chi2 = ((np.bincount(a[1].cpu().numpy(), minlength=len(F)) - expected) ** 2 / expected).sum()
    assert stats.chi2.sf(chi2, len(F) - 1) > 1e-3
    Bc = a[0].cpu().numpy()
    assert stats.kstest(Bc[:, 1] + Bc[:, 2], lambda t: t ** 2).pvalue > 1e-3


# ---------------------------------------------------------------- measure_geometry
def _run_case(name, device):
    import panic3d_b200.metrics3d as m3
    case = METRICS3D_CASES[name]
    mcd, (gv, gf) = pred_mc(case), gt_mesh(case)
    bits = injected_bits(case)
    if device:
        mcd = {k: torch.from_numpy(v).to(DEV) for k, v in mcd.items()}
        gv, gf = torch.from_numpy(gv).to(DEV), torch.from_numpy(gf).to(DEV)
    return m3.measure_geometry(mcd, gv, gf, case['roi'], bw=case['bw'], n_sample=case['n_sample'], seed=case['bn'],
                               injected=(bits, bits))


@pytest.mark.parametrize('name', sorted(METRICS3D_CASES))
def test_measure_geometry_equals_reference_fixture(name):
    import panic3d_b200.metrics3d as m3
    g = np.load(os.path.join(GOLDEN, f'metrics3d_{name}.npz'))
    case = METRICS3D_CASES[name]
    out = _run_case(name, device=False)
    for k, v in out.items():
        if k.startswith(('precision_', 'recall_', 'f1_')):
            assert v == g[k], k                                   # exact counts over n
        else:
            assert abs(v - g[k]) <= 1e-12 * abs(g[k]), k           # torch sum vs numpy's pairwise sum
    # the pieces, bit for bit
    mcd, (gv, gf) = pred_mc(case), gt_mesh(case)
    pv = mcd['verts'].astype(np.float64) * np.array([-1.0, 1.0, 1.0])
    fp = m3.filter_mesh(pv, mcd['faces'], case['roi'], case['bw'])
    fg = m3.filter_mesh(gv, gf, case['roi'], case['bw'])
    for got, k in ((fp['verts'], 'pred_verts'), (fp['faces'], 'pred_faces'), (fg['verts'], 'gt_verts'), (fg['faces'], 'gt_faces')):
        assert got.dtype == g[k].dtype and np.array_equal(got, g[k]), k
    gvt = g['gt_verts'].astype(np.float64) * np.array([-1.0, 1.0, -1.0])
    assert np.array_equal(m3.get_point_mesh_distance(g['points_pred'], gvt, g['gt_faces']), g['p2s_all'])
    assert np.array_equal(m3.get_point_mesh_distance(g['points_gt'], g['pred_verts'], g['pred_faces']), g['s2p_all'])
    r = m3.point_mesh_f1(g['p2s_all'], g['s2p_all'], 0.05)
    assert r['precision'] == g['precision_050'] and r['recall'] == g['recall_050'] and r['f1'] == g['f1_050']


@pytest.mark.parametrize('name', sorted(METRICS3D_CASES))
def test_measure_geometry_numpy_route_equals_device_route(name):
    a, b = _run_case(name, device=False), _run_case(name, device=True)
    assert a.keys() == b.keys() and all(a[k] == b[k] for k in a)


def test_errors():
    import panic3d_b200.metrics3d as m3
    case = METRICS3D_CASES['blob32_gt64']
    mcd, (gv, gf) = pred_mc(case), gt_mesh(case)
    with pytest.raises(ValueError, match='no faces'):
        m3.measure_geometry(mcd, gv, gf, ((0, 0), (2, 2)), n_sample=100, seed=0)
    with pytest.raises(RuntimeError, match='no CPU path'):
        m3.point_mesh_squared_distance(torch.zeros(4, 3), torch.from_numpy(gv).to(DEV), torch.from_numpy(gf).to(DEV))
    with pytest.raises(RuntimeError, match='no CPU path'):
        m3.random_points_on_mesh(10, torch.from_numpy(gv), torch.from_numpy(gf), seed=0)
    with pytest.raises(ValueError, match='no faces'):
        m3.point_mesh_squared_distance(np.zeros((4, 3)), gv, gf[:0])
    with pytest.raises(ValueError, match='zero area'):
        m3.random_points_on_mesh(10, np.zeros((3, 3)), np.array([[0, 1, 2]]), seed=0)


def test_whole_size_self_and_offset():
    """measure_geometry at the reference's 10k samples on the 256^3 volume-query mesh: against itself every distance is
    0 up to the rounding of the sampled point (the ground truth is the predicted mesh mapped into its frame), against a
    copy moved by 0.01 none exceeds the offset."""
    import panic3d_b200.mesh as pm
    import panic3d_b200.metrics3d as m3
    from tests.test_mesh_gpu import _query
    vol, bw = _query(256, want_coordinates=False)
    m = pm.marching_cubes_device(vol['densities'][0, 0], 0.5)
    V = m['verts'].double() / 256 * bw - 0.5 * bw
    F = m['faces']
    roi = ((0, 0), (512, 512))
    # the ground truth lives in the frame that diag(-1, 1, -1) maps onto the mirrored prediction
    gt = V * torch.tensor([1.0, 1.0, -1.0], dtype=torch.float64, device=DEV)
    out = m3.measure_geometry({'verts': V, 'faces': F}, gt, F, roi, bw=bw, seed='self')
    assert out['p2s'] <= 1e-15 and out['s2p'] <= 1e-15 and out['cd'] <= 1e-15
    assert all(out[f'f1_{int(t * 1000):03d}'] == 1.0 for t in m3.THRESHOLDS)
    off = gt + torch.tensor([0.0, 0.0, 0.01], dtype=torch.float64, device=DEV)
    out = m3.measure_geometry({'verts': V, 'faces': F}, off, F, roi, bw=bw, seed='offset')
    assert 0 < out['p2s'] <= 0.01 * (1 + 1e-9) and 0 < out['s2p'] <= 0.01 * (1 + 1e-9)
    assert out['f1_050'] == 1.0 and out['f1_500'] == 1.0      # at 0.01 itself the last bit of a distance decides
