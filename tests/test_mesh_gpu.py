"""GPU: marching cubes (p3d_mc_count / p3d_mc_emit through panic3d_b200.mesh) against the CPU oracle array for array,
the drop-in against the reference fixtures, and mesh properties on a 256^3 volume-query output."""
import os

import numpy as np
import pytest
import torch

from oracle import mesh_oracle as mo
from tests import mesh_checks as mc
from tests.golden.cases import VOLUME_CASES, build_case_inputs
from tests.golden.cases_mesh import MESH_CASES, mesh_case_inputs
from tests.test_render_gpu import make_decoder

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def _device(vol, level, rgb=None):
    import panic3d_b200.mesh as pm
    m = pm.marching_cubes_device(torch.from_numpy(vol).to(DEV), level, None if rgb is None else torch.from_numpy(rgb).to(DEV))
    return {k: (None if v is None else v.cpu().numpy()) for k, v in m.items()}


def _assert_equals_oracle(vol, level, rgb=None):
    verts, faces, normals, values = mo.marching_cubes(vol, level)
    got = _device(vol, level, rgb)
    assert np.array_equal(got['verts'], verts)
    assert np.array_equal(got['faces'], faces)
    assert np.array_equal(got['values'], values)
    assert np.abs(got['normals'] - normals).max() <= 1e-6
    if rgb is not None:
        a, b, c = verts.astype(int).T
        assert np.array_equal(got['colors'], rgb[:, a, b, c].T)
    return got


def _query(res, **kw):
    import panic3d_b200.volume as pv
    from panic3d_b200.training.volumetric_rendering.renderer import ImportanceRenderer
    # the fixture case's crop / cull options: at generate.py's cull_clouds=0.5 these synthetic planes are culled entirely
    case = dict(VOLUME_CASES['vol_crop_cull16'], res=res)
    planes, dec, _, _, _, _, opts = build_case_inputs(case)
    out = pv.query_volume(planes.to(DEV), make_decoder(dec, DEV), opts, resolution=res, triplane_crop=case['triplane_crop'],
                          cull_clouds=case['cull_clouds'], renderer=ImportanceRenderer(use_triplane=True), **kw)
    torch.cuda.synchronize()
    return out, opts['box_warp']


@pytest.mark.parametrize('name', sorted(MESH_CASES))
def test_kernel_equals_oracle_on_fixture_inputs(name):
    vol, rgbs = mesh_case_inputs(MESH_CASES[name])
    _assert_equals_oracle(vol, MESH_CASES[name]['level'], np.ascontiguousarray(rgbs))


@pytest.mark.parametrize('field', ['sphere', 'torus', 'smooth_random', 'on_level_corners'])
def test_kernel_equals_oracle_on_analytic_fields(field):
    vol = getattr(mc, field)()
    got = _assert_equals_oracle(vol, 0.0)
    mc.assert_closed_oriented(got['verts'], got['faces'])


def test_kernel_equals_oracle_on_volume_query_96():
    out, _ = _query(96, want_coordinates=False)
    vol = out['densities'][0, 0].cpu().numpy()
    rgb = np.ascontiguousarray(out['rgbs'][0, :3].cpu().numpy())
    got = _assert_equals_oracle(vol, 0.5, rgb)
    assert len(got['faces']) > 1000


@pytest.mark.parametrize('name', sorted(MESH_CASES))
def test_dropin_equals_reference_fixture(name):
    import panic3d_b200.mesh as pm
    case = MESH_CASES[name]
    vol, rgbs = mesh_case_inputs(case)
    got = pm.marching_cubes(vol, rgbs, case['boxwarp'], level=case['level'])
    g = np.load(os.path.join(GOLDEN, f'mesh_{name}.npz'))
    for k in ('verts', 'faces', 'normals', 'values', 'colors'):
        assert got[k].dtype == g[k].dtype and got[k].shape == g[k].shape, k
        if k == 'normals':
            assert np.abs(got[k] - g[k]).max() <= 1e-6
        else:
            assert np.array_equal(got[k], g[k]), k
    assert got.verts is got['verts']


def test_dropin_numpy_route_equals_in_place_route():
    """generate.py's call (numpy from .cpu().numpy()) and the in-place call on the device tensors, including the strided
    ['rgbs'][0,:3] view of the channels-last buffer, give the same mesh."""
    import panic3d_b200.mesh as pm
    vol, bw = _query(64, want_coordinates=False)
    assert not vol['rgbs'][0, :3].is_contiguous()
    a = pm.marching_cubes(vol['densities'].cpu().numpy()[0, 0], vol['rgbs'].cpu().numpy()[0, :3], bw, level=0.5)
    b = pm.marching_cubes(vol['densities'][0, 0], vol['rgbs'][0, :3], bw, level=0.5)
    for k in ('verts', 'faces', 'normals', 'values', 'colors'):
        assert np.array_equal(a[k], b[k]), k


def test_errors_like_skimage():
    import panic3d_b200.mesh as pm
    v = torch.from_numpy(mc.sphere(8, 2.0)).to(DEV)
    with pytest.raises(ValueError):
        pm.marching_cubes_device(v, float(v.max()) + 1)
    with pytest.raises(RuntimeError, match='No surface'):
        pm.marching_cubes_device(torch.zeros(4, 4, 4, device=DEV), 0.0)
    with pytest.raises(ValueError):
        pm.marching_cubes_device(torch.zeros(1, 4, 4, device=DEV), 0.0)


def test_volume_query_256_mesh_properties():
    import panic3d_b200.mesh as pm
    vol, bw = _query(256, want_coordinates=False)
    R = 256
    dens, rgb = vol['densities'][0, 0], vol['rgbs'][0, :3]
    m1 = pm.marching_cubes_device(dens, 0.5, rgb)
    m2 = pm.marching_cubes_device(dens, 0.5, rgb)
    for k in m1:
        assert torch.equal(m1[k], m2[k]), k                         # bit-identical run to run
    verts, faces = m1['verts'].cpu().numpy(), m1['faces'].cpu().numpy()
    assert len(faces) > 10000
    edges, cnt = mc.edge_face_counts(faces)
    assert cnt.max() <= 2
    open_ = edges[cnt == 1]
    if len(open_):                                                   # open edges only on the volume's outer faces
        p, q = verts[open_[:, 0]], verts[open_[:, 1]]
        on = ((p == 0) & (q == 0)) | ((p == R - 1) & (q == R - 1))
        assert on.any(1).all()
    assert mc.consistently_oriented(faces)
    mc.assert_no_degenerates(verts, faces)
    d = pm.marching_cubes(dens, rgb, bw, level=0.5)
    assert (np.abs(d['verts']) <= bw / 2).all()
    assert np.array_equal(d['faces'], faces)
