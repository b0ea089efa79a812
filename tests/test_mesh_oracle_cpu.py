"""CPU: the marching-cubes contract (oracle/mesh_oracle.py) - single cells, shared faces, closed analytic surfaces,
degenerate removal, skimage's errors - and the product module's refusal to run without a device."""
import itertools

import numpy as np
import pytest
import torch

from oracle import mesh_oracle as mo
from tests import mesh_checks as mc

F32 = np.float32


def _cell_values(bits, rng):
    """2x2x2 values (corner order mo.CORNERS) realising the inside bits, with magnitudes spread over 3 decades so the
    decider of every ambiguous face goes both ways across draws."""
    mag = (10.0 ** rng.uniform(-1.5, 1.5, 8)).astype(F32)
    return np.where([(bits >> c) & 1 for c in range(8)], mag, -mag).astype(F32)


def _ambiguous_outcomes(bits, f):
    out = []
    for _, _, lat in mo.FACES:
        ins = [(bits >> c) & 1 for c in lat]
        if ins in ([1, 0, 0, 1], [0, 1, 1, 0]):
            a, b, c, d = (f[x] for x in lat)
            det = F32(a * d) - F32(b * c)
            out.append(bool(det > 0) if ins[0] else bool(det < 0))
    return tuple(out)


def _check_cell(bits, f):
    inside = [(bits >> c) & 1 for c in range(8)]
    crossing = {e for e, (c, a) in enumerate(mo.EDGES) if inside[c] != inside[c | (1 << (2 - a))]}
    loops = mo.cell_loops(inside, f)
    used = [e for lp in loops for e in lp]
    assert sorted(used) == sorted(crossing)                          # every crossing edge exactly once
    assert [lp[0] for lp in loops] == sorted(lp[0] for lp in loops)  # loops in order of their smallest id
    for lp in loops:
        assert lp[0] == min(lp) and len(lp) >= 3
        for x, y in zip(lp, lp[1:] + lp[:1]):                        # each segment lies on one cube face
            assert any(x in ce and y in ce for _, ce, _ in mo.FACES), (bits, lp)
    tris = mo.cell_triangles(inside, f)
    assert len(tris) == len(crossing) - 2 * len(loops)
    assert all(set(t) <= crossing for t in tris)


def test_every_sign_configuration_and_decider_outcome():
    rng = np.random.default_rng(0)
    for bits in range(256):
        seen = set()
        n_amb = None
        for draw in range(400):
            f = _cell_values(bits, rng)
            _check_cell(bits, f)
            o = _ambiguous_outcomes(bits, f)
            n_amb = len(o)
            seen.add(o)
            if len(seen) == 2 ** n_amb:
                break
        # each ambiguous face was both joined and separated at least once
        for k in range(n_amb):
            assert {o[k] for o in seen} == {False, True}, bits


def test_decider_ties_count_as_separated():
    f = np.array([1, -1, -1, 1, 1, -1, -1, 1], F32)                   # every face a*d - b*c == 0 exactly
    bits = sum(1 << c for c in range(8) if f[c] > 0)
    assert _ambiguous_outcomes(bits, f) == (False,) * len(_ambiguous_outcomes(bits, f))
    _check_cell(bits, f)


@pytest.mark.parametrize('axis', [0, 1, 2])
def test_cells_sharing_a_face_agree_on_its_segments(axis):
    rng = np.random.default_rng(10 + axis)
    shape = [2, 2, 2]
    shape[axis] = 3
    D = tuple(shape)
    for _ in range(300):
        V = (rng.standard_normal(D) * 10.0 ** rng.uniform(-1, 1, D)).astype(F32)
        segs = []
        for lo in (0, 1):
            p = [0, 0, 0]
            p[axis] = lo
            vals = [V[p[0] + o[0], p[1] + o[1], p[2] + o[2]] for o in mo.CORNERS]
            inside = [v > 0 for v in vals]
            keys = [3 * np.ravel_multi_index((p[0] + mo.CORNERS[c][0], p[1] + mo.CORNERS[c][1], p[2] + mo.CORNERS[c][2]), D) + a
                    for c, a in mo.EDGES]
            shared = {keys[e] for e, (c, a) in enumerate(mo.EDGES) if a != axis and mo.CORNERS[c][axis] == 1 - lo}
            s = set()
            for lp in mo.cell_loops(inside, [F32(v) for v in vals]):
                for x, y in zip(lp, lp[1:] + lp[:1]):
                    if keys[x] in shared and keys[y] in shared:
                        s.add((keys[x], keys[y]))
            segs.append(s)
        assert segs[0] == {(y, x) for x, y in segs[1]}                 # same segments, opposite directions


def test_sphere_closed_area_normals_winding():
    V = mc.sphere(64, 25.0)
    verts, faces, normals, values = mo.marching_cubes(V, 0.0)
    mc.assert_closed_oriented(verts, faces)
    assert mc.euler_characteristic(verts, faces) == 2
    fn = mc.face_normals(verts, faces)
    assert 0.99 < 0.5 * np.linalg.norm(fn, axis=1).sum() / (4 * np.pi * 25.0 ** 2) < 1.01
    c = (64 - 1) / 2
    radial = verts - c
    radial /= np.linalg.norm(radial, axis=1, keepdims=True)
    assert ((normals * radial).sum(1) > 0.99).all()
    # winding: the right-hand normal points the way the (outward, 'descent') vertex normals do
    assert ((fn * normals[faces].sum(1)).sum(1) > 0).all()
    assert verts.dtype == np.float32 and faces.dtype == np.int32 and normals.dtype == np.float32 and values.dtype == np.float32
    # values: the max of the lowest-index cell around the edge, so never below the level
    assert (values >= 0).all()


def test_torus_genus_one():
    verts, faces, _, _ = mo.marching_cubes(mc.torus(), 0.0)
    mc.assert_closed_oriented(verts, faces)
    assert mc.euler_characteristic(verts, faces) == 0


def test_saddle_rich_field_is_a_closed_oriented_manifold():
    V = mc.smooth_random(40, seed=3)
    verts, faces, _, _ = mo.marching_cubes(V, 0.0)
    n_amb = 0                                                           # the field does exercise the decider
    for i, j, k in itertools.product(range(39), repeat=3):
        fc = [V[i + o[0], j + o[1], k + o[2]] for o in mo.CORNERS]
        bits = sum(1 << c for c in range(8) if fc[c] > 0)
        n_amb += len(_ambiguous_outcomes(bits, fc))
    assert n_amb > 20
    mc.assert_closed_oriented(verts, faces)


def test_corners_on_level_are_merged():
    V = mc.on_level_corners()
    assert (V == 0).mean() > 0.01
    verts, faces, _, _ = mo.marching_cubes(V, 0.0)
    mc.assert_no_degenerates(verts, faces)
    mc.assert_closed_oriented(verts, faces)
    assert (verts == np.round(verts)).all(1).sum() > 100                # many vertices do sit on lattice corners


def test_vertex_positions_and_order():
    V = mc.blob(16, seed=1)
    verts, faces, _, _ = mo.marching_cubes(V, 0.5)
    a = np.argmax(verts != np.round(verts), axis=1)                     # the edge axis (non-integer coordinate)
    lo = np.floor(verts).astype(np.int64)
    keys = 3 * np.ravel_multi_index(tuple(lo.T), V.shape) + a
    assert (np.diff(keys) > 0).all()                                    # ascending edge key
    hi = lo.copy()
    hi[np.arange(len(hi)), a] += 1
    vlo, vhi = V[tuple(lo.T)], V[tuple(hi.T)]
    assert ((vlo > 0.5) != (vhi > 0.5)).all()
    t = (F32(0.5) - vlo) / (vhi - vlo)
    assert np.array_equal(verts[np.arange(len(a)), a], lo[np.arange(len(a)), a].astype(F32) + t)


def test_errors_like_skimage():
    V = mc.sphere(8, 2.0)
    with pytest.raises(ValueError):
        mo.marching_cubes(V, float(V.max()) + 1)
    with pytest.raises(ValueError):
        mo.marching_cubes(V, float(V.min()) - 1)
    with pytest.raises(RuntimeError):
        mo.marching_cubes(np.zeros((4, 4, 4), F32), 0.0)               # in range, nothing crosses
    with pytest.raises(ValueError):
        mo.marching_cubes(np.zeros((1, 4, 4), F32), 0.0)


def test_mesh_module_has_no_cpu_path():
    import panic3d_b200.mesh as pm
    with pytest.raises(RuntimeError, match='no CPU path'):
        pm.marching_cubes_device(torch.zeros(4, 4, 4))
