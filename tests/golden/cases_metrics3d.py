"""Geometry-metric fixture cases (tests/golden/make_golden_metrics3d.py): inputs are regenerated, never stored.

Predicted meshes are the marching-cubes fixtures ``mesh_*.npz`` (the drop-in's output in world units); ground-truth
meshes are a seeded bumpy sphere in their own frame; the region of interest is synthetic.  The fp32 case moves one
vertex exactly onto the fp32 rounding of a crop bound that rounds inward, so it is dropped when compared in fp32 (the
reference's numpy semantics) but would be kept in float64."""
from __future__ import annotations

import os
import zlib

import numpy as np

from oracle import metrics3d_oracle as mo

HERE = os.path.dirname(os.path.abspath(__file__))

METRICS3D_CASES = {
    'vol_crop_cull16_gt32': dict(pred='mesh_vol_crop_cull16', gt_seed=3, gt_dtype='float32', roi=((118, 140), (270, 236)),
                                 bn='daredemoE/fandom_align/synthA/0003/front', n_sample=2000, bw=0.7),
    'blob32_gt64': dict(pred='mesh_blob32', gt_seed=7, gt_dtype='float64', roi=((96, 120), (300, 290)),
                        bn='daredemoE/fandom_align/synthB/0007/front', n_sample=2000, bw=0.7),
}


def bumpy_sphere(seed, n_theta=40, n_phi=64, radius=0.2):
    """Closed genus-0 mesh: poles + rings, radius modulated by a few seeded harmonics, seeded centre."""
    rng = np.random.default_rng(seed)
    th = np.linspace(0, np.pi, n_theta + 1)[1:-1]
    ph = np.linspace(0, 2 * np.pi, n_phi, endpoint=False)
    T, P = np.meshgrid(th, ph, indexing='ij')
    r = radius * np.ones_like(T)
    for _ in range(4):
        k, m, amp, ph0 = rng.integers(1, 5), rng.integers(1, 5), rng.uniform(0.03, 0.1), rng.uniform(0, 2 * np.pi)
        r = r * (1 + amp * np.sin(k * T) * np.cos(m * P + ph0))
    c = rng.uniform(-0.04, 0.04, 3)
    ring = np.stack([r * np.sin(T) * np.cos(P), r * np.cos(T), r * np.sin(T) * np.sin(P)], -1).reshape(-1, 3) + c
    verts = np.concatenate([(c + [0, radius, 0])[None], ring, (c - [0, radius, 0])[None]])
    faces = []
    idx = lambda i, j: 1 + i * n_phi + (j % n_phi)       # noqa: E731
    for j in range(n_phi):
        faces.append((0, idx(0, j + 1), idx(0, j)))
        for i in range(n_theta - 2):
            faces += [(idx(i, j), idx(i, j + 1), idx(i + 1, j)), (idx(i, j + 1), idx(i + 1, j + 1), idx(i + 1, j))]
        faces.append((len(verts) - 1, idx(n_theta - 2, j), idx(n_theta - 2, j + 1)))
    return verts, np.asarray(faces, np.int64)


def on_bound_vertex(verts, roi, bw):
    """Move the vertex nearest to a crop bound whose fp32 rounding lies inside the box exactly onto that rounding.
    Returns (verts, index)."""
    x_lo, x_hi, y_lo, y_hi = mo.roi_bounds(roi, bw)
    inside = mo.filter_mask(verts.astype(np.float64), roi, bw)
    for axis, b, inward in ((0, x_lo, 1), (0, x_hi, -1), (1, y_lo, 1), (1, y_hi, -1)):
        b32 = np.float32(b)
        if (float(b32) - b) * inward > 0:
            cand = np.where(inside)[0]
            i = cand[np.argmin(np.abs(verts[cand, axis] - b))]
            v = verts.copy()
            v[i, axis] = b32
            return v, int(i)
    raise AssertionError('no crop bound of this roi rounds inward in fp32')


def gt_mesh(case):
    v, f = bumpy_sphere(case['gt_seed'])
    if case['gt_dtype'] == 'float32':
        v, _ = on_bound_vertex(v.astype(np.float32), case['roi'], case['bw'])
        return v, f
    return v.astype(np.float64), f


def pred_mc(case):
    z = np.load(os.path.join(HERE, case['pred'] + '.npz'))
    return {'verts': z['verts'], 'faces': z['faces']}


def injected_bits(case):
    """The bits the fixture's stub igl drew inside np_seed(bn): the legacy global stream seeded with adler32(bn), the
    same for both meshes of a subject (both calls reseed with bn)."""
    rs = np.random.RandomState(zlib.adler32(bytes(case['bn'], encoding='utf-8')))
    n = case['n_sample']
    return draw_bits(rs, n)


def draw_bits(rs, n):
    face_bits = rs.randint(0, 2 ** 64, size=n, dtype=np.uint64)
    bary_u = rs.random_sample((n, 2))
    return face_bits, bary_u
