"""TEST INFRASTRUCTURE ONLY - numpy float64 restatement of the eval geometry metrics that ``p3d_surface_sample`` /
``p3d_bvh_build`` / ``p3d_point_mesh_distance`` (include/p3d_geom.h, csrc/point_mesh.cu) and ``panic3d_b200.metrics3d``
implement: the 3-D block of the reference's ``_scripts/eval/measure.py`` (helpers :54-99, per subject :141-201; the
sampler ``sample_points_near_surface`` / ``bary2cart`` of ``_databacks/lustrous_gltf_v0_measurable.py``).

The contract (shared bit for bit with the kernels; every numpy operation below is one separately rounded IEEE op):
  * crop (``filter_mesh``): the open box of ``roi_bounds`` (Python floats in the reference's operation order), compared
    in the dtype of the vertices - numpy treats a Python float as a weak scalar, so fp32 vertices meet bounds rounded
    to fp32 and float64 vertices exact ones; faces kept iff all three vertices are, re-indexed by cumsum(mask)-1;
    kept vertices that no kept face uses stay;
  * frames: the predicted vertices are mirrored in x (``* [-1,1,1]``, float64 from there on); the ground truth is
    cropped in its own frame, then mapped by diag(-1, 1, -1) (exact up to the sign of a zero);
  * sampler: face weight ``floor(|cross(b-a, c-a)| / max * 2^32)`` (uint64), CDF = its exact cumulative sum; sample i
    with 64-bit word k and uniforms (a, b) takes the first face with cdf > mulhi64(k, total), flips (a, b) to
    (1-a, 1-b) when a + b > 1, barycentrics (1-a-b, a, b), point (v0*b0 + v1*b1) + v2*b2.  On the device the bits
    come from Philox4x32-10 (key seed, counter i, stream); here they are injected;
  * closest point: Ericson's ClosestPtPointTriangle (Real-Time Collision Detection 5.1.5) in float64; a zero
    denominator in any division falls back to the nearest of the segments ab, bc, ca (first on ties; a segment clamps
    its projection t to [0, |ab|^2] before dividing); the point is then clamped into the face's bounding box (so the
    BVH's box bounds hold for the computed point).  dist2 = (dx*dx + dy*dy) + dz*dz.  Over a mesh: exhaustive
    search, the smallest dist2, ties to the smallest face id (np.argmin);
  * metrics: p2s = sqrt(dist2) of the predicted points to the ground-truth mesh, s2p the other way; cd =
    (mean(p2s) + mean(s2p)) / 2; precision / recall = mean(d <= th); f1 = 2*pre*rec / (pre+rec), 0 when both are 0.

Deviations from the reference: igl's random stream cannot be reproduced, so sample parity with igl is UNPINNED (the
sampler is ours; the fixtures pin ``bary2cart`` and everything around it).  igl's closest point may differ from ours in
the last bits and on degenerate faces (unpinned).  The means on the device are torch sums, not numpy's pairwise sums
(last bits).  A crop that leaves no face raises ValueError in ``panic3d_b200.metrics3d``; igl's behaviour there is not
pinned.  Inputs are assumed finite, with squared distances that are 0 or normal numbers (no fp64 underflow).
``measure.py:201`` assigns ``ans3d['f1_...']`` instead of appending, so its printed F1 is the last subject's; the
per-subject values here are what it computes per subject.
Only ``tests/`` may import this module; the product path is ``panic3d_b200.metrics3d``.
"""
from __future__ import annotations

import numpy as np

THRESHOLDS = (0.005, 0.01, 0.05, 0.1, 0.5)
_M32 = np.uint64(0xffffffff)


# ---------------------------------------------------------------- crop
def roi_bounds(roi, bw, size=512):
    """(x_lo, x_hi, y_lo, y_hi) of the open crop box, Python floats."""
    (a0, a1), (s0, s1) = roi
    x_lo = -bw / 2 + (a1 / size) * bw
    y_hi = bw / 2 - (a0 / size) * bw
    return x_lo, x_lo + bw * (s1 / size), y_hi - bw * (s0 / size), y_hi


def filter_mask(v, roi, bw, size=512):
    x_lo, x_hi, y_lo, y_hi = (np.asarray(b, dtype=v.dtype) for b in roi_bounds(roi, bw, size))
    return (v[:, 0] > x_lo) & (v[:, 0] < x_hi) & (v[:, 1] > y_lo) & (v[:, 1] < y_hi)


def filter_mesh(v, f, roi, bw, size=512):
    keep = filter_mask(v, roi, bw, size)
    fkeep = keep[f].all(axis=1)
    new_id = np.cumsum(keep) - 1
    return {'verts': v[keep], 'faces': new_id[f[fkeep]]}


# ---------------------------------------------------------------- vector helpers (one rounding per op)
def _dot(u, w):
    return (u[..., 0] * w[..., 0] + u[..., 1] * w[..., 1]) + u[..., 2] * w[..., 2]


def _cross(u, w):
    return np.stack([u[..., 1] * w[..., 2] - u[..., 2] * w[..., 1],
                     u[..., 2] * w[..., 0] - u[..., 0] * w[..., 2],
                     u[..., 0] * w[..., 1] - u[..., 1] * w[..., 0]], -1)


def _col(x):
    return x[..., None]


# ---------------------------------------------------------------- closest point
def closest_on_segment(p, a, b):
    ab = b - a
    t = _dot(p - a, ab)
    den = _dot(ab, ab)
    with np.errstate(divide='ignore', invalid='ignore'):
        q = a + _col(t / den) * ab
    q = np.where(_col(t >= den), b, q)
    return np.where(_col(~(t > 0)), a, q)


def closest_on_triangle(p, a, b, c):
    """Closest point of each triangle (a, b, c) to p (all broadcast to (..., 3)) and its squared distance."""
    p, a, b, c = np.broadcast_arrays(p, a, b, c)
    ab, ac, ap = b - a, c - a, p - a
    d1, d2 = _dot(ab, ap), _dot(ac, ap)
    bp = p - b
    d3, d4 = _dot(ab, bp), _dot(ac, bp)
    vc = d1 * d4 - d3 * d2
    cp = p - c
    d5, d6 = _dot(ab, cp), _dot(ac, cp)
    vb = d5 * d2 - d1 * d6
    va = d3 * d6 - d5 * d4
    e43, e56 = d4 - d3, d5 - d6
    den_ab, den_ac, den_bc = d1 - d3, d2 - d6, e43 + e56
    tot = (va + vb) + vc
    with np.errstate(divide='ignore', invalid='ignore', over='ignore'):
        q_ab = a + _col(d1 / den_ab) * ab
        q_ac = a + _col(d2 / den_ac) * ac
        q_bc = b + _col(e43 / den_bc) * (c - b)
        inv = 1.0 / tot
        q_in = (a + _col(vb * inv) * ab) + _col(vc * inv) * ac
    # Ericson's regions in his order: first true wins
    conds = [(d1 <= 0) & (d2 <= 0), (d3 >= 0) & (d4 <= d3), (vc <= 0) & (d1 >= 0) & (d3 <= 0),
             (d6 >= 0) & (d5 <= d6), (vb <= 0) & (d2 >= 0) & (d6 <= 0), (va <= 0) & (e43 >= 0) & (e56 >= 0)]
    region = np.select(conds, [0, 1, 2, 3, 4, 5], 6)
    q = np.select([_col(region == k) for k in range(6)], [a, b, q_ab, c, q_ac, q_bc], q_in)
    degenerate = (((region == 2) & (den_ab == 0)) | ((region == 4) & (den_ac == 0)) | ((region == 5) & (den_bc == 0))
                  | ((region == 6) & (tot == 0)))
    if degenerate.any():
        q0, q1, q2 = closest_on_segment(p, a, b), closest_on_segment(p, b, c), closest_on_segment(p, c, a)
        best = _dot(p - q0, p - q0)
        e1 = _dot(p - q1, p - q1)
        m1 = e1 < best
        qd = np.where(_col(m1), q1, q0)
        best = np.where(m1, e1, best)
        qd = np.where(_col(_dot(p - q2, p - q2) < best), q2, qd)
        q = np.where(_col(degenerate), qd, q)
    lo = np.fmin(np.fmin(a, b), c)
    hi = np.fmax(np.fmax(a, b), c)
    q = np.fmin(np.fmax(q, lo), hi)
    d = p - q
    return q, _dot(d, d)


def point_mesh_squared_distance(P, V, F, chunk=1 << 21):
    """Exhaustive search over every face: (dist2 (n,), face (n,) int64, closest (n,3)), ties to the smallest face id."""
    P, V = np.asarray(P, np.float64), np.asarray(V, np.float64)
    F = np.asarray(F, np.int64)
    a, b, c = V[F[:, 0]], V[F[:, 1]], V[F[:, 2]]
    n = len(P)
    d2 = np.empty(n)
    face = np.empty(n, np.int64)
    closest = np.empty((n, 3))
    step = max(1, chunk // max(1, len(F)))
    for s in range(0, n, step):
        p = P[s:s + step, None, :]
        q, e = closest_on_triangle(p, a[None], b[None], c[None])
        j = np.argmin(e, axis=1)
        r = np.arange(len(j))
        d2[s:s + step], face[s:s + step], closest[s:s + step] = e[r, j], j, q[r, j]
    return d2, face, closest


# ---------------------------------------------------------------- sampler
def face_areas(V, F):
    """|cross(b-a, c-a)| (twice the area) per face, float64."""
    V = np.asarray(V, np.float64)
    a, b, c = V[F[:, 0]], V[F[:, 1]], V[F[:, 2]]
    x = _cross(b - a, c - a)
    return np.sqrt(_dot(x, x))


def face_weights(V, F):
    area = face_areas(V, F)
    m = area.max()
    if not m > 0:
        return np.zeros(len(area), np.uint64)
    return np.floor(area / m * 4294967296.0).astype(np.uint64)


def face_cdf(V, F):
    return np.cumsum(face_weights(V, F), dtype=np.uint64)


def mulhi64(k, t):
    """floor(k * t / 2^64) elementwise for uint64 k and a uint64 scalar t, in 32-bit limbs."""
    k, t = np.asarray(k, np.uint64), np.uint64(t)
    s32 = np.uint64(32)
    kh, kl, th, tl = k >> s32, k & _M32, t >> s32, t & _M32
    ll, hl, lh, hh = kl * tl, kh * tl, kl * th, kh * th
    mid = (ll >> s32) + (hl & _M32) + lh
    return hh + (hl >> s32) + (mid >> s32)


def sample_from_bits(V, F, face_bits, bary_u):
    """The sampler with injected bits: (B (n,3), FI (n,) int64, points (n,3))."""
    V = np.asarray(V, np.float64)
    F = np.asarray(F, np.int64)
    cdf = face_cdf(V, F)
    total = cdf[-1]
    if total == 0:
        raise ValueError('every face has zero area')
    fi = np.searchsorted(cdf, mulhi64(face_bits, total), side='right').astype(np.int64)
    a, b = bary_u[:, 0].astype(np.float64), bary_u[:, 1].astype(np.float64)
    flip = (a + b) > 1
    a, b = np.where(flip, 1 - a, a), np.where(flip, 1 - b, b)
    b0 = (1 - a) - b
    B = np.stack([b0, a, b], 1)
    f = F[fi]
    pts = (V[f[:, 0]] * b0[:, None] + V[f[:, 1]] * a[:, None]) + V[f[:, 2]] * b[:, None]
    return B, fi, pts


# ---------------------------------------------------------------- metrics
def point_mesh_f1(p2s, s2p, th):
    pre, rec = (p2s <= th).mean(), (s2p <= th).mean()
    f1 = 2 * pre * rec / (pre + rec) if not (pre == 0 and rec == 0) else 0.0
    return {'precision': pre, 'recall': rec, 'threshold': th, 'f1': f1}


def measure_geometry(mc_verts, mc_faces, gt_verts, gt_faces, roi, bw, bits_pred, bits_gt, thresholds=THRESHOLDS):
    """One subject of measure.py:141-201 with injected sampler bits ((face_bits, bary_u) per mesh).  Returns the
    per-subject numbers and the intermediate arrays."""
    pv = np.asarray(mc_verts).astype(np.float64) * np.array([-1.0, 1.0, 1.0])
    pred = filter_mesh(pv, np.asarray(mc_faces), roi, bw)
    gt = filter_mesh(np.asarray(gt_verts), np.asarray(gt_faces), roi, bw)
    if len(pred['faces']) == 0 or len(gt['faces']) == 0:
        raise ValueError('the region of interest leaves no faces')
    gv = gt['verts'].astype(np.float64) * np.array([-1.0, 1.0, -1.0])
    pts_pred = sample_from_bits(pred['verts'], pred['faces'], *bits_pred)[2]
    pts_gt = sample_from_bits(gv, gt['faces'], *bits_gt)[2]
    p2s = np.sqrt(point_mesh_squared_distance(pts_pred, gv, gt['faces'])[0])
    s2p = np.sqrt(point_mesh_squared_distance(pts_gt, pred['verts'], pred['faces'])[0])
    out = {'p2s': p2s.mean(), 's2p': s2p.mean(), 'cd': (p2s.mean() + s2p.mean()) / 2}
    for th in thresholds:
        r = point_mesh_f1(p2s, s2p, th)
        name = f'{int(th * 1000):03d}'
        out[f'precision_{name}'], out[f'recall_{name}'], out[f'f1_{name}'] = r['precision'], r['recall'], r['f1']
    arrays = {'pred_verts': pred['verts'], 'pred_faces': pred['faces'], 'gt_verts': gt['verts'], 'gt_faces': gt['faces'],
              'points_pred': pts_pred, 'points_gt': pts_gt, 'p2s_all': p2s, 's2p_all': s2p}
    return out, arrays
