"""TEST INFRASTRUCTURE ONLY - CPU restatement of the marching-cubes contract that ``p3d_mc_count`` / ``p3d_mc_emit``
(include/p3d_mesh.h, csrc/marching_cubes.cu) implement: the configuration the reference hard-codes in
``_util/eg3d_metrics3d.py:186-210`` (``skimage.measure.marching_cubes(vol, level, spacing=(1,1,1),
gradient_direction='descent', step_size=1, allow_degenerate=False, method='lewiner', mask=None)``).

The contract (shared bit for bit with the kernel):
  * a corner is inside iff V > level (level cast to fp32); edge = lattice corner (i,j,k) + axis a, key 3*lin(i,j,k)+a
    with lin row-major over (D0,D1,D2); an edge whose two corners differ in inside-ness carries ONE vertex, shared by
    every cell around it; vertices are ordered by key;
  * position in index space (axis0, axis1, axis2): idx + t along the edge, t = (level - v_lo) / (v_hi - v_lo), every
    fp32 operation rounded separately;
  * per cell face: 2 crossings are paired; 4 crossings are paired by the asymptotic decider (Nielson & Hamann 1991):
    det = a*d - b*c of the face's values minus level in the face's lattice order, compared with the sign of the
    denominator a+d-b-c (positive iff a, d are the inside pair).  det of that sign joins the inside corners across the
    face, anything else (a tie included) separates them.  Both cells of a face compute the same bits;
  * segments are directed so that each triangle's right-hand normal points from inside to outside ('descent'): walking
    a face's corners counter-clockwise about its outward normal, a segment runs from an outside->inside crossing to the
    next crossing (separated) or the previous one (joined).  The segments chain into closed loops; each loop is fanned
    from its smallest vertex id, loops in order of their smallest vertex id, cells in linear order;
  * normals: -grad V (numpy.gradient) at the two corners, interpolated with t, normalised (zero stays zero);
  * values: max of the 8 corner values of the lowest-index cell containing the edge;
  * allow_degenerate=False: vertices at identical fp32 positions (only possible on lattice corners) merge onto the
    lowest id; faces with a repeated index are dropped, then unreferenced vertices, survivors keep their order.

Deviation from the reference (stated as for kornia / torchvision elsewhere in oracle/): the vertex SET is the one
skimage produces on the same volume (one per crossing edge, at the linearly interpolated point; last-ulp parity of t
unpinned), but the in-cell triangulation is our own, and Lewiner's interior tests (cases 4, 6, 7, 10, 12, 13) that
sometimes add a tunnel and a cell-centre vertex are not implemented, so in those cells the surface differs from
skimage's.  Parity with skimage output is therefore UNPINNED (skimage is not installed where this project runs);
the downstream metrics (measure.py) consume only verts / faces and sample points on the surface.
``tests/golden/make_golden_mesh.py`` pins what the reference's own ``marching_cubes`` does around the skimage call
(call arguments, the colour rule, the scaling) with this oracle's raw mesh standing in for skimage's.
Only ``tests/`` may import this module; the product path is ``panic3d_b200.mesh``.
"""
from __future__ import annotations

import numpy as np

F32 = np.float32

# cell corner c = 4*d0 + 2*d1 + d2 (offsets along axis 0, 1, 2): ascending c is ascending linear index
CORNERS = [((c >> 2) & 1, (c >> 1) & 1, c & 1) for c in range(8)]
# the 12 cell edges (corner, axis) in ascending global key order
EDGES = [(c, a) for c in range(8) for a in range(3) if CORNERS[c][a] == 0]
EDGE_ID = {e: n for n, e in enumerate(EDGES)}


def _corner(off):
    return 4 * off[0] + 2 * off[1] + off[2]


def _edge_between(c0, c1):
    a = [CORNERS[c0][x] != CORNERS[c1][x] for x in range(3)].index(True)
    return EDGE_ID[(c0 if CORNERS[c0][a] == 0 else c1, a)]


def _faces():
    """Per cell face: corners counter-clockwise about the outward normal, the edge after each of them, and the
    corners in the face's lattice order (a, b, c, d) for the decider."""
    out = []
    for n in range(3):
        for s in (0, 1):
            up, wp = (n + 1) % 3, (n + 2) % 3                # e_up x e_wp = e_n
            ring = [(1, 0), (1, 1), (0, 1), (0, 0)] if s else [(0, 0), (0, 1), (1, 1), (1, 0)]
            cyc = []
            for pu, pw in ring:
                off = [0, 0, 0]
                off[n], off[up], off[wp] = s, pu, pw
                cyc.append(_corner(off))
            u, w = sorted((up, wp))
            lat = []
            for pu, pw in ((0, 0), (0, 1), (1, 0), (1, 1)):
                off = [0, 0, 0]
                off[n], off[u], off[w] = s, pu, pw
                lat.append(_corner(off))
            out.append((cyc, [_edge_between(cyc[q], cyc[(q + 1) % 4]) for q in range(4)], lat))
    return out


FACES = _faces()


def cell_loops(inside, f):
    """Closed vertex loops of one cell as lists of local edge ids (EDGES order), each starting at its smallest id,
    loops in order of that id.  inside: 8 bools; f: 8 fp32 values minus level (corner order CORNERS)."""
    nxt = {}
    for cyc, cedge, lat in FACES:
        ins = [bool(inside[c]) for c in cyc]
        cross = [q for q in range(4) if ins[q] != ins[(q + 1) % 4]]
        if not cross:
            continue
        joined = False
        if len(cross) == 4:
            a, b, c, d = (F32(f[x]) for x in lat)
            det = F32(a * d) - F32(b * c)
            joined = bool(det > 0) if inside[lat[0]] else bool(det < 0)
        for n, q in enumerate(cross):
            if not ins[q]:                                  # outside -> inside along the counter-clockwise walk
                nxt[cedge[q]] = cedge[cross[(n + (-1 if joined else 1)) % len(cross)]]
    loops, seen = [], set()
    for e in sorted(nxt):
        if e in seen:
            continue
        loop = [e]
        seen.add(e)
        while nxt[loop[-1]] != e:
            loop.append(nxt[loop[-1]])
            seen.add(loop[-1])
        loops.append(loop)
    return loops


def cell_triangles(inside, f):
    """Fan triangulation of cell_loops: (v0, vk, vk+1) per loop, local edge ids."""
    return [(lp[0], lp[k], lp[k + 1]) for lp in cell_loops(inside, f) for k in range(1, len(lp) - 1)]


def _edge_t(lo, hi, level):
    return (level - lo) / (hi - lo)


def marching_cubes(V, level=0.5):
    """(verts (V,3) fp32 index space, faces (F,3) int32, normals (V,3) fp32, values (V,) fp32) - what the reference
    reads from skimage.measure.marching_cubes.  Raises ValueError / RuntimeError as skimage does."""
    V = np.ascontiguousarray(V, dtype=F32)
    if V.ndim != 3 or min(V.shape) < 2:
        raise ValueError('Input volume should be a 3D numpy array with every dimension >= 2.')
    level = F32(level)
    if not V.min() <= level <= V.max():
        raise ValueError('Surface level must be within volume data range.')
    D = V.shape
    inside = V > level
    grad = np.gradient(V)
    cellmax = V[:-1, :-1, :-1]
    for c in range(1, 8):
        o = CORNERS[c]
        cellmax = np.maximum(cellmax, V[o[0]:D[0] - 1 + o[0], o[1]:D[1] - 1 + o[1], o[2]:D[2] - 1 + o[2]])

    # ---- vertices: one per crossing edge, ordered by key 3*lin + a
    keys, pos, nrm, val = [], [], [], []
    for a in range(3):
        lo_sl = tuple(slice(0, D[x] - 1) if x == a else slice(None) for x in range(3))
        hi_sl = tuple(slice(1, D[x]) if x == a else slice(None) for x in range(3))
        cr = np.argwhere(inside[lo_sl] != inside[hi_sl])
        if len(cr) == 0:
            continue
        hi_idx = cr.copy()
        hi_idx[:, a] += 1
        vlo, vhi = V[tuple(cr.T)], V[tuple(hi_idx.T)]
        t = _edge_t(vlo, vhi, level)
        p = cr.astype(F32)
        p[:, a] = p[:, a] + t
        glo = np.stack([-grad[x][tuple(cr.T)] for x in range(3)], 1)
        ghi = np.stack([-grad[x][tuple(hi_idx.T)] for x in range(3)], 1)
        n = glo + t[:, None] * (ghi - glo)
        norm = np.sqrt(n[:, 0] * n[:, 0] + n[:, 1] * n[:, 1] + n[:, 2] * n[:, 2])
        n = np.where(norm[:, None] > 0, n / np.where(norm > 0, norm, F32(1))[:, None], F32(0))
        cell = cr.copy()                                       # lowest-index cell containing the edge
        for x in range(3):
            if x != a:
                cell[:, x] = np.maximum(cell[:, x] - 1, 0)
        keys.append(3 * np.ravel_multi_index(tuple(cr.T), D).astype(np.int64) + a)
        pos.append(p); nrm.append(n.astype(F32)); val.append(cellmax[tuple(cell.T)])
    if not keys:
        raise RuntimeError('No surface found at the given iso value.')
    keys = np.concatenate(keys)
    order = np.argsort(keys, kind='stable')
    keys, pos, nrm, val = keys[order], np.concatenate(pos)[order], np.concatenate(nrm)[order], np.concatenate(val)[order]
    vid = {int(k): n for n, k in enumerate(keys)}

    # ---- faces: loop over the cells that have a crossing, in linear order
    ins_c = np.stack([inside[o[0]:D[0] - 1 + o[0], o[1]:D[1] - 1 + o[1], o[2]:D[2] - 1 + o[2]] for o in CORNERS], -1)
    active = np.argwhere(ins_c.any(-1) & ~ins_c.all(-1))     # argwhere is row-major: ascending cell index
    fval = V - level
    faces = []
    for i, j, k in active:
        tris = cell_triangles(ins_c[i, j, k], [fval[i + o[0], j + o[1], k + o[2]] for o in CORNERS])
        base = [3 * (((i + CORNERS[c][0]) * D[1] + j + CORNERS[c][1]) * D[2] + k + CORNERS[c][2]) + a for c, a in EDGES]
        faces.extend((vid[base[x]], vid[base[y]], vid[base[z]]) for x, y, z in tris)
    faces = np.asarray(faces, dtype=np.int64).reshape(-1, 3)

    # ---- allow_degenerate=False: merge identical positions (lattice corners) onto the lowest id
    on_corner = np.all(pos == np.floor(pos), axis=1)
    rep = np.arange(len(keys))
    if on_corner.any():
        ids = np.nonzero(on_corner)[0]
        ck = np.ravel_multi_index(tuple(pos[ids].astype(np.int64).T), D)
        first = {}
        for n, c in zip(ids, ck):                               # ids ascend: the first one seen is the lowest
            rep[n] = first.setdefault(int(c), int(n))
    faces = rep[faces]
    keep = (faces[:, 0] != faces[:, 1]) & (faces[:, 1] != faces[:, 2]) & (faces[:, 0] != faces[:, 2])
    faces = faces[keep]
    used = np.zeros(len(keys), bool)
    used[faces.ravel()] = True
    remap = np.cumsum(used) - 1
    return pos[used], remap[faces].astype(np.int32), nrm[used], val[used]


def postprocess(verts, faces, normals, values, rgbs, boxwarp, shape_res):
    """eg3d_metrics3d.py:198-210 after the skimage call: colours rgbs[:3, a, b, c] at the truncated vertex indices, then
    the index -> world scaling (numpy keeps fp32 with Python scalars)."""
    colors = np.stack([rgbs[:3, a, b, c] for a, b, c in verts.astype(int)])
    bw = boxwarp
    return {'verts': verts / shape_res * bw - 0.5 * bw, 'faces': faces, 'normals': normals, 'values': values, 'colors': colors}
