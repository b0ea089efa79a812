"""Eval geometry metrics on the device - the 3-D half of the reference's ``_scripts/eval/measure.py`` (lines 54-99 and
141-201): Chamfer distance and F1 between the predicted mesh and the ground-truth mesh of one subject.

The reference runs ``igl.random_points_on_mesh`` and ``igl.point_mesh_squared_distance`` (a host AABB tree, built twice
per subject over meshes of ~372k faces); igl is not a dependency here.  ``p3d_surface_sample``, ``p3d_bvh_build`` and
``p3d_point_mesh_distance`` (include/p3d_geom.h) do that work in float64 on the device: an area-weighted sampler with an
exact integer CDF, an LBVH, and a traversal that equals exhaustive search bit for bit.  Filtering, the frame flips and
the final means are torch operations on the device.

    ``filter_mesh``                   measure.py:54-76 (the region-of-interest crop)
    ``random_points_on_mesh``         igl's name: (barycentrics (n,3), faces (n,))
    ``point_mesh_squared_distance``   igl's name and triple: (dist2, face, closest point)
    ``get_point_mesh_distance``       measure.py:77-86
    ``point_mesh_f1``                 measure.py:87-99
    ``measure_geometry``              the per-subject block measure.py:141-201

Every function accepts numpy arrays or CUDA tensors; numpy in gives numpy out, CUDA tensors in give CUDA tensors out.
There is no CPU path: the work always runs on a CUDA device (CPU tensors raise ``RuntimeError``).  The contract is
written out in oracle/metrics3d_oracle.py.
"""
from __future__ import annotations

import secrets
import zlib

import numpy as np
import torch

from . import _lib
from .volume import _AttrDict

THRESHOLDS = (0.005, 0.01, 0.05, 0.1, 0.5)
GEOM_ZERO_AREA, GEOM_STACK_OVERFLOW = 1, 2          # status bits of include/p3d_geom.h
_U64 = 1 << 64


# ---------------------------------------------------------------- input plumbing
def _is_numpy(*xs):
    return any(isinstance(x, np.ndarray) for x in xs)


def _device(*xs):
    for x in xs:
        if torch.is_tensor(x):
            if not x.is_cuda:
                raise RuntimeError('panic3d_b200.metrics3d has no CPU path: pass numpy arrays or CUDA tensors')
            return x.device
    return torch.device('cuda', torch.cuda.current_device())


def _cuda(x, dev, dtype=None):
    if torch.is_tensor(x):
        if not x.is_cuda:
            raise RuntimeError('panic3d_b200.metrics3d has no CPU path: pass numpy arrays or CUDA tensors')
        t = x.detach().to(dev)
    else:
        t = torch.from_numpy(np.ascontiguousarray(x)).to(dev)
    return (t if dtype is None else t.to(dtype)).contiguous()


def _out(t, numpy):
    return t.cpu().numpy() if numpy else t


def seed_value(seed):
    """The 64-bit Philox key of ``seed``: an int as is (mod 2^64), a str through adler32 of its UTF-8 bytes as the
    reference's ``np_seed`` does (_util/util_v1.py:102-113), None a fresh random key (``np_seed(None)`` reseeds from
    the OS too)."""
    if seed is None:
        return secrets.randbits(64)
    if isinstance(seed, str):
        return zlib.adler32(bytes(seed, encoding='utf-8'))
    return int(seed) % _U64


def _check_status(s: int):
    if s & GEOM_ZERO_AREA:
        raise ValueError('panic3d_b200.metrics3d: every face of the mesh has zero area; cannot sample its surface')
    if s & GEOM_STACK_OVERFLOW:
        raise RuntimeError('panic3d_b200.metrics3d: BVH traversal stack overflow (p3d_point_mesh_distance)')


def _mesh(V, F, who):
    if V.dim() != 2 or V.shape[1] != 3 or F.dim() != 2 or F.shape[1] != 3:
        raise ValueError(f'panic3d_b200.metrics3d.{who}: verts must be (V,3) and faces (F,3), got {tuple(V.shape)}, {tuple(F.shape)}')
    if F.shape[0] == 0:
        raise ValueError(f'panic3d_b200.metrics3d.{who}: the mesh has no faces')
    return V.double().contiguous(), F.to(torch.int32).contiguous()


# ---------------------------------------------------------------- device primitives (no host synchronisation)
def _sample(V, F, n, key, stream_id, face_bits, bary_u, status):
    dev = V.device
    nf = int(F.shape[0])
    L = _lib.lib()
    nbytes = L.p3d_surface_sample_workspace_bytes(nf)
    if nbytes == 0:
        _lib.check(-1)
    ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    bary = torch.empty((n, 3), dtype=torch.float64, device=dev)
    face = torch.empty((n,), dtype=torch.int64, device=dev)
    pts = torch.empty((n, 3), dtype=torch.float64, device=dev)
    if face_bits is not None:
        if bary_u is None or tuple(face_bits.shape) != (n,) or tuple(bary_u.shape) != (n, 2):
            raise ValueError(f'panic3d_b200.metrics3d: face_bits must be ({n},) and bary_u ({n},2), given together')
    with torch.cuda.device(dev):
        _lib.check(L.p3d_surface_sample(V.data_ptr(), F.data_ptr(), nf, n, key, stream_id, _lib.ptr(face_bits), _lib.ptr(bary_u),
                                        ws.data_ptr(), nbytes, bary.data_ptr(), face.data_ptr(), pts.data_ptr(), status.data_ptr(),
                                        _lib.stream_ptr(dev)))
    return bary, face, pts


def _distance(P, V, F, status):
    dev = V.device
    nf, n = int(F.shape[0]), int(P.shape[0])
    L = _lib.lib()
    nbytes = L.p3d_bvh_workspace_bytes(nf)
    if nbytes == 0:
        _lib.check(-1)
    bvh = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    d2 = torch.empty((n,), dtype=torch.float64, device=dev)
    face = torch.empty((n,), dtype=torch.int64, device=dev)
    closest = torch.empty((n, 3), dtype=torch.float64, device=dev)
    with torch.cuda.device(dev):
        stream = _lib.stream_ptr(dev)
        _lib.check(L.p3d_bvh_build(V.data_ptr(), F.data_ptr(), nf, bvh.data_ptr(), nbytes, stream))
        _lib.check(L.p3d_point_mesh_distance(P.data_ptr(), n, V.data_ptr(), F.data_ptr(), nf, bvh.data_ptr(), nbytes, d2.data_ptr(),
                                             face.data_ptr(), closest.data_ptr(), status.data_ptr(), stream))
    return d2, face, closest


def roi_bounds(roi, bw, size=512):
    """The open box ``(x_lo, x_hi, y_lo, y_hi)`` of the region of interest ``roi = ((a0, a1), (s0, s1))`` (pixel origin
    and size in a ``size`` x ``size`` front view spanning ``bw``), as Python floats with measure.py's operation order."""
    (a0, a1), (s0, s1) = roi
    x_lo = -bw / 2 + (a1 / size) * bw
    y_hi = bw / 2 - (a0 / size) * bw
    return x_lo, x_lo + bw * (s1 / size), y_hi - bw * (s0 / size), y_hi


def _filter_masks(v, f, roi, bw, size):
    """measure.py:54-69: the box scalars as Python floats, compared in the dtype of ``v`` (numpy treats a Python float
    as a weak scalar, so an fp32 mesh meets bounds rounded to fp32)."""
    x_lo, x_hi, y_lo, y_hi = roi_bounds(roi, bw, size)

    def s(x):
        return torch.tensor(x, dtype=v.dtype, device=v.device)
    vmask = (v[:, 0] > s(x_lo)) & (v[:, 0] < s(x_hi)) & (v[:, 1] > s(y_lo)) & (v[:, 1] < s(y_hi))
    fmask = vmask[f.long()].all(dim=1)
    return vmask, fmask


def _compact(v, f, vmask, fmask, nv, nf):
    """v[vmask] and (cumsum(vmask)-1)[f[fmask]] with the sizes already known: no further host synchronisation (rows that
    are dropped land in a discarded slot)."""
    pos = torch.cumsum(vmask, 0) - 1
    vt = torch.where(vmask, pos, nv)
    verts = torch.empty((nv + 1, 3), dtype=v.dtype, device=v.device).index_copy_(0, vt, v)[:nv]
    ft = torch.where(fmask, torch.cumsum(fmask, 0) - 1, nf)
    faces = torch.empty((nf + 1, 3), dtype=torch.int64, device=v.device).index_copy_(0, ft, pos[f.long()])[:nf]
    return verts, faces


# ---------------------------------------------------------------- public API
def filter_mesh(v, f, roi, bw, size=512):
    """``measure.py:54-76``: keep the vertices strictly inside the region of interest in x and y, the faces whose three
    vertices are all kept (re-indexed), and the kept vertices no face references.  Returns ``{'verts', 'faces'}`` with
    verts in the dtype of ``v`` and int64 faces."""
    numpy = _is_numpy(v, f)
    dev = _device(v, f)
    V, Fc = _cuda(v, dev), _cuda(f, dev)
    vmask, fmask = _filter_masks(V, Fc, roi, bw, size)
    nv, nf = torch.stack([vmask.sum(), fmask.sum()]).tolist()
    verts, faces = _compact(V, Fc, vmask, fmask, nv, nf)
    return {'verts': _out(verts, numpy), 'faces': _out(faces, numpy)}


def random_points_on_mesh(n, V, F, seed=None, stream=0, face_bits=None, bary_u=None):
    """Area-weighted uniform points on the mesh, as ``igl.random_points_on_mesh(n, V, F)``: returns barycentrics
    ``B (n,3) fp64`` and faces ``FI (n,) int64``, the pair ``bary2cart`` consumes.  ``seed`` (int or str) and ``stream``
    select the Philox stream; ``face_bits (n,) uint64`` with ``bary_u (n,2) fp64`` replace the random bits."""
    numpy = _is_numpy(V, F)
    dev = _device(V, F, face_bits, bary_u)
    Vd, Fd = _mesh(_cuda(V, dev), _cuda(F, dev), 'random_points_on_mesh')
    fb = None if face_bits is None else _cuda(face_bits, dev, torch.uint64)
    bu = None if bary_u is None else _cuda(bary_u, dev, torch.float64)
    status = torch.zeros((1,), dtype=torch.int32, device=dev)
    B, FI, _ = _sample(Vd, Fd, int(n), seed_value(seed), int(stream), fb, bu, status)
    _check_status(int(status.item()))
    return _out(B, numpy), _out(FI, numpy)


def point_mesh_squared_distance(P, V, F):
    """``igl.point_mesh_squared_distance(P, V, F)``: for each point the squared distance to the mesh, the face it is
    attained on (ties to the smallest id) and the closest point - ``(dist2 (n,) fp64, face (n,) int64, closest (n,3)
    fp64)``, equal to exhaustive search over all faces."""
    numpy = _is_numpy(P, V, F)
    dev = _device(P, V, F)
    Vd, Fd = _mesh(_cuda(V, dev), _cuda(F, dev), 'point_mesh_squared_distance')
    Pd = _cuda(P, dev, torch.float64)
    if Pd.dim() != 2 or Pd.shape[1] != 3:
        raise ValueError(f'panic3d_b200.metrics3d.point_mesh_squared_distance: points must be (n,3), got {tuple(Pd.shape)}')
    status = torch.zeros((1,), dtype=torch.int32, device=dev)
    d2, face, closest = _distance(Pd, Vd, Fd, status)
    _check_status(int(status.item()))
    return _out(d2, numpy), _out(face, numpy), _out(closest, numpy)


def get_point_mesh_distance(queries, v, f):
    """``measure.py:77-86``: ``sqrt`` of ``point_mesh_squared_distance``."""
    d2, _, _ = point_mesh_squared_distance(queries, v, f)
    return np.sqrt(d2) if isinstance(d2, np.ndarray) else torch.sqrt(d2)


def point_mesh_f1(p2s, s2p, thresh):
    """``measure.py:87-99``: precision ``mean(p2s <= thresh)``, recall ``mean(s2p <= thresh)``, their F1 (0 when both
    are 0).  Returns ``{'precision', 'recall', 'threshold', 'f1'}`` (numpy float64 or 0-d CUDA tensors)."""
    numpy = _is_numpy(p2s, s2p)
    dev = _device(p2s, s2p)
    a, b = _cuda(p2s, dev, torch.float64), _cuda(s2p, dev, torch.float64)
    # count / n, as numpy's mean of a bool array: an exact integer sum, one division (by a device tensor: torch turns
    # a division by a Python scalar into a multiplication by its reciprocal, which can differ in the last bit)
    def n_of(x):
        return torch.full((), x.numel(), dtype=torch.float64, device=dev)
    pre = (a <= thresh).sum().double() / n_of(a)
    rec = (b <= thresh).sum().double() / n_of(b)
    f1 = torch.where((pre == 0) & (rec == 0), torch.zeros_like(pre), 2 * pre * rec / (pre + rec))
    if numpy:
        pre, rec, f1 = (np.float64(x) for x in torch.stack([pre, rec, f1]).tolist())
    return _AttrDict({'precision': pre, 'recall': rec, 'threshold': thresh, 'f1': f1})


def measure_geometry(mc, gt_verts, gt_faces, roi, bw=0.7, n_sample=10000, seed=None, thresholds=THRESHOLDS, injected=None):
    """The per-subject geometry block of ``measure.py:141-201`` for one subject.

    ``mc``: the predicted mesh, either the ``marching_cubes`` drop-in's dict (numpy, world units) or
    ``marching_cubes_device``'s output scaled to world units (``verts`` (V,3), ``faces`` (F,3)); ``gt_verts`` /
    ``gt_faces``: the ground-truth head mesh in its own frame (numpy or CUDA, any float dtype - the crop compares in
    it).  ``roi`` is the subject's ``area_of_interest``, ``seed`` the subject name (or an int).

    Steps: mirror the predicted x (float64 from here on); crop both meshes (``filter_mesh``); map the ground truth by
    ``diag(-1, 1, -1)``; sample ``n_sample`` points on each (Philox streams 0 and 1 of ``seed``); ``p2s`` = distances
    of the predicted points to the ground-truth mesh, ``s2p`` = of the ground-truth points to the predicted mesh.
    ``injected = ((face_bits, bary_u) predicted, (face_bits, bary_u) ground truth)`` replaces the random bits.

    Returns ``{'p2s', 's2p', 'cd', 'precision_XXX', 'recall_XXX', 'f1_XXX'}`` (XXX = ``int(th*1000):03d``, the
    reference's key) as numpy float64 - per subject; averaging over subjects is the caller's.  The meshes stay on the
    device; there are two host synchronisations, the cropped mesh sizes (to size the BVHs, and to raise ``ValueError``
    on an empty crop before any kernel runs) and the final numbers."""
    dev = _device(mc['verts'], mc['faces'], gt_verts, gt_faces)
    pv = _cuda(mc['verts'], dev, torch.float64) * torch.tensor([-1.0, 1.0, 1.0], dtype=torch.float64, device=dev)
    pf = _cuda(mc['faces'], dev)
    gv, gf = _cuda(gt_verts, dev), _cuda(gt_faces, dev)
    if not gv.is_floating_point():
        gv = gv.double()
    pvm, pfm = _filter_masks(pv, pf, roi, bw, 512)
    gvm, gfm = _filter_masks(gv, gf, roi, bw, 512)
    nvp, nfp, nvg, nfg = torch.stack([pvm.sum(), pfm.sum(), gvm.sum(), gfm.sum()]).tolist()     # host sync 1
    if nfp == 0 or nfg == 0:
        raise ValueError(f'panic3d_b200.metrics3d.measure_geometry: the region of interest leaves no faces '
                         f'(predicted {nfp}, ground truth {nfg})')
    pv, pf = _compact(pv, pf, pvm, pfm, nvp, nfp)
    gv, gf = _compact(gv, gf, gvm, gfm, nvg, nfg)
    gv = gv.double() * torch.tensor([-1.0, 1.0, -1.0], dtype=torch.float64, device=dev)      # cv2our_world_inv[:3,:3]
    pf, gf = pf.to(torch.int32).contiguous(), gf.to(torch.int32).contiguous()
    pv, gv = pv.contiguous(), gv.contiguous()
    key = seed_value(seed)
    n = int(n_sample)
    inj = [(None, None), (None, None)] if injected is None else [
        (_cuda(fb, dev, torch.uint64), _cuda(bu, dev, torch.float64)) for fb, bu in injected]
    status = torch.zeros((1,), dtype=torch.int32, device=dev)
    _, _, pts_pred = _sample(pv, pf, n, key, 0, *inj[0], status)
    _, _, pts_gt = _sample(gv, gf, n, key, 1, *inj[1], status)
    p2s = torch.sqrt(_distance(pts_pred, gv, gf, status)[0])
    s2p = torch.sqrt(_distance(pts_gt, pv, pf, status)[0])
    th = torch.tensor(thresholds, dtype=torch.float64, device=dev)
    row = torch.cat([torch.stack([p2s.sum(), s2p.sum(), status[0].double()]),
                     (p2s[None, :] <= th[:, None]).sum(1).double(), (s2p[None, :] <= th[:, None]).sum(1).double()])
    vals = row.tolist()                                                                         # host sync 2
    _check_status(int(vals[2]))
    p2s_mean, s2p_mean = np.float64(vals[0]) / n, np.float64(vals[1]) / n
    out = _AttrDict({'p2s': p2s_mean, 's2p': s2p_mean, 'cd': (p2s_mean + s2p_mean) / 2})
    k = len(thresholds)
    for i, t in enumerate(thresholds):
        pre, rec = np.float64(vals[3 + i]) / n, np.float64(vals[3 + k + i]) / n
        name = f'{int(t * 1000):03d}'
        out[f'precision_{name}'] = pre
        out[f'recall_{name}'] = rec
        out[f'f1_{name}'] = 2 * pre * rec / (pre + rec) if not pre == rec == 0.0 else np.float64(0.0)
    return out
