"""Marching cubes on the device - the B200 replacement for ``marching_cubes`` (reference
``_util/eg3d_metrics3d.py:186-210``; SURVEY.md section 8f-2), the geometry step of ``_scripts/eval/generate.py:97-105``.

The reference runs ``skimage.measure.marching_cubes(method='lewiner')`` on the host over the 255^3 cells of the
volume, then looks up every vertex colour in a Python loop.  Here ``p3d_mc_count`` / ``p3d_mc_emit``
(include/p3d_mesh.h) extract the mesh with one host synchronisation (the mesh size), and the colours are gathered on
the device from only the three channels at the vertex voxels.

    ``marching_cubes_device``   CUDA volume (+ optional (3,D0,D1,D2) rgb view, any strides) -> dict of CUDA tensors
    ``marching_cubes``          drop-in for the reference function: same arguments, same returned dict of numpy arrays

The triangulation contract (and how it deviates from skimage's Lewiner tables) is stated in oracle/mesh_oracle.py.
``egm.marching_cubes = panic3d_b200.mesh.marching_cubes`` rebinds the reference name (INTEGRATION.md).  No CPU path:
the extraction always runs on a CUDA device.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from .volume import _AttrDict


def marching_cubes_device(density, level=0.5, rgb=None):
    """Iso-surface of ``density`` (CUDA tensor (D0,D1,D2)) at ``level`` (cast to fp32; inside is ``density > level``).

    Returns ``{'verts' (V,3) fp32 in index space (axis0, axis1, axis2), 'faces' (F,3) int32, 'normals' (V,3),
    'values' (V,), 'colors' (V,3) or None}`` as CUDA tensors.  ``rgb`` is a (3,D0,D1,D2) fp32 view on the same device,
    read in place with its strides; ``colors`` are its values at the truncated vertex positions.  Raises
    ``ValueError`` when ``level`` is outside the volume's range and ``RuntimeError`` when nothing crosses it, like
    skimage."""
    if not (torch.is_tensor(density) and density.is_cuda):
        raise RuntimeError('panic3d_b200.mesh.marching_cubes_device has no CPU path: density must be a CUDA tensor')
    if density.dim() != 3 or min(density.shape) < 2:
        raise ValueError(f'panic3d_b200.mesh: density must be (D0,D1,D2) with every dimension >= 2, got {tuple(density.shape)}')
    dev = density.device
    vol = density.detach().float().contiguous()
    D0, D1, D2 = (int(x) for x in vol.shape)
    if rgb is not None:
        if not (torch.is_tensor(rgb) and rgb.device == dev and tuple(rgb.shape) == (3, D0, D1, D2)):
            raise ValueError(f'panic3d_b200.mesh: rgb must be a (3,{D0},{D1},{D2}) tensor on {dev}')
        rgb = rgb.detach()
        if rgb.dtype != torch.float32:
            rgb = rgb.float()
    L = _lib.lib()
    nbytes = L.p3d_mc_workspace_bytes(D0, D1, D2)
    if nbytes == 0:
        _lib.check(-1)
    lvl = float(np.float32(level))
    with torch.cuda.device(dev):
        stream = _lib.stream_ptr(dev)
        ws = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        counts, rng = (C.c_int64 * 3)(), (C.c_float * 2)()
        _lib.check(L.p3d_mc_count(vol.data_ptr(), D0, D1, D2, lvl, ws.data_ptr(), nbytes, counts, rng, stream))
        if not rng[0] <= lvl <= rng[1]:
            raise ValueError('Surface level must be within volume data range.')
        if counts[2] == 0:
            raise RuntimeError('No surface found at the given iso value.')
        nv, nf = int(counts[0]), int(counts[1])
        verts = torch.empty((nv, 3), dtype=torch.float32, device=dev)
        normals = torch.empty((nv, 3), dtype=torch.float32, device=dev)
        values = torch.empty((nv,), dtype=torch.float32, device=dev)
        colors = torch.empty((nv, 3), dtype=torch.float32, device=dev) if rgb is not None else None
        faces = torch.empty((nf, 3), dtype=torch.int32, device=dev)
        strides = rgb.stride() if rgb is not None else (0, 0, 0, 0)
        _lib.check(L.p3d_mc_emit(vol.data_ptr(), D0, D1, D2, lvl, ws.data_ptr(), nbytes, _lib.ptr(rgb), *strides,
                                 verts.data_ptr(), normals.data_ptr(), values.data_ptr(), _lib.ptr(colors), faces.data_ptr(),
                                 stream))
    return {'verts': verts, 'faces': faces, 'normals': normals, 'values': values, 'colors': colors}


def _to_device(x, dev):
    if torch.is_tensor(x):
        return x if x.is_cuda else x.to(dev)
    return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(dev)


def marching_cubes(vol, rgbs, boxwarp, level=0.5):
    """Drop-in for ``_util.eg3d_metrics3d.marching_cubes`` (eg3d_metrics3d.py:186-210): same arguments, same returned
    dict (``verts``, ``faces``, ``normals``, ``values``, ``colors``) of numpy arrays.

    ``vol`` (R,R,R) and ``rgbs`` (>=3,R,R,R) may be numpy arrays, as ``generate.py`` passes them (uploaded), or CUDA
    tensors such as ``query_volume(...)['densities'][0,0]`` and ``['rgbs'][0,:3]``, read in place: then only the three
    colour channels at the vertex voxels are read instead of copying all 32 channels (2.15 GB at 256^3) to the host.
    The colour lookup and the index -> world scaling are the reference's own lines, applied to the device results."""
    shape_res = vol.shape[-1]
    assert vol.shape[0] == vol.shape[1] == vol.shape[2]
    dev = vol.device if torch.is_tensor(vol) and vol.is_cuda else torch.device('cuda', torch.cuda.current_device())
    m = marching_cubes_device(_to_device(vol, dev), level=level, rgb=_to_device(rgbs[:3], dev))
    mc_vert = m['verts'].cpu().numpy()
    bw = boxwarp
    mc_vert = mc_vert / shape_res * bw - 0.5 * bw
    return _AttrDict({
        'verts': mc_vert,
        'faces': m['faces'].cpu().numpy(),
        'normals': m['normals'].cpu().numpy(),
        'values': m['values'].cpu().numpy(),
        'colors': m['colors'].cpu().numpy(),
    })
