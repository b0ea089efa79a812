"""ctypes binding of lib/libp3d.so (the C ABI declared in include/p3d_render.h, include/p3d_ops.h, include/p3d_mesh.h and
include/p3d_geom.h).

The library is loaded lazily on first use and the load FAILS LOUDLY: there is no CPU or
PyTorch fallback behind any op of this package."""
from __future__ import annotations

import ctypes as C
import os
import threading

PKG = os.path.dirname(os.path.abspath(__file__))
# P3D_LIBP3D: load another build of the library (A/B experiments: profiles/experiments/build_variants.py); default in-tree
LIB_PATH = os.environ.get('P3D_LIBP3D') or os.path.join(PKG, 'lib', 'libp3d.so')

P3D_PLANES_EG3D, P3D_PLANES_PANIC3D = 0, 1
P3D_RAYS_NUMERIC, P3D_RAYS_AUTOBOX = 0, 1
P3D_MLP_FP32_SIMT, P3D_MLP_TC_3XBF16, P3D_MLP_TC_BF16 = 0, 1, 2


class RenderParams(C.Structure):
    """Mirror of ``p3d_render_params`` (include/p3d_render.h) - field order and types must match."""
    _fields_ = [
        ('n_views', C.c_int32), ('n_rays', C.c_int32), ('n_coarse', C.c_int32), ('n_fine', C.c_int32),
        ('channels', C.c_int32), ('plane_h', C.c_int32), ('plane_w', C.c_int32),
        ('hidden', C.c_int32), ('out_dim', C.c_int32),
        ('stride_view', C.c_int64), ('stride_plane', C.c_int64), ('stride_row', C.c_int64), ('stride_col', C.c_int64),
        ('planes_bf16', C.c_int32),
        ('box_warp', C.c_double), ('ray_start', C.c_double), ('ray_end', C.c_double),
        ('ray_mode', C.c_int32), ('disparity', C.c_int32), ('white_back', C.c_int32), ('plane_mode', C.c_int32),
        ('triplane_crop', C.c_double), ('cull_clouds', C.c_double), ('binarize_clouds', C.c_double),
        ('w1_gain', C.c_float), ('b1_gain', C.c_float), ('w2_gain', C.c_float), ('b2_gain', C.c_float),
        ('force_sigmoid', C.c_int32), ('mlp_mode', C.c_int32),
        ('seed', C.c_uint64),
        ('defer_depth_clamp', C.c_int32), ('reserved0', C.c_int32),
    ]


_lock = threading.Lock()
_lib = None

_VP = C.c_void_p
_PROTOS = {
    # name: (restype, argtypes)
    'p3d_version': (C.c_char_p, []),
    'p3d_last_error': (C.c_char_p, []),
    'p3d_launch_count': (C.c_uint64, []),
    'p3d_planes_to_channels_last': (C.c_int, [_VP, _VP, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _VP]),
    'p3d_raygen_pinhole': (C.c_int, [_VP, _VP, C.c_int32, C.c_int32, _VP, _VP, _VP]),
    'p3d_raygen_ortho': (C.c_int, [_VP, _VP, C.c_int32, C.c_int32, C.c_double, _VP, _VP, _VP]),
    'p3d_render_workspace_bytes': (C.c_size_t, [C.POINTER(RenderParams)]),
    'p3d_render_fused_supported': (C.c_int, [C.POINTER(RenderParams)]),
    'p3d_decode_tc_supported': (C.c_int, [C.POINTER(RenderParams), C.c_int64]),
    'p3d_render_forward': (C.c_int, [C.POINTER(RenderParams)] + [_VP] * 9 + [_VP, C.c_size_t] + [_VP] * 5),
    'p3d_decode_points': (C.c_int, [C.POINTER(RenderParams)] + [_VP] * 6 + [C.c_int64, _VP, _VP, _VP]),
    'p3d_decode_points_backward': (C.c_int, [C.POINTER(RenderParams)] + [_VP] * 6 + [C.c_int64] + [_VP] * 7 + [_VP]),
    'p3d_volume_query': (C.c_int, [C.POINTER(RenderParams)] + [_VP] * 5 + [C.c_int32, C.c_double, C.c_double, C.c_double] + [_VP] * 5),
    'p3d_render_forward_host': (C.c_int, [C.POINTER(RenderParams)] + [_VP] * 7 + [C.c_int32] + [_VP] * 6),
    'p3d_render_backward_scratch_bytes': (C.c_size_t, [C.POINTER(RenderParams)]),
    'p3d_render_backward': (C.c_int, [C.POINTER(RenderParams)] + [_VP] * 7 + [_VP, C.c_size_t] + [_VP] * 5 + [_VP, C.c_size_t] + [_VP] * 6),
    'p3d_render_depth_bounds': (C.c_int, [_VP, _VP, _VP]),
    'p3d_depth_finalize': (C.c_int, [_VP, C.c_int64, _VP, _VP]),
    'p3d_host_arena_release': (None, []),
    'p3d_ipc_alloc': (C.c_int, [C.c_size_t, C.POINTER(_VP), C.c_char_p]),
    'p3d_ipc_open': (C.c_int, [C.c_char_p, C.POINTER(_VP)]),
    'p3d_ipc_close': (C.c_int, [_VP]),
    'p3d_ipc_free': (C.c_int, [_VP]),
    'p3d_copy_async': (C.c_int, [_VP, _VP, C.c_size_t, _VP]),
    'p3d_profile_enable': (None, [C.c_int]),
    'p3d_profile_read': (C.c_int, [C.POINTER(C.c_double), C.POINTER(C.c_uint64), C.c_int, C.c_int]),
    # include/p3d_mesh.h (marching cubes, panic3d_b200.mesh)
    'p3d_mc_workspace_bytes': (C.c_size_t, [C.c_int32] * 3),
    'p3d_mc_count': (C.c_int, [_VP] + [C.c_int32] * 3 + [C.c_double, _VP, C.c_size_t, C.POINTER(C.c_int64), C.POINTER(C.c_float), _VP]),
    'p3d_mc_emit': (C.c_int, [_VP] + [C.c_int32] * 3 + [C.c_double, _VP, C.c_size_t, _VP] + [C.c_int64] * 4 + [_VP] * 5 + [_VP]),
    # include/p3d_geom.h (surface sampling, BVH, point-to-mesh distance; panic3d_b200.metrics3d)
    'p3d_surface_sample_workspace_bytes': (C.c_size_t, [C.c_int64]),
    'p3d_surface_sample': (C.c_int, [_VP, _VP, C.c_int64, C.c_int64, C.c_uint64, C.c_uint32, _VP, _VP, _VP, C.c_size_t] + [_VP] * 5),
    'p3d_bvh_workspace_bytes': (C.c_size_t, [C.c_int64]),
    'p3d_bvh_build': (C.c_int, [_VP, _VP, C.c_int64, _VP, C.c_size_t, _VP]),
    'p3d_point_mesh_distance': (C.c_int, [_VP, C.c_int64, _VP, _VP, C.c_int64, _VP, C.c_size_t] + [_VP] * 5),
}


def declared_symbols():
    """Every symbol the headers declare and the binding expects (used by the CPU export test)."""
    return sorted(_PROTOS)


def register_protos(protos: dict):
    """Other modules (ops) add their entry points here before the first load."""
    _PROTOS.update(protos)
    if _lib is not None:
        _bind(_lib, protos)


def _bind(lib, protos):
    for name, (res, args) in protos.items():
        fn = getattr(lib, name)          # AttributeError if the .so does not export it
        fn.restype = res
        fn.argtypes = args


def lib():
    """Load (once) and return the shared library; raises RuntimeError if it is missing."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        f'{LIB_PATH} is missing: build it with `python -c "import __graft_entry__ as g; g.build()"` '
                        '(there is no CPU / PyTorch fallback for the panic3d_b200 ops)')
                handle = C.CDLL(LIB_PATH)
                _bind(handle, _PROTOS)
                _lib = handle
    return _lib


def check(rc: int):
    if rc != 0:
        msg = lib().p3d_last_error().decode('utf-8', 'replace')
        raise RuntimeError(f'p3d error {rc}: {msg}')


def launch_count() -> int:
    return int(lib().p3d_launch_count())


def ptr(t):
    """data_ptr of a tensor or None -> NULL."""
    return None if t is None else t.data_ptr()


def stream_ptr(device=None):
    import torch
    return torch.cuda.current_stream(device).cuda_stream
