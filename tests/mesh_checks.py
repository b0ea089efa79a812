"""Shared mesh properties and test fields for the marching-cubes tests (oracle on the CPU, kernel on the GPU)."""
from __future__ import annotations

import numpy as np


def _edges(faces):
    return np.stack([faces[:, [0, 1]], faces[:, [1, 2]], faces[:, [2, 0]]], 1).reshape(-1, 2).astype(np.int64)


def edge_face_counts(faces):
    """Undirected edges (E,2) and the number of faces around each."""
    return np.unique(np.sort(_edges(faces), 1), axis=0, return_counts=True)


def consistently_oriented(faces):
    """Every directed edge appears once: neighbouring faces traverse their shared edge in opposite directions."""
    d = _edges(faces)
    return len(np.unique(d, axis=0)) == len(d)


def euler_characteristic(verts, faces):
    e, _ = edge_face_counts(faces)
    return len(verts) - len(e) + len(faces)


def assert_closed_oriented(verts, faces):
    _, cnt = edge_face_counts(faces)
    assert (cnt == 2).all(), np.unique(cnt, return_counts=True)
    assert consistently_oriented(faces)
    assert len(np.unique(faces)) == len(verts)                    # no unreferenced vertex


def assert_no_degenerates(verts, faces):
    assert ((faces[:, 0] != faces[:, 1]) & (faces[:, 1] != faces[:, 2]) & (faces[:, 0] != faces[:, 2])).all()
    assert len(np.unique(verts, axis=0)) == len(verts)


def face_normals(verts, faces):
    v = verts.astype(np.float64)
    return np.cross(v[faces[:, 1]] - v[faces[:, 0]], v[faces[:, 2]] - v[faces[:, 0]])


# ---------------------------------------------------------------- fields (fp32, outside padded so surfaces close)
def _grid(n):
    x = np.arange(n, dtype=np.float64) - (n - 1) / 2
    return np.meshgrid(x, x, x, indexing='ij')


def sphere(n=64, r=25.0):
    X, Y, Z = _grid(n)
    return (r - np.sqrt(X * X + Y * Y + Z * Z)).astype(np.float32)


def torus(n=64, big=18.0, small=7.0):
    X, Y, Z = _grid(n)
    q = np.sqrt(X * X + Y * Y) - big
    return (small - np.sqrt(q * q + Z * Z)).astype(np.float32)


def smooth_random(n=48, seed=0, sigma=2.0):
    """Gaussian-filtered noise: saddle-rich, with many ambiguous faces; the one-voxel border is outside."""
    from scipy.ndimage import gaussian_filter
    g = gaussian_filter(np.random.default_rng(seed).standard_normal((n, n, n)), sigma)
    g = (g / g.std()).astype(np.float32)
    g[[0, -1], :, :] = -1
    g[:, [0, -1], :] = -1
    g[:, :, [0, -1]] = -1
    return g


def on_level_corners(n=40, r=13.0):
    """Sphere distance quantised to 1/2: a large share of lattice corners sit exactly on level 0."""
    return (np.round(sphere(n, r) * 2) / 2).astype(np.float32)


def blob(n=32, seed=0):
    """Seeded sum of Gaussian blobs (level 0.5 crosses it), outside on the border."""
    rng = np.random.default_rng(seed)
    X, Y, Z = _grid(n)
    v = np.zeros_like(X)
    for _ in range(5):
        c = rng.uniform(-n / 5, n / 5, 3)
        s = rng.uniform(n / 10, n / 6)
        v += np.exp(-((X - c[0]) ** 2 + (Y - c[1]) ** 2 + (Z - c[2]) ** 2) / (2 * s * s))
    v[[0, -1], :, :] = 0
    v[:, [0, -1], :] = 0
    v[:, :, [0, -1]] = 0
    return v.astype(np.float32)
