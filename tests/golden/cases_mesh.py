"""Marching-cubes fixture cases (tests/golden/make_golden_mesh.py): inputs are regenerated, never stored."""
from __future__ import annotations

import os

import numpy as np

from tests import mesh_checks as mc

HERE = os.path.dirname(os.path.abspath(__file__))

MESH_CASES = {
    # the reference's own get_eg3d_volume output (the one committed volume that crosses 0.5), sliced as generate.py does
    'vol_crop_cull16': dict(source='volume_vol_crop_cull16', boxwarp=0.7, level=0.5),
    'blob32': dict(source='blob', res=32, seed=5, boxwarp=0.7, level=0.5),
}


def mesh_case_inputs(case):
    """(vol (R,R,R) fp32, rgbs (3,R,R,R) fp32) numpy arrays, as generate.py:98-103 passes them."""
    if case['source'] == 'blob':
        R = case['res']
        vol = mc.blob(R, seed=case['seed'])
        rgbs = np.random.default_rng(case['seed'] + 1).random((3, R, R, R), dtype=np.float32)
        return vol, rgbs
    z = np.load(os.path.join(HERE, case['source'] + '.npz'))
    return z['densities'][0, 0], z['rgbs'][0, :3]
