"""CPU: the marching-cubes oracle put through the drop-in post-processing equals the fixtures made by the reference's
own ``marching_cubes`` (tests/golden/make_golden_mesh.py), bit for bit."""
import os

import numpy as np
import pytest

from oracle import mesh_oracle as mo
from tests.golden.cases_mesh import MESH_CASES, mesh_case_inputs

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


@pytest.mark.parametrize('name', sorted(MESH_CASES))
def test_mesh_oracle_matches_reference_fixture(name):
    case = MESH_CASES[name]
    g = np.load(os.path.join(GOLDEN, f'mesh_{name}.npz'))
    vol, rgbs = mesh_case_inputs(case)
    out = mo.postprocess(*mo.marching_cubes(vol, case['level']), rgbs, case['boxwarp'], vol.shape[-1])
    for k in ('verts', 'faces', 'normals', 'values', 'colors'):
        assert out[k].dtype == g[k].dtype and out[k].shape == g[k].shape, k
        assert np.array_equal(out[k], g[k]), k
    assert len(g['faces']) > 1000
