"""CPU: the geometry-metric oracle, run through its restatement of measure.py's per-subject block, equals the fixtures
made by the reference's own code (tests/golden/make_golden_metrics3d.py), bit for bit."""
import os

import numpy as np
import pytest

from oracle import metrics3d_oracle as mo
from tests.golden.cases_metrics3d import METRICS3D_CASES, gt_mesh, injected_bits, pred_mc

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


@pytest.mark.parametrize('name', sorted(METRICS3D_CASES))
def test_metrics3d_oracle_matches_reference_fixture(name):
    case = METRICS3D_CASES[name]
    g = np.load(os.path.join(GOLDEN, f'metrics3d_{name}.npz'))
    mc = pred_mc(case)
    gv, gf = gt_mesh(case)
    bits = injected_bits(case)
    out, arrays = mo.measure_geometry(mc['verts'], mc['faces'], gv, gf, case['roi'], case['bw'], bits, bits)
    for k, v in arrays.items():
        assert v.dtype == g[k].dtype and v.shape == g[k].shape, k
        assert np.array_equal(v, g[k]), k
    for k, v in out.items():
        assert np.float64(v) == g[k], k
    assert str(g['gt_verts'].dtype) == case['gt_dtype']
    assert len(g['pred_faces']) > 100 and len(g['gt_faces']) > 1000
