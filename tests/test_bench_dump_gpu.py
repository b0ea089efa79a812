"""GPU: `bench.py --dump-outputs DIR` writes the last timed step's rays and renderer outputs, and two runs with the same
arguments write identical arrays (the comparison two builds of the project rely on)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SHAPES = {'ray_origins': (8, 16384, 3), 'ray_directions': (8, 16384, 3), 'rgb': (8, 16384, 32), 'depth': (8, 16384, 1),
          'weights_sum': (8, 16384, 1), 'xyz': (8, 16384, 3)}


def _bench(out_dir):
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--gpus', '1', '--steps', '2', '--warmup', '1', '--no-e2e',
                        '--no-variants', '--no-cpu-baseline', '--dump-outputs', str(out_dir)],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    d = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith('{')][-1])
    assert d['steps'] == 2 and d['value'] > 0
    return {f[:-len('.npy')]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


def test_dump_outputs_are_complete_and_repeatable(tmp_path):
    a, b = _bench(tmp_path / 'a'), _bench(tmp_path / 'b')
    assert {k: v.shape for k, v in a.items()} == SHAPES
    assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in a.values())
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert (a['weights_sum'] > 0).any() and a['rgb'].std() > 0
    for k in a:
        assert np.array_equal(a[k], b[k]), k
