"""Generate tests/golden/metrics3d_*.npz with the reference's own geometry-metric code (_scripts/eval/measure.py).

    python tests/golden/make_golden_metrics3d.py

Sliced out of the reference by AST line range and executed (the modules' top-level imports need CLIP, LPIPS, pyvista,
igl, ...): ``filter_mesh``, ``get_point_mesh_distance``, ``point_mesh_f1`` and the per-subject 3-D block of the loop in
measure.py; ``sample_points_near_surface`` and ``bary2cart`` of _databacks/lustrous_gltf_v0_measurable.py; ``np_seed``
of _util/util_v1.py.  They run with a stub ``igl`` (not installed here) whose ``random_points_on_mesh`` draws
(face_bits, bary_u) from the numpy stream that ``np_seed(bn)`` seeded and returns oracle/metrics3d_oracle.py's samples
for those bits, and whose ``point_mesh_squared_distance`` is the oracle's exhaustive search; a stub ``pload`` returns the
predicted mesh, a stub ``uvrm`` the ground-truth mesh, and a small ``Dict`` shim stands in for addict.

What the fixtures pin to the reference's code: the x mirror and its float64 promotion, the crop (bounds, dtype of the
comparison, face re-indexing), the ground-truth frame map, ``bary2cart``, and the Chamfer / F1 formulas.  Sample parity
with igl itself is unpinnable (its random stream is its own).  Only outputs are stored; inputs are regenerated.
"""
from __future__ import annotations

import ast
import contextlib
import json
import os
import sys
import textwrap
import threading
import types
import zlib
from collections import defaultdict

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = '/root/reference'
sys.path[:0] = [ROOT]

from oracle import metrics3d_oracle as mo      # noqa: E402
from tests.golden.cases_metrics3d import METRICS3D_CASES, draw_bits, gt_mesh, pred_mc   # noqa: E402


def _source(rel):
    path = os.path.join(REF, rel)
    src = open(path).read()
    return path, src, src.splitlines(keepends=True), ast.parse(src)


def _lines(lines, node):
    start = min([node.lineno] + [d.lineno for d in getattr(node, 'decorator_list', [])])
    return textwrap.dedent(''.join(lines[start - 1:node.end_lineno]))


def _functions(rel, names, ns):
    path, _, lines, tree = _source(rel)
    for node in ast.walk(tree):
        if isinstance(node, ast.FunctionDef) and node.name in names:
            exec(compile(_lines(lines, node), path, 'exec'), ns)
    missing = [n for n in names if n not in ns]
    assert not missing, missing


def _subject_block():
    """The statements of measure.py's per-subject loop from the predicted-mesh load to the end (the 3-D metrics)."""
    path, _, lines, tree = _source('_scripts/eval/measure.py')
    (loop,) = [n for n in tree.body if isinstance(n, ast.For) and ast.unparse(n.target) == 'bn']
    start = [i for i, s in enumerate(loop.body)
             if isinstance(s, ast.Assign) and any(ast.unparse(t) == 'fn_march' for t in s.targets)][0]
    first, last = loop.body[start], loop.body[-1]
    return compile(textwrap.dedent(''.join(lines[first.lineno - 1:last.end_lineno])), path, 'exec')


class Dict(dict):
    __getattr__ = dict.__getitem__


def main():
    block = _subject_block()
    for name, case in METRICS3D_CASES.items():
        mc = pred_mc(case)
        gv, gf = gt_mesh(case)
        drawn = []

        def random_points_on_mesh(n, v, f):
            fb, bu = draw_bits(np.random, n)
            drawn.append((fb, bu))
            B, FI, _ = mo.sample_from_bits(v, f, fb, bu)
            return B, FI

        def point_mesh_squared_distance(P, V, F):
            assert P.dtype == np.float64 and V.dtype == np.float64
            return mo.point_mesh_squared_distance(P, V, F)

        igl = types.SimpleNamespace(random_points_on_mesh=random_points_on_mesh, point_mesh_squared_distance=point_mesh_squared_distance)

        class Head:
            def __init__(self, gltf):
                self.verts, self.faces = gv, gf

        ns = dict(np=np, igl=igl, Dict=Dict, contextlib=contextlib, zlib=zlib, threading=threading,
                  _np_seed_lock=threading.Lock())
        _functions('_util/util_v1.py', ['np_seed'], ns)
        _functions('_databacks/lustrous_gltf_v0_measurable.py', ['bary2cart', 'sample_points_near_surface'], ns)
        _functions('_scripts/eval/measure.py', ['filter_mesh', 'get_point_mesh_distance', 'point_mesh_f1'], ns)
        Head.sample_points_near_surface = staticmethod(ns['sample_points_near_surface'])
        gltf = types.SimpleNamespace(remove_innards=lambda: gltf)
        ns['uvrm'] = types.SimpleNamespace(LustrousGLTF=lambda path: gltf, LustrousGLTFDecapitated=Head)
        ns['pload'] = lambda fn: {'verts': mc['verts'].copy(), 'faces': mc['faces'].copy()}
        ns.update(bn=case['bn'], roi=case['roi'], edn='./temp/eval/fixture', bw=case['bw'], n_sample=case['n_sample'],
                  ans3d=defaultdict(list))
        exec(block, ns)

        p2s, s2p, a3 = ns['p2s'], ns['s2p'], ns['ans3d']
        out = {'p2s': a3['p2s'][-1], 's2p': a3['s2p'][-1], 'cd': a3['cd'][-1]}
        for th in mo.THRESHOLDS:
            r = ns['point_mesh_f1'](p2s, s2p, th)
            key = f'{int(th * 1000):03d}'
            assert r['f1'] == a3[f'f1_{key}']
            out[f'precision_{key}'], out[f'recall_{key}'], out[f'f1_{key}'] = r['precision'], r['recall'], r['f1']
        assert len(drawn) == 2 and all(np.array_equal(drawn[0][k], drawn[1][k]) for k in (0, 1))
        np.savez_compressed(
            os.path.join(HERE, f'metrics3d_{name}.npz'), case=json.dumps(case),
            pred_verts=ns['mesh_pred']['verts'], pred_faces=ns['mesh_pred']['faces'],
            gt_verts=ns['mesh_gt']['verts'], gt_faces=ns['mesh_gt']['faces'],
            points_pred=ns['points_pred'], points_gt=ns['points_gt'], p2s_all=p2s, s2p_all=s2p,
            **{k: np.float64(v) for k, v in out.items()})
        print(f'metrics3d_{name}: pred F={len(ns["mesh_pred"]["faces"])}/{len(mc["faces"])} gt F={len(ns["mesh_gt"]["faces"])}/{len(gf)} '
              f'gt verts {ns["mesh_gt"]["verts"].dtype}; cd={out["cd"]:.6f} f1_010={out["f1_010"]:.4f} f1_050={out["f1_050"]:.4f}')


if __name__ == '__main__':
    main()
