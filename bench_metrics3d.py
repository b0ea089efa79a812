"""Eval geometry metrics per subject on one GPU: the 3-D block of _scripts/eval/measure.py:141-201.

    python bench_metrics3d.py [--res 256] [--iters 20] [--warmup 3] [--n-sample 10000]

The predicted mesh is the marching-cubes mesh of the volume query on seeded random tri-planes (the input of
bench_mesh.py: the fixtures' generator, cull_clouds=0.35), in world units; the ground truth is the same mesh moved by
0.005 in z and mapped into the ground-truth frame, so both meshes have the volume-query mesh's size.  The region of
interest is the whole front view.  Reported, CUDA events after warm-up unless stated:
  * BVH build on the predicted mesh (p3d_bvh_build);
  * 10k + 10k queries: n_sample points against each mesh (p3d_point_mesh_distance, the trees prebuilt);
  * the whole measure_geometry on device tensors (host clock around its two synchronisations, median);
  * the same with both meshes passed as numpy arrays (upload included; host clock, median).
There is no reference arm: the reference calls igl.point_mesh_squared_distance / random_points_on_mesh, and igl is not
installed where this runs, so its cost is reported as not measured (the exhaustive-search oracle is a test restatement,
not a stand-in for igl's AABB tree).  Prints one JSON line; writes nothing.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bench_mesh import card, events_ms, host_ms, tri_plane_volume  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--res', type=int, default=256)
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--n-sample', type=int, default=10000)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_metrics3d.py needs a CUDA device')
    import panic3d_b200.mesh as pm
    import panic3d_b200.metrics3d as m3
    query, bw = tri_plane_volume(args.res)
    vol = query()
    m = pm.marching_cubes_device(vol['densities'][0, 0], 0.5)
    dev = m['verts'].device
    pred_v = m['verts'].double() / args.res * bw - 0.5 * bw
    faces = m['faces']
    gt_v = pred_v * torch.tensor([1.0, 1.0, -1.0], dtype=torch.float64, device=dev) + torch.tensor([0.0, 0.0, -0.005], dtype=torch.float64, device=dev)
    roi = ((0, 0), (512, 512))
    mcd = {'verts': pred_v, 'faces': faces}
    mc_np = {'verts': pred_v.cpu().numpy(), 'faces': faces.cpu().numpy()}
    gt_np, faces_np = gt_v.cpu().numpy(), faces.cpu().numpy()
    n = args.n_sample

    # the primitives on the (uncropped) meshes, as measure_geometry calls them
    pv = (pred_v * torch.tensor([-1.0, 1.0, 1.0], dtype=torch.float64, device=dev)).contiguous()
    gv = (gt_v * torch.tensor([-1.0, 1.0, -1.0], dtype=torch.float64, device=dev)).contiguous()
    f32 = faces.to(torch.int32).contiguous()
    status = torch.zeros(1, dtype=torch.int32, device=dev)
    L = m3._lib.lib()
    nf = int(f32.shape[0])
    nbytes = L.p3d_bvh_workspace_bytes(nf)
    bvh_p = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    bvh_g = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    stream = m3._lib.stream_ptr(dev)
    _, _, pts_p = m3._sample(pv, f32, n, 1, 0, None, None, status)
    _, _, pts_g = m3._sample(gv, f32, n, 1, 1, None, None, status)
    outs = [torch.empty(n, dtype=torch.float64, device=dev), torch.empty(n, dtype=torch.int64, device=dev),
            torch.empty((n, 3), dtype=torch.float64, device=dev)]

    def build():
        m3._lib.check(L.p3d_bvh_build(pv.data_ptr(), f32.data_ptr(), nf, bvh_p.data_ptr(), nbytes, stream))

    def build_g():
        m3._lib.check(L.p3d_bvh_build(gv.data_ptr(), f32.data_ptr(), nf, bvh_g.data_ptr(), nbytes, stream))

    def queries():
        for P, V, ws in ((pts_p, gv, bvh_g), (pts_g, pv, bvh_p)):
            m3._lib.check(L.p3d_point_mesh_distance(P.data_ptr(), n, V.data_ptr(), f32.data_ptr(), nf, ws.data_ptr(), nbytes,
                                                    outs[0].data_ptr(), outs[1].data_ptr(), outs[2].data_ptr(), status.data_ptr(), stream))

    def sample():
        m3._sample(pv, f32, n, 1, 0, None, None, status)
        m3._sample(gv, f32, n, 1, 1, None, None, status)

    def device_route():
        return m3.measure_geometry(mcd, gt_v, faces, roi, bw=bw, n_sample=n, seed='daredemoE/fandom_align/bench/0000/front')

    def numpy_route():
        return m3.measure_geometry(mc_np, gt_np, faces_np, roi, bw=bw, n_sample=n, seed='daredemoE/fandom_align/bench/0000/front')

    build_g()
    for fn in (build, queries, sample, device_route, numpy_route):
        for _ in range(args.warmup):
            fn()
    torch.cuda.synchronize()
    assert int(status.item()) == 0
    t_build = events_ms(build, args.iters)
    t_query = events_ms(queries, args.iters)
    t_sample = events_ms(sample, args.iters)
    t_dev = host_ms(device_route, args.iters)
    t_np = host_ms(numpy_route, max(3, args.iters // 2))
    a, b = device_route(), numpy_route()
    assert all(a[k] == b[k] for k in a)
    res = {'bench': 'metrics3d', **card(), 'reference_ms': 'not measured (igl is not installed)',
           'res': args.res, 'faces': nf, 'verts': int(pred_v.shape[0]), 'n_sample': n,
           'bvh_build_ms': round(t_build, 4), 'queries_2x_ms': round(t_query, 4),
           'query_points_per_s': round(2 * n / (t_query * 1e-3), 1), 'sample_2x_ms': round(t_sample, 4),
           'measure_geometry_device_ms': round(t_dev, 3), 'measure_geometry_numpy_ms': round(t_np, 3),
           'cd': float(a['cd']), 'f1_010': float(a['f1_010'])}
    print(json.dumps(res))


if __name__ == '__main__':
    main()
