"""Marching cubes per 256^3 subject on one GPU: the geometry step of _scripts/eval/generate.py:97-105.

    python bench_mesh.py [--res 256] [--iters 20] [--warmup 3]

Two inputs: the volume query on seeded random tri-planes (the test fixtures' generator, triplane_crop=0.1 as generate.py
passes it, cull_clouds=0.35 because generate.py's 0.5 culls these synthetic planes entirely; a noisy surface with many
triangles) and a smooth analytic blob.  For each it reports
  * query_volume + marching_cubes_device per pass, and marching_cubes_device alone (CUDA events after warm-up);
  * cells/s, V and F, and the share of the HBM bound: compulsory bytes (the fp32 volume once, plus the mesh written)
    over the data-sheet 7.7 TB/s, divided by the measured marching-cubes time;
  * the generate.py route: the caller's .cpu().numpy() copies of densities and all rgb channels, then the drop-in
    marching_cubes on numpy, host clock around a synchronise; and the drop-in on the device tensors in place.
There is no reference arm: the reference calls skimage.measure.marching_cubes, which is not installed where this
runs, so its cost is reported as not measured (the CPU oracle is a test restatement, not a stand-in for skimage).
Prints one JSON line; writes nothing.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

HBM_BYTES_PER_S = 7.7e12


def card():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power = (x.strip() for x in q.split(','))
    except Exception:
        name, power = torch.cuda.get_device_name(0), 'not measured'
    return {'gpu': name, 'power_limit': power}


def tri_plane_volume(res):
    """Seeded random tri-planes and decoder of the vol_crop_cull16 fixture case through query_volume at `res`."""
    import panic3d_b200.volume as pv
    from panic3d_b200.training.triplane import OSGDecoder
    from tests.golden.cases import VOLUME_CASES, build_case_inputs
    case = dict(VOLUME_CASES['vol_crop_cull16'], res=res)
    planes, dec, _, _, _, _, opts = build_case_inputs(case)
    d = OSGDecoder(32, {'decoder_lr_mul': dec['lr_mul'], 'decoder_output_dim': 32})
    with torch.no_grad():
        d.net[0].weight.copy_(dec['w1']); d.net[0].bias.copy_(dec['b1'])
        d.net[2].weight.copy_(dec['w2']); d.net[2].bias.copy_(dec['b2'])
    d = d.cuda().requires_grad_(False)
    planes = planes.cuda()

    def run():
        return pv.query_volume(planes, d, opts, resolution=res, triplane_crop=case['triplane_crop'], cull_clouds=case['cull_clouds'],
                               want_coordinates=False)
    return run, opts['box_warp']


def blob_volume(res):
    x = torch.linspace(-1, 1, res, device='cuda')
    X, Y, Z = torch.meshgrid(x, x, x, indexing='ij')
    d = torch.exp(-((X - 0.2) ** 2 + Y ** 2 + Z ** 2) / 0.18) + torch.exp(-((X + 0.35) ** 2 + (Y - 0.1) ** 2 + (Z + 0.2) ** 2) / 0.08)
    dens = d[None, None].contiguous()
    rgb = torch.rand(1, res, res, res, 32, device='cuda').permute(0, 4, 1, 2, 3)   # channels-last like query_volume
    out = {'densities': dens, 'rgbs': rgb}
    return (lambda: out), 0.7


def events_ms(fn, iters):
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(iters):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / iters


def host_ms(fn, iters):
    ts = []
    for _ in range(iters):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return sorted(ts)[len(ts) // 2]


def bench_input(name, make, res, iters, warmup):
    import panic3d_b200.mesh as pm
    query, bw = make(res)
    vol = query()
    dens, rgb = vol['densities'][0, 0], vol['rgbs'][0, :3]

    def mc_only():
        return pm.marching_cubes_device(dens, 0.5, rgb)

    def full():
        v = query()
        return pm.marching_cubes_device(v['densities'][0, 0], 0.5, v['rgbs'][0, :3])

    def generate_route():
        v = query()
        return pm.marching_cubes(v['densities'].cpu().numpy()[0, 0], v['rgbs'].cpu().numpy()[0, :3], bw, level=0.5)

    def in_place_route():
        v = query()
        return pm.marching_cubes(v['densities'][0, 0], v['rgbs'][0, :3], bw, level=0.5)

    for fn in (mc_only, full, generate_route, in_place_route):
        for _ in range(warmup):
            fn()
    m = mc_only()
    V, F = int(m['verts'].shape[0]), int(m['faces'].shape[0])
    t_mc = events_ms(mc_only, iters)
    t_full = events_ms(full, iters)
    t_query = events_ms(query, iters)
    compulsory = 4 * res ** 3 + V * (12 + 12 + 4 + 12) + F * 12
    return {
        'input': name, 'res': res, 'verts': V, 'faces': F,
        'mc_ms': round(t_mc, 4), 'query_ms': round(t_query, 4), 'query_plus_mc_ms': round(t_full, 4),
        'cells_per_s': round((res - 1) ** 3 / (t_mc * 1e-3), 1),
        'compulsory_bytes': compulsory, 'hbm_bound_share': round(compulsory / HBM_BYTES_PER_S / (t_mc * 1e-3), 4),
        'generate_route_ms': round(host_ms(generate_route, max(3, iters // 4)), 2),
        'in_place_dropin_ms': round(host_ms(in_place_route, max(3, iters // 4)), 2),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--res', type=int, default=256)
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('bench_mesh.py needs a CUDA device')
    import panic3d_b200  # noqa: F401
    res = {'bench': 'marching_cubes', **card(), 'reference_ms': 'not measured (skimage is not installed)',
           'inputs': [bench_input('tri_planes', tri_plane_volume, args.res, args.iters, args.warmup),
                      bench_input('blob', blob_volume, args.res, args.iters, args.warmup)]}
    print(json.dumps(res))


if __name__ == '__main__':
    main()
