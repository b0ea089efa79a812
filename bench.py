#!/usr/bin/env python
"""bench.py - rendered views/sec of the tri-plane volumetric renderer hot path.

Workload (BASELINE.json configs[1]): per GPU a batch of 8 views, 128x128 rays, 96 coarse + 96
importance samples per ray, 8 distinct 3x32x512x512 fp32 tri-planes, OSGDecoder 32->64->33.
A "step" = one pass of the hot path over that batch: layout pre-pass (NCHW -> channels-last
texels) + ray generation + ImportanceRenderer.forward.  Synthetic data, random-init decoder.

    python bench.py [--gpus N] [--steps K] [--warmup W]           our arm (CUDA, one rank per GPU)
    python bench.py [...] --dump-outputs DIR                      also write the last timed step's outputs as DIR/*.npy
    python bench.py --impl reference [...]                        the reference's CPU algorithm (oracle port)

Prints ONE JSON line (rank 0).  See DESIGN.md section "Measurement" for how every field is derived.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'rendered views/sec @128x128 rays x96 samples, 512^2x32ch tri-plane'
UNIT = 'views/s'
R, S, SF, P, C, VIEWS = 128, 96, 96, 512, 32, 8
FLOP_PER_SAMPLE = 2 * 32 * 64 + 2 * 64 * 33            # 8,320 tensor-eligible FLOP (SURVEY 8d)
BYTES_PER_VIEW = 3 * C * P * P * 4 + R * R * 37 * 4    # tri-plane read once + 37 floats/ray out
# dram__bytes_read.sum + dram__bytes_write.sum of ONE launch of the default fused kernel on this workload, from the committed
# `ncu --set full` capture of the default bench command (profiles/r2_final_ws3_raw.csv: 632.8 MB read + 22.6 MB written)
FUSED_TRAFFIC = 655.4e6


# rendering_options of BASELINE configs[1] (train_eclustrousC.py:409-440 + eg3dc_v0.py:30-31,55-56)
RENDER_OPTS = dict(box_warp=0.7, ray_start=0.5, ray_end=1.5, depth_resolution=96, depth_resolution_importance=96,
                   disparity_space_sampling=False, clamp_mode='softplus', white_back=True, triplane_depth=1)


def workload_config(n_gpus, mlp_mode='tc_3xbf16', planes='fp32'):
    return {'workload': f'{VIEWS} views/GPU x {R}x{R} rays x ({S}+{SF}) samples, {VIEWS} distinct 3x{C}x{P}x{P} fp32 tri-planes/GPU',
            'views_per_gpu': VIEWS, 'rays': R * R, 'samples_coarse': S, 'samples_importance': SF, 'plane': P,
            'decoder': '32-64-33 softplus', 'mlp_mode': mlp_mode, 'plane_storage': planes, 'parallelism': f'views sharded x{n_gpus}',
            'l2': 'inputs (805 MB of tri-planes re-laid out every step) exceed the 126 MB L2; no explicit flush'}


def read_peaks():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as f:
            pk = json.load(f)
        return pk['hbm_gbs'], pk.get('bf16_tflops_sustained', pk['bf16_tflops']), 'measured (MEASURED_PEAKS.json, sustained)'
    except Exception:
        return 6650.0, 1400.0, 'fallback (B200_PROFILING.md)'


class ClockSampler:
    """nvidia-smi clocks + throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = 'index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,' \
        'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-lms', '100', '-i', str(self.index)], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
            self.t.join(timeout=5)

    def summary(self):
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        busy = sorted(sm)[len(sm) // 2:]      # upper half = samples under load
        return {'sm_mhz': statistics.median(busy), 'sm_max_mhz': max(mx), 'reasons': sorted(reasons), 'samples': len(sm)}


# --------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's own CPU implementation of the path, on the box's host cores.
#   kind "reference": baseline/_ref holds the UNMODIFIED reference tree (installed by baseline/install_ref.sh in the build
#                     container; git-ignored, shipped to the GPU box) -> its ImportanceRenderer / RaySampler / OSGDecoder are
#                     imported exactly as SURVEY.md section 8c describes and timed on CPU
#   kind "port":      no baseline/_ref -> the oracle restatement (torch CPU, the reference's own ATen op chain)
# One step = ONE view of the 8-view workload (a bounded sample: ~2.4 s of CPU work; the metric is per view).
# --------------------------------------------------------------------------------------------
REF_TREE = os.path.join(ROOT, 'baseline', '_ref')


def _import_reference():
    """-> (ImportanceRenderer, RaySampler, OSGDecoder, camera_params_to_matrix) of the unmodified reference, or None."""
    src = os.path.join(REF_TREE, '_train', 'eg3dc', 'src')
    if not os.path.isdir(os.path.join(src, 'training', 'volumetric_rendering')):
        return None
    from baseline import ref_env
    ref_env.setup()                                                       # PROJECT_DN, sys.path, kornia stub, plugin finder
    try:
        import training.triplane as ref_tp
        from training.volumetric_rendering.renderer import ImportanceRenderer
        from training.volumetric_rendering.ray_sampler import RaySampler
        import _databacks.lustrous_renders_v1 as ref_dk
    except Exception as e:                                                 # a broken install must not look like a fast reference
        print(f'[bench] baseline/_ref present but not importable ({type(e).__name__}: {e}); timing the oracle port', file=sys.stderr)
        return None
    if 'baseline/_ref' not in os.path.abspath(sys.modules[ImportanceRenderer.__module__].__file__).replace(os.sep, '/'):
        return None                                                       # our drop-in modules shadow these names: never time those as "reference"
    return ImportanceRenderer, RaySampler, ref_tp.OSGDecoder, ref_dk.camera_params_to_matrix


def cpu_reference_time(steps, warmup, views=1, cap_s=240.0):
    """Times `views` view(s) of the bench workload per step on the host CPU: the imported reference when baseline/_ref
    exists, else oracle.render (gather='aten').  Stops early once `cap_s` seconds of timed steps have accumulated.
    -> (times, threads, kind)"""
    import torch
    from oracle import renderer_oracle as orc
    g = torch.Generator().manual_seed(0)
    ref = _import_reference()
    opts = dict(RENDER_OPTS)
    planes = torch.randn(views, 3, C, P, P, generator=g)
    w1, w2 = torch.randn(64, C, generator=g), torch.randn(33, 64, generator=g)
    if ref is not None:
        RefRenderer, RefSampler, RefDecoder, ref_cam = ref
        renderer, sampler = RefRenderer(use_triplane=True), RefSampler()
        decoder = RefDecoder(C, {'decoder_lr_mul': 1, 'decoder_output_dim': 32}).requires_grad_(False)
        with torch.no_grad():
            decoder.net[0].weight.copy_(w1); decoder.net[2].weight.copy_(w2)
        labels = torch.stack([ref_cam('eg3d_lustrousB', elev=0.0, azim=-180.0 + 30.0 * i, dist=1.0, fov=30.0)['camera_label'] for i in range(views)])
        c2w, K = labels[:, :16].view(-1, 4, 4), labels[:, 16:25].view(-1, 3, 3)

        def render(res, u_c, u_f):                                        # the reference draws its own jitter (torch.rand_like)
            ro, rd = sampler(c2w, K, res)
            return renderer(planes if res == R else planes[:1], decoder, ro if res == R else ro[:1], rd if res == R else rd[:1], opts)
    else:
        dec = dict(w1=w1, b1=torch.zeros(64), w2=w2, b2=torch.zeros(33), lr_mul=1.0, force_sigmoid=False)
        cams = [orc.camera_params_to_matrix(0.0, -180.0 + 30.0 * i, 1.0, 30.0) for i in range(views)]
        c2w, K = torch.stack([c[0] for c in cams]), torch.stack([c[1] for c in cams])

        def render(res, u_c, u_f):
            ro, rd = orc.ray_sampler(c2w if res == R else c2w[:1], K if res == R else K[:1], res)
            return orc.render(planes if res == R else planes[:1], dec, ro, rd, opts, u_c, u_f, use_triplane=True, gather='aten')
    # torch's CPU ops do not scale to every core of a 100+-core host on tensors this size: probe a
    # quarter-size render at a few thread counts and give the baseline the fastest one.
    ncpu = os.cpu_count() or 1
    cands = sorted({c for c in (ncpu, 64, 32, 16, 8) if c <= ncpu}, reverse=True)
    best = (ncpu, 1e30)
    if len(cands) > 1:
        pu_c, pu_f = torch.rand(1, 64 * 64, S, 1, generator=g), torch.rand(64 * 64, SF, generator=g)
        for c in cands:
            torch.set_num_threads(c)
            with torch.no_grad():
                t0 = time.perf_counter()
                render(64, pu_c, pu_f)
                dt = time.perf_counter() - t0
            if dt < best[1]:
                best = (c, dt)
    torch.set_num_threads(best[0])
    times = []
    with torch.no_grad():
        for i in range(warmup + steps):
            u_c = torch.rand(views, R * R, S, 1, generator=g)
            u_f = torch.rand(views * R * R, SF, generator=g)
            t0 = time.perf_counter()
            render(R, u_c, u_f)
            dt = time.perf_counter() - t0
            if i >= warmup:
                times.append(dt)
                if sum(times) > cap_s:
                    break
    return times, torch.get_num_threads(), ('reference' if ref is not None else 'port')


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    times, cores, kind = cpu_reference_time(steps, warmup, views=1)
    total = sum(times)
    v = len(times) / total
    what = ('the unmodified reference ImportanceRenderer.forward imported from baseline/_ref' if kind == 'reference'
            else 'the oracle port (oracle/renderer_oracle.py, the reference\'s ATen op chain)')
    sample = (f'{what} on the host CPU, {cores} threads; each step = 1 of the workload\'s 8 views (128x128 rays, 96+96 samples, '
              f'512^2 planes; views/s is per view); {len(times)} timed steps after {warmup} warm-up'
              + ('' if len(times) == steps else f' (stopped at the 240 s cap, {steps} requested)'))
    out = {'impl': 'reference', 'metric': METRIC, 'value': v, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': len(times),
           'warmup': warmup, 'ms_per_step': 1e3 * total / len(times), 'higher_is_better': True, 'scaling': 'weak',
           'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic', 'config': workload_config(args.gpus, args.mlp, args.planes),
           'cpu_baseline': {'value': v, 'unit': UNIT, 'cores': cores, 'kind': kind, 'sample': sample},
           'e2e': {'value': v, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}, 'gpu_launches': 0}
    print(json.dumps(out), flush=True)


# --------------------------------------------------------------------------------------------
# our arm
# --------------------------------------------------------------------------------------------
def run_ours(args):
    import ctypes as Ct
    import torch
    import torch.distributed as dist
    import panic3d_b200  # noqa: F401
    from panic3d_b200 import _lib, cameras
    from panic3d_b200.training.volumetric_rendering.renderer import ImportanceRenderer
    from panic3d_b200.training.volumetric_rendering.ray_sampler import RaySampler
    from panic3d_b200.training.triplane import OSGDecoder

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
    L = _lib.lib()

    mlp_mode = {'fp32_simt': 0, 'tc_3xbf16': 1, 'tc_bf16': 2}[args.mlp]
    torch.manual_seed(1234 + rank)
    planes = torch.randn(VIEWS, 3, C, P, P, device=dev)                         # NCHW fp32, as the backbone emits
    decoder = OSGDecoder(C, {'decoder_lr_mul': 1, 'decoder_output_dim': 32}).to(dev).requires_grad_(False)
    spin = cameras.cam60[cameras.camsubs['spin12']]
    labels = torch.stack([cameras.camera_params_to_matrix(elev=float(spin[(rank * VIEWS + i) % 12][0]),
                                                          azim=float(spin[(rank * VIEWS + i) % 12][1]), dist=1.0, fov=30.0)['camera_label']
                          for i in range(VIEWS)])
    labels_dev = labels.to(dev)
    opts = dict(RENDER_OPTS)                     # the GPU arm never touches oracle/ (only cpu_reference_time does)
    renderer, sampler = ImportanceRenderer(use_triplane=True), RaySampler()
    renderer.mlp_mode = mlp_mode
    renderer.planes_bf16 = args.planes == 'bf16'
    # rendered images -> rank 0 (BASELINE configs[3]): peer-to-peer DMA into rank 0's buffer on a side stream (views.PeerGather),
    # overlapped with the next step's render; P3D_BENCH_GATHER=nccl selects the blocking NCCL all-gather of round 1 for A/B
    from panic3d_b200 import views as pviews
    gather_mode = os.environ.get('P3D_BENCH_GATHER', 'p2p') if world > 1 else 'none'
    gather_buf = torch.empty((world * VIEWS, R * R, 32), device=dev) if gather_mode == 'nccl' else None
    peer = pviews.PeerGather((VIEWS, R * R, 32), torch.float32, dev, dst=0) if gather_mode == 'p2p' else None
    step_no = [0]
    last = {}                                                                 # the most recent step's results, for --dump-outputs

    def step():
        c2w, K = labels_dev[:, :16].view(-1, 4, 4), labels_dev[:, 16:25].view(-1, 3, 3)
        ro, rd = sampler(c2w, K, R)
        renderer._planes.key = None                                           # distinct tri-planes every step: redo the layout pass
        rgb, depth, wsum, xyz = renderer(planes, decoder, ro, rd, opts)
        last.update(ray_origins=ro, ray_directions=rd, rgb=rgb, depth=depth, weights_sum=wsum, xyz=xyz)
        if gather_mode == 'nccl':
            dist.all_gather_into_tensor(gather_buf, rgb)
        elif gather_mode == 'p2p':
            peer.push(rgb, step_no[0])
            step_no[0] += 1
        return rgb

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    with torch.no_grad(), ClockSampler(local) as clk:            # nvidia-smi polls through warm-up + timed region
        for _ in range(max(args.warmup, 3)):
            step()
        barrier()
        # ---- timed region: device time (CUDA events on the launching stream), max over ranks
        L.p3d_profile_read(None, None, 0, 1)
        n0 = _lib.launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(args.steps):
            step()
        if peer is not None:
            peer.join_current_stream()                                          # the last image copies are inside the bracket
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        launches = _lib.launch_count() - n0
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, last)
    with torch.no_grad():
        # ---- per-kernel device time for the roofline (separate short run with event brackets enabled)
        L.p3d_profile_enable(1)
        for _ in range(3):
            step()
        torch.cuda.synchronize()
        slot_ms = (Ct.c_double * 8)()
        slot_n = (Ct.c_uint64 * 8)()
        L.p3d_profile_read(slot_ms, slot_n, 8, 1)
        L.p3d_profile_enable(0)
        # ---- the other operating points SURVEY 8(d) asks for, same inputs, 10 device-timed steps each (N=1 only; context for
        #      the headline, not part of it): training-time 48+48 sampling, bf16-stored planes, the single-pass bf16 decoder
        #      and the fp32 SIMT parity kernels
        variants = None
        if world == 1 and not args.no_variants:
            variants = {}
            for name, ov, mm, pb in (('48+48 samples', dict(depth_resolution=48, depth_resolution_importance=48), mlp_mode, renderer.planes_bf16),
                                     ('bf16-stored planes', {}, mlp_mode, True), ('tc_bf16 decoder (1 pass)', {}, 2, renderer.planes_bf16),
                                     ('fp32_simt kernels', {}, 0, renderer.planes_bf16)):
                rv = ImportanceRenderer(use_triplane=True)
                rv.mlp_mode, rv.planes_bf16 = mm, pb
                vo = dict(opts, **ov)

                def vstep():
                    c2w, K = labels_dev[:, :16].view(-1, 4, 4), labels_dev[:, 16:25].view(-1, 3, 3)
                    ro, rd = sampler(c2w, K, R)
                    rv._planes.key = None
                    return rv(planes, decoder, ro, rd, vo)
                for _ in range(3):
                    vstep()
                v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                v0.record()
                for _ in range(10):
                    vstep()
                v1.record()
                torch.cuda.synchronize()
                variants[name] = {'value': round(VIEWS * 10 / (v0.elapsed_time(v1) * 1e-3), 1), 'unit': UNIT, 'steps': 10}
                del rv
        if variants is not None:
            # the tri-planes arrive as a (N,96,H,W) torch.channels_last tensor (what a channels-last backbone emits): the renderer
            # reads them in place - no layout pre-pass, the step moves only the algorithmic bytes
            pl_cl = planes.reshape(VIEWS, 3 * C, P, P).contiguous(memory_format=torch.channels_last).view(VIEWS, 3, C, P, P)
            rv = ImportanceRenderer(use_triplane=True)
            rv.mlp_mode = mlp_mode

            def zstep():
                c2w, K = labels_dev[:, :16].view(-1, 4, 4), labels_dev[:, 16:25].view(-1, 3, 3)
                ro, rd = sampler(c2w, K, R)
                return rv(pl_cl, decoder, ro, rd, opts)
            for _ in range(3):
                zstep()
            v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            v0.record()
            for _ in range(10):
                zstep()
            v1.record()
            torch.cuda.synchronize()
            variants['channels_last tri-planes consumed zero-copy (no layout pre-pass)'] = {'value': round(VIEWS * 10 / (v0.elapsed_time(v1) * 1e-3), 1), 'unit': UNIT, 'steps': 10}
            del rv, pl_cl
            torch.cuda.empty_cache()
            # SURVEY 8(f)-2: the 256^3 sigma/rgb grid of get_eg3d_volume for one subject, one launch (reference: 168 chunks)
            from panic3d_b200 import volume as pvol
            for _ in range(2):
                pvol.query_volume(planes[:1], decoder, opts, resolution=256, triplane_crop=0.1, cull_clouds=0.5, renderer=renderer)
            v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            v0.record()
            for _ in range(3):
                pvol.query_volume(planes[:1], decoder, opts, resolution=256, triplane_crop=0.1, cull_clouds=0.5, renderer=renderer)
            v1.record()
            torch.cuda.synchronize()
            variants['volume query 256^3 (sigma+rgb+density+coords)'] = {'value': round(v0.elapsed_time(v1) / 3, 3), 'unit': 'ms/subject', 'steps': 3}
            torch.cuda.empty_cache()
            # training-path context (BASELINE configs[4] shape: batch_gpu 4, R=64, 48+48, 256^2 planes): forward + backward
            # through the autograd Function (p3d_render_forward / p3d_render_backward), gradients to planes and decoder
            with torch.enable_grad():
                tp = torch.randn(4, 3, C, 256, 256, device=dev, requires_grad=True)
                tdec = OSGDecoder(C, {'decoder_lr_mul': 1, 'decoder_output_dim': 32}).to(dev)
                tro, trd = sampler(labels_dev[:4, :16].view(-1, 4, 4), labels_dev[:4, 16:25].view(-1, 3, 3), 64)
                topts = dict(opts, depth_resolution=48, depth_resolution_importance=48)
                rt = ImportanceRenderer(use_triplane=True)

                def tstep():
                    rgb, depth, wsum, _ = rt(tp, tdec, tro, trd, topts)
                    (rgb.mean() + 0.1 * depth.mean() + 0.1 * wsum.mean()).backward()
                    tp.grad = None
                for _ in range(3):
                    tstep()
                v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                v0.record()
                for _ in range(10):
                    tstep()
                v1.record()
                torch.cuda.synchronize()
                variants['training fwd+bwd (4 views, 64^2 rays, 48+48, 256^2 planes)'] = {'value': round(v0.elapsed_time(v1) / 10, 3), 'unit': 'ms/step', 'steps': 10}
                del tp, tdec, rt
            torch.cuda.empty_cache()
        # ---- the reference's own GPU path beside ours (SURVEY 8d): the UNMODIFIED ImportanceRenderer from baseline/_ref - ~60
        #      eager PyTorch CUDA ops per pass - on this same GPU, same planes / decoder / cameras, one view per call
        #      (its intermediates are ~15 GB per view; views/s is per view)
        if variants is not None:
            ref = _import_reference()
            if ref is not None:
                RefRenderer, RefSampler, RefDecoder, _cam = ref
                rr, rs = RefRenderer(use_triplane=True).to(dev), RefSampler()
                rdec = RefDecoder(C, {'decoder_lr_mul': 1, 'decoder_output_dim': 32}).to(dev).requires_grad_(False)
                rdec.load_state_dict(decoder.state_dict())
                c2w1, K1 = labels_dev[:1, :16].view(-1, 4, 4), labels_dev[:1, 16:25].view(-1, 3, 3)

                def rstep():
                    ro, rd = rs(c2w1, K1, R)
                    return rr(planes[:1], rdec, ro, rd, opts)
                for _ in range(2):
                    rstep()
                v0, v1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                v0.record()
                for _ in range(5):
                    rstep()
                v1.record()
                torch.cuda.synchronize()
                variants['reference renderer (unmodified, eager PyTorch) on this GPU, 1 view/call'] = {
                    'value': round(5 / (v0.elapsed_time(v1) * 1e-3), 2), 'unit': UNIT, 'steps': 5}
                del rr, rdec
                torch.cuda.empty_cache()
        # ---- e2e through the host-buffer C-ABI entry point (pinned host planes in, images out)
        e2e = None
        if not args.no_e2e:
            e2e = run_e2e(L, _lib, planes, decoder, labels, opts, mlp_mode, args, barrier)

    comm_ms = None
    if world > 1:                                                    # the exchange alone (device time, max over ranks), for the `comm` field
        with torch.no_grad():
            rgb_probe = step()
            barrier()
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            for i in range(5):
                if gather_mode == 'nccl':
                    dist.all_gather_into_tensor(gather_buf, rgb_probe)
                else:
                    peer.push(rgb_probe, i)
            if peer is not None:
                peer.join_current_stream()
            c1.record()
            barrier()
            tc = torch.tensor([c0.elapsed_time(c1) / 5], device=dev, dtype=torch.float64)
            dist.all_reduce(tc, op=dist.ReduceOp.MAX)
            comm_ms = float(tc.item())
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    if e2e is not None:
        te = torch.tensor([e2e['ms']], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e['ms'] = float(te.item())
    clocks = clk.summary()

    if rank == 0:
        value = world * VIEWS * args.steps / (ms_max * 1e-3)
        hbm_gbs, tc_tf, peak_src = read_peaks()
        fused = slot_n[5] > 0
        slot = 5 if fused else 0
        kern_ms = slot_ms[slot] / max(1, slot_n[slot])                         # avg duration of ONE launch of the dominant kernel
        samples_per_launch = VIEWS * R * R * (S + SF) / (1 if fused else 2)     # v1: coarse and fine are separate launches
        flops = FLOP_PER_SAMPLE * samples_per_launch
        byts = BYTES_PER_VIEW * VIEWS / (1 if fused else 2)
        t_tensor, t_hbm = flops / (tc_tf * 1e12), byts / (hbm_gbs * 1e9)
        if t_tensor >= t_hbm:
            roof = {'bound': 'tensor', 'achieved': flops / (kern_ms * 1e-3) / 1e12, 'peak': tc_tf, 'unit': 'TFLOP/s'}
        else:
            roof = {'bound': 'hbm', 'achieved': byts / (kern_ms * 1e-3) / 1e9, 'peak': hbm_gbs, 'unit': 'GB/s'}
        # dram__bytes_read.sum + dram__bytes_write.sum of one launch, from the committed `ncu --set full` capture of this
        # command (profiles/r1_final_ws_raw.csv: 630.5 MB + 22.3 MB); only valid for the default kernel / workload
        traffic = FUSED_TRAFFIC if (fused and args.planes == 'fp32' and os.environ.get('P3D_FUSED_IMPL', 'v5') == 'v5') else None
        roof.update({'frac': roof['achieved'] / roof['peak'], 'traffic': traffic,
                     'kernel': ('k_render_ws3' if os.environ.get('P3D_FUSED_IMPL', 'v5') == 'v5' else 'k_render_ws') if fused else 'k_sample_decode',
                     'kernel_ms_per_launch': kern_ms,
                     'launches_timed': int(slot_n[slot]), 'peak_source': peak_src,
                     'step_breakdown_ms': {'sample_decode': slot_ms[0] / 3, 'importance': slot_ms[1] / 3, 'composite': slot_ms[2] / 3,
                                           'layout': slot_ms[3] / 3, 'raygen': slot_ms[4] / 3, 'fused': slot_ms[5] / 3}})
        out = {'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': max(args.warmup, 3),
               'ms_per_step': ms_max / args.steps, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
               'dtype': 'f32', 'data': 'synthetic', 'config': workload_config(world, args.mlp, args.planes), 'clocks': clocks,
               'gpu_launches': int(launches), 'roofline': roof}
        if world > 1:
            out['comm'] = {'mode': gather_mode if (peer is None or peer.p2p) else 'nccl (p2p unavailable on this box)', 'bytes_per_rank_per_step': VIEWS * R * R * 32 * 4, 'ms_per_step': comm_ms,
                           'note': 'rendered feature images -> rank 0; p2p = NVLink DMA on a side stream under the next render'}
        if e2e is not None:
            out['e2e'] = {'value': world * VIEWS * e2e['steps'] / (e2e['ms'] * 1e-3), 'unit': UNIT,
                          'h2d_bytes_per_step': e2e['h2d'], 'd2h_bytes_per_step': e2e['d2h'], 'steps': e2e['steps'],
                          'api': 'p3d_render_forward_host (C-ABI, pinned host buffers)'}
        if variants:
            out['variants'] = variants
        if world == 1 and not args.no_cpu_baseline:
            times, cores, kind = cpu_reference_time(steps=3, warmup=1, views=1)
            out['cpu_baseline'] = {'value': len(times) / sum(times), 'unit': UNIT, 'cores': cores, 'kind': kind,
                                   'sample': f'{len(times)} timed renders of 1 view of the same workload ('
                                             + ('unmodified reference from baseline/_ref' if kind == 'reference' else 'oracle port')
                                             + f', torch CPU, {cores} threads) after 1 warm-up'}
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_e2e(L, _lib, planes, decoder, labels, opts, mlp_mode, args, barrier):
    """Same step through p3d_render_forward_host: NCHW planes, decoder and cameras start in pinned HOST memory,
    results land in pinned host memory; H2D and D2H copies are inside the timed region every step."""
    import ctypes as Ct
    import torch
    p = _lib.RenderParams()
    p.n_views, p.n_rays, p.n_coarse, p.n_fine = VIEWS, R * R, S, SF
    p.channels, p.plane_h, p.plane_w, p.hidden, p.out_dim = C, P, P, 64, 33
    p.box_warp, p.ray_start, p.ray_end = opts['box_warp'], opts['ray_start'], opts['ray_end']
    p.ray_mode, p.disparity, p.white_back, p.plane_mode = 0, 0, 1, 1
    fc1, fc2 = decoder.net[0], decoder.net[2]
    p.w1_gain, p.b1_gain, p.w2_gain, p.b2_gain = float(fc1.weight_gain), float(fc1.bias_gain), float(fc2.weight_gain), float(fc2.bias_gain)
    p.mlp_mode, p.seed = mlp_mode, 7
    p.planes_bf16 = 1 if args.planes == 'bf16' else 0
    h_planes = planes.cpu().pin_memory()
    h_w = [t.detach().cpu().float().contiguous().pin_memory() for t in (fc1.weight, fc1.bias, fc2.weight, fc2.bias)]
    h_c2w = labels[:, :16].contiguous().pin_memory()
    h_K = labels[:, 16:25].contiguous().pin_memory()
    outs = [torch.empty(s, dtype=torch.float32).pin_memory() for s in ((VIEWS, R * R, 32), (VIEWS, R * R), (VIEWS, R * R), (VIEWS, R * R, 3))]

    def call():
        _lib.check(L.p3d_render_forward_host(Ct.byref(p), h_planes.data_ptr(), *[w.data_ptr() for w in h_w], h_c2w.data_ptr(),
                                             h_K.data_ptr(), R, None, None, *[o.data_ptr() for o in outs]))
    for _ in range(2):
        call()
    steps = max(1, min(args.steps, 10))
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        call()                                     # synchronises internally (results are on the host when it returns)
    ms = (time.perf_counter() - t0) * 1e3
    barrier()
    L.p3d_host_arena_release()
    h2d = h_planes.numel() * 4 + sum(w.numel() for w in h_w) * 4 + (h_c2w.numel() + h_K.numel()) * 4
    d2h = sum(o.numel() for o in outs) * 4
    return {'ms': ms, 'steps': steps, 'h2d': h2d, 'd2h': d2h}


def dump_outputs(out_dir, tensors):
    """Write each tensor as out_dir/<name>.npy in float32, whole: the last timed step's rays and the four renderer outputs
    come to 22.5 MB.  The inputs are seeded (tri-planes, decoder, cameras, and the per-call jitter seed drawn from the
    torch CPU generator), so the same command line renders the same step on every build."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in tensors.items():
        np.save(os.path.join(out_dir, name + '.npy'), t.detach().float().cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=100)
    ap.add_argument('--warmup', type=int, default=10)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--mlp', default=os.environ.get('P3D_BENCH_MLP', 'tc_3xbf16'), choices=['fp32_simt', 'tc_3xbf16', 'tc_bf16'])
    ap.add_argument('--planes', default=os.environ.get('P3D_BENCH_PLANES', 'fp32'), choices=['fp32', 'bf16'],
                    help='storage type of the channels-last tri-plane copy the gather reads (bf16 = fast mode, not parity)')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-variants', action='store_true', help='skip the 48+48 / bf16 / fp32_simt context measurements')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write the last timed step\'s ray origins / directions and rgb / depth / '
                         'weights_sum / xyz (rank 0\'s views) as DIR/<name>.npy, float32')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference' and args.dump_outputs:
        ap.error('--dump-outputs writes what the CUDA arm computed; it does not apply to --impl reference')
    if args.impl == 'reference':
        run_reference(args)
    else:
        world = int(os.environ.get('WORLD_SIZE', '1'))
        if world != args.gpus and args.gpus > 1 and world == 1:
            raise SystemExit('--gpus N>1 must be launched with torch.distributed.run (one rank per GPU)')
        run_ours(args)


if __name__ == '__main__':
    main()
