"""CPU: the drop-in mechanism.  The reference's own TriPlaneGenerator must pick up this package's renderer / ray sampler
by import name, unchanged."""
import os
import subprocess
import sys
import textwrap

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_install_registers_modules():
    code = textwrap.dedent('''
        import sys
        sys.path.insert(0, %r)
        import panic3d_b200.dropin as d
        names = d.install()
        assert 'training.volumetric_rendering.renderer' in names, names
        import panic3d_b200.training.volumetric_rendering.renderer as ours
        assert sys.modules['training.volumetric_rendering.renderer'] is ours
        print('ok')
    ''' % ROOT)
    r = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True)
    assert r.returncode == 0 and 'ok' in r.stdout, r.stderr[-2000:]


def test_reference_generator_uses_dropin_modules():
    """The reference's TriPlaneGenerator reaches the renderer and ray sampler by import name and ``paste_front`` by module
    global.  tests/golden/dropin_reference.json records those names, the constructor and hook signatures and what a built
    generator holds, from the unmodified reference (tests/golden/make_golden_dropin.py): after install() / install_paste()
    every name resolves to this package, and this package's classes and hooks match what was recorded."""
    code = textwrap.dedent('''
        import importlib, inspect, json, sys, types
        sys.path.insert(0, %(root)r)
        ref = json.load(open(%(golden)r))
        import panic3d_b200.dropin as d
        served = d.install()
        import panic3d_b200.training.volumetric_rendering.renderer as ours_r
        import panic3d_b200.training.volumetric_rendering.ray_sampler as ours_s
        import panic3d_b200.training.triplane as ours_tp
        import panic3d_b200.paste as ours_p
        ours = {'ImportanceRenderer': ours_r.ImportanceRenderer, 'RaySampler': ours_s.RaySampler}
        for name, mod in ref['triplane_imports'].items():            # triplane.py: `from <mod> import <name>`
            assert getattr(importlib.import_module(mod), name) is ours[name], (name, mod)
        # every renderer module the reference loads is served, and every served module is one the reference loads
        assert sorted(m for m in served if m.startswith('training.')) == \\
            [m for m in ref['modules_loaded'] if m.startswith('training.volumetric_rendering.')], served
        assert set(served) <= set(ref['modules_loaded']), served
        params = lambda fn: [[p.name, p.kind.name, None if p.default is inspect.Parameter.empty else repr(p.default)]
                             for p in inspect.signature(fn).parameters.values()]
        assert params(ours_r.ImportanceRenderer.__init__)[1:] == ref['renderer_init']
        assert params(ours_s.RaySampler.__init__)[1:] == ref['ray_sampler_init']
        gen = ref['generator']                                       # built with rendering_kwargs use_triplane=True
        renderer, sampler = ours_r.ImportanceRenderer(use_triplane=True), ours_s.RaySampler()
        assert renderer.plane_axes.tolist() == gen['renderer_plane_axes']
        assert sum(p.numel() for p in renderer.parameters()) == gen['renderer_parameters']
        assert sum(p.numel() for p in sampler.parameters()) == gen['ray_sampler_parameters']
        dec = ours_tp.OSGDecoder(32, {'decoder_lr_mul': 1, 'decoder_output_dim': 32})
        assert {n: list(p.shape) for n, p in dec.named_parameters()} == gen['decoder_parameters']
        assert all(hasattr(dec.net[i], a) for i in (0, 2) for a in gen['decoder_gains'])
        # G.f resolves `paste_front` in its module's globals at call time, so rebinding the module attribute is the whole
        # plug-in: a stand-in `training.triplane` whose f calls the recorded globals
        tp = types.ModuleType('training.triplane')
        for name in ref['hooks']:
            setattr(tp, name, lambda *a, **k: 'reference')
        exec('def f(*a):\\n    return [%%s]\\n' %% ', '.join(n + '(*a)' for n in ref['f_module_globals']), tp.__dict__)
        sys.modules['training.triplane'] = tp
        ref_paste = tp.paste_front
        assert d.install_paste() == list(ref['hooks'])               # finds training.triplane by name
        assert tp.paste_front is ours_p.paste_front and tp._p3d_reference_paste_front is ref_paste
        assert tp.f.__globals__['paste_front'] is ours_p.paste_front and ref['f_module_globals'] == ['paste_front']
        for name, want in ref['hooks'].items():
            assert getattr(tp, name) is getattr(ours_p, name) and params(getattr(ours_p, name)) == want, name
        print('ok')
    ''' % dict(root=ROOT, golden=os.path.join(ROOT, 'tests', 'golden', 'dropin_reference.json')))
    r = subprocess.run([sys.executable, '-c', code], capture_output=True, text=True)
    assert r.returncode == 0 and 'ok' in r.stdout, (r.stdout[-1000:], r.stderr[-3000:])


def test_plane_reuse_memo_runs_backbone_once_per_subject():
    """SURVEY 8f-1: repeated G.f-style calls with the same (ws, cond) hit the memo; changed latents, in-place edits,
    training-mode calls and non-const noise do not."""
    import torch
    from panic3d_b200 import dropin

    class Backbone:
        def __init__(self):
            self.calls = 0

        def synthesis(self, ws, cond, update_emas=False, **kw):
            self.calls += 1
            return ws.sum() + torch.zeros(1, 96, 4, 4) + self.calls

    class G:
        pass
    g = G()
    g.backbone = Backbone()
    memo = dropin.enable_plane_reuse(g)
    assert dropin.enable_plane_reuse(g) is memo                                   # idempotent
    ws = torch.randn(1, 14, 512)
    cond = {'image': torch.randn(1, 3, 8, 8), 'levels': [torch.ones(2), torch.zeros(3)]}
    a = g.backbone.synthesis(ws, cond, update_emas=False, noise_mode='const')
    for _ in range(15):                                                           # the other views of the sweep: fresh, equal ws
        b = g.backbone.synthesis(ws.clone(), {'image': cond['image'].clone(), 'levels': cond['levels']}, update_emas=False, noise_mode='const')
        assert b is a
    assert (memo.misses, memo.hits) == (1, 15)
    ws2 = ws.clone(); ws2[0, 0, 0] += 1
    assert g.backbone.synthesis(ws2, cond, noise_mode='const') is not a           # different subject
    ws2.mul_(2.0)                                                                 # in-place edit of the cached key tensor's twin
    c = g.backbone.synthesis(ws2, cond, noise_mode='const')
    assert memo.misses == 3 and g.backbone.synthesis(ws2, cond, noise_mode='const') is c
    n = memo.misses
    g.backbone.synthesis(ws2, cond, noise_mode='random')                          # stochastic noise: never cached
    g.backbone.synthesis(ws2, cond, update_emas=True, noise_mode='const')
    wsg = ws2.clone().requires_grad_(True)
    g.backbone.synthesis(wsg, cond, noise_mode='const')                           # autograd call (training): bypass
    assert memo.misses == n
    with torch.no_grad():
        assert g.backbone.synthesis(wsg, cond, noise_mode='const') is c           # same values under no_grad: reuse
    big = {'image': torch.randn(1, 3, 256, 256)}                                  # kept by reference + version counter
    d = g.backbone.synthesis(ws2, big, noise_mode='const')
    assert g.backbone.synthesis(ws2, big, noise_mode='const') is d
    big['image'].add_(1.0)                                                        # in-place write -> value compare -> miss
    assert g.backbone.synthesis(ws2, big, noise_mode='const') is not d
    memo.clear()
    assert g.backbone.synthesis(ws2, cond, noise_mode='const') is not c


def test_plane_reuse_memo_noise_mode_of_calls_that_do_not_name_one():
    """G.f / G.synthesis never pass noise_mode (the reference's layers then draw fresh noise per call).  The memo either
    passes an explicit 'const' on (default: deterministic sweep, cached) or, with default_noise_mode=None, leaves the call
    alone and does not cache it - it never replays one random draw for all views."""
    import torch
    from panic3d_b200 import dropin

    class Backbone:
        def __init__(self):
            self.modes = []

        def synthesis(self, ws, cond, update_emas=False, noise_mode='random', **kw):
            self.modes.append(noise_mode)
            return ws.sum() + torch.zeros(1, 96, 4, 4) + len(self.modes)

    class G:
        pass
    ws = torch.randn(1, 14, 512)
    g = G(); g.backbone = Backbone()
    bb = g.backbone
    memo = dropin.enable_plane_reuse(g)
    a = g.backbone.synthesis(ws, None)
    assert g.backbone.synthesis(ws.clone(), None) is a
    assert bb.modes == ['const'] and (memo.misses, memo.hits) == (1, 1)
    g2 = G(); g2.backbone = Backbone()
    bb2 = g2.backbone
    memo2 = dropin.enable_plane_reuse(g2, default_noise_mode=None)
    x = g2.backbone.synthesis(ws, None)
    y = g2.backbone.synthesis(ws, None)
    assert x is not y and bb2.modes == ['random', 'random'] and (memo2.misses, memo2.hits) == (0, 0)
    z = g2.backbone.synthesis(ws, None, noise_mode='const')
    assert g2.backbone.synthesis(ws, None, noise_mode='const') is z and memo2.hits == 1
