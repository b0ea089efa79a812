"""Golden facts about the UNMODIFIED reference's ``training/triplane.py`` that the drop-in relies on:

    python tests/golden/make_golden_dropin.py <reference checkout>

The reference's generator reaches the renderer, the ray sampler and ``paste_front`` by import name and module
global; this records those names, the constructor and ``paste_front`` signatures, the modules importing it loads and
what a built ``TriPlaneGenerator`` holds, as ``dropin_reference.json``.  Only names, signatures, shapes and the
renderer's plane axes are stored: ``tests/test_dropin_cpu.py`` checks this package against them without the reference tree."""
import inspect
import json
import os
import sys
import types

HERE = os.path.dirname(os.path.abspath(__file__))


def _params(fn):
    return [[p.name, p.kind.name, None if p.default is inspect.Parameter.empty else repr(p.default)]
            for p in inspect.signature(fn).parameters.values()]


def main(ref):
    ref = os.path.abspath(ref)
    os.environ['PROJECT_DN'] = ref
    sys.path[:0] = [ref, ref + '/_train/eg3dc/src']
    sys.modules['kornia'] = types.ModuleType('kornia')            # imported by triplane.py, not used by what is recorded
    import training.triplane as tp
    assert tp.__file__.startswith(ref)
    rk = dict(superresolution_module='training.superresolution.SuperresolutionHybrid8XDC', sr_antialias=True,
              use_triplane=True, c_gen_conditioning_zero=True, decoder_lr_mul=1, box_warp=0.7)
    G = tp.TriPlaneGenerator(z_dim=64, c_dim=25, w_dim=64, img_resolution=512, img_channels=3, rendering_kwargs=rk,
                             cond_mode='none', mapping_kwargs=dict(num_layers=1), channel_base=2048, channel_max=32,
                             sr_kwargs=dict(channel_base=2048, channel_max=32, fused_modconv_default='inference_only'))
    hooks = ('paste_front', 'get_front_occlusion', 'get_front_weights')
    facts = {
        'triplane_imports': {n: getattr(tp, n).__module__ for n in ('ImportanceRenderer', 'RaySampler')},
        'modules_loaded': sorted(m for m in sys.modules if m.startswith(('training.volumetric_rendering.', 'torch_utils.ops.'))),
        'renderer_init': _params(tp.ImportanceRenderer.__init__)[1:],
        'ray_sampler_init': _params(tp.RaySampler.__init__)[1:],
        'generator': {
            'renderer_plane_axes': G.renderer.plane_axes.tolist(),
            'renderer_parameters': sum(p.numel() for p in G.renderer.parameters()),
            'ray_sampler_parameters': sum(p.numel() for p in G.ray_sampler.parameters()),
            'decoder_parameters': {n: list(p.shape) for n, p in G.decoder.named_parameters()},
            'decoder_gains': sorted(a for a in ('weight_gain', 'bias_gain') if hasattr(G.decoder.net[0], a)),
        },
        'f_module_globals': sorted(n for n in hooks if n in tp.TriPlaneGenerator.f.__code__.co_names),
        'hooks': {n: _params(getattr(tp, n)) for n in hooks},
    }
    with open(os.path.join(HERE, 'dropin_reference.json'), 'w') as f:
        f.write('{\n' + ',\n'.join(f' {json.dumps(k)}: {json.dumps(v)}' for k, v in facts.items()) + '\n}\n')
    print(sorted(facts))


if __name__ == '__main__':
    main(sys.argv[1] if len(sys.argv) > 1 else os.environ['PROJECT_DN'])
