"""The drop-in seam itself (SURVEY.md section 8b, B1): ``nerf_from_image_b200.render.render``
and ``ParallelModel`` called exactly as run.py calls the reference's.

Everything ``render`` does on the host is exercised for real -- the generator front-end call,
lifting planes / palette / decoder weights out of the ``sampler`` closure (``extract_field``,
no-copy plane join), the two random draws in the reference's order, flag and extra-output
handling -- and only the CUDA core (``fused_render``) is stood in for by the CPU oracle (test
infrastructure).  ``target_model`` is tests/helpers_dropin.py's stand-in for the reference's
``Generator``, loaded with the same scene; what the reference's ``render`` returned for it with
the same seed, and the generator's front-end results, are recorded in
tests/golden/reference/render_dropin.npz (tests/golden/make_golden_reference.py).
"""
import os
import types

import numpy as np
import pytest
import torch

from nerf_from_image_b200 import _lib
from nerf_from_image_b200 import render as R
from oracle import render_oracle as O
from tests import helpers as Hh
from tests import helpers_dropin as HD

H, W, S = 10, 14, 8


def oracle_core(calls):
    """Stand-in for fused.fused_render with the same signature, on the CPU oracle."""
    def core(planes, w1, b1, w2, b2, palette, beta, alpha, c2w, focal, center, bbox, cfg,
             height, width, num_samples, noise_t=None, noise_u=None, extra_mode=0,
             cam_grad=True, compute_normals=False, out=None, planes_layout='channel_first',
             view=None):
        assert planes_layout == 'channel_first'   # the reference Generator's own planes
        calls.append(dict(planes=planes, cfg=cfg, extra_mode=extra_mode, cam_grad=cam_grad,
                          noise_t=noise_t, noise_u=noise_u, view=view))
        vkw = dict(view_features=view[0], w3=view[1], b3=view[2]) if view is not None else {}
        o = O.render_oracle(planes, w1, b1, w2, b2, palette, beta, alpha, c2w, focal, center,
                            bbox, height, width, num_samples, noise_t, noise_u,
                            scene_range=cfg.scene_range, white_background=cfg.white_background,
                            use_sdf=cfg.use_sdf, fine_sampling=cfg.fine_sampling,
                            compute_normals=compute_normals,
                            compute_semantics=extra_mode == _lib.EXTRA_SEMANTICS,
                            compute_coords=extra_mode == _lib.EXTRA_COORDS,
                            force_no_cam_grad=not cam_grad, **vkw)
        extra = o['semantics'] if extra_mode != _lib.EXTRA_NONE else None
        res = (o['rgb'], o['depth'], o['mask'], extra)
        return res + ((o['normals'],) if compute_normals else ())
    return core


def scene_of(case, A=10, viewdir=False):
    scene, cams = Hh.make_case(case, seed=21, batch=2, plane_res=16, attention_values=A)
    if viewdir:
        from fixtures import synthetic
        scene = synthetic.add_view_mapper(scene)
    return scene, cams


def recorded(key):
    return Hh.reference_golden('render_dropin', key)


def setup(monkeypatch, case='p3d_bbox', A=10, use_sdf=True, fine=True, viewdir=False):
    scene, cams = scene_of(case, A, viewdir)
    g = HD.SceneGenerator(scene, use_sdf=use_sdf)
    calls = []
    monkeypatch.setattr(R, 'fused_render', oracle_core(calls))
    R.configure(types.SimpleNamespace(use_viewdir=viewdir, use_sdf=use_sdf, attention_values=A,
                                      fine_sampling=fine),
                {'scene_range': scene['scene_range'],
                 'white_background': scene['white_background']})
    ws = torch.zeros(2, 15 if A > 0 else 14, 512)
    extra_in = {'attention_values': scene['palette']} if A > 0 else {}
    return scene, cams, g, ws, extra_in, calls


RETURNS_CASES = [
    ('p3d_bbox', {}),
    ('cub_ortho', {}),
    ('chairs_white_center', {}),
    ('p3d_bbox', dict(randomize=False)),
    ('p3d_plain', dict(compute_semantics=True)),
    ('p3d_plain', dict(compute_coords=True, compute_semantics=True)),  # coords win, run.py:337
    ('p3d_plain', dict(compute_normals=True)),
    ('p3d_plain', dict(force_no_cam_grad=True)),
    # --use_viewdir (CARLA; run.py:216-221): the model is called with the unit view directions
    ('chairs_white_center', dict(viewdir=True)),
    ('p3d_bbox', dict(viewdir=True, compute_semantics=True)),
    ('cub_ortho', dict(viewdir=True, force_no_cam_grad=True)),
]


def returns_key(case, kw):
    return 'returns_%s_%s' % (case, '_'.join('%s=%s' % i for i in sorted(kw.items())) or 'default')


@pytest.mark.parametrize('case,kw', RETURNS_CASES)
def test_render_returns_what_the_reference_returns(monkeypatch, case, kw):
    ref = recorded(returns_key(case, kw))
    kw = dict(kw)
    scene, cams, g, ws, extra_in, calls = setup(monkeypatch, case, viewdir=kw.pop('viewdir', False))
    ref_kw = dict(kw)
    randomize = ref_kw.pop('randomize', True)
    torch.manual_seed(33)
    got = R.render(g, H, W, cams['c2w'], cams['focal'], cams['center'], cams['bbox'], ws, S,
                   randomize=randomize, extra_model_inputs=extra_in, **ref_kw)
    # both consumed the default generator identically: the next draw agrees
    assert torch.equal(torch.rand(3), ref['next'])
    assert len(got) == 6
    for i, name in enumerate(('rgb', 'depth', 'mask', 'normals', 'extra')):
        assert (got[i] is None) == (name not in ref), name
        if name in ref:
            assert got[i].shape == ref[name].shape, name
            assert (got[i] - ref[name]).abs().max().item() < (1e-4 if name == 'normals' else 2e-5), name
    assert got[5] == {}
    (call,) = calls
    assert call['cam_grad'] == (not kw.get('force_no_cam_grad', False))
    assert (call['noise_t'] is None) == (not randomize)
    if 'view_mapper' in scene:
        vf, w3, b3 = call['view']
        assert vf.shape == (2, H, W, 32)
        assert torch.allclose(w3, scene['w3'], rtol=1e-6, atol=0) and torch.allclose(b3, scene['b3'], rtol=1e-6, atol=0)
        # the view directions reach the mapper attached to the cameras unless force_no_cam_grad
        assert vf.requires_grad  # (the mapper's parameters; the cameras unless force_no_cam_grad)


def test_viewdir_gradients_reach_the_mapper_and_the_cameras(monkeypatch):
    """--use_viewdir: d rgb / d(ViewDirectionMapper parameters) and the camera gradient THROUGH the
    view directions agree with the reference's autograd (the per-ray trunk stays under autograd;
    the kernel returns d/d view_features, d/d w3, d/d b3)."""
    want = recorded('viewdir_grads')
    scene, cams, g, ws, extra_in, calls = setup(monkeypatch, 'p3d_plain', viewdir=True)
    cam = dict(cams, c2w=cams['c2w'].clone().requires_grad_())
    vm = g.viewdir_mapper
    leaves = [cam['c2w'], vm.fc0.weight, vm.fc3.weight, vm.norm2.bias, vm.output.weight, vm.output.bias]
    torch.manual_seed(4)
    got = R.render(g, H, W, cam['c2w'], cam['focal'], cam['center'], cam['bbox'], ws, S,
                   extra_model_inputs=extra_in)
    have = torch.autograd.grad(got[0].square().sum() + got[2].sum(), leaves)
    for i, a in enumerate(have):
        assert Hh.rel_l2(a, want['grad%d' % i]) < 1e-4


def test_stand_in_closes_over_what_the_generator_closes_over():
    """extract_field / extract_view read the sampler closure's and the mapper closure's free
    variables by name: the stand-in's are among those of the original Generator's closures
    (recorded) and include every name render() reads."""
    z = np.load(os.path.join(Hh.REFERENCE_GOLDEN, 'render_dropin.npz'))
    scene, _ = scene_of('p3d_plain', viewdir=True)
    d = torch.nn.functional.normalize(torch.randn(2, 4, 4, 1, 3), dim=-1)
    sampler = HD.SceneGenerator(scene)(d, torch.zeros(2, 15, 512), ['sampler'],
                                       {'attention_values': scene['palette']})['sampler']
    read = {'xy', 'xz', 'yz', 'attention_values', 'viewdir_mapper_closure'}
    assert read <= set(sampler.__code__.co_freevars) <= set(map(str, z['sampler_freevars']))
    mapper = R._closure_vars(sampler)['viewdir_mapper_closure']
    assert {'x'} <= set(mapper.__code__.co_freevars) <= set(map(str, z['mapper_freevars']))


def test_planes_are_lifted_without_a_copy(monkeypatch):
    scene, cams, g, ws, extra_in, calls = setup(monkeypatch)
    R.render(g, H, W, cams['c2w'], cams['focal'], None, cams['bbox'], ws, S,
             extra_model_inputs=extra_in)
    planes = calls[0]['planes']
    assert planes.shape == (2, 3, 32, 16, 16)
    assert planes.data_ptr() == g.synthesis_network.planes.data_ptr()  # a view of the synthesis output


VARIANT_CASES = ((0, True, True), (10, False, True), (10, True, False))


def variant_key(A, use_sdf, fine):
    return 'variants_A%d_sdf%d_fine%d' % (A, int(use_sdf), int(fine))


def test_variants_and_model_outputs(monkeypatch):
    # direct colours (A = 0), density model, no fine pass, and an extra model output
    for A, use_sdf, fine in VARIANT_CASES:
        ref = recorded(variant_key(A, use_sdf, fine))
        scene, cams, g, ws, extra_in, calls = setup(monkeypatch, 'p3d_plain', A, use_sdf, fine)
        torch.manual_seed(5)
        got = R.render(g, H, W, cams['c2w'], cams['focal'], None, None, ws, S,
                       extra_model_inputs=extra_in)
        for a, k in zip(got[:3], ('rgb', 'depth', 'mask')):
            assert (a - ref[k]).abs().max().item() < 2e-5
        assert calls[0]['cfg'].attention_values == A and calls[0]['cfg'].use_sdf == use_sdf
        assert (calls[0]['noise_u'] is None) == (not fine)
    scene, cams, g, ws, extra_in, calls = setup(monkeypatch)
    out = R.render(g, H, W, cams['c2w'], cams['focal'], None, None, ws, S,
                   extra_model_outputs=['attention_values'], extra_model_inputs=extra_in)
    assert list(out[5]) == ['attention_values']          # 'sampler' is not leaked to the caller
    assert torch.equal(out[5]['attention_values'], scene['palette'])


def test_error_behaviour(monkeypatch):
    scene, cams, g, ws, extra_in, calls = setup(monkeypatch)
    a = (g, H, W, cams['c2w'], cams['focal'], None, None, ws, S)
    R.args.use_viewdir = True                             # model built without use_viewdir
    with pytest.raises(_lib.NfiError):
        R.render(*a, extra_model_inputs=extra_in)
    R.args.use_viewdir = False
    R.args.attention_values = 0
    with pytest.raises(AssertionError):                   # run.py:232
        R.render(*a, compute_semantics=True, extra_model_inputs=extra_in)
    R.args.attention_values = 10
    R.args.use_sdf = False
    with pytest.raises(AssertionError):                   # run.py:229
        R.render(*a, compute_normals=True, extra_model_inputs=extra_in)
    with pytest.raises(AttributeError):
        R.configure({'use_sdf': True}, {'scene_range': 1.0, 'white_background': False})
    with pytest.raises(KeyError):
        R.configure(dict(use_viewdir=False, use_sdf=True, attention_values=10,
                         fine_sampling=True), {'scene_range': 1.0})

    class NoPlanes(torch.nn.Module):
        def forward(self, *a, **k):
            return {'sampler': lambda x: x}
    with pytest.raises(_lib.NfiError):
        R.configure(dict(use_viewdir=False, use_sdf=True, attention_values=10,
                         fine_sampling=True), {'scene_range': 1.0, 'white_background': False})
        R.render(NoPlanes(), H, W, cams['c2w'], cams['focal'], None, None, ws, S)


def test_parallel_model_forward(monkeypatch):
    scene, cams, g, ws, extra_in, calls = setup(monkeypatch)
    pm = R.ParallelModel(H, model=g, model_ema=g)
    R.depth_samples_per_ray = S
    torch.manual_seed(8)
    out = pm(cams['c2w'], cams['focal'], None, cams['bbox'], ws, use_ema=True,
             extra_model_inputs=extra_in)
    ref = recorded('parallel')
    assert out[0].shape == (2, H, H, 3)
    assert (out[0] - ref['rgb']).abs().max().item() < 2e-5
    # closure form (run.py:612-615): called with (self, rgb, mask, extra, model_outputs, **params)
    seen = {}
    def closure(self_, rgb, mask, extra, model_outputs, tag):
        seen.update(tag=tag, rgb=rgb, mask=mask)
        return 'closed'
    assert pm(cams['c2w'], cams['focal'], None, cams['bbox'], ws, closure=closure,
              closure_params={'tag': 7}, extra_model_inputs=extra_in) == 'closed'
    assert seen['tag'] == 7 and seen['rgb'].shape == (2, H, H, 3)
    # res / ray multipliers (run.py:600-603)
    pm(cams['c2w'], cams['focal'], None, cams['bbox'], ws, res_multiplier=0.5, ray_multiplier=2,
       extra_model_inputs=extra_in)
    assert calls[-1]['noise_t'].shape == (2, H // 2, H // 2, 2 * S)


def front_end_inputs(z, w_full):
    return (('z', z), ('w1', w_full[:, :1].contiguous()), ('w', w_full))


def palette_bias():
    return torch.randn(2, 10, 3, generator=torch.Generator().manual_seed(6))


def test_front_end_latent_handling_matches_the_generator():
    """generator.resolve_ws / resolve_palette (the host logic of both sm_100a front-ends) feed
    the synthesis network and the palette exactly what Generator.forward fed them
    (models/generator.py:423-468, recorded with its real mapping network and texture mapper), for
    z, a single broadcast w and a complete w."""
    from nerf_from_image_b200 import generator as G
    rec = recorded('front_end')
    torch.manual_seed(2)
    z = torch.randn(2, 512)
    g = HD.RecordedFrontEnd(rec, z)
    for name, c in front_end_inputs(z, rec['w_full']):
        w2, batch = G.resolve_ws(g, c)
        pal, w_syn = G.resolve_palette(g, w2, ['sampler'], {})
        assert batch == 2
        assert torch.equal(w_syn, rec[name + '_ws'])
        assert torch.equal(pal, rec[name + '_attention_values'])
    bias = palette_bias()
    pal, _ = G.resolve_palette(g, rec['w_full'], ['sampler'], {'attention_values_bias': bias})
    assert torch.equal(pal, rec['bias_attention_values'])
    assert G.FusedGeneratorFront.supports(['sampler'], {}) is False          # grad mode on
    with torch.no_grad():
        assert G.FusedGeneratorFront.supports(['sampler', 'attention_values'], {})
        assert not G.FusedGeneratorFront.supports(['sampler', 'sdf_eikonal_loss'], {})
    assert G.HeadsGeneratorFront.supports(['sampler', 'entropy_loss', 'path_length'], {})
    assert not G.HeadsGeneratorFront.supports(['sampler'], {})
