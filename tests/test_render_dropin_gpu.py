"""The drop-in seam on hardware: ``render()`` / ``ParallelModel`` with the reference's REAL
``Generator`` (mapping + texture mapper + the full StyleGAN2 synthesis network, random init,
seeded) on CUDA, against the UNMODIFIED reference ``render`` (run.py:176-350, lifted by AST)
running eagerly in fp32 on the same GPU from the same seed.

The original project's files are staged, unmodified, into the git-ignored ``oracle/_ref/`` by
``__graft_entry__.build()`` when NFI_REFERENCE_ROOT names a checkout of it; without them these
tests skip and say so.

What this pins that the CPU seam test (tests/test_render_dropin.py, CUDA core stood in for
by the oracle) cannot: closure introspection on CUDA tensors, the no-copy plane join, the
fused kernels behind the real front-end, and that both consume the CUDA default generator
identically (``torch.rand_like`` inside TorchScript vs ``torch.rand`` here).
"""
import types

import pytest
import torch

from oracle import reference_lift as RL

pytestmark = [pytest.mark.gpu,
              pytest.mark.skipif(not RL.available(),
                                 reason='original project not staged (oracle/_ref)')]

H = W = 32
S = 16


def _rel(a, b):
    return ((a - b).norm() / b.norm().clamp_min(1e-12)).item()


def _setup(dataset='p3d_car', A=10, B=2, seed=1234, use_viewdir=False):
    from nerf_from_image_b200 import render as R
    from fixtures import synthetic
    torch.backends.cuda.matmul.allow_tf32 = False   # run.py:59-60
    torch.backends.cudnn.allow_tf32 = False
    _, generator = RL._import_reference()
    cfg = synthetic.DATASET_CONFIGS[dataset]
    torch.manual_seed(seed)                        # the reference's own seed, run.py:413
    g = generator.Generator(512, cfg['scene_range'], attention_values=A, use_sdf=True,
                            disable_stylegan_noise=True, use_viewdir=use_viewdir).cuda().eval()
    g.requires_grad_(False)                        # inversion setting, run.py:628-629
    with torch.no_grad():                          # the random-init SDF head is ~ N(1.13, 0.27):
        g.decoder.net[2].bias[0] = -1.15           # shift it so it crosses zero (mask ~ 0.5-0.6)
        if use_viewdir:                            # the mapper's output layer starts at zero
            g.viewdir_mapper.output.weight.normal_()   # (generator.py:217-218): make it matter
            g.viewdir_mapper.output.bias.normal_(0, 0.1)
    cams = synthetic.make_cameras(seed, B, ortho=cfg['ortho'], radius=cfg['radius'],
                                  with_bbox=not cfg['ortho'], device='cuda')
    z = torch.randn(B, 512, device='cuda')
    with torch.no_grad():
        ws = g.mapping_network(z, None)
    args = types.SimpleNamespace(use_viewdir=use_viewdir, use_sdf=True, attention_values=A,
                                 fine_sampling=True)
    dcfg = {'scene_range': cfg['scene_range'], 'white_background': cfg['white_background']}
    R.configure(args, dcfg)
    ref_render = RL.lift_render(cfg['scene_range'], cfg['white_background'], use_sdf=True,
                                attention_values=A, fine_sampling=True, use_viewdir=use_viewdir)
    return R, g, cams, ws, ref_render


@pytest.mark.parametrize('dataset', ['p3d_car', 'cub'])
@pytest.mark.parametrize('kw', [{}, dict(compute_coords=True), dict(force_no_cam_grad=True)])
def test_render_equals_the_reference_on_cuda(cuda_lib, dataset, kw):
    R, g, cams, ws, ref_render = _setup(dataset)
    a = (g, H, W, cams['c2w'], cams['focal'], cams['center'], cams['bbox'], ws, S)
    with torch.no_grad():
        torch.manual_seed(77)
        ref = ref_render(*a, **kw)
        state_ref = torch.cuda.get_rng_state()
        torch.manual_seed(77)
        got = R.render(*a, **kw)
        state_got = torch.cuda.get_rng_state()
    assert len(got) == len(ref) == 6
    assert 0.02 < ref[2].mean().item() < 0.98, 'degenerate fixture: mask %.3f' % ref[2].mean().item()
    for i, name in enumerate(('rgb', 'depth', 'mask', 'normals', 'extra')):
        assert (got[i] is None) == (ref[i] is None), name
        if ref[i] is not None:
            assert got[i].shape == ref[i].shape and got[i].device == ref[i].device, name
            assert _rel(got[i], ref[i]) < 1e-3, (name, _rel(got[i], ref[i]))
    assert torch.equal(state_ref, state_got), 'RNG consumption differs from the reference'


@pytest.mark.parametrize('kw', [{}, dict(compute_semantics=True), dict(force_no_cam_grad=True)])
def test_render_with_viewdir_equals_the_reference_on_cuda(cuda_lib, kw):
    """--use_viewdir (the CARLA models, run.py:216-221): the reference Generator built with
    use_viewdir=True, called with the unit view directions, its ViewDirectionMapper's per-sample
    closure evaluated inside the fused kernels."""
    R, g, cams, ws, ref_render = _setup('p3d_car', use_viewdir=True)
    a = (g, H, W, cams['c2w'], cams['focal'], cams['center'], cams['bbox'], ws, S)
    with torch.no_grad():
        torch.manual_seed(77)
        ref = ref_render(*a, **kw)
        state_ref = torch.cuda.get_rng_state()
        torch.manual_seed(77)
        got = R.render(*a, **kw)
        state_got = torch.cuda.get_rng_state()
    for i, name in enumerate(('rgb', 'depth', 'mask', 'normals', 'extra')):
        assert (got[i] is None) == (ref[i] is None), name
        if ref[i] is not None:
            assert _rel(got[i], ref[i]) < 1e-3, (name, _rel(got[i], ref[i]))
    assert torch.equal(state_ref, state_got), 'RNG consumption differs from the reference'
    # and the pose gradient, which now also flows through the view directions
    grads = []
    for fn in (ref_render, R.render):
        c2w = cams['c2w'].clone().requires_grad_()
        torch.manual_seed(5)
        out = fn(g, H, W, c2w, cams['focal'], None, cams['bbox'], ws, S)
        grads.append(torch.autograd.grad(out[0].square().mean() + out[2].mean(), [c2w])[0])
    assert _rel(grads[1], grads[0]) < 5e-3


def test_viewdir_with_the_fused_front_ends(cuda_lib):
    """--use_viewdir together with enable_fused_synthesis (planes from the tcgen05 synthesis
    kernels, mapper trunk by the reference module) and enable_fused_heads (regulariser outputs)."""
    R, g, cams, ws, ref_render = _setup('p3d_car', use_viewdir=True)
    a = (g, H, W, cams['c2w'], cams['focal'], cams['center'], cams['bbox'], ws, S)
    try:
        R.enable_fused_synthesis(g)
        with torch.no_grad():
            torch.manual_seed(31)
            ref = ref_render(*a)
            torch.manual_seed(31)
            got = R.render(*a)
        assert _rel(got[0], ref[0]) < 2e-3 and _rel(got[2], ref[2]) < 2e-3   # bf16-pair synthesis
        R.enable_fused_heads(g)
        g.train()                                   # generator.py:517: the eikonal head is a training loss
        heads = ['sdf_eikonal_loss', 'entropy_loss']
        torch.manual_seed(32)
        ref = ref_render(*a, extra_model_outputs=heads)
        torch.manual_seed(32)
        got = R.render(*a, extra_model_outputs=heads)
        assert _rel(got[0], ref[0]) < 1e-3
        for k in heads:
            assert _rel(got[5][k], ref[5][k]) < 1e-3, k
    finally:
        g.eval()
        R.enable_fused_synthesis(g, False)
        R.enable_fused_heads(g, False)


def test_inversion_gradients_flow_to_the_latents_like_the_reference(cuda_lib):
    """One inversion-style step (run.py:2256-2317): loss on rgb and mask, gradients w.r.t. the
    per-image latents (through the reference's synthesis autograd on both sides) and the pose."""
    R, g, cams, ws, ref_render = _setup('p3d_car')
    grads = []
    for fn in (ref_render, R.render):
        w = ws.clone().requires_grad_()
        c2w = cams['c2w'].clone().requires_grad_()
        focal = cams['focal'].clone().requires_grad_()
        torch.manual_seed(5)
        out = fn(g, H, W, c2w, focal, None, cams['bbox'], w, S)
        loss = out[0].square().mean() + (out[2] - 0.5).square().mean()
        grads.append(torch.autograd.grad(loss, [w, c2w, focal]))
    for n, a, b in zip(('ws', 'c2w', 'focal'), grads[1], grads[0]):
        assert b.abs().sum() > 0, n
        assert _rel(a, b) < 5e-3, (n, _rel(a, b))


def test_parallel_model_on_cuda(cuda_lib):
    R, g, cams, ws, ref_render = _setup('p3d_car')
    pm = R.ParallelModel(H, model=g, model_ema=g)
    R.depth_samples_per_ray = S
    with torch.no_grad():
        torch.manual_seed(9)
        out = pm(cams['c2w'], cams['focal'], None, cams['bbox'], ws, use_ema=True)
        torch.manual_seed(9)
        ref = ref_render(g, H, W, cams['c2w'], cams['focal'], None, cams['bbox'], ws, S)
    assert _rel(out[0], ref[0]) < 1e-3 and _rel(out[2], ref[2]) < 1e-3
    # the planes handed to the kernels are a VIEW of the synthesis output (no stack copy)
    from nerf_from_image_b200.render import _closure_vars, _join_planes
    mo = g(None, ws, ['sampler'], {})
    cv = _closure_vars(mo['sampler'])
    joined = _join_planes(cv['xy'], cv['xz'], cv['yz'])
    assert joined.data_ptr() == cv['xy'].data_ptr() and joined.shape[1:3] == (3, 32)


@pytest.mark.parametrize('input_kind', ['ws', 'z', 'w1'])
def test_render_with_the_fused_plane_producer(cuda_lib, input_kind):
    """w (or z) -> image entirely on the sm_100a kernels: ``enable_fused_synthesis`` routes the
    no_grad calls through generator.FusedGeneratorFront (synthesis network on tcgen05, planes
    channel-last into the render kernels); the reference render, eager fp32, is the yardstick."""
    R, g, cams, ws, ref_render = _setup('p3d_car')
    model_input = {'ws': ws, 'z': torch.randn(ws.shape[0], 512, device='cuda'),
                   'w1': ws[:, :1].contiguous()}[input_kind]
    a = (g, H, W, cams['c2w'], cams['focal'], None, cams['bbox'], model_input, S)
    R.enable_fused_synthesis(g)
    try:
        with torch.no_grad():
            torch.manual_seed(21)
            ref = ref_render(*a, extra_model_outputs=['attention_values'])
            s_ref = torch.cuda.get_rng_state()
            torch.manual_seed(21)
            got = R.render(*a, extra_model_outputs=['attention_values'])
            s_got = torch.cuda.get_rng_state()
        assert torch.equal(s_ref, s_got)
        for i in (0, 1, 2):
            assert _rel(got[i], ref[i]) < 1e-3, (i, _rel(got[i], ref[i]))
        assert torch.equal(got[5]['attention_values'], ref[5]['attention_values'])
        # a call that needs autograd through the synthesis network keeps the reference module
        w = ws.clone().requires_grad_()
        out = R.render(g, H, W, cams['c2w'], cams['focal'], None, cams['bbox'], w, S)
        out[0].mean().backward()
        assert w.grad is not None and w.grad.abs().sum() > 0
    finally:
        R.enable_fused_synthesis(g, False)


def test_regulariser_outputs_through_render(cuda_lib):
    """A GAN generator-step style call (run.py:1007-1044): render + the regulariser entries of
    ``model_outputs``, gradients to the latents and the decoder.  With ``enable_fused_heads`` the
    entries come from the fused point evaluator; the reference computes them with the unfused
    decoder and a double backward."""
    R, g, cams, ws, ref_render = _setup('p3d_car')
    g.requires_grad_(True)
    g.train()                                            # the eikonal head asserts self.training
    extra = ['sdf_eikonal_loss', 'total_variation_loss', 'entropy_loss']
    params = [g.decoder.net[0].weight, g.decoder.net[2].weight, g.beta]
    res = []
    try:
        for fn, fused in ((ref_render, False), (R.render, True)):
            R.enable_fused_heads(g, fused)
            w = ws.clone().requires_grad_()
            torch.manual_seed(31)
            out = fn(g, H, W, cams['c2w'], cams['focal'], None, cams['bbox'], w, S,
                     extra_model_outputs=list(extra))
            mo = out[5]
            loss = out[0].square().mean() + 0.1 * mo['sdf_eikonal_loss'].mean() \
                + mo['total_variation_loss'].mean() + 0.01 * mo['entropy_loss'].mean()
            grads = torch.autograd.grad(loss, [w] + params)
            res.append((mo, grads, torch.cuda.get_rng_state()))
    finally:
        R.enable_fused_heads(g, False)
        g.eval()
        g.requires_grad_(False)
    (mo_r, gr, s_r), (mo_f, gf, s_f) = res
    assert torch.equal(s_r, s_f), 'RNG consumption differs'
    for k in extra:
        assert mo_f[k].shape == mo_r[k].shape
        assert _rel(mo_f[k], mo_r[k]) < 1e-3, (k, _rel(mo_f[k], mo_r[k]))
    for n, a, b in zip(('ws', 'w1', 'w2', 'beta'), gf, gr):
        assert _rel(a, b) < 5e-3, (n, _rel(a, b))
    # SDF pre-training branch of ParallelModel (run.py:598-600)
    pm = R.ParallelModel(H, model=g, model_ema=g)
    g.train()
    try:
        torch.manual_seed(3)
        a = pm(None, None, None, None, ws, pretrain_sdf=True)
        R.enable_fused_heads(g)
        torch.manual_seed(3)
        b = pm(None, None, None, None, ws, pretrain_sdf=True)
    finally:
        R.enable_fused_heads(g, False)
        g.eval()
    for k in ('sdf_distance_loss', 'sdf_eikonal_loss'):
        assert _rel(b[k], a[k]) < 1e-3, k
