"""Records what the original project's own code returns for the inputs of
tests/test_oracle_vs_reference.py, tests/test_heads_oracle.py, tests/test_render_dropin.py and
tests/test_synthesis_oracle.py, so that those comparisons run from this repository alone:

    NFI_REFERENCE_ROOT=<checkout of the original nerf-from-image> \
        python tests/golden/make_golden_reference.py

The inputs (scenes, cameras, points, poses) come from the seeded fixtures and are rebuilt by the
tests; mostly only the reference's outputs are stored, one tests/golden/reference/<test>.npz per
test function (per test module for the drop-in seam), keyed '<parameter set>/<output>'.  The
synthesis network's block-by-block record also holds the small network's parameters.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from fixtures import synthetic  # noqa: E402
from oracle import reference_lift as RL  # noqa: E402
from oracle import render_oracle as O  # noqa: E402
from oracle import synthesis_oracle as SO  # noqa: E402
from tests import helpers as Hh  # noqa: E402
from tests import helpers_dropin as HD  # noqa: E402
from tests import test_render_dropin as TD  # noqa: E402
from tests import test_synthesis_oracle as TS  # noqa: E402
from tests import test_heads_oracle as TH  # noqa: E402
from tests import test_oracle_vs_reference as T  # noqa: E402

OUT = os.path.join(HERE, 'reference')
RENDER_OUTPUTS = ('rgb', 'depth', 'mask', 'normals', 'extra')


def put(arrays, prefix, **tensors):
    for k, v in tensors.items():
        if v is not None:
            arrays[prefix + '/' + k] = v.detach().cpu().numpy()


def put_render(arrays, prefix, out):
    put(arrays, prefix, **dict(zip(RENDER_OUTPUTS, out[:5])))


def render_cases():
    a = {}
    for case in Hh.CASES:
        for randomize in (True, False):
            scene, cams = Hh.make_case(case, seed=2, batch=2, plane_res=24)
            out, _, _ = RL.reference_render(scene, cams, 12, 20, 12, seed=4, randomize=randomize)
            put_render(a, T.render_key(case, randomize), out)
    return a


def render_variants():
    a = {}
    for kw in T.VARIANTS:
        scene, cams = Hh.make_case('p3d_bbox', seed=3, batch=2, plane_res=24)
        out, _, _ = RL.reference_render(scene, cams, 12, 12, 10, seed=5, **kw)
        put_render(a, T.kw_key(kw), out)
    return a


def view_direction_conditioning():
    a = {}
    for case, A, kw in T.VIEWDIR_CASES:
        key = T.viewdir_key(case, A, kw)
        scene, cams = Hh.make_case(case, seed=2, batch=2, plane_res=24, attention_values=A)
        scene = synthetic.add_view_mapper(scene)
        out, _, _ = RL.reference_render(scene, cams, 12, 20, 12, seed=4, **kw)
        put_render(a, key, out)
        g = RL.build_reference_generator(scene)
        closure = g.viewdir_mapper(T.trunk_directions())
        x = dict(zip(closure.__code__.co_freevars,
                     (c.cell_contents for c in closure.__closure__)))['x']
        gains = {}
        for i in range(7):
            fc = getattr(g.viewdir_mapper, 'fc%d' % i)
            gains['gain_fc%d_w' % i] = torch.tensor(float(fc.weight_gain))
            if fc.bias is not None:
                gains['gain_fc%d_b' % i] = torch.tensor(float(fc.bias_gain))
        put(a, key, trunk_x=x, **gains)
    return a


def stage_functions():
    a = {}
    nerf_utils, _ = RL._import_reference()
    scene, _ = Hh.make_case('p3d_bbox', seed=6, batch=2)
    for cam_case in T.STAGE_CAMERAS:
        _, cams = Hh.make_case(cam_case, seed=6, batch=2)
        ro, rd = nerf_utils.get_ray_bundle(9, 13, cams['focal'], cams['c2w'], cams['bbox'],
                                           cams['center'])
        dn = torch.nn.functional.normalize(rd, dim=-1)
        rn, rf = nerf_utils.compute_near_far_planes(ro, dn, scene['scene_range'])
        put(a, cam_case, origins=ro, dirs=rd, near=rn, far=rf)
    w, bins = T.pdf_inputs()
    torch.manual_seed(1)
    put(a, 'sample_pdf', random=nerf_utils.sample_pdf(bins, w[..., 1:-1], 16, deterministic=False),
        deterministic=nerf_utils.sample_pdf(bins, w[..., 1:-1], 16, deterministic=True))
    return a


def sampler():
    a = {}
    for A, use_sdf, request in T.SAMPLER_CASES:
        scene, _ = Hh.make_case('p3d_plain', seed=12, batch=2, plane_res=24, attention_values=A)
        x = T.sampler_points(scene, 2, 200, 3)
        with torch.no_grad():
            ref = RL.reference_sampler(scene, x, request, use_sdf=use_sdf)
        put(a, T.sampler_key(A, use_sdf, request), **ref)
    return a


def sampler_normals_and_bbox():
    a = {}
    scene, _ = Hh.make_case('p3d_plain', seed=13, batch=2, plane_res=24)
    x = T.sampler_points(scene, 2, 200, 4)
    ref = RL.reference_sampler(scene, x.clone(), ['normals', 'sigma'])
    put(a, 'normals', **ref)
    with torch.no_grad():
        ref = RL.reference_sampler(scene, x, ['sigma', 'coords'], bbox_debug=True)
    put(a, 'bbox', **ref)
    return a


def pose_to_matrix():
    a = {}
    pu = RL.reference_pose_utils()
    for persp in (True, False):
        for flipped in (True, False):
            z0, t2, s, q = T.pose_inputs(5, 6, persp)
            leaves = [t.clone().requires_grad_() for t in (z0, t2, s, q) if t is not None]
            args = (leaves[0], leaves[1], leaves[2], leaves[3]) if persp else \
                (None, leaves[0], leaves[1], leaves[2])
            mat, focal = pu.pose_to_matrix(*args, flipped)
            grads = torch.autograd.grad(T.pose_loss(mat, focal), leaves)
            put(a, T.pose_key(persp, flipped), matrix=mat, focal=focal,
                **{'grad%d' % i: g for i, g in enumerate(grads)})
    return a


def heads():
    a = {}
    B, R, nstrata = TH.B, TH.R, TH.NSTRATA
    scene, _ = Hh.make_case('p3d_plain', seed=3, batch=B, plane_res=R)
    g = RL.build_reference_generator(scene)
    g.train()   # the eikonal head asserts self.training (generator.py:531)
    planes = scene['planes'].clone().requires_grad_()
    g.synthesis_network.planes = planes.reshape(B, 96, R, R)
    ws = torch.zeros(B, 15, 512)
    torch.manual_seed(TH.SEED)
    ref = g(None, ws, request_model_outputs=TH.REQ,
            model_inputs={'attention_values': scene['palette']})
    l1, l2 = g.decoder.net[0], g.decoder.net[2]
    loss = sum(w * ref[k].sum() for w, k in zip(TH.WEIGHTS, TH.REQ))
    gr = torch.autograd.grad(loss, [planes, l1.weight, l2.weight, g.beta])
    put(a, 'out', **{k: ref[k] for k in TH.REQ})
    put(a, 'leaf', w1=l1.weight * l1.weight_gain, b1=l1.bias * l1.bias_gain,
        w2=l2.weight * l2.weight_gain, b2=l2.bias * l2.bias_gain, beta=g.beta,
        w1_gain=torch.tensor(float(l1.weight_gain)), w2_gain=torch.tensor(float(l2.weight_gain)))
    put(a, 'grad', planes=gr[0], w1_raw=gr[1], w2_raw=gr[2], beta=gr[3])
    return a


def reference_dropin_generator(scene, use_sdf=True):
    """The original Generator loaded with ``scene``, after checking that the stand-in the tests
    use in its place has bit-identical effective weights."""
    g = RL.build_reference_generator(scene, use_sdf=use_sdf)
    h = HD.SceneGenerator(scene, use_sdf=use_sdf)
    for a, b in zip((g.decoder.net[0], g.decoder.net[2]), (h.decoder.net[0], h.decoder.net[2])):
        assert torch.equal(a.weight * a.weight_gain, b.weight * b.weight_gain)
        assert torch.equal(a.bias * a.bias_gain, b.bias * b.bias_gain)
    if h.use_viewdir:
        ma, wa, ba = O.effective_view_mapper_weights(g.viewdir_mapper)
        mb = h.viewdir_mapper.effective()
        assert sorted(ma) == sorted(mb) and all(torch.equal(ma[k], mb[k]) for k in ma)
        out = h.viewdir_mapper.output
        assert torch.equal(wa, out.weight * out.weight_gain) and torch.equal(ba, out.bias * out.bias_gain)
    B, _, C, R, _ = scene['planes'].shape
    g.synthesis_network.planes = scene['planes'].reshape(B, 3 * C, R, R)
    return g


def render_dropin():
    a = {}
    H, W, S = TD.H, TD.W, TD.S
    for case, kw in TD.RETURNS_CASES:
        key = TD.returns_key(case, kw)
        kw = dict(kw)
        scene, cams = TD.scene_of(case, viewdir=kw.pop('viewdir', False))
        g = reference_dropin_generator(scene)
        randomize = kw.pop('randomize', True)
        out, _, _ = RL.reference_render(scene, cams, H, W, S, seed=33, randomize=randomize,
                                        generator=g, **kw)
        put_render(a, key, out)
        put(a, key, next=torch.rand(3))
    scene, cams = TD.scene_of('p3d_plain', viewdir=True)
    g = reference_dropin_generator(scene)
    cam = dict(cams, c2w=cams['c2w'].clone().requires_grad_())
    vm = g.viewdir_mapper
    leaves = [cam['c2w'], vm.fc0.weight, vm.fc3.weight, vm.norm2.bias, vm.output.weight, vm.output.bias]
    ref, _, _ = RL.reference_render(scene, cam, H, W, S, seed=4, generator=g)
    grads = torch.autograd.grad(ref[0].square().sum() + ref[2].sum(), leaves)
    put(a, 'viewdir_grads', **{'grad%d' % i: t for i, t in enumerate(grads)})
    # the names the original closures close over (extract_field / extract_view read them)
    d = torch.nn.functional.normalize(torch.randn(2, 4, 4, 1, 3), dim=-1)
    sampler = g(d, torch.zeros(2, 15, 512), ['sampler'],
                {'attention_values': scene['palette']})['sampler']
    a['sampler_freevars'] = np.array(sampler.__code__.co_freevars)
    mapper = dict(zip(sampler.__code__.co_freevars, sampler.__closure__))['viewdir_mapper_closure']
    a['mapper_freevars'] = np.array(mapper.cell_contents.__code__.co_freevars)
    for A, use_sdf, fine in TD.VARIANT_CASES:
        scene, cams = TD.scene_of('p3d_plain', A)
        g = reference_dropin_generator(scene, use_sdf)
        ref, _, _ = RL.reference_render(scene, dict(cams, center=None, bbox=None), H, W, S, seed=5,
                                        generator=g, use_sdf=use_sdf, fine_sampling=fine)
        put_render(a, TD.variant_key(A, use_sdf, fine), ref)
    scene, cams = TD.scene_of('p3d_bbox')
    g = reference_dropin_generator(scene)
    ref, _, _ = RL.reference_render(scene, dict(cams, center=None), H, H, S, seed=8, generator=g)
    put(a, 'parallel', rgb=ref[0])
    # the front-end's latent handling (models/generator.py:423-468) on the real mapping network
    seen = {}
    stub = g.synthesis_network

    def spy(w, **kw):
        seen['ws'] = w.clone()
        return stub.planes
    stub.forward = spy
    torch.manual_seed(2)
    z = torch.randn(2, 512)
    w_full = g.mapping_network(z, None).detach()
    rec = dict(w_full=w_full, texture_w14=g.texture_mapper(w_full[:, 14]),
               texture_w0=g.texture_mapper(w_full[:, 0]))
    for name, c in TD.front_end_inputs(z, w_full):
        out = g(None, c, ['sampler', 'attention_values'], {})
        rec[name + '_ws'] = seen['ws']
        rec[name + '_attention_values'] = out['attention_values']
    bias = TD.palette_bias()
    out = g(None, w_full, ['sampler', 'attention_values'], {'attention_values_bias': bias})
    rec['bias_attention_values'] = out['attention_values']
    put(a, 'front_end', **rec)
    return a


def synthesis_blocks():
    RL._import_reference()
    from models import stylegan
    p = TS.blocks_params()
    meta = p.pop('meta')
    net = stylegan.SynthesisNetwork(TS.BLOCKS_W_DIM, TS.BLOCKS_RES, 96,
                                    channel_base=4096, channel_max=128).eval()
    missing, unexpected = net.load_state_dict(p, strict=False)
    assert not unexpected and all(k.endswith('resample_filter') for k in missing)
    layers = SO.extract_params(net)['meta']['layers']   # the module's own flags
    ws = TS.blocks_ws(net.num_ws)
    a = {}
    with torch.no_grad():
        x = img = None
        w_idx = 0
        for i, r in enumerate(net.block_resolutions):
            blk = getattr(net, 'b%d' % r)
            cur = ws.narrow(1, w_idx, blk.num_conv + blk.num_torgb)
            w_idx += blk.num_conv
            x, img = blk(x, img, cur, noise_mode='const')
            for j, (name, t) in enumerate((('x', x), ('img', img))):
                put(a, 'b%d_%s' % (r, name), **TS.block_summary(t, 2 * i + j))
    assert net.num_ws == 2 * len(meta['resolutions'])
    a['layers'] = np.array(list(layers))
    put(a, 'flags', up=torch.tensor([v['up'] for v in layers.values()]),
        use_noise=torch.tensor([v['use_noise'] for v in layers.values()]))
    return a


FILES = {
    'render_matches_reference': render_cases,
    'render_variants_match_reference': render_variants,
    'view_direction_conditioning_matches_reference': view_direction_conditioning,
    'stage_functions_match_reference': stage_functions,
    'sampler_matches_reference': sampler,
    'sampler_normals_and_bbox_match_reference': sampler_normals_and_bbox,
    'pose_to_matrix_matches_reference': pose_to_matrix,
    'heads_match_the_reference': heads,
    'render_dropin': render_dropin,
    'synthesis_blocks': synthesis_blocks,
}


def main():
    if not RL.available():
        raise SystemExit('set NFI_REFERENCE_ROOT to a checkout of the original project')
    os.makedirs(OUT, exist_ok=True)
    for name, fn in FILES.items():
        if sys.argv[1:] and name not in sys.argv[1:]:   # re-record only the files named
            continue
        arrays = fn()
        path = os.path.join(OUT, name + '.npz')
        np.savez_compressed(path, **arrays)
        print('%-50s %3d arrays %8d bytes' % (name, len(arrays), os.path.getsize(path)))


if __name__ == '__main__':
    main()
