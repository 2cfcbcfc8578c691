"""Shared helpers for the parity tests (oracle side and CUDA side)."""
import os

import numpy as np
import torch

from fixtures import synthetic
from oracle import render_oracle as O

REFERENCE_GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference')


def reference_golden(test, key):
    """{output name: tensor} the original project returned for parameter set ``key`` of
    ``test`` (recorded by tests/golden/make_golden_reference.py)."""
    z = np.load(os.path.join(REFERENCE_GOLDEN, test + '.npz'))
    out = {k[len(key) + 1:]: torch.from_numpy(z[k]) for k in z.files if k.startswith(key + '/')}
    assert out, 'no stored reference outputs for %s / %s' % (test, key)
    return out

CASES = {
    # name: (dataset, camera kwargs, scene kwargs)
    'p3d_bbox': ('p3d_car', dict(with_bbox=True), {}),
    'p3d_plain': ('p3d_car', dict(), {}),
    'cub_ortho': ('cub', dict(), {}),
    'cub_ortho_bbox': ('cub', dict(with_bbox=True), {}),
    'chairs_white_center': ('shapenet_chairs', dict(with_center=True), {}),
}


def make_case(name, seed=1, batch=2, plane_res=32, attention_values=10, device='cpu'):
    ds, cam_kw, sc_kw = CASES[name]
    cfg = synthetic.DATASET_CONFIGS[ds]
    scene = synthetic.make_scene(seed, batch, plane_res=plane_res,
                                 attention_values=attention_values,
                                 scene_range=cfg['scene_range'],
                                 white_background=cfg['white_background'],
                                 object_radius=cfg['object_radius'], device=device, **sc_kw)
    cams = synthetic.make_cameras(seed, batch, ortho=cfg['ortho'], radius=cfg['radius'],
                                  device=device, **cam_kw)
    return scene, cams


def to_device(d, device):
    return {k: (v.to(device) if torch.is_tensor(v) else v) for k, v in d.items()}


def view_features(scene, cams, H, W, cam_grad=True):
    """[B,H,W,32] ViewDirectionMapper trunk output of the rays of ``cams`` for a scene from
    ``synthetic.add_view_mapper`` (what the reference's Generator computes from the view
    directions render() hands it, run.py:216-221), with the oracle's restatement."""
    _, d = O.ray_bundle(H, W, cams['focal'], cams['c2w'], cams['bbox'], cams['center'])
    d = torch.nn.functional.normalize(d, dim=-1)
    if not cam_grad:
        d = d.detach()
    return O.view_mapper_trunk(d, scene['view_mapper'])


def run_oracle(scene, cams, H, W, S, noise_t, noise_u, **kw):
    if 'view_mapper' in scene and 'view_features' not in kw:
        kw = dict(kw, view_features=view_features(scene, cams, H, W,
                                                  not kw.get('force_no_cam_grad', False)),
                  w3=scene['w3'], b3=scene['b3'])
    return O.render_oracle(scene['planes'], scene['w1'], scene['b1'], scene['w2'],
                           scene['b2'], scene['palette'], scene['beta'], scene['alpha'],
                           cams['c2w'], cams['focal'], cams['center'], cams['bbox'],
                           H, W, S, noise_t, noise_u, scene_range=scene['scene_range'],
                           white_background=scene['white_background'], **kw)


MLP_MODE = 0  # tests/test_parity_gpu.py switches this (0 auto, 1 SIMT, 2 tensor core)


def run_cuda(scene, cams, H, W, S, noise_t, noise_u, use_sdf=True, fine_sampling=True,
             extra_mode=0, cam_grad=True, device='cuda', mlp_mode=None, compute_normals=False):
    from nerf_from_image_b200.fused import RenderConfig, fused_render
    sc = to_device(scene, device)
    cm = to_device(cams, device)
    view = None
    if 'view_mapper' in sc:
        vm = {k: v.to(device) for k, v in sc['view_mapper'].items()}
        view = (view_features(dict(sc, view_mapper=vm), cm, H, W, cam_grad), sc['w3'], sc['b3'])
    A = sc['palette'].shape[1] if sc['palette'] is not None else 0
    cfg = RenderConfig(scene_range=sc['scene_range'], white_background=sc['white_background'],
                       use_sdf=use_sdf, fine_sampling=fine_sampling, attention_values=A,
                       mlp_mode=MLP_MODE if mlp_mode is None else mlp_mode)
    nt = noise_t.to(device) if noise_t is not None else None
    nu = noise_u.to(device) if noise_u is not None else None
    return fused_render(sc['planes'], sc['w1'], sc['b1'], sc['w2'], sc['b2'], sc['palette'],
                        sc['beta'], sc['alpha'], cm['c2w'], cm['focal'], cm['center'],
                        cm['bbox'], cfg, H, W, S, nt, nu, extra_mode, cam_grad,
                        compute_normals=compute_normals, view=view)


def rel_l2(a, b):
    return ((a - b).norm() / b.norm().clamp_min(1e-12)).item()
