"""Golden vectors produced by the reference itself (tests/golden/make_golden.py).

CPU: the oracle reproduces every fixture (forward and reference-autograd
gradients) -- this is what pins the oracle to the reference on a machine that
has no checkout of the original project.  GPU: the CUDA path reproduces them through the C ABI.
"""
import glob
import os

import numpy as np
import pytest
import torch

from tests import helpers as Hh

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
FILES = sorted(glob.glob(os.path.join(GOLDEN_DIR, '*.npz')))
GRAD_NAMES = ['planes', 'w1', 'b1', 'w2', 'b2', 'c2w', 'palette', 'beta', 'alpha', 'w3', 'b3',
              'vm_fc0_w', 'vm_fc4_w', 'vm_norm3_b']  # vm_*: ViewDirectionMapper trunk (--use_viewdir)


def load(path, device='cpu'):
    z = np.load(path)
    t = lambda k: torch.from_numpy(z[k]).to(device) if k in z.files else None
    meta = {k[5:]: z[k].item() for k in z.files if k.startswith('meta_')}
    scene = {k: t('in_' + k) for k in ('planes', 'w1', 'b1', 'w2', 'b2', 'palette', 'beta', 'alpha')}
    if 'in_w3' in z.files:
        scene.update(w3=t('in_w3'), b3=t('in_b3'),
                     view_mapper={k[6:]: t(k) for k in z.files if k.startswith('in_vm_')})
    scene['scene_range'] = float(meta['scene_range'])
    scene['white_background'] = bool(meta['white_background'])
    cams = {k: t('cam_' + k) for k in ('c2w', 'focal', 'center', 'bbox')}
    expect = {k: t(k) for k in z.files if not k.startswith(('in_', 'cam_', 'meta_', 'noise_'))}
    return scene, cams, t('noise_t'), t('noise_u'), meta, expect


def loss_of(rgb, mask):
    g = torch.Generator().manual_seed(99)
    wr = torch.randn(rgb.shape, generator=g).to(rgb.device)
    wm = torch.randn(mask.shape, generator=g).to(rgb.device)
    return (rgb * wr).sum() + (mask * wm).sum()


def with_leaves(scene, cams):
    sc = {k: (v.clone().requires_grad_() if (torch.is_tensor(v) and k in GRAD_NAMES) else v)
          for k, v in scene.items()}
    if 'view_mapper' in scene:
        sc['view_mapper'] = {k: (v.clone().requires_grad_() if 'vm_' + k in GRAD_NAMES else v)
                             for k, v in scene['view_mapper'].items()}
    cm = dict(cams)
    cm['c2w'] = cams['c2w'].clone().requires_grad_()
    return sc, cm


def leaf_of(sc, cm, n):
    if n == 'c2w':
        return cm['c2w']
    return sc['view_mapper'][n[3:]] if n.startswith('vm_') else sc[n]


def test_fixture_set_is_complete():
    assert len(FILES) >= 9


@pytest.mark.parametrize('path', FILES, ids=[os.path.basename(f)[:-4] for f in FILES])
def test_oracle_reproduces_reference_golden(path):
    scene, cams, nt, nu, m, exp = load(path)
    sc, cm = with_leaves(scene, cams)
    out = Hh.run_oracle(sc, cm, m['H'], m['W'], m['S'], nt, nu, use_sdf=bool(m['use_sdf']),
                        fine_sampling=bool(m['fine_sampling']),
                        compute_semantics=bool(m['compute_semantics']),
                        compute_coords=bool(m['compute_coords']))
    for k in ('rgb', 'depth', 'mask'):
        assert (out[k] - exp[k]).abs().max().item() < 2e-5, k
    if 'extra' in exp:
        assert (out['semantics'] - exp['extra']).abs().max().item() < 2e-5
    names = [n for n in GRAD_NAMES if ('grad_' + n) in exp]
    leaves = [leaf_of(sc, cm, n) for n in names]
    grads = torch.autograd.grad(loss_of(out['rgb'], out['mask']), leaves)
    for n, g in zip(names, grads):
        assert Hh.rel_l2(g, exp['grad_' + n]) < 1e-4, n


@pytest.mark.gpu
@pytest.mark.parametrize('path', FILES, ids=[os.path.basename(f)[:-4] for f in FILES])
def test_cuda_reproduces_reference_golden(cuda_lib, path):
    scene, cams, nt, nu, m, exp = load(path, 'cuda')
    sc, cm = with_leaves(scene, cams)
    extra_mode = 1 if m['compute_coords'] else (2 if m['compute_semantics'] else 0)
    rgb, depth, mask, extra = Hh.run_cuda(sc, cm, m['H'], m['W'], m['S'], nt, nu,
                                          use_sdf=bool(m['use_sdf']),
                                          fine_sampling=bool(m['fine_sampling']),
                                          extra_mode=extra_mode)
    assert Hh.rel_l2(rgb, exp['rgb']) < 2e-4
    assert Hh.rel_l2(mask, exp['mask']) < 2e-4
    assert Hh.rel_l2(depth, exp['depth']) < 2e-4
    if 'extra' in exp:
        assert Hh.rel_l2(extra, exp['extra']) < 2e-4
    names = [n for n in GRAD_NAMES if ('grad_' + n) in exp]
    leaves = [leaf_of(sc, cm, n) for n in names]
    grads = torch.autograd.grad(loss_of(rgb, mask), leaves)
    for n, g in zip(names, grads):
        assert Hh.rel_l2(g, exp['grad_' + n]) < 2e-3, n
