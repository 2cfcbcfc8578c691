"""Size-independent properties of the render path, checked on the oracle (CPU).

They hold for the reference by construction (citations inline) and are what the GPU parity
tests rely on implicitly at sizes where no fixture exists: colour is linear in the palette,
the background only enters through 1 - mask, images are independent of each other, fine
depths stay inside [near, far], and the deterministic mode has no hidden draw.
"""
import torch

from fixtures import synthetic
from oracle import render_oracle as O
from tests import helpers as Hh

H, W, S = 12, 16, 12


def case(seed=3, name='p3d_bbox', batch=3):
    scene, cams = Hh.make_case(name, seed=seed, batch=batch, plane_res=24)
    nt, nu = synthetic.make_noise(seed, batch, H, W, S)
    return scene, cams, nt, nu


def test_colour_is_linear_in_the_palette():
    """rgb = sum_i w_i softmax(f_i) @ palette (generator.py:668-679, nerf_utils.py:151)."""
    scene, cams, nt, nu = case()
    g = torch.Generator().manual_seed(1)
    p1, p2 = torch.rand(3, 10, 3, generator=g), torch.rand(3, 10, 3, generator=g)
    r = lambda pal: Hh.run_oracle(dict(scene, palette=pal), cams, H, W, S, nt, nu)
    a, b, c = r(p1), r(p2), r(0.3 * p1 - 1.7 * p2)
    assert (c['rgb'] - (0.3 * a['rgb'] - 1.7 * b['rgb'])).abs().max().item() < 1e-5
    for k in ('mask', 'depth'):  # geometry does not see the palette
        assert torch.equal(a[k], b[k]) and torch.equal(a[k], c[k])


def test_white_background_only_adds_one_minus_mask():
    """nerf_utils.py:157-158."""
    scene, cams, nt, nu = case()
    black = Hh.run_oracle(dict(scene, white_background=False), cams, H, W, S, nt, nu)
    white = Hh.run_oracle(dict(scene, white_background=True), cams, H, W, S, nt, nu)
    assert (white['rgb'] - (black['rgb'] + (1 - black['mask'])[..., None])).abs().max().item() < 1e-6
    assert torch.equal(white['mask'], black['mask']) and torch.equal(white['depth'], black['depth'])


def test_images_are_independent():
    """No cross-image arithmetic (SURVEY.md section 8e): any permutation or subset of the batch
    renders to the same pixels -- the premise of sharding by image.  Both renders run on one CPU
    thread: with 16 or more, ATen splits the oracle's work by position in the batch, and the last
    bit of a pixel can then depend on where its image sits."""
    scene, cams, nt, nu = case()
    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        full = Hh.run_oracle(scene, cams, H, W, S, nt, nu)
        perm = torch.tensor([2, 0, 1])
        per_image = ('planes', 'palette', 'c2w', 'focal', 'center', 'bbox')
        sel = lambda d: {k: (v[perm] if (k in per_image and v is not None) else v)
                         for k, v in d.items()}
        out = Hh.run_oracle(sel(scene), sel(cams), H, W, S, nt[perm],
                            nu.view(3, H * W, S)[perm].reshape(-1, S))
    finally:
        torch.set_num_threads(threads)
    for k in ('rgb', 'depth', 'mask'):
        assert torch.equal(out[k], full[k][perm]), k


def test_ranges():
    scene, cams, nt, nu = case(name='chairs_white_center')
    out = Hh.run_oracle(scene, cams, H, W, S, nt, nu)
    assert out['mask'].min() >= 0 and out['mask'].max() <= 1 + 1e-5
    # sample_pdf returns the fine depths in draw order (nerf_utils.py:201-222; the union is
    # sorted later, run.py:283); the CUDA path sorts the uniforms first -- same set
    z = out['z_fine'].view(3, H, W, S)
    o, d = O.ray_bundle(H, W, cams['focal'], cams['c2w'], cams['bbox'], cams['center'])
    near, far, _ = O.near_far_planes(o, torch.nn.functional.normalize(d, dim=-1),
                                     scene['scene_range'])
    assert (z >= near[..., None] - 1e-5).all() and (z <= far[..., None] + 1e-5).all()
    assert (out['depth'] <= far * out['mask'] + 1e-4).all()  # depth = sum w t <= far * sum w


def test_deterministic_mode_is_deterministic():
    scene, cams, _, _ = case()
    a = Hh.run_oracle(scene, cams, H, W, S, None, None)
    torch.manual_seed(123)
    torch.rand(7)
    b = Hh.run_oracle(scene, cams, H, W, S, None, None)
    for k in ('rgb', 'depth', 'mask'):
        assert torch.equal(a[k], b[k]), k
