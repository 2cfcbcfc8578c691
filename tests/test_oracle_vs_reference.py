"""Pins the oracle against the original project's own code (CPU).

What the original code returned for these inputs is stored under tests/golden/reference/
(tests/golden/make_golden_reference.py re-records it from a checkout of the original project);
the inputs are rebuilt here from the seeded fixtures.
"""
import pytest
import torch

from oracle import pose_oracle as PO
from oracle import render_oracle as O
from tests import helpers as Hh


def render_key(case, randomize):
    return '%s_randomize%d' % (case, int(randomize))


def kw_key(kw):
    return '_'.join('%s=%s' % (k, v) for k, v in sorted(kw.items())) or 'default'


def reference_noise(seed, B, H, W, S, randomize=True, fine_sampling=True):
    """The two draws the reference's render made after ``torch.manual_seed(seed)``
    (oracle/reference_lift.py replays them the same way)."""
    if not randomize:
        return None, None
    torch.manual_seed(seed)
    nt = torch.rand(B, H, W, S)
    nu = torch.rand(B * H * W, S) if fine_sampling else None
    return nt, nu


def assert_render_matches(ref, o):
    for k in ('rgb', 'depth', 'mask'):
        assert (ref[k] - o[k]).abs().max().item() < 2e-5, k
    if 'normals' in ref:
        assert (ref['normals'] - o['normals']).abs().max().item() < 1e-4
    if 'extra' in ref:
        assert (ref['extra'] - o['semantics']).abs().max().item() < 2e-5


@pytest.mark.parametrize('case', list(Hh.CASES))
@pytest.mark.parametrize('randomize', [True, False])
def test_render_matches_reference(case, randomize):
    ref = Hh.reference_golden('render_matches_reference', render_key(case, randomize))
    scene, cams = Hh.make_case(case, seed=2, batch=2, plane_res=24)
    nt, nu = reference_noise(4, 2, 12, 20, 12, randomize)
    o = Hh.run_oracle(scene, cams, 12, 20, 12, nt, nu)
    assert_render_matches(ref, o)


VARIANTS = [dict(fine_sampling=False), dict(use_sdf=False), dict(compute_semantics=True),
            dict(compute_coords=True), dict(compute_normals=True), dict(force_no_cam_grad=True)]


@pytest.mark.parametrize('kw', VARIANTS)
def test_render_variants_match_reference(kw):
    ref = Hh.reference_golden('render_variants_match_reference', kw_key(kw))
    scene, cams = Hh.make_case('p3d_bbox', seed=3, batch=2, plane_res=24)
    nt, nu = reference_noise(5, 2, 12, 12, 10, fine_sampling=kw.get('fine_sampling', True))
    o = Hh.run_oracle(scene, cams, 12, 12, 10, nt, nu, **kw)
    assert_render_matches(ref, o)
    assert ('normals' in ref) == bool(kw.get('compute_normals'))
    assert ('extra' in ref) == bool(kw.get('compute_semantics') or kw.get('compute_coords'))


VIEWDIR_CASES = [('p3d_plain', 10, {}), ('chairs_white_center', 0, {}),
                 ('cub_ortho', 10, dict(compute_semantics=True)),
                 ('p3d_bbox', 10, dict(force_no_cam_grad=True)),
                 ('p3d_plain', 10, dict(compute_normals=True))]


def viewdir_key(case, A, kw):
    return '%s_A%d_%s' % (case, A, kw_key(kw))


def trunk_directions():
    g = torch.Generator().manual_seed(7)
    return torch.nn.functional.normalize(torch.randn(3, 5, 1, 3, generator=g), dim=-1)


@pytest.mark.parametrize('case,A,kw', VIEWDIR_CASES)
def test_view_direction_conditioning_matches_reference(case, A, kw):
    """--use_viewdir (run.py:216-221, models/generator.py:189-253,662-663): the reference
    Generator built with use_viewdir=True and given the oracle scene's ViewDirectionMapper
    weights, called by the reference's own render(), against the oracle's restatement of the
    mapper trunk (per ray) and closure (per sample)."""
    from fixtures import synthetic
    ref = Hh.reference_golden('view_direction_conditioning_matches_reference',
                              viewdir_key(case, A, kw))
    scene, cams = Hh.make_case(case, seed=2, batch=2, plane_res=24, attention_values=A)
    scene = synthetic.add_view_mapper(scene)
    nt, nu = reference_noise(4, 2, 12, 20, 12)
    o = Hh.run_oracle(scene, cams, 12, 20, 12, nt, nu, **kw)
    assert_render_matches(ref, o)
    # the trunk alone, against the module (bit-identical: same ops in the same order).  The
    # module holds weight / gain and uses weight * gain (render_oracle.effective_view_mapper_weights)
    m = dict(scene['view_mapper'])
    for k, gain in ref.items():
        if k.startswith('gain_'):
            m[k[len('gain_'):]] = (m[k[len('gain_'):]] / gain) * gain
    assert len(m) == len(scene['view_mapper'])
    assert torch.equal(O.view_mapper_trunk(trunk_directions(), m), ref['trunk_x'])


STAGE_CAMERAS = ('p3d_bbox', 'cub_ortho_bbox', 'chairs_white_center')


def pdf_inputs():
    torch.manual_seed(0)
    w = torch.rand(50, 16)
    bins = torch.sort(torch.rand(50, 15), dim=-1).values
    return w, bins


def test_stage_functions_match_reference():
    scene, cams = Hh.make_case('p3d_bbox', seed=6, batch=2)
    for cam_case in STAGE_CAMERAS:
        ref = Hh.reference_golden('stage_functions_match_reference', cam_case)
        _, cams = Hh.make_case(cam_case, seed=6, batch=2)
        o, d = O.ray_bundle(9, 13, cams['focal'], cams['c2w'], cams['bbox'], cams['center'])
        assert (ref['origins'] - o).abs().max() < 1e-6 and (ref['dirs'] - d).abs().max() < 1e-6
        dn = torch.nn.functional.normalize(ref['dirs'], dim=-1)
        n, f, _ = O.near_far_planes(o, dn, scene['scene_range'])
        assert torch.equal(ref['near'], n) and torch.equal(ref['far'], f)
    ref = Hh.reference_golden('stage_functions_match_reference', 'sample_pdf')
    w, bins = pdf_inputs()
    torch.manual_seed(1)
    u = torch.rand(50, 16)
    assert torch.allclose(ref['random'], O.inverse_cdf_samples(bins, w[..., 1:-1], u), atol=1e-6)
    assert torch.allclose(ref['deterministic'], O.inverse_cdf_samples(
        bins, w[..., 1:-1], O.deterministic_u(16, 50)), atol=1e-6)


def test_missed_rays_do_not_need_the_global_fallback():
    """The CUDA path skips lib/nerf_utils.py:258-259; images must not change."""
    scene, cams = Hh.make_case('p3d_plain', seed=8, batch=2)
    cams['focal'] = torch.tensor([0.35, 0.4])  # wide field of view: corner rays miss the cube
    from fixtures import synthetic
    nt, nu = synthetic.make_noise(1, 2, 16, 16, 8)
    a = Hh.run_oracle(scene, cams, 16, 16, 8, nt, nu, global_near_far_fallback=True)
    b = Hh.run_oracle(scene, cams, 16, 16, 8, nt, nu, global_near_far_fallback=False)
    o, d = O.ray_bundle(16, 16, cams['focal'], cams['c2w'], cams['bbox'], None)
    hit = O.near_far_planes(o, torch.nn.functional.normalize(d, dim=-1), scene['scene_range'])[2]
    assert (~hit).any() and hit.any()
    for k in ('rgb', 'depth', 'mask'):
        assert torch.equal(a[k], b[k]), k


def sampler_points(scene, batch, n, seed):
    """Points filling the cube and a margin outside it (the out-of-box mask must trigger)."""
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(batch, 5, n // 5, 3, generator=g) * 2 - 1) * 1.15 * scene['scene_range']


SAMPLER_CASES = [
    (10, True, ['sigma', 'rgb']),
    (10, True, ['sdf_distance', 'sigma', 'rgb', 'semantics', 'coords']),
    (0, True, ['sigma', 'rgb', 'sdf_distance']),
    (10, False, ['sigma', 'rgb']),
]


def sampler_key(A, use_sdf, request):
    return 'A%d_sdf%d_%s' % (A, int(use_sdf), '+'.join(request))


@pytest.mark.parametrize('A,use_sdf,request_', SAMPLER_CASES)
def test_sampler_matches_reference(A, use_sdf, request_):
    ref = Hh.reference_golden('sampler_matches_reference', sampler_key(A, use_sdf, request_))
    scene, _ = Hh.make_case('p3d_plain', seed=12, batch=2, plane_res=24, attention_values=A)
    x = sampler_points(scene, 2, 200, 3)
    with torch.no_grad():
        o = O.sampler(x, scene['planes'], scene['w1'], scene['b1'], scene['w2'], scene['b2'],
                      scene['palette'], scene['beta'], scene['alpha'], scene['scene_range'],
                      request=request_, use_sdf=use_sdf)
    assert sorted(ref) == sorted(o)
    for k in ref:
        assert ref[k].shape == o[k].shape, k
        assert (ref[k] - o[k]).abs().max().item() < 2e-5, k


def test_sampler_normals_and_bbox_match_reference():
    scene, _ = Hh.make_case('p3d_plain', seed=13, batch=2, plane_res=24)
    x = sampler_points(scene, 2, 200, 4)
    ref = Hh.reference_golden('sampler_normals_and_bbox_match_reference', 'normals')
    o = O.sampler(x, scene['planes'], scene['w1'], scene['b1'], scene['w2'], scene['b2'],
                  scene['palette'], scene['beta'], scene['alpha'], scene['scene_range'],
                  request=['normals', 'sigma'])
    assert ref['normals'].shape == o['normals'].shape == x.shape
    assert (ref['normals'] - o['normals']).abs().max().item() < 1e-4
    assert (ref['sigma'] - o['sigma']).abs().max().item() < 2e-5
    ref = Hh.reference_golden('sampler_normals_and_bbox_match_reference', 'bbox')
    with torch.no_grad():
        o = O.sampler(x, scene['planes'], scene['w1'], scene['b1'], scene['w2'], scene['b2'],
                      scene['palette'], scene['beta'], scene['alpha'], scene['scene_range'],
                      request=['sigma', 'coords'], bbox_debug=True)
    assert (ref['sigma'] > 50).any()
    assert (ref['sigma'] - o['sigma']).abs().max().item() < 2e-5


def pose_inputs(seed, batch, persp):
    g = torch.Generator().manual_seed(seed)
    q = torch.nn.functional.normalize(torch.randn(batch, 4, generator=g), dim=-1)
    t2 = 0.3 * torch.randn(batch, 2, generator=g)
    s = 0.8 + 0.5 * torch.rand(batch, generator=g)
    z0 = 0.5 * torch.randn(batch, generator=g) if persp else None
    return z0, t2, s, q


def pose_loss(m, f):
    g = torch.Generator().manual_seed(9)
    wm = torch.randn(6, 4, 4, generator=g)
    wf = torch.randn(6, generator=g)
    return (m * wm).sum() + ((f * wf).sum() if f is not None else 0)


def pose_key(persp, flipped):
    return 'persp%d_flipped%d' % (int(persp), int(flipped))


@pytest.mark.parametrize('persp', [True, False])
@pytest.mark.parametrize('flipped', [True, False])
def test_pose_to_matrix_matches_reference(persp, flipped):
    ref = Hh.reference_golden('pose_to_matrix_matches_reference', pose_key(persp, flipped))
    z0, t2, s, q = pose_inputs(5, 6, persp)
    leaves = [t.clone().requires_grad_() for t in (z0, t2, s, q) if t is not None]
    args = (leaves[0], leaves[1], leaves[2], leaves[3]) if persp else \
        (None, leaves[0], leaves[1], leaves[2])
    mat, f = PO.pose_to_matrix(*args, flipped)
    assert torch.equal(ref['matrix'], mat)
    assert ('focal' in ref) == (f is not None)
    if f is not None:
        assert torch.equal(ref['focal'], f)
    grads = torch.autograd.grad(pose_loss(mat, f), leaves)
    assert len(grads) == len([k for k in ref if k.startswith('grad')])
    for i, g in enumerate(grads):
        assert (ref['grad%d' % i] - g).abs().max().item() < 1e-5
    # (lib/pose_utils.py:72 matrix_to_pose, the reference's inverse, does not run under
    # numpy >= 2 -- np.array(copy=False) -- so the round trip is not checked through it)
    rows = PO.quaternion_rows(q)
    eye = torch.eye(3).expand(6, 3, 3)
    assert (rows @ rows.transpose(-1, -2) - eye).abs().max().item() < 1e-5
