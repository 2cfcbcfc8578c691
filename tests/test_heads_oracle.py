"""oracle/heads_oracle.py against the original project's Generator regulariser heads
(models/generator.py:520-585; its synthesis network stubbed to return the planes under test),
values and gradients w.r.t. planes / decoder / beta, with the same random draws.  What the
original module returned is stored in tests/golden/reference/heads_match_the_reference.npz
(tests/golden/make_golden_reference.py)."""
import torch

from oracle import heads_oracle as HO
from tests import helpers as Hh

REQ = ['sdf_eikonal_loss', 'sdf_distance_loss', 'total_variation_loss', 'entropy_loss']
WEIGHTS = torch.tensor([1.0, 0.1, 3.0, 0.5])
B, R, NSTRATA, SEED = 2, 16, 32, 11


def test_heads_match_the_reference():
    ref = Hh.reference_golden('heads_match_the_reference', 'out')
    leaf = Hh.reference_golden('heads_match_the_reference', 'leaf')
    grad = Hh.reference_golden('heads_match_the_reference', 'grad')
    scene, _ = Hh.make_case('p3d_plain', seed=3, batch=B, plane_res=R)
    # replay the module's two draws: rand_like(bins) (ops.py:23), then randn_like(eik_coords) (:554)
    torch.manual_seed(SEED)
    n = NSTRATA - 1
    noise = torch.rand(B, n, n, n, 3)
    perturb = torch.randn(B, 1, n ** 3, 3).view(B, n ** 3, 3)
    leaves = {k: leaf[k].clone().requires_grad_() for k in ('w1', 'b1', 'w2', 'b2', 'beta')}
    for k in ('w1', 'b1', 'w2', 'b2'):   # the fixture's weights, through the EqualizedLinear gains
        assert torch.allclose(leaves[k], scene[k], rtol=1e-6, atol=1e-7), k
    planes2 = scene['planes'].clone().requires_grad_()
    pts = HO.stratified_points(B, NSTRATA, scene['scene_range'], noise)
    got = HO.heads(planes2, leaves['w1'], leaves['b1'], leaves['w2'], leaves['b2'], leaves['beta'],
                   scene['scene_range'], pts, REQ, perturb)
    for k in REQ:
        assert got[k].shape == ref[k].shape == (B,)
        assert (got[k] - ref[k]).abs().max().item() < 2e-5 * max(1.0, ref[k].abs().max().item()), k
    loss_g = sum(w * got[k].sum() for w, k in zip(WEIGHTS, REQ))
    gg = torch.autograd.grad(loss_g, [planes2, leaves['w1'], leaves['w2'], leaves['beta']])
    assert Hh.rel_l2(gg[0], grad['planes']) < 1e-4
    # d/d raw weight = gain * d/d effective
    assert Hh.rel_l2(gg[1] * leaf['w1_gain'], grad['w1_raw']) < 1e-4
    assert Hh.rel_l2((gg[2] * leaf['w2_gain'])[:1], grad['w2_raw'][:1]) < 1e-4
    assert Hh.rel_l2(gg[3], grad['beta']) < 1e-4
