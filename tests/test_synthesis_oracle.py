"""oracle/synthesis_oracle.py (the restatement of the reference's plane producer, SURVEY.md
section 8f N1) against the golden fixtures the reference produced: its output, and the
UNMODIFIED models.stylegan.SynthesisNetwork block by block (recorded by
tests/golden/make_golden_reference.py)."""
import os

import numpy as np
import pytest
import torch

from oracle import synthesis_oracle as SO
from tests import helpers as Hh
from tests import helpers_synth as HS


@pytest.mark.parametrize('case', HS.CASES)
def test_oracle_reproduces_the_reference_fixtures(case):
    p, ws, img, mode = HS.load_case(case)
    noises = HS.const_noises(p) if mode == 'const' else None
    with torch.no_grad():
        got = SO.synthesis_forward(p, ws, noises)
    assert got.shape == img.shape
    assert (got - img).abs().max().item() < 2e-5 * max(1.0, img.abs().max().item())


# the recorded network: the original SynthesisNetwork(512, 32, 96, channel_base=4096,
# channel_max=128) -- four blocks of 128 channels -- in eval mode, its weights loaded from
# fixtures.synthetic.make_synthesis_params(BLOCKS_SEED, ...), const noise.  Its block outputs are
# too large to store whole: the record keeps BLOCKS_SAMPLE elements of each at seeded positions,
# each tensor's largest magnitude, and the mean and mean square of every (image, channel) plane.
BLOCKS_SEED, BLOCKS_RES, BLOCKS_CHANNELS, BLOCKS_W_DIM, BLOCKS_BATCH = 3, 32, (128,) * 4, 512, 2
BLOCKS_SAMPLE = 8192


def blocks_params():
    from fixtures import synthetic
    return synthetic.make_synthesis_params(BLOCKS_SEED, BLOCKS_RES, BLOCKS_CHANNELS, BLOCKS_W_DIM)


def blocks_ws(num_ws):
    return torch.randn(BLOCKS_BATCH, num_ws, BLOCKS_W_DIM,
                       generator=torch.Generator().manual_seed(BLOCKS_SEED + 1))


def block_summary(t, seed):
    """What the record keeps of a block output ``t`` [B, C, H, W]."""
    n = t.numel()
    idx = torch.randperm(n, generator=torch.Generator().manual_seed(seed))[:min(n, BLOCKS_SAMPLE)]
    d = t.double().flatten(2)
    return dict(sample=t.flatten()[idx], absmax=t.abs().max(), mean=d.mean(-1),
                mean_square=d.square().mean(-1))


def test_oracle_matches_the_reference_module_block_by_block():
    p = blocks_params()
    z = np.load(os.path.join(Hh.REFERENCE_GOLDEN, 'synthesis_blocks.npz'))
    recorded_layers = {str(k): dict(use_noise=bool(u), up=bool(up)) for k, u, up in
                       zip(z['layers'], z['flags/use_noise'], z['flags/up'])}
    assert p['meta']['layers'] == recorded_layers      # the module's own layer flags
    ws = blocks_ws(2 * len(p['meta']['resolutions']))
    with torch.no_grad():
        img, blocks = SO.synthesis_forward(p, ws, HS.const_noises(p), return_blocks=True)
    for i, r in enumerate(p['meta']['resolutions']):
        for j, (name, got) in enumerate(zip(('x', 'img'), blocks['b%d' % r])):
            ref = Hh.reference_golden('synthesis_blocks', 'b%d_%s' % (r, name))
            o = block_summary(got, 2 * i + j)
            scale = max(1.0, ref['absmax'].item())
            assert (o['sample'] - ref['sample']).abs().max().item() < 1e-4 * scale, (r, name)
            assert abs(o['absmax'] - ref['absmax']).item() < 1e-4 * scale, (r, name)
            # implied by an elementwise bound of 1e-4 * scale everywhere
            assert (o['mean'] - ref['mean']).abs().max().item() < 1e-4 * scale, (r, name)
            assert (o['mean_square'] - ref['mean_square']).abs().max().item() < 3e-4 * scale ** 2, (r, name)
    assert torch.equal(img, blocks['b%d' % BLOCKS_RES][1])


def test_up_layer_is_the_composition_the_kernels_implement():
    """The stride-2 transposed conv as four parity-phase convolutions over the input grid
    (4 + 2 + 2 + 1 taps) followed by the 4x4 FIR -- the decomposition of csrc/nfi_synth.cu --
    equals conv_transpose2d + filter (stylegan.py:98-102)."""
    import torch.nn.functional as F
    torch.manual_seed(0)
    x = torch.randn(2, 8, 5, 7)
    w = torch.randn(6, 8, 3, 3)
    f = SO.fir_kernel()
    ref = F.conv_transpose2d(x, w.transpose(0, 1), stride=2)
    H, W = x.shape[2:]
    raw = torch.zeros(2, 6, 2 * H + 1, 2 * W + 1)
    xp = F.pad(x, (1, 1, 1, 1))
    for py in range(2):
        for px in range(2):
            DH, DW = (H if py else H + 1), (W if px else W + 1)
            acc = torch.zeros(2, 6, DH, DW)
            for ky in range(py, 3, 2):
                for kx in range(px, 3, 2):
                    dy, dx = -(ky // 2), -(kx // 2)
                    patch = xp[:, :, 1 + dy:1 + dy + DH, 1 + dx:1 + dx + DW]
                    acc += torch.einsum('bchw,oc->bohw', patch, w[:, :, ky, kx])
            raw[:, :, py::2, px::2] = acc
    assert (raw - ref).abs().max().item() < 1e-4
    # image upsampling weights of the ToRGB epilogue: out[2i] = 3/4 in[i] + 1/4 in[i-1], ...
    img = torch.randn(1, 3, 4, 4)
    up = SO.upsample_img(img, f)
    k = torch.tensor([0.25, 0.75, 0.75, 0.25])
    man = torch.zeros(1, 3, 8, 8)
    for u in range(8):
        for v in range(8):
            iy, ix = u // 2, v // 2
            jy, jx = (iy + 1 if u % 2 else iy - 1), (ix + 1 if v % 2 else ix - 1)
            val = 0.75 * 0.75 * img[:, :, iy, ix]
            if 0 <= jx < 4:
                val = val + 0.75 * 0.25 * img[:, :, iy, jx]
            if 0 <= jy < 4:
                val = val + 0.25 * 0.75 * img[:, :, jy, ix]
            if 0 <= jx < 4 and 0 <= jy < 4:
                val = val + 0.25 * 0.25 * img[:, :, jy, jx]
            man[:, :, u, v] = val
    assert (man - up).abs().max().item() < 1e-5
