"""The sm_100a tri-plane producer (csrc/nfi_synth.cu through nfi_synthesis_forward) against
(1) the fixtures the reference produced, (2) the oracle restatement on a seeded mid-size
network, and (3) -- where the original project is staged (oracle/_ref) -- the UNMODIFIED
models.stylegan.SynthesisNetwork at the real size (256^2 planes, 512 channels), including RNG
consumption of the noise draws.  Bar: <= 1e-3 relative L2 (BASELINE north_star); 3xTF32 leaves
about 1e-6, the asserts use 5e-5."""
import pytest
import torch

from fixtures import synthetic
from oracle import reference_lift as RL
from oracle import synthesis_oracle as SO
from tests import helpers_synth as HS

pytestmark = pytest.mark.gpu
TOL = 5e-5


def _rel(a, b):
    return ((a - b).norm() / b.norm().clamp_min(1e-12)).item()


def _cf(planes_cl):
    from nerf_from_image_b200.synthesis import planes_channel_first
    return planes_channel_first(planes_cl)


@pytest.mark.parametrize('case', HS.CASES)
def test_fixtures(cuda_lib, case):
    from nerf_from_image_b200.synthesis import FusedSynthesis
    p, ws, img, mode = HS.load_case(case, 'cuda')
    fs = FusedSynthesis.from_params(p)
    with torch.no_grad():
        planes = fs(ws, noise_mode='const')
    assert planes.shape == (ws.shape[0], 3, 32, 32, 32) and planes.is_contiguous()
    assert _rel(_cf(planes), img) < TOL, _rel(_cf(planes), img)


@pytest.mark.parametrize('channels,batch', [((128, 128, 64, 32), 3), ((256, 128, 128, 96, 64), 2)])
def test_against_the_oracle(cuda_lib, channels, batch):
    """Ragged tile grids (4x4 .. 64x64 positions, batch 3), N tiles of 128 / 96 / 64 / 32,
    explicit noise on every layer."""
    from nerf_from_image_b200.synthesis import FusedSynthesis
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    res = 4 << (len(channels) - 1)
    p = synthetic.make_synthesis_params(5, res, channels, 512, 'cuda')
    ws = torch.randn(batch, 2 * len(channels), 512, generator=torch.Generator().manual_seed(6)).cuda()
    with torch.no_grad():
        ref = SO.synthesis_forward(p, ws, HS.const_noises(p))
        got = _cf(FusedSynthesis.from_params(p)(ws, noise_mode='const'))
    assert _rel(got, ref) < TOL, _rel(got, ref)


staged = pytest.mark.skipif(not RL.available(),
                            reason='original project not staged (oracle/_ref)')


@staged
def test_full_size_against_the_reference_module(cuda_lib):
    """256^2 x 96 planes from the 512-channel network of the p3d_car / cub / chairs configs
    (models/generator.py:366-372), eval mode."""
    from nerf_from_image_b200.synthesis import FusedSynthesis
    torch.backends.cuda.matmul.allow_tf32 = False   # run.py:59-60
    torch.backends.cudnn.allow_tf32 = False
    RL._import_reference()
    from models import stylegan
    torch.manual_seed(1234)
    net = stylegan.SynthesisNetwork(512, 256, 96).cuda().eval().requires_grad_(False)
    ws = torch.randn(2, net.num_ws, 512, device='cuda')
    with torch.no_grad():
        ref = net(ws)
        got = FusedSynthesis(net)(ws)
        truth = net.double()(ws.double())     # the module's own arithmetic in float64
        net.float()
    assert got.shape == (2, 3, 256, 256, 32)
    # the stated bar, against the reference as it runs (eager fp32, cuDNN)
    assert _rel(_cf(got), ref) < 1e-3, _rel(_cf(got), ref)
    # and against ground truth.  Measured r2: 1.35e-4 for this kernel, 3.8e-6 for cuDNN's fp32:
    # the 3xTF32 operands are exact to 2^-22, but the tensor core accumulates the 9 x 512 x 3
    # products of an output in ONE fp32 TMEM accumulator with truncating adds, a bias that grows
    # with K (the small-K decoder GEMMs of the render kernels are unaffected; DESIGN.md 4.8)
    e_ours, e_ref = _rel(_cf(got).double(), truth), _rel(ref.double(), truth)
    assert e_ours < 3e-4, (e_ours, e_ref)


@staged
def test_random_noise_draws_consume_the_generator_like_the_reference(cuda_lib):
    from nerf_from_image_b200.synthesis import FusedSynthesis
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    RL._import_reference()
    from models import stylegan
    torch.manual_seed(7)
    net = stylegan.SynthesisNetwork(512, 64, 96, channel_base=8192, channel_max=128).cuda()
    net.requires_grad_(False)
    with torch.no_grad():
        for n, q in net.named_parameters():
            if n.endswith('noise_strength'):
                q.fill_(0.1)
    net.train()   # training mode draws noise for every layer (stylegan.py:332-337)
    ws = torch.randn(2, net.num_ws, 512, device='cuda')
    with torch.no_grad():
        torch.manual_seed(99)
        ref = net(ws, noise_mode='random')
        s_ref = torch.cuda.get_rng_state()
        torch.manual_seed(99)
        got = FusedSynthesis(net)(ws, noise_mode='random')
        s_got = torch.cuda.get_rng_state()
    assert torch.equal(s_ref, s_got)
    assert _rel(_cf(got), ref) < TOL


def test_forward_only_and_no_cpu_path(cuda_lib):
    from nerf_from_image_b200 import _lib
    from nerf_from_image_b200.synthesis import FusedSynthesis
    p, ws, img, mode = HS.load_case(HS.CASES[0], 'cuda')
    fs = FusedSynthesis.from_params(p)
    with pytest.raises(_lib.NfiError):
        fs(ws.clone().requires_grad_())
    with pytest.raises(_lib.NfiError):
        with torch.no_grad():
            fs(ws.cpu())
