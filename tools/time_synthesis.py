"""Times the plane producer at BASELINE config-2 size (B images, 256^2 x 96 planes, 512-channel
StyleGAN2 synthesis): the sm_100a kernels (FusedSynthesis) and, where the reference files are
staged, the reference module in PyTorch eager fp32 (TF32 off, run.py:59-60) on the same GPU.
Usage: python tools/time_synthesis.py [batch] [steps]"""
import sys
import torch
sys.path.insert(0, '.')
from oracle import reference_lift as RL
from nerf_from_image_b200.synthesis import FusedSynthesis
torch.backends.cuda.matmul.allow_tf32 = False
torch.backends.cudnn.allow_tf32 = False
B = int(sys.argv[1]) if len(sys.argv) > 1 else 32
K = int(sys.argv[2]) if len(sys.argv) > 2 else 5
if not RL.available():
    raise SystemExit('original project not staged (oracle/_ref)')
RL._import_reference()
from models import stylegan
torch.manual_seed(1234)
net = stylegan.SynthesisNetwork(512, 256, 96).cuda().eval().requires_grad_(False)
ws = torch.randn(B, net.num_ws, 512, device='cuda')
fs = FusedSynthesis(net)
# dense FLOPs of the convolutions as executed (transposed convs on the input grid)
ch = [min(32768 // r, 512) for r in net.block_resolutions]
fl = 0
for i, r in enumerate(net.block_resolutions):
    if i:
        fl += 2 * ch[i - 1] * ch[i] * 9 * (r // 2) ** 2
    fl += 2 * ch[i] * ch[i] * 9 * r * r + 2 * ch[i] * 96 * r * r
def timeit(fn, n):
    for _ in range(2):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / n
with torch.no_grad():
    ms = timeit(lambda: fs(ws), K)
    print('fused synthesis   B=%d: %.2f ms per forward  (%.1f images/s, %.1f TFLOP/s dense fp32-equivalent, %.2f GFLOP/image)'
          % (B, ms, B / ms * 1e3, B * fl / ms / 1e9, fl / 1e9))
    try:
        ms_r = timeit(lambda: net(ws), max(2, K // 2))
        print('reference eager   B=%d: %.2f ms per forward  (%.1f images/s)  -> %.2fx' % (B, ms_r, B / ms_r * 1e3, ms_r / ms))
    except Exception as e:
        print('reference eager: unavailable', repr(e)[:120])
    torch.cuda.empty_cache()
    print('peak memory %.1f GB' % (torch.cuda.max_memory_allocated() / 2 ** 30))
