"""CPU/torch restatement of the reference's plane producer -- TEST INFRASTRUCTURE.

The StyleGAN2 synthesis network that ``Generator.forward`` runs to produce the tri-planes
(/root/reference/models/generator.py:475-477 -> models/stylegan.py:438-490), restated as plain
functions over a flat parameter dict so that it can be compared stage by stage with the
sm_100a kernels of ``nerf_from_image_b200/csrc/nfi_synth.cu`` (SURVEY.md section 8f, N1).
Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s reference legs import it.

Pinned to the reference: ``tests/test_synthesis_oracle.py`` runs the UNMODIFIED
``models.stylegan.SynthesisNetwork`` (imported from the staged
``oracle/_ref``) on the same weights and latents and compares every block; the fixtures under
``tests/golden/synth/`` were produced by the reference (``tests/golden/make_golden_synth.py``).

Per layer (models/stylegan.py:114-145 ``conv_modulated2d``, :293-356 ``SynthesisLayer``):
    s      = affine(w)                      EqualizedLinear 512 -> Cin, bias init 1   (:148-180)
    d[b,o] = rsqrt(sum_{i,k} (W[o,i,k] s[b,i])^2 + 1e-8)
    x      = x * s                          activations scaled, weights shared by the batch
    x      = conv3x3(x, W, pad 1)           or, with up: conv_transpose2d(stride 2) followed by
                                            the [1,3,3,1]x[1,3,3,1]/64 FIR with gain 4, pad 1 (:98-102)
    x      = x * d + noise                  (addcmul; noise = randn * noise_strength or absent)
    x      = leaky_relu((x + bias) * sqrt(2), 0.2)
ToRGB (:359-380): 1x1 modulated conv without demodulation, styles * 1/sqrt(Cin), + bias; the
running image is FIR-upsampled (:71-75) and the block's ToRGB output added (:420-435).
"""
import math

import torch
import torch.nn.functional as F


def fir_kernel(device=None, dtype=torch.float32):
    """models/stylegan.py:48-52: outer([1,3,3,1]) normalised to sum 1."""
    h = torch.tensor([1., 3., 3., 1.], device=device, dtype=dtype)
    h = h[:, None] * h[None, :]
    return h / h.sum()


def block_resolutions(img_resolution):
    return [2 ** i for i in range(2, int(math.log2(img_resolution)) + 1)]


def extract_params(net):
    """Flat dict of the tensors of a reference ``SynthesisNetwork`` (or anything with the same
    attribute layout): ``params['b8.conv0.weight']`` etc., plus static ints under ``'meta'``."""
    p = {k: v.detach() for k, v in net.state_dict().items()}
    res = block_resolutions(net.img_resolution)
    layers = {}
    for r in res:
        blk = getattr(net, 'b%d' % r)
        for name in ('conv0', 'conv1'):
            if hasattr(blk, name):
                layer = getattr(blk, name)
                layers['b%d.%s' % (r, name)] = dict(use_noise=bool(layer.use_noise), up=bool(layer.up))
    p['meta'] = dict(img_resolution=net.img_resolution, img_channels=net.img_channels,
                     w_dim=net.w_dim, resolutions=res, layers=layers)
    return p


def affine(p, prefix, w):
    """EqualizedLinear(w_dim, Cin, init_bias_one): weight / sqrt(w_dim), bias (lr multiplier 1)."""
    wt = p[prefix + '.affine.weight']
    return F.linear(w, wt * (1.0 / math.sqrt(wt.shape[1])), p[prefix + '.affine.bias'])


def upsample_img(img, f):
    """models/stylegan.py:71-75: zero-insertion x2 then the FIR with gain 4 (one transposed conv)."""
    B, C, H, W = img.shape
    y = F.conv_transpose2d(img.reshape(B * C, 1, H, W), (f * 4)[None, None], stride=2, padding=1)
    return y.view(B, C, y.shape[2], y.shape[3])


def modulated_conv(x, weight, styles, noise, up, f):
    B = x.shape[0]
    wmod = weight.unsqueeze(0) * styles.reshape(B, 1, -1, 1, 1)
    dcoef = (wmod.square().sum(dim=[2, 3, 4]) + 1e-8).rsqrt()
    x = x * styles.reshape(B, -1, 1, 1)
    if up:
        x = F.conv_transpose2d(x, weight.transpose(0, 1), stride=2)
        C = x.shape[1]
        x = F.conv2d(x.reshape(B * C, 1, x.shape[2], x.shape[3]), (f * 4)[None, None], padding=1)
        x = x.view(B, C, x.shape[2], x.shape[3])
    else:
        x = F.conv2d(x, weight, padding=weight.shape[-1] // 2)
    x = x * dcoef.reshape(B, -1, 1, 1)
    if noise is not None:
        x = x + noise
    return x


def synthesis_layer(p, prefix, x, w, noise, up, f):
    s = affine(p, prefix, w)
    x = modulated_conv(x, p[prefix + '.weight'], s, noise, up, f)
    x = (x + p[prefix + '.bias'].view(1, -1, 1, 1)) * math.sqrt(2)
    return F.leaky_relu(x, 0.2)


def to_rgb(p, prefix, x, w):
    wt = p[prefix + '.weight']
    s = affine(p, prefix, w) * (1.0 / math.sqrt(wt.shape[1]))
    y = F.conv2d(x * s.reshape(x.shape[0], -1, 1, 1), wt)
    return y + p[prefix + '.bias'].view(1, -1, 1, 1)


def synthesis_forward(p, ws, noises=None, return_blocks=False):
    """ws [B, num_ws, 512] -> img [B, img_channels, R, R] (channel-first, as the reference).

    ``noises``: optional dict ``{'b8.conv0': [B,1,8,8] tensor ALREADY multiplied by
    noise_strength, ...}`` standing in for the ``torch.randn`` draws of :334-340; a missing key
    means no noise for that layer (eval mode with strength 0, or ``disable_stylegan_noise``)."""
    meta = p['meta']
    f = fir_kernel(ws.device, ws.dtype)
    noises = noises or {}
    x = img = None
    w_idx = 0
    blocks = {}
    for r in meta['resolutions']:
        pre = 'b%d' % r
        if r == 4:
            x = p[pre + '.const'].unsqueeze(0).repeat(ws.shape[0], 1, 1, 1)
            n_conv = 1
        else:
            x = synthesis_layer(p, pre + '.conv0', x, ws[:, w_idx], noises.get(pre + '.conv0'),
                                True, f)
            n_conv = 2
        x = synthesis_layer(p, pre + '.conv1', x, ws[:, w_idx + n_conv - 1],
                            noises.get(pre + '.conv1'), False, f)
        y = to_rgb(p, pre + '.torgb', x, ws[:, w_idx + n_conv])
        img = y if img is None else upsample_img(img, f) + y
        w_idx += n_conv
        if return_blocks:
            blocks[pre] = (x, img)
    return (img, blocks) if return_blocks else img
