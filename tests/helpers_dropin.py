"""A stand-in for the original project's ``Generator`` at the seam that
``nerf_from_image_b200.render`` reads (models/generator.py:407-502,587): EqualizedLinear decoder
layers (``weight * weight_gain``), ``beta`` / ``alpha``, a ViewDirectionMapper whose per-ray trunk
output ``x`` the mapper closure closes over, and a ``sampler`` closure over ``xy`` / ``xz`` / ``yz``
(views of one synthesis output), ``attention_values`` and ``viewdir_mapper_closure``.

It carries a ``fixtures.synthetic`` scene, as ``oracle.reference_lift.build_reference_generator``
loads one into the original module; what the original returned for the same scene is recorded in
tests/golden/reference/render_dropin.npz (tests/golden/make_golden_reference.py), and the recorder
checks that the effective weights of both are bit-identical."""
import math

import torch
from torch import nn

from oracle import render_oracle as O


class EqualizedLinear(nn.Module):
    """Holds ``effective / gain`` and uses ``weight * weight_gain`` (stylegan.py:148-180)."""

    def __init__(self, w_eff, b_eff=None):
        super().__init__()
        self.weight_gain = 1 / math.sqrt(w_eff.shape[1])
        self.bias_gain = 1
        self.weight = nn.Parameter(w_eff / self.weight_gain)
        self.bias = nn.Parameter(b_eff / self.bias_gain) if b_eff is not None else None


class ViewDirectionMapper(nn.Module):
    def __init__(self, m, w3, b3):
        super().__init__()
        for i in range(7):
            setattr(self, 'fc%d' % i, EqualizedLinear(m['fc%d_w' % i], m.get('fc%d_b' % i)))
        for i in range(1, 5):
            norm = nn.Module()
            norm.weight, norm.bias = nn.Parameter(m['norm%d_w' % i]), nn.Parameter(m['norm%d_b' % i])
            setattr(self, 'norm%d' % i, norm)
        self.output = EqualizedLinear(w3, b3)

    def effective(self):
        m = {}
        for i in range(7):
            fc = getattr(self, 'fc%d' % i)
            m['fc%d_w' % i] = fc.weight * fc.weight_gain
            if fc.bias is not None:
                m['fc%d_b' % i] = fc.bias * fc.bias_gain
        for i in range(1, 5):
            norm = getattr(self, 'norm%d' % i)
            m['norm%d_w' % i], m['norm%d_b' % i] = norm.weight, norm.bias
        return m

    def forward(self, viewdir):
        x = O.view_mapper_trunk(viewdir, self.effective())

        def mapper_closure(features):
            raise NotImplementedError('the per-sample mapper runs inside the fused kernels', x)
        return mapper_closure


class PlaneStub(nn.Module):
    """Synthesis network stand-in: returns the [B,96,R,R] planes it holds."""

    def __init__(self, planes):
        super().__init__()
        self.planes = planes

    def forward(self, ws, **kwargs):
        return self.planes


class SceneGenerator(nn.Module):
    def __init__(self, scene, use_sdf=True):
        super().__init__()
        B, _, C, R, _ = scene['planes'].shape
        self.attention_values = scene['palette'].shape[1] if scene['palette'] is not None else 0
        self.use_viewdir = 'view_mapper' in scene
        self.synthesis_network = PlaneStub(scene['planes'].reshape(B, 3 * C, R, R))
        self.decoder = nn.Module()
        self.decoder.net = nn.ModuleList([EqualizedLinear(scene['w1'], scene['b1']), nn.Softplus(),
                                          EqualizedLinear(scene['w2'], scene['b2'])])
        if use_sdf:
            self.beta = nn.Parameter(scene['beta'].view(1).clone())
            self.alpha = nn.Parameter(scene['alpha'].view(1).clone())
        if self.use_viewdir:
            self.viewdir_mapper = ViewDirectionMapper(scene['view_mapper'], scene['w3'], scene['b3'])

    def forward(self, viewdir, c, request_model_outputs=['sampler'], model_inputs={}):
        if self.attention_values > 0:
            attention_values = model_inputs['attention_values']
        if self.use_viewdir and viewdir is not None:
            viewdir_mapper_closure = self.viewdir_mapper(viewdir)
        planes = self.synthesis_network(c)
        planes = planes.view(c.shape[0], 3, 32, planes.shape[-2], planes.shape[-1])
        model_outputs = {}
        if 'attention_values' in request_model_outputs:
            model_outputs['attention_values'] = attention_values
        xy, xz, yz = planes[:, 0], planes[:, 1], planes[:, 2]

        def sampler(x_in, request_sampler_outputs=['sigma', 'rgb']):
            raise NotImplementedError('the fused renderer reads the closure, it does not call it',
                                      xy, xz, yz, attention_values, viewdir_mapper_closure)
        model_outputs['sampler'] = sampler
        return model_outputs


class RecordedFrontEnd:
    """The attributes ``generator.resolve_ws`` / ``resolve_palette`` read, with the mapping network
    and texture mapper answering from outputs recorded from the original modules."""
    use_encoder = False
    num_classes = 0

    def __init__(self, rec, z):
        self.attention_values = 10
        w_full = rec['w_full']

        def mapping_network(c, label):
            assert label is None and torch.equal(c, z)
            return w_full
        mapping_network.backbone = type('Backbone', (), {'num_ws': w_full.shape[1]})
        self.mapping_network = mapping_network
        self.textures = [(w_full[:, 14], rec['texture_w14']), (w_full[:, 0], rec['texture_w0'])]

    def texture_mapper(self, w):
        for w_in, out in self.textures:
            if torch.equal(w, w_in):
                return out
        raise AssertionError('texture mapper input not recorded')
