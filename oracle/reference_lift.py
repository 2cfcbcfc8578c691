"""Run the UNMODIFIED original project's hot path -- TEST / BASELINE INFRASTRUCTURE.

The original project is optional: ``build()`` stages the files used here, unmodified, from its
checkout into the git-ignored ``oracle/_ref/`` (``oracle/stage_reference.py``), and
``available()`` says whether they can be imported.  Callers
are the golden-data generators under ``tests/golden/``, the on-GPU drop-in tests that need the
original ``Generator`` module, and ``bench.py``'s reference legs (``--impl reference``,
``cpu_baseline``) -- never the product path.  No original source is copied into the
repository: ``render`` (run.py:176-350) is taken from the original file by AST at run
time (run.py itself cannot be imported -- it parses argv, loads datasets and
imports lpips/pytorch_fid at module level), and the radiance field is the
original's own ``models.generator.Generator`` whose synthesis network is
swapped for a stub that returns the planes under test.
"""

import ast
import os
import sys
import types
import warnings

import torch
import torch.nn.functional as F

_STAGED = os.path.join(os.path.dirname(os.path.abspath(__file__)), '_ref')


def _find_root():
    """NFI_REFERENCE_ROOT, else the copy build() staged, else the original checkout itself."""
    from oracle.stage_reference import DEFAULT_SOURCE
    for cand in (os.environ.get('NFI_REFERENCE_ROOT'), _STAGED, DEFAULT_SOURCE):
        if cand and os.path.isfile(os.path.join(cand, 'run.py')):
            return cand
    return _STAGED


REFERENCE_ROOT = _find_root()


def available():
    return os.path.isfile(os.path.join(REFERENCE_ROOT, 'run.py'))


def _import_reference():
    if REFERENCE_ROOT not in sys.path:
        sys.path.insert(0, REFERENCE_ROOT)
    with warnings.catch_warnings():
        warnings.simplefilter('ignore')
        from lib import nerf_utils  # noqa
        from models import generator  # noqa
    return nerf_utils, generator


def lift_render(scene_range, white_background, use_sdf=True,
                attention_values=10, fine_sampling=True, use_viewdir=False):
    """Returns the reference's ``render`` bound to the two module globals it
    reads (``args`` and ``dataset_config``; SURVEY.md section 1)."""
    nerf_utils, _ = _import_reference()
    with open(os.path.join(REFERENCE_ROOT, 'run.py')) as f:
        tree = ast.parse(f.read())
    fn = [n for n in tree.body
          if isinstance(n, ast.FunctionDef) and n.name == 'render'][0]
    ns = {
        'nerf_utils': nerf_utils, 'F': F, 'torch': torch,
        'args': types.SimpleNamespace(use_viewdir=use_viewdir, use_sdf=use_sdf,
                                      attention_values=attention_values,
                                      fine_sampling=fine_sampling),
        'dataset_config': {'scene_range': scene_range,
                           'white_background': white_background},
    }
    exec(compile(ast.Module(body=[fn], type_ignores=[]), 'run.py', 'exec'), ns)
    return ns['render']


class _PlaneStub(torch.nn.Module):
    """Stands in for SynthesisNetwork: returns the [B,96,R,R] planes given."""

    def __init__(self):
        super().__init__()
        self.planes = None

    def forward(self, ws, **kwargs):
        return self.planes


def build_reference_generator(scene, use_sdf=True):
    """Reference Generator carrying ``scene``'s decoder weights, beta/alpha (and, for a scene from
    ``fixtures.synthetic.add_view_mapper``, its ViewDirectionMapper: ``use_viewdir=True``).

    ``scene`` is a dict from ``fixtures.synthetic.make_scene``:
    effective decoder weights are divided by the EqualizedLinear gains so the
    reference module reproduces them (models/stylegan.py:168-177).
    """
    _, generator = _import_reference()
    A = scene['palette'].shape[1] if scene['palette'] is not None else 0
    vd = 'view_mapper' in scene
    g = generator.Generator(512, scene['scene_range'], attention_values=A,
                            use_sdf=use_sdf, disable_stylegan_noise=True, use_viewdir=vd)
    g.synthesis_network = _PlaneStub()
    l1, l2 = g.decoder.net[0], g.decoder.net[2]
    with torch.no_grad():
        if vd:
            vm, m = g.viewdir_mapper, scene['view_mapper']
            for i in range(7):
                fc = getattr(vm, 'fc%d' % i)
                fc.weight.copy_(m['fc%d_w' % i] / fc.weight_gain)
                if fc.bias is not None:
                    fc.bias.copy_(m['fc%d_b' % i] / fc.bias_gain)
            for i in range(1, 5):
                getattr(vm, 'norm%d' % i).weight.copy_(m['norm%d_w' % i])
                getattr(vm, 'norm%d' % i).bias.copy_(m['norm%d_b' % i])
            vm.output.weight.copy_(scene['w3'] / vm.output.weight_gain)
            vm.output.bias.copy_(scene['b3'] / vm.output.bias_gain)
        l1.weight.copy_(scene['w1'] / l1.weight_gain)
        l1.bias.copy_(scene['b1'] / l1.bias_gain)
        l2.weight.copy_(scene['w2'] / l2.weight_gain)
        l2.bias.copy_(scene['b2'] / l2.bias_gain)
        if use_sdf:
            g.beta.copy_(scene['beta'].view(1))
            g.alpha.copy_(scene['alpha'].view(1))
    g.eval()
    return g


def reference_render(scene, cams, height, width, num_samples, seed=None,
                     randomize=True, fine_sampling=True, use_sdf=True,
                     compute_normals=False, compute_semantics=False,
                     compute_coords=False, force_no_cam_grad=False,
                     generator=None, planes=None, palette=None):
    """Calls the lifted reference ``render``; returns (outputs, noise_t, noise_u).

    The reference draws its noise with ``torch.rand_like`` / ``torch.rand``
    inside TorchScript functions; seeding the default generator and replaying
    the same two draws afterwards reproduces the tensors (the stubbed
    generator forward consumes no random numbers in between).
    """
    A = scene['palette'].shape[1] if scene['palette'] is not None else 0
    render = lift_render(scene['scene_range'], scene['white_background'],
                         use_sdf=use_sdf, attention_values=A,
                         fine_sampling=fine_sampling, use_viewdir='view_mapper' in scene)
    g = generator if generator is not None else build_reference_generator(
        scene, use_sdf)
    planes = scene['planes'] if planes is None else planes
    palette = scene['palette'] if palette is None else palette
    B, _, C, R, _ = planes.shape
    g.synthesis_network.planes = planes.reshape(B, 3 * C, R, R)
    ws = torch.zeros(B, 15 if A > 0 else 14, 512)
    extra_in = {'attention_values': palette} if A > 0 else {}
    if seed is not None:
        torch.manual_seed(seed)
    out = render(g, height, width, cams['c2w'], cams['focal'], cams['center'],
                 cams['bbox'], ws, num_samples, randomize=randomize,
                 compute_normals=compute_normals,
                 compute_semantics=compute_semantics,
                 compute_coords=compute_coords,
                 extra_model_inputs=extra_in,
                 force_no_cam_grad=force_no_cam_grad)
    noise_t = noise_u = None
    if randomize and seed is not None:
        torch.manual_seed(seed)
        noise_t = torch.rand(B, height, width, num_samples)
        if fine_sampling:
            noise_u = torch.rand(B * height * width, num_samples)
    return out, noise_t, noise_u


def reference_sampler(scene, x_in, request, use_sdf=True, bbox_debug=False, generator=None):
    """Calls the reference Generator's own ``sampler`` closure
    (models/generator.py:587-681) at ``x_in`` [B, ..., S, 3]; returns its dict."""
    A = scene['palette'].shape[1] if scene['palette'] is not None else 0
    g = generator if generator is not None else build_reference_generator(scene, use_sdf)
    planes = scene['planes']
    B, _, C, R, _ = planes.shape
    g.synthesis_network.planes = planes.reshape(B, 3 * C, R, R)
    ws = torch.zeros(B, 15 if A > 0 else 14, 512)
    extra_in = {'attention_values': scene['palette']} if A > 0 else {}
    outputs = ['sampler'] + (['bbox'] if bbox_debug else [])
    closure = g(None, ws, request_model_outputs=outputs, model_inputs=extra_in)['sampler']
    return closure(x_in, request_sampler_outputs=list(request))


def reference_pose_utils():
    """The reference's lib.pose_utils module (lib/pose_utils.py)."""
    _import_reference()
    from lib import pose_utils  # noqa
    return pose_utils
