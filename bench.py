#!/usr/bin/env python
"""Benchmark of the fused tri-plane render (BASELINE.json metric: rays/s at 128x128, 64 coarse +
64 fine samples per ray).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
                    [--config 2|3|4|5] [--scaling weak|strong]

Workloads (BASELINE.json `configs`):
  --config 2 (default)  p3d_car generator forward: batch 32 per GPU, 256^2 x 32ch fp32 tri-planes
             -> 128x128 rays x (64 + 64) samples -> rgb / depth / mask.
               value     render with the planes resident in HBM in the layout the sm_100a plane
                         producer emits (channel-last), CUDA events, max over ranks
               e2e       w -> image through the public API: latents in pinned host memory -> H2D
                         -> synthesis network (tcgen05 kernels) -> render -> D2H of rgb/depth/mask
               roofline  render_forward_pipe against the algorithmic tensor-FLOP bound (SURVEY 8d)
               cpu_baseline / --impl reference: the reference's own render on the host cores
  --config 3  cub --run_inversion: orthographic, scene_range 2, GLOBAL batch 16 sharded over the
             GPUs (4 images per GPU at N=4), 30 steps of forward + backward (gradients to planes,
             palette, pose), rays/s of forward+backward.
  --config 4  shapenet_chairs GAN generator step on the path: global batch 32, forward + backward
             with decoder-weight / beta / alpha gradients too, all-reduce of those gradients.
  --config 5  inversion sweep: resolution {128, 256} x samples/ray {32, 64, 128}, forward and
             forward+backward, 8 images per GPU; one JSON line with a `sweep` list.
--scaling strong (config 2): global batch 32 split over the GPUs instead of 32 per GPU.

Inputs (>= 0.8 GB per GPU at config 2) are far larger than the 126 MB L2, so consecutive steps
cannot be served from cache.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'rays_per_sec_128x128_64+64spp'
UNIT = 'rays/s'
CFG = dict(batch=32, height=128, width=128, samples=64, plane_res=256, attention_values=10,
           dataset='p3d_car')
FLOPS_PER_POINT = 2 * 32 * 64 + 2 * 64 * 11 + 2 * 10 * 3  # 5,564 (SURVEY.md 8d)
WORKLOADS = {
    2: 'config 2: p3d_car generator forward, render 128x128, 64 coarse + 64 fine samples/ray, '
       'batch %d per GPU, 256^2x32ch fp32 tri-planes -> rgb/depth/mask',
    3: 'config 3: cub --run_inversion step (orthographic, scene_range 2.0): render forward + '
       'backward (grads to planes, palette, tform_cam2world), 128x128, 64+64 samples/ray, GLOBAL '
       'batch %d sharded over the GPUs',
    4: 'config 4: shapenet_chairs GAN generator step on the render path: forward + backward incl. '
       'decoder-weight / beta / alpha gradients + their all-reduce, 128x128, 64+64 samples/ray, '
       'GLOBAL batch %d sharded over the GPUs',
    5: 'config 5: p3d_car inversion sweep, resolution {128,256} x samples/ray {32,64,128}, %d '
       'images per GPU, forward and forward+backward',
}


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(path):
        p = json.load(open(path))
        return dict(hbm_gbs=p['hbm_gbs'], tflops=p.get('bf16_tflops_sustained', p['bf16_tflops']),
                    source='measured (MEASURED_PEAKS.json, bf16 sustained)')
    return dict(hbm_gbs=6650.0, tflops=1590.0, source='fallback (B200_PROFILING.md)')


def measured_traffic(kernel, batch):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` from the committed
    `ncu --set full` capture (profiles/traffic.json: written from the raw csv by
    tools/ncu_summary.py); None when no capture of this batch size exists."""
    path = os.path.join(ROOT, 'profiles', 'traffic.json')
    if not os.path.isfile(path):
        return None, None
    for row in json.load(open(path)):
        if row['kernel'] == kernel and row['batch'] == batch:
            return row['dram_bytes'], row['source']
    return None, None


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons sampled DURING the timed region (NVML, every ~10 ms; falls
    back to nvidia-smi if pynvml is missing)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False
        self.max_mhz = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nvml = None

    def run(self):
        while not self.stop_flag:
            try:
                if self.nvml is not None:
                    n = self.nvml
                    mhz = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
                    bits = n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)
                    self.rows.append((mhz, bits))
                    time.sleep(0.01)
                else:
                    q = 'clocks.sm,clocks.max.sm,clocks_event_reasons.active'
                    out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q,
                                          '--format=csv,noheader,nounits'], capture_output=True,
                                         text=True, timeout=5).stdout.strip().split(',')
                    self.max_mhz = int(out[1])
                    self.rows.append((int(out[0]), int(out[2], 16)))
            except Exception:
                time.sleep(0.05)

    def summary(self):
        self.stop_flag = True
        self.join(timeout=6)
        if not self.rows:
            return dict(sm_mhz=None, sm_max_mhz=self.max_mhz, reasons=['unsampled'])
        sm = sorted(r[0] for r in self.rows)
        names = {0x8: 'hw_slowdown', 0x40: 'hw_thermal_slowdown', 0x20: 'sw_thermal_slowdown',
                 0x4: 'sw_power_cap'}
        seen = 0
        for _, bits in self.rows:
            seen |= bits
        return dict(sm_mhz=sm[len(sm) // 2], sm_max_mhz=self.max_mhz,
                    reasons=[n for b, n in names.items() if seen & b], samples=len(self.rows))


# ------------------------------------------------------------------ the reference on the host
def _cpu_case(n_images):
    from fixtures import synthetic
    ds = synthetic.DATASET_CONFIGS[CFG['dataset']]
    scene = synthetic.make_scene(1234, n_images, plane_res=CFG['plane_res'],
                                 attention_values=CFG['attention_values'],
                                 scene_range=ds['scene_range'],
                                 white_background=ds['white_background'])
    cams = synthetic.make_cameras(1234, n_images, radius=ds['radius'])
    nt, nu = synthetic.make_noise(1234, n_images, CFG['height'], CFG['width'], CFG['samples'])
    return scene, cams, nt, nu


def reference_kind():
    """'reference' when the unmodified original project can run here (staged into oracle/_ref
    by build() from the original checkout), else 'port' (the oracle)."""
    from oracle import reference_lift as RL
    return 'reference' if RL.available() else 'port'


def cpu_render(case, kind, seed=77):
    """One pass of the reference's render on the host cores; returns (seconds, rgb)."""
    scene, cams, nt, nu = case
    H, W, S = CFG['height'], CFG['width'], CFG['samples']
    t0 = time.perf_counter()
    with torch.no_grad():
        if kind == 'reference':
            # run.py:176-350 lifted by AST, reference Generator carrying the scene's decoder,
            # planes given (its synthesis network is the NEXT row of SURVEY.md section 8)
            from oracle import reference_lift as RL
            out, _, _ = RL.reference_render(scene, cams, H, W, S, seed=seed, generator=case_generator(case))
            rgb = out[0]
        else:
            from oracle import render_oracle as O
            rgb = O.render_oracle(scene['planes'], scene['w1'], scene['b1'], scene['w2'],
                                  scene['b2'], scene['palette'], scene['beta'], scene['alpha'],
                                  cams['c2w'], cams['focal'], None, None, H, W, S, nt, nu,
                                  scene_range=scene['scene_range'],
                                  white_background=scene['white_background'])['rgb']
    return time.perf_counter() - t0, rgb


_GEN = {}


def case_generator(case):
    from oracle import reference_lift as RL
    key = id(case[0])
    if key not in _GEN:
        _GEN[key] = RL.build_reference_generator(case[0])
    return _GEN[key]


def best_cpu_threads(kind):
    """The reference's CPU path is plain PyTorch; its intra-op scaling saturates well before all
    cores of a big host, so probe a few thread counts on a small sample of the same workload and
    keep the fastest (reported as `cores`)."""
    from fixtures import synthetic
    from oracle import render_oracle as O
    ds = synthetic.DATASET_CONFIGS[CFG['dataset']]
    scene = synthetic.make_scene(7, 1, plane_res=64, scene_range=ds['scene_range'])
    cams = synthetic.make_cameras(7, 1, radius=ds['radius'])
    nt, nu = synthetic.make_noise(7, 1, 32, 32, 32)
    total = os.cpu_count() or 1
    best, best_t = total, None
    for th in sorted({t for t in (8, 16, 32, 64, total) if t <= total}):
        torch.set_num_threads(th)
        ts = []
        for _ in range(3):
            t0 = time.perf_counter()
            with torch.no_grad():
                O.render_oracle(scene['planes'], scene['w1'], scene['b1'], scene['w2'],
                                scene['b2'], scene['palette'], scene['beta'], scene['alpha'],
                                cams['c2w'], cams['focal'], None, None, 32, 32, 32, nt, nu,
                                scene_range=scene['scene_range'])
            ts.append(time.perf_counter() - t0)
        if best_t is None or min(ts) < best_t:
            best, best_t = th, min(ts)
    torch.set_num_threads(best)
    return best


def config_block(args, world, batch_per_gpu, global_batch):
    """The same for both arms (the driver compares the two lines' `config`)."""
    return {'workload': WORKLOADS[args.config] % (global_batch if args.config in (3, 4) else batch_per_gpu),
            'global_batch': global_batch, 'scaling': args.scaling,
            'parallelism': 'images sharded over the GPUs, all_gather of [rgb,depth,mask] tiles '
                           'when N > 1 (the reference arm runs on host CPU cores, rank 0 only)',
            'cache': 'inputs larger than L2; no flush needed', 'randomize': True}


def run_reference(args):
    """--impl reference: the reference's own CPU path on the host cores, bounded sample."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    kind = reference_kind()
    threads = best_cpu_threads(kind)
    n_img = 1
    case = _cpu_case(n_img)
    for _ in range(max(1, args.warmup)):
        cpu_render(case, kind)
    times = [cpu_render(case, kind)[0] for _ in range(args.steps)]
    rays = n_img * CFG['height'] * CFG['width']
    total = sum(times)
    value = rays * len(times) / total
    B = args.batch or CFG['batch']
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT,
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': 1e3 * total / len(times), 'higher_is_better': True, 'scaling': args.scaling,
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': config_block(args, args.gpus, B, args.gpus * B if args.scaling == 'weak' else B),
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': threads,
                         'host_cores': os.cpu_count(), 'kind': kind,
                         'sample': '%d image(s) of the batch per step (same geometry; images are '
                                   'independent, the rate is per ray), torch CPU fp32, no_grad; %s'
                                   % (n_img, 'unmodified reference render (run.py:176-350 lifted '
                                      'from oracle/_ref), planes given' if kind == 'reference'
                                      else 'oracle port of the reference ops')},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line))


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, outputs):
    """Writes each [batch, ...] output as out_dir/<name>.npy in float32, so that two builds can be
    compared output for output on the same seeded inputs.  Past DUMP_LIMIT_BYTES in all, only the
    leading images of the batch are written (the same ones every run)."""
    import numpy as np
    per_image = sum(t[0].numel() for t in outputs.values()) * 4
    keep = max(1, min(min(len(t) for t in outputs.values()), DUMP_LIMIT_BYTES // per_image))
    os.makedirs(out_dir, exist_ok=True)
    for name, t in outputs.items():
        np.save(os.path.join(out_dir, name + '.npy'), t[:keep].detach().float().cpu().numpy())


# ------------------------------------------------------------------ the B200 arm
class Bench:
    def __init__(self, args):
        import torch.distributed as dist
        from nerf_from_image_b200 import _lib, fused, parallel
        from fixtures import synthetic
        self.args, self.dist, self.fused, self.parallel, self.synthetic = args, dist, fused, parallel, synthetic
        self._lib = _lib
        self.world = int(os.environ.get('WORLD_SIZE', '1'))
        self.rank = int(os.environ.get('RANK', '0'))
        self.local_rank = int(os.environ.get('LOCAL_RANK', '0'))
        if not torch.cuda.is_available():
            raise SystemExit('bench.py needs a CUDA device: the fused renderer has no CPU path')
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device('cuda', self.local_rank)
        if self.world > 1:
            dist.init_process_group('nccl', device_id=self.dev)
        self.lib = _lib.load()

    # -------------------------------------------------------------- helpers
    def barrier(self):
        torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()

    def max_over_ranks(self, x):
        if self.world == 1:
            return x
        t = torch.tensor([x], device=self.dev, dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.item()

    def min_over_ranks(self, x):
        if self.world == 1:
            return x
        t = torch.tensor([float(x)], device=self.dev, dtype=torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return t.item()

    def timed(self, fn, steps, warmup):
        for _ in range(warmup):
            fn()
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        self.barrier()
        return self.max_over_ranks(e0.elapsed_time(e1)) / steps

    def scene(self, dataset, batch, seed, H, W, S, res=None, layout='channel_last'):
        syn = self.synthetic
        ds = syn.DATASET_CONFIGS[dataset]
        sc = syn.make_scene(seed, batch, plane_res=res or CFG['plane_res'],
                            attention_values=CFG['attention_values'], scene_range=ds['scene_range'],
                            white_background=ds['white_background'],
                            object_radius=ds['object_radius'], device=self.dev)
        if layout == 'channel_last':   # what the sm_100a plane producer emits
            sc['planes'] = sc['planes'].permute(0, 1, 3, 4, 2).contiguous()
        cams = syn.make_cameras(seed, batch, ortho=ds['ortho'], radius=ds['radius'], device=self.dev)
        nt, nu = syn.make_noise(seed, batch, H, W, S, device=self.dev)
        cfg = self.fused.RenderConfig(scene_range=sc['scene_range'],
                                      white_background=sc['white_background'],
                                      attention_values=CFG['attention_values'],
                                      mlp_mode=self.args.mlp_mode)
        return sc, cams, nt, nu, cfg

    def render(self, sc, cams, nt, nu, cfg, H, W, S, out=None, layout='channel_last', peers=None,
               **leaves):
        g = lambda k: leaves.get(k, sc[k] if k in sc else cams[k])
        return self.fused.fused_render(
            g('planes'), g('w1'), g('b1'), g('w2'), g('b2'), g('palette'), g('beta'), g('alpha'),
            g('c2w'), cams['focal'], None, None, cfg, H, W, S, nt, nu, out=out,
            planes_layout=layout, peers=peers)

    # -------------------------------------------------------------- config 2
    def config2(self):
        a, world, rank, dev = self.args, self.world, self.rank, self.dev
        fused, parallel, dist = self.fused, self.parallel, self.dist
        H, W, S = CFG['height'], CFG['width'], CFG['samples']
        if a.scaling == 'strong':
            gb = a.batch or CFG['batch']
            if gb % world:
                raise SystemExit('--scaling strong needs batch %% gpus == 0')
            B = gb // world
        else:
            B = a.batch or CFG['batch']
            gb = world * B
        sc, cams, nt, nu, cfg = self.scene(CFG['dataset'], B, 1234 + rank, H, W, S)
        kernel_events = []
        gather_events = []

        # N > 1: the exchange fused into the kernel where symmetric memory is available on this
        # box ('auto' falls back to the in-place NCCL all-gather, and says so in `exchange`)
        peer_ex, exchange_note = None, ('nccl' if world > 1 else None)
        if world > 1 and a.exchange in ('peer', 'auto'):
            try:
                peer_ex = parallel.PeerExchange(gb, H, W, dev)
                ok, why = 1.0, ''
            except Exception as exc:
                ok, why = 0.0, repr(exc)[:120]
            if self.min_over_ranks(ok) < 1.0:
                if a.exchange == 'peer':
                    raise SystemExit('--exchange peer: symmetric memory unavailable: ' + why)
                peer_ex, exchange_note = None, 'nccl (peer exchange unavailable: %s)' % why
            else:
                exchange_note = 'peer'

        def step(time_kernel=False):
            with torch.no_grad():
                if time_kernel:
                    fused.KERNEL_EVENTS = kernel_events
                out = full = peers = None
                if peer_ex is not None:
                    # the exchange fused into the kernel: tiles stored into every rank's buffers
                    # over NVLink (symmetric memory), one device-side barrier, no collective call
                    full, out, peers = peer_ex.begin()
                elif world > 1:
                    # the path's one exchange step, in place: the kernel writes this rank's tiles
                    # into its slice of the full-batch buffers, one NCCL launch all-gathers them
                    full = parallel.gathered_buffers(gb, H, W, dev)
                    out = parallel.shard_views(full, gb, world, rank)
                res = self.render(sc, cams, nt, nu, cfg, H, W, S, out=out, peers=peers)
                fused.KERNEL_EVENTS = None
                if world > 1:
                    if time_kernel:
                        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        g0.record()
                    if peer_ex is not None:
                        peer_ex.finish()
                        res = full
                    else:
                        res = parallel.all_gather_inplace(full, gb)
                    if time_kernel:
                        g1.record()
                        gather_events.append((g0, g1))
            return res[:3]

        for _ in range(a.warmup):
            step()
        self.barrier()
        sampler = ClockSampler(self.local_rank)
        if rank == 0:
            sampler.start()
        torch.cuda.synchronize()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        for _ in range(a.steps):
            last = step(time_kernel=True)
        ev1.record()
        self.barrier()
        clocks = sampler.summary() if rank == 0 else None
        ms_step = self.max_over_ranks(ev0.elapsed_time(ev1)) / a.steps
        if a.dump_outputs and rank == 0:
            dump_outputs(a.dump_outputs, dict(zip(('rgb', 'depth', 'mask'), last)))
        rays_step = gb * H * W
        value = rays_step / (ms_step * 1e-3)
        k_ms = sum(x.elapsed_time(y) for x, y in kernel_events) / max(1, len(kernel_events))
        coll_ms = (self.max_over_ranks(sum(x.elapsed_time(y) for x, y in gather_events)
                                       / max(1, len(gather_events))) if world > 1 else None)

        # ---- N > 1: the gathered buffers are checked, not assumed
        gathered = None
        if world > 1:
            with torch.no_grad():
                mine = self.render(sc, cams, nt, nu, cfg, H, W, S)
                a0, b0 = parallel.shard_range(gb, world, rank)
                own_ok = all(torch.equal(x[a0:b0], y) for x, y in zip(last, mine[:3]))
                # every rank re-renders its right-hand neighbour's images from that rank's seed
                peer = (rank + 1) % world
                scp, cmp_, ntp, nup, cfgp = self.scene(CFG['dataset'], B, 1234 + peer, H, W, S)
                theirs = self.render(scp, cmp_, ntp, nup, cfgp, H, W, S)
                a1, b1 = parallel.shard_range(gb, world, peer)
                peer_ok = all(torch.equal(x[a1:b1], y) for x, y in zip(last, theirs[:3]))
                del scp, ntp, nup, theirs
            gathered = {'own_slice_bit_exact_on_every_rank': bool(self.min_over_ranks(own_ok)),
                        'neighbour_slice_bit_exact_on_every_rank': bool(self.min_over_ranks(peer_ok)),
                        'how': 'after the timed steps each rank compares its slice of the '
                               'all-gathered rgb/depth/mask with a private render, and the slice of '
                               'rank+1 with a local render of that rank\'s seeded inputs'}

        # ---- e2e: w -> image through the public API, host latents in, host image out
        e2e = self.e2e_generator_forward(B, gb, H, W, S) if not a.no_e2e else None
        e2e_planes = self.e2e_planes_from_host(sc, cams, cfg, B, gb, H, W, S) \
            if not (a.no_e2e or a.quick) else None

        # ---- render with channel-first planes (the reference module's layout): re-layout pass
        cf = None
        if not a.quick:
            sc_cf = dict(sc, planes=sc['planes'].permute(0, 1, 4, 2, 3).contiguous())
            with torch.no_grad():
                ms_cf = self.timed(lambda: self.render(sc_cf, cams, nt, nu, cfg, H, W, S,
                                                       layout='channel_first'), 5, 2)
            cf = {'value': B * world * H * W / (ms_cf * 1e-3) if a.scaling == 'weak'
                  else gb * H * W / (ms_cf * 1e-3), 'unit': UNIT, 'ms_per_step': ms_cf,
                  'what': 'same render fed with [B,3,32,R,R] planes as the reference synthesis '
                          'module leaves them: + nfi_planes_to_channel_last (1.6 GB moved)'}
            del sc_cf
            torch.cuda.empty_cache()

        fwd_bwd = self.fwd_bwd(sc, cams, nt, nu, cfg, H, W, S, gb) if not a.no_backward else None
        pretrained = self.fixture_pretrained(B, H, W, S) if (world == 1 and not a.quick
                                                             and not a.no_cpu_baseline) else None
        if rank != 0:
            return
        pk = peaks()
        flops_launch = float(B * H * W) * (2 * S) * FLOPS_PER_POINT
        hbm_bytes_launch = float(B) * 3 * 32 * CFG['plane_res'] ** 2 * 4 + B * H * W * 20.0
        achieved_tf = flops_launch / (k_ms * 1e-3) / 1e12 if k_ms > 0 else 0.0
        traffic, traffic_src = measured_traffic('render_forward_pipe', B)
        roofline = {
            'bound': 'tensor', 'achieved': achieved_tf, 'peak': pk['tflops'], 'unit': 'TFLOP/s',
            'frac': achieved_tf / pk['tflops'], 'traffic': traffic, 'traffic_source': traffic_src,
            'kernel': 'render_forward_pipe (dominant kernel of the step)', 'kernel_ms': k_ms,
            'kernel_share_of_step': k_ms / ms_step if ms_step > 0 else None,
            'algorithmic_flops_per_launch': flops_launch,
            'algorithmic_hbm_bytes_per_launch': hbm_bytes_launch,
            'hbm_achieved_gbs': hbm_bytes_launch / (k_ms * 1e-3) / 1e9 if k_ms > 0 else 0.0,
            'hbm_peak_gbs': pk['hbm_gbs'], 'peak_source': pk['source'],
        }
        if fwd_bwd is not None:
            # the backward sweep re-runs the two layers and adds dL/dH = dOut W2 (2 x 11 x 64) and
            # dL/dF = dpre W1 (2 x 64 x 32) per point: 5,504 FLOPs on top of the recompute's 5,564
            bwd_flops = float(B * H * W) * (2 * S) * (FLOPS_PER_POINT + 5504.0)
            step_s = fwd_bwd['ms_per_step'] * 1e-3
            ach = (flops_launch + bwd_flops) / step_s / 1e12
            fwd_bwd['roofline'] = {
                'bound': 'tensor', 'achieved': ach, 'peak': pk['tflops'], 'unit': 'TFLOP/s',
                'frac': ach / pk['tflops'],
                'algorithmic_flops_per_step': flops_launch + bwd_flops,
                'what': 'render_forward_pipe + render_backward_pipe (pose gradients on) of one '
                        'inversion step; the backward is bound by its three line-rate passes per '
                        'point -- gather, red.global.add.v4 scatter, pose re-read (DESIGN.md 8.2)'}
        cpu_baseline = parity = eager = None
        if world == 1 and not a.no_cpu_baseline:
            cpu_baseline, parity = self.cpu_baseline_and_parity(cfg, H, W, S)
            eager = self.eager_gpu(H, W, S)
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': a.steps,
            'warmup': a.warmup, 'ms_per_step': ms_step, 'higher_is_better': True,
            'scaling': a.scaling, 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': config_block(a, world, B, gb),
            'clocks': clocks, 'e2e': e2e,
            # per step: prep_weight_image, render_forward_pipe
            'gpu_launches': 2 * a.steps,
            'roofline': roofline, 'fwd_bwd': fwd_bwd, 'cpu_baseline': cpu_baseline,
            'torch_eager_gpu': eager, 'parity': parity, 'gathered_check': gathered,
            'collective_ms': coll_ms, 'exchange': exchange_note,
            'render_from_channel_first_planes': cf,
            'e2e_planes_from_host': e2e_planes, 'fixture_pretrained_generator': pretrained,
        }
        print(json.dumps(line))

    def e2e_generator_forward(self, B, gb, H, W, S):
        """w -> image end to end: the per-step inputs (latents, cameras) start in pinned host
        memory, the image ends in pinned host memory; synthesis network and render both on the
        sm_100a kernels.  With the reference files staged the call is the public drop-in
        ``render()`` on the reference's own Generator; otherwise the same two stages are called
        directly on seeded synthesis parameters."""
        from nerf_from_image_b200 import render as R
        from nerf_from_image_b200.synthesis import FusedSynthesis
        from oracle import reference_lift as RL  # availability probe only
        dev, rank, world = self.dev, self.rank, self.world
        syn = self.synthetic
        ds = syn.DATASET_CONFIGS[CFG['dataset']]
        cams = syn.make_cameras(99 + rank, B, radius=ds['radius'], device='cpu')
        host = {'c2w': cams['c2w'].pin_memory(), 'focal': cams['focal'].pin_memory(),
                'ws': torch.randn(B, 15, 512, generator=torch.Generator().manual_seed(5 + rank)).pin_memory(),
                'rgb': torch.empty(B, H, W, 3).pin_memory(), 'depth': torch.empty(B, H, W).pin_memory(),
                'mask': torch.empty(B, H, W).pin_memory()}
        api = None
        try:
            if not RL.available():
                raise RuntimeError('reference files not staged')
            import types
            _, generator = RL._import_reference()
            torch.manual_seed(1234)
            g = generator.Generator(512, ds['scene_range'], attention_values=CFG['attention_values'],
                                    use_sdf=True, disable_stylegan_noise=True).to(dev).eval()
            g.requires_grad_(False)
            with torch.no_grad():
                g.decoder.net[2].bias[0] = -1.15   # random-init SDF head shifted to cross zero
            R.configure(types.SimpleNamespace(use_viewdir=False, use_sdf=True,
                                              attention_values=CFG['attention_values'],
                                              fine_sampling=True, mlp_mode=self.args.mlp_mode),
                        {'scene_range': ds['scene_range'], 'white_background': ds['white_background']})
            R.enable_fused_synthesis(g)

            def step():
                with torch.no_grad():
                    ws = host['ws'].to(dev, non_blocking=True)
                    c2w = host['c2w'].to(dev, non_blocking=True)
                    focal = host['focal'].to(dev, non_blocking=True)
                    out = R.render(g, H, W, c2w, focal, None, None, ws, S)
                    host['rgb'].copy_(out[0], non_blocking=True)
                    host['depth'].copy_(out[1], non_blocking=True)
                    host['mask'].copy_(out[2], non_blocking=True)
                torch.cuda.synchronize()
            api = ('nerf_from_image_b200.render.render (drop-in of run.py:176-350) on the reference '
                   'Generator with enable_fused_synthesis: mapping-free w input -> texture mapper -> '
                   'FusedSynthesis (tcgen05) -> fused render')
            fs_only = FusedSynthesis(g.synthesis_network)
            ws_dev = host['ws'].to(dev)
            synth_only = lambda: fs_only(ws_dev[:, :14])
        except Exception as exc:
            why = repr(exc)[:80]
            chans = [min(32768 // r, 512) for r in (4, 8, 16, 32, 64, 128, 256)]
            fs = FusedSynthesis.from_params(syn.make_synthesis_params(3, 256, chans, 512, dev))
            sc, _, _, _, cfg = self.scene(CFG['dataset'], B, 7, H, W, S)

            def step():
                with torch.no_grad():
                    ws = host['ws'].to(dev, non_blocking=True)
                    c2w = host['c2w'].to(dev, non_blocking=True)
                    focal = host['focal'].to(dev, non_blocking=True)
                    planes = fs(ws[:, :14])
                    nt = torch.rand(B, H, W, S, device=dev)
                    nu = torch.rand(B * H * W, S, device=dev)
                    out = self.fused.fused_render(planes, sc['w1'], sc['b1'], sc['w2'], sc['b2'],
                                                  sc['palette'], sc['beta'], sc['alpha'], c2w, focal,
                                                  None, None, cfg, H, W, S, nt, nu,
                                                  planes_layout='channel_last')
                    host['rgb'].copy_(out[0], non_blocking=True)
                    host['depth'].copy_(out[1], non_blocking=True)
                    host['mask'].copy_(out[2], non_blocking=True)
                torch.cuda.synchronize()
            api = ('FusedSynthesis + fused_render called directly on seeded parameters (%s)' % why)
            ws_dev = host['ws'].to(dev)
            synth_only = lambda: fs(ws_dev[:, :14])
        for _ in range(2):
            step()
        self.barrier()
        n = max(2, self.args.e2e_steps)
        t0 = time.perf_counter()
        for _ in range(n):
            step()
        dt = self.max_over_ranks((time.perf_counter() - t0) / n)
        R._FRONTS.clear()
        # the plane producer on its own (CUDA events): dense conv FLOPs as executed (transposed convs
        # on the input grid), x3 for the three bf16 MMAs per product, against the measured bf16 peak
        with torch.no_grad():
            ms_syn = self.timed(synth_only, 5, 2)
        chans = [min(32768 // r, 512) for r in (4, 8, 16, 32, 64, 128, 256)]
        fl = 0.0
        for i, r in enumerate((4, 8, 16, 32, 64, 128, 256)):
            if i:
                fl += 2.0 * chans[i - 1] * chans[i] * 9 * (r // 2) ** 2
            fl += 2.0 * chans[i] * chans[i] * 9 * r * r + 2.0 * chans[i] * 96 * r * r
        pk = peaks()
        mma_tf = 3 * B * fl / (ms_syn * 1e-3) / 1e12
        synthesis = {'ms_per_forward': ms_syn, 'images_per_s': world * B / (ms_syn * 1e-3),
                     'dense_gflop_per_image': fl / 1e9,
                     'fp32_equivalent_tflops': B * fl / (ms_syn * 1e-3) / 1e12,
                     'bf16_mma_tflops': mma_tf, 'frac_of_measured_bf16_peak': mma_tf / pk['tflops'],
                     'what': 'FusedSynthesis alone, %d images, 256^2 x 96 planes, 512-channel '
                             'StyleGAN2 synthesis (13 modulated 3x3 convs + 7 ToRGB); bf16 hi/lo '
                             'pairs, three MMAs per product' % B}
        h2d = sum(host[k].numel() * 4 for k in ('ws', 'c2w', 'focal'))
        d2h = sum(host[k].numel() * 4 for k in ('rgb', 'depth', 'mask'))
        torch.cuda.empty_cache()
        return {'value': gb * H * W / dt, 'unit': UNIT, 'h2d_bytes_per_step': h2d,
                'd2h_bytes_per_step': d2h, 'ms_per_step': dt * 1e3,
                'mask_mean': host['mask'].mean().item(), 'api': api, 'synthesis': synthesis,
                'what': 'generator forward, w -> image: latents + cameras H2D from pinned memory, '
                        'synthesis network and render on the sm_100a kernels (both random draws '
                        'made on the device like the reference), rgb/depth/mask D2H; wall clock '
                        'incl. synchronisation, max over ranks'}

    def fixture_pretrained(self, B, H, W, S, steps=120):
        """SURVEY.md section 8d's fixture, to show that `value` does not hinge on the analytic
        scene: the reference Generator (seed 1234) SDF-pre-trained with the reference's own
        objective (run.py:821-868: sdf_distance + 0.1 * sdf_eikonal, Adam 2.5e-3; `steps`
        instead of 1000 steps, 4 latents each) -- its two losses computed by the fused point
        evaluator (enable_fused_heads) -- then 32 latents -> planes (FusedSynthesis) -> render."""
        from nerf_from_image_b200 import render as R
        from nerf_from_image_b200.synthesis import FusedSynthesis
        from oracle import reference_lift as RL  # availability probe + module import only
        if not RL.available():
            return {'unavailable': 'original project not staged (oracle/_ref)'}
        try:
            import types
            dev = self.dev
            syn = self.synthetic
            ds = syn.DATASET_CONFIGS[CFG['dataset']]
            _, generator = RL._import_reference()
            torch.manual_seed(1234)
            g = generator.Generator(512, ds['scene_range'], attention_values=CFG['attention_values'],
                                    use_sdf=True, disable_stylegan_noise=True).to(dev).train()
            R.configure(types.SimpleNamespace(use_viewdir=False, use_sdf=True,
                                              attention_values=CFG['attention_values'],
                                              fine_sampling=True, mlp_mode=self.args.mlp_mode),
                        {'scene_range': ds['scene_range'], 'white_background': ds['white_background']})
            R.enable_fused_heads(g)
            pm = R.ParallelModel(H, model=g, model_ema=g)
            opt = torch.optim.Adam(g.parameters(), lr=2.5e-3)
            t0 = time.perf_counter()
            first = last = None
            for i in range(steps):
                losses = pm(None, None, None, None, c=torch.randn(4, 512, device=dev), pretrain_sdf=True)
                loss = losses['sdf_distance_loss'].mean() + 0.1 * losses['sdf_eikonal_loss'].mean()
                loss.backward()
                opt.step()
                opt.zero_grad(set_to_none=True)
                if i == 0:
                    first = loss.item()
                last = loss.item() if i == steps - 1 else last
            torch.cuda.synchronize()
            train_s = time.perf_counter() - t0
            R.enable_fused_heads(g, False)
            g.eval().requires_grad_(False)
            cams = syn.make_cameras(4321, B, radius=ds['radius'], device=dev)
            cfg = self.fused.RenderConfig(scene_range=ds['scene_range'], white_background=False,
                                          attention_values=CFG['attention_values'],
                                          mlp_mode=self.args.mlp_mode)
            with torch.no_grad():
                ws = g.mapping_network(torch.randn(B, 512, device=dev), None)
                planes = FusedSynthesis(g.synthesis_network)(ws[:, :14])
                palette = g.texture_mapper(ws[:, 14])
                l1, l2 = g.decoder.net[0], g.decoder.net[2]
                w = (l1.weight * l1.weight_gain, l1.bias * l1.bias_gain, l2.weight * l2.weight_gain,
                     l2.bias * l2.bias_gain)
                nt = torch.rand(B, H, W, S, device=dev)
                nu = torch.rand(B * H * W, S, device=dev)
                fn = lambda: self.fused.fused_render(planes, *w, palette, g.beta, g.alpha, cams['c2w'],
                                                     cams['focal'], None, None, cfg, H, W, S, nt, nu,
                                                     planes_layout='channel_last')
                ms = self.timed(fn, 10, 3)
                mask = fn()[2].mean().item()
            del g, opt, planes
            torch.cuda.empty_cache()
            return {'value': B * H * W / (ms * 1e-3), 'unit': UNIT, 'ms_per_step': ms,
                    'mask_mean': mask, 'pretrain_steps': steps, 'pretrain_seconds': train_s,
                    'pretrain_loss_first_last': [first, last],
                    'what': 'render of %d images whose planes come from the SDF-pre-trained reference '
                            'Generator through FusedSynthesis (losses of the pre-training from the '
                            'fused point evaluator); same kernel, same geometry as `value`' % B}
        except Exception as exc:
            return {'unavailable': repr(exc)[:200]}

    def e2e_planes_from_host(self, sc, cams, cfg, B, gb, H, W, S):
        """Round 1's end-to-end figure, kept for continuity: PLANES from the host (805 MB per
        step over PCIe) through the C-ABI host entry point."""
        _lib, lib = self._lib, self.lib
        pin = lambda t: t.detach().cpu().contiguous().pin_memory()
        host = {k: pin(sc[k]) for k in ('w1', 'b1', 'w2', 'b2', 'palette', 'beta', 'alpha')}
        host['planes'] = pin(sc['planes'].permute(0, 1, 4, 2, 3))   # channel-first, as the ABI takes
        host['c2w'], host['focal'] = pin(cams['c2w']), pin(cams['focal'])
        host['rgb'] = torch.empty(B, H, W, 3).pin_memory()
        host['depth'] = torch.empty(B, H, W).pin_memory()
        host['mask'] = torch.empty(B, H, W).pin_memory()
        p = _lib.RenderParams()
        p.batch, p.height, p.width, p.num_samples = B, H, W, S
        p.plane_res, p.n_attention = CFG['plane_res'], CFG['attention_values']
        p.scene_range = sc['scene_range']
        p.white_background = int(sc['white_background'])
        p.use_sdf, p.fine_sampling, p.noise_mode = 1, 1, _lib.NOISE_PHILOX
        p.noise_seed = 1234 + self.rank
        p.mlp_mode = self.args.mlp_mode
        in_keys = ('planes', 'w1', 'b1', 'w2', 'b2', 'palette', 'beta', 'alpha', 'c2w', 'focal')
        for k in in_keys + ('rgb', 'depth', 'mask'):
            setattr(p, k, ctypes.c_void_p(host[k].data_ptr()))
        h2d = sum(host[k].numel() * 4 for k in in_keys)
        d2h = sum(host[k].numel() * 4 for k in ('rgb', 'depth', 'mask'))
        _lib.check(lib.nfi_render_forward_host(ctypes.byref(p), self.local_rank))
        self.barrier()
        t0 = time.perf_counter()
        for _ in range(2):
            _lib.check(lib.nfi_render_forward_host(ctypes.byref(p), self.local_rank))
        dt = self.max_over_ranks((time.perf_counter() - t0) / 2)
        return {'value': gb * H * W / dt, 'unit': UNIT, 'h2d_bytes_per_step': h2d,
                'd2h_bytes_per_step': d2h, 'ms_per_step': dt * 1e3,
                'api': 'nfi_render_forward_host (C ABI): planes H2D every step -- PCIe-bound'}

    def fwd_bwd(self, sc, cams, nt, nu, cfg, H, W, S, gb, weights=False, steps=None):
        """Forward + backward through the autograd.Function: the inversion step (grads to planes,
        palette, pose; decoder frozen: run.py:628-629,2256-2317) or, with `weights`, the GAN
        generator step (grads to planes, palette, decoder, beta, alpha; the cameras are sampled
        data there, run.py:1007-1044)."""
        leaves = {k: sc[k].detach().clone().requires_grad_() for k in ('planes', 'palette')}
        if not weights:
            leaves['c2w'] = cams['c2w'].detach().clone().requires_grad_()
        if weights:
            for k in ('w1', 'b1', 'w2', 'b2', 'beta', 'alpha'):
                leaves[k] = sc[k].detach().clone().requires_grad_()

        def step():
            rgb, depth, mask, _ = self.render(sc, cams, nt, nu, cfg, H, W, S, **leaves)
            (rgb.square().mean() + mask.mean()).backward()
            if weights and self.world > 1:
                self.parallel.all_reduce_grads([leaves[k] for k in ('w1', 'b1', 'w2', 'b2', 'beta', 'alpha')])
            for v in leaves.values():
                v.grad = None

        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        nb = steps or max(2, min(5, self.args.steps))
        ms_b = self.timed(step, nb, 3)
        torch.cuda.empty_cache()
        return {'value': gb * H * W / (ms_b * 1e-3), 'unit': UNIT, 'ms_per_step': ms_b,
                'what': 'fused_render forward + backward through the autograd.Function (grads to '
                        'planes, palette, %s)' % (
                            'decoder weights (render_wgrad_pipe, tcgen05), beta, alpha (+ their '
                            'all-reduce); cameras are data' if weights
                            else 'tform_cam2world; decoder frozen')}

    def cpu_baseline_and_parity(self, cfg, H, W, S):
        kind = reference_kind()
        n_img = 2
        cores = best_cpu_threads(kind)
        case = _cpu_case(n_img)
        cpu_render(case, kind)          # untimed: thread pool and allocator warm-up
        reps, dt, ref_rgb = 0, 0.0, None
        while dt < 10.0 and reps < 8:
            t, ref_rgb = cpu_render(case, kind)
            dt += t
            reps += 1
        rate = reps * n_img * H * W / dt
        cpu = {'value': rate, 'unit': UNIT, 'cores': cores, 'host_cores': os.cpu_count(), 'kind': kind,
               'sample': '%d of the 32 images (same geometry) x %d passes, %.1f s, torch CPU fp32 '
                         'no_grad, %s' % (n_img, reps, dt, 'unmodified reference render lifted from '
                                          'oracle/_ref' if kind == 'reference' else 'oracle port')}
        # parity of the CUDA path on exactly those images, against the oracle with the same
        # injected noise (the reference draws its own: same distribution, different numbers)
        from oracle import render_oracle as O
        scene, cams, nt, nu = case
        with torch.no_grad():
            ref = O.render_oracle(scene['planes'], scene['w1'], scene['b1'], scene['w2'],
                                  scene['b2'], scene['palette'], scene['beta'], scene['alpha'],
                                  cams['c2w'], cams['focal'], None, None, H, W, S, nt, nu,
                                  scene_range=scene['scene_range'],
                                  white_background=scene['white_background'])
            dev = self.dev
            sg = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in scene.items()}
            rgb_g, dep_g, msk_g, _ = self.fused.fused_render(
                sg['planes'], sg['w1'], sg['b1'], sg['w2'], sg['b2'], sg['palette'], sg['beta'],
                sg['alpha'], cams['c2w'].to(dev), cams['focal'].to(dev), None, None, cfg, H, W, S,
                nt.to(dev), nu.to(dev))
        parity = {'rgb_rel_l2': O.rel_l2(rgb_g.cpu(), ref['rgb']),
                  'rgb_psnr_db': O.psnr(rgb_g.cpu(), ref['rgb']),
                  'mask_rel_l2': O.rel_l2(msk_g.cpu(), ref['mask']),
                  'depth_rel_l2': O.rel_l2(dep_g.cpu(), ref['depth']),
                  'against': 'CPU oracle (pinned to the reference), identical injected noise, '
                             '%d images' % n_img}
        return cpu, parity

    def eager_gpu(self, H, W, S):
        """The same torch ops as the reference's render (the oracle port), fp32 with TF32 off like
        run.py:59-60, on this GPU -- the number the fused kernel has to beat."""
        try:
            from oracle import render_oracle as O
            torch.backends.cuda.matmul.allow_tf32 = False
            torch.backends.cudnn.allow_tf32 = False
            n_img = 2
            sc, cm, nt, nu, _ = self.scene(CFG['dataset'], n_img, 77, H, W, S, layout='channel_first')

            def fn():
                with torch.no_grad():
                    O.render_oracle(sc['planes'], sc['w1'], sc['b1'], sc['w2'], sc['b2'],
                                    sc['palette'], sc['beta'], sc['alpha'], cm['c2w'], cm['focal'],
                                    None, None, H, W, S, nt, nu, scene_range=sc['scene_range'],
                                    white_background=sc['white_background'])
            ms = self.timed(fn, 3, 2)
            torch.cuda.empty_cache()
            return {'value': n_img * H * W / (ms * 1e-3), 'unit': UNIT, 'ms_per_step': ms,
                    'sample': '%d images per step (same geometry), torch eager fp32 on this GPU, '
                              'no_grad, oracle port of the reference ops' % n_img}
        except Exception as exc:
            return {'unavailable': repr(exc)[:200]}

    # -------------------------------------------------------------- configs 3 / 4
    def config34(self):
        a, world, rank = self.args, self.world, self.rank
        H, W, S = CFG['height'], CFG['width'], CFG['samples']
        inv = a.config == 3
        gb = a.batch or (16 if inv else 32)
        if gb % world:
            raise SystemExit('global batch %d is not divisible by %d GPUs' % (gb, world))
        B = gb // world
        ds = 'cub' if inv else 'shapenet_chairs'
        sc, cams, nt, nu, cfg = self.scene(ds, B, 1234 + rank, H, W, S)
        steps = a.steps if a.steps_given else (30 if inv else 20)
        sampler = ClockSampler(self.local_rank)
        if rank == 0:
            sampler.start()
        res = self.fwd_bwd(sc, cams, nt, nu, cfg, H, W, S, gb, weights=not inv, steps=steps)
        clocks = sampler.summary() if rank == 0 else None
        with torch.no_grad():
            ms_f = self.timed(lambda: self.render(sc, cams, nt, nu, cfg, H, W, S), 10, 3)
        if rank != 0:
            return
        tiles = B * (H // 8) * (W // 16)
        line = {
            'metric': 'rays_per_sec_fwd_bwd_128x128_64+64spp', 'value': res['value'], 'unit': UNIT,
            'n_gpus': world, 'steps': steps, 'warmup': 3, 'ms_per_step': res['ms_per_step'],
            'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f32',
            'data': 'synthetic', 'config': config_block(a, world, B, gb), 'clocks': clocks,
            'forward_only': {'value': gb * H * W / (ms_f * 1e-3), 'unit': UNIT, 'ms_per_step': ms_f},
            'images_per_gpu': B,
            'tiles_per_gpu': tiles, 'waves_of_148_ctas': tiles / 148.0,
            # per step: weight image + render_forward_pipe, weight images + render_backward_pipe,
            # with decoder gradients also weight images + render_wgrad_pipe
            'what': res['what'], 'gpu_launches': (5 if inv else 8) * steps,
        }
        print(json.dumps(line))

    # -------------------------------------------------------------- config 5
    def config5(self):
        a, world, rank = self.args, self.world, self.rank
        B = a.batch or 8
        rows = []
        for res in (128, 256):
            for S in (32, 64, 128):
                sc, cams, nt, nu, cfg = self.scene(CFG['dataset'], B, 1234 + rank, res, res, S)
                with torch.no_grad():
                    ms_f = self.timed(lambda: self.render(sc, cams, nt, nu, cfg, res, res, S), 5, 3)
                fb = self.fwd_bwd(sc, cams, nt, nu, cfg, res, res, S, world * B, steps=3)
                rays = world * B * res * res
                flops = float(rays) * 2 * S * FLOPS_PER_POINT
                rows.append({'resolution': res, 'samples_per_ray': S,
                             'forward_rays_per_s': rays / (ms_f * 1e-3), 'forward_ms': ms_f,
                             'forward_points_per_s': rays * 2 * S / (ms_f * 1e-3),
                             'forward_tensor_tflops': flops / (ms_f * 1e-3) / 1e12,
                             'fwd_bwd_rays_per_s': fb['value'], 'fwd_bwd_ms': fb['ms_per_step']})
                del sc, nt, nu
                torch.cuda.empty_cache()
        if rank != 0:
            return
        pk = peaks()
        for r in rows:
            r['forward_roofline_frac'] = r['forward_tensor_tflops'] / world / pk['tflops']
        base = [r for r in rows if r['resolution'] == 128 and r['samples_per_ray'] == 64][0]
        print(json.dumps({
            'metric': METRIC, 'value': base['forward_rays_per_s'], 'unit': UNIT, 'n_gpus': world,
            'steps': 5, 'warmup': 3, 'ms_per_step': base['forward_ms'], 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': config_block(a, world, B, world * B), 'sweep': rows,
            'roofline_peak': pk, 'gpu_launches': 2 * 5}))

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=None)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--config', type=int, default=2, choices=[2, 3, 4, 5])
    ap.add_argument('--scaling', default='weak', choices=['weak', 'strong'])
    ap.add_argument('--exchange', default='auto', choices=['auto', 'nccl', 'peer'],
                    help='N > 1: in-place NCCL all-gather, or stores into the peers\' buffers from the kernel')
    ap.add_argument('--batch', type=int, default=None)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-e2e', action='store_true')
    ap.add_argument('--no-backward', action='store_true')
    ap.add_argument('--quick', action='store_true', help='skip the side legs (ncu, A/B runs)')
    ap.add_argument('--e2e-steps', type=int, default=3)
    ap.add_argument('--mlp-mode', type=lambda x: int(x, 0), default=0)
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='config 2: write rgb / depth / mask of the last timed step to '
                         'DIR/<name>.npy (float32, at most 64 MB in all)')
    args = ap.parse_args()
    args.steps_given = args.steps is not None
    if args.steps is None:
        args.steps = 20 if args.impl == 'b200' else 3
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'b200' or args.config != 2):
        ap.error('--dump-outputs writes the outputs of the timed render of --config 2')
    if args.impl == 'reference':
        return run_reference(args)
    args.warmup = max(args.warmup, 3)
    if args.quick:
        args.no_cpu_baseline = args.no_backward = True
    b = Bench(args)
    try:
        if args.config == 2:
            b.config2()
        elif args.config in (3, 4):
            b.config34()
        else:
            b.config5()
    finally:
        b.close()


if __name__ == '__main__':
    main()
