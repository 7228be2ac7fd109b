#!/usr/bin/env python
"""Headline benchmark: rays/sec of the render-and-relight hot path.

A step = one full view of BASELINE.json configs[1] ("lego_3072 geometry: 800x800,
128 spp, 512 light dirs, microfacet BRDF"): ray generation -> 128-sample sigma-MLP
march -> surface points (Stage A), then normal / light-visibility / albedo /
roughness MLPs, GGX BRDF and the 512-light rendering equation (Stage B) -> sRGB.
Synthetic data, random-init networks of the reference architecture.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--dump-outputs DIR]

N > 1 runs under torchrun (one rank per GPU): every rank renders its own full view
(weak scaling, north star "rays shard naturally"), and one NCCL all-gather per
step assembles all images on every rank.  Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

FLOP_SIGMA = 982528
FLOP_NERF = 982528 + 2 * (256 * 256 + 283 * 128 + 128 * 3)   # + bottleneck + colour branch
       # per sample  (BASELINE.md section 2)
FLOP_LVIS = 144640        # per (ray, light)
FLOP_POINT = 131328       # per ray, normal / albedo nets (rough: 130816)
FALLBACK_PEAKS = {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--imh', type=int, default=800)
    ap.add_argument('--imw', type=int, default=800)
    ap.add_argument('--spp', type=int, default=128, help='sigma-MLP samples per ray')
    ap.add_argument('--light-h', type=int, default=16)
    ap.add_argument('--sigma-precision', default=os.environ.get('NF_SIGMA_PREC', 'auto'))
    ap.add_argument('--cpu-sample-rays', type=int, default=8192)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-secondary', action='store_true',
                    help='skip the bounded secondary measurements (other BASELINE configs)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write the arrays the last timed step returned as DIR/<name>.npy (float32)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    return args


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(pred, out_dir):
    """Writes every array of one ViewRenderer.render result as <out_dir>/<name>.npy (float32), so
    that two builds can be compared output for output.  Above DUMP_MAX_BYTES in all, the same
    seeded sample of rays is kept from every array."""
    arrs = {k: v.detach().float().cpu().numpy() for k, v in pred.items()
            if isinstance(v, torch.Tensor)}
    total = sum(a.nbytes for a in arrs.values())
    if total > DUMP_MAX_BYTES:
        n = next(iter(arrs.values())).shape[0]
        keep = np.sort(np.random.default_rng(0).choice(n, n * DUMP_MAX_BYTES // total, replace=False))
        arrs = {k: a[keep] for k, a in arrs.items()}
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrs.items():
        np.save(os.path.join(out_dir, k + '.npy'), np.ascontiguousarray(a))


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        d['source'] = 'measured (MEASURED_PEAKS.json)'
        return d
    d = dict(FALLBACK_PEAKS)
    d['source'] = 'fallback (B200_PROFILING.md)'
    return d


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.rows, self.stop = index, [], threading.Event()
        self.t = threading.Thread(target=self.run, daemon=True)

    def run(self):
        while not self.stop.is_set():
            try:
                o = subprocess.run(
                    ['nvidia-smi', '-i', str(self.index), '--query-gpu=' + self.Q,
                     '--format=csv,noheader,nounits'], capture_output=True, text=True,
                    timeout=5).stdout.strip()
                if o:
                    self.rows.append([x.strip() for x in o.split(',')])
            except Exception:
                pass
            self.stop.wait(0.2)

    def __enter__(self):
        self.t.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.t.join(timeout=6)

    def summary(self):
        if not self.rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unsampled']}
        sm = sorted(float(r[0]) for r in self.rows)
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names)
                   if any(r[3 + i].lower().startswith('active') for r in self.rows)]
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': float(self.rows[0][1]),
                'power_w_max': max(float(r[2]) for r in self.rows), 'reasons': reasons,
                'samples': len(self.rows)}


def host_cores():
    """Cores this process may actually use: affinity mask capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, 'sched_getaffinity') else os.cpu_count()
    try:
        q, per = open('/sys/fs/cgroup/cpu.max').read().split()
        if q != 'max':
            n = max(1, min(n, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    return n


# ------------------------------------------------------------------ reference arm
def cpu_reference_rays_per_s(args, n_rays, steps, warmup):
    """The oracle (op-for-op CPU restatement of the reference; TF cannot run here) on a
    bounded sample of the same workload: n_rays rays at the same S and L."""
    from oracle import stage_a, stage_b, brdf as obrdf
    from nerfactor_b200 import synth
    torch.set_num_threads(host_cores())
    lh = args.light_h
    params = synth.make_stage_b_params(0, 'microfacet', light_hw=(lh, 2 * lh))
    nerf = synth.make_nerf_params(0)
    lxyz, lareas = obrdf.gen_light_xyz(lh, 2 * lh)
    om = stage_b.StageB(params, {'brdf': 'microfacet'}, lxyz=lxyz, lareas=lareas)
    rayo, rayd = stage_a.gen_rays(synth.look_at_c2w(), synth.CAM_ANGLE_X, args.imh, args.imw)
    sel = np.linspace(0, args.imh * args.imw - 1, n_rays).astype(np.int64)
    ro = torch.tensor(rayo.reshape(-1, 3)[sel])
    rd = stage_a.l2_normalize(torch.tensor(rayd.reshape(-1, 3)[sel]), 1)

    def step():
        a = stage_a.march_single_pass(nerf, ro, rd, 2., 6., args.spp, use_fine=True)
        alpha = torch.clamp(a['occu'], 0., 1.)[:, None]
        xyz = a['surf'] * alpha
        z3 = torch.zeros((n_rays, 3))
        batch = (None, None, ro, rd, z3, alpha, xyz, z3, torch.zeros((n_rays, 2 * lh * lh)))
        return om.call(batch, 'test')[0]['rgb']

    with torch.no_grad():
        for _ in range(warmup):
            step()
        t0 = time.perf_counter()
        for _ in range(steps):
            step()
        dt = (time.perf_counter() - t0) / steps
    return n_rays / dt, dt


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    n = args.cpu_sample_rays
    rps, dt = cpu_reference_rays_per_s(args, n, max(1, args.steps), max(1, min(args.warmup, 1)))
    sample = '%d of %d rays per step, same S=%d and L=%d' % (
        n, args.imh * args.imw, args.spp, 2 * args.light_h ** 2)
    line = {
        'impl': 'reference', 'metric': 'rays/sec', 'value': rps, 'unit': 'rays/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': dt * 1e3, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args, 'cpu'),
        'cpu_baseline': {'value': rps, 'unit': 'rays/s', 'cores': host_cores(),
                         'kind': 'port', 'sample': sample},
        'e2e': {'value': rps, 'unit': 'rays/s', 'h2d_bytes_per_step': 0,
                'd2h_bytes_per_step': 0},
        'note': 'restated reference (PyTorch-CPU oracle); TensorFlow 2.2 is not installable here'}
    print(json.dumps(line), flush=True)


def workload_config(args, sigma_prec):
    return {'workload': 'configs[1]: %dx%d view, %d sigma-MLP samples/ray (single pass), '
                        '%d light dirs, microfacet BRDF' % (
                            args.imw, args.imh, args.spp, 2 * args.light_h ** 2),
            'rays_per_view': args.imh * args.imw, 'samples_per_ray': args.spp,
            'light_dirs': 2 * args.light_h ** 2, 'brdf': 'microfacet',
            'precision': {'sigma_mlp': {'f16e': 'f16 operands (encoding as f16 hi+lo pair) / f32 accum',
                                        'f16': 'f16 operands / f32 accum'}.get(sigma_prec, sigma_prec),
                          'lvis_mlp': 'f16 operands / f32 accum',
                          'point_mlps': 'f16 hi/lo split x3 (fp32-accurate) / f32 accum',
                          'render': 'f32'},
            'l2_policy': 'per-step working set (lvis 1.3 GB, sigma 0.33 GB) exceeds the 126 MB L2',
            'stage_b': 'per-point networks, then nf_stageB_fused_fwd (visibility net -> GGX -> rendering '
                       'equation over L2-resident point chunks; no [N, L] tensor kept in HBM)',
            'lvis_lights': 'the visibility tensor is not an output of the timed call, so the visibility '
                           'network runs on the front-lit lights of each point only (cos(normal, light) > '
                           '-1e-5): the reference multiplies the visibility of all others by zero '
                           '(nerfactor.py:329-330) and evaluates its BRDF on front-lit pairs only itself '
                           '(:429-458).  Colours are bit-identical to evaluating every light '
                           '(parity.stage_b.front_lit_vs_all_lights...); secondary.step_all_lights times '
                           'the same step with every light evaluated',
            'parallelism': 'one view per GPU (same synthetic camera on every rank) + all_gather of images '
                           '(asynchronous, overlapping the next step)'}


def secondary_rows(ctx, nerf, kt):
    """Bounded measurements of the other BASELINE configs (parity-tested in tests/; these are
    context rows, not the headline): reference-exact hierarchical Stage A, the surface->light
    visibility march, learned-BRDF relighting at L = 1024, and one train step."""
    from nerfactor_b200 import _lib, synth, config as nfconfig
    from nerfactor_b200 import geometry_from_nerf as gfn
    from nerfactor_b200.models.nerfactor import Model as LearnedModel
    from nerfactor_b200.trainvali import Trainer
    from nerfactor_b200.brdf.renderer import gen_light_xyz
    out = {}
    cfg = nfconfig.default_config('nerf')
    # (1) compute_depth_and_normal: 128 coarse + 320 fine samples with d sigma/dx normals
    h = w = 200
    ro, rd = _lib.gen_rays(ctx, synth.look_at_c2w(), synth.CAM_ANGLE_X, h, w, normalize=True)
    t = kt(lambda: gfn.compute_depth_and_normal(nerf, ro, rd, cfg, precision=nerf.precision), 2)
    out['stage_a_hierarchical'] = {
        'what': 'geometry_from_nerf.compute_depth_and_normal, 128 coarse + 320 fine, '
                'tcgen05 sigma kernel (%s) + forward / input-gradient kernel (f16)' % nerf.precision,
        'rays': h * w, 'ms': t, 'rays_per_s': h * w / (t * 1e-3)}
    h = w = 96
    ro, rd = _lib.gen_rays(ctx, synth.look_at_c2w(), synth.CAM_ANGLE_X, h, w, normalize=True)
    t = kt(lambda: gfn.compute_depth_and_normal(nerf, ro, rd, cfg, precision='fp32'), 2)
    out['stage_a_hierarchical_fp32'] = {
        'what': 'same, FP32 CUDA-core kernels throughout (the bit-level parity path)',
        'rays': h * w, 'ms': t, 'rays_per_s': h * w / (t * 1e-3)}
    # (1b) the step before Stage A: NeRF colour rendering (nerf.py:149-252), 64 coarse + 192 fine
    h = w = 400
    ro, rd = _lib.gen_rays(ctx, synth.look_at_c2w(), synth.CAM_ANGLE_X, h, w, normalize=False)
    nb = ('bench', (h, w), ro, rd, None)
    t = kt(lambda: nerf.call(nb, 'test', precision='f16'), 2)
    out['nerf_render_rgb'] = {
        'what': 'nerf Model.call (coarse 64 + fine 192 samples, view-dependent colour), fused '
                'tcgen05 trunk + bottleneck + colour kernel (f16)',
        'rays': h * w, 'ms': t, 'rays_per_s': h * w / (t * 1e-3),
        'tflops': h * w * (64 + 192) * FLOP_NERF / (t * 1e-3) / 1e12}
    # (2) compute_light_visibility: every front-lit (point, light) pair marched 128 + 320 samples
    npts = 256
    surf = (ro[:npts] + rd[:npts] * 3.0).contiguous()
    nrm = (-rd[:npts]).contiguous()
    t = kt(lambda: gfn.compute_light_visibility(nerf, surf, nrm, cfg, light_h=16), 2)
    lx16, _ = gen_light_xyz(16, 32)
    _, _, fl = _lib.lvis_rays(ctx, surf, nrm, torch.as_tensor(
        np.asarray(lx16, np.float32).reshape(-1, 3)).to(ctx.device))
    marched = int(fl.sum().item())                # only front-lit pairs are marched (gfn.py:205-215)
    out['stage_a_light_visibility'] = {
        'what': 'geometry_from_nerf.compute_light_visibility, 512 lights, 128 + 320 samples per '
                'front-lit pair, %s' % nerf.precision,
        'points': npts, 'pairs': npts * 512, 'marched_pairs': marched, 'ms': t,
        'marched_pairs_per_s': marched / (t * 1e-3)}
    # (3) configs[2]: learned-MERL BRDF, 1024 light dirs on a 16x32 env-map, one 200x200 view
    lm = LearnedModel(nfconfig.default_config('nerfactor'),
                      params=synth.make_stage_b_params(0, 'learned'), ctx=ctx, precision='f16')
    lxyz, lareas = gen_light_xyz(16, 64)
    lm.set_lights(lxyz.reshape(-1, 3), lareas.reshape(-1),
                  light_idx=synth.light_index_map((16, 32), (16, 64)))
    n = 40000
    b = list(synth.make_stage_b_batch(1, n, 1, fg_frac=1.0))
    b[8] = None
    bt = tuple(torch.as_tensor(x).to(ctx.device) if isinstance(x, np.ndarray) and
               x.dtype != np.dtype('S9') and x.dtype.kind == 'f' else x for x in b)
    t = kt(lambda: lm.call(bt, 'test'), 2)
    out['stage_b_learned_L1024'] = {
        'what': 'nerfactor Model.call (learned BRDF), 1024 light dirs, 16x32 env-map',
        'rays': n, 'ms': t, 'rays_per_s': n / (t * 1e-3)}
    # (4) configs[3] semantics: one optimizer step, 1024 rays x 512 lights, fp32 training kernels
    lm2 = LearnedModel(nfconfig.default_config('nerfactor'),
                       params=synth.make_stage_b_params(0, 'learned'), ctx=ctx, precision='fp32')
    tb = synth.make_stage_b_batch(2, 1024, 512, fg_frac=1.0)
    tr = Trainer(lm2, precision='bf16')
    t = kt(lambda: tr.train_step(tb), 3)
    out['train_step'] = {'what': 'Trainer.train_step, 1024 rays x 512 lights, jitter on, '
                                 'tcgen05 Dense kernels (bf16 operands, fp32 accumulate / master)',
                         'ms': t, 'rays_per_s': 1024 / (t * 1e-3)}
    tr = Trainer(lm2, precision='fp32')
    t = kt(lambda: tr.train_step(tb), 3)
    out['train_step_fp32'] = {'what': 'same, FP32 CUDA-core Dense kernels',
                              'ms': t, 'rays_per_s': 1024 / (t * 1e-3)}
    # (5) the stage before Stage A: one NeRF train step (trainvali.NerfTrainer), in a subprocess
    try:
        r = subprocess.run([sys.executable, os.path.join(ROOT, 'tools', 'bench_nerf_train.py')],
                           capture_output=True, text=True, timeout=300)
        line = [l for l in r.stdout.splitlines() if l.startswith('{')]
        out['nerf_train_step'] = json.loads(line[-1]) if (r.returncode == 0 and line) else {
            'error': (r.stderr or r.stdout)[-400:]}
    except Exception as e:
        out['nerf_train_step'] = {'error': repr(e)}
    return out


def timed_mode_parity(ctx, nerf, model, vr, args, sigma_prec):
    """Measured error of the precision modes this run TIMES, against the library's own FP32
    CUDA-core kernels (which tests/ pin to the oracle and to the reference's fixtures): the sigma
    network on a ray subset of the benchmark view, the Stage-B networks + renderer on identical
    surface points, and the whole chain on the well-conditioned sphere-like field with smooth
    Stage-B networks (same construction as tests/test_gpu_stage_a_precision.py, where the same
    chain is compared with the CPU oracle).  Outside the timed region."""
    from nerfactor_b200 import _lib, synth, config as nfconfig
    from nerfactor_b200 import geometry_from_nerf as gfn
    from nerfactor_b200.models.nerf import Model as NerfModel
    from nerfactor_b200.models.nerfactor_microfacet import Model
    from nerfactor_b200.pipeline import ViewRenderer
    from nerfactor_b200.brdf.renderer import gen_light_xyz
    rl2 = lambda a, b: float((a - b).norm() / b.norm().clamp_min(1e-30))
    out = {'reference': 'FP32 CUDA-core kernels of this library (oracle-pinned in tests/)'}
    ro, rd = _lib.gen_rays(ctx, synth.look_at_c2w(4.0, 30.0, 30.0), synth.CAM_ANGLE_X, args.imh,
                           args.imw, normalize=True)
    sel = torch.linspace(0, ro.shape[0] - 1, 4096, device=ctx.device).long()
    ro, rd = ro[sel].contiguous(), rd[sel].contiguous()
    a_t = gfn.march_single_pass(nerf, ro, rd, args.spp, use_fine=True, precision=sigma_prec)
    a_r = gfn.march_single_pass(nerf, ro, rd, args.spp, use_fine=True, precision='fp32')
    dd = (a_t['depth'] - a_r['depth']).abs()
    out['stage_a'] = {'rays': 4096, 'sigma_rel_l2': rl2(a_t['sigma'], a_r['sigma']),
                      'depth_abs_err_median': float(dd.median()),
                      'depth_abs_err_p99': float(torch.quantile(dd, .99)),
                      'occupancy_abs_err_max': float((a_t['occu'] - a_r['occu']).abs().max())}
    alpha = torch.clamp(a_r['occu'], 0., 1.)[:, None]
    z3 = torch.zeros((4096, 3), device=ctx.device)
    batch = (None, None, ro, rd, z3, alpha.contiguous(), (a_r['surf'] * alpha).contiguous(), z3, None)
    p16 = model.call(batch, 'test')[0]
    model.precision = 'fp32'
    try:
        p32 = model.call(batch, 'test')[0]
    finally:
        model.precision = 'f16'
    out['stage_b'] = {'rays': 4096, 'rgb_rel_l2': rl2(p16['rgb'], p32['rgb']),
                      'lvis_rel_l2': rl2(p16['lvis'], p32['lvis'])}
    # the timed Stage-B path (nf_stageB_fused_fwd over point chunks) against the separate
    # full-size kernels of Model.call, on the whole benchmark view
    full_f = vr.render(synth.look_at_c2w(4.0, 30.0, 30.0), synth.CAM_ANGLE_X, args.imh, args.imw)
    full_c = vr.render(synth.look_at_c2w(4.0, 30.0, 30.0), synth.CAM_ANGLE_X, args.imh, args.imw,
                       fused=False)
    out['stage_b']['fused_op_vs_separate_kernels_rgb_rel_l2_full_view'] = rl2(full_f['rgb'], full_c['rgb'])
    full_a = vr.render(synth.look_at_c2w(4.0, 30.0, 30.0), synth.CAM_ANGLE_X, args.imh, args.imw,
                       all_lights=True)
    out['stage_b']['front_lit_vs_all_lights_rgb_max_abs_diff_full_view'] = float(
        (full_f['rgb'] - full_a['rgb']).abs().max())
    del full_f, full_c, full_a
    # end to end on the sphere-like field
    lh = args.light_h
    lxyz, lareas = gen_light_xyz(lh, 2 * lh)
    sb = synth.make_stage_b_params(4, 'microfacet', light_hw=(lh, 2 * lh), xyz_freq_decay=1.0)
    blob = synth.make_blob_nerf_params(5)
    chain = {}
    for tag, pa, pb in (('timed', sigma_prec, 'f16'), ('fp32', 'fp32', 'fp32')):
        nm = NerfModel(nfconfig.default_config('nerf'), params=blob, ctx=ctx, precision=pa)
        mm = Model(nfconfig.default_config('nerfactor_microfacet', light_h=lh), params=sb, ctx=ctx,
                   precision=pb)
        mm.set_lights(lxyz.reshape(-1, 3), lareas.reshape(-1))
        chain[tag] = ViewRenderer(nm, mm, n_samples=args.spp, use_fine=True).render(
            synth.look_at_c2w(), synth.CAM_ANGLE_X, 64, 64)
    same = (chain['timed']['alpha'] > 0) == (chain['fp32']['alpha'] > 0)
    fg = (same & (chain['fp32']['alpha'] > 0))[:, 0]
    out['end_to_end_sphere_field'] = {
        'what': 'camera -> %d-sample march -> Stage B -> sRGB, 64 x 64 view of the analytic '
                'sphere-like density field, smooth Stage-B networks' % args.spp,
        'rgb_rel_l2': rl2(chain['timed']['rgb'][fg], chain['fp32']['rgb'][fg]),
        'foreground_rays': int(fg.sum()), 'mask_flips': int((~same).sum()),
        'north_star_tolerance': 1e-4}
    return out


def multi_rank_rows(ctx, vr, model, args, dist, world, rank):
    """Rows every rank takes part in (N = 1 too): (1) STRONG scaling -- one 800 x 800 view
    ray-sharded over the ranks (pipeline.shard_range), image assembled with one all-gather
    (pipeline.gather_image); (2) BASELINE configs[4] as written -- 8 novel views x 8 env-maps
    (one integrate pass relights under all 8 probes), views split over the ranks, all images
    gathered.  CUDA events between barriers, max over ranks."""
    from nerfactor_b200 import synth
    from nerfactor_b200.pipeline import shard_range, gather_image
    n_rays = args.imh * args.imw

    def timed(fn, steps=2, warmup=1):
        for _ in range(warmup):
            fn()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        if world > 1:
            t = torch.tensor([ms], device=ctx.device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    out = {}
    c2w = synth.look_at_c2w(4.0, 30.0, 30.0)
    a, b = shard_range(n_rays, rank, world)

    per = (n_rays + world - 1) // world
    peer = None
    if world > 1 and os.environ.get('NF_GATHER', 'push') == 'push':
        try:
            from nerfactor_b200.pipeline import PeerImageGather
            peer = PeerImageGather(per, (3,), world, rank, ctx.device)
        except Exception:
            peer = None

    def strong():
        pred = vr.render(c2w, synth.CAM_ANGLE_X, args.imh, args.imw, ray_range=(a, b))
        if world == 1:
            return pred['rgb']
        if peer is None:
            return gather_image(pred['rgb'], n_rays, rank, world)
        rgb = pred['rgb']
        if rgb.shape[0] < per:                    # last shard of a ragged split
            rgb = torch.cat((rgb, torch.zeros((per - rgb.shape[0], 3), device=ctx.device)), 0)
        peer.push(rgb)
        return peer.finish().reshape(-1, 3)[:n_rays]      # the image is complete on every rank
    ms = timed(strong)
    out['strong_scaling_one_view'] = {
        'what': 'ONE %dx%d view, rays [rank] of %d contiguous shards, image assembled on every rank '
                'inside the timed region (%s)' % (args.imw, args.imh, world,
                                                 'peer pushes' if peer is not None else 'NCCL all-gather'),
        'scaling': 'strong', 'ms': ms, 'rays_per_s': n_rays / (ms * 1e-3), 'n_gpus': world}
    # configs[4]: 8 views x 8 env-maps
    n_views, n_maps = 8, 8
    probes = synth.make_probes(3, n_maps, light_hw=(args.light_h, 2 * args.light_h))
    saved = model.novel_probes
    from collections import OrderedDict
    model.novel_probes = OrderedDict(('probe%d' % i, torch.as_tensor(p).to(ctx.device))
                                     for i, p in enumerate(probes))
    mine = [v for v in range(n_views) if v % world == rank]
    per = (n_views + world - 1) // world

    def sweep():
        imgs = []
        for v in mine:
            pred = vr.render(synth.look_at_c2w(4.0, 30.0 + 45.0 * v, 30.0), synth.CAM_ANGLE_X,
                             args.imh, args.imw, relight_probes=True)
            imgs.append(pred['rgb_probes'])                      # [n_rays, 8, 3]
        while len(imgs) < per:                                   # ragged split: pad for the gather
            imgs.append(torch.zeros_like(imgs[0]) if imgs else
                        torch.zeros((n_rays, n_maps, 3), device=ctx.device))
        local = torch.stack(imgs, 0)
        if world > 1:
            full = torch.empty((world,) + tuple(local.shape), device=ctx.device)
            dist.all_gather_into_tensor(full, local)
            return full
        return local
    try:
        ms = timed(sweep, steps=1 if world == 1 else 2)
    finally:
        model.novel_probes = saved
    # configs[3]: one data-parallel optimizer step (forward + backward + gradient all-reduce +
    # AMSGrad), 1024 rays x 512 lights per rank, bf16 tensor-core Dense kernels
    try:
        from nerfactor_b200 import config as nfconfig
        from nerfactor_b200.models.nerfactor import Model as LearnedModel
        from nerfactor_b200.trainvali import Trainer
        lm = LearnedModel(nfconfig.default_config('nerfactor'),
                          params=synth.make_stage_b_params(0, 'learned'), ctx=ctx, precision='fp32')
        tb = synth.make_stage_b_batch(2 + rank, 1024, 512, fg_frac=1.0)
        tr = Trainer(lm, world_size=world, rank=rank, precision='bf16')
        t_ms = timed(lambda: tr.train_step(tb), steps=5, warmup=3)
        out['train_step_data_parallel'] = {
            'what': 'BASELINE configs[3]: Trainer.train_step (learned-BRDF NeRFactor, jitter on), 1024 '
                    'rays x 512 lights PER RANK, bf16 tcgen05 Dense kernels, one NCCL all-reduce of the '
                    'flat gradient inside the timed region, AMSGrad',
            'ms': t_ms, 'rays_per_s': world * 1024 / (t_ms * 1e-3), 'n_gpus': world,
            'global_batch_rays': world * 1024}
        del tr, lm
    except Exception as e:
        out['train_step_data_parallel'] = {'error': repr(e)}
        if world > 1:
            raise
    out['config5_relight_sweep'] = {
        'what': 'BASELINE configs[4]: %d novel views x %d env-maps at %dx%d, views split over the '
                'ranks, NCCL all-gather of every relit image' % (n_views, n_maps, args.imw, args.imh),
        'ms': ms, 'rays_per_s': n_views * n_rays / (ms * 1e-3),
        'relit_images_per_s': n_views * n_maps / (ms * 1e-3), 'n_gpus': world,
        'gathered_bytes': int(n_views * n_rays * n_maps * 3 * 4)}
    return out


# ------------------------------------------------------------------------ our arm
def main():
    args = parse()
    if args.impl == 'reference':
        return run_reference(args)
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        # keep stdout to the single JSON line: NCCL's banner / debug output goes to stderr
        if os.environ.get('NCCL_DEBUG', 'VERSION').upper() == 'VERSION':
            os.environ['NCCL_DEBUG'] = 'WARN'
        os.environ.setdefault('NCCL_DEBUG_FILE', '/dev/stderr')
        import torch.distributed as dist
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    from nerfactor_b200 import _lib, synth, config as nfconfig
    from nerfactor_b200.models.nerfactor_microfacet import Model
    from nerfactor_b200.models.nerf import Model as NerfModel
    from nerfactor_b200.pipeline import ViewRenderer

    ctx = _lib.Context(local)
    lh = args.light_h
    L = 2 * lh * lh
    n_rays = args.imh * args.imw
    sigma_prec = args.sigma_precision
    nerf = NerfModel(nfconfig.default_config('nerf'), params=synth.make_nerf_params(0), ctx=ctx,
                     precision='f16')
    if sigma_prec == 'auto':
        # 'f16e' = fp16 operands with the positional encoding as an fp16 hi + lo pair: the mode
        # whose end-to-end RGB parity is demonstrated (tests/test_gpu_stage_a_precision.py)
        sigma_prec = 'f16e'
    nerf.precision = sigma_prec
    model = Model(nfconfig.default_config('nerfactor_microfacet', light_h=lh),
                  params=synth.make_stage_b_params(0, 'microfacet', light_hw=(lh, 2 * lh)),
                  ctx=ctx, precision='f16')
    vr = ViewRenderer(nerf, model, n_samples=args.spp, use_fine=True)
    # one view per rank; weak scaling = identical per-GPU work, so every rank renders the same
    # synthetic camera (a different azimuth changes the foreground fraction and with it the
    # Stage-B work, which would measure the scene, not the system)
    c2w = synth.look_at_c2w(4.0, 30.0, 30.0)
    light_host = torch.rand((lh, 2 * lh, 3)).pin_memory()
    rgb_host = torch.empty((n_rays, 3)).pin_memory()
    alpha_host = torch.empty((n_rays, 1)).pin_memory()
    gathered = torch.empty((world * n_rays, 3), device=ctx.device) if world > 1 else None
    # N > 1: images are exchanged by one-sided pushes over NVLink peer memory (copy engines, no SM
    # kernel, no per-step rendezvous: pipeline.PeerImageGather); NCCL all_gather is the fallback
    peer = None
    gather_how = 'none'
    if world > 1:
        gather_how = 'NCCL all_gather_into_tensor (async)'
        if os.environ.get('NF_GATHER', 'push') == 'push':
            try:
                from nerfactor_b200.pipeline import PeerImageGather
                peer = PeerImageGather(n_rays, (3,), world, rank, ctx.device)
                gather_how = 'one-sided pushes into symmetric peer memory (NVLink, copy engines)'
            except Exception as e:           # symmetric memory not available in this build
                peer = None
                gather_how += ' [symmetric memory unavailable: %r]' % (e,)

    # The image all-gather of step k is issued asynchronously (NCCL's own stream, after the
    # step's last kernel) and overlaps the kernels of step k + 1; the next gather -- and the end of
    # the timed region -- wait for it.  Ranks are therefore not lock-stepped kernel by kernel.
    pending = [None]

    def gather(rgb):
        if peer is not None:
            peer.push(rgb)
            return
        if pending[0] is not None:
            pending[0].wait()
        pending[0] = dist.all_gather_into_tensor(gathered, rgb.contiguous(), async_op=True)

    def drain():
        if peer is not None:
            if peer.step:
                peer.finish()
            return
        if pending[0] is not None:
            pending[0].wait()
            pending[0] = None

    last_pred = [None]

    def step_device():
        pred = vr.render(c2w, synth.CAM_ANGLE_X, args.imh, args.imw)
        if world > 1:
            gather(pred['rgb'])
        if args.dump_outputs:
            last_pred[0] = pred
        return pred

    def step_e2e():
        pred = vr.render_to_host(c2w, synth.CAM_ANGLE_X, args.imh, args.imw, light_host,
                                 rgb_host, alpha_host)
        if world > 1:
            gather(pred['rgb'])
        return pred

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        if world > 1:
            drain()
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ctx.launches
        e0.record()
        for _ in range(steps):
            fn()
        if world > 1:
            drain()                   # the last image is assembled inside the timed region
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=ctx.device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dist.barrier()
            ms = float(t.item())
        return ms, ctx.launches - l0

    # clocks / throttle reasons are sampled on rank 0 only (its line is the one printed): one
    # nvidia-smi poller per rank would put 5 N queries per second on the box during the timed region
    if rank == 0:
        with ClockSampler(local) as cs:
            ms, launches = timed(step_device, args.steps, max(3, args.warmup))
        clocks = cs.summary()
    else:
        ms, launches = timed(step_device, args.steps, max(3, args.warmup))
        clocks = None
    if args.dump_outputs and rank == 0:
        dump_outputs(last_pred[0], args.dump_outputs)
    last_pred[0] = None
    ms_step = ms / args.steps
    value = world * n_rays / (ms_step * 1e-3)
    ms_e2e, _ = timed(step_e2e, args.steps, 1)
    e2e_value = world * n_rays / (ms_e2e / args.steps * 1e-3)

    def step_all_lights():
        pred = vr.render(c2w, synth.CAM_ANGLE_X, args.imh, args.imw, all_lights=True)
        if world > 1:
            gather(pred['rgb'])
        return pred
    ms_all, _ = timed(step_all_lights, args.steps, 1)
    all_lights_row = {'what': 'the timed step with the visibility network evaluated for EVERY light '
                              '(config.lvis_lights); same images bit for bit',
                      'ms': ms_all / args.steps, 'rays_per_s': world * n_rays / (ms_all / args.steps * 1e-3)}

    multi = None
    if not args.no_secondary:
        try:
            multi = multi_rank_rows(ctx, vr, model, args, dist, world, rank)
        except Exception as e:                    # context rows must not take the headline down
            multi = {'error': repr(e)}
            if world > 1:
                raise
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- per-kernel device times (CUDA events on the launching stream) + rooflines
    pk = peaks()
    a = vr.stage_a(c2w, synth.CAM_ANGLE_X, args.imh, args.imw)
    mask = a['alpha'][:, 0] > 0
    xyz_m = a['xyz'][mask].contiguous()
    n_fg = int(xyz_m.shape[0])

    def kt(fn, reps=3):
        fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    rayo, rayd = a['rayo'], a['rayd']
    z = _lib.gen_z(ctx, nerf.near, nerf.far, args.spp, n_rays)
    t_sigma = kt(lambda: _lib.sigma_fwd(ctx, nerf.packed_sigma(True), rayo, rayd, z, None,
                                        sigma_prec), 2 if sigma_prec == 'fp32' else 3)
    z3 = torch.zeros_like(a['xyz'])
    batch_b = (None, None, a['rayo'], a['rayd'], z3, a['alpha'], a['xyz'], z3, None)
    t_lvis = kt(lambda: model._pred_lvis_at(xyz_m))
    lvis = model._pred_lvis_at(xyz_m)
    t_point = kt(lambda: model._pred_normal_at(xyz_m))
    nrm = model._pred_normal_at(xyz_m)
    alb = model._pred_albedo_at(xyz_m)
    rough = model._pred_brdf_at(xyz_m)
    cam = rayo[mask].contiguous()
    light = model.light.reshape(1, -1, 3).contiguous()
    t_int = kt(lambda: _lib.integrate_fwd(ctx, xyz_m, nrm, cam, alb, lvis, model.lxyz,
                                          model.lareas, light, rough=rough, f0=0.04))
    tensor_peak = pk['bf16_tflops_sustained']
    alg_sigma = n_rays * args.spp * 4 * 2 + n_rays * 24          # z in, sigma out, rays
    alg_lvis = n_fg * L * 4 + n_fg * 12
    alg_int = n_fg * (4 * L + 64 + 12)
    rf_sigma = {'kernel': 'nf_sigma_fwd (%s)' % sigma_prec, 'bound': 'tensor',
                'achieved': n_rays * args.spp * FLOP_SIGMA / (t_sigma * 1e-3) / 1e12,
                'peak': tensor_peak, 'unit': 'TFLOP/s', 'ms': t_sigma, 'traffic': None,
                'algorithmic_bytes': alg_sigma}
    rf_sigma_plain = None
    if sigma_prec == 'f16e':        # context: the same kernel without the split encoding
        t_plain = kt(lambda: _lib.sigma_fwd(ctx, nerf.packed_sigma(True), rayo, rayd, z, None, 'f16'), 3)
        rf_sigma_plain = {'kernel': 'nf_sigma_fwd (f16, positional encoding NOT split; not the timed mode)',
                          'bound': 'tensor', 'ms': t_plain, 'peak': tensor_peak, 'unit': 'TFLOP/s',
                          'achieved': n_rays * args.spp * FLOP_SIGMA / (t_plain * 1e-3) / 1e12}
        rf_sigma_plain['frac'] = rf_sigma_plain['achieved'] / tensor_peak
    # Stage B as the timed step runs it (front-lit lights only) and with every light
    t_sb_fl = kt(lambda: model.render_rgb(batch_b))
    t_sb_all = kt(lambda: model.render_rgb(batch_b, all_lights=True))
    rf_lvis = {'kernel': 'nf_lvis_fwd (lvis_tc3_kernel f16, every light: %d x %d rows)' % (n_fg, L),
               'bound': 'tensor',
               'achieved': n_fg * L * FLOP_LVIS / (t_lvis * 1e-3) / 1e12,
               'peak': tensor_peak, 'unit': 'TFLOP/s', 'ms': t_lvis, 'traffic': None,
               'algorithmic_bytes': alg_lvis,
               'executed_tflops': n_fg * L * 131328 / (t_lvis * 1e-3) / 1e12,
               'note': 'achieved = the reference\'s FLOPs per (point, light) pair / time; the kernel '
                       'EXECUTES 131 328 per pair (the xyz part of the input is folded into a '
                       'per-point bias once per point: -22 % of the K; the bias rides in the MMA as '
                       'a K = 16 block: +12.5 %), which is why `frac` can exceed 1 against the '
                       'sustained cuBLAS figure',
               'stage_b_ms': {'front_lit_lights_only (timed mode)': t_sb_fl, 'every_light': t_sb_all,
                              'what': 'Model.render_rgb on the view\'s foreground points: per-point '
                                      'networks + nf_stageB_fused_fwd'}}
    rf_int = {'kernel': 'nf_integrate_fwd (microfacet)', 'bound': 'hbm',
              'achieved': alg_int / (t_int * 1e-3) / 1e9,
              'peak': pk['hbm_gbs'], 'unit': 'GB/s', 'ms': t_int, 'traffic': None,
              'algorithmic_bytes': alg_int,
              'note': 'ALU-bound with the analytic GGX lobe (SURVEY 7 hard parts)'}
    # the other integrate variant (nf_integrate_fwd brdf_kind = 1: pre-computed learned-BRDF lobe,
    # SURVEY 8b "pre-computed-BRDF variant"): reads the lvis AND spec rows (8L + 76 B / ray) and has
    # no GGX arithmetic, i.e. the memory-heavier of the two.  Context row; never the headline.
    rf_int_spec = None
    try:
        spec = torch.rand_like(lvis)
        t_int1 = kt(lambda: _lib.integrate_fwd(ctx, xyz_m, nrm, cam, alb, lvis, model.lxyz,
                                               model.lareas, light, spec=spec, spec_scale=1.0))
        alg_int1 = n_fg * (8 * L + 64 + 12)
        rf_int_spec = {'kernel': 'nf_integrate_fwd (pre-computed BRDF lobe)', 'bound': 'hbm',
                       'achieved': alg_int1 / (t_int1 * 1e-3) / 1e9, 'peak': pk['hbm_gbs'],
                       'unit': 'GB/s', 'ms': t_int1, 'traffic': None,
                       'algorithmic_bytes': alg_int1}
        rf_int_spec['frac'] = rf_int_spec['achieved'] / rf_int_spec['peak']
        del spec
    except Exception as e:                                  # context row only
        rf_int_spec = {'kernel': 'nf_integrate_fwd (pre-computed BRDF lobe)', 'error': repr(e)}
    rf_point = {'kernel': 'nf_point_mlp_fwd (tcgen05 f16x3 split, per net; x3 per step)', 'bound': 'latency',
                'achieved': n_fg * FLOP_POINT / (t_point * 1e-3) / 1e12, 'peak': None,
                'unit': 'TFLOP/s', 'ms': t_point, 'traffic': None}
    for r in (rf_sigma, rf_lvis, rf_int):
        r['frac'] = r['achieved'] / r['peak']
    # both denominators for the tensor-bound kernels: `peak` is the sustained cuBLAS figure (the
    # kernels run 40-70 ms per launch on a power-capped part, the regime that figure describes);
    # `frac_burst` uses the best-of-10 short-GEMM figure
    for r in (rf_sigma, rf_lvis):
        if pk.get('bf16_tflops'):
            r['peak_burst'] = pk['bf16_tflops']
            r['frac_burst'] = r['achieved'] / pk['bf16_tflops']
    # DRAM bytes per launch from the committed ncu --set full capture of this exact workload
    tpath = os.path.join(ROOT, 'profiles', 'r2_traffic.json')
    if not os.path.exists(tpath):
        tpath = os.path.join(ROOT, 'profiles', 'r1_traffic.json')
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        wl = tj['workload']
        if (wl['imh'], wl['imw'], wl['spp'], wl['light_dirs']) == (args.imh, args.imw, args.spp, L):
            for r, key in ((rf_sigma, 'sigma'), (rf_lvis, 'lvis'), (rf_int, 'integrate'),
                           (rf_point, 'point')):
                if (key == 'sigma' and sigma_prec == 'fp32') or key not in tj['kernels']:
                    continue
                r['traffic'] = tj['kernels'][key]['dram_bytes']
                r['ncu_tensor_pipe_active_pct'] = tj['kernels'][key].get('tensor_pipe_active_pct')
                r['traffic_source'] = tj['source']
    dominant = max((rf_sigma, rf_lvis, rf_int), key=lambda r: r['ms'])
    dominant = dict(dominant, peak_source=pk['source'] + ', sustained bf16 cuBLAS' if
                    dominant['bound'] == 'tensor' else pk['source'])

    secondary = None
    if not args.no_secondary:
        secondary = secondary_rows(ctx, nerf, kt) if world == 1 else {}
        secondary.update(multi or {})
        secondary['step_all_lights'] = all_lights_row
    parity = timed_mode_parity(ctx, nerf, model, vr, args, sigma_prec)

    cpu = None
    if not args.no_cpu_baseline:
        rps, dt = cpu_reference_rays_per_s(args, args.cpu_sample_rays, 3, 1)
        cpu = {'value': rps, 'unit': 'rays/s', 'cores': host_cores(), 'kind': 'port',
               'sample': '%d of %d rays, same S=%d and L=%d, 1 warm-up + 3 timed passes '
                         '(%.1f s each)' % (args.cpu_sample_rays, n_rays, args.spp, L, dt)}

    line = {
        'metric': 'rays/sec', 'value': value, 'unit': 'rays/s', 'n_gpus': world,
        'steps': args.steps, 'warmup': max(3, args.warmup), 'ms_per_step': ms_step,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'f16' if sigma_prec != 'fp32' else 'f32+f16', 'data': 'synthetic',
        'config': dict(workload_config(args, sigma_prec), image_exchange=gather_how),
        'e2e': {'value': e2e_value, 'unit': 'rays/s',
                'h2d_bytes_per_step': int(light_host.numel() * 4 + 16 * 8 + 8),
                'd2h_bytes_per_step': int(rgb_host.numel() * 4 + alpha_host.numel() * 4)},
        'gpu_launches': launches, 'clocks': clocks,
        # the same step with the visibility network evaluated for every light instead of the
        # front-lit ones (config.lvis_lights): identical images, more tensor work
        'every_light': {'value': all_lights_row['rays_per_s'], 'unit': 'rays/s',
                        'ms_per_step': all_lights_row['ms']},
        'roofline': dominant,
        'rooflines': [rf_sigma, rf_lvis, rf_int, rf_point] + ([rf_int_spec] if rf_int_spec else []) +
                     ([rf_sigma_plain] if rf_sigma_plain else []),
        'foreground_rays': n_fg,
        'cpu_baseline': cpu,
        'parity': parity,
        'secondary': secondary,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
