"""Kernel time of nf_integrate_bwd (CUDA events around replays of a CUDA graph of 10 calls) at the
train step's size (1024 points x 512 lights) and at 65 536 x 512, both BRDF kinds, with every
gradient the NeRFactor train step asks for; beside it, the same gradients through torch autograd
of the element-wise composition the op replaces (autodiff.microfacet_brdf / albedo / pi + spec *
scale, then autodiff.render: forward + backward), and nf_integrate_fwd.  One JSON object, with the
GPU's name and power limit."""
import json
import math
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from nerfactor_b200 import _lib, synth                                     # noqa: E402
from nerfactor_b200 import autodiff as ad                                  # noqa: E402


def _time(fn, per_graph=10, replays=5):
    """ms per fn(): `per_graph` calls captured in one CUDA graph (as the train step replays them,
    so host launch overhead is left out), replayed `replays` times after one warm-up replay."""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(2):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for _ in range(per_graph):
            fn()
    g.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(replays):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (per_graph * replays)


def main():
    ctx = _lib.default_context()
    gpu = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader',
                          '-i', str(torch.cuda.current_device())],
                         capture_output=True, text=True).stdout.strip()
    out = {'gpu': gpu, 'cases': []}
    L = 512
    for n in (1024, 65536):
        batch = synth.make_stage_b_batch(1, n, L, fg_frac=1.0)
        rng = np.random.default_rng(2)
        dev = lambda a: torch.as_tensor(np.ascontiguousarray(a, np.float32)).cuda()
        xyz, nrm, cam, lvis = [dev(batch[i]) for i in (6, 7, 2, 8)]
        d = rng.standard_normal((L, 3))
        d[:, 2] = np.abs(d[:, 2]) + 0.3
        lxyz = dev(100. * d / np.linalg.norm(d, axis=1, keepdims=True))
        lareas = dev(np.full(L, 2 * math.pi / L))
        light = dev(rng.uniform(0., 2., (L, 3)))
        albedo = dev(rng.uniform(0.05, 0.9, (n, 3)))
        d_rgb = dev(rng.standard_normal((n, 3)))
        for kind in (0, 1):
            prop = dev(rng.uniform(0.2, 0.8, (n, 1))) if kind == 0 else dev(rng.uniform(0, 1, (n, L)))
            rough, spec = (prop, None) if kind == 0 else (None, prop)
            need = ['lvis', 'normal', 'albedo', 'rough' if kind == 0 else 'spec', 'light']
            t_bwd = _time(lambda: _lib.integrate_bwd(
                ctx, xyz, nrm, cam, albedo, lvis, lxyz, lareas, light, d_rgb, rough=rough,
                spec=spec, f0=0.04, spec_scale=1.0, linear2srgb=True, need=need))
            t_fwd = _time(lambda: _lib.integrate_fwd(
                ctx, xyz, nrm, cam, albedo, lvis, lxyz, lareas, light[None], rough=rough, spec=spec,
                f0=0.04, spec_scale=1.0, linear2srgb=True))

            def eager():
                leaves = [x.detach().requires_grad_(True) for x in (lvis, nrm, albedo, prop, light)]
                lv, nr, al, pr, li = leaves
                surf2l = ad.safe_l2_normalize(lxyz.reshape(1, -1, 3) - xyz[:, None, :], 2)
                surf2c = ad.safe_l2_normalize(cam - xyz, 1)
                nn = ad.safe_l2_normalize(nr, 1)
                if kind == 0:
                    brdf = ad.microfacet_brdf(surf2l, surf2c, nn, al, pr, 0.04)
                else:
                    brdf = al[:, None, :] / math.pi + pr[:, :, None].expand(n, L, 3)
                rgb = ad.render(lv, brdf, surf2l, nn, li, lareas, True)
                torch.autograd.grad(rgb, leaves, d_rgb)

            t_eager = _time(eager)
            out['cases'].append({'n': n, 'L': L, 'kind': kind, 'nf_integrate_bwd_ms': t_bwd,
                                 'nf_integrate_fwd_ms': t_fwd,
                                 'torch_autograd_fwd_bwd_ms': t_eager})
    print(json.dumps(out))


if __name__ == '__main__':
    main()
