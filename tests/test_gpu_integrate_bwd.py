"""nf_integrate_bwd -- the backward of the rendering equation -- on the GPU: gradients against fp64
autograd of the torch composition it replaces, NULL outputs, run-to-run determinism, and the
NeRFactor train step on the library's kernels against the reference's own tape."""
import ctypes as C
import math
import os
from importlib import import_module

import numpy as np
import pytest
import torch

from nerfactor_b200 import _lib, synth, config as nfconfig
from nerfactor_b200 import autodiff as ad

pytestmark = pytest.mark.gpu

F0, SPEC_SCALE = 0.04, 0.7
NAMES = ('lvis', 'normal', 'albedo', 'prop', 'light')


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


@pytest.fixture(scope='module')
def ctx():
    return _lib.default_context()


def _case(kind, n, L, seed=0):
    """Inputs that reach every branch of the adjoint: normals around a sphere seen from one camera
    (front, grazing and back-facing views), raw normals of random length, roughness 0.7 / 0.4 / 0.2,
    lights on the upper hemisphere with a few 30x brighter ones (rgb > 1: gradient 0), points
    facing down (every light back-lit) or with lvis = 0 (linear sum exactly 0: the gradient passes
    the clip), points with lvis * 1e-4 (below the sRGB knee)."""
    rng = np.random.default_rng(seed + 1000 * kind + n + 7 * L)
    batch = synth.make_stage_b_batch(seed, n, L, fg_frac=1.0)
    xyz, nrm, cam, lvis = batch[6], batch[7].copy(), batch[2], batch[8].copy()
    nrm[5::13] = [0.02, -0.01, -1.]
    nrm *= rng.uniform(0.5, 2., (n, 1))
    lvis[2::7] = 0.
    lvis[3::11] *= 1e-4
    d = rng.standard_normal((L, 3))
    d[:, 2] = np.abs(d[:, 2]) + 0.3
    lxyz = 100. * d / np.linalg.norm(d, axis=1, keepdims=True)
    lareas = rng.uniform(0.5, 1.5, L) * 2 * math.pi / L
    light = rng.uniform(0., 3., (L, 3))
    light[rng.uniform(size=L) < 0.05] *= 30.
    albedo = rng.uniform(0.05, 0.9, (n, 3))
    if kind == 0:
        prop = np.array([0.7, 0.4, 0.2])[np.arange(n) % 3][:, None]
    else:
        prop = rng.uniform(0., 1., (n, L))
    d_rgb = rng.standard_normal((n, 3))
    f32 = lambda a: torch.as_tensor(np.ascontiguousarray(a, np.float32))
    return dict(lvis=f32(lvis), normal=f32(nrm), albedo=f32(albedo), prop=f32(prop),
                light=f32(light), xyz=f32(xyz), cam=f32(cam), lxyz=f32(lxyz), lareas=f32(lareas),
                d_rgb=f32(d_rgb))


def _autograd(c, kind, srgb, dtype, device='cuda'):
    """Gradients of autodiff.microfacet_brdf (or albedo / pi + spec * scale) + autodiff.render after
    the normalisation of the raw normal -- the CPU branch of autodiff.integrate, run here as plain
    torch ops in `dtype`."""
    t = {k: v.to(device=device, dtype=dtype) for k, v in c.items()}
    leaves = [t[k].clone().requires_grad_(True) for k in NAMES]
    lvis, normal, albedo, prop, light = leaves
    surf2l = ad.safe_l2_normalize(t['lxyz'].reshape(1, -1, 3) - t['xyz'][:, None, :], 2)
    surf2c = ad.safe_l2_normalize(t['cam'] - t['xyz'], 1)
    nn = ad.safe_l2_normalize(normal, 1)
    if kind == 0:
        brdf = ad.microfacet_brdf(surf2l, surf2c, nn, albedo, prop, F0)
    else:
        n, L = prop.shape
        brdf = albedo[:, None, :] / math.pi + (prop.reshape(n, L, 1) * SPEC_SCALE).expand(n, L, 3)
    rgb = ad.render(lvis, brdf, surf2l, nn, light, t['lareas'], srgb)
    grads = torch.autograd.grad(rgb, leaves, t['d_rgb'])
    return {k: g.detach().double().cpu() for k, g in zip(NAMES, grads)}


def _kernel(ctx, c, kind, srgb, need=NAMES):
    t = {k: v.cuda() for k, v in c.items()}
    pname = 'rough' if kind == 0 else 'spec'
    out = _lib.integrate_bwd(ctx, t['xyz'], t['normal'], t['cam'], t['albedo'], t['lvis'],
                             t['lxyz'], t['lareas'], t['light'], t['d_rgb'],
                             rough=t['prop'] if kind == 0 else None,
                             spec=t['prop'] if kind == 1 else None, f0=F0, spec_scale=SPEC_SCALE,
                             linear2srgb=srgb, need=[pname if k == 'prop' else k for k in need])
    return {('prop' if k == pname else k): v for k, v in out.items()}


@pytest.mark.parametrize('L', [8, 512, 1000])
@pytest.mark.parametrize('n', [1, 33, 3000])
@pytest.mark.parametrize('srgb', [True, False])
@pytest.mark.parametrize('kind', [0, 1])
def test_integrate_bwd_vs_fp64_autograd(ctx, kind, srgb, n, L):
    """Every gradient of nf_integrate_bwd against fp64 autograd of the torch composition, with the
    bar max(3 x the same autograd's own error in fp32, 1e-5) in relative L2 per tensor.
    Measured on a B200 (printed per case): learned lobe <= 4.1e-7 everywhere; microfacet lvis,
    albedo <= 4.8e-7, roughness <= 2.6e-6, light <= 3.8e-6, normal <= 1.9e-5 except at n = 3000,
    L = 1000: 7.7e-4 / 1.0e-3 with sRGB on / off (fp32 autograd: 1.2e-3 / 1.6e-3; grazing views).
    The worst case uses 0.30 of its bar."""
    c = _case(kind, n, L)
    truth = _autograd(c, kind, srgb, torch.float64)
    fp32 = _autograd(c, kind, srgb, torch.float32)
    got = _kernel(ctx, c, kind, srgb)
    torch.cuda.synchronize()
    line = []
    for k in NAMES:
        want = truth[k].numpy().reshape(-1)
        e_k = rel_l2(got[k].cpu().numpy().reshape(-1), want)
        e_32 = rel_l2(fp32[k].numpy().reshape(-1), want)
        line.append('%s %.1e (fp32 autograd %.1e)' % (k, e_k, e_32))
        assert np.isfinite(e_k) and e_k <= max(3 * e_32, 1e-5), (k, e_k, e_32)
    print('integrate_bwd kind %d srgb %d n %d L %d: %s' % (kind, srgb, n, L, ', '.join(line)))


def _raw_call(ctx, t, kind, outs):
    """nf_integrate_bwd through ctypes with caller-owned output buffers (None = NULL)."""
    a = _lib._integrate_args(t['xyz'], t['normal'], t['cam'], t['albedo'], t['lvis'], t['lxyz'],
                             t['lareas'], t['prop'].reshape(-1) if kind == 0 else None,
                             t['prop'] if kind == 1 else None, t['light'].reshape(1, -1, 3),
                             None, None, F0, SPEC_SCALE, True)
    g = _lib.IntegrateGrads()
    g.d_rgb_d = _lib._f32(t['d_rgb'])
    for k, buf in outs.items():
        field = {'prop': 'd_rough_d' if kind == 0 else 'd_spec_d'}.get(k, 'd_%s_d' % k)
        setattr(g, field, _lib._f32(buf) if buf is not None else None)
    nbytes = ctx.lib.nf_integrate_bwd_workspace_bytes(C.byref(a))
    work = torch.empty((nbytes,), dtype=torch.uint8, device='cuda')
    ctx.check(ctx.lib.nf_integrate_bwd(ctx.h, C.byref(a), C.byref(g), _lib._ptr(work), nbytes,
                                       _lib._stream()))


@pytest.mark.parametrize('kind', [0, 1])
def test_null_outputs_are_neither_computed_nor_written(ctx, kind):
    """A subset of the outputs gives those bit-identical to the full call; the buffers of the
    others (not passed: NULL) keep their contents."""
    c = _case(kind, 700, 512, seed=3)
    t = {k: v.cuda() for k, v in c.items()}
    shapes = {k: tuple(t[k].reshape(-1).shape if k == 'prop' and kind == 0 else t[k].shape)
              for k in NAMES}
    full = {k: torch.full(shapes[k], float('nan'), device='cuda') for k in NAMES}
    _raw_call(ctx, t, kind, full)
    for subset in (('normal', 'prop'), ('lvis',), ('light',), ('albedo', 'prop'), ('lvis', 'light')):
        bufs = {k: torch.full(shapes[k], -7.25, device='cuda') for k in NAMES}
        _raw_call(ctx, t, kind, {k: (bufs[k] if k in subset else None) for k in NAMES})
        torch.cuda.synchronize()
        for k in NAMES:
            if k in subset:
                assert torch.equal(bufs[k], full[k]), (subset, k)
            else:
                assert bool((bufs[k] == -7.25).all()), (subset, k)
    assert all(bool(torch.isfinite(v).all()) for v in full.values())


@pytest.mark.parametrize('kind', [0, 1])
def test_two_calls_are_bit_identical(ctx, kind):
    c = _case(kind, 3000, 512, seed=5)
    a = _kernel(ctx, c, kind, True)
    b = _kernel(ctx, c, kind, True)
    for k in NAMES:
        assert torch.equal(a[k], b[k]), k


def test_unsupported_arguments_are_errors(ctx):
    """More than one env-map, a light index map, or d_rough for the learned lobe."""
    c = _case(0, 16, 8)
    t = {k: v.cuda() for k, v in c.items()}
    two = torch.stack((t['light'], t['light']))
    idx = torch.arange(8, dtype=torch.int32, device='cuda')
    d_alb = torch.empty((16, 3), device='cuda')
    for light, light_idx, rough, spec in ((two, None, t['prop'].reshape(-1), None),
                                          (t['light'][None], idx, t['prop'].reshape(-1), None),
                                          (t['light'][None], None, None, t['lvis'])):
        a = _lib._integrate_args(t['xyz'], t['normal'], t['cam'], t['albedo'], t['lvis'], t['lxyz'],
                                 t['lareas'], rough, spec, light, light_idx)
        g = _lib.IntegrateGrads()
        g.d_rgb_d, g.d_albedo_d = _lib._f32(t['d_rgb']), _lib._f32(d_alb)
        if spec is not None:
            g.d_rough_d = _lib._f32(d_alb)
        rc = ctx.lib.nf_integrate_bwd(ctx.h, C.byref(a), C.byref(g), None, 0, _lib._stream())
        assert rc in (-1, -2) and ctx.lib.nf_last_error_string(ctx.h)


@pytest.mark.parametrize('kind', ['microfacet', 'learned'])
def test_trainer_on_the_kernels_vs_reference_tape(ctx, kind, monkeypatch):
    """`Trainer(m, precision='fp32').loss_and_grad` on CUDA (every network on the library's Dense
    kernels, the rendering equation and its adjoint on nf_integrate_fwd / nf_integrate_bwd) against
    the gradients the REFERENCE's train_step produced through the shim
    (tests/golden/ref_tfshim_train_grad_*.npz): per-ray loss and all 41 gradient tensors."""
    from nerfactor_b200.trainvali import Trainer
    calls = []
    real = _lib.integrate_bwd

    def counted(*a, **kw):
        calls.append(kw.get('need'))
        return real(*a, **kw)

    monkeypatch.setattr(_lib, 'integrate_bwd', counted)
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden',
                             'ref_tfshim_train_grad_%s.npz' % kind))
    name = 'nerfactor_microfacet' if kind == 'microfacet' else 'nerfactor'
    Model = import_module('nerfactor_b200.models.' + name).Model
    lh, n = int(g['light_h']), int(g['n_rays'])
    params = synth.make_stage_b_params(int(g['seed_params']), kind, light_hw=(lh, 2 * lh))
    m = Model(nfconfig.default_config(name, light_h=lh), params=params, ctx=ctx, precision='fp32')
    batch = synth.make_stage_b_batch(int(g['seed_batch']), n, 2 * lh * lh, fg_frac=1.0)
    tr = Trainer(m, precision='fp32')
    loss, grad = tr.loss_and_grad(batch, xyz_noise=g['xyz_noise'])
    assert len(calls) == 1 and set(calls[0]) == {
        'lvis', 'normal', 'albedo', 'rough' if kind == 'microfacet' else 'spec', 'light'}
    assert np.allclose(loss.cpu().numpy(), g['per_example_loss'], atol=1e-5, rtol=1e-4)
    gv = tr.views(grad)
    keys = [k for k in g.files if k.startswith('grad/')]
    assert len(keys) == len(gv) == 41
    worst = 0.
    for k in keys:
        parts = k.split('/')
        key = ('light', 0, 'light') if parts[1] == 'light' else (parts[1], int(parts[2]), parts[3])
        want = g[k]
        got = gv[key].cpu().numpy().reshape(want.shape)
        err = np.abs(got - want).max() / max(np.abs(want).max(), 1e-8)
        worst = max(worst, err)
        assert err <= 2e-3, k
    print('trainer (%s) on the kernels vs reference tape: worst max-abs error / max %.2e'
          % (kind, worst))
