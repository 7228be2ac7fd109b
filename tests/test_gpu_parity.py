"""Parity of the CUDA path (through the C ABI) against the CPU oracle.

Tolerances: fp32 kernels 1e-5 (rel-L2); tcgen05 f16 path: rendered RGB within the
north-star's 1e-4 relative L2; bit-exact for ray generation / pixel indexing."""
import os

import numpy as np
import pytest
import torch

from oracle import brdf as obrdf, stage_a, stage_b, networks as onets
from nerfactor_b200 import synth, config as nfconfig

pytestmark = pytest.mark.gpu


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


@pytest.fixture(scope='module')
def ctx():
    from nerfactor_b200 import _lib
    return _lib.default_context()


def dev(x, ctx, dtype=torch.float32):
    return torch.as_tensor(np.ascontiguousarray(x), dtype=dtype).to(ctx.device)


# ------------------------------------------------------------- tcgen05 bring-up
@pytest.mark.parametrize('K', [16, 32, 64, 128])
def test_tcgen05_single_tile_exact(ctx, K):
    """One 128x128xK tile through the TMEM-A / K-major no-swizzle smem-B layouts the fused
    kernels use, and one 256x128xK CTA-pair (cta_group::2) tile: exact on small integers."""
    from nerfactor_b200 import _lib
    rng = np.random.default_rng(K)
    a = rng.integers(-4, 5, (256, K)).astype(np.float32)
    b = rng.integers(-4, 5, (128, K)).astype(np.float32)
    one = _lib.selftest_umma(ctx, dev(a[:128], ctx), dev(b, ctx)).cpu().numpy()
    assert np.array_equal(one, a[:128] @ b.T)
    pair = _lib.selftest_umma2(ctx, dev(a, ctx), dev(b, ctx)).cpu().numpy()
    assert np.array_equal(pair, a @ b.T)


# ------------------------------------------------------------------- Stage A
@pytest.mark.parametrize('hw', [(64, 64), (800, 800), (37, 53)])
def test_gen_rays_bit_exact(ctx, hw):
    from nerfactor_b200 import _lib
    h, w = hw
    c2w = synth.look_at_c2w(4.0, 30.0, 30.0)
    ro, rd = stage_a.gen_rays(c2w, synth.CAM_ANGLE_X, h, w)
    go, gd = _lib.gen_rays(ctx, c2w, synth.CAM_ANGLE_X, h, w)
    assert np.array_equal(go.cpu().numpy(), ro.reshape(-1, 3))
    assert np.array_equal(gd.cpu().numpy(), rd.reshape(-1, 3))     # ray n = y*W + x


def _nerf_model(ctx, seed=3, precision='fp32'):
    from nerfactor_b200.models.nerf import Model
    return Model(nfconfig.default_config('nerf'), params=synth.make_nerf_params(seed),
                 ctx=ctx, precision=precision)


def _rays(ctx, h, w):
    from nerfactor_b200 import _lib
    return _lib.gen_rays(ctx, synth.look_at_c2w(), synth.CAM_ANGLE_X, h, w, normalize=True)


def test_march_single_pass_fp32_vs_oracle_and_golden(ctx, golden_dir):
    from nerfactor_b200 import geometry_from_nerf as gfn
    g = np.load(os.path.join(golden_dir, 'oracle_stage_a.npz'))
    model = _nerf_model(ctx, int(g['seed_nerf']))
    ro, rd = _rays(ctx, 8, 8)
    out = gfn.march_single_pass(model, ro, rd, 32, precision='fp32', want_weights=True)
    assert rel_l2(out['sigma'].cpu(), g['sp_sigma']) < 2e-5
    assert rel_l2(out['weights'].cpu(), g['sp_weights']) < 2e-5
    assert rel_l2(out['depth'].cpu(), g['sp_depth']) < 1e-5
    assert rel_l2(out['occu'].cpu(), g['sp_occu']) < 1e-5
    assert rel_l2(out['surf'].cpu(), g['sp_surf']) < 1e-5


@pytest.fixture(params=['cluster1', 'cluster2', 'pair'])
def sigma_variant(request, monkeypatch):
    """The streamed-weight sigma kernel has three variants (single CTA, 2-CTA multicast
    cluster = default, cta_group::2 CTA pair); all must give the same results."""
    monkeypatch.delenv('NF_SIGMA_PAIR', raising=False)
    monkeypatch.delenv('NF_SIGMA_CLUSTER', raising=False)
    if request.param == 'pair':
        monkeypatch.setenv('NF_SIGMA_PAIR', '1')
    else:
        monkeypatch.setenv('NF_SIGMA_CLUSTER', request.param[-1])
    return request.param


@pytest.mark.parametrize('shape', [(8, 8, 32), (37, 5, 128), (50, 41, 77)])
def test_sigma_tcgen05_vs_fp32_kernel_and_oracle(ctx, shape, sigma_variant):
    """tcgen05 f16 sigma kernel (ragged tile counts, S not a tile divisor) against the
    FP32 kernel; the FP32 kernel against the oracle; bbox masking is exact."""
    from nerfactor_b200 import _lib
    h, w, S = shape
    model = _nerf_model(ctx, 3)
    ro, rd = _rays(ctx, h, w)
    z = _lib.gen_z(ctx, 2., 6., S, h * w)
    mlp_s = model.packed_sigma(True)
    s32 = _lib.sigma_fwd(ctx, mlp_s, ro, rd, z, None, 'fp32')
    s16 = _lib.sigma_fwd(ctx, mlp_s, ro, rd, z, None, 'f16')
    sbf = _lib.sigma_fwd(ctx, mlp_s, ro, rd, z, None, 'bf16')
    assert rel_l2(s16.cpu(), s32.cpu()) < 3e-3
    assert rel_l2(sbf.cpu(), s32.cpu()) < 3e-2
    if h * w * S <= 4096:
        pts = (ro[:, None, :] + rd[:, None, :] * z[:, :, None]).reshape(-1, 3).cpu()
        so = stage_a.eval_sigma_mlp(synth.make_nerf_params(3), pts, True).reshape(h * w, S)
        assert rel_l2(s32.cpu(), so) < 5e-5
    bb = [-1., 1., -1., 1., -1., 1.]
    pts = ro[:, None, :] + rd[:, None, :] * z[:, :, None]
    outside = ((pts < -1.) | (pts > 1.)).any(-1)
    for prec in ('fp32', 'f16'):
        sb = _lib.sigma_fwd(ctx, mlp_s, ro, rd, z, bb, prec)
        assert float(sb[outside].abs().max()) == 0.
        ref = s32 if prec == 'fp32' else s16
        assert torch.equal(sb[~outside], ref[~outside])
    _, occ32, d32, _, _ = _lib.composite(ctx, s32, z, ro, rd)
    _, occ16, d16, _, _ = _lib.composite(ctx, s16, z, ro, rd)
    # fp16 operands: sigma is good to ~1e-3 relative; depth / occupancy follow, except on
    # the rare ray whose LAST sample has sigma within rounding of 0: its delta is 1e10
    # (nerf.py:188-191), so alpha_last jumps between 0 and 1 -- a discontinuity of the
    # reference algorithm itself.  Hence percentiles, not max.
    dd, do = (d32 - d16).abs(), (occ32 - occ16).abs()
    assert float(dd.mean()) < 3e-3 and float(torch.quantile(dd, 0.99)) < 2e-2
    assert float(torch.quantile(do, 0.99)) < 5e-3


def test_sigma_normal_kernel_vs_oracle_autograd(ctx):
    """-l2_normalize(d relu(sigma) / d xyz) (geometry_from_nerf.py:285-300) vs torch autograd."""
    from nerfactor_b200 import _lib
    model = _nerf_model(ctx, 3)
    ro, rd = _rays(ctx, 7, 9)
    S = 19                                             # 63 x 19 rows: ragged last CTA
    z = _lib.gen_z(ctx, 2., 6., S, 63)
    sig, nrm = _lib.sigma_normal_fwd(ctx, model.packed_sigma(True), ro, rd, z)
    pts = (ro[:, None, :] + rd[:, None, :] * z[:, :, None]).reshape(-1, 3).cpu()
    so, no = stage_a.sigma_and_normal(synth.make_nerf_params(3), pts)
    assert rel_l2(sig.cpu().reshape(-1), so.reshape(-1)) < 5e-5
    got, exp = nrm.cpu().reshape(-1, 3).numpy(), no.numpy()
    live = np.linalg.norm(exp, axis=1) > 0.5           # where relu is active
    assert live.sum() > 100
    assert np.abs(got[live] - exp[live]).max() < 2e-3
    assert np.abs(got[~live]).max() < 1e-6             # zero gradient -> zero normal
    # the fp32 forward inside the gradient kernel equals the plain fp32 kernel
    s32 = _lib.sigma_fwd(ctx, model.packed_sigma(True), ro, rd, z, None, 'fp32')
    assert rel_l2(sig.cpu(), s32.cpu()) < 1e-6


def _emulate_sigma_normal_mixed(params, pts, dt):
    """The tcgen05 gradient kernel's arithmetic restated with torch ops on the device:
    operands rounded to `dt` (fp16 / bf16), products accumulated in fp32, ReLU patterns
    taken from the fp32 pre-activations, the backward seed scaled by a power of two.
    Independent of the kernel's tiling / TMEM / barrier structure."""
    q = lambda x: x.to(dt).float()
    dev = pts.device
    Ws = [torch.as_tensor(w, device=dev) for w, _ in params['fine_enc']['layers']]
    bs = [torch.as_tensor(b, device=dev) for _, b in params['fine_enc']['layers']]
    w_out = torch.as_tensor(params['fine_sigma_out']['layers'][0][0], device=dev)[:, 0]
    b_out = float(params['fine_sigma_out']['layers'][0][1][0])
    cols = [pts]
    for f0 in range(0, 10, 3):                    # octaves 0,3,6,9 + double-angle steps
        s, c = torch.sin(pts * float(2 ** f0)), torch.cos(pts * float(2 ** f0))
        for j in range(3):
            if f0 + j < 10:
                cols += [s, c]
                s, c = 2. * s * c, 1. - 2. * s * s
    E = q(torch.cat(cols, 1))                     # [N, 63]
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        h, masks, hf = E, [], None
        for l in range(8):
            if l == 0:
                pre = E @ q(Ws[0]) + bs[0]
            elif l == 5:
                pre = h @ q(Ws[5][:256]) + E @ q(Ws[5][256:]) + bs[5]
            else:
                pre = h @ q(Ws[l]) + bs[l]
            masks.append(pre > 0)
            hf = torch.relu(pre)
            h = q(hf)
        raw = hf @ w_out + b_out
        gs = 2. ** (1 - int(np.frexp(float(w_out.abs().max()))[1]))
        g = q(gs * w_out[None, :] * masks[7])
        GE = torch.zeros_like(E)
        for l in range(7, 0, -1):
            if l == 5:
                GE = GE + g @ q(Ws[5][256:]).t()
            g = q((g @ q(Ws[l][:256]).t()) * masks[l - 1])
        GE = GE + g @ q(Ws[0]).t()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
    grad = GE[:, :3].clone()
    for f in range(10):
        sn, cs = E[:, 3 + 6 * f:6 + 6 * f], E[:, 6 + 6 * f:9 + 6 * f]
        grad = grad + float(2 ** f) * (cs * GE[:, 3 + 6 * f:6 + 6 * f] - sn * GE[:, 6 + 6 * f:9 + 6 * f])
    grad = grad * (raw > 0).float()[:, None] / gs
    nrm = -grad * torch.rsqrt(torch.clamp((grad * grad).sum(1, keepdim=True), min=1e-12))
    return torch.relu(raw), nrm


@pytest.mark.parametrize('prec', ['f16', 'bf16'])
def test_sigma_normal_tcgen05(ctx, prec):
    """nf_sigma_normal_fwd on the tensor cores (forward + input gradient, fp16 / bf16 operands):
    sigma bit-identical to the forward-only kernel; normals (a) agree with a torch restatement
    of the same mixed-precision arithmetic, (b) are independent of which tile / CTA iteration
    a sample lands in, (c) track the FP32 kernel within the operand precision."""
    from nerfactor_b200 import _lib
    model = _nerf_model(ctx, 3)
    mlp = model.packed_sigma(True)
    ro, rd = _rays(ctx, 64, 64)
    S = 19                                              # 77824 samples: 608 tiles, ragged tail
    z = _lib.gen_z(ctx, 2., 6., S, ro.shape[0])
    sig, nrm = _lib.sigma_normal_fwd(ctx, mlp, ro, rd, z, None, prec)
    assert torch.equal(sig, _lib.sigma_fwd(ctx, mlp, ro, rd, z, None, prec))
    assert not torch.isnan(nrm).any()
    # (b) first 147 tiles on their own (one tile per CTA) == the same samples in the long run
    k = 990
    sig_k, nrm_k = _lib.sigma_normal_fwd(ctx, mlp, ro[:k].contiguous(), rd[:k].contiguous(),
                                         z[:k].contiguous(), None, prec)
    assert torch.equal(nrm_k, nrm[:k]) and torch.equal(sig_k, sig[:k])
    # (a) same arithmetic, different machinery
    pts = (ro[:, None, :] + rd[:, None, :] * z[:, :, None]).reshape(-1, 3)
    se, ne = _emulate_sigma_normal_mixed(synth.make_nerf_params(3), pts,
                                         torch.float16 if prec == 'f16' else torch.bfloat16)
    live = (ne.norm(dim=1) > 0.5) & (nrm.reshape(-1, 3).norm(dim=1) > 0.5)
    assert float(live.float().mean()) > 0.1
    d = (nrm.reshape(-1, 3) - ne).abs().max(dim=1).values[live]
    print(prec, 'vs emulation: median', float(d.median()), 'q99', float(torch.quantile(d, .99)),
          'max', float(d.max()))
    assert float(d.median()) < 2e-4 and float(torch.quantile(d, .99)) < 2e-2
    # (c) against the FP32 CUDA-core kernel
    s32, n32 = _lib.sigma_normal_fwd(ctx, mlp, ro, rd, z)
    both = (n32.norm(dim=2) > 0.5) & (nrm.norm(dim=2) > 0.5)
    d32 = (n32 - nrm).abs().max(dim=2).values[both]
    print(prec, 'vs fp32: median', float(d32.median()), 'q90', float(torch.quantile(d32, .9)))
    assert float(d32.median()) < (2e-3 if prec == 'f16' else 6e-2)
    # zero gradient where relu(raw) is off
    off = sig.reshape(-1) == 0
    assert float(nrm.reshape(-1, 3)[off].abs().max()) < 1e-6


def test_compute_depth_and_normal_vs_golden(ctx, golden_dir):
    """Hierarchical camera->surface march (geometry_from_nerf.py:249-319), 32 + 48 samples."""
    from nerfactor_b200 import geometry_from_nerf as gfn
    g = np.load(os.path.join(golden_dir, 'oracle_stage_a.npz'))
    model = _nerf_model(ctx, int(g['seed_nerf']))
    ro, rd = _rays(ctx, 8, 8)
    cfg = nfconfig.default_config('nerf', n_samples_coarse=-32, n_samples_fine=-16)
    occu, depth, normal = gfn.compute_depth_and_normal(model, ro, rd, cfg, precision='fp32')
    d = np.abs(depth.cpu().numpy() - g['h_depth'])
    assert np.median(d) < 1e-4 and np.quantile(d, 0.95) < 5e-3
    assert np.abs(occu.cpu().numpy() - g['h_occu']).max() < 1e-3
    dn = np.abs(normal.cpu().numpy() - g['h_normal']).max(axis=1)
    assert np.median(dn) < 1e-3 and np.quantile(dn, 0.95) < 2e-2


def test_process_view_buffers_vs_oracle(ctx):
    """geometry_from_nerf.process_view (:93-174) without file I/O: alpha / xyz / normal / lvis
    buffers of a 6x6 view against the oracle chain."""
    from nerfactor_b200 import geometry_from_nerf as gfn
    model = _nerf_model(ctx, 3)
    h = w = 6
    ro, rd = _rays(ctx, h, w)
    cfg = nfconfig.default_config('nerf', n_samples_coarse=-32, n_samples_fine=-16)
    out = gfn.process_view(model, ro, rd, (h, w), cfg, light_h=2, precision='fp32')
    nerf = synth.make_nerf_params(3)
    occu, depth, normal = stage_a.compute_depth_and_normal(
        nerf, ro.cpu(), rd.cpu(), 2., 6., n_samples_coarse=-32, n_samples_fine=-16)
    a_o, xyz_o, n_o, surf_o = stage_a.postprocess_view(occu, depth, normal, ro.cpu(), rd.cpu(), (h, w))
    assert np.abs(out['alpha'].cpu().numpy() - a_o.numpy()).max() < 1e-3
    d = np.abs(out['xyz'].cpu().numpy() - xyz_o.numpy()).max(axis=2)
    assert np.median(d) < 1e-3
    assert out['normal'].shape == (h, w, 3) and out['lvis'].shape == (h, w, 8)
    nn = np.linalg.norm(out['normal'].cpu().numpy(), axis=2)
    assert np.allclose(nn, 1., atol=1e-4)
    lv = out['lvis'].cpu().numpy()
    assert lv.min() >= 0. and lv.max() <= 1.


def test_gen_z_and_gen_z_fine_vs_oracle(ctx):
    from nerfactor_b200 import _lib
    rng = np.random.default_rng(0)
    n, sc, sf = 257, 40, 56
    u = rng.uniform(size=(n, sc)).astype(np.float32)
    z_o = stage_a.gen_z(2., 6., sc, n, perturb_u=u)
    z_g = _lib.gen_z(ctx, 2., 6., sc, n, False, dev(u, ctx))
    assert np.allclose(z_g.cpu().numpy(), z_o.numpy(), atol=1e-6)
    w = rng.uniform(size=(n, sc)).astype(np.float32) ** 4
    w[:5] = 0.                                            # empty rays: denom -> eps
    zf_o = stage_a.gen_z_fine(z_o, torch.tensor(w), sf)
    zf_g = _lib.gen_z_fine(ctx, z_g, dev(w, ctx), sf)
    got = zf_g.cpu().numpy()
    assert np.all(np.diff(got, axis=1) >= 0)              # sortedness
    # inv_transform_sample is discontinuous where a cdf bin is ~1e-5 wide
    # (`denom < eps -> 1`, util/math.py:90-91): a 1-ulp difference in the cumsum can
    # move such a sample inside its bin.  Everything else agrees to fp32 rounding.
    d = np.abs(got - zf_o.numpy())
    assert (d > 2e-5).mean() < 1e-3 and d.max() < 4. / sc


def test_composite_weights_vs_oracle(ctx):
    from nerfactor_b200 import _lib
    rng = np.random.default_rng(1)
    n, s = 300, 77
    sigma = (rng.standard_normal((n, s)) * 5).astype(np.float32)
    z = np.sort(rng.uniform(2, 6, (n, s)).astype(np.float32), axis=1)
    rd = rng.standard_normal((n, 3)).astype(np.float32)
    ro = rng.standard_normal((n, 3)).astype(np.float32)
    nrm = rng.standard_normal((n, s, 3)).astype(np.float32)
    w_o = stage_a.accumulate_sigma(torch.tensor(sigma), torch.tensor(z), torch.tensor(rd))
    w, occu, depth, surf, en = _lib.composite(
        ctx, dev(sigma, ctx), dev(z, ctx), dev(ro, ctx), dev(rd, ctx), dev(nrm, ctx))
    assert np.allclose(w.cpu().numpy(), w_o.numpy(), atol=2e-6)
    assert np.allclose(occu.cpu().numpy(), w_o.sum(-1).numpy(), atol=1e-5)
    assert np.allclose(depth.cpu().numpy(), (w_o * torch.tensor(z)).sum(-1).numpy(), atol=2e-5)
    en_o = (w_o[:, :, None] * torch.tensor(nrm)).sum(-2).numpy()
    assert np.allclose(en.cpu().numpy(), en_o, atol=2e-5)


def test_light_visibility_march_fp32_vs_oracle(ctx):
    from nerfactor_b200 import geometry_from_nerf as gfn
    model = _nerf_model(ctx, 3)
    cfg = nfconfig.default_config('nerf', n_samples_coarse=-32, n_samples_fine=-16)
    rng = np.random.default_rng(5)
    surf = rng.uniform(-1, 1, (24, 3)).astype(np.float32)
    nrm = rng.standard_normal((24, 3)).astype(np.float32)
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    lx, _ = obrdf.gen_light_xyz(2, 4)
    model.precision = 'fp32'
    got = gfn.compute_light_visibility(model, dev(surf, ctx), dev(nrm, ctx), cfg, lxyz=lx)
    nerf = synth.make_nerf_params(3)
    exp = stage_a.compute_light_visibility(nerf, torch.tensor(surf), torch.tensor(nrm), lx,
                                           n_samples_coarse=-32, n_samples_fine=-16)
    assert np.allclose(got.cpu().numpy(), exp.numpy(), atol=3e-4)


# ------------------------------------------------------------------- Stage B
def _stage_b(ctx, brdf, lh, lw, seed=7, precision='f16', **kw):
    name = 'nerfactor_microfacet' if brdf == 'microfacet' else 'nerfactor'
    from importlib import import_module
    Model = import_module('nerfactor_b200.models.' + name).Model
    params = synth.make_stage_b_params(seed, brdf, light_hw=(lh, lw))
    cfg = nfconfig.default_config(name, light_h=lh)
    m = Model(cfg, params=params, ctx=ctx, precision=precision, **kw)
    lxyz, lareas = obrdf.gen_light_xyz(lh, lw)
    m.set_lights(lxyz.reshape(-1, 3), lareas.reshape(-1))
    m.light_res = (lh, lw)
    om = stage_b.StageB(params, {'brdf': brdf}, lxyz=lxyz, lareas=lareas)
    return m, om, params


@pytest.mark.parametrize('brdf', ['microfacet', 'learned'])
@pytest.mark.parametrize('precision', ['fp32', 'f16'])
def test_model_call_matches_golden(ctx, golden_dir, brdf, precision):
    """Config-1-like case (96 rays, L=16): full Model.call vs the frozen oracle vectors."""
    g = np.load(os.path.join(golden_dir, 'oracle_stage_b_%s.npz' % brdf))
    lh, lw = int(g['lh']), int(g['lw'])
    m, _, _ = _stage_b(ctx, brdf, lh, lw, int(g['seed_params']), precision)
    batch = synth.make_stage_b_batch(int(g['seed_batch']), int(g['n_rays']), lh * lw)
    probes = synth.make_probes(int(g['seed_probes']), 3, (lh, lw))
    for i, p in enumerate(probes):
        m.novel_probes['p%d' % i] = p
    pred, gt, lk, _ = m.call(batch, 'test', relight_probes=True)
    tol_net = 1e-5 if precision == 'fp32' else 3e-3
    assert rel_l2(pred['normal'].cpu(), g['normal']) < 1e-5
    assert rel_l2(pred['albedo'].cpu(), g['albedo']) < 1e-5
    assert rel_l2(pred['brdf'].cpu(), g['brdf']) < 1e-5
    assert rel_l2(pred['lvis'].cpu(), g['lvis']) < tol_net
    tol_rgb = 1e-5 if precision == 'fp32' else 1e-4      # north-star bar on RGB
    assert rel_l2(pred['rgb'].cpu(), g['rgb']) < tol_rgb
    assert rel_l2(pred['rgb_probes'].cpu(), g['rgb_relit']) < tol_rgb
    bg = batch[5][:, 0] == 0
    assert np.all(pred['rgb'].cpu().numpy()[bg] == 0)    # background rows stay zero


@pytest.mark.parametrize('brdf', ['microfacet', 'learned'])
def test_stage_b_l512_rgb_within_1e4(ctx, brdf):
    """Reference-native light grid (16x32 = 512 lights), ragged N (not a tile multiple)."""
    m, om, _ = _stage_b(ctx, brdf, 16, 32, seed=21, precision='f16')
    batch = synth.make_stage_b_batch(22, 203, 512)
    pred, _, _, _ = m.call(batch, 'test', relight_olat=True)
    opred, _, _ = om.call(batch, 'test', relight_lights=om.novel_olat((16, 32))[:40])
    assert rel_l2(pred['rgb'].cpu(), opred['rgb']) < 1e-4
    assert rel_l2(pred['lvis'].cpu(), opred['lvis']) < 3e-3
    assert rel_l2(pred['rgb_olat'].cpu().numpy()[:, :40], opred['rgb_relit']) < 1e-4


@pytest.mark.parametrize('brdf,lh,lw,n', [('microfacet', 16, 32, 1000), ('microfacet', 10, 20, 203),
                                          ('learned', 16, 32, 333), ('microfacet', 16, 64, 150)])
@pytest.mark.parametrize('single', [False, True])
def test_fused_stage_b_equals_model_call(ctx, brdf, lh, lw, n, single, monkeypatch, request):
    """Model.render_rgb (nf_stageB_fused_fwd) against Model.call on the same batch: the
    single-kernel case (microfacet, one env-map, L <= 512: rendering equation inside the head
    epilogue of the visibility network; ragged L = 200 too), the chunked cases (learned lobe;
    L = 1024; several env-maps), with and without the optional lvis output -- and against the
    oracle for RGB."""
    if single and os.environ.get('NF_STAGEB_SINGLE') != '1':
        # the library reads NF_STAGEB_SINGLE once per process: run this case in a fresh one
        import subprocess
        import sys
        r = subprocess.run([sys.executable, '-m', 'pytest', '-q', '-p', 'no:cacheprovider',
                            request.node.nodeid], cwd=str(request.config.rootpath),
                           env=dict(os.environ, NF_STAGEB_SINGLE='1'), capture_output=True,
                           text=True, timeout=900)
        assert r.returncode == 0 and '1 passed' in r.stdout, r.stdout[-4000:] + r.stderr[-2000:]
        return
    m, om, _ = _stage_b(ctx, brdf, lh, lw, seed=13, precision='f16')
    for i, p in enumerate(synth.make_probes(5, 3, light_hw=(lh, lw))):
        m.novel_probes['p%d' % i] = p
    batch = synth.make_stage_b_batch(31, n, lh * lw)
    ref = m.call(batch, 'test', relight_probes=True)[0]
    out = m.render_rgb(batch)
    out_l = m.render_rgb(batch, want_lvis=True)
    out_a = m.render_rgb(batch, all_lights=True)
    out_p = m.render_rgb(batch, relight_probes=True, want_lvis=True)
    for k in ('normal', 'albedo', 'brdf'):
        assert torch.equal(out[k], ref[k])
    assert torch.equal(out_l['lvis'], ref['lvis']) and torch.equal(out_p['lvis'], ref['lvis'])
    # without the lvis output the visibility network skips the lights facing away from the normal
    # (zero weight in the renderer, nerfactor.py:329-330): rows are independent, so the sums are
    # the same bit for bit as with every light evaluated
    assert torch.equal(out['rgb'], out_l['rgb']) and torch.equal(out_a['rgb'], out_l['rgb'])
    assert rel_l2(out['rgb'].cpu(), ref['rgb'].cpu()) < 1e-5
    assert rel_l2(out_p['rgb_probes'].cpu(), ref['rgb_probes'].cpu()) < 1e-5
    assert float(out['rgb'][torch.as_tensor(batch[5][:, 0] == 0)].abs().max()) == 0.
    opred = om.call(batch, 'test')[0]
    assert rel_l2(out['rgb'].cpu(), opred['rgb']) < 1e-4       # north-star bar vs the oracle
    empty = tuple(x[:0] if isinstance(x, np.ndarray) else x for x in batch)
    assert m.render_rgb(empty)['rgb'].shape == (0, 3)


def test_front_lit_culling_with_unlit_points(ctx):
    """nf_stageB_fused_fwd without the lvis output evaluates the visibility network only for the
    lights facing the shading normal (nerfactor.py:329-330 zeroes the others).  Lights on the upper
    cap only + normals pointing down make whole points unlit: runs of such points at the start,
    in the middle and at the end of a worker group's point sequence, and alternating ones, must
    neither hang the kernel's point pipeline nor change a colour (bit-equal to all lights)."""
    from nerfactor_b200 import _lib
    m, _, _ = _stage_b(ctx, 'microfacet', 16, 32, seed=7, precision='f16')
    lx_all, la_all = m.lxyz.reshape(-1, 3), m.lareas.reshape(-1)
    keep = lx_all[:, 2] > 30.
    lxyz, lareas = lx_all[keep].contiguous(), la_all[keep].contiguous()
    L = int(lxyz.shape[0])
    assert 100 < L < 400
    n_groups = 2 * int(ctx.sm_count)
    n = 6 * n_groups
    rng = np.random.default_rng(17)
    seq, grp = np.arange(n) // n_groups, np.arange(n) % n_groups
    unlit = ((grp % 4 == 0) & np.isin(seq, (1, 2))) | ((grp % 4 == 1) & np.isin(seq, (0, 1))) | \
            ((grp % 4 == 2) & np.isin(seq, (4, 5))) | ((grp % 4 == 3) & (seq % 2 == 0))
    nrm = rng.standard_normal((n, 3)).astype(np.float32)
    nrm[:, 2] = np.abs(nrm[:, 2]) + 0.5
    nrm /= np.linalg.norm(nrm, axis=1, keepdims=True)
    nrm[unlit] = (0., 0., -1.)
    xyz = dev(rng.uniform(-.5, .5, (n, 3)).astype(np.float32), ctx)
    normal = dev(nrm, ctx)
    cam = dev((rng.standard_normal((n, 3)) * .1 + (0., 0., 4.)).astype(np.float32), ctx)
    albedo = dev(rng.uniform(.1, .9, (n, 3)).astype(np.float32), ctx)
    rough = dev(rng.uniform(.2, .8, (n,)).astype(np.float32), ctx)
    light = dev(rng.uniform(0., 2., (1, L, 3)).astype(np.float32), ctx)
    mlp = m._packed_mlp('lvis', 'lvis', n_freqs_a=m.embedder['xyz'].n_freqs,
                        n_freqs_b=m.embedder['ldir'].n_freqs)
    run = lambda **kw: _lib.stageB_fused_fwd(ctx, mlp, xyz, normal, cam, albedo, lxyz, lareas, light,
                                             rough=rough, precision='f16', **kw)
    rgb_c, _ = run()
    rgb_a, _ = run(all_lights=True)
    rgb_f, lv_f = run(want_lvis=True, all_lights='front_lit')
    rgb_l, lv = run(want_lvis=True)
    assert torch.equal(rgb_c, rgb_a) and torch.equal(rgb_f, rgb_a) and torch.equal(rgb_l, rgb_a)
    u = torch.as_tensor(unlit, device=lv.device)
    assert float(lv_f[u].abs().max()) == 0. and float(rgb_c[u].abs().max()) == 0.
    nz = lv_f != 0
    assert 0.2 < float(nz[~u].float().mean()) <= 1.
    assert torch.equal(lv_f[nz], lv[nz])


def test_composite_ops_are_chunk_invariant(ctx):
    """The one-call ops process their input in chunks (32768 rays; 2^19 (point, light) pairs;
    <= 48 MB of visibility rows): a multi-chunk call must equal the concatenation of single-chunk
    calls bit for bit (every ray / pair / point is independent)."""
    from nerfactor_b200 import geometry_from_nerf as gfn
    model = _nerf_model(ctx, 3, precision='f16e')
    cfg = nfconfig.default_config('nerf', n_samples_coarse=-48, n_samples_fine=-52)   # 16 + 12 samples
    ro, rd = _rays(ctx, 210, 200)                                                      # 42000 rays: 2 chunks
    occu, depth, normal = gfn.compute_depth_and_normal(model, ro, rd, cfg)
    k = 32768
    for lo, hi in ((0, k), (k, ro.shape[0])):
        o2, d2, n2 = gfn.compute_depth_and_normal(model, ro[lo:hi].contiguous(), rd[lo:hi].contiguous(), cfg)
        assert torch.equal(occu[lo:hi], o2) and torch.equal(depth[lo:hi], d2) and torch.equal(normal[lo:hi], n2)
    # light march: 1300 points x 512 lights = 665600 pairs (2 chunks; the boundary falls inside a point)
    rng = np.random.default_rng(8)
    surf = dev(rng.uniform(-1, 1, (1300, 3)).astype(np.float32), ctx)
    nrm = rng.standard_normal((1300, 3)).astype(np.float32)
    nrm = dev(nrm / np.linalg.norm(nrm, axis=1, keepdims=True), ctx)
    lv = gfn.compute_light_visibility(model, surf, nrm, cfg, light_h=16)
    for lo, hi in ((0, 700), (700, 1300)):
        part = gfn.compute_light_visibility(model, surf[lo:hi].contiguous(), nrm[lo:hi].contiguous(), cfg,
                                            light_h=16)
        assert torch.equal(lv[lo:hi], part)
    # 1 - sum(w) with w from the +1e-6 cumprod (util/math.py:67-68) may undershoot 0 by ~1e-5;
    # the caller clips (gfn.py:160)
    assert float(lv.min()) >= -1e-3 and float(lv.max()) <= 1. + 1e-6
    frac_lit = float((lv != 0).float().mean())
    assert 0.3 < frac_lit < 0.7                       # back-lit pairs stay exactly 0
    # fused Stage B: 60000 points x 512 lights = 3 chunks of 24576 points
    m, _, _ = _stage_b(ctx, 'microfacet', 16, 32, seed=5, precision='f16')
    batch = synth.make_stage_b_batch(9, 60000, 1, fg_frac=1.0)
    big = m.render_rgb(batch)['rgb']
    ref = m.call(batch, 'test')[0]['rgb']
    assert rel_l2(big.cpu(), ref.cpu()) < 1e-6
    sub = tuple(x[20000:40000] if isinstance(x, np.ndarray) else x for x in batch)
    assert torch.equal(m.render_rgb(sub)['rgb'], big[20000:40000])


def test_lvis_jitter_semantics_tensor_core_path(ctx):
    """shape.py:170 / nerfactor.py:225: the jittered visibility is the network at xyz + noise with
    the light directions of xyz.  nf_lvis_dirs_fwd (fp16 operands) against the oracle, and it
    differs from evaluating everything at the jittered point."""
    m, om, _ = _stage_b(ctx, 'microfacet', 10, 20, seed=3, precision='f16')
    rng = np.random.default_rng(2)
    xyz = torch.as_tensor(rng.uniform(-1, 1, (301, 3)).astype(np.float32))
    noise = torch.as_tensor((0.05 * rng.standard_normal((301, 3))).astype(np.float32))
    got = m._pred_lvis_jitter_at(dev(xyz + noise, ctx), dev(xyz, ctx)).cpu()
    want = om.pred_lvis_at(xyz + noise, om.calc_ldir(xyz))
    assert rel_l2(got, want) < 3e-3
    moved = om.pred_lvis_at(xyz + noise, om.calc_ldir(xyz + noise))
    assert rel_l2(got, moved) > 3 * rel_l2(got, want)
    # same inputs for both origins == the plain kernel, bit for bit
    a = m._pred_lvis_jitter_at(dev(xyz, ctx), dev(xyz, ctx))
    assert torch.equal(a, m._pred_lvis_at(dev(xyz, ctx)))


def test_config3_learned_brdf_1024_lights_on_16x32_envmap(ctx):
    """BASELINE configs[2]: learned-MERL BRDF, L = 1024 light directions (16x64 grid) looking
    up a 16x32 HDR env-map through the nearest-pixel index map (SURVEY 8d caveat on L)."""
    from nerfactor_b200.models.nerfactor import Model
    params = synth.make_stage_b_params(41, 'learned', light_hw=(16, 32))
    lxyz, lareas = obrdf.gen_light_xyz(16, 64)
    idx = synth.light_index_map((16, 32), (16, 64))
    m = Model(nfconfig.default_config('nerfactor'), params=params, ctx=ctx, precision='f16')
    m.set_lights(lxyz.reshape(-1, 3), lareas.reshape(-1), light_idx=idx)
    om = stage_b.StageB(params, {'brdf': 'learned'}, lxyz=lxyz, lareas=lareas, light_idx=idx)
    batch = synth.make_stage_b_batch(42, 77, 1024)
    probes = synth.make_probes(43, 2, (16, 32))
    for i, p_ in enumerate(probes):
        m.novel_probes['hdr%d' % i] = p_
    pred, _, _, _ = m.call(batch, 'test', relight_probes=True)
    opred, _, _ = om.call(batch, 'test', relight_lights=[p_ for p_ in probes])
    assert pred['lvis'].shape == (77, 1024)
    assert rel_l2(pred['rgb'].cpu(), opred['rgb']) < 1e-4
    assert rel_l2(pred['rgb_probes'].cpu(), opred['rgb_relit']) < 1e-4


def test_config5_relight_sweep_eight_envmaps(ctx):
    """BASELINE configs[4] per-GPU slice: one view relit under 8 env-maps in one call
    (two passes of four inside nf_integrate_fwd)."""
    m, om, _ = _stage_b(ctx, 'learned', 16, 32, seed=51, precision='f16')
    batch = synth.make_stage_b_batch(52, 150, 512)
    probes = synth.make_probes(53, 8, (16, 32))
    for i, p_ in enumerate(probes):
        m.novel_probes['env%d' % i] = p_
    pred, _, _, _ = m.call(batch, 'test', relight_probes=True)
    opred, _, _ = om.call(batch, 'test', relight_lights=[p_ for p_ in probes])
    assert pred['rgb_probes'].shape == (150, 8, 3)
    assert rel_l2(pred['rgb_probes'].cpu(), opred['rgb_relit']) < 1e-4
    # overrides of test.py:91-132: global albedo override and BRDF-latent override
    z = np.array([0.01, -0.02, 0.005], np.float32)
    alb = np.array([0.3, 0.5, 0.7], np.float32)
    p2, _, _, _ = m.call(batch, 'test', albedo_override=alb, brdf_z_override=z)
    o2, _, _ = om.call(batch, 'test', albedo_override=alb, brdf_z_override=z)
    assert rel_l2(p2['rgb'].cpu(), o2['rgb']) < 1e-4
    assert rel_l2(p2['albedo'].cpu(), o2['albedo']) < 1e-6


def test_ragged_light_count_xyz_scale_and_ambient_olat(ctx):
    """L = 200 (10 x 20 grid: two tiles per point, the second one ragged), xyz_scale != 1
    (shape.py:47-48), and OLAT relighting with ambient light (nerfactor.py:68-84)."""
    from nerfactor_b200.models.nerfactor import Model
    lh, lw = 10, 20
    params = synth.make_stage_b_params(61, 'learned', light_hw=(lh, lw))
    lxyz, lareas = obrdf.gen_light_xyz(lh, lw)
    cfg = nfconfig.default_config('nerfactor', light_h=lh, xyz_scale=0.37, ambient_inten=0.25)
    m = Model(cfg, params=params, ctx=ctx, precision='f16')
    m.set_lights(lxyz.reshape(-1, 3), lareas.reshape(-1))
    m.light_res = (lh, lw)
    om = stage_b.StageB(params, {'brdf': 'learned', 'xyz_scale': 0.37, 'ambient_inten': 0.25},
                        lxyz=lxyz, lareas=lareas)
    batch = synth.make_stage_b_batch(62, 45, lh * lw)
    pred, _, _, _ = m.call(batch, 'test', relight_olat=True)
    olats = om.novel_olat((lh, lw))
    opred, _, _ = om.call(batch, 'test', relight_lights=olats[:25] + olats[-5:])
    assert pred['lvis'].shape == (45, 200)
    assert rel_l2(pred['lvis'].cpu(), opred['lvis']) < 3e-3
    assert rel_l2(pred['rgb'].cpu(), opred['rgb']) < 1e-4
    got = pred['rgb_olat'].cpu().numpy()
    sel = np.concatenate((got[:, :25], got[:, -5:]), axis=1)
    assert rel_l2(sel, opred['rgb_relit']) < 1e-4
    for prec, tol in (('fp32', 1e-5), ('bf16', 2e-3)):
        m.precision = prec
        p2, _, _, _ = m.call(batch, 'test')
        assert rel_l2(p2['rgb'].cpu(), opred['rgb']) < tol, prec


@pytest.mark.parametrize('n', [1, 127, 128, 1000])
def test_point_networks_f16x3_tcgen05_vs_fp32_and_oracle(ctx, n):
    """Per-point nets on tensor cores with the 3-term fp16 split: fp32-level accuracy."""
    from nerfactor_b200 import _lib
    m, om, _ = _stage_b(ctx, 'learned', 2, 8, seed=5)
    xyz = np.random.default_rng(n).uniform(-1.5, 1.5, (n, 3)).astype(np.float32)
    xt = dev(xyz, ctx)
    for name in ('normal', 'albedo', 'brdf_z'):
        pm = m._packed_mlp(name, 'point', n_freqs_a=10)
        a32 = _lib.point_mlp_fwd(ctx, pm, xt, 1.0, 'fp32').cpu().numpy()
        a3 = _lib.point_mlp_fwd(ctx, pm, xt, 1.0, 'f16x3').cpu().numpy()
        o = om._point_mlp(name, torch.tensor(xyz)).numpy()
        assert rel_l2(a32, o) < 2e-6 and rel_l2(a3, o) < 1e-5, name
    with pytest.raises(_lib.NfError):
        _lib.point_mlp_fwd(ctx, pm, xt, 1.0, 'f16')       # plain fp16 is refused for these nets


def test_lvis_and_brdf_kernels_fp32_vs_f16_vs_oracle(ctx):
    from nerfactor_b200 import _lib
    m, om, params = _stage_b(ctx, 'learned', 16, 32, seed=5, precision='f16')
    rng = np.random.default_rng(9)
    n = 70
    xyz = rng.uniform(-1.2, 1.2, (n, 3)).astype(np.float32)
    xt = dev(xyz, ctx)
    surf2l = om.calc_ldir(torch.tensor(xyz))
    lv_o = om.pred_lvis_at(torch.tensor(xyz), surf2l).numpy()
    mlp_l = m._packed_mlp('lvis', 'lvis', n_freqs_a=10, n_freqs_b=4)
    lv32 = _lib.lvis_fwd(ctx, mlp_l, xt, m.lxyz, 1.0, 'fp32').cpu().numpy()
    lv16 = _lib.lvis_fwd(ctx, mlp_l, xt, m.lxyz, 1.0, 'f16').cpu().numpy()
    lvbf = _lib.lvis_fwd(ctx, mlp_l, xt, m.lxyz, 1.0, 'bf16').cpu().numpy()
    assert np.abs(lv32 - lv_o).max() < 2e-5
    assert np.abs(lv16 - lv_o).max() < 4e-3 and rel_l2(lv16, lv_o) < 1.5e-3
    assert np.abs(lvbf - lv_o).max() < 3e-2 and rel_l2(lvbf, lv_o) < 1e-2


def test_empty_and_all_background(ctx):
    m, _, _ = _stage_b(ctx, 'microfacet', 2, 8)
    batch = list(synth.make_stage_b_batch(3, 33, 16))
    batch[5] = np.zeros_like(batch[5])                     # alpha = 0 everywhere
    pred, _, _, _ = m.call(tuple(batch), 'test')
    assert pred['rgb'].shape == (33, 3) and float(pred['rgb'].abs().sum()) == 0.
    with pytest.raises(ValueError):
        m.call(tuple(batch), 'predict')                    # models/base.py:107-110


def test_loss_matches_oracle(ctx):
    m, om, _ = _stage_b(ctx, 'learned', 2, 8, seed=7, precision='fp32')
    batch = synth.make_stage_b_batch(11, 64, 16)
    nfg = int((batch[5][:, 0] > 0).sum())
    noise = (0.01 * np.random.default_rng(2).standard_normal((nfg, 3))).astype(np.float32)
    pred, gt, lk, _ = m.call(batch, 'train', xyz_noise=noise)
    loss = m.compute_loss(pred, gt, **lk)
    opred, ogt, olk = om.call(batch, 'train', xyz_noise=noise)
    oloss = om.compute_loss(opred, ogt, **olk)
    assert np.allclose(loss.cpu().numpy(), oloss.numpy(), atol=2e-6, rtol=1e-4)


def test_full_size_properties(ctx):
    """800x800-scale properties the oracle cannot check in seconds: linearity of the
    rendering equation in the env-map before tonemapping, permutation equivariance
    over rays, and OLAT consistency (sum of OLAT renders == white-light render)."""
    from nerfactor_b200 import _lib
    m, _, _ = _stage_b(ctx, 'microfacet', 16, 32, seed=31)
    n = 20000
    batch = synth.make_stage_b_batch(32, n, 512, fg_frac=1.0)
    xyz, nrm, cam = dev(batch[6], ctx), dev(batch[7], ctx), dev(batch[2], ctx)
    albedo = dev(np.full((n, 3), .5, np.float32), ctx)
    rough = dev(np.full((n, 1), .4, np.float32), ctx)
    lvis = m._pred_lvis_at(xyz)
    args = dict(lxyz=m.lxyz, lareas=m.lareas, rough=rough, f0=0.04, linear2srgb=False)
    la = torch.rand((1, 512, 3), device=ctx.device) * 1e-3     # small: stay below the clip
    lb = torch.rand((1, 512, 3), device=ctx.device) * 1e-3
    ra = _lib.integrate_fwd(ctx, xyz, nrm, cam, albedo, lvis, light=la, **args)
    rb = _lib.integrate_fwd(ctx, xyz, nrm, cam, albedo, lvis, light=lb, **args)
    rab = _lib.integrate_fwd(ctx, xyz, nrm, cam, albedo, lvis, light=la + lb, **args)
    assert rel_l2((ra + rb).cpu(), rab.cpu()) < 1e-5
    perm = torch.randperm(n, device=ctx.device)
    lvis_p = m._pred_lvis_at(xyz[perm].contiguous())
    assert torch.equal(lvis_p, lvis[perm])                  # rays are independent
    olat = _lib.integrate_olat_fwd(ctx, xyz, nrm, cam, albedo, lvis, olat_inten=1e-3,
                                   ambient=0., **args)
    white = _lib.integrate_fwd(ctx, xyz, nrm, cam, albedo, lvis,
                               light=torch.full((1, 512, 3), 1e-3, device=ctx.device), **args)
    assert rel_l2(olat.sum(1).cpu(), white[:, 0].cpu()) < 1e-4


def test_integrate_kernel_vs_reference_sphere_renderer(ctx, golden_dir):
    """nf_integrate_fwd / nf_integrate_olat_fwd against numbers produced by the REFERENCE ITSELF:
    its NumPy light-stage renderer (brdf/renderer.py SphereRenderer, run in the build container by
    tests/golden/make_golden.py) on its sphere scene, Lambertian BRDF, seeded env-map with one
    bright texel.  Pins light directions, cosine, area weights, front-lit mask, env-map lookup and
    the hemisphere sum of the kernels without going through the oracle."""
    from nerfactor_b200 import _lib
    g = np.load(os.path.join(golden_dir, 'ref_sphere_renderer.npz'))
    fg = g['is_fg']
    n = int(fg.sum())
    L = g['lxyz'].shape[0] * g['lxyz'].shape[1]
    xyz, nrm, alb = [dev(g[k][fg].astype(np.float32), ctx) for k in ('xyz', 'normal', 'albedo')]
    cam = dev(np.tile(g['cam_loc'].astype(np.float32)[None], (n, 1)), ctx)
    lvis = torch.ones((n, L), device=ctx.device)
    zeros = torch.zeros((n, L), device=ctx.device)
    lxyz = dev(g['lxyz'].reshape(-1, 3).astype(np.float32), ctx)
    lareas = dev(g['lareas'].reshape(-1).astype(np.float32), ctx)
    light = dev(g['envmap'].reshape(1, L, 3).astype(np.float32), ctx)
    want = g['render'][fg]
    # pre-computed-lobe variant with a zero lobe = pure Lambert albedo / pi
    rgb = _lib.integrate_fwd(ctx, xyz, nrm, cam, alb, lvis, lxyz, lareas, light, spec=zeros,
                             spec_scale=1.0, linear2srgb=False)[:, 0]
    assert rel_l2(rgb.cpu(), want) < 5e-6
    # eight copies of the env-map in one call (EC = 8 path), each scaled differently
    scales = torch.arange(1, 9, device=ctx.device, dtype=torch.float32)[:, None, None] / 8
    rgb8 = _lib.integrate_fwd(ctx, xyz, nrm, cam, alb, lvis, lxyz, lareas,
                              (light * scales).contiguous(), spec=zeros, spec_scale=1.0,
                              linear2srgb=False)
    for e in range(8):
        assert rel_l2(rgb8[:, e].cpu(), want * (e + 1) / 8) < 5e-6, e
    # OLAT kernel: env-map = inten * onehot(l); summing the one-light renders weighted by the
    # texel values reproduces the env-map render (per channel)
    olat = _lib.integrate_olat_fwd(ctx, xyz, nrm, cam, alb, lvis, lxyz, lareas, olat_inten=1.0,
                                   ambient=0., spec=zeros, spec_scale=1.0, linear2srgb=False)
    recon = torch.einsum('nlc,lc->nc', olat, light[0])
    assert rel_l2(recon.cpu(), want) < 5e-6


def test_integrate_kernels_vs_fp64_incl_grazing_views(ctx):
    """Both rendering-equation kernels (packed-FP32 nf_integrate_fwd, scalar nf_integrate_olat_fwd)
    against an fp64 evaluation of the reference formulas, LINEAR output (no clip / tone curve to
    hide errors), normals that put many points at grazing view angles (n.v -> 0, where the GGX
    normalisation |l + v| -> 0 is ill-conditioned).  The fp32 reference formulas themselves sit at
    ~1e-6 (rough 0.4) / ~6e-5 (rough 0.2) from fp64 here."""
    import cpu_backend as cb
    from nerfactor_b200 import _lib
    from nerfactor_b200.brdf.renderer import gen_light_xyz
    n, L = 3000, 512
    batch = synth.make_stage_b_batch(32, n, L, fg_frac=1.0)
    lxyz, lareas = gen_light_xyz(16, 32)
    lx = torch.as_tensor(lxyz.reshape(-1, 3).astype(np.float32))
    la = torch.as_tensor(lareas.reshape(-1).astype(np.float32))
    xyz, nrm, cam = [torch.as_tensor(batch[i]) for i in (6, 7, 2)]
    lvis = torch.as_tensor(batch[8])
    alb = torch.full((n, 3), .5)
    # packed kernel: the GGX normalisation is formed from the component of l + v orthogonal to n
    # (csrc/nf_integrate.cu), which keeps it within 1e-4 of fp64 down to roughness 0.2
    for rough_v, tol_packed, tol_scalar in ((0.7, 2e-6, 1e-6), (0.4, 1e-5, 5e-6), (0.2, 1e-4, 3e-4)):
        rough = torch.full((n, 1), rough_v)
        c64 = cb._pair_terms(xyz.double(), nrm.double(), cam.double(), alb.double(), lvis.double(),
                             lx.double(), la.double(), rough.double(), None, 0.04, 1.0)
        truth = (c64.sum(1) * 1e-3).numpy()
        args = dict(lxyz=dev(lx, ctx), lareas=dev(la, ctx), rough=dev(rough, ctx), f0=0.04,
                    linear2srgb=False)
        pts = [dev(t, ctx) for t in (xyz, nrm, cam, alb, lvis)]
        white = torch.full((1, L, 3), 1e-3, device=ctx.device)
        packed = _lib.integrate_fwd(ctx, *pts, light=white, **args)[:, 0]
        scalar = _lib.integrate_olat_fwd(ctx, *pts, olat_inten=1e-3, ambient=0., **args).sum(1)
        print('integrate vs fp64, roughness %.1f: packed %.2e  scalar %.2e'
              % (rough_v, rel_l2(packed.cpu(), truth), rel_l2(scalar.cpu(), truth)))
        assert rel_l2(packed.cpu(), truth) < tol_packed, rough_v
        assert rel_l2(scalar.cpu(), truth) < tol_scalar, rough_v


def test_microfacet_class_callable_vs_oracle(ctx):
    """`Microfacet(...)(pts2l, pts2c, normal, albedo, rough)` -- the reference's class surface
    (brdf/microfacet/microfacet.py:30-72) -- through nf_microfacet_brdf_fwd, against the oracle's
    restatement; defaults (albedo None, rough None), lambert_only, un-normalised inputs."""
    from nerfactor_b200.brdf.microfacet.microfacet import Microfacet
    rng = np.random.default_rng(4)
    n, L = 257, 33
    pts2l = rng.standard_normal((n, L, 3)).astype(np.float32) * 3.
    pts2c = rng.standard_normal((n, 3)).astype(np.float32)
    nrm = rng.standard_normal((n, 3)).astype(np.float32)
    alb = rng.uniform(0, 1, (n, 3)).astype(np.float32)
    rough = rng.uniform(0.15, 1, (n, 1)).astype(np.float32)
    for kw, a, r in ((dict(f0=0.04), alb, rough), (dict(), None, None),
                     (dict(lambert_only=True), alb, None)):
        got = Microfacet(**kw)(pts2l, pts2c, nrm, a, r).cpu()
        t = lambda x: None if x is None else torch.as_tensor(x)
        want = obrdf.Microfacet(**kw)(t(pts2l), t(pts2c), t(nrm), t(a), t(r))
        assert got.shape == (n, L, 3)
        assert rel_l2(got, want) < 2e-5, kw
    with pytest.raises(ValueError):
        Microfacet()(pts2l[:, 0], pts2c, nrm)


def test_network_call_on_cuda_tensors_vs_oracle(ctx):
    """`mlp.Network.__call__` / `seq.Network.__call__` / `Embedder.__call__` (networks/mlp.py:39-50,
    seq.py:33-38, embedder.py:39-47) on CUDA tensors through the FP32 Dense kernels."""
    from nerfactor_b200.networks import mlp, seq
    from nerfactor_b200.networks.embedder import Embedder
    rng = np.random.default_rng(9)
    p = synth.init_mlp(rng, 27, [128] * 4, ['relu'] * 4, [2], 0.05)
    net = mlp.Network([128] * 4, act=['relu'] * 4, skip_at=[2]).build(27).load(p)
    head = mlp.Network([3], act=['sigmoid']).build(128)
    emb = Embedder(in_dims=3, log2_max_freq=3, n_freqs=4)
    x = torch.as_tensor(rng.uniform(-1, 1, (1000, 3)).astype(np.float32))
    y = head(net(emb(x.to(ctx.device)))).cpu()
    hp = {'layers': head.weights(), 'act': ['sigmoid'], 'skip_at': None}
    want = onets.mlp_forward(hp, onets.mlp_forward(p, onets.embed(x, 4)))
    assert y.shape == (1000, 3) and rel_l2(y, want) < 1e-5
    s = seq.Network()
    s.layers = head.layers
    assert torch.equal(s(net(emb(x.to(ctx.device)))).cpu(), y)
    with pytest.raises(TypeError):
        net(emb(x))                                   # CPU tensor: no CPU path


# ------------------------------------------------------------------ NeRF colour branch (8f.2)
def test_nerf_eval_fp32_layered_vs_oracle(ctx):
    """Model._eval_nerf_at (nerf.py:254-290) on the FP32 Dense kernels vs the oracle."""
    from nerfactor_b200 import _lib
    model = _nerf_model(ctx, 3)
    ro, rd = _rays(ctx, 6, 7)
    z = _lib.gen_z(ctx, 2., 6., 11, ro.shape[0])
    rgbs = model._eval_nerf_at(ro, rd, z, use_fine=True, precision='fp32')
    pts = (ro[:, None, :] + rd[:, None, :] * z[:, :, None]).reshape(-1, 3).cpu()
    views = rd[:, None, :].expand(-1, 11, 3).reshape(-1, 3).cpu()
    ref = stage_a.eval_nerf_at(synth.make_nerf_params(3), pts, views, True)
    assert rel_l2(rgbs.cpu().reshape(-1, 4)[:, :3], ref[:, :3]) < 2e-5
    assert rel_l2(rgbs.cpu().reshape(-1, 4)[:, 3], ref[:, 3]) < 2e-5


@pytest.mark.parametrize('prec', ['f16', 'bf16'])
def test_nerf_tcgen05_kernel(ctx, prec):
    """nf_nerf_fwd: sigma column bit-identical to the sigma-only kernel (same trunk, same head
    order), colours within operand precision of the FP32 path, results independent of the tile
    a sample lands in (ragged sizes, several tiles per CTA)."""
    from nerfactor_b200 import _lib
    model = _nerf_model(ctx, 3)
    ro, rd = _rays(ctx, 64, 64)
    S = 19
    z = _lib.gen_z(ctx, 2., 6., S, ro.shape[0])
    rgbs = model._eval_nerf_at(ro, rd, z, use_fine=True, precision=prec)
    assert rgbs.shape == (4096, S, 4) and not torch.isnan(rgbs).any()
    sig = _lib.sigma_fwd(ctx, model.packed_sigma(True), ro, rd, z, None, prec)
    assert torch.equal(torch.relu(rgbs[:, :, 3]), sig)
    k = 990                                              # 147 tiles: one per CTA
    sub = model._eval_nerf_at(ro[:k].contiguous(), rd[:k].contiguous(), z[:k].contiguous(),
                              use_fine=True, precision=prec)
    assert torch.equal(sub, rgbs[:k])
    kk = 300
    ref = model._eval_nerf_at(ro[:kk].contiguous(), rd[:kk].contiguous(), z[:kk].contiguous(),
                              use_fine=True, precision='fp32')
    tol = 3e-3 if prec == 'f16' else 3e-2
    assert rel_l2(rgbs[:kk, :, :3].cpu(), ref[:, :, :3].cpu()) < tol
    assert rel_l2(rgbs[:kk, :, 3].cpu(), ref[:, :, 3].cpu()) < tol


def test_nerf_render_rays_vs_oracle(ctx):
    """Model.call / _render_rays (nerf.py:100-118, 149-252): coarse 16 + fine 24 samples, white
    background, against the oracle chain; then the tensor-core path against the FP32 one."""
    model = _nerf_model(ctx, 3)
    model.config.set('DEFAULT', 'n_samples_coarse', '16')
    model.n_samples_fine = 24
    ro, rd = _rays(ctx, 8, 8)
    batch = ('view', (8, 8), ro * 1.0, rd * 3.0, torch.zeros_like(ro))   # un-normalised rayd
    pred, gt, lk, vis = model.call(batch, 'test', precision='fp32')
    oc, of = stage_a.nerf_render_rays(synth.make_nerf_params(3), ro.cpu(), (rd * 3.0).cpu(),
                                      2., 6., 16, 24, False, True)
    assert pred['coarse'].shape == (64, 3) and lk == {}
    assert np.abs(pred['coarse'].cpu().numpy() - oc['rgb'].numpy()).max() < 2e-4
    d = np.abs(pred['fine'].cpu().numpy() - of['rgb'].numpy())
    assert np.median(d) < 1e-4 and np.quantile(d, 0.95) < 5e-3      # gen_z_fine discontinuities
    assert np.abs(vis['coarse_occu'].cpu().numpy() - oc['occu'].numpy()).max() < 1e-4
    assert np.abs(vis['coarse_disp'].cpu().numpy() - oc['disp'].numpy()).max() < 1e-3
    p16, _, _, _ = model.call(batch, 'test', precision='f16')
    d16 = (p16['coarse'] - pred['coarse']).abs()
    assert float(d16.mean()) < 2e-3 and float(d16.max()) < 3e-2
