"""Differentiable train-mode forward of the NeRFactor models (SURVEY.md 8a a21-a23).

A train step works on `n_rays_per_step` = 1024 rays (nerfactor.ini:93), i.e. 0.5 M
(ray, light) rows -- three orders of magnitude less than a test-time view.  The Dense
contractions (>99.9 % of the step's FLOPs) run in this library's CUDA kernels through
`DenseFn` (nf_dense_fwd / nf_dense_bwd), the rendering equation through `IntegrateFn`
(nf_integrate_fwd / nf_integrate_bwd); the rest of the O(N L) element-wise math around
them is expressed in torch ops on the device so torch.autograd provides its adjoint,
with the reference's custom gradients (nerfactor/util/math.py:24-60) kept as explicit
autograd Functions.  Forward values equal the fused inference kernels' (same formulas).
"""
import math

import os

import torch
import torch.nn.functional as F

from . import _lib


# ------------------------------------------------------------------ Dense layers

# NF_MLP_CHAIN=0: layer-by-layer Dense calls (fp32 activations in HBM) also for tensor-core precisions
CHAIN = os.environ.get('NF_MLP_CHAIN', '1') != '0'


class DenseFn(torch.autograd.Function):
    """act([x1 | x2] @ w + b) through nf_dense_fwd / nf_dense_bwd.  `prec`: 'fp32' (CUDA
    cores) or 'bf16' / 'f16' (tcgen05, operands rounded to 16 bit, fp32 accumulation)."""

    @staticmethod
    def forward(ctx, x1, x2, w, b, act, prec='fp32'):
        c = _lib.default_context()
        x1 = x1.contiguous()
        x2c = None if x2 is None else x2.contiguous()
        w, b = w.contiguous(), b.contiguous()
        if w.data_ptr() % 16:            # cp.async needs 16-byte aligned weight rows
            w = w.clone()
        y = _lib.dense_fwd(c, x1, x2c, w, b, act, prec)
        ctx.save_for_backward(x1, x2c if x2c is not None else x1.new_empty(0), w, y)
        ctx.has_x2, ctx.act, ctx.prec = x2c is not None, act, prec
        return y

    @staticmethod
    def backward(ctx, dy):
        x1, x2, w, y = ctx.saved_tensors
        x2 = x2 if ctx.has_x2 else None
        c = _lib.default_context()
        n1, n2 = ctx.needs_input_grad[0], ctx.has_x2 and ctx.needs_input_grad[1]
        dx1, dx2, dw, db = _lib.dense_bwd(c, x1, x2, w, y, dy.contiguous(), ctx.act, n1, n2,
                                          ctx.prec)
        return dx1, dx2, dw, db, None, None


class MlpChainFn(torch.autograd.Function):
    """A whole mlp.Network (hidden layers + head) through nf_mlp_chain_fwd / nf_mlp_chain_bwd: one
    call each way, activations kept as 16-bit rows in a private workspace.  Arguments after `prec`:
    w0, b0, w1, b1, ... (already padded the way mlp_apply pads them)."""

    @staticmethod
    def forward(ctx, x, acts, skip_layer, prec, *wb):
        c = _lib.default_context()
        x = x.contiguous()
        ws = [t.contiguous() for t in wb[0::2]]
        bs = [t.contiguous() for t in wb[1::2]]
        ws = [w.clone() if w.data_ptr() % 16 else w for w in ws]
        y, work = _lib.mlp_chain_fwd(c, x, ws, bs, acts, skip_layer, prec)
        ctx.save_for_backward(y, *ws, *bs)
        ctx.work = work                 # the library's private workspace (not an autograd variable)
        ctx.acts, ctx.skip_layer, ctx.prec, ctx.in_dim, ctx.nl = acts, skip_layer, prec, x.shape[1], len(ws)
        return y

    @staticmethod
    def backward(ctx, dy):
        y, work = ctx.saved_tensors[0], ctx.work
        ws = list(ctx.saved_tensors[1:1 + ctx.nl])
        bs = list(ctx.saved_tensors[1 + ctx.nl:])
        c = _lib.default_context()
        dx, dws, dbs = _lib.mlp_chain_bwd(c, ws, bs, ctx.acts, ctx.skip_layer, ctx.in_dim, y,
                                          dy.contiguous(), work, ctx.needs_input_grad[0], ctx.prec)
        grads = []
        for dw, db in zip(dws, dbs):
            grads += [dw, db]
        return (dx, None, None, None) + tuple(grads)


def _pad_to4(n):
    return (n + 3) // 4 * 4


def mlp_apply(x, layers, acts, skip_at, prec='fp32', in_dim=None):
    """mlp.Network.__call__ (nerfactor/networks/mlp.py:39-50) + seq.Network for the head.
    layers: [(W[in,out], b[out]), ...] torch tensors (Keras layout).  Inputs / outputs
    whose width is not a multiple of 4 are zero-padded for the kernels (and sliced back);
    `in_dim`: true input width when `x` already arrives zero-padded to a multiple of 4."""
    if in_dim is None:
        in_dim = x.shape[1]
    in_pad = _pad_to4(in_dim)
    assert x.shape[1] in (in_dim, in_pad)
    xp = F.pad(x, (0, in_pad - in_dim)) if x.shape[1] != in_pad else x
    widths = [_pad_to4(w.shape[1]) for w, _ in layers]
    skips = sorted(skip_at) if skip_at is not None else []
    if (prec in ('bf16', 'f16') and CHAIN and len(skips) <= 1 and (not skips or skips[0] + 1 < len(layers))
            and _lib.mlp_chain_supported(in_pad, widths, [in_pad] + [
                widths[i] + (in_pad if skips and i == skips[0] else 0) for i in range(len(layers) - 1)])):
        # one call for the whole network; weights padded exactly as in the layer-by-layer path below
        wb = []
        for i, (w, b) in enumerate(layers):
            n, n_pad = w.shape[1], widths[i]
            if skips and i == skips[0] + 1:
                wh, wx = w[:w.shape[0] - in_dim], w[w.shape[0] - in_dim:]
                wfull = torch.cat((wh, F.pad(wx, (0, 0, 0, in_pad - in_dim))), 0)
            elif i == 0:
                wfull = F.pad(w, (0, 0, 0, in_pad - in_dim)) if in_pad != in_dim else w
            else:
                wfull = w
            if n_pad != n:
                wfull, b = F.pad(wfull, (0, n_pad - n)), F.pad(b, (0, n_pad - n))
            wb += [wfull, b]
        y = MlpChainFn.apply(xp, tuple(acts), skips[0] + 1 if skips else 0, prec, *wb)
        n_out = layers[-1][0].shape[1]
        return y[:, :n_out] if y.shape[1] != n_out else y
    h, h_skip = xp, None
    for i, ((w, b), act) in enumerate(zip(layers, acts)):
        n = w.shape[1]
        n_pad = _pad_to4(n)
        if h_skip is not None:                      # layer after the skip: [hidden | input]
            wh, wx = w[:w.shape[0] - in_dim], w[w.shape[0] - in_dim:]
            wx = F.pad(wx, (0, 0, 0, in_pad - in_dim))
            wfull = torch.cat((wh, wx), 0)
            x1, x2 = h, h_skip
        else:
            wfull = F.pad(w, (0, 0, 0, h.shape[1] - w.shape[0])) if h.shape[1] != w.shape[0] else w
            x1, x2 = h, None
        if n_pad != n:
            wfull = F.pad(wfull, (0, n_pad - n))
            bfull = F.pad(b, (0, n_pad - n))
        else:
            bfull = b
        y = DenseFn.apply(x1, x2, wfull, bfull, act, prec)
        h = y[:, :n] if n_pad != n else y
        h_skip = xp if (skip_at is not None and i in skip_at) else None
    return h


def embed(x, n_freqs):
    """nerfactor/networks/embedder.py:46-47."""
    out = [x]
    for k in range(n_freqs):
        out += [torch.sin(x * float(2 ** k)), torch.cos(x * float(2 ** k))]
    return torch.cat(out, -1)


# ------------------------------------------------------- TF semantics with custom grads

_CONSTS = {}


def _const(vals, device):
    """Small constant vectors, uploaded once per device (a host->device copy of a Python tuple
    cannot be captured into a CUDA graph)."""
    key = (tuple(vals), str(device))
    if key not in _CONSTS:
        _CONSTS[key] = torch.tensor(vals, dtype=torch.float32, device=device)
    return _CONSTS[key]


def safe_l2_normalize(x, axis, eps=1e-6):
    """nerfactor/util/math.py:63-64 (tf.linalg.l2_normalize)."""
    sq = torch.sum(x * x, dim=axis, keepdim=True)
    return x * torch.rsqrt(torch.clamp(sq, min=eps))


class SafeAcos(torch.autograd.Function):
    """nerfactor/util/math.py:42-60."""

    @staticmethod
    def forward(ctx, x):
        xc = torch.clamp(x, -1., 1.)
        ctx.save_for_backward(xc)
        return torch.acos(xc)

    @staticmethod
    def backward(ctx, dy):
        (xc,) = ctx.saved_tensors
        denom = torch.sqrt(1. - xc ** 2 + 1e-6) + 1e-6
        return dy * (-1. / denom)


class SafeAtan2(torch.autograd.Function):
    """nerfactor/util/math.py:24-39: z = atan2(x, y)."""

    @staticmethod
    def forward(ctx, x, y):
        ctx.save_for_backward(x, y)
        return torch.atan2(x, y)

    @staticmethod
    def backward(ctx, dz):
        x, y = ctx.saved_tensors
        denom = x ** 2 + y ** 2 + 1e-6
        return dz * (y / denom), dz * (-x / denom)


def divide_no_nan(a, b):
    a, b = torch.broadcast_tensors(a, b)
    safe = torch.where(b == 0, torch.ones_like(b), b)
    return torch.where(b == 0, torch.zeros_like(a), a / safe)


def gen_world2local(normal, eps=1e-6):
    """nerfactor/util/geom.py:119-149."""
    normal = safe_l2_normalize(normal, 1)
    z = (_const((0., 0., 1.), normal.device) + eps)[None, :].expand_as(normal)
    t = safe_l2_normalize(torch.linalg.cross(normal, z), 1)
    b = safe_l2_normalize(torch.linalg.cross(normal, t), 1)
    return torch.stack((t, b, normal), dim=1)


def dir2rusink(a, b):
    """nerfactor/util/geom.py:152-192."""
    a = safe_l2_normalize(a, 1)
    b = safe_l2_normalize(b, 1)
    h = safe_l2_normalize((a + b) / 2, 1)
    theta_h = SafeAcos.apply(h[:, 2])
    phi_h = SafeAtan2.apply(h[:, 1], h[:, 0])
    binormal = _const((0., 1., 0.), a.device)
    normal = _const((0., 0., 1.), a.device)

    def rot_vec(vector, axis, angle):
        cos_ang, sin_ang = torch.cos(angle).reshape(-1), torch.sin(angle).reshape(-1)
        axis = axis.reshape(1, 3)
        return vector * cos_ang[:, None] + \
            axis * (vector @ axis.t()) * (1 - cos_ang)[:, None] + \
            torch.linalg.cross(axis.expand_as(vector), vector) * sin_ang[:, None]

    diff = rot_vec(rot_vec(b, normal, -phi_h), binormal, -theta_h)
    theta_d = SafeAcos.apply(diff[:, 2])
    at = SafeAtan2.apply(diff[:, 1], diff[:, 0])
    phi_d = at - torch.floor(at / math.pi) * math.pi          # tf.math.floormod
    return torch.stack((phi_d, theta_h, theta_d), dim=1)


def microfacet_brdf(pts2l, pts2c, normal, albedo, rough, f0):
    """brdf/microfacet/microfacet.py:30-111."""
    pts2l = safe_l2_normalize(pts2l, 2)
    pts2c = safe_l2_normalize(pts2c, 1)
    normal = safe_l2_normalize(normal, 1)
    h = safe_l2_normalize(pts2l + pts2c[:, None, :], 2)
    f = f0 + (1 - f0) * (1 - torch.einsum('ijk,ijk->ij', pts2l, h)) ** 5
    alpha = rough ** 2
    cos_theta_m = torch.einsum('ijk,ik->ij', h, normal)
    chi = (cos_theta_m > 0).to(h.dtype)
    cm2 = cos_theta_m ** 2
    tm2 = divide_no_nan(1 - cm2, cm2)
    d = divide_no_nan(alpha ** 2 * chi, math.pi * cm2 ** 2 * (alpha ** 2 + tm2) ** 2)
    cos_theta_v = torch.einsum('ij,ij->i', normal, pts2c)
    div = divide_no_nan(torch.einsum('ijk,ik->ij', h, pts2c), cos_theta_v[:, None])
    chi_g = (div > 0).to(h.dtype)
    cv2 = torch.clamp(cos_theta_v ** 2, 0., 1.)
    tv2 = torch.clamp(divide_no_nan(1 - cv2, cv2), min=0.)
    g = divide_no_nan(chi_g * 2, 1 + torch.sqrt(1 + alpha ** 2 * tv2[:, None]))
    l_dot_n = torch.einsum('ijk,ik->ij', pts2l, normal)
    denom = 4 * torch.abs(l_dot_n) * torch.abs(cos_theta_v)[:, None]
    spec = divide_no_nan(f * g * d, denom)
    return spec[:, :, None] + (albedo / math.pi)[:, None, :]


def linear2srgb(x):
    """nerfactor/util/img.py:140-163."""
    x = torch.clamp(x, 0., 1.)
    # pow(0, 1/2.4) has an infinite derivative: TF evaluates it too and selects afterwards
    nonlin = 1.055 * torch.pow(torch.clamp(x, min=1e-30), 1 / 2.4) - 0.055
    return torch.where(x <= 0.0031308, x * 12.92, nonlin)


def render(lvis, brdf, surf2l, normal, light_flat, lareas, srgb):
    """nerfactor/models/nerfactor.py:315-342 for one env-map."""
    cos = torch.einsum('ijk,ik->ij', surf2l, normal)
    front_lit = (cos > 0).to(cos.dtype)
    lv = front_lit * lvis
    contrib = brdf * (lv[:, :, None] * light_flat[None, :, :]) * cos[:, :, None] * \
        lareas.reshape(1, -1, 1)
    rgb = torch.clamp(torch.sum(contrib, dim=1), 0., 1.)
    return linear2srgb(rgb) if srgb else rgb


class IntegrateFn(torch.autograd.Function):
    """The rendering equation through nf_integrate_fwd, its adjoint through nf_integrate_bwd (only
    the gradients autograd asks for; the backward recomputes the sum from the saved inputs)."""

    @staticmethod
    def forward(ctx, lvis, normal, albedo, brdf_prop, light_flat, xyz, cam, lxyz, lareas, kind,
                f0, spec_scale, srgb):
        c = _lib.default_context()
        ins = [t.contiguous() for t in (lvis, normal, albedo, brdf_prop, light_flat, xyz, cam,
                                        lxyz.reshape(-1, 3), lareas.reshape(-1))]
        lvis, normal, albedo, prop, light_flat, xyz, cam, lxyz, lareas = ins
        rough, spec = (prop, None) if kind == 0 else (None, prop)
        rgb = _lib.integrate_fwd(c, xyz, normal, cam, albedo, lvis, lxyz, lareas,
                                 light_flat.reshape(1, -1, 3), rough=rough, spec=spec, f0=f0,
                                 spec_scale=spec_scale, linear2srgb=srgb)
        ctx.save_for_backward(*ins)
        ctx.kind, ctx.f0, ctx.spec_scale, ctx.srgb = kind, f0, spec_scale, srgb
        return rgb.reshape(-1, 3)

    @staticmethod
    def backward(ctx, d_rgb):
        lvis, normal, albedo, prop, light_flat, xyz, cam, lxyz, lareas = ctx.saved_tensors
        names = ('lvis', 'normal', 'albedo', 'rough' if ctx.kind == 0 else 'spec', 'light')
        need = [k for k, want in zip(names, ctx.needs_input_grad[:5]) if want]
        rough, spec = (prop, None) if ctx.kind == 0 else (None, prop)
        g = _lib.integrate_bwd(_lib.default_context(), xyz, normal, cam, albedo, lvis, lxyz, lareas,
                               light_flat, d_rgb.contiguous(), rough=rough, spec=spec, f0=ctx.f0,
                               spec_scale=ctx.spec_scale, linear2srgb=ctx.srgb, need=need)
        return tuple(g.get(k) for k in names) + (None,) * 8


def integrate(lvis, normal, albedo, brdf_prop, light_flat, xyz, cam, lxyz, lareas, kind, f0,
              spec_scale, srgb):
    """Differentiable rendering equation for one env-map (nerfactor.py:212, 315-342 with the BRDF
    of microfacet.py:30-111 or nerfactor.py:457-461) -> rgb [n, 3].
    lvis [n, L]; normal [n, 3] raw (normalised here, nerfactor.py:212); albedo [n, 3];
    brdf_prop: rough [n, 1] (kind 0, microfacet) or the front-masked learned spec [n, L] (kind 1);
    light_flat [L, 3] (one texel per light, >= 0); xyz / cam [n, 3]; lxyz [L, 3]; lareas [L].
    CUDA tensors run nf_integrate_fwd / nf_integrate_bwd, which give no gradient for xyz, cam,
    lxyz or lareas; CPU tensors run the torch composition below."""
    if lvis.is_cuda:
        return IntegrateFn.apply(lvis, normal, albedo, brdf_prop, light_flat, xyz, cam, lxyz,
                                 lareas, kind, f0, spec_scale, srgb)
    surf2l = safe_l2_normalize(lxyz.reshape(1, -1, 3) - xyz[:, None, :], 2)   # shape.py:128-135
    surf2c = safe_l2_normalize(cam - xyz, 1)                                  # shape.py:137-144
    normal = safe_l2_normalize(normal, 1)
    if kind == 0:
        brdf = microfacet_brdf(surf2l, surf2c, normal, albedo, brdf_prop, f0)
    else:
        n, L = brdf_prop.shape
        brdf = albedo[:, None, :] / math.pi + (brdf_prop.reshape(n, L, 1) * spec_scale).expand(n, L, 3)
    return render(lvis, brdf, surf2l, normal, light_flat, lareas, srgb)
