"""nf_integrate_bwd (backward of the rendering equation) without a GPU: the host-only workspace
query, and the CPU branch of autodiff.integrate, which must stay the torch composition it
replaces in the train step."""
import ctypes as C
import math

import numpy as np
import pytest
import torch

from nerfactor_b200 import _lib
from nerfactor_b200 import autodiff as ad


def _args(n, L, n_envmaps=1):
    a = _lib.IntegrateArgs()
    a.n, a.n_lights, a.n_envmaps, a.envmap_pixels = n, L, n_envmaps, L
    return a


def test_workspace_query_is_host_only_and_grows_with_n_up_to_its_cap():
    lib = _lib.load_library()
    ws = lambda n, L, e=1: lib.nf_integrate_bwd_workspace_bytes(C.byref(_args(n, L, e)))
    assert ws(0, 512) == 0
    sizes = [ws(n, 512) for n in (1, 8, 9, 100, 1024, 8192, 65536, 1 << 20)]
    assert sizes[0] > 0
    assert all(b >= a for a, b in zip(sizes, sizes[1:]))
    assert sizes[1] < sizes[2] < sizes[3] < sizes[4]
    # per-block partial sums of d_light ([blocks, 3, L] floats): capped, so the large sizes agree
    assert sizes[-1] == sizes[-2] == sizes[-3]
    assert sizes[-1] % (3 * 512 * 4) == 0
    assert ws(65536, 1000) > ws(65536, 512)
    assert lib.nf_integrate_bwd_workspace_bytes(None) == 0


def test_workspace_query_is_zero_for_unsupported_arguments():
    lib = _lib.load_library()
    for n_envmaps in (0, 2, 9):
        assert lib.nf_integrate_bwd_workspace_bytes(C.byref(_args(1024, 512, n_envmaps))) == 0
    assert lib.nf_integrate_bwd_workspace_bytes(C.byref(_args(1024, 5000))) == 0


def _inputs(kind, n=37, L=24, seed=0):
    rng = np.random.default_rng(seed)
    t = lambda a: torch.as_tensor(np.asarray(a, np.float32))
    xyz = t(rng.uniform(-1, 1, (n, 3)))
    cam = t(np.tile([[0., 0., 4.]], (n, 1)))
    normal = t(rng.standard_normal((n, 3)) * rng.uniform(0.5, 2., (n, 1)))
    albedo = t(rng.uniform(0.05, 0.9, (n, 3)))
    lvis = t(rng.uniform(0, 1, (n, L)))
    lxyz = t(rng.standard_normal((L, 3)) * 50.)
    lareas = t(rng.uniform(0.5, 1.5, L) * 4 * math.pi / L)
    light = t(rng.uniform(0, 3, (L, 3)))
    prop = t(rng.uniform(0.2, 0.8, (n, 1))) if kind == 0 else t(rng.uniform(0, 1, (n, L)))
    return lvis, normal, albedo, prop, light, xyz, cam, lxyz, lareas


@pytest.mark.parametrize('kind', [0, 1])
@pytest.mark.parametrize('srgb', [True, False])
def test_cpu_branch_is_the_torch_composition(kind, srgb):
    """On CPU tensors autodiff.integrate is microfacet_brdf (or albedo / pi + spec * scale) and
    render after the normalisation of the raw normal: same values and gradients, bit for bit."""
    ins = _inputs(kind)
    lvis, normal, albedo, prop, light, xyz, cam, lxyz, lareas = ins
    leaves = [x.clone().requires_grad_(True) for x in (lvis, normal, albedo, prop, light)]
    got = ad.integrate(*leaves, xyz, cam, lxyz, lareas, kind, 0.04, 0.7, srgb)
    d = torch.as_tensor(np.random.default_rng(1).standard_normal(got.shape).astype(np.float32))
    g_got = torch.autograd.grad(got, leaves, d)

    ref_leaves = [x.clone().requires_grad_(True) for x in (lvis, normal, albedo, prop, light)]
    lv, nr, al, pr, li = ref_leaves
    surf2l = ad.safe_l2_normalize(lxyz.reshape(1, -1, 3) - xyz[:, None, :], 2)
    surf2c = ad.safe_l2_normalize(cam - xyz, 1)
    nn = ad.safe_l2_normalize(nr, 1)
    if kind == 0:
        brdf = ad.microfacet_brdf(surf2l, surf2c, nn, al, pr, 0.04)
    else:
        n, L = pr.shape
        brdf = al[:, None, :] / math.pi + (pr.reshape(n, L, 1) * 0.7).expand(n, L, 3)
    want = ad.render(lv, brdf, surf2l, nn, li, lareas, srgb)
    g_want = torch.autograd.grad(want, ref_leaves, d)
    assert got.shape == (lvis.shape[0], 3)
    assert torch.equal(got, want)
    for a, b in zip(g_got, g_want):
        assert torch.equal(a, b)
