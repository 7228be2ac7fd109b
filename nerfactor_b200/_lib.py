"""ctypes binding of libnerfactor_b200.so (the C ABI in include/nerfactor_b200.h).

PyTorch is only the owner of device memory and streams here: every wrapper
passes raw device pointers and the current CUDA stream to the library.  There is
no CPU or PyTorch fallback: a missing library or a missing sm_100 GPU raises.
"""
import ctypes as C
import os

import numpy as np
import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libnerfactor_b200.so')

NF_OK = 0
ERRORS = {-1: 'NF_ERR_INVALID_ARG', -2: 'NF_ERR_UNSUPPORTED', -3: 'NF_ERR_CUDA',
          -4: 'NF_ERR_NO_DEVICE'}
ACT = {None: 0, 'relu': 1, 'sigmoid': 2, 'softplus': 3}
KIND = {'point': 0, 'lvis': 1, 'brdf': 2, 'sigma': 3}
PREC = {'fp32': 0, 'f16': 1, 'bf16': 2, 'f16x3': 3, 'f16e': 4}

# every symbol include/nerfactor_b200.h declares (tests check the .so exports all)
EXPORTS = [
    'nf_version', 'nf_ctx_create', 'nf_ctx_destroy', 'nf_last_error_string',
    'nf_ctx_sm_count', 'nf_mlp_create', 'nf_mlp_destroy', 'nf_mlp_device_bytes',
    'nf_mlp_upload', 'nf_point_mlp_fwd', 'nf_lvis_fwd', 'nf_brdf_learned_fwd',
    'nf_integrate_fwd', 'nf_integrate_olat_fwd', 'nf_gen_rays', 'nf_gen_z',
    'nf_sigma_fwd', 'nf_sigma_normal_fwd', 'nf_mlp_attach_rgb', 'nf_nerf_fwd', 'nf_composite', 'nf_gen_z_fine',
    'nf_lvis_rays', 'nf_selftest_umma', 'nf_selftest_umma2', 'nf_dense_fwd',
    'nf_dense_fwd_workspace_bytes', 'nf_dense_bwd_workspace_bytes',
    'nf_dense_bwd', 'nf_mlp_chain_workspace_bytes', 'nf_mlp_chain_fwd', 'nf_mlp_chain_bwd',
    'nf_adam_amsgrad_step', 'nf_microfacet_brdf_fwd', 'nf_selftest_tmem',
    'nf_raymarch_depth_normal_workspace_bytes', 'nf_raymarch_depth_normal_fwd',
    'nf_raymarch_lvis_workspace_bytes', 'nf_raymarch_lvis_fwd',
    'nf_stageB_fused_workspace_bytes', 'nf_stageB_fused_fwd', 'nf_lvis_dirs_fwd', 'nf_lvis_inputs_fwd',
    'nf_integrate_bwd_workspace_bytes', 'nf_integrate_bwd']


class NfError(RuntimeError):
    pass


class MlpDesc(C.Structure):
    _fields_ = [('kind', C.c_int), ('in_dim', C.c_int), ('width', C.c_int),
                ('depth', C.c_int), ('skip_at', C.c_int), ('out_dim', C.c_int),
                ('out_act', C.c_int), ('n_freqs_a', C.c_int), ('n_freqs_b', C.c_int),
                ('z_dim', C.c_int), ('W', C.POINTER(C.c_void_p)),
                ('b', C.POINTER(C.c_void_p))]


class NerfRgbDesc(C.Structure):
    _fields_ = [('n_freqs_view', C.c_int), ('hidden', C.c_int),
                ('w_bottleneck', C.c_void_p), ('b_bottleneck', C.c_void_p),
                ('w_rgb0', C.c_void_p), ('b_rgb0', C.c_void_p),
                ('w_rgb1', C.c_void_p), ('b_rgb1', C.c_void_p)]


class IntegrateArgs(C.Structure):
    _fields_ = [('n', C.c_int), ('n_lights', C.c_int), ('n_envmaps', C.c_int),
                ('envmap_pixels', C.c_int), ('brdf_kind', C.c_int),
                ('linear2srgb', C.c_int), ('f0', C.c_float), ('spec_scale', C.c_float),
                ('xyz_d', C.c_void_p), ('normal_d', C.c_void_p), ('cam_d', C.c_void_p),
                ('albedo_d', C.c_void_p), ('rough_d', C.c_void_p), ('spec_d', C.c_void_p),
                ('lvis_d', C.c_void_p), ('lxyz_d', C.c_void_p), ('lareas_d', C.c_void_p),
                ('light_d', C.c_void_p), ('light_idx_d', C.c_void_p), ('rgb_d', C.c_void_p)]


class IntegrateGrads(C.Structure):
    _fields_ = [('d_rgb_d', C.c_void_p), ('d_lvis_d', C.c_void_p), ('d_normal_d', C.c_void_p),
                ('d_albedo_d', C.c_void_p), ('d_rough_d', C.c_void_p), ('d_spec_d', C.c_void_p),
                ('d_light_d', C.c_void_p)]


class StageBArgs(C.Structure):
    _fields_ = [('n', C.c_int), ('n_lights', C.c_int), ('n_envmaps', C.c_int),
                ('envmap_pixels', C.c_int), ('brdf_kind', C.c_int), ('linear2srgb', C.c_int),
                ('z_dim', C.c_int), ('f0', C.c_float), ('spec_scale', C.c_float),
                ('xyz_scale', C.c_float), ('xyz_d', C.c_void_p), ('normal_d', C.c_void_p),
                ('cam_d', C.c_void_p), ('albedo_d', C.c_void_p), ('rough_d', C.c_void_p),
                ('z_d', C.c_void_p), ('lxyz_d', C.c_void_p), ('lareas_d', C.c_void_p),
                ('light_d', C.c_void_p), ('light_idx_d', C.c_void_p), ('lvis_d', C.c_void_p),
                ('rgb_d', C.c_void_p), ('lvis_all_lights', C.c_int)]


CHAIN_MAX = 8


class MlpChain(C.Structure):
    _fields_ = [('depth', C.c_int), ('in_dim', C.c_int), ('skip_layer', C.c_int),
                ('width', C.c_int * CHAIN_MAX), ('act', C.c_int * CHAIN_MAX),
                ('w', C.c_void_p * CHAIN_MAX), ('b', C.c_void_p * CHAIN_MAX)]


_lib = None


def load_library():
    """Loads the shared library (no GPU needed to load / inspect symbols)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NfError(
            'libnerfactor_b200.so is not built: run `python -c "import '
            '__graft_entry__ as g; g.build()"` (nerfactor_b200/csrc/build.sh). '
            'There is no CPU fallback.')
    lib = C.CDLL(LIB_PATH)
    vp, i, f, d = C.c_void_p, C.c_int, C.c_float, C.c_double
    lib.nf_version.restype = i
    lib.nf_ctx_create.argtypes = [C.POINTER(vp), i]
    lib.nf_ctx_destroy.argtypes = [vp]
    lib.nf_last_error_string.argtypes = [vp]
    lib.nf_last_error_string.restype = C.c_char_p
    lib.nf_ctx_sm_count.argtypes = [vp]
    lib.nf_mlp_create.argtypes = [vp, C.POINTER(MlpDesc), C.POINTER(vp)]
    lib.nf_mlp_destroy.argtypes = [vp]
    lib.nf_mlp_device_bytes.argtypes = [vp]
    lib.nf_mlp_device_bytes.restype = C.c_size_t
    lib.nf_mlp_upload.argtypes = [vp, vp, vp, vp]
    lib.nf_mlp_chain_workspace_bytes.argtypes = [C.POINTER(MlpChain), C.c_longlong]
    lib.nf_mlp_chain_workspace_bytes.restype = C.c_size_t
    lib.nf_mlp_chain_fwd.argtypes = [vp, C.POINTER(MlpChain), vp, C.c_longlong, vp, vp, i, vp]
    lib.nf_mlp_chain_bwd.argtypes = [vp, C.POINTER(MlpChain), C.c_longlong, vp, vp, vp,
                                     C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), vp, i, vp]
    lib.nf_point_mlp_fwd.argtypes = [vp, vp, vp, i, f, vp, i, vp]
    lib.nf_lvis_fwd.argtypes = [vp, vp, vp, i, f, vp, i, vp, i, vp]
    lib.nf_lvis_inputs_fwd.argtypes = [vp, vp, vp, i, vp, i, f, i, i, i, vp, vp]
    lib.nf_lvis_dirs_fwd.argtypes = [vp, vp, vp, vp, i, f, vp, i, vp, i, vp]
    lib.nf_brdf_learned_fwd.argtypes = [vp, vp, vp, vp, vp, vp, i, vp, i, vp, i, vp]
    lib.nf_integrate_fwd.argtypes = [vp, C.POINTER(IntegrateArgs), vp]
    lib.nf_integrate_olat_fwd.argtypes = [vp, C.POINTER(IntegrateArgs), f, f, vp, vp]
    lib.nf_integrate_bwd_workspace_bytes.argtypes = [C.POINTER(IntegrateArgs)]
    lib.nf_integrate_bwd_workspace_bytes.restype = C.c_size_t
    lib.nf_integrate_bwd.argtypes = [vp, C.POINTER(IntegrateArgs), C.POINTER(IntegrateGrads), vp,
                                     C.c_size_t, vp]
    lib.nf_microfacet_brdf_fwd.argtypes = [vp, vp, vp, vp, vp, vp, i, i, f, i, f, vp, vp]
    lib.nf_gen_rays.argtypes = [vp, C.POINTER(d), d, i, i, i, vp, vp, vp]
    lib.nf_gen_z.argtypes = [vp, f, f, i, i, i, vp, vp, vp]
    lib.nf_sigma_fwd.argtypes = [vp, vp, vp, vp, vp, i, i, C.POINTER(f), vp, i, vp]
    lib.nf_mlp_attach_rgb.argtypes = [vp, vp, C.POINTER(NerfRgbDesc)]
    lib.nf_nerf_fwd.argtypes = [vp, vp, vp, vp, vp, i, i, vp, i, vp]
    lib.nf_sigma_normal_fwd.argtypes = [vp, vp, vp, vp, vp, i, i, C.POINTER(f), vp, vp, i, vp]
    lib.nf_composite.argtypes = [vp, vp, vp, vp, vp, vp, i, i, vp, vp, vp, vp, vp, vp]
    lib.nf_gen_z_fine.argtypes = [vp, vp, vp, i, i, i, vp, vp]
    lib.nf_lvis_rays.argtypes = [vp, vp, vp, i, vp, i, vp, vp, vp, vp]
    lib.nf_selftest_umma.argtypes = [vp, vp, vp, i, i, vp, vp]
    lib.nf_selftest_umma2.argtypes = [vp, vp, vp, i, vp, vp]
    lib.nf_selftest_tmem.argtypes = [vp, i, i, i, i, vp, vp]
    lib.nf_raymarch_depth_normal_workspace_bytes.argtypes = [i, i, i]
    lib.nf_raymarch_depth_normal_workspace_bytes.restype = C.c_size_t
    lib.nf_raymarch_depth_normal_fwd.argtypes = [vp, vp, vp, vp, vp, i, f, f, i, i, i, C.POINTER(f),
                                                 i, vp, C.c_size_t, vp, vp, vp, vp]
    lib.nf_stageB_fused_workspace_bytes.argtypes = [C.POINTER(StageBArgs), i]
    lib.nf_stageB_fused_workspace_bytes.restype = C.c_size_t
    lib.nf_stageB_fused_fwd.argtypes = [vp, vp, vp, C.POINTER(StageBArgs), i, vp, C.c_size_t, vp]
    lib.nf_raymarch_lvis_workspace_bytes.argtypes = [i, i, i, i]
    lib.nf_raymarch_lvis_workspace_bytes.restype = C.c_size_t
    lib.nf_raymarch_lvis_fwd.argtypes = [vp, vp, vp, vp, vp, i, vp, i, f, f, i, i, i, C.POINTER(f),
                                         i, vp, C.c_size_t, vp, vp]
    ll = C.c_longlong
    lib.nf_dense_fwd.argtypes = [vp, vp, i, vp, i, vp, vp, ll, i, i, vp, vp, i, vp]
    lib.nf_dense_fwd_workspace_bytes.argtypes = [i, i, i, i]
    lib.nf_dense_fwd_workspace_bytes.restype = C.c_size_t
    lib.nf_dense_bwd_workspace_bytes.argtypes = [ll, i, i, i, i]
    lib.nf_dense_bwd_workspace_bytes.restype = C.c_size_t
    lib.nf_dense_bwd.argtypes = [vp, vp, i, vp, i, vp, vp, vp, ll, i, i, vp, vp, vp, vp, vp, i, vp]
    lib.nf_adam_amsgrad_step.argtypes = [vp, vp, vp, vp, vp, vp, ll, f, f, f, f, ll, vp]
    for name in EXPORTS:
        if name not in ('nf_last_error_string', 'nf_mlp_device_bytes',
                        'nf_dense_bwd_workspace_bytes', 'nf_dense_fwd_workspace_bytes',
                        'nf_raymarch_depth_normal_workspace_bytes',
                        'nf_raymarch_lvis_workspace_bytes', 'nf_stageB_fused_workspace_bytes',
                        'nf_integrate_bwd_workspace_bytes'):
            getattr(lib, name).restype = i
    _lib = lib
    return lib


def _ptr(t):
    if t is None:
        return None
    assert t.is_cuda and t.is_contiguous(), 'need a contiguous CUDA tensor'
    return C.c_void_p(t.data_ptr())


def _f32(t):
    assert t.dtype == torch.float32, 'fp32 tensor expected'
    return _ptr(t)


def _stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class Context:
    """nf_ctx wrapper; one per process / GPU."""

    def __init__(self, device=None):
        self.lib = load_library()
        if not torch.cuda.is_available():
            raise NfError('no CUDA device: nerfactor_b200 has no CPU fallback')
        if device is None:
            device = torch.cuda.current_device()
        self.device = torch.device('cuda', device)
        h = C.c_void_p()
        rc = self.lib.nf_ctx_create(C.byref(h), int(device))
        if rc != NF_OK:
            raise NfError('nf_ctx_create failed: %s (an sm_100 GPU is required)'
                          % ERRORS.get(rc, rc))
        self.h = h
        self.launches = 0      # kernels of this library enqueued so far

    def check(self, rc):
        if rc != NF_OK:
            msg = self.lib.nf_last_error_string(self.h).decode()
            raise NfError('%s: %s' % (ERRORS.get(rc, rc), msg))

    def launch(self, rc):
        """check() for calls that enqueue one of this library's kernels."""
        self.launches += 1
        self.check(rc)

    @property
    def sm_count(self):
        return self.lib.nf_ctx_sm_count(self.h)

    def __del__(self):
        try:
            if getattr(self, 'h', None):
                self.lib.nf_ctx_destroy(self.h)
                self.h = None
        except Exception:
            pass


_default_ctx = None


def default_context():
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context()
    return _default_ctx


class PackedMlp:
    """nf_mlp wrapper: packs a trunk + head on the host and uploads it into a
    torch-owned device buffer."""

    def __init__(self, ctx, kind, layers, skip_at, out_act, n_freqs_a=0, n_freqs_b=0,
                 z_dim=0, rgb=None):
        """layers: [(W[in,out], b[out]) ...] fp32 NumPy, trunk layers then head.
        rgb (sigma nets): {'bottleneck': (W, b), 'rgb_out': [(W0, b0), (W1, b1)],
        'n_freqs_view': F} -- the NeRF colour branch (nf_mlp_attach_rgb)."""
        self.ctx = ctx
        depth = len(layers) - 1
        Ws = [np.ascontiguousarray(w, dtype=np.float32) for w, _ in layers]
        bs = [np.ascontiguousarray(b, dtype=np.float32) for _, b in layers]
        self._keep = (Ws, bs)
        d = MlpDesc()
        d.kind, d.in_dim, d.width = KIND[kind], Ws[0].shape[0], Ws[0].shape[1]
        d.depth, d.skip_at = depth, skip_at
        d.out_dim, d.out_act = Ws[-1].shape[1], ACT[out_act]
        d.n_freqs_a, d.n_freqs_b, d.z_dim = n_freqs_a, n_freqs_b, z_dim
        Wp = (C.c_void_p * (depth + 1))(*[w.ctypes.data for w in Ws])
        bp = (C.c_void_p * (depth + 1))(*[b.ctypes.data for b in bs])
        d.W, d.b = Wp, bp
        self.kind, self.out_dim, self.depth, self.width = kind, d.out_dim, depth, d.width
        h = C.c_void_p()
        ctx.check(ctx.lib.nf_mlp_create(ctx.h, C.byref(d), C.byref(h)))
        self.h = h
        self.has_rgb = rgb is not None
        if rgb is not None:
            c32 = lambda a: np.ascontiguousarray(a, dtype=np.float32)
            arrs = [c32(rgb['bottleneck'][0]), c32(rgb['bottleneck'][1]),
                    c32(rgb['rgb_out'][0][0]), c32(rgb['rgb_out'][0][1]),
                    c32(rgb['rgb_out'][1][0]), c32(rgb['rgb_out'][1][1])]
            self._keep_rgb = arrs
            rd = NerfRgbDesc(int(rgb['n_freqs_view']), int(arrs[2].shape[1]),
                             *[a.ctypes.data for a in arrs])
            assert arrs[0].shape == (256, 256) and arrs[4].shape == (arrs[2].shape[1], 3)
            assert arrs[2].shape[0] == 256 + 3 * (1 + 2 * int(rgb['n_freqs_view']))
            ctx.check(ctx.lib.nf_mlp_attach_rgb(ctx.h, h, C.byref(rd)))
        nbytes = ctx.lib.nf_mlp_device_bytes(h)
        self.buf = torch.empty(nbytes + 256, dtype=torch.uint8, device=ctx.device)
        off = (-self.buf.data_ptr()) % 256
        self.dev_ptr = self.buf.data_ptr() + off
        ctx.check(ctx.lib.nf_mlp_upload(ctx.h, h, C.c_void_p(self.dev_ptr), _stream()))

    def __del__(self):
        try:
            if getattr(self, 'h', None):
                self.ctx.lib.nf_mlp_destroy(self.h)
                self.h = None
        except Exception:
            pass


# ------------------------------------------------------------------ forward ops

def point_mlp_fwd(ctx, mlp, xyz, xyz_scale=1.0, precision='fp32'):
    n = xyz.shape[0]
    out = torch.empty((n, mlp.out_dim), dtype=torch.float32, device=xyz.device)
    ctx.launch(ctx.lib.nf_point_mlp_fwd(ctx.h, mlp.h, _f32(xyz), n, float(xyz_scale),
                                       _f32(out), PREC[precision], _stream()))
    return out


def lvis_fwd(ctx, mlp, xyz, lxyz, xyz_scale=1.0, precision='f16'):
    lxyz = lxyz.reshape(-1, 3)
    n, L = xyz.shape[0], lxyz.shape[0]
    out = torch.empty((n, L), dtype=torch.float32, device=xyz.device)
    ctx.launch(ctx.lib.nf_lvis_fwd(ctx.h, mlp.h, _f32(xyz), n, float(xyz_scale), _f32(lxyz),
                                  L, _f32(out), PREC[precision], _stream()))
    return out


def lvis_inputs_fwd(ctx, xyz, xyz_dir, lxyz, xyz_scale, n_freqs_xyz, n_freqs_ldir):
    """[embed(xyz_scale xyz) | embed(l2n(lxyz - xyz_dir))] rows, zero-padded to a multiple of 4
    columns -> (rows [n * L, ld], true width)."""
    lxyz = lxyz.reshape(-1, 3)
    n, L = xyz.shape[0], lxyz.shape[0]
    width = 3 * (1 + 2 * n_freqs_xyz) + 3 * (1 + 2 * n_freqs_ldir)
    ld = (width + 3) // 4 * 4
    out = torch.empty((n * L, ld), dtype=torch.float32, device=xyz.device)
    ctx.launch(ctx.lib.nf_lvis_inputs_fwd(ctx.h, _f32(xyz), _f32(xyz_dir), n, _f32(lxyz), L,
                                         float(xyz_scale), int(n_freqs_xyz), int(n_freqs_ldir),
                                         ld, _f32(out), _stream()))
    return out, width


def lvis_dirs_fwd(ctx, mlp, xyz, xyz_dir, lxyz, xyz_scale=1.0, precision='f16'):
    """Visibility network at `xyz` with the light directions of `xyz_dir` (shape.py:170)."""
    lxyz = lxyz.reshape(-1, 3)
    n, L = xyz.shape[0], lxyz.shape[0]
    out = torch.empty((n, L), dtype=torch.float32, device=xyz.device)
    ctx.launch(ctx.lib.nf_lvis_dirs_fwd(ctx.h, mlp.h, _f32(xyz), _f32(xyz_dir), n, float(xyz_scale),
                                       _f32(lxyz), L, _f32(out), PREC[precision], _stream()))
    return out


def brdf_learned_fwd(ctx, mlp, xyz, normal, cam, z, lxyz, precision='f16'):
    lxyz = lxyz.reshape(-1, 3)
    n, L = xyz.shape[0], lxyz.shape[0]
    out = torch.empty((n, L), dtype=torch.float32, device=xyz.device)
    ctx.launch(ctx.lib.nf_brdf_learned_fwd(
        ctx.h, mlp.h, _f32(xyz), _f32(normal), _f32(cam), _f32(z), n, _f32(lxyz), L,
        _f32(out), PREC[precision], _stream()))
    return out


def _integrate_args(xyz, normal, cam, albedo, lvis, lxyz, lareas, rough=None, spec=None,
                    light=None, light_idx=None, rgb=None, f0=0.04, spec_scale=1.0,
                    linear2srgb=True):
    a = IntegrateArgs()
    lxyz, lareas = lxyz.reshape(-1, 3), lareas.reshape(-1)
    a.n, a.n_lights = xyz.shape[0], lxyz.shape[0]
    a.brdf_kind = 0 if spec is None else 1
    a.linear2srgb, a.f0, a.spec_scale = int(linear2srgb), float(f0), float(spec_scale)
    a.xyz_d, a.normal_d, a.cam_d = _f32(xyz), _f32(normal), _f32(cam)
    a.albedo_d, a.lvis_d = _f32(albedo), _f32(lvis)
    a.rough_d = _f32(rough) if rough is not None else None
    a.spec_d = _f32(spec) if spec is not None else None
    a.lxyz_d, a.lareas_d = _f32(lxyz), _f32(lareas)
    if light is not None:
        a.n_envmaps, a.envmap_pixels = light.shape[0], light.shape[1]
        a.light_d = _f32(light)
    a.light_idx_d = _ptr(light_idx) if light_idx is not None else None
    a.rgb_d = _f32(rgb) if rgb is not None else None
    return a


def integrate_fwd(ctx, xyz, normal, cam, albedo, lvis, lxyz, lareas, light, rough=None,
                  spec=None, light_idx=None, f0=0.04, spec_scale=1.0, linear2srgb=True):
    """light: [E, P, 3] (clipped >= 0). Returns rgb [n, E, 3]."""
    n, E = xyz.shape[0], light.shape[0]
    rgb = torch.empty((n, E, 3), dtype=torch.float32, device=xyz.device)
    if light_idx is not None:
        assert light_idx.dtype == torch.int32
    a = _integrate_args(xyz, normal, cam, albedo, lvis, lxyz, lareas, rough, spec, light,
                        light_idx, rgb, f0, spec_scale, linear2srgb)
    ctx.launch(ctx.lib.nf_integrate_fwd(ctx.h, C.byref(a), _stream()))
    return rgb


def integrate_bwd(ctx, xyz, normal, cam, albedo, lvis, lxyz, lareas, light, d_rgb, rough=None,
                  spec=None, f0=0.04, spec_scale=1.0, linear2srgb=True, need=()):
    """Gradients of integrate_fwd with one env-map, light [L, 3] (one texel per light, >= 0), given
    d_rgb [n, 3].  `need`: names out of 'lvis', 'normal', 'albedo', 'rough' (with rough), 'spec'
    (with spec), 'light'; only those are computed.  -> {name: gradient} (normal: with respect to
    the raw normal, spec: before spec_scale, light: summed over the points, rough: shape of rough)."""
    n, L = xyz.shape[0], lxyz.reshape(-1, 3).shape[0]
    light = light.reshape(1, L, 3)
    a = _integrate_args(xyz, normal, cam, albedo, lvis, lxyz, lareas,
                        None if rough is None else rough.reshape(-1), spec, light, None, None, f0,
                        spec_scale, linear2srgb)
    shapes = {'lvis': (n, L), 'normal': (n, 3), 'albedo': (n, 3), 'light': (L, 3),
              'rough': (n,), 'spec': (n, L)}
    out = {k: torch.empty(shapes[k], dtype=torch.float32, device=xyz.device) for k in need}
    g = IntegrateGrads()
    g.d_rgb_d = _f32(d_rgb)
    for k, t in out.items():
        setattr(g, 'd_%s_d' % k, _f32(t))
    nbytes = ctx.lib.nf_integrate_bwd_workspace_bytes(C.byref(a)) if 'light' in out else 0
    work = torch.empty((nbytes,), dtype=torch.uint8, device=xyz.device) if nbytes else None
    if 'light' in out:
        ctx.launches += 1                    # the ordered sum of the per-block d_light partials
    ctx.launch(ctx.lib.nf_integrate_bwd(ctx.h, C.byref(a), C.byref(g), _ptr(work), nbytes,
                                        _stream()))
    if 'rough' in out:
        out['rough'] = out['rough'].reshape(rough.shape)
    return out


def integrate_olat_fwd(ctx, xyz, normal, cam, albedo, lvis, lxyz, lareas, olat_inten,
                       ambient, rough=None, spec=None, f0=0.04, spec_scale=1.0,
                       linear2srgb=True):
    n, L = xyz.shape[0], lxyz.reshape(-1, 3).shape[0]
    out = torch.empty((n, L, 3), dtype=torch.float32, device=xyz.device)
    a = _integrate_args(xyz, normal, cam, albedo, lvis, lxyz, lareas, rough, spec, None,
                        None, None, f0, spec_scale, linear2srgb)
    ctx.launch(ctx.lib.nf_integrate_olat_fwd(ctx.h, C.byref(a), float(olat_inten),
                                            float(ambient), _f32(out), _stream()))
    return out


def stageB_fused_fwd(ctx, mlp_lvis, xyz, normal, cam, albedo, lxyz, lareas, light, rough=None,
                     z=None, mlp_brdf=None, light_idx=None, f0=0.04, spec_scale=1.0, xyz_scale=1.0,
                     linear2srgb=True, precision='f16', want_lvis=False, all_lights=False):
    """Light-visibility net -> BRDF -> rendering equation in one C call (nf_stageB_fused_fwd).
    light [E, P, 3] -> rgb [n, E, 3] (and lvis [n, L] when want_lvis).  Without `want_lvis` the
    visibility network only runs on the front-lit lights of each point (the renderer multiplies
    the others by zero, nerfactor.py:329-330) unless `all_lights`."""
    lxyz, lareas = lxyz.reshape(-1, 3), lareas.reshape(-1)
    n, L, E = xyz.shape[0], lxyz.shape[0], light.shape[0]
    dev = xyz.device
    rgb = torch.empty((n, E, 3), dtype=torch.float32, device=dev)
    lvis = torch.empty((n, L), dtype=torch.float32, device=dev) if want_lvis else None
    a = StageBArgs()
    a.n, a.n_lights, a.n_envmaps, a.envmap_pixels = n, L, E, light.shape[1]
    a.brdf_kind = 0 if z is None else 1
    a.linear2srgb, a.f0, a.spec_scale, a.xyz_scale = int(linear2srgb), float(f0), float(spec_scale), float(xyz_scale)
    a.xyz_d, a.normal_d, a.cam_d, a.albedo_d = _f32(xyz), _f32(normal), _f32(cam), _f32(albedo)
    if z is None:
        rough = rough.reshape(-1)
        a.rough_d = _f32(rough)
    else:
        a.z_d, a.z_dim = _f32(z), z.shape[1]
    a.lxyz_d, a.lareas_d, a.light_d = _f32(lxyz), _f32(lareas), _f32(light)
    if light_idx is not None:
        assert light_idx.dtype == torch.int32
        a.light_idx_d = _ptr(light_idx)
    a.lvis_d = _f32(lvis) if lvis is not None else None
    a.rgb_d = _f32(rgb)
    a.lvis_all_lights = 2 if all_lights == 'front_lit' else int(bool(all_lights))
    nbytes = ctx.lib.nf_stageB_fused_workspace_bytes(C.byref(a), PREC[precision])
    work = torch.empty((nbytes + 256,), dtype=torch.uint8, device=dev) if nbytes else None
    wptr = C.c_void_p(work.data_ptr() + (-work.data_ptr()) % 256) if nbytes else None
    if nbytes:          # chunked path: 2-3 kernels per chunk of <= 48 MB rows
        cpts = max(256, ((48 << 20) // (L * 4)) // 256 * 256)
        ctx.launches += (2 + (z is not None)) * max(1, (n + cpts - 1) // cpts) - 1
    ctx.launch(ctx.lib.nf_stageB_fused_fwd(
        ctx.h, mlp_lvis.h, mlp_brdf.h if mlp_brdf is not None else None, C.byref(a),
        PREC[precision], wptr, nbytes, _stream()))
    return rgb, lvis


def microfacet_brdf_fwd(ctx, pts2l, pts2c, normal, albedo=None, rough=None, default_rough=0.3,
                        lambert_only=False, f0=0.91):
    """Microfacet.__call__ (brdf/microfacet/microfacet.py:30-72) -> brdf [n, L, 3]."""
    n, L = pts2l.shape[0], pts2l.shape[1]
    out = torch.empty((n, L, 3), dtype=torch.float32, device=pts2l.device)
    ctx.launch(ctx.lib.nf_microfacet_brdf_fwd(
        ctx.h, _f32(pts2l), _f32(pts2c), _f32(normal),
        _f32(albedo) if albedo is not None else None, _f32(rough) if rough is not None else None,
        n, L, float(default_rough), int(bool(lambert_only)), float(f0), _f32(out), _stream()))
    return out


def gen_rays(ctx, c2w, cam_angle_x, h, w, normalize=False):
    c2w = np.ascontiguousarray(np.asarray(c2w, dtype=np.float64).reshape(16))
    rayo = torch.empty((h * w, 3), dtype=torch.float32, device=ctx.device)
    rayd = torch.empty((h * w, 3), dtype=torch.float32, device=ctx.device)
    ctx.launch(ctx.lib.nf_gen_rays(
        ctx.h, c2w.ctypes.data_as(C.POINTER(C.c_double)), float(cam_angle_x), h, w,
        int(normalize), _f32(rayo), _f32(rayd), _stream()))
    return rayo, rayd


def gen_z(ctx, near, far, n_samples, n_rays, lin_in_disp=False, perturb_u=None):
    z = torch.empty((n_rays, n_samples), dtype=torch.float32, device=ctx.device)
    ctx.launch(ctx.lib.nf_gen_z(ctx.h, float(near), float(far), n_samples, n_rays,
                               int(lin_in_disp),
                               _f32(perturb_u) if perturb_u is not None else None,
                               _f32(z), _stream()))
    return z


def _bbox(bbox):
    if bbox is None:
        return None
    arr = (C.c_float * 6)(*[float(v) for v in bbox])
    return arr


def sigma_fwd(ctx, mlp, rayo, rayd, z, bbox=None, precision='f16'):
    n, S = z.shape
    sigma = torch.empty((n, S), dtype=torch.float32, device=z.device)
    bb = _bbox(bbox)
    ctx.launch(ctx.lib.nf_sigma_fwd(ctx.h, mlp.h, _f32(rayo), _f32(rayd), _f32(z), n, S,
                                   bb, _f32(sigma), PREC[precision], _stream()))
    return sigma


def nerf_fwd(ctx, mlp, rayo, rayd, z, precision='f16'):
    """-> rgbs [n, S, 4] = (raw r, g, b, raw sigma), nerf.py:254-290 (use_views)."""
    n, S = z.shape
    out = torch.empty((n, S, 4), dtype=torch.float32, device=z.device)
    ctx.launch(ctx.lib.nf_nerf_fwd(ctx.h, mlp.h, _f32(rayo), _f32(rayd), _f32(z), n, S,
                                  _f32(out), PREC[precision], _stream()))
    return out


def sigma_normal_fwd(ctx, mlp, rayo, rayd, z, bbox=None, precision='fp32'):
    n, S = z.shape
    sigma = torch.empty((n, S), dtype=torch.float32, device=z.device)
    normal = torch.empty((n, S, 3), dtype=torch.float32, device=z.device)
    bb = _bbox(bbox)
    ctx.launch(ctx.lib.nf_sigma_normal_fwd(ctx.h, mlp.h, _f32(rayo), _f32(rayd), _f32(z), n,
                                          S, bb, _f32(sigma), _f32(normal), PREC[precision],
                                          _stream()))
    return sigma, normal


def composite(ctx, sigma, z, rayo, rayd, normal=None, want_weights=True, want_surf=True):
    n, S = sigma.shape
    dev = sigma.device
    weights = torch.empty((n, S), dtype=torch.float32, device=dev) if want_weights else None
    occu = torch.empty((n,), dtype=torch.float32, device=dev)
    depth = torch.empty((n,), dtype=torch.float32, device=dev)
    surf = torch.empty((n, 3), dtype=torch.float32, device=dev) if want_surf else None
    en = torch.empty((n, 3), dtype=torch.float32, device=dev) if normal is not None else None
    ctx.launch(ctx.lib.nf_composite(
        ctx.h, _f32(sigma), _f32(z), _f32(rayo), _f32(rayd),
        _f32(normal) if normal is not None else None, n, S,
        _f32(weights) if weights is not None else None, _f32(occu), _f32(depth),
        _f32(surf) if surf is not None else None, _f32(en) if en is not None else None,
        _stream()))
    return weights, occu, depth, surf, en


def gen_z_fine(ctx, z_coarse, weights, n_fine):
    n, Sc = z_coarse.shape
    z_all = torch.empty((n, Sc + n_fine), dtype=torch.float32, device=z_coarse.device)
    ctx.launch(ctx.lib.nf_gen_z_fine(ctx.h, _f32(z_coarse), _f32(weights), n, Sc, n_fine,
                                    _f32(z_all), _stream()))
    return z_all


def lvis_rays(ctx, surf, normal, lxyz):
    n, L = surf.shape[0], lxyz.shape[0]
    dev = surf.device
    rayo = torch.empty((n * L, 3), dtype=torch.float32, device=dev)
    rayd = torch.empty((n * L, 3), dtype=torch.float32, device=dev)
    fl = torch.empty((n * L,), dtype=torch.uint8, device=dev)
    ctx.launch(ctx.lib.nf_lvis_rays(ctx.h, _f32(surf), _f32(normal), n, _f32(lxyz), L,
                                   _f32(rayo), _f32(rayd), _ptr(fl), _stream()))
    return rayo, rayd, fl.view(n, L)


def raymarch_depth_normal_fwd(ctx, mlp_coarse, mlp_fine, rayo, rayd, near, far, n_coarse, n_fine,
                              lin_in_disp=False, bbox=None, precision='f16e'):
    """compute_depth_and_normal (gfn.py:249-319) in one C call -> (occu [n], depth [n],
    normal [n, 3]); n_coarse / n_fine are the actual sample counts."""
    n = rayo.shape[0]
    dev = rayo.device
    occu = torch.empty((n,), dtype=torch.float32, device=dev)
    depth = torch.empty((n,), dtype=torch.float32, device=dev)
    normal = torch.empty((n, 3), dtype=torch.float32, device=dev)
    nbytes = ctx.lib.nf_raymarch_depth_normal_workspace_bytes(n, n_coarse, n_fine)
    work = torch.empty((nbytes + 256,), dtype=torch.uint8, device=dev)
    wptr = work.data_ptr() + (-work.data_ptr()) % 256
    n_chunks = max(1, (n + 32767) // 32768)
    ctx.launches += 6 * n_chunks - 1
    ctx.launch(ctx.lib.nf_raymarch_depth_normal_fwd(
        ctx.h, mlp_coarse.h, mlp_fine.h, _f32(rayo), _f32(rayd), n, float(near), float(far),
        int(n_coarse), int(n_fine), int(lin_in_disp), _bbox(bbox), PREC[precision],
        C.c_void_p(wptr), nbytes, _f32(occu), _f32(depth), _f32(normal), _stream()))
    return occu, depth, normal


def raymarch_lvis_fwd(ctx, mlp_coarse, mlp_fine, surf, normal, lxyz, lvis_near, lvis_far,
                      n_coarse, n_fine, lin_in_disp=False, bbox=None, precision='f16e'):
    """compute_light_visibility (gfn.py:177-246) in one C call -> lvis_hit [m, L]."""
    m, L = surf.shape[0], lxyz.shape[0]
    dev = surf.device
    lvis = torch.empty((m, L), dtype=torch.float32, device=dev)
    if m == 0:
        return lvis
    nbytes = ctx.lib.nf_raymarch_lvis_workspace_bytes(m, L, n_coarse, n_fine)
    work = torch.empty((nbytes + 256,), dtype=torch.uint8, device=dev)
    wptr = work.data_ptr() + (-work.data_ptr()) % 256
    ctx.launches += 8 * max(1, (m * L + (1 << 19) - 1) >> 19) - 1
    ctx.launch(ctx.lib.nf_raymarch_lvis_fwd(
        ctx.h, mlp_coarse.h, mlp_fine.h, _f32(surf), _f32(normal), m, _f32(lxyz), L,
        float(lvis_near), float(lvis_far), int(n_coarse), int(n_fine), int(lin_in_disp),
        _bbox(bbox), PREC[precision], C.c_void_p(wptr), nbytes, _f32(lvis), _stream()))
    return lvis


def selftest_umma(ctx, a, b, swap_lbo_sbo=False):
    """a, b: [128, K] fp32 CUDA tensors -> a @ b.T through one tcgen05 tile."""
    K = a.shape[1]
    out = torch.empty((128, 128), dtype=torch.float32, device=a.device)
    ctx.launch(ctx.lib.nf_selftest_umma(ctx.h, _f32(a), _f32(b), K, int(swap_lbo_sbo),
                                       _f32(out), _stream()))
    return out


# ------------------------------------------------------------------ training ops

def dense_fwd(ctx, x1, x2, w, b, act, precision='fp32'):
    """y = act([x1 | x2] @ w + b); x2 may be None.  All dims multiples of 4."""
    m, k1 = x1.shape
    k2 = 0 if x2 is None else x2.shape[1]
    n = w.shape[1]
    assert w.shape[0] == k1 + k2
    y = torch.empty((m, n), dtype=torch.float32, device=x1.device)
    nbytes = ctx.lib.nf_dense_fwd_workspace_bytes(n, k1, k2, PREC[precision])
    work = torch.empty((nbytes,), dtype=torch.uint8, device=x1.device) if nbytes else None
    ctx.launch(ctx.lib.nf_dense_fwd(ctx.h, _f32(x1), k1, _f32(x2) if x2 is not None else None,
                                    k2, _f32(w), _f32(b), m, n, ACT[act], _f32(y),
                                    _ptr(work) if work is not None else None, PREC[precision],
                                    _stream()))
    return y


def dense_bwd(ctx, x1, x2, w, y, dy, act, need_dx1, need_dx2, precision='fp32'):
    """-> (dx1 | None, dx2 | None, dw, db) for one Dense layer."""
    m, k1 = x1.shape
    k2 = 0 if x2 is None else x2.shape[1]
    n = w.shape[1]
    dev = x1.device
    dx1 = torch.empty((m, k1), dtype=torch.float32, device=dev) if need_dx1 else None
    dx2 = torch.empty((m, k2), dtype=torch.float32, device=dev) if (need_dx2 and k2) else None
    dw = torch.zeros((k1 + k2, n), dtype=torch.float32, device=dev)
    db = torch.zeros((n,), dtype=torch.float32, device=dev)
    nbytes = ctx.lib.nf_dense_bwd_workspace_bytes(m, n, k1, k2, PREC[precision])
    work = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    ctx.launch(ctx.lib.nf_dense_bwd(
        ctx.h, _f32(x1), k1, _f32(x2) if x2 is not None else None, k2, _f32(w), _f32(y),
        _f32(dy), m, n, ACT[act], _f32(dx1) if dx1 is not None else None,
        _f32(dx2) if dx2 is not None else None, _f32(dw), _f32(db), _ptr(work), PREC[precision],
        _stream()))
    return dx1, dx2, dw, db


def _chain_struct(ws, bs, acts, skip_layer, in_dim):
    ch = MlpChain()
    ch.depth, ch.in_dim, ch.skip_layer = len(ws), int(in_dim), int(skip_layer)
    for l, (w, b, a) in enumerate(zip(ws, bs, acts)):
        ch.width[l], ch.act[l] = int(w.shape[1]), ACT[a]
        ch.w[l], ch.b[l] = w.data_ptr(), b.data_ptr()
    return ch


def mlp_chain_supported(in_dim, widths, n_rows_in):
    """Shapes nf_mlp_chain_fwd / _bwd take (include/nerfactor_b200.h): widths[-1] is the head."""
    if not 2 <= len(widths) <= CHAIN_MAX or in_dim % 4 or widths[-1] % 4:
        return False
    k0p = (in_dim + 15) // 16 * 16
    if any(w % 16 or w > 256 for w in widths[:-1]) or k0p > 256:
        return False
    return all(k <= 256 for k in n_rows_in)


def mlp_chain_fwd(ctx, x, ws, bs, acts, skip_layer, precision='bf16'):
    """Whole mlp.Network forward in one call (nf_mlp_chain_fwd).  ws[l] [in_l, width_l] (the skip
    layer's [width + in_dim, width]), all fp32 contiguous.  -> (y [rows, width[-1]], workspace):
    the workspace holds the 16-bit activations the backward call needs."""
    rows, in_dim = x.shape
    ch = _chain_struct(ws, bs, acts, skip_layer, in_dim)
    nbytes = ctx.lib.nf_mlp_chain_workspace_bytes(C.byref(ch), rows)
    if rows and not nbytes:
        raise NfError('nf_mlp_chain: unsupported network shape')
    work = torch.empty((max(nbytes, 16),), dtype=torch.uint8, device=x.device)
    y = torch.empty((rows, ws[-1].shape[1]), dtype=torch.float32, device=x.device)
    ctx.launches += 2 * len(ws)
    ctx.launch(ctx.lib.nf_mlp_chain_fwd(ctx.h, C.byref(ch), _f32(x), rows, _f32(y), _ptr(work),
                                        PREC[precision], _stream()))
    return y, work


def mlp_chain_bwd(ctx, ws, bs, acts, skip_layer, in_dim, y, dy, work, need_dx, precision='bf16'):
    """-> (dx | None, [dw_l], [db_l]) for the network nf_mlp_chain_fwd just ran on `work`."""
    rows = y.shape[0]
    dev = y.device
    ch = _chain_struct(ws, bs, acts, skip_layer, in_dim)
    dx = torch.empty((rows, in_dim), dtype=torch.float32, device=dev) if need_dx else None
    dws = [torch.zeros_like(w) for w in ws]
    dbs = [torch.zeros_like(b) for b in bs]
    pw = (C.c_void_p * CHAIN_MAX)(*([t.data_ptr() for t in dws] + [None] * (CHAIN_MAX - len(ws))))
    pb = (C.c_void_p * CHAIN_MAX)(*([t.data_ptr() for t in dbs] + [None] * (CHAIN_MAX - len(bs))))
    ctx.launches += 6 * len(ws)
    ctx.launch(ctx.lib.nf_mlp_chain_bwd(ctx.h, C.byref(ch), rows, _f32(y), _f32(dy),
                                        _f32(dx) if dx is not None else None, pw, pb, _ptr(work),
                                        PREC[precision], _stream()))
    return dx, dws, dbs


def adam_amsgrad_step(ctx, param, grad, m, v, vhat, lr, step, beta1=0.9, beta2=0.999,
                      eps=1e-7):
    ctx.launch(ctx.lib.nf_adam_amsgrad_step(
        ctx.h, _f32(param), _f32(grad), _f32(m), _f32(v), _f32(vhat), param.numel(), float(lr),
        float(beta1), float(beta2), float(eps), int(step), _stream()))


def selftest_tmem(ctx, reader_warps, iters, mma_iters, mode):
    """-> (reader cycles, MMA-stream cycles) of the TMEM throughput microbenchmark."""
    out = torch.zeros((4,), dtype=torch.int64, device=ctx.device)
    ctx.launch(ctx.lib.nf_selftest_tmem(ctx.h, reader_warps, iters, mma_iters, mode, _ptr(out),
                                       _stream()))
    o = out.cpu().tolist()
    return o[0], o[1]


def selftest_umma2(ctx, a, b):
    """a: [256, K], b: [128, K] fp32 CUDA tensors -> a @ b.T through one CTA-pair tcgen05 tile."""
    K = a.shape[1]
    out = torch.empty((256, 128), dtype=torch.float32, device=a.device)
    ctx.launch(ctx.lib.nf_selftest_umma2(ctx.h, _f32(a), _f32(b), K, _f32(out), _stream()))
    return out
