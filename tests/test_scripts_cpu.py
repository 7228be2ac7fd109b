"""Host side of the drop-in scripts (nerfactor/test.py, trainvali.py, geometry_from_nerf.py) and
of the models' `vis_batch` / `compile_batch_vis` (SURVEY.md 8f.4): everything that does not need
the GPU.  The end-to-end run of the three scripts on a B200 is tests/test_zz_gpu_scripts.py."""
import os
from collections import OrderedDict

import numpy as np
import pytest

from nerfactor_b200 import config as nfconfig
from nerfactor_b200 import test as nftest
from nerfactor_b200 import trainvali, geometry_from_nerf as gfn
from nerfactor_b200.models._visualize import NeRFactorVis, ShapeVis, NerfVis
from nerfactor_b200.util import img as imgutil, io as ioutil

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'ref_host_code.npz')


# ------------------------------------------------------------------------------ test.py
def test_albedo_overrides():
    xyz = np.array([[-1.6, 0, 0], [-1.5, 0, 0], [-1.0, 0, 0], [0.0, 0, 0], [1.49, 0, 0],
                    [1.5, 0, 0]], np.float32)
    assert np.allclose(nftest.get_albedo_override(xyz, 'gold'), (1, 0.843, 0))
    assert np.allclose(nftest.get_albedo_override(xyz, 'aluminium'), (0.913, 0.921, 0.925))
    rb = nftest.get_albedo_override(xyz, 'rainbow')
    # 7 bands over [-1.5, 1.5): outside stays black (test.py:105-119)
    assert np.allclose(rb[0], 0) and np.allclose(rb[5], 0)
    assert np.allclose(rb[1], (0.58, 0, 0.83)) and np.allclose(rb[4], (1, 0, 0))
    assert np.allclose(rb[3], (0, 1, 0))
    rb_y = nftest.get_albedo_override(xyz, 'rainbow', sv_axis_i=1)
    assert np.allclose(rb_y, (0, 1, 0))                  # y = 0 everywhere -> the middle band
    tb = nftest.get_albedo_override(xyz, 'turbo')
    assert tb.shape == (6, 3) and np.allclose(tb[0], 0) and tb.min() >= 0 and tb.max() <= 1
    with pytest.raises(NotImplementedError):
        nftest.get_albedo_override(xyz, 'plaid')


def test_turbo_fit_against_reference_table():
    """nftest.turbo vs the reference's turbo table and its interpolate_or_clip
    (third_party/turbo_colormap.py), values stored by tests/golden/make_golden_host.py."""
    g = np.load(GOLDEN)
    xs = np.linspace(0, 1, 501)
    assert np.abs(nftest.turbo(xs) - g['turbo/table']).max() < 0.011
    assert list(g['turbo/below']) == [0.0, 0.0, 0.0]
    assert list(g['turbo/above']) == [1.0, 1.0, 1.0]


def test_compute_rgb_scales(tmp_path):
    """test.py:46-88 on a hand-made run directory: prediction = 0.5 x ground truth (linear)."""
    run = tmp_path / 'out' / 'lr5e-3'
    cfg = nfconfig.default_config('nerfactor', data_root=str(tmp_path / 'data'))
    ioutil.write_config(cfg, str(run) + '.ini')
    rng = np.random.default_rng(0)
    gt_lin = rng.uniform(0.2, 0.9, size=(8, 8, 3))
    alpha = np.ones((8, 8))
    alpha[:2] = 0
    gt_rgba = np.concatenate([gt_lin, alpha[..., None]], -1)
    imgutil.write_arr(gt_rgba, str(tmp_path / 'data' / 'val_000' / 'albedo.png'))
    bd = run / 'vis_vali' / 'epoch000000010' / 'batch000000000'
    imgutil.write_arr((0.5 * gt_lin) ** (1 / 2.2), str(bd / 'pred_albedo.png'))
    ioutil.write_json({'id': 'val_000'}, str(bd / 'metadata.json'))
    scales = nftest.compute_rgb_scales(str(run / 'checkpoints' / 'ckpt-10'))
    assert scales.shape == (3,) and np.allclose(scales, 2.0, atol=0.06)   # 8-bit round trips


def test_flag_names_match_reference():
    a = nftest.parse_args(['--ckpt', '/o/x/checkpoints/ckpt-3', '--tgt_albedo', 'gold',
                           '--sv_axis_i', '2', '--color_correct_albedo'])
    assert a.ckpt.endswith('ckpt-3') and a.tgt_albedo == 'gold' and a.sv_axis_i == 2
    assert a.color_correct_albedo and a.sv_axis_min == -1.5 and a.sv_axis_max == 1.5
    t = trainvali._parse_args(['--config', 'shape.ini', '--config_override', 'imh=64,lr=1e-3'])
    assert t.config == 'shape.ini' and t.device == 'gpu' and not t.debug
    g = gfn._parse_args(['--trained_nerf', '/n', '--out_root', '/o', '--light_h', '8',
                         '--scene_bbox=-1,1,-1,1,0,2', '--occu_thres', '0.5'])
    assert g.lvis_far == 1. and g.light_h == 8 and g.spp == 1 and g.mlp_chunk == 1_500_000
    assert gfn.parse_bbox(g.scene_bbox) == [-1., 1., -1., 1., 0., 2.]


def test_load_config_and_prune(tmp_path):
    cfg = trainvali.load_config('nerfactor_microfacet.ini', 'imh=64,lr=1e-3,xname=run{lr}')
    assert cfg.getint('DEFAULT', 'imh') == 64 and cfg.get('DEFAULT', 'model') == 'nerfactor_microfacet'
    from nerfactor_b200.util import config as configutil
    assert cfg.get('DEFAULT', 'xname').format(**configutil.config2dict(cfg)) == 'run1e-3'
    ioutil.write_config(cfg, str(tmp_path / 'my.ini'))
    assert trainvali.load_config(str(tmp_path / 'my.ini')).getfloat('DEFAULT', 'lr') == 1e-3
    d = tmp_path / 'checkpoints'
    d.mkdir()
    for s in (1, 2, 10):
        for ext in ('index', 'data-00000-of-00001'):
            (d / ('ckpt-%d.%s' % (s, ext))).write_bytes(b'x')
    trainvali._prune(str(d), -1)
    assert len(list(d.iterdir())) == 6
    trainvali._prune(str(d), 2)
    assert sorted(p.name for p in d.iterdir()) == [
        'ckpt-10.data-00000-of-00001', 'ckpt-10.index', 'ckpt-2.data-00000-of-00001', 'ckpt-2.index']


# -------------------------------------------------------------------------- vis_batch
class _FakeBase:
    white_bg, debug = True, False

    @staticmethod
    def _validate_mode(mode):
        if mode not in ('train', 'vali', 'test'):
            raise ValueError(mode)


class _FakeNeRFactor(NeRFactorVis, _FakeBase):
    shape_mode = 'finetune'
    light_res = (4, 8)

    def __init__(self, data_root):
        rng = np.random.default_rng(1)
        self.config = nfconfig.default_config('nerfactor_microfacet', light_h=4,
                                              data_root=data_root)
        self.lareas = np.ones((4, 8), np.float32)
        self.light = rng.random((4, 8, 3)).astype(np.float32)
        self.novel_probes = OrderedDict(p0=(rng.random((4, 8, 3)) * 5).astype(np.float32))
        self.novel_olat = OrderedDict()
        for i in range(4):
            for j in range(8):
                env = np.zeros((4, 8, 3), np.float32)
                env[i, j] = 200.
                self.novel_olat['%04d-%04d' % (i, j)] = env

    def _brdf_prop_as_img(self, brdf_prop):
        return np.concatenate([brdf_prop] * 3, axis=2)


def _to_vis(h, w, L, id_, seed=0):
    r = np.random.default_rng(seed)
    n = h * w
    return {'id': id_, 'hw': (h, w), 'pred_rgb': r.random((n, 3)),
            'pred_normal': r.random((n, 3)) * 2 - 1, 'pred_lvis': r.random((n, L)),
            'pred_albedo': r.random((n, 3)), 'pred_brdf': r.random((n, 1)),
            'pred_rgb_probes': r.random((n, 1, 3)), 'pred_rgb_olat': r.random((n, L, 3)),
            'gt_rgb': r.random((n, 3)), 'gt_normal': r.random((n, 3)) * 2 - 1,
            'gt_lvis': r.random((n, L)), 'gt_alpha': (r.random((n, 1)) > 0.3).astype(np.float32)}


def test_nerfactor_vis_batch_vali_and_test(tmp_path):
    m = _FakeNeRFactor(str(tmp_path / 'data'))
    tv = _to_vis(12, 10, 32, 'val_000')
    vdir = str(tmp_path / 'vis_vali' / 'epoch000000001' / 'batch000000000')
    keep = dict(tv)
    m.vis_batch(tv, vdir, mode='vali')
    assert set(tv) == set(keep)                        # the caller's dict is left intact
    names = set(os.listdir(vdir))
    assert {'pred_rgb.png', 'gt_rgb.png', 'pred_albedo.png', 'pred_brdf.png', 'pred_normal.png',
            'pred_lvis.png', 'pred-vs-gt_rgb.apng', 'pred-vs-gt_normal.apng',
            'pred-vs-gt_lvis.apng', 'metadata.json', 'pred_rgb_probes_p0.png'} <= names
    assert os.path.exists(os.path.join(os.path.dirname(vdir), 'pred_light.png'))
    meta = ioutil.read_json(os.path.join(vdir, 'metadata.json'))
    assert meta['id'] == 'val_000' and 3 < meta['psnr'] < 20
    # written RGB = alpha-blend onto white with the stricter alpha, truncated to 8 bit
    alpha = keep['gt_alpha'].reshape(12, 10)
    want = (np.clip(keep['pred_rgb'].reshape(12, 10, 3) * alpha[..., None] +
                    (1 - alpha[..., None]), 0, 1) * 255).astype(np.uint8)
    assert np.array_equal(imgutil.read(os.path.join(vdir, 'pred_rgb.png')), want)
    html = m.compile_batch_vis([vdir], os.path.join(os.path.dirname(vdir), 'all'), mode='vali')
    assert html.endswith('all.html') and 'pred-vs-gt_rgb.apng' in open(html).read()
    assert m.vis_batch(dict(keep), vdir + 'x', mode='train') is None and not os.path.exists(vdir + 'x')
    with pytest.raises(ValueError):
        m.vis_batch(dict(keep), vdir, mode='bogus')
    # test mode: OLAT renders for the upper hemisphere, per-light visibility, then the video
    tdirs = []
    for i in range(2):
        tdir = str(tmp_path / 'vis_test' / ('batch%09d' % i))
        tv = _to_vis(12, 10, 32, 'test_%03d' % i, seed=i)
        if i == 0:
            tv['pred_rgb_olat'] = None
        m.vis_batch(tv, tdir, mode='test', olat_vis=(i == 1))
        tdirs.append(tdir)
    last = set(os.listdir(tdirs[1]))
    assert sum(n.startswith('pred_rgb_olat_') for n in last) == 16
    assert sum(n.startswith('pred_lvis_olat_') for n in last) == 16
    assert ioutil.read_json(os.path.join(tdirs[0], 'metadata.json')) == {'id': 'test_000'}
    mp4 = m.compile_batch_vis(tdirs, str(tmp_path / 'vis_test' / 'all'), mode='test')
    assert mp4.endswith('all.mp4') and os.path.getsize(mp4) > 1000


class _FakeShape(ShapeVis, _FakeBase):
    config = nfconfig.default_config('shape')


def test_shape_vis_batch(tmp_path):
    m = _FakeShape()
    tv = {k: v for k, v in _to_vis(8, 8, 16, 'val_001').items()
          if k in ('id', 'hw', 'pred_normal', 'pred_lvis', 'gt_normal', 'gt_lvis', 'gt_alpha')}
    # the reference's per-ray tiled id / hw are accepted too (nerf_shape.py:79-81)
    tv['id'] = np.array([b'val_001'] * 64)
    tv['hw'] = np.tile(np.array([[8, 8]], np.int32), (64, 1))
    vdir = str(tmp_path / 'e' / 'batch000000000')
    m.vis_batch(tv, vdir, mode='vali')
    assert {'pred-vs-gt_normal.apng', 'pred-vs-gt_lvis.apng', 'gt_alpha.png',
            'metadata.json'} <= set(os.listdir(vdir))
    assert m.compile_batch_vis([vdir], str(tmp_path / 'e' / 'all'), 'vali').endswith('.html')
    with pytest.raises(NotImplementedError):
        m.compile_batch_vis([vdir], str(tmp_path / 'e' / 'all'), 'test')


class _FakeNerf(NerfVis, _FakeBase):
    config = nfconfig.default_config('nerf')
    near, far = 2., 6.


def test_nerf_vis_batch(tmp_path):
    m = _FakeNerf()
    r = np.random.default_rng(0)
    n = 36
    tv = {'id': 'val_000', 'hw': (6, 6), 'gt_rgb': r.random((n, 3))}
    for p in ('coarse_', 'fine_'):
        tv.update({p + 'rgb': r.random((n, 3)), p + 'occu': r.random(n),
                   p + 'depth': r.uniform(2, 6, n), p + 'disp': r.uniform(1 / 6, 1 / 2, n)})
    vdir = str(tmp_path / 'e' / 'batch000000000')
    m.vis_batch(tv, vdir, mode='vali')
    assert {'fine-vs-gt_rgb.apng', 'fine-vs-coarse_depth.apng', 'fine_occu.png',
            'metadata.json'} <= set(os.listdir(vdir))
    # white background: occupancy is written inverted (nerf.py:337-338)
    occ = imgutil.read(os.path.join(vdir, 'fine_occu.png'))
    assert np.array_equal(occ, ((1 - tv['fine_occu'].reshape(6, 6)) * 255).astype(np.uint8))
    assert m.compile_batch_vis([vdir], str(tmp_path / 'e' / 'all'), 'vali').endswith('.html')
    assert m.compile_batch_vis([vdir], str(tmp_path / 'e' / 'vid'), 'test').endswith('.mp4')


def test_vis_batch_equals_reference_vis_batch(tmp_path, monkeypatch):
    """The reference's NeRFactor `vis_batch` (nerfactor.py:562-739, its own file, run through the
    TensorFlow shim on the reference model's own outputs by tests/golden/make_golden_host.py) vs
    `vis_batch` here on the same `to_vis`: same files, same pixels (text-free images), incl. OLAT /
    probe renders composited on the average light and the per-light visibility maps."""
    import json
    import torch
    import cpu_backend
    from nerfactor_b200 import synth
    from nerfactor_b200.models.nerfactor_microfacet import Model
    g = np.load(GOLDEN)
    lh, h, w = 2, 6, 5
    params = synth.make_stage_b_params(7, 'microfacet', light_hw=(lh, 2 * lh))
    probes = synth.make_probes(5, 2, (lh, 2 * lh))
    mine_in = {k[len('vis/in/'):]: g[k].copy() for k in g.files if k.startswith('vis/in/')}
    mine_in['id'], mine_in['hw'] = 'test_007', (h, w)
    mdir = str(tmp_path / 'mine')
    # ---- the model here (host code only: vis_batch never touches the kernels)
    ctx = cpu_backend.install(monkeypatch)
    m = Model(nfconfig.default_config('nerfactor_microfacet', light_h=lh), params=params,
              ctx=ctx, precision='fp32')
    for i, p in enumerate(probes):
        m.novel_probes['p%d' % i] = torch.as_tensor(p)
    m.vis_batch(mine_in, mdir, mode='test', olat_vis=True)
    rf, mf = list(g['vis/files']), sorted(os.listdir(mdir))
    assert rf == mf and len(rf) > 20
    assert json.loads(str(g['vis/metadata'])) == ioutil.read_json(os.path.join(mdir, 'metadata.json'))
    for f in rf:
        if f.endswith('.png'):
            a = g['vis/png/' + f].astype(int)
            b = imgutil.read(os.path.join(mdir, f)).astype(int)
            assert a.shape == b.shape and np.abs(a - b).max() <= 1, f


def test_stage_a_files_equal_reference_process_view(tmp_path, monkeypatch):
    """geometry_from_nerf.process_view of the reference (its own file through the shim: march,
    occupancy threshold, alpha / xyz / normal maps, hit mask, light visibility, alpha masking,
    file writers; stored by tests/golden/make_golden_host.py) vs `process_view` +
    `write_view_buffers` here on the CPU test double: the four buffers a Stage-B dataset reads."""
    import torch
    import cpu_backend
    from nerfactor_b200 import synth
    from nerfactor_b200.models.nerf import Model
    from nerfactor_b200.util import geom_io
    from oracle import stage_a
    g = np.load(GOLDEN)
    lh, h, w = 2, 5, 6
    mdir = str(tmp_path / 'mine')
    params = synth.make_nerf_params(3)
    rayo, rayd = stage_a.gen_rays(synth.look_at_c2w(), synth.CAM_ANGLE_X, h, w)
    rayo, rayd = rayo.reshape(-1, 3), rayd.reshape(-1, 3)
    # ---- here, kernels replaced by the test double
    ctx = cpu_backend.install(monkeypatch)
    model = Model(nfconfig.default_config('nerf', n_samples_coarse=-48, n_samples_fine=8),
                  params=params, ctx=ctx, precision='fp32')
    ro = torch.as_tensor(rayo)
    rd = torch.as_tensor(rayd)
    rd = rd * torch.rsqrt(torch.clamp((rd * rd).sum(1, keepdim=True), min=1e-12))
    buffers = gfn.process_view(model, ro, rd, (h, w), model.config, occu_thres=0.9,
                               lvis_far=1., light_h=lh, precision='fp32')
    md_ = os.path.join(mdir, 'train_003')
    geom_io.write_view_buffers(buffers, md_)
    assert geom_io.view_done(md_)
    a_r = g['process_view/alpha.png'].astype(int)
    a_m = imgutil.read(os.path.join(md_, 'alpha.png')).astype(int)
    assert a_r.shape == a_m.shape and np.abs(a_r - a_m).max() <= 1
    assert 0 < (a_r > 0).mean() < 1                   # the threshold removed some pixels
    for f, tol in (('xyz.npy', 2e-5), ('normal.npy', 2e-4), ('lvis.npy', 5e-5)):
        r, m_ = g['process_view/' + f], np.load(os.path.join(md_, f))
        assert r.shape == m_.shape and r.dtype == m_.dtype == np.float32
        assert np.abs(r - m_).max() < tol, (f, np.abs(r - m_).max())
