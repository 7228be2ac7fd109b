"""Host-side data formats either side of the hot path (SURVEY.md 8f): dataset classes
(nerfactor/datasets/{base,nerf,nerf_shape}.py), light-probe loading (nerfactor.py:85-92,
169-179), image helpers.  The mirrors of the reference's own loaders, writers and image helpers
are compared with what that code returned on the same inputs (tests/golden/ref_host_code.npz,
written by tests/golden/make_golden_host.py)."""
import os

import numpy as np
import pytest

from nerfactor_b200 import config as nfconfig, synth
from nerfactor_b200.datasets import get_dataset_class
from nerfactor_b200.util import img as imgutil, light as lightutil, io as ioutil, \
    config as configutil

HERE = os.path.dirname(os.path.abspath(__file__))


def _golden():
    return np.load(os.path.join(HERE, 'golden', 'ref_host_code.npz'))


def _cfg(root, nerf_root=None, **kw):
    cfg = nfconfig.default_config('nerfactor', imh=8, data_root=str(root),
                                  n_rays_per_step=32, cache=True, **kw)
    if nerf_root is not None:
        cfg.set('DEFAULT', 'data_nerf_root', str(nerf_root))
    return cfg


def test_nerf_dataset_modes(tmp_path):
    root = tmp_path / 'scene'
    synth.write_scene(str(root), imh=16, imw=16, n_train=3, n_val=1, n_test=2)
    cfg = _cfg(root)
    D = get_dataset_class('nerf')
    train = D(cfg, 'train', seed=0)
    assert train.get_n_views() == 3 and train.bs == 32
    pipe = train.build_pipeline(no_batch=True)
    epoch = list(pipe)
    assert len(epoch) == 3
    id_, hw, rayo, rayd, rgb = epoch[0]
    assert hw == (8, 8) and tuple(rayo.shape) == (32, 3) and tuple(rgb.shape) == (32, 3)
    assert sorted(e[0] for e in epoch) == ['train_000', 'train_001', 'train_002']
    # a second epoch reshuffles and resamples but serves the cached decode
    assert len(list(pipe)) == 3
    vali = D(cfg, 'vali')
    assert vali.bs == 64
    (id_, hw, rayo, rayd, rgb), = list(vali.build_pipeline(no_batch=True))
    assert id_ == 'val_000' and tuple(rgb.shape) == (64, 3)
    # white background where the RGBA image is transparent (nerf.py:165-168)
    assert float(rgb.max()) <= 1. and float(rgb[0].min()) == 1.
    test = D(cfg, 'test')
    out = list(test.build_pipeline(no_batch=True, no_shuffle=True))
    assert [o[0] for o in out] == ['test_000', 'test_001']
    assert float(out[0][4].abs().max()) == 0.          # placeholder RGB (nerf.py:155-157)


def test_gen_rays_matches_geom_io_and_row_major(tmp_path):
    from nerfactor_b200.util import geom_io
    root = tmp_path / 'scene'
    synth.write_scene(str(root), imh=8, imw=8, n_train=1, n_val=0, n_test=0)
    ds = get_dataset_class('nerf')(_cfg(root), 'train', always_all_rays=True)
    c2w = synth.look_at_c2w()
    o, d = ds._gen_rays(c2w, synth.CAM_ANGLE_X, 6, 10)
    o2, d2 = geom_io.gen_rays_host(c2w, synth.CAM_ANGLE_X, 6, 10)
    assert np.array_equal(o, o2) and np.array_equal(d, d2)
    # pixel (y, x) -> ray y * W + x, pixel corners (no half-pixel offset), datasets/nerf.py:180-191
    fl = .5 * 10 / np.tan(.5 * synth.CAM_ANGLE_X)
    local = np.array([(3 - 5.) / fl, -(2 - 3.) / fl, -1.])
    assert np.allclose(d.reshape(-1, 3)[2 * 10 + 3], c2w[:3, :3] @ local, rtol=0, atol=1e-15)


def test_nerf_shape_dataset(tmp_path):
    root, nroot = tmp_path / 'scene', tmp_path / 'nerf_out'
    synth.write_scene(str(root), imh=8, imw=8, n_train=2, n_val=1, n_test=1,
                      nerf_root=str(nroot), n_lights=16)
    # a view without buffers is skipped (nerf_shape.py:44-63)
    os.remove(str(nroot / 'train_001' / 'lvis.npy'))
    cfg = _cfg(root, nroot, use_nerf_alpha=False)
    D = get_dataset_class('nerf_shape')
    train = D(cfg, 'train', seed=1)
    assert [os.path.basename(os.path.dirname(f)) for f in train.files] == ['train_000']
    batch, = list(train.build_pipeline(no_batch=True))
    id_, hw, rayo, rayd, rgb, alpha, xyz, normal, lvis = batch
    assert id_ == 'train_000' and hw == (8, 8)
    assert tuple(alpha.shape) == (32, 1) and tuple(lvis.shape) == (32, 16)
    assert float(alpha.min()) > 0.9                     # foreground-only sampling (:84-107)
    assert np.allclose(np.linalg.norm(normal.numpy(), axis=1), 1., atol=1e-5)
    test = D(cfg, 'test')
    id_, hw, rayo, rayd, rgb, alpha, xyz, normal, lvis = next(iter(
        test.build_pipeline(no_batch=True, no_shuffle=True)))
    assert tuple(xyz.shape) == (64, 3) and float(rgb.abs().max()) == 0.
    # row-major flatten of the stored buffers
    ref_xyz = np.load(str(nroot / 'test_000' / 'xyz.npy')).reshape(-1, 3)
    assert np.array_equal(xyz.numpy(), ref_xyz)


def test_pipeline_take_and_error_propagation(tmp_path):
    root = tmp_path / 'scene'
    synth.write_scene(str(root), imh=8, imw=8, n_train=3, n_val=2, n_test=0)
    ds = get_dataset_class('nerf')(_cfg(root), 'vali')
    pipe = ds.build_pipeline(no_batch=True)
    assert len(list(pipe.take(1))) == 1 and len(pipe.take(1)) == 1
    os.remove(ds.meta2img[ds.files[1]])
    ds2 = get_dataset_class('nerf')(_cfg(root), 'vali')
    assert ds2.get_n_views() == 1                       # unpaired camera skipped (nerf.py:78-88)
    pipe._cached.clear()
    with pytest.raises(FileNotFoundError):
        list(pipe)                                      # loader-thread error reaches the consumer


def test_light_probe_loading(tmp_path):
    envdir = tmp_path / 'envmaps'
    synth.write_scene(str(tmp_path / 's'), n_train=0, n_val=0, n_test=0,
                      envmap_dir=str(envdir), n_probes=2)
    probes = lightutil.load_probes(str(envdir), 16)
    assert list(probes) == ['probe0', 'probe1']
    p = probes['probe0']
    assert p.shape == (16, 32, 3) and p.dtype == np.float32 and p.min() >= 0
    # energy-preserving box-like average: the antialiased resize of a constant is the constant
    const = np.full((64, 128, 3), 3.5, np.float32)
    assert np.allclose(imgutil.resize(const, new_h=16), 3.5, atol=1e-5)
    vis = lightutil.vis_light(p, h=32)
    assert vis.shape == (32, 64, 3) and vis.dtype == np.uint8 and vis.max() == 255
    assert len(lightutil.vis_olat_lights(2, 8)) == 8


def test_resize_matches_pillow_antialias():
    """tf.image.resize(bilinear, antialias=True) follows Pillow's reducing BILINEAR filter
    (half-pixel centres, triangle support scaled by the ratio, renormalised weights)."""
    from PIL import Image
    rng = np.random.default_rng(0)
    for h, w, nh in ((64, 128, 16), (100, 200, 16), (16, 32, 32), (37, 74, 16)):
        a = (rng.random((h, w)) * 10).astype(np.float32)
        r = imgutil.resize(a, new_h=nh)
        p = np.array(Image.fromarray(a, mode='F').resize((r.shape[1], r.shape[0]),
                                                         Image.BILINEAR))
        assert np.abs(r - p).max() < 5e-6


def test_image_helpers_roundtrip(tmp_path):
    a = np.random.default_rng(0).random((12, 10, 3))
    u = imgutil.write_arr(a, str(tmp_path / 'a.png'), clip=True)
    assert np.array_equal(u, (a * 255).astype(np.uint8))            # truncation, io/img.py:150
    assert np.array_equal(imgutil.read(str(tmp_path / 'a.png')), u)
    with pytest.raises(AssertionError):
        imgutil.write_arr(a + 1, str(tmp_path / 'b.png'))
    psnr = imgutil.PSNR('uint8')
    with np.errstate(divide='ignore'):
        assert psnr(u, u.copy()) == np.inf
    v = u.copy()
    v[0, 0, :] ^= 8
    assert 40 < psnr(u, v) < 80
    cfg = nfconfig.default_config('nerfactor')
    ioutil.write_config(cfg, str(tmp_path / 'x' / 'run.ini'))
    back = ioutil.read_config(str(tmp_path / 'x' / 'run.ini'))
    assert configutil.config2dict(back) == configutil.config2dict(cfg)
    assert configutil.get_config_ini('/o/run/checkpoints/ckpt-3') == '/o/run.ini'


def test_against_importable_reference_helpers(tmp_path):
    g = _golden()
    rng = np.random.default_rng(3)
    a = rng.random((20, 30, 3))
    u8 = (a * 255).astype(np.uint8)
    assert np.array_equal(imgutil.normalize_uint(u8), g['helpers/normalize_uint'])
    assert np.array_equal(imgutil.denormalize_float(a), g['helpers/denormalize_float'])
    hdr = (rng.random((8, 16, 3)) * 30).astype(np.float32)
    assert np.array_equal(imgutil.tonemap(hdr, gamma=4), g['helpers/tonemap'])
    assert np.array_equal(imgutil.resize_cv2(a, new_h=10), g['helpers/resize'])
    assert np.array_equal(imgutil.alpha_blend(a, a[:, :, 0]), g['helpers/alpha_blend'])
    assert abs(imgutil.PSNR('uint8')(u8, u8[::-1].copy()) - float(g['helpers/psnr'])) < 1e-12
    lightutil.write_hdr(hdr, str(tmp_path / 'p.hdr'))
    # xm.io.hdr.read itself calls np.fromstring (removed in NumPy 2); same two cv2 calls by hand
    import cv2
    buf = np.frombuffer(open(str(tmp_path / 'p.hdr'), 'rb').read(), np.uint8)
    want = cv2.cvtColor(cv2.imdecode(buf, cv2.IMREAD_UNCHANGED), cv2.COLOR_BGR2RGB)
    assert np.array_equal(lightutil.read_hdr(str(tmp_path / 'p.hdr')), want)
    open(str(tmp_path / 'b.txt'), 'w').close()
    open(str(tmp_path / 'a.txt'), 'w').close()
    assert [os.path.relpath(p, str(tmp_path)) for p in ioutil.sortglob(
        str(tmp_path), '*', ext='txt')] == list(g['helpers/sortglob'])


# ---- the reference's own loaders / writers, run on the same inputs by make_golden_host.py ------
def _rel(files, base):
    return [os.path.relpath(f, str(base)) for f in files]


def _check_loads(ds, g, pre):
    """Every view `ds` serves loads to what the reference's loader returned for it."""
    for i, path in enumerate(ds.files):
        m = ds._load_data(path)
        assert m[0] == g[pre + '%d/id' % i].item() and len(m) - 1 == int(g[pre + '%d/n' % i])
        for j, b in enumerate(m[1:]):
            a = g[pre + '%d/%d' % (i, j)]
            assert a.shape == np.shape(b) and np.array_equal(np.asarray(a, np.float32), b), (pre, j)


def test_dataset_loaders_equal_reference_loaders(tmp_path):
    """nerfactor/datasets/{nerf,nerf_shape}.py `_glob` + `_load_data` (the reference's files,
    unmodified) vs the loaders here, on a synthetic scene in the reference's layout, incl. the
    resize-on-load path (imh != stored height)."""
    g = _golden()
    root, nroot = tmp_path / 'scene', tmp_path / 'surf'
    synth.write_scene(str(root), imh=16, imw=16, n_train=2, n_val=1, n_test=1,
                      nerf_root=str(nroot), n_lights=8)
    for imh in (16, 8):
        cfg = _cfg(root, nroot, use_nerf_alpha=False, no_batch=True)
        cfg.set('DEFAULT', 'imh', str(imh))
        for mode in ('train', 'vali', 'test'):
            pre = 'loaders/shape/%d/%s/' % (imh, mode)
            mine = get_dataset_class('nerf_shape')(cfg, mode)
            assert _rel(mine.files, tmp_path) == list(g[pre + 'files'])
            _check_loads(mine, g, pre)
        # ray generation incl. the NDC branch and 2 x 2 sub-pixel samples (nerf.py:172-214)
        for ndc in ('False', 'True'):
            cfg.set('DEFAULT', 'ndc', ndc)
            for sps in (1, 2):
                mm = get_dataset_class('nerf').__new__(get_dataset_class('nerf'))
                mm.config, mm.sps = cfg, sps
                c2w = synth.look_at_c2w(3.0, 40.0, 25.0)
                got = mm._gen_rays(c2w, 0.7, 6, 9)
                assert len(got) == 2
                for k, b in enumerate(got):
                    a = g['loaders/rays/%d/%s/%d/%d' % (imh, ndc, sps, k)]
                    assert a.shape == b.shape and np.allclose(a, b, rtol=1e-13, atol=1e-13)
        cfg.set('DEFAULT', 'ndc', 'False')
        minen = get_dataset_class('nerf')(cfg, 'train')
        assert _rel(minen.files, tmp_path) == list(g['loaders/nerf/%d/files' % imh])
        for i, path in enumerate(minen.files):
            m = minen._load_data(path)
            assert m[0] == g['loaders/nerf/%d/%d/id' % (imh, i)].item()
            assert len(m) - 1 == int(g['loaders/nerf/%d/%d/n' % (imh, i)])
            assert all(np.array_equal(g['loaders/nerf/%d/%d/%d' % (imh, i, j)], b)
                       for j, b in enumerate(m[1:]))


def test_geometry_buffer_writers_equal_reference_writers(tmp_path):
    """nerfactor/util/geom.py write_alpha / write_xyz / write_normal (and the raw + averaged part
    of write_lvis) vs util/geom_io.py: same .npy bytes, same PNG pixels."""
    from nerfactor_b200.util import geom_io
    g = _golden()
    rng = np.random.default_rng(0)
    alpha = rng.random((9, 7)).astype(np.float32)
    xyz = (rng.standard_normal((9, 7, 3)) * alpha[..., None]).astype(np.float32)
    nrm = rng.standard_normal((9, 7, 3)).astype(np.float32)
    nrm /= np.linalg.norm(nrm, axis=2, keepdims=True)
    lvis = rng.random((9, 7, 8)).astype(np.float32)
    md = str(tmp_path / 'mine')
    geom_io.write_view_buffers({'alpha': alpha, 'xyz': xyz, 'normal': nrm, 'lvis': lvis}, md)
    for f in ('xyz.npy', 'normal.npy', 'lvis.npy'):
        assert open(os.path.join(md, f), 'rb').read() == g['writers/' + f].tobytes(), f
    for f in ('alpha.png', 'xyz.png', 'normal.png', 'lvis.png'):
        a, b = g['writers/' + f], imgutil.read(os.path.join(md, f))
        assert a.shape == b.shape and np.array_equal(a, b), f


def _write_mvs_scene(root, imh=8):
    """The MVS layout (datasets/mvs_shape.py): everything of a view in <mvs_root>/<view>/, the
    metadata carries `cam_loc`, the lights sit in <mvs_root>/lights.npz."""
    import json
    import shutil
    from nerfactor_b200.brdf.renderer import gen_light_xyz
    tmp = str(root) + '_src'
    synth.write_scene(tmp, imh=imh, imw=imh, n_train=2, n_val=1, n_test=1,
                      nerf_root=tmp + '_buf', n_lights=8)
    for id_ in sorted(os.listdir(tmp)):
        d = os.path.join(str(root), id_)
        shutil.copytree(os.path.join(tmp, id_), d)
        for f in os.listdir(os.path.join(tmp + '_buf', id_)):
            shutil.copy(os.path.join(tmp + '_buf', id_, f), d)
        meta = json.load(open(os.path.join(d, 'metadata.json')))
        c2w = np.array([float(x) for x in meta['cam_transform_mat'].split(',')]).reshape(4, 4)
        meta['cam_loc'] = [float(x) for x in c2w[:3, 3]]
        json.dump(meta, open(os.path.join(d, 'metadata.json'), 'w'))
    lxyz, lareas = gen_light_xyz(2, 4)
    np.savez(os.path.join(str(root), 'lights.npz'), lxyzs=lxyz * 0.5, lareas=lareas)


def test_mvs_shape_dataset(tmp_path):
    root = tmp_path / 'mvs'
    _write_mvs_scene(root)
    cfg = _cfg(tmp_path / 'unused', None, mvs_root=str(root), use_nerf_alpha=True)
    ds = get_dataset_class('mvs_shape')(cfg, 'train', seed=0)
    assert ds.get_n_views() == 2
    id_, hw, rayo, rayd, rgb, alpha, xyz, normal, lvis = next(iter(ds.build_pipeline()))
    assert hw == (8, 8) and tuple(lvis.shape) == (32, 8)
    assert float(rayd.abs().max()) == 0.                      # dummy directions
    assert np.allclose(np.linalg.norm(rayo.numpy(), axis=1), 4., atol=1e-5)   # the camera location


def test_mvs_shape_loader_equals_reference_loader(tmp_path):
    g = _golden()
    root = tmp_path / 'mvs'
    _write_mvs_scene(root)
    cfg = _cfg(tmp_path / 'unused', None, mvs_root=str(root), use_nerf_alpha=False)
    for mode in ('train', 'vali', 'test'):
        mine = get_dataset_class('mvs_shape')(cfg, mode)
        assert _rel(mine.files, tmp_path) == list(g['mvs/%s/files' % mode]) and mine.files
        _check_loads(mine, g, 'mvs/%s/' % mode)
