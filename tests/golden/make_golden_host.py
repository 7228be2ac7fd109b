"""Runs the reference's host-side code (loaders, buffer writers, image helpers, `vis_batch`,
`process_view`, the turbo table, the shipped .ini files) on the same seeded inputs the tests
build, and writes what it returned to tests/golden/ref_host_code.npz.

Needs a checkout of the reference next to the TensorFlow shim (see make_golden_tfshim.py):

    python tests/golden/make_golden_host.py

The tests in test_datasets_cpu.py, test_scripts_cpu.py and test_host_e2e_cpu.py compare the code
here with these arrays; they build their inputs with the same helpers this script imports.
"""
import json
import os
import sys
import tempfile
from configparser import ConfigParser

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
TESTS = os.path.dirname(HERE)
sys.path.insert(0, HERE)
import make_golden_tfshim as gen  # noqa: E402  (sys.path: shim, reference, repository root)
sys.path.insert(0, TESTS)
import test_datasets_cpu as tdc  # noqa: E402  (the tests' own input builders)

import torch  # noqa: E402
from nerfactor_b200 import synth  # noqa: E402

REF = gen.REF
OUT = {}


def _load_all(ds, files, pre):
    for i, path in enumerate(files):
        r = ds._load_data(path)
        OUT[pre + '%d/id' % i] = np.array(r[0])
        OUT[pre + '%d/n' % i] = np.array(len(r) - 1)
        for j, a in enumerate(r[1:]):
            OUT[pre + '%d/%d' % (i, j)] = np.asarray(a)


def configs():
    cdir = os.path.join(REF, 'nerfactor', 'config')
    for ini in sorted(f for f in os.listdir(cdir) if f.endswith('.ini')):
        cfg = ConfigParser()
        with open(os.path.join(cdir, ini)) as h:
            cfg.read_file(h)
        d = {s: dict(cfg.items(s, raw=True)) if s != 'DEFAULT' else dict(cfg.defaults())
             for s in ['DEFAULT'] + cfg.sections()}
        OUT['configs/' + ini] = np.array(json.dumps(d, sort_keys=True))


def helpers(tmp):
    from third_party.xiuminglib import xiuminglib as xm
    rng = np.random.default_rng(3)
    a = rng.random((20, 30, 3))
    u8 = (a * 255).astype(np.uint8)
    hdr = (rng.random((8, 16, 3)) * 30).astype(np.float32)
    OUT['helpers/normalize_uint'] = xm.img.normalize_uint(u8)
    OUT['helpers/denormalize_float'] = xm.img.denormalize_float(a)
    OUT['helpers/tonemap'] = xm.img.tonemap(hdr, gamma=4)
    OUT['helpers/resize'] = xm.img.resize(a, new_h=10)
    OUT['helpers/alpha_blend'] = xm.img.alpha_blend(a, a[:, :, 0])
    OUT['helpers/psnr'] = np.array(xm.metric.PSNR('uint8')(u8, u8[::-1].copy()))
    open(os.path.join(tmp, 'b.txt'), 'w').close()
    open(os.path.join(tmp, 'a.txt'), 'w').close()
    OUT['helpers/sortglob'] = np.array([os.path.relpath(p, tmp) for p in
                                        xm.os.sortglob(tmp, '*', ext='txt')])


def loaders(tmp):
    from nerfactor.datasets.nerf import Dataset as RefNerf
    from nerfactor.datasets.nerf_shape import Dataset as RefShape
    root, nroot = os.path.join(tmp, 'scene'), os.path.join(tmp, 'surf')
    synth.write_scene(root, imh=16, imw=16, n_train=2, n_val=1, n_test=1, nerf_root=nroot,
                      n_lights=8)
    rel = lambda fs: [os.path.relpath(f, tmp) for f in fs]
    for imh in (16, 8):
        cfg = tdc._cfg(root, nroot, use_nerf_alpha=False, no_batch=True)
        cfg.set('DEFAULT', 'imh', str(imh))
        for mode in ('train', 'vali', 'test'):
            ref = RefShape.__new__(RefShape)            # skip tf.data-related __init__ parts
            ref.config, ref.mode, ref.debug = cfg, mode, False
            ref.meta2buf, ref.meta2img, ref.sps = {}, {}, 1
            ref.files = ref._glob()
            _load_all(ref, ref.files, 'loaders/shape/%d/%s/' % (imh, mode))
            OUT['loaders/shape/%d/%s/files' % (imh, mode)] = np.array(rel(ref.files))
        for ndc in ('False', 'True'):
            cfg.set('DEFAULT', 'ndc', ndc)
            for sps in (1, 2):
                rr = RefNerf.__new__(RefNerf)
                rr.config, rr.sps = cfg, sps
                c2w = synth.look_at_c2w(3.0, 40.0, 25.0)
                for k, a in enumerate(rr._gen_rays(c2w, 0.7, 6, 9)):
                    OUT['loaders/rays/%d/%s/%d/%d' % (imh, ndc, sps, k)] = np.asarray(a)
        cfg.set('DEFAULT', 'ndc', 'False')
        refn = RefNerf.__new__(RefNerf)
        refn.config, refn.mode, refn.debug, refn.meta2img, refn.sps = cfg, 'train', False, {}, 1
        refn.files = refn._glob()
        _load_all(refn, refn.files, 'loaders/nerf/%d/' % imh)
        OUT['loaders/nerf/%d/files' % imh] = np.array(rel(refn.files))


def writers(tmp):
    from nerfactor.util import geom as refgeom
    from third_party.xiuminglib import xiuminglib as xm
    from nerfactor_b200.util import img as imgutil
    rng = np.random.default_rng(0)
    alpha = rng.random((9, 7)).astype(np.float32)
    xyz = (rng.standard_normal((9, 7, 3)) * alpha[..., None]).astype(np.float32)
    nrm = rng.standard_normal((9, 7, 3)).astype(np.float32)
    nrm /= np.linalg.norm(nrm, axis=2, keepdims=True)
    lvis = rng.random((9, 7, 8)).astype(np.float32)
    rd = os.path.join(tmp, 'ref')
    os.makedirs(rd)
    refgeom.write_alpha(alpha, rd)
    refgeom.write_xyz(xyz, rd)
    refgeom.write_normal(nrm, rd)
    np.save(os.path.join(rd, 'lvis.npy'), lvis)             # geom.py:30-32
    xm.io.img.write_arr(np.mean(lvis, axis=2), os.path.join(rd, 'lvis.png'))   # geom.py:34-36
    for f in ('xyz.npy', 'normal.npy', 'lvis.npy'):
        OUT['writers/' + f] = np.frombuffer(open(os.path.join(rd, f), 'rb').read(), np.uint8)
    for f in ('alpha.png', 'xyz.png', 'normal.png', 'lvis.png'):
        OUT['writers/' + f] = imgutil.read(os.path.join(rd, f))


def mvs(tmp):
    from nerfactor.datasets.mvs_shape import Dataset as RefMvs
    root = os.path.join(tmp, 'mvs')
    tdc._write_mvs_scene(root)
    cfg = tdc._cfg(os.path.join(tmp, 'unused'), None, mvs_root=root, use_nerf_alpha=False)
    for mode in ('train', 'vali', 'test'):
        ref = RefMvs.__new__(RefMvs)
        ref.config, ref.mode, ref.debug, ref.meta2buf, ref.meta2img, ref.sps = \
            cfg, mode, False, {}, {}, 1
        ref.files = ref._glob()
        _load_all(ref, ref.files, 'mvs/%s/' % mode)
        OUT['mvs/%s/files' % mode] = np.array([os.path.relpath(f, tmp) for f in ref.files])


def turbo():
    from third_party.turbo_colormap import turbo_colormap_data, interpolate_or_clip
    xs = np.linspace(0, 1, 501)
    OUT['turbo/table'] = np.array([interpolate_or_clip(turbo_colormap_data, float(x)) for x in xs])
    OUT['turbo/below'] = np.array(interpolate_or_clip(turbo_colormap_data, -0.1))
    OUT['turbo/above'] = np.array(interpolate_or_clip(turbo_colormap_data, 1.1))


def vis_batch(tmp):
    """The reference's NeRFactor model: call (test mode, OLAT + probes) -> to_vis -> vis_batch."""
    from collections import OrderedDict
    from nerfactor.util import light as reflight
    from nerfactor_b200.util import img as imgutil
    lh, h, w = 2, 6, 5
    model, cfg, params = gen.build_stage_b('microfacet', lh, os.path.join(tmp, 'cfg'), 7)
    L = 2 * lh * lh
    batch_np = list(synth.make_stage_b_batch(11, h * w, L))
    batch_np[1] = np.tile(np.array([[h, w]], np.int32), (h * w, 1))

    class _Id:                                   # an eager string tensor: x[0].numpy() -> bytes
        def __getitem__(self, i):
            return self

        def numpy(self):
            return b'test_007'
    batch = tuple(_Id() if i == 0 else gen.t32(x) if i > 1 else torch.as_tensor(x)
                  for i, x in enumerate(batch_np))
    probes = synth.make_probes(5, 2, (lh, 2 * lh))
    model.novel_probes = OrderedDict(('p%d' % i, gen.t32(p)) for i, p in enumerate(probes))
    model.novel_probes_uint = {k: reflight.vis_light(v, h=model.embed_light_h)
                               for k, v in model.novel_probes.items()}
    _, _, _, to_vis = model.call(batch, mode='test', relight_olat=True, relight_probes=True)
    for k, v in to_vis.items():
        if isinstance(v, torch.Tensor):
            OUT['vis/in/' + k] = v.detach().numpy().copy()
        elif k not in ('id', 'hw'):
            raise TypeError('to_vis[%r]: %r' % (k, type(v)))
    rdir = os.path.join(tmp, 'ref')
    model.vis_batch(to_vis, rdir, mode='test', olat_vis=True)
    files = sorted(os.listdir(rdir))
    OUT['vis/files'] = np.array(files)
    OUT['vis/metadata'] = np.array(open(os.path.join(rdir, 'metadata.json')).read())
    for f in files:
        if f.endswith('.png'):
            OUT['vis/png/' + f] = imgutil.read(os.path.join(rdir, f))


def process_view(tmp):
    """geometry_from_nerf.process_view of the reference on a 5 x 6 view of a random-init NeRF."""
    from nerfactor import geometry_from_nerf as refgfn
    from nerfactor.models.nerf import Model as RefNerf
    from third_party.xiuminglib import xiuminglib as xm
    from nerfactor_b200.util import img as imgutil
    from oracle import stage_a
    xm.vis.video.make_video = lambda *a, **k: None          # lvis.mp4: visualisation only
    lh, h, w = 2, 5, 6
    rdir = os.path.join(tmp, 'ref')
    if not refgfn.FLAGS.is_parsed():
        refgfn.FLAGS(['t'])
    refgfn.FLAGS.light_h, refgfn.FLAGS.out_root = lh, rdir
    refgfn.FLAGS.occu_thres, refgfn.FLAGS.spp = 0.9, 1
    cfg = gen.read_ini('nerf.ini', n_samples_coarse=-48, n_samples_fine=8, data_root=tmp,
                       outroot=tmp)
    ref_model = RefNerf(cfg)
    gen.set_weights(ref_model.net, synth.make_nerf_params(3))
    rayo, rayd = stage_a.gen_rays(synth.look_at_c2w(), synth.CAM_ANGLE_X, h, w)
    rayo, rayd = rayo.reshape(-1, 3), rayd.reshape(-1, 3)

    class _Id:
        def __getitem__(self, i):
            return self

        def numpy(self):
            return b'train_003'
    batch = (_Id(), torch.tensor([[h, w]] * (h * w), dtype=torch.int32), gen.t32(rayo),
             gen.t32(rayd), None)
    refgfn.process_view(cfg, ref_model, batch)
    vd = os.path.join(rdir, 'train_003')
    from nerfactor_b200.util import geom_io
    assert geom_io.view_done(vd)
    OUT['process_view/alpha.png'] = imgutil.read(os.path.join(vd, 'alpha.png'))
    for f in ('xyz.npy', 'normal.npy', 'lvis.npy'):
        OUT['process_view/' + f] = np.load(os.path.join(vd, f))


if __name__ == '__main__':
    configs()
    turbo()
    for fn in (helpers, loaders, writers, mvs, vis_batch, process_view):
        with tempfile.TemporaryDirectory() as tmp:
            fn(tmp)
    path = os.path.join(HERE, 'ref_host_code.npz')
    np.savez_compressed(path, **OUT)
    print(path, os.path.getsize(path), 'bytes,', len(OUT), 'arrays')
