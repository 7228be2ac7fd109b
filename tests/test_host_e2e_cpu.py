"""Host logic of the drop-in scripts end to end on the CPU test double (tests/cpu_backend.py):
file formats, dataset -> batch -> Model.call glue, loss, optimizer bookkeeping, checkpoint
naming / resume, visualisation tree.  The same scenario runs on the real kernels in
tests/test_zz_gpu_scripts.py."""
import numpy as np
import pytest
import torch

import cpu_backend
import e2e_scenario
from nerfactor_b200 import config as nfconfig, synth


def test_scripts_end_to_end_on_test_double(tmp_path, monkeypatch):
    cpu_backend.install(monkeypatch)
    e2e_scenario.run(tmp_path, imh=8, light_h=2, n_samples=8, epochs=2, n_rays=32)


def test_model_call_glue_matches_oracle_on_test_double(monkeypatch):
    """Model.call's compaction / scatter / override glue vs the oracle's Model.call on a batch
    with background rays (the kernels themselves are replaced, so this isolates the host code)."""
    from oracle import stage_b, brdf as obrdf
    ctx = cpu_backend.install(monkeypatch)
    from nerfactor_b200.models.nerfactor_microfacet import Model
    lh, lw = 2, 8
    params = synth.make_stage_b_params(7, 'microfacet', light_hw=(lh, lw))
    m = Model(nfconfig.default_config('nerfactor_microfacet', light_h=lh), params=params, ctx=ctx)
    lxyz, lareas = obrdf.gen_light_xyz(lh, lw)
    m.set_lights(lxyz.reshape(-1, 3), lareas.reshape(-1))
    m.light_res = (lh, lw)
    batch = synth.make_stage_b_batch(11, 40, lh * lw, fg_frac=0.6)
    probes = synth.make_probes(3, 2, (lh, lw))
    for i, p in enumerate(probes):
        m.novel_probes['p%d' % i] = torch.as_tensor(p)
    pred, gt, lk, to_vis = m.call(batch, 'test', relight_probes=True, relight_olat=True,
                                  albedo_scales=np.array([0.5, 1., 2.], np.float32))
    om = stage_b.StageB(params, {'brdf': 'microfacet'}, lxyz=lxyz, lareas=lareas)
    olat = om.novel_olat((lh, lw))                      # the 16 one-hot env-maps, (i, j) order
    opred, _, _ = om.call(batch, 'test', relight_lights=list(probes) + olat,
                          albedo_scales=np.array([0.5, 1., 2.], np.float32))
    want = {k: opred[k].numpy() for k in ('rgb', 'normal', 'lvis', 'albedo', 'brdf')}
    want['rgb_probes'] = opred['rgb_relit'].numpy()[:, :2]
    want['rgb_olat'] = opred['rgb_relit'].numpy()[:, 2:]
    for k, b in want.items():
        a = pred[k].numpy()
        assert a.shape == b.shape, k
        assert np.abs(a - b).max() < 2e-5, (k, np.abs(a - b).max())
    bg = batch[5][:, 0] == 0
    assert bg.any() and np.all(pred['rgb'].numpy()[bg] == 0)           # nerfactor.py:268-293
    assert to_vis['pred_rgb'] is pred['rgb'] and set(lk) == {
        'mode', 'normal_jitter', 'lvis_jitter', 'brdf_prop_jitter', 'albedo_jitter'}
    with pytest.raises(ValueError):
        m.call(batch, 'predict')


def test_shape_model_call_and_loss_equal_reference_code(monkeypatch):
    """nerfactor_b200.models.shape.Model (host code; kernels replaced by the test double) against
    the REFERENCE'S shape.py Model.call + compute_loss run through the TensorFlow shim
    (tests/golden/ref_tfshim_shape.npz): predictions, jittered predictions, per-ray loss."""
    import os
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden',
                             'ref_tfshim_shape.npz'))
    ctx = cpu_backend.install(monkeypatch)
    from nerfactor_b200.models.shape import Model
    lh, n = int(g['light_h']), int(g['n_rays'])
    params = synth.make_stage_b_params(int(g['seed_params']), 'learned', light_hw=(lh, 2 * lh))
    cfg = nfconfig.default_config('shape', light_h=lh, normal_smooth_weight=0.01,
                                  lvis_smooth_weight=0.5)      # as in the generator
    m = Model(cfg, params=params, ctx=ctx, precision='fp32')
    batch = synth.make_stage_b_batch(int(g['seed_batch']), n, 2 * lh * lh)
    pred, gt, lk, _ = m.call(batch, 'train', xyz_noise=g['xyz_noise'])
    for k in ('normal', 'lvis'):
        assert np.abs(pred[k].numpy() - g['pred_' + k]).max() < 2e-6, k
    assert np.abs(lk['normal_jitter'].numpy() - g['normal_jitter']).max() < 2e-6
    # the jittered visibility: net at xyz + noise, light directions of the UN-jittered point
    # (shape.py:151, 170) -- `_pred_lvis_jitter_at`
    assert np.abs(lk['lvis_jitter'].numpy() - g['lvis_jitter']).max() < 2e-6
    # ... and its documented fallback for batches too big to materialise (directions then follow
    # the jittered point: lights at radius 100, jitter 0.01 -> below 1e-4)
    monkeypatch.setattr(Model, 'JITTER_EXACT_MAX_PAIRS', 0)
    _, _, lk_big, _ = m.call(batch, 'train', xyz_noise=g['xyz_noise'])
    d = np.abs(lk_big['lvis_jitter'].numpy() - g['lvis_jitter']).max()
    assert 0 < d < 1e-4
    loss = m.compute_loss(pred, gt, **lk)
    assert loss.shape == (n,) and np.abs(loss.numpy() - g['loss']).max() < 2e-6


@pytest.mark.parametrize('kind', ['microfacet'])
def test_nerfactor_model_call_equals_reference_code(monkeypatch, kind):
    """Same for the NeRFactor model's host glue (mask / compaction / scatter, overrides, probe and
    OLAT relighting, loss) against tests/golden/ref_tfshim_stage_b_microfacet.npz."""
    import os
    from importlib import import_module
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden',
                             'ref_tfshim_stage_b_%s.npz' % kind))
    ctx = cpu_backend.install(monkeypatch)
    Model = import_module('nerfactor_b200.models.nerfactor_microfacet').Model
    lh = int(g['light_h'])
    params = synth.make_stage_b_params(int(g['seed_params']), kind, light_hw=(lh, 2 * lh))
    m = Model(nfconfig.default_config('nerfactor_microfacet', light_h=lh), params=params, ctx=ctx,
              precision='fp32')
    batch = synth.make_stage_b_batch(int(g['seed_batch']), int(g['n_rays']), 2 * lh * lh)
    for i, p in enumerate(g['probes']):
        m.novel_probes['p%d' % i] = p
    pred, _, _, _ = m.call(batch, 'test', relight_probes=True, relight_olat=True)
    for k in ('rgb', 'normal', 'lvis', 'albedo', 'brdf', 'rgb_probes', 'rgb_olat'):
        assert np.abs(pred[k].numpy() - g['test_' + k]).max() < 5e-6, k
    pr, gt, lk, _ = m.call(batch, 'train', xyz_noise=g['xyz_noise'])
    for k in ('normal_jitter', 'lvis_jitter', 'albedo_jitter', 'brdf_prop_jitter'):
        assert np.abs(lk[k].numpy() - g['train_' + k]).max() < 2e-6, k
    loss = m.compute_loss(pr, gt, **lk)
    assert np.abs(loss.numpy() - g['train_loss']).max() < 1e-6
    pv, gtv, lkv, _ = m.call(batch, 'vali')
    assert np.abs(m.compute_loss(pv, gtv, **lkv).numpy() - g['vali_loss']).max() < 2e-6


@pytest.mark.parametrize('kind', ['microfacet', 'learned'])
def test_trainer_gradients_equal_reference_tape(monkeypatch, kind):
    """`Trainer.loss_and_grad` (trainvali.forward + autodiff.py: the differentiable host path of
    the train step, Dense kernels replaced by the test double) against the gradients the
    REFERENCE's train_step produced through the shim (tests/golden/ref_tfshim_train_grad_*.npz):
    per-ray loss and all 41 gradient tensors, frozen BRDF prior excluded."""
    import os
    from importlib import import_module
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden',
                             'ref_tfshim_train_grad_%s.npz' % kind))
    ctx = cpu_backend.install(monkeypatch)
    name = 'nerfactor_microfacet' if kind == 'microfacet' else 'nerfactor'
    Model = import_module('nerfactor_b200.models.' + name).Model
    from nerfactor_b200.trainvali import Trainer
    lh, n = int(g['light_h']), int(g['n_rays'])
    params = synth.make_stage_b_params(int(g['seed_params']), kind, light_hw=(lh, 2 * lh))
    m = Model(nfconfig.default_config(name, light_h=lh), params=params, ctx=ctx, precision='fp32')
    batch = synth.make_stage_b_batch(int(g['seed_batch']), n, 2 * lh * lh, fg_frac=1.0)
    tr = Trainer(m, precision='fp32')
    loss, grad = tr.loss_and_grad(batch, xyz_noise=g['xyz_noise'])
    assert np.allclose(loss.numpy(), g['per_example_loss'], atol=2e-6, rtol=1e-5)
    gv = tr.views(grad)
    keys = [k for k in g.files if k.startswith('grad/')]
    assert len(keys) == len(gv) == 41
    for k in keys:
        parts = k.split('/')
        key = ('light', 0, 'light') if parts[1] == 'light' else (parts[1], int(parts[2]), parts[3])
        want = g[k]
        got = gv[key].numpy().reshape(want.shape)
        assert np.abs(got - want).max() <= 2e-5 * max(np.abs(want).max(), 1e-8), k


import os as _os

_GOLDEN = _os.path.join(_os.path.dirname(_os.path.abspath(__file__)), 'golden', 'ref_host_code.npz')


@pytest.mark.parametrize('ini', ['nerfactor.ini', 'nerfactor_microfacet.ini', 'nerfactor_mvs.ini',
                                 'nerfactor_no_geom_opt.ini', 'nerfactor_no_geom_pretrain.ini',
                                 'nerfactor_no_smooth.ini', 'shape.ini', 'shape_mvs.ini',
                                 'nerf.ini', 'brdf.ini'])
def test_every_shipped_reference_config_drives_the_models(monkeypatch, tmp_path, ini):
    """The reference's own .ini files (their keys and values as stored by
    tests/golden/make_golden_host.py, written back to an .ini and read as such, site paths
    replaced): model construction, a forward pass and the loss on the CPU test double -- every key
    the models read is present or has the reference's fallback."""
    import json
    from configparser import ConfigParser
    import numpy as _np
    from nerfactor_b200 import models
    from nerfactor_b200.brdf.renderer import gen_light_xyz
    from nerfactor_b200.util import io as ioutil
    ctx = cpu_backend.install(monkeypatch)
    stored = ConfigParser()
    stored.read_dict(json.loads(str(np.load(_GOLDEN)['configs/' + ini])))
    with open(str(tmp_path / ini), 'w') as h:
        stored.write(h)
    cfg = ioutil.read_config(str(tmp_path / ini))
    lh = 2
    for k in ('data_root', 'data_nerf_root', 'outroot', 'test_envmap_dir'):
        if cfg.has_option('DEFAULT', k):
            cfg.set('DEFAULT', k, str(tmp_path / k))
    for k in ('shape_model_ckpt', 'brdf_model_ckpt'):
        if cfg.has_option('DEFAULT', k):
            cfg.set('DEFAULT', k, str(tmp_path / k / 'lr' / 'checkpoints' / 'ckpt-1'))
    if cfg.has_option('DEFAULT', 'light_h'):
        cfg.set('DEFAULT', 'light_h', str(lh))
    if cfg.has_option('DEFAULT', 'mvs_root'):
        _os.makedirs(str(tmp_path / 'mvs'))
        lxyz, lareas = gen_light_xyz(lh, 2 * lh)
        _np.savez(str(tmp_path / 'mvs' / 'lights.npz'), lxyzs=lxyz, lareas=lareas)
        cfg.set('DEFAULT', 'mvs_root', str(tmp_path / 'mvs'))
    name = cfg.get('DEFAULT', 'model')
    kw = {}
    if name.startswith('nerfactor'):
        # the checkpoints the .ini names do not exist here: like the reference, construction fails
        # hard on that (a typo must not give a random frozen prior) ...
        if name == 'nerfactor' or cfg.get('DEFAULT', 'shape_mode') in ('frozen', 'finetune'):
            with pytest.raises(FileNotFoundError):
                models.get_model_class(name)(cfg, ctx=ctx, precision='fp32')
        kw['allow_uninitialised_prior'] = True       # ... unless explicitly opted out
    model = models.get_model_class(name)(cfg, ctx=ctx, precision='fp32', **kw)
    model.register_trainable()
    assert model.trainable_registered
    if name == 'brdf':
        assert model.latent_code.z.shape[1] == 3 and cfg.get('DEFAULT', 'loss_transform') == 'log'
        return
    if name == 'nerf':
        assert set(model.net) >= {'coarse_enc', 'fine_enc', 'coarse_sigma_out', 'fine_rgb_out'}
        return
    if name == 'nerfactor':                 # the learned lobe has no test double: microfacet-free
        assert model.brdf_model is not None and model.z_dim == 3
        return
    batch = synth.make_stage_b_batch(1, 12, 2 * lh * lh)
    pred, gt, lk, to_vis = model.call(batch, 'train')
    loss = model.compute_loss(pred, gt, **lk)
    assert tuple(loss.shape) == (12,) and bool(torch.isfinite(loss).all())


def test_nerf_trainer_equals_reference_train_step(monkeypatch):
    """`NerfTrainer` (stratified + hierarchical sampling, both networks, density noise, L2 on both
    renderings; Dense kernels replaced by the test double) against the REFERENCE's NeRF train
    step run through the shim with all four random draws recorded
    (tests/golden/ref_tfshim_nerf_train_grad.npz): renderings, per-ray loss, 48 gradient tensors
    (big kernels are stored as fp16 in the fixture)."""
    g = np.load(_os.path.join(_os.path.dirname(_os.path.abspath(__file__)), 'golden',
                              'ref_tfshim_nerf_train_grad.npz'))
    ctx = cpu_backend.install(monkeypatch)
    from nerfactor_b200.models.nerf import Model
    from nerfactor_b200.trainvali import make_trainer, NerfTrainer
    cfg = nfconfig.default_config('nerf', n_samples_coarse=int(g['n_c']),
                                  n_samples_fine=int(g['n_f']), perturb=True,
                                  noise_std=float(g['noise_std']))
    m = Model(cfg, params=synth.make_nerf_params(int(g['seed_nerf'])), ctx=ctx, precision='fp32')
    tr = make_trainer(m, precision='fp32')
    assert isinstance(tr, NerfTrainer)
    batch = (None, None, g['rayo'], g['rayd'], g['rgb'])
    draws = dict(perturb_u=g['perturb_u'], fine_u=g['fine_u'],
                 sigma_noise=(g['noise_coarse'], g['noise_fine']))
    with torch.no_grad():
        loss_f, pred = tr.forward(tr.flat, batch, 'train', **draws)
    assert np.abs(pred['coarse'].numpy() - g['pred_coarse']).max() < 2e-6
    # the fine samples go through a discontinuous inverse-CDF lookup and a 2^9-frequency
    # encoding: 1-ulp differences of the sample positions show up at the 1e-5 level on single rays
    assert np.abs(pred['fine'].numpy() - g['pred_fine']).max() < 5e-5
    assert np.median(np.abs(pred['fine'].numpy() - g['pred_fine'])) < 1e-6
    assert np.median(np.abs(tr.last_z_all.numpy() - g['z_all'])) < 1e-6
    # gradients with the reference's recorded samples replayed (no gradient flows through them)
    replay = dict(draws, z_all=g['z_all'])
    with torch.no_grad():
        _, pred = tr.forward(tr.flat, batch, 'train', **replay)
    assert np.abs(pred['fine'].numpy() - g['pred_fine']).max() < 2e-6
    loss, grad = tr.loss_and_grad(batch, **replay)
    assert np.allclose(loss.numpy(), g['per_example_loss'], atol=2e-6, rtol=1e-5)
    gv = tr.views(grad)
    keys = [k for k in g.files if k.startswith('grad/')]
    assert len(keys) == len(gv) == 48
    for k in keys:
        _, net, li, kind = k.split('/')
        want = g[k].astype(np.float32)
        got = gv[(net, int(li), kind)].numpy()
        # fp16-stored big kernels: 2^-11 of the element; everything else tight
        rel = 6e-4 if g[k].dtype == np.float16 else 5e-5
        tol = rel * max(np.abs(want).max(), 1e-8)
        assert np.abs(got - want).max() <= tol, k
    # one optimizer step moves the weights and a few more reduce the loss on this batch
    l0 = float(tr.train_step(batch, **draws))
    for _ in range(5):
        l1 = float(tr.train_step(batch, **draws))
    assert l1 < l0


def test_nerf_training_script_then_stage_a(tmp_path, monkeypatch):
    """The stage before Stage A through the scripts: `trainvali --config <nerf .ini>` trains the
    NeRF (NerfTrainer), checkpoints under the reference's variable names and writes the validation
    visualisation; `geometry_from_nerf --trained_nerf <that run>` then finds the latest checkpoint
    and its .ini and produces the geometry buffers.  CPU test double, FP32 layered NeRF path."""
    cpu_backend.install(monkeypatch)
    from nerfactor_b200 import trainvali, geometry_from_nerf as gfn
    from nerfactor_b200.util import io as ioutil, tfckpt
    data = str(tmp_path / 'data')
    ids = synth.write_scene(data, imh=8, imw=8, n_train=2, n_val=1, n_test=1)
    cfg = nfconfig.default_config(
        'nerf', data_root=data, imh=6, n_samples_coarse=6, n_samples_fine=6, n_rays_per_step=24,
        epochs=2, ckpt_period=1, vali_period=2, vali_batches=1, outroot=str(tmp_path / 'out'))
    ini = str(tmp_path / 'nerf.ini')
    ioutil.write_config(cfg, ini)
    outdir = trainvali.main(['--config', ini, '--precision', 'fp32'])
    ckpt = ioutil.latest_checkpoint(_os.path.join(outdir, 'checkpoints'))
    assert ckpt.endswith('ckpt-2')
    names = tfckpt.read_checkpoint(ckpt)
    assert 'net/net_coarse_enc_layer0/kernel/.ATTRIBUTES/VARIABLE_VALUE' in names
    assert 'net/net_fine_rgb_out_layer1/bias/.OPTIMIZER_SLOT/optimizer/vhat/.ATTRIBUTES/VARIABLE_VALUE' in names
    vdir = _os.path.join(outdir, 'vis_vali', 'epoch000000002')
    assert _os.path.exists(_os.path.join(vdir, 'all.html'))
    assert _os.path.exists(_os.path.join(vdir, 'batch000000000', 'fine-vs-gt_rgb.apng'))
    # nerf_test.py: the test cameras rendered with the trained NeRF, compiled into a video
    from nerfactor_b200 import nerf_test
    vroot, view_at = nerf_test.main(['--ckpt', ckpt, '--precision', 'fp32'])
    assert _os.path.exists(_os.path.join(vroot, 'batch000000000', 'fine_rgb.png'))
    assert ioutil.read_json(_os.path.join(vroot, 'batch000000000', 'metadata.json')) == {
        'id': 'test_000'}
    assert view_at.endswith('ckpt-2.mp4') and _os.path.getsize(view_at) > 0
    surf = str(tmp_path / 'surf')
    done = gfn.main(['--trained_nerf', outdir, '--out_root', surf, '--light_h', '2',
                     '--precision', 'fp32'])
    assert sorted(done) == sorted(ids)
    assert np.load(_os.path.join(surf, 'test_000', 'lvis.npy')).shape == (6, 6, 8)


def test_brdf_prior_trainer_equals_reference_train_step(monkeypatch, tmp_path):
    """`BrdfTrainer` + models/brdf.py `call` / `compute_loss` (BRDF prior: softplus MLP on
    [z | embed(rusink)] and the reciprocal coordinates, log-space L2, latent codes optimised with
    the network) against the reference's train step through the shim
    (tests/golden/ref_tfshim_brdf_train_grad.npz): predictions, per-row loss, the 10 Dense
    gradients and the latent-code gradient (non-zero only in the step's material row)."""
    g = np.load(_os.path.join(_os.path.dirname(_os.path.abspath(__file__)), 'golden',
                              'ref_tfshim_brdf_train_grad.npz'))
    ctx = cpu_backend.install(monkeypatch)
    from nerfactor_b200.models.brdf import Model
    from nerfactor_b200.trainvali import make_trainer, BrdfTrainer
    names = [str(x) for x in g['names']]
    params = synth.make_stage_b_params(5, 'learned')
    m = Model(nfconfig.default_config('brdf', lr=1e-3), params=params, brdf_names=names)
    m.latent_code.z = g['z0']
    i = int(g['i'])
    batch = (names[i], i, 16, 128, 1, g['rusink'], g['refl'])
    pred, gt, lk, to_vis = m.call(batch, 'vali')
    assert np.abs(pred['brdf'].numpy() - g['pred_brdf']).max() < 1e-6
    assert np.abs(pred['brdf_reci'].numpy() - g['pred_brdf_reci']).max() < 1e-6
    loss = m.compute_loss(pred, gt, keep_batch=True, **lk)
    assert np.allclose(loss.numpy(), g['per_example_loss'], atol=1e-6, rtol=1e-5)
    tr = make_trainer(m)
    assert isinstance(tr, BrdfTrainer)
    loss, grad = tr.loss_and_grad(batch)
    assert np.allclose(loss.numpy(), g['per_example_loss'], atol=1e-6, rtol=1e-5)
    gv = tr.views(grad)
    keys = [k for k in g.files if k.startswith('grad/')]
    assert len(keys) == len(gv) == 11
    for k in keys:
        parts = k.split('/')
        key = ('z', 0, 'z') if parts[1] == 'z' else (parts[1], int(parts[2]), parts[3])
        want = g[k]
        assert np.abs(gv[key].numpy() - want).max() <= 2e-5 * max(np.abs(want).max(), 1e-8), k
    gz = gv[('z', 0, 'z')].numpy()
    assert np.abs(gz[i]).max() > 0 and np.abs(np.delete(gz, i, axis=0)).max() == 0
    l0 = float(tr.train_step(batch))
    for _ in range(30):
        l1 = float(tr.train_step(batch))
    assert l1 < l0
    tr.sync_to_model()
    assert not np.array_equal(m.latent_code.z[i], g['z0'][i])       # the code moved ...
    assert np.array_equal(np.delete(m.latent_code.z, i, 0), np.delete(g['z0'], i, 0))  # only it
    # novel identity at test time: interpolated latent code (brdf.py:89-97)
    pi, _, _, _ = m.call(('000000_0.250000_%s_0.750000_%s' % (names[0], names[2]), -1, 16, 128, 1,
                          g['rusink'], np.zeros_like(g['refl'])), 'test')
    z_mix = 0.25 * m.latent_code.z[0] + 0.75 * m.latent_code.z[2]
    m2 = Model(nfconfig.default_config('brdf'), params=params, brdf_names=['mix'])
    for k in ('brdf_mlp', 'brdf_out'):
        m2.net[k].load({'layers': m.net[k].weights()})
    m2.latent_code.z = z_mix[None]
    p2, _, _, _ = m2.call(('mix', 0, 16, 128, 1, g['rusink'], g['refl']), 'vali')
    assert np.abs(pi['brdf'].numpy() - p2['brdf'].numpy()).max() < 1e-6


def test_brdf_prior_training_script_feeds_nerfactor(tmp_path, monkeypatch):
    """`trainvali --config <brdf .ini>` on synthetic MERL-style tables: checkpoints carry the MLP
    and the latent codes under the reference's names (`net/latent_code/_z`), and a NeRFactor model
    whose config names that checkpoint restores the prior (network, codes, material names) the
    way nerfactor.py:36-60 does."""
    cpu_backend.install(monkeypatch)
    from nerfactor_b200 import trainvali
    from nerfactor_b200.util import io as ioutil, tfckpt
    from nerfactor_b200.models.nerfactor import Model as NeRFactor
    data = str(tmp_path / 'merl')
    names = synth.write_merl_npz(data, n_rows=96)
    cfg = nfconfig.default_config('brdf', data_root=data, n_rays_per_step=32, epochs=2,
                                  ckpt_period=1, vali_period=2, vali_batches=1, lr=1e-3,
                                  outroot=str(tmp_path / 'out'))
    ini = str(tmp_path / 'brdf.ini')
    ioutil.write_config(cfg, ini)
    outdir = trainvali.main(['--config', ini])
    ckpt = ioutil.latest_checkpoint(_os.path.join(outdir, 'checkpoints'))
    t = tfckpt.read_checkpoint(ckpt)
    z = t['net/latent_code/_z/.ATTRIBUTES/VARIABLE_VALUE']
    assert z.shape == (3, 3) and 'net/net_brdf_mlp_layer0/kernel/.ATTRIBUTES/VARIABLE_VALUE' in t
    assert int(t['optimizer/iter/.ATTRIBUTES/VARIABLE_VALUE']) == 2 * len(names)
    assert _os.path.exists(_os.path.join(outdir, 'vis_vali', 'epoch000000002', 'batch000000000',
                                         'log10_brdf.npy'))
    # explore_brdf_space.py: every seen material + the interpolated identities on the test coords
    from nerfactor_b200 import explore_brdf_space
    vroot, n_done = explore_brdf_space.main(['--ckpt', ckpt])
    assert n_done == 3 + 2 * 11                      # 3 materials, 2 pairs x 11 blends
    assert ioutil.read_json(_os.path.join(vroot, 'batch000000000', 'metadata.json'))['id'] == \
        sorted(names)[0]
    lb = np.load(_os.path.join(vroot, 'batch000000004', 'log10_brdf.npy'))
    assert lb.shape[1] == 2 and np.isfinite(lb).all()
    assert explore_brdf_space.main(['--ckpt', ckpt])[1] == 0          # all done: skipped
    ncfg = nfconfig.default_config('nerfactor', light_h=2, brdf_model_ckpt=ckpt,
                                   shape_mode='scratch')
    m = NeRFactor(ncfg)
    assert m.brdf_model.brdf_names == sorted(names)
    assert np.array_equal(np.asarray(m.brdf_model.latent_code.z), z)
    w_ckpt = t['net/net_brdf_out_layer0/kernel/.ATTRIBUTES/VARIABLE_VALUE']
    assert np.array_equal(m.brdf_model.net['brdf_out'].weights()[0][0], w_ckpt)
