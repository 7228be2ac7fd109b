"""Mirror of the train / validation step of nerfactor/trainvali.py (:110-127 optimizer,
:273-295 distributed_train_step, :301-317 vali step) for the shape and NeRFactor models.

    trainer = Trainer(model, config)          # model: nerfactor_b200.models.{shape,nerfactor,...}
    loss = trainer.train_step(batch)          # forward (train mode) + backward + AMSGrad
    trainer.sync_to_model()                   # push weights back for the inference kernels

Data parallelism (trainvali.py:259-295, MirroredStrategy): one process per GPU; each rank
gets its own rays, the per-ray loss is divided by the GLOBAL batch size
(tf.nn.compute_average_loss, :282-283) and the flat gradient buffer is summed with ONE
NCCL all-reduce before the optimizer step.
"""

import numpy as np
import torch

from . import _lib
from . import autodiff as ad
from .models.shape import to_device


class Trainer:
    def __init__(self, model, config=None, world_size=1, rank=0, precision=None):
        """precision: arithmetic of the Dense layers -- 'fp32' (CUDA cores), 'bf16' or 'f16'
        (tcgen05: 16-bit operands, fp32 accumulation, fp32 master weights / optimizer state).
        Default: 'fp32' for an fp32 model, else 'bf16' (BASELINE configs[3])."""
        self.precision = precision or ('fp32' if model.precision == 'fp32' else 'bf16')
        self.model = model
        self.ctx = model.ctx
        self.device = model.device
        cfg = config or model.config
        self.lr0 = cfg.getfloat('DEFAULT', 'lr', fallback=5e-3)
        self.lr_decay_steps = cfg.getint('DEFAULT', 'lr_decay_steps', fallback=-1)
        self.lr_decay_rate = cfg.getfloat('DEFAULT', 'lr_decay_rate', fallback=0.1)
        self.world_size, self.rank = world_size, rank
        self.iterations = 0
        # ---- flat parameter buffer: every trainable Dense kernel / bias, then the light
        self.names, shapes = [], []
        for net_name, net in model.net.items():
            for li, layer in enumerate(net.layers):
                if layer.trainable:
                    self.names += [(net_name, li, 'kernel'), (net_name, li, 'bias')]
                    shapes += [layer.kernel.shape, layer.bias.shape]
        # trainable tensors that are not Dense layers: the light probe (nerfactor.py:367-375), the
        # latent codes of the BRDF prior (networks/layers.py:24-45)
        self.has_light = hasattr(model, '_light')
        extras = {}
        if self.has_light:
            extras['light'] = model._light
        if hasattr(model, 'latent_code'):
            extras['z'] = torch.as_tensor(np.asarray(model.latent_code._z, np.float32))
        for kind, t in extras.items():
            self.names.append((kind, 0, kind))
            shapes.append(tuple(t.shape))
        sizes = [int(np.prod(s)) for s in shapes]
        # every view starts on a 16-byte boundary (the kernels stream weights with cp.async 16)
        padded = [(n + 3) // 4 * 4 for n in sizes]
        self.offsets = np.concatenate(([0], np.cumsum(padded))).astype(np.int64)
        total = int(self.offsets[-1])
        self.flat = torch.zeros(total, device=self.device)
        for (net_name, li, kind), off, shp in zip(self.names, self.offsets[:-1], shapes):
            if kind in extras:
                src = extras[kind]
            else:
                layer = model.net[net_name].layers[li]
                src = torch.as_tensor(getattr(layer, kind))
            self.flat[off:off + src.numel()] = src.reshape(-1).to(self.device)
        self.shapes = shapes
        self.m = torch.zeros_like(self.flat)
        self.v = torch.zeros_like(self.flat)
        self.vhat = torch.zeros_like(self.flat)
        # frozen layers (trainable = False) and the frozen BRDF prior (nerfactor.py:58-60): device copies
        self._frozen = {}
        for net_name, net in model.net.items():
            for li, layer in enumerate(net.layers):
                if not layer.trainable:
                    self._frozen[(net_name, li)] = (to_device(layer.kernel, self.device),
                                                    to_device(layer.bias, self.device))
        self._graphs = {}
        self.brdf_layers = None
        if getattr(model, 'brdf_model', None) is not None:
            bm = model.brdf_model
            self.brdf_layers = [(to_device(w, self.device), to_device(b, self.device))
                                for w, b in bm.net['brdf_mlp'].weights() + bm.net['brdf_out'].weights()]

    # ------------------------------------------------------------------ params
    def views(self, flat=None):
        """name -> tensor views of the flat buffer (autograd leaf = the flat buffer)."""
        flat = self.flat if flat is None else flat
        out = {}
        for (net_name, li, kind), off, shp in zip(self.names, self.offsets[:-1], self.shapes):
            n = int(np.prod(shp))
            out[(net_name, li, kind)] = flat[off:off + n].view(*shp)
        return out

    def net_layers(self, views, name):
        """[(W, b), ...] of trunk + head `name` ('normal', 'lvis', 'albedo', 'brdf_z')."""
        layers = []
        for part in ('_mlp', '_out'):
            net = self.model.net[name + part]
            for li, layer in enumerate(net.layers):
                key = (name + part, li, 'kernel')
                if key in views:
                    layers.append((views[key], views[(name + part, li, 'bias')]))
                else:      # frozen layer
                    layers.append(self._frozen[(name + part, li)])
        trunk = self.model.net[name + '_mlp']
        head = self.model.net[name + '_out']
        acts = [l.activation for l in trunk.layers] + [l.activation for l in head.layers]
        return layers, acts, trunk.skip_at

    def sync_to_model(self):
        """Writes the trained weights back into model.net / model._light (re-packs lazily)."""
        v = self.views()
        for (net_name, li, kind), t in v.items():
            if kind == 'light':
                self.model._light = t.detach().clone()
            elif kind == 'z':
                self.model.latent_code.z = t.detach().cpu().numpy().copy()
            else:
                layer = self.model.net[net_name].layers[li]
                arr = t.detach().cpu().numpy().copy()
                if kind == 'kernel':
                    layer.kernel = arr
                else:
                    layer.bias = arr
        self.model.weights_changed()

    def learning_rate(self):
        """ExponentialDecay(lr, decay_steps, decay_rate), continuous -- only when
        lr_decay_steps > 0; otherwise (the reference's fallback -1) a constant rate
        (trainvali.py:111-117)."""
        if self.lr_decay_steps <= 0:
            return self.lr0
        return self.lr0 * self.lr_decay_rate ** (self.iterations / self.lr_decay_steps)

    # ------------------------------------------------------------------ forward
    def _point(self, views, name, pts):
        layers, acts, skip = self.net_layers(views, name)
        e = ad.embed(self.model.xyz_scale * pts, self.model.embedder['xyz'].n_freqs)
        return ad.mlp_apply(e, layers, acts, skip, self.precision)

    def _lvis(self, views, pts, surf2l, pts_dir=None):
        """shape.py:213-237 on materialised rows.  Neither the surface points nor the light
        directions carry gradients, so the [n L, 90] input rows ([embed(pts) | embed(surf2l)],
        surf2l = directions of `pts_dir`: the un-jittered point for the jittered evaluation,
        shape.py:170) are built by one kernel (nf_lvis_inputs_fwd) instead of ~30 torch ops."""
        layers, acts, skip = self.net_layers(views, 'lvis')
        n, L = surf2l.shape[0], surf2l.shape[1]
        m = self.model
        if pts.is_cuda and not pts.requires_grad:
            e, width = _lib.lvis_inputs_fwd(
                self.ctx, pts.contiguous(), (pts if pts_dir is None else pts_dir).contiguous(),
                m.lxyz.reshape(-1, 3), m.xyz_scale, m.embedder['xyz'].n_freqs,
                m.embedder['ldir'].n_freqs)
            return ad.mlp_apply(e, layers, acts, skip, self.precision, in_dim=width).reshape(n, L)
        e_x = ad.embed(m.xyz_scale * pts, m.embedder['xyz'].n_freqs)
        e_l = ad.embed(surf2l.reshape(-1, 3), m.embedder['ldir'].n_freqs)
        e = torch.cat((e_x[:, None, :].expand(n, L, e_x.shape[1]).reshape(n * L, -1), e_l), -1)
        return ad.mlp_apply(e, layers, acts, skip, self.precision).reshape(n, L)

    def _brdf_learned(self, surf2l, surf2c, normal, z):
        """nerfactor.py:413-457 -> the front-masked spec [n, L] (all pairs evaluated; back-lit ones
        are zeroed, :454-455); albedo / pi + spec * scale (:458-461) is formed by ad.integrate."""
        m = self.model
        n, L = surf2l.shape[0], surf2l.shape[1]
        w2l = ad.gen_world2local(normal)
        vdir = torch.einsum('jkl,jl->jk', w2l, surf2c)
        ldir = torch.einsum('jkl,jnl->jnk', w2l, surf2l)
        ldir_flat = ldir.reshape(-1, 3)
        vdir_flat = vdir[:, None, :].expand(n, L, 3).reshape(-1, 3)
        rusink = ad.dir2rusink(ldir_flat, vdir_flat)
        z_flat = z[:, None, :].expand(n, L, z.shape[1]).reshape(n * L, -1)
        front = (ldir_flat[:, 2] > 0).to(z.dtype)
        e = torch.cat((z_flat, ad.embed(rusink, m.embedder['rusink'].n_freqs)), 1)
        trunk = m.brdf_model.net['brdf_mlp']
        acts = [l.activation for l in trunk.layers] + ['softplus']
        spec = ad.mlp_apply(e, self.brdf_layers, acts, trunk.skip_at, self.precision)[:, 0] * front
        return spec.reshape(n, L)

    def forward(self, flat, batch, mode, xyz_noise=None, all_fg=False):
        """Differentiable `Model.call` (shape.py:146-182 / nerfactor.py:181-313) + loss.
        all_fg: the caller guarantees alpha > 0 for every ray (what the train-mode sampler
        produces, nerf_shape.py:84-121), so the foreground compaction is the identity and the
        step has static shapes (CUDA-graph capturable)."""
        m = self.model
        views = self.views(flat)
        dev = self.device
        _, _, rayo, _, rgb, alpha, xyz, normal, lvis = batch
        rayo, rgb, alpha, xyz, normal, lvis = [to_device(x, dev) for x in
                                               (rayo, rgb, alpha, xyz, normal, lvis)]
        is_shape = not hasattr(m, 'shape_mode')
        jitter_std = m.config.getfloat('DEFAULT', 'xyz_jitter_std')
        if is_shape or all_fg:
            sel = lambda x: x
            ind = None
        else:
            mask = alpha[:, 0] > 0
            ind = torch.nonzero(mask, as_tuple=False)[:, 0]
            sel = lambda x: x.index_select(0, ind)
        rayo_m, rgb_m, xyz_m, normal_m, lvis_m = [sel(x) for x in (rayo, rgb, xyz, normal, lvis)]
        if xyz_noise is None and jitter_std > 0:
            xyz_noise = torch.randn_like(xyz_m) * jitter_std
        elif xyz_noise is not None:
            xyz_noise = to_device(xyz_noise, dev)
        lxyz = m.lxyz.reshape(1, -1, 3)
        surf2l = ad.safe_l2_normalize(lxyz - xyz_m[:, None, :], 2)          # shape.py:128-135
        xyz_j = None if xyz_noise is None else xyz_m + xyz_noise

        n_full = alpha.shape[0]

        def scatter(v):
            if v is None or ind is None:
                return v
            out = torch.zeros((n_full,) + tuple(v.shape[1:]), dtype=v.dtype, device=dev)
            return out.index_copy(0, ind, v)

        if is_shape:
            normal_pred = ad.safe_l2_normalize(self._point(views, 'normal', xyz_m) + 1e-6, 1)
            normal_j = None
            if xyz_j is not None and m.normal_smooth_weight > 0:
                normal_j = ad.safe_l2_normalize(self._point(views, 'normal', xyz_j) + 1e-6, 1)
            lvis_pred = self._lvis(views, xyz_m, surf2l)
            lvis_j = None
            if xyz_j is not None and m.lvis_smooth_weight > 0:
                lvis_j = self._lvis(views, xyz_j, surf2l, xyz_m)
            pred = {'normal': normal_pred, 'lvis': lvis_pred}
            gt = {'normal': normal, 'lvis': lvis, 'alpha': alpha}
            loss = m.compute_loss(pred, gt, normal_jitter=normal_j, lvis_jitter=lvis_j)
            return loss, pred

        surf2c = ad.safe_l2_normalize(rayo_m - xyz_m, 1)                     # shape.py:137-144
        if m.shape_mode == 'nerf':
            normal_pred, normal_j = normal_m, None
            lvis_pred, lvis_j = torch.clamp(lvis_m, 1e-8, 1.), None
        else:
            normal_pred = self._point(views, 'normal', xyz_m) + 1e-6
            normal_j = None if xyz_j is None else self._point(views, 'normal', xyz_j) + 1e-6
            lvis_pred = self._lvis(views, xyz_m, surf2l)
            lvis_j = None if xyz_j is None else self._lvis(views, xyz_j, surf2l, xyz_m)
        normal_raw = normal_pred                       # ad.integrate normalises it itself (:212)
        normal_pred = ad.safe_l2_normalize(normal_pred, 1)
        if normal_j is not None:
            normal_j = ad.safe_l2_normalize(normal_j, 1)
        slope = m.config.getfloat('DEFAULT', 'albedo_slope', fallback=0.7)
        bias = m.config.getfloat('DEFAULT', 'albedo_bias', fallback=0.1)
        albedo = slope * self._point(views, 'albedo', xyz_m) + bias
        albedo_j = None if xyz_j is None else slope * self._point(views, 'albedo', xyz_j) + bias
        z = self._point(views, 'brdf_z', xyz_m)
        z_j = None if xyz_j is None else self._point(views, 'brdf_z', xyz_j)
        if m.normalize_brdf_z:
            z = ad.safe_l2_normalize(z, 1)
            z_j = None if z_j is None else ad.safe_l2_normalize(z_j, 1)
        light = torch.clamp(views[('light', 0, 'light')], min=0.)
        light_flat = light.reshape(-1, 3)
        if m.light_idx is not None:
            light_flat = light_flat[m.light_idx.long()]
        srgb = m.config.getboolean('DEFAULT', 'linear2srgb')
        if getattr(m, 'brdf_model', None) is not None:
            spec = self._brdf_learned(surf2l, surf2c, normal_pred, z)
            rgb_pred = ad.integrate(lvis_pred, normal_raw, albedo, spec, light_flat, xyz_m, rayo_m,
                                    m.lxyz, m.lareas, 1, 0., m.config.getfloat(
                                        'DEFAULT', 'learned_brdf_scale'), srgb)
        else:
            rgb_pred = ad.integrate(lvis_pred, normal_raw, albedo, z, light_flat, xyz_m, rayo_m,
                                    m.lxyz, m.lareas, 0, m.config.getfloat('DEFAULT', 'fresnel_f0'),
                                    1., srgb)
        pred = {'rgb': scatter(rgb_pred), 'normal': scatter(normal_pred),
                'lvis': scatter(lvis_pred), 'albedo': scatter(albedo), 'brdf': scatter(z)}
        gt = {'rgb': scatter(rgb_m), 'normal': scatter(normal_m), 'lvis': scatter(lvis_m),
              'alpha': alpha}
        m_light = m._light
        m._light = views[('light', 0, 'light')]       # compute_loss reads self.light (TV prior)
        try:
            loss = m.compute_loss(pred, gt, mode=mode, normal_jitter=scatter(normal_j),
                                  lvis_jitter=scatter(lvis_j), brdf_prop_jitter=scatter(z_j),
                                  albedo_jitter=scatter(albedo_j))
        finally:
            m._light = m_light
        return loss, pred

    # ------------------------------------------------------------------ steps
    def loss_and_grad(self, batch, xyz_noise=None, global_batch=None, all_fg=False):
        """-> (per-ray loss [N], flat gradient of sum(loss) / global_batch)."""
        flat = self.flat.detach().requires_grad_(True)
        loss, _ = self.forward(flat, batch, 'train', xyz_noise, all_fg)
        gb = global_batch or (loss.shape[0] * self.world_size)
        total = torch.sum(loss) / gb                      # tf.nn.compute_average_loss
        (grad,) = torch.autograd.grad(total, flat)
        return loss.detach(), grad

    # ---- CUDA-graph replay of forward + backward (the ~2000 small launches of one step)
    def _all_foreground(self, alpha):
        a = alpha[:, 0] if getattr(alpha, 'ndim', 2) == 2 else alpha
        return bool((a > 0).all())

    def _graphed_loss_and_grad(self, batch, xyz_noise):
        """Captures loss_and_grad once per input-shape signature and replays it; inputs are copied
        into static device buffers.  Returns None when the batch is not graphable."""
        is_shape = not hasattr(self.model, 'shape_mode')
        if not is_shape and not self._all_foreground(batch[5]):
            return None
        fields = (2, 4, 5, 6, 7, 8)                      # rayo, rgb, alpha, xyz, normal, lvis
        key = tuple(tuple(batch[i].shape) for i in fields) + (xyz_noise is not None,)
        st = self._graphs.get(key)
        if st is None:
            bufs = {i: torch.empty(tuple(batch[i].shape), dtype=torch.float32, device=self.device)
                    for i in fields}
            nbuf = None if xyz_noise is None else torch.empty(
                tuple(xyz_noise.shape), dtype=torch.float32, device=self.device)
            static = tuple(bufs.get(i, batch[i] if i < 2 else None) for i in range(9))
            st = {'bufs': bufs, 'noise': nbuf, 'batch': static, 'graph': None}
            self._graphs[key] = st
        for i, bt in st['bufs'].items():
            bt.copy_(torch.as_tensor(batch[i]), non_blocking=True)
        if st['noise'] is not None:
            st['noise'].copy_(torch.as_tensor(xyz_noise), non_blocking=True)
        if st['graph'] is None:
            cur = torch.cuda.current_stream()
            side = torch.cuda.Stream()
            side.wait_stream(cur)
            with torch.cuda.stream(side):                # warm-up off the capture stream
                self.loss_and_grad(st['batch'], st['noise'], all_fg=True)
            cur.wait_stream(side)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                st['loss'], st['grad'] = self.loss_and_grad(st['batch'], st['noise'], all_fg=True)
            st['graph'] = g
        st['graph'].replay()
        return st['loss'], st['grad']

    def train_step(self, batch, xyz_noise=None, graph=True):
        """trainvali.py:273-295: one optimizer iteration; returns the summed loss / global bs.
        graph=True replays forward + backward as one CUDA graph when the batch allows it."""
        out = self._graphed_loss_and_grad(batch, xyz_noise) if (
            graph and self.device.type == 'cuda') else None
        loss, grad = out if out is not None else self.loss_and_grad(batch, xyz_noise)
        if self.world_size > 1:
            import torch.distributed as dist
            dist.all_reduce(grad, op=dist.ReduceOp.SUM)   # gradient all-reduce (one flat buffer)
        lr = self.learning_rate()
        self.iterations += 1
        _lib.adam_amsgrad_step(self.ctx, self.flat, grad.contiguous(), self.m, self.v, self.vhat,
                               lr, self.iterations)
        total = torch.sum(loss) / (loss.shape[0] * self.world_size)
        if self.world_size > 1:
            import torch.distributed as dist
            dist.all_reduce(total, op=dist.ReduceOp.SUM)
        return total

    # ------------------------------------------------------------ checkpoint / resume
    def _var_path(self, key):
        net_name, li, kind = key
        if kind in ('light', 'z'):
            return 'net/_light' if kind == 'light' else 'net/latent_code/_z'
        return 'net/net_%s_layer%d/%s' % (net_name, li, kind)

    def save_checkpoint(self, ckpt_dir, step):
        """trainvali.py:134-141, 197-200: writes `ckpt_dir/ckpt-<step>` in TensorFlow's tensor-
        bundle format under the reference's variable names (weights, light, `step`, AMSGrad
        `iter` / `m` / `v` / `vhat` slots) and updates the `checkpoint` state file."""
        import os
        from .util import tfckpt
        sfx = '/.ATTRIBUTES/VARIABLE_VALUE'
        tensors = {'step' + sfx: np.asarray(step, np.int32),
                   'optimizer/iter' + sfx: np.asarray(self.iterations, np.int64)}
        host = {n: t.detach().cpu().numpy() for n, t in
                (('p', self.flat), ('m', self.m), ('v', self.v), ('vhat', self.vhat))}
        for key, off, shp in zip(self.names, self.offsets[:-1], self.shapes):
            n = int(np.prod(shp))
            path = self._var_path(key)
            tensors[path + sfx] = host['p'][off:off + n].reshape(shp)
            for slot in ('m', 'v', 'vhat'):
                tensors['%s/.OPTIMIZER_SLOT/optimizer/%s%s' % (path, slot, sfx)] = \
                    host[slot][off:off + n].reshape(shp)
        prefix = os.path.join(ckpt_dir, 'ckpt-%d' % step)
        tfckpt.write_checkpoint(prefix, tensors)
        with open(os.path.join(ckpt_dir, 'checkpoint'), 'w') as f:
            f.write('model_checkpoint_path: "ckpt-%d"\nall_model_checkpoint_paths: "ckpt-%d"\n'
                    % (step, step))
        return prefix

    def restore_checkpoint(self, prefix):
        """Resumes weights, light, optimizer slots and iteration count from `prefix` (a file
        written by save_checkpoint or by the reference's CheckpointManager); variables the
        checkpoint lacks keep their values.  Returns the stored `step` (0 if absent)."""
        from .util import tfckpt
        sfx = '/.ATTRIBUTES/VARIABLE_VALUE'
        t = tfckpt.read_checkpoint(prefix)
        bufs = {'p': self.flat, 'm': self.m, 'v': self.v, 'vhat': self.vhat}
        for key, off, shp in zip(self.names, self.offsets[:-1], self.shapes):
            n = int(np.prod(shp))
            path = self._var_path(key)
            for slot, buf in bufs.items():
                name = path + sfx if slot == 'p' else \
                    '%s/.OPTIMIZER_SLOT/optimizer/%s%s' % (path, slot, sfx)
                if name in t:
                    if tuple(t[name].shape) != tuple(shp):
                        raise ValueError("%s: shape %s, expected %s" % (name, t[name].shape, shp))
                    buf[off:off + n] = torch.as_tensor(
                        np.ascontiguousarray(t[name], np.float32).reshape(-1)).to(self.device)
        if 'optimizer/iter' + sfx in t:
            self.iterations = int(t['optimizer/iter' + sfx])
        self.sync_to_model()
        return int(t['step' + sfx]) if 'step' + sfx in t else 0

    @torch.no_grad()
    def vali_step(self, batch):
        """trainvali.py:301-317: forward in 'vali' mode through the fused inference kernels."""
        self.sync_to_model()
        pred, gt, loss_kwargs, _ = self.model.call(batch, 'vali')
        return self.model.compute_loss(pred, gt, **loss_kwargs)


class NerfTrainer(Trainer):
    """Train step of the NeRF itself (the stage before Stage A; nerfactor/models/nerf.py:100-300
    driven by trainvali.py:273-295): stratified + hierarchical sampling, both networks, L2 on the
    coarse and the fine rendering.  The Dense contractions run in nf_dense_fwd / nf_dense_bwd
    (8 x 256 trunk with the skip, sigma head, bottleneck, view-dependent colour head); sampling,
    compositing and the loss are torch ops on the device, so autograd supplies their adjoint.
    The hierarchical samples carry no gradient (tf.stop_gradient, nerf.py:143).

    Random draws of the reference (tf.random.uniform for the stratified / importance samples,
    nerf.py:133, util/math.py:81; tf.random.normal for the density noise, nerf.py:196) are explicit
    optional inputs (`perturb_u`, `fine_u`, `sigma_noise`), drawn with torch when not given.
    `z_all` replays the sorted union of coarse and importance samples itself (they carry no
    gradient): the inverse-CDF lookup is discontinuous in the coarse weights, so a comparison of
    gradients with another implementation fixes the samples and leaves the lookup out."""

    def __init__(self, model, config=None, world_size=1, rank=0, precision=None):
        super().__init__(model, config, world_size, rank, precision or 'fp32')
        cfg = config or model.config
        self.n_c = cfg.getint('DEFAULT', 'n_samples_coarse')
        self.n_f = cfg.getint('DEFAULT', 'n_samples_fine')
        self.lin_in_disp = cfg.getboolean('DEFAULT', 'lin_in_disp')
        self.perturb = cfg.getboolean('DEFAULT', 'perturb')
        self.noise_std = cfg.getfloat('DEFAULT', 'noise_std')

    # ---- pieces -------------------------------------------------------------------
    def _layers(self, views, name):
        net = self.model.net[name]
        out = []
        for li in range(len(net.layers)):
            key = (name, li, 'kernel')
            out.append((views[key], views[(name, li, 'bias')]) if key in views
                       else self._frozen[(name, li)])
        return out

    def _eval(self, views, pref, rayo, rayd, z):
        """nerf.py:254-290 (use_views): rgbs [n, S, 4] = (raw rgb, raw sigma)."""
        m = self.model
        n, S = z.shape
        pts = (rayo[:, None, :] + rayd[:, None, :] * z[:, :, None]).reshape(-1, 3)
        vdir = rayd[:, None, :].expand(n, S, 3).reshape(-1, 3)
        enc = m.net[pref + 'enc']
        feat = ad.mlp_apply(ad.embed(pts, m.embedder['xyz'].n_freqs), self._layers(views, pref + 'enc'),
                            ['relu'] * len(enc.layers), enc.skip_at, self.precision)
        sigma = ad.mlp_apply(feat, self._layers(views, pref + 'sigma_out'), [None], None,
                             self.precision)
        bott = ad.mlp_apply(feat, self._layers(views, pref + 'bottleneck'), [None], None,
                            self.precision)
        fv = torch.cat((bott, ad.embed(vdir, m.embedder['view'].n_freqs)), -1)
        rgb = ad.mlp_apply(fv, self._layers(views, pref + 'rgb_out'), ['relu', None], None,
                           self.precision)
        return torch.cat((rgb, sigma), -1).reshape(n, S, 4)

    def _accumulate(self, rgbs, z, rayd, sigma_noise=None, inf=1e10, eps=1e-6):
        """nerf.py:184-252: weights, colour composited onto the background, occupancy."""
        dist = torch.cat((z[:, 1:] - z[:, :-1], torch.full_like(z[:, :1], inf)), -1)
        dist = dist * torch.linalg.norm(rayd[:, None, :], dim=-1)
        sigma = rgbs[:, :, 3]
        if sigma_noise is not None:
            sigma = sigma + sigma_noise
        elif self.noise_std > 0:
            sigma = sigma + torch.randn_like(sigma) * self.noise_std
        density = 1. - torch.exp(-torch.relu(sigma) * dist)
        t = 1. - density + eps                                   # util/math.py:67-68
        trans = torch.cat((torch.ones_like(t[:, :1]), torch.cumprod(t, -1)[:, :-1]), -1)
        weights = density * trans
        occu = weights.sum(-1)
        rgb = (weights[:, :, None] * torch.sigmoid(rgbs[:, :, :3])).sum(-2)
        bg = 1. if self.model.white_bg else 0.
        return rgb * occu[:, None] + bg * (1. - occu[:, None]), weights

    @staticmethod
    def _inv_transform_sample(val, weights, n_samples, u=None, eps=1e-5):
        """util/math.py:71-94 (searchsorted side='right'); deterministic u = linspace(0, 1, n)
        when `u` is None and perturbation is off."""
        pdf = weights / (weights.sum(-1, keepdim=True) + eps)
        cdf = torch.cat((torch.zeros_like(pdf[:, :1]), torch.cumsum(pdf, -1)), -1)
        ind = torch.searchsorted(cdf.contiguous(), u.contiguous(), right=True)
        below = torch.clamp(ind - 1, min=0)
        above = torch.clamp(ind, max=cdf.shape[-1] - 1)
        c0, c1 = torch.gather(cdf, 1, below), torch.gather(cdf, 1, above)
        v0, v1 = torch.gather(val, 1, below), torch.gather(val, 1, above)
        denom = c1 - c0
        denom = torch.where(denom < eps, torch.ones_like(denom), denom)
        return v0 + (u - c0) / denom * (v1 - v0)

    # ---- step ---------------------------------------------------------------------
    def forward(self, flat, batch, mode='train', perturb_u=None, fine_u=None, sigma_noise=None,
                z_all=None):
        """-> (per-ray loss [N], {'coarse': rgb, 'fine': rgb})."""
        m, dev = self.model, self.device
        views = self.views(flat)
        _, _, rayo, rayd, rgb_gt = batch
        rayo, rayd, rgb_gt = [to_device(x, dev) for x in (rayo, rayd, rgb_gt)]
        rayd = rayd * torch.rsqrt(torch.clamp((rayd * rayd).sum(1, keepdim=True), min=1e-12))
        n = rayo.shape[0]
        perturb = self.perturb and mode == 'train'
        t = torch.linspace(0., 1., self.n_c, device=dev)
        if self.lin_in_disp:
            z = 1. / (1. / m.near * (1. - t) + 1. / m.far * t)
        else:
            z = m.near * (1. - t) + m.far * t
        z = z[None, :].expand(n, self.n_c)
        if perturb or perturb_u is not None:                       # nerf.py:129-135
            mid = .5 * (z[:, 1:] + z[:, :-1])
            upper, lower = torch.cat((mid, z[:, -1:]), -1), torch.cat((z[:, :1], mid), -1)
            u = to_device(perturb_u, dev) if perturb_u is not None else torch.rand_like(lower)
            z = lower + (upper - lower) * u
        sn = (None, None) if sigma_noise is None else [to_device(x, dev) for x in sigma_noise]
        rgb_c, w = self._accumulate(self._eval(views, 'coarse_', rayo, rayd, z), z, rayd, sn[0])
        mse = lambda a: torch.mean((a - rgb_gt) ** 2, dim=-1)
        loss, pred = mse(rgb_c), {'coarse': rgb_c, 'fine': None}
        if self.n_f > 0:
            with torch.no_grad():                                   # tf.stop_gradient, nerf.py:143
                if z_all is not None:
                    z_all = to_device(z_all, dev).contiguous()
                    assert z_all.shape == (n, self.n_c + self.n_f)
                else:
                    if fine_u is not None:
                        u = to_device(fine_u, dev)
                    elif perturb:
                        u = torch.rand((n, self.n_f), device=dev)
                    else:
                        u = torch.linspace(0., 1., self.n_f, device=dev)[None, :].expand(n, self.n_f)
                    z_f = self._inv_transform_sample(.5 * (z[:, 1:] + z[:, :-1]),
                                                     w[:, 1:-1].detach(), self.n_f, u.contiguous())
                    z_all = torch.sort(torch.cat((z, z_f), -1), -1).values
            self.last_z_all = z_all               # sample depths of the fine pass (diagnostics)
            rgb_f, _ = self._accumulate(self._eval(views, 'fine_', rayo, rayd, z_all), z_all, rayd,
                                        sn[1])
            loss = loss + mse(rgb_f)
            pred['fine'] = rgb_f
        return loss, pred

    def loss_and_grad(self, batch, global_batch=None, **draws):
        flat = self.flat.detach().requires_grad_(True)
        loss, _ = self.forward(flat, batch, 'train', **draws)
        gb = global_batch or (loss.shape[0] * self.world_size)
        (grad,) = torch.autograd.grad(torch.sum(loss) / gb, flat)
        return loss.detach(), grad

    def _graphed_loss_and_grad(self, batch, xyz_noise):
        return None                  # data-dependent hierarchical sampling: eager

    def train_step(self, batch, graph=False, **draws):
        loss, grad = self.loss_and_grad(batch, **draws)
        if self.world_size > 1:
            import torch.distributed as dist
            dist.all_reduce(grad, op=dist.ReduceOp.SUM)
        lr = self.learning_rate()
        self.iterations += 1
        _lib.adam_amsgrad_step(self.ctx, self.flat, grad.contiguous(), self.m, self.v, self.vhat,
                               lr, self.iterations)
        total = torch.sum(loss) / (loss.shape[0] * self.world_size)
        if self.world_size > 1:
            import torch.distributed as dist
            dist.all_reduce(total, op=dist.ReduceOp.SUM)
        return total

    @torch.no_grad()
    def vali_step(self, batch):
        self.sync_to_model()
        pred, gt, loss_kwargs, _ = self.model.call(batch, 'vali')
        return self.model.compute_loss(pred, gt, keep_batch=True, **loss_kwargs)


class BrdfTrainer(Trainer):
    """Training of the BRDF prior (nerfactor/models/brdf.py under trainvali.py:273-295): one
    material per step, `n_rays_per_step` random entries of its MERL table; the softplus MLP on
    [z | embed(rusink)] and on the reciprocal coordinates, log-space L2 against the measured
    reflectance; the MLP AND the per-material latent codes are optimised (Generative Latent
    Optimization), so only the row of the step's material receives a gradient."""

    def __init__(self, model, config=None, world_size=1, rank=0, precision=None):
        if not hasattr(model, 'ctx'):           # the prior's model is host-only until trained
            model.ctx = _lib.default_context()
            model.device, model.precision = model.ctx.device, 'fp32'
        super().__init__(model, config, world_size, rank, precision or 'fp32')

    def forward(self, flat, batch, mode='train'):
        m, dev = self.model, self.device
        views = self.views(flat)
        _, i, _, _, _, rusink, refl = batch
        rusink, refl = to_device(rusink, dev), to_device(refl, dev)
        layers = [(views[(name, li, 'kernel')], views[(name, li, 'bias')])
                  for name in ('brdf_mlp', 'brdf_out') for li in range(len(m.net[name].layers))]
        z_all = views[('z', 0, 'z')]
        if m.latent_code.normalize:
            z_all = ad.safe_l2_normalize(z_all, 1)
        i0 = int(np.asarray(i).reshape(-1)[0])
        z = z_all[i0:i0 + 1].expand(rusink.shape[0], -1)
        brdf, brdf_reci = m._eval_brdf_at(z, rusink, layers, self.precision)
        pred = {'brdf': brdf, 'brdf_reci': brdf_reci}
        return m.compute_loss(pred, {'brdf': refl}, keep_batch=True), pred

    def loss_and_grad(self, batch, global_batch=None):
        flat = self.flat.detach().requires_grad_(True)
        loss, _ = self.forward(flat, batch, 'train')
        gb = global_batch or (loss.shape[0] * self.world_size)
        (grad,) = torch.autograd.grad(torch.sum(loss) / gb, flat)
        return loss.detach(), grad

    def _graphed_loss_and_grad(self, batch, xyz_noise):
        return None

    def train_step(self, batch, graph=False):
        return NerfTrainer.train_step(self, batch)


def make_trainer(model, config=None, **kw):
    """The trainer for a model: NeRF (models/nerf.py), the BRDF prior, or shape / NeRFactor."""
    net = getattr(model, 'net', {})
    if 'coarse_enc' in net:
        return NerfTrainer(model, config, **kw)
    if 'brdf_mlp' in net:
        return BrdfTrainer(model, config, **kw)
    return Trainer(model, config, **kw)


# =============================================================================== script
def _parse_args(argv=None):
    import argparse
    ap = argparse.ArgumentParser(
        description="Mirror of nerfactor/trainvali.py's command line (trainvali.py:33-39)")
    ap.add_argument('--config', default='nerfactor.ini',
                    help="base .ini file in config/ or a full path")
    ap.add_argument('--config_override', default='', help="e.g., 'key1=value1,key2=value2'")
    ap.add_argument('--debug', action='store_true')
    ap.add_argument('--device', default='gpu', choices=['gpu'],
                    help="the reference's 'cpu' strategy does not exist here: no CPU fallback")
    ap.add_argument('--precision', default=None, choices=[None, 'bf16', 'f16', 'fp32'],
                    help="arithmetic of the training Dense kernels (default bf16)")
    return ap.parse_args(argv)


def load_config(path, override=''):
    """trainvali.py:53-62: a full path, or a name resolved against the built-in defaults
    (`nerfactor.ini`, `nerfactor_microfacet.ini`, `shape.ini`; the reference ships these under
    nerfactor/config/ with site-specific paths), then `key=value,...` overrides."""
    import os
    from .config import default_config
    from .util import io as ioutil
    if os.path.exists(path):
        config = ioutil.read_config(path)
    else:
        config = default_config(os.path.basename(path)[:-len('.ini')]
                                if path.endswith('.ini') else path)
    if override:
        for kv in override.split(','):
            k, v = kv.split('=', 1)
            config.set('DEFAULT', k, v)
    return config


def _prune(ckptdir, keep):
    """tf.train.CheckpointManager(max_to_keep=keep): drop all but the newest `keep` checkpoints."""
    import glob
    import os
    if not keep or keep <= 0:
        return
    steps = sorted(int(os.path.basename(p)[len('ckpt-'):-len('.index')])
                   for p in glob.glob(os.path.join(ckptdir, 'ckpt-*.index')))
    for s in steps[:-keep]:
        for p in glob.glob(os.path.join(ckptdir, 'ckpt-%d.*' % s)):
            os.remove(p)


def main(argv=None):
    """trainvali.py:45-256: config -> output directory -> datasets -> model + AMSGrad ->
    resume -> epochs of (one gradient step per training view) with periodic checkpoints and
    validation visualisations.  One process per GPU under torchrun: every rank draws its share
    of `n_rays_per_step` rays of the same view, gradients meet in one all-reduce."""
    import json
    import os
    import time
    from os.path import join
    from . import datasets, models
    from .util import io as ioutil, config as configutil

    FLAGS = _parse_args(argv)
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if torch.cuda.is_available():          # without a GPU the model constructor raises (no CPU path)
        torch.cuda.set_device(int(os.environ.get('LOCAL_RANK', '0')))
    if world > 1:
        import torch.distributed as dist
        if not dist.is_initialized():
            dist.init_process_group('nccl')
    config = load_config(FLAGS.config, FLAGS.config_override)
    config_dict = configutil.config2dict(config)
    xname = config.get('DEFAULT', 'xname', fallback='lr{lr}').format(**config_dict)
    outdir = join(config.get('DEFAULT', 'outroot'), xname)
    if rank == 0:
        ioutil.prepare_outdir(outdir, overwrite=config.getboolean('DEFAULT', 'overwrite',
                                                                  fallback=False))
        ioutil.write_config(config, outdir.rstrip('/') + '.ini')
    if world > 1:
        dist.barrier()
    # ---- data (trainvali.py:76-100)
    Dataset = datasets.get_dataset_class(config.get('DEFAULT', 'dataset', fallback='nerf_shape'))
    dataset_train = Dataset(config, 'train', debug=FLAGS.debug, seed=1000 + rank)
    global_bs_train = dataset_train.bs
    dataset_train.bs = max(1, global_bs_train // world)       # this rank's share of the rays
    datapipe_train = dataset_train.build_pipeline(no_batch=True, seed=0)   # same view order
    vali_batches = None
    try:
        dataset_vali = Dataset(config, 'vali', debug=FLAGS.debug)
        vali_batches = dataset_vali.build_pipeline(no_batch=True).take(
            config.getint('DEFAULT', 'vali_batches', fallback=4))
    except (FileNotFoundError, AssertionError):
        pass
    # ---- model + optimizer (trainvali.py:102-127)
    Model = models.get_model_class(config.get('DEFAULT', 'model'))
    model = Model(config, debug=FLAGS.debug, precision='fp32' if FLAGS.precision == 'fp32'
                  else 'f16')
    model.register_trainable()
    for k in ('clipnorm', 'clipvalue'):
        if config.getfloat('DEFAULT', k, fallback=-1) > 0:
            raise NotImplementedError("%s > 0 (the reference's configs all use -1)" % k)
    trainer = make_trainer(model, config, world_size=world, rank=rank, precision=FLAGS.precision)
    # ---- resume (trainvali.py:129-146)
    ckptdir = join(outdir, 'checkpoints')
    keep = config.getint('DEFAULT', 'keep_recent_epochs', fallback=-1)
    latest = ioutil.latest_checkpoint(ckptdir) if os.path.isdir(ckptdir) else None
    step = trainer.restore_checkpoint(latest) if latest else 0
    print("Resumed from step:\n\t%s" % latest if latest else "Started from scratch")
    epochs = config.getint('DEFAULT', 'epochs')
    ckpt_period = config.getint('DEFAULT', 'ckpt_period')
    vali_period = config.getint('DEFAULT', 'vali_period')
    vali_vis_epoch_dir = join(outdir, 'vis_vali', 'epoch{e:09d}')

    def log(name, rec):
        if rank == 0:
            with open(join(outdir, name + '.jsonl'), 'a') as f:
                f.write(json.dumps(rec) + '\n')

    # ---- training loop (trainvali.py:168-256); an "epoch" = one step per training view
    while step < epochs:
        batch_loss, batch_time = [], []
        for batch in datapipe_train:
            t0 = time.time()
            loss = trainer.train_step(batch)
            batch_loss.append(float(loss))
            batch_time.append(time.time() - t0)
            if FLAGS.debug:
                break
        assert batch_time, "Dataset is empty"
        step += 1
        if step % ckpt_period == 0:
            if rank == 0:
                saved = trainer.save_checkpoint(ckptdir, step)
                _prune(ckptdir, keep)
                print("Checkpointed step %s:\n\t%s" % (step, saved))
            log('summary_train', {'step': step, 'loss_train': float(np.mean(batch_loss)),
                                  'batch_time_train': float(np.mean(batch_time))})
        if vali_batches is not None and vali_period > 0 and step % vali_period == 0 and rank == 0:
            trainer.sync_to_model()
            losses, vis_dirs = [], []
            for batch_i, batch in enumerate(vali_batches):
                with torch.no_grad():
                    pred, gt, loss_kwargs, to_vis = model.call(batch, 'vali')
                    loss_kwargs['keep_batch'] = True
                    per_ray = model.compute_loss(pred, gt, **loss_kwargs)
                losses.append(float(per_ray.sum() / per_ray.shape[0]))
                vis_dir = join(vali_vis_epoch_dir.format(e=step), 'batch{b:09d}'.format(b=batch_i))
                model.vis_batch(to_vis, vis_dir, mode='vali')
                vis_dirs.append(vis_dir)
            view_at = model.compile_batch_vis(
                vis_dirs, join(vali_vis_epoch_dir.format(e=step), 'all'), mode='vali')
            log('summary_vali', {'step': step, 'loss_vali': float(np.mean(losses)),
                                 'vis_vali': view_at})
        if world > 1:
            dist.barrier()
    return outdir


if __name__ == '__main__':
    main()
