"""The view-parallel scripts under a 2-process launch (torchrun's environment, gloo instead of
NCCL, CPU test double for the kernels): geometry_from_nerf and test.py split the views round-robin
over the ranks -- every view is produced exactly once, rank 0 compiles the video after a barrier."""
import os
import socket
import sys

import pytest
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))


def _worker(rank, world, port, tmp, q):
    import torch
    torch.set_num_threads(1)
    for p in (HERE, os.path.dirname(HERE)):
        if p not in sys.path:
            sys.path.insert(0, p)
    # CUDA_VISIBLE_DEVICES='': the kernels are the CPU test double, so the scripts must not pick
    # cuda:<LOCAL_RANK> (which does not exist on a one-GPU machine) either
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank),
                      WORLD_SIZE=str(world), LOCAL_RANK=str(rank), CUDA_VISIBLE_DEVICES='')
    import cpu_backend
    mpatch = pytest.MonkeyPatch()
    cpu_backend.install(mpatch)
    from nerfactor_b200 import geometry_from_nerf as gfn, test as nftest
    nerf_dir, surf, ckpt = (os.path.join(tmp, 'out', 'nerf', 'lr1e-4'), os.path.join(tmp, 'surf'),
                            os.path.join(tmp, 'out', 'nerfactor', 'lr5e-3', 'checkpoints', 'ckpt-1'))
    done = gfn.main(['--trained_nerf', nerf_dir, '--out_root', surf, '--light_h', '2',
                     '--imh', '6', '--precision', 'fp32'])
    import torch.distributed as dist
    dist.init_process_group('gloo', rank=rank, world_size=world)
    dist.barrier()                                     # Stage A of every view before Stage B
    outroot, view_at = nftest.main(['--ckpt', ckpt, '--precision', 'fp32'])
    q.put((rank, sorted(done), outroot, view_at))
    dist.destroy_process_group()
    mpatch.undo()


def test_stage_a_and_test_script_split_views_over_two_ranks(tmp_path):
    sys.path.insert(0, HERE)
    from nerfactor_b200 import config as nfconfig, synth
    from nerfactor_b200.util import io as ioutil, tfckpt
    tmp = str(tmp_path)
    data = os.path.join(tmp, 'data')
    ids = synth.write_scene(data, imh=6, imw=6, n_train=1, n_val=0, n_test=3,
                            envmap_dir=os.path.join(tmp, 'env'), n_probes=1, light_hw=(2, 4))
    nerf_dir = os.path.join(tmp, 'out', 'nerf', 'lr1e-4')
    ioutil.write_config(nfconfig.default_config('nerf', data_root=data, imh=6, n_samples_coarse=-56,
                                                n_samples_fine=4), nerf_dir + '.ini')
    tfckpt.write_checkpoint(os.path.join(nerf_dir, 'checkpoints', 'ckpt-1'),
                            tfckpt.tensors_from_params(synth.make_nerf_params(0), step=1))
    run = os.path.join(tmp, 'out', 'nerfactor', 'lr5e-3')
    cfg = nfconfig.default_config(
        'nerfactor_microfacet', data_root=data, data_nerf_root=os.path.join(tmp, 'surf'), imh=6,
        light_h=2, shape_mode='scratch', test_envmap_dir=os.path.join(tmp, 'env'))
    ioutil.write_config(cfg, run + '.ini')
    params = synth.make_stage_b_params(3, 'microfacet', light_hw=(2, 4))
    tfckpt.write_checkpoint(os.path.join(run, 'checkpoints', 'ckpt-1'),
                            tfckpt.tensors_from_params(params, step=1))
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    mctx = mp.get_context('spawn')
    q = mctx.Queue()
    procs = [mctx.Process(target=_worker, args=(r, 2, port, tmp, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted([q.get(timeout=600) for _ in procs], key=lambda t: t[0])
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    (_, done0, outroot, view0), (_, done1, _, view1) = res
    assert not set(done0) & set(done1) and sorted(done0 + done1) == sorted(ids)   # each view once
    assert len(done0) == 2 and len(done1) == 2
    batches = sorted(d for d in os.listdir(outroot) if d.startswith('batch'))
    assert batches == ['batch%09d' % i for i in range(3)]
    assert all(os.path.exists(os.path.join(outroot, b, 'pred_rgb.png')) for b in batches)
    # OLAT relighting only on the final view, whichever rank owned it (test.py:176)
    assert any(f.startswith('pred_rgb_olat_') for f in os.listdir(os.path.join(outroot, batches[2])))
    assert not any(f.startswith('pred_rgb_olat_') for f in os.listdir(os.path.join(outroot, batches[0])))
    assert view0 is not None and view0.endswith('.mp4') and view1 is None       # rank 0 compiles


def _train_worker(rank, world, port, ini, q):
    import torch
    torch.set_num_threads(1)
    for p in (HERE, os.path.dirname(HERE)):
        if p not in sys.path:
            sys.path.insert(0, p)
    # CUDA_VISIBLE_DEVICES='': the kernels are the CPU test double, so the scripts must not pick
    # cuda:<LOCAL_RANK> (which does not exist on a one-GPU machine) either
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank),
                      WORLD_SIZE=str(world), LOCAL_RANK=str(rank), CUDA_VISIBLE_DEVICES='')
    import cpu_backend
    mpatch = pytest.MonkeyPatch()
    cpu_backend.install(mpatch)
    import torch.distributed as dist
    dist.init_process_group('gloo', rank=rank, world_size=world)     # main() would ask for nccl
    from nerfactor_b200 import trainvali
    outdir = trainvali.main(['--config', ini, '--precision', 'fp32'])
    q.put((rank, outdir))
    dist.destroy_process_group()
    mpatch.undo()


def test_trainvali_script_data_parallel_two_ranks(tmp_path):
    """trainvali.main under a 2-rank launch: every rank draws its half of n_rays_per_step from the
    same view, one gradient all-reduce per step, rank 0 checkpoints and validates while the other
    waits at the epoch barrier; the optimizer has taken epochs x views steps."""
    sys.path.insert(0, HERE)
    from nerfactor_b200 import config as nfconfig, synth
    from nerfactor_b200.util import io as ioutil, tfckpt
    tmp = str(tmp_path)
    data, surf = os.path.join(tmp, 'data'), os.path.join(tmp, 'surf')
    synth.write_scene(data, imh=6, imw=6, n_train=2, n_val=1, n_test=0, nerf_root=surf, n_lights=8)
    cfg = nfconfig.default_config(
        'nerfactor_microfacet', data_root=data, data_nerf_root=surf, imh=6, light_h=2,
        shape_mode='scratch', n_rays_per_step=16, epochs=2, ckpt_period=1, vali_period=2,
        vali_batches=1, outroot=os.path.join(tmp, 'out'))
    ini = os.path.join(tmp, 'run.ini')
    ioutil.write_config(cfg, ini)
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    mctx = mp.get_context('spawn')
    q = mctx.Queue()
    procs = [mctx.Process(target=_train_worker, args=(r, 2, port, ini, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=600) for _ in procs]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    outdir = res[0][1]
    ckpt = ioutil.latest_checkpoint(os.path.join(outdir, 'checkpoints'))
    assert ckpt.endswith('ckpt-2')
    t = tfckpt.read_checkpoint(ckpt)
    assert int(t['optimizer/iter/.ATTRIBUTES/VARIABLE_VALUE']) == 4           # 2 epochs x 2 views
    assert os.path.exists(os.path.join(outdir, 'vis_vali', 'epoch000000002', 'all.html'))
