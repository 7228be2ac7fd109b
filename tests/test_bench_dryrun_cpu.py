"""bench.py's control flow on the CPU test double (tests/cpu_backend.py) with CUDA events faked:
guards the JSON contract and the N > 1 path (asynchronous image all-gather, drain inside the timed
region, barrier, max-over-ranks) against Python-level regressions.  The numbers are meaningless;
real runs happen on the B200 box."""
import json
import os
import socket
import sys
import time

import pytest
import torch
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
ARGV = ['bench.py', '--imh', '8', '--imw', '8', '--spp', '8', '--light-h', '2', '--steps', '2',
        '--warmup', '1', '--no-secondary', '--no-cpu-baseline']


class _Event:
    def __init__(self, enable_timing=True):
        self.t = 0.

    def record(self):
        self.t = time.time()

    def elapsed_time(self, other):
        return max((other.t - self.t) * 1e3, 1e-3)


def _patch(mpatch):
    for p in (HERE, ROOT):
        if p not in sys.path:
            sys.path.insert(0, p)
    import cpu_backend
    cpu_backend.install(mpatch)
    mpatch.setattr(torch.cuda, 'Event', _Event)
    mpatch.setattr(torch.cuda, 'synchronize', lambda *a: None)
    mpatch.setattr(torch.cuda, 'set_device', lambda *a: None)
    mpatch.setattr(torch.Tensor, 'pin_memory', lambda self: self)


def _check_line(line, n_gpus):
    d = json.loads(line)
    for k in ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step',
              'higher_is_better', 'scaling', 'vs_baseline', 'dtype', 'data', 'config', 'e2e',
              'gpu_launches', 'clocks', 'roofline', 'cpu_baseline'):
        assert k in d, k
    assert d['n_gpus'] == n_gpus and d['metric'] == 'rays/sec' and d['unit'] == 'rays/s'
    assert d['warmup'] >= 3 and d['scaling'] == 'weak' and d['higher_is_better'] is True
    assert 'workload' in d['config'] and 'model' not in d['config']
    assert set(d['e2e']) >= {'value', 'unit', 'h2d_bytes_per_step', 'd2h_bytes_per_step'}
    rf = d['roofline']
    assert rf['bound'] in ('hbm', 'tensor') and {'achieved', 'peak', 'unit', 'frac', 'traffic'} <= set(rf)
    assert d['gpu_launches'] > 0
    kernels = [r['kernel'] for r in d['rooflines']]
    assert any('pre-computed BRDF lobe' in k for k in kernels)
    return d


def test_bench_single_rank_line(monkeypatch, capsys):
    _patch(monkeypatch)
    monkeypatch.setattr(sys, 'argv', list(ARGV))
    import bench
    bench.main()
    lines = [l for l in capsys.readouterr().out.splitlines() if l.startswith('{')]
    assert len(lines) == 1                               # ONE JSON line on stdout
    d = _check_line(lines[0], 1)
    assert d['value'] == pytest.approx(64 / (d['ms_per_step'] * 1e-3))


def test_bench_dump_outputs_repeatable(monkeypatch, capsys, tmp_path):
    """--dump-outputs writes the last timed step's render result as float32 .npy files, and two
    runs with the same arguments write the same arrays."""
    import numpy as np
    _patch(monkeypatch)
    import bench
    dumps = []
    for run in ('a', 'b'):
        monkeypatch.setattr(sys, 'argv', list(ARGV) + ['--dump-outputs', str(tmp_path / run)])
        bench.main()
        dumps.append({f[:-4]: np.load(str(tmp_path / run / f))
                      for f in sorted(os.listdir(str(tmp_path / run)))})
    capsys.readouterr()
    assert {'rgb', 'alpha', 'xyz', 'normal', 'albedo', 'brdf'} <= set(dumps[0])
    for k, a in dumps[0].items():
        assert a.dtype == np.float32 and a.shape[0] == 64, k
        assert np.array_equal(a, dumps[1][k]), k
    assert dumps[0]['alpha'].max() > 0                   # the view has foreground rays


def test_dump_outputs_samples_rays_above_the_cap(monkeypatch, tmp_path):
    import numpy as np
    if ROOT not in sys.path:
        sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setattr(bench, 'DUMP_MAX_BYTES', 1000)
    pred = {'rgb': torch.arange(300.).reshape(100, 3), 'alpha': torch.arange(100.)[:, None],
            'note': 'not an array'}
    for run in ('a', 'b'):
        bench.dump_outputs(pred, str(tmp_path / run))
    assert sorted(os.listdir(str(tmp_path / 'a'))) == ['alpha.npy', 'rgb.npy']
    rgb, alpha = np.load(str(tmp_path / 'a' / 'rgb.npy')), np.load(str(tmp_path / 'a' / 'alpha.npy'))
    assert rgb.nbytes + alpha.nbytes <= 1000 and rgb.shape[0] == alpha.shape[0] > 0
    assert np.array_equal(rgb[:, 0], 3 * alpha[:, 0])    # the same rays from every array
    assert np.array_equal(rgb, np.load(str(tmp_path / 'b' / 'rgb.npy')))


def _worker(rank, port, q):
    torch.set_num_threads(1)
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank),
                      WORLD_SIZE='2', LOCAL_RANK=str(rank))
    mpatch = pytest.MonkeyPatch()
    _patch(mpatch)
    import io
    import contextlib
    import torch.distributed as dist
    orig = dist.init_process_group
    mpatch.setattr(dist, 'init_process_group',
                   lambda backend, **kw: orig('gloo', rank=rank, world_size=2))
    sys.argv = list(ARGV) + ['--gpus', '2']
    import bench
    buf = io.StringIO()
    with contextlib.redirect_stdout(buf):
        bench.main()
    q.put((rank, [l for l in buf.getvalue().splitlines() if l.startswith('{')]))
    mpatch.undo()


def test_bench_two_ranks_gloo():
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=300) for _ in procs)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert len(res[0]) == 1 and res[1] == []             # rank 0 alone prints
    d = _check_line(res[0][0], 2)
    assert d['value'] == pytest.approx(2 * 64 / (d['ms_per_step'] * 1e-3))   # whole-job aggregate
