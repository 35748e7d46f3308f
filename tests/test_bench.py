"""bench.py --dump-outputs: what the last timed step computed, as .npy files of bounded size (float32 / float64; larger
arrays sampled at fixed positions), the same from run to run; --steps sets the number of timed steps."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from tests.helpers import rel_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load(d):
    return {f[:-len('.npy')]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_write_outputs_bounds_and_sample_positions(tmp_path):
    import bench
    n = bench.DUMP_CAP['params'] + 1000
    flat = torch.arange(n, dtype=torch.float32)
    arrays = {'params': flat, 'grads': -flat, 'z': torch.ones(4, 3, dtype=torch.float64),
              'loss': torch.tensor([2.5]), 'logits': torch.arange(2000000)}
    bench.write_outputs(str(tmp_path / 'a'), arrays)
    bench.write_outputs(str(tmp_path / 'b'), arrays)
    a, b = _load(tmp_path / 'a'), _load(tmp_path / 'b')
    assert sorted(a) == sorted(arrays)
    assert sum(os.path.getsize(tmp_path / 'a' / f) for f in os.listdir(tmp_path / 'a')) <= 64 * 1000 * 1000
    for k in a:
        assert a[k].dtype in (np.float32, np.float64) and np.array_equal(a[k], b[k]), k
    assert a['z'].dtype == np.float64 and a['z'].shape == (4, 3)
    assert a['loss'].tolist() == [2.5]
    p = a['params']
    assert p.shape == (bench.DUMP_CAP['params'],) and np.all(np.diff(p) > 0) and p[-1] < n     # distinct, in order
    assert np.array_equal(a['grads'], -p)                              # the same positions in params and grads
    assert a['logits'].dtype == np.float32 and a['logits'].size == 1000000


@pytest.mark.gpu
def test_bench_dumps_the_last_timed_step(tmp_path):
    env = dict(os.environ, IMPFLOW_BENCH_NOSAMPLER='1')

    def run(out):
        r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--workload', 'toy', '--steps', '3',
                            '--warmup', '1', '--no-cpu-baseline', '--dump-outputs', str(out)],
                           cwd=str(tmp_path), env=env, capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-4000:]
        lines = r.stdout.strip().splitlines()
        assert len(lines) == 1, r.stdout[-4000:]
        return json.loads(lines[0]), _load(out)

    line, a = run(tmp_path / 'a')
    assert line['steps'] == 3 and len(line['per_step_ms']) == 3
    assert sorted(a) == ['grads', 'logdet', 'loss', 'params', 'z']
    batch, d = line['config']['per_gpu_batch'], 2
    assert a['z'].shape == (batch, d) and a['logdet'].shape == (batch, 1) and a['loss'].shape == (1,)
    assert a['params'].shape == a['grads'].shape and a['params'].size > 0
    assert all(np.isfinite(v).all() for v in a.values())
    _, b = run(tmp_path / 'b')
    for k in a:
        assert rel_err(b[k], a[k]) < 1e-4, k
