"""bench.py --dump-outputs: what the writer stores (CPU), and that two runs of the b200 arm with the same arguments dump
the same sampler outputs (GPU, tiny shape)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_types_and_size_cap(tmp_path):
    g = torch.Generator().manual_seed(0)
    arrays = {'xh': torch.randn((5000, 13), generator=g), 'mask': torch.arange(5000), 'sizes': torch.tensor([2500, 2500])}
    bench.dump_outputs(arrays, str(tmp_path / 'full'))
    for name, t in arrays.items():
        a = np.load(tmp_path / 'full' / f'{name}.npy')
        assert a.dtype == (np.float32 if t.is_floating_point() else np.float64)
        assert np.array_equal(a, t.numpy())
    limit = 100_000                     # a third of what the arrays hold
    for d in ('a', 'b'):
        bench.dump_outputs(arrays, str(tmp_path / d), limit=limit)
        assert sum(os.path.getsize(tmp_path / d / f) for f in os.listdir(tmp_path / d)) <= limit
    got = {n: np.load(tmp_path / 'a' / f'{n}.npy') for n in arrays}
    for n in arrays:
        assert np.array_equal(got[n], np.load(tmp_path / 'b' / f'{n}.npy'))
    rows = got['mask'].astype(np.int64)
    assert 0 < len(rows) < 5000 and np.all(np.diff(rows) > 0)
    assert np.array_equal(got['xh'], arrays['xh'].numpy()[rows])      # arrays with as many rows keep the same rows


@pytest.mark.gpu
def test_b200_arm_dumps_the_same_outputs_twice(tmp_path):
    argv = ['--steps', '1', '--warmup', '1', '--batch', '2', '--timesteps', '10', '--no-cpu-baseline', '--no-e2e',
            '--profile-calls', '1']
    for d in ('a', 'b'):
        r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), *argv, '--dump-outputs', str(tmp_path / d)],
                           capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads([l for l in r.stdout.splitlines() if l.startswith('{')][-1])['steps'] == 1
    names = ['xh_lig_all', 'lig_sizes_all', 'xh_lig', 'xh_pocket', 'lig_mask', 'pocket_mask']
    assert sorted(os.listdir(tmp_path / 'a')) == sorted(n + '.npy' for n in names)
    a = {n: np.load(tmp_path / 'a' / f'{n}.npy') for n in names}
    b = {n: np.load(tmp_path / 'b' / f'{n}.npy') for n in names}
    assert a['xh_lig'].shape == (2 * 25, 13) and a['xh_lig'].dtype == np.float32
    assert np.array_equal(a['xh_lig_all'], a['xh_lig'])
    for n in ('lig_sizes_all', 'lig_mask', 'pocket_mask'):
        assert np.array_equal(a[n], b[n])
    # same seeded inputs and noise; the tensor-core kernels may sum a receiver's messages in another order
    scale = float(np.abs(a['xh_pocket'][:, :3]).max())
    for n in ('xh_lig', 'xh_pocket'):
        np.testing.assert_allclose(b[n][:, :3], a[n][:, :3], rtol=0, atol=1e-3 * scale)
        assert np.array_equal(a[n][:, 3:], b[n][:, 3:])
