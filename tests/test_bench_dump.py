"""bench.py --dump-outputs: what the last timed step returned, as float32 .npy files under 64 MB, identical from run to
run with the same arguments (so that two builds can be compared output for output)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT


def test_dump_outputs_budget_and_fixed_row_sample(tmp_path):
    import bench
    g = torch.Generator().manual_seed(0)
    res = {'verts': torch.randn(1000, 6890, 3, generator=g), 'poses': torch.randn(1000, 63, generator=g).double(),
           'joints': torch.randn(1000, 45, 3, generator=g)}
    for d in ('a', 'b'):
        bench.dump_outputs(res, str(tmp_path / d))
    files = sorted(os.listdir(tmp_path / 'a'))
    assert files == ['joints.npy', 'poses.npy', 'verts.npy']
    assert sum(os.path.getsize(tmp_path / 'a' / f) for f in files) <= 64 * 10 ** 6
    out = {f[:-4]: np.load(tmp_path / 'a' / f) for f in files}
    for f in files:
        assert np.array_equal(np.load(tmp_path / 'b' / f), out[f[:-4]])
    assert all(v.dtype == np.float32 for v in out.values())
    # the outputs that fit are written whole; the 82.7 MB one keeps ascending rows of a seed-0 permutation
    assert np.array_equal(out['poses'], res['poses'].float().numpy())
    assert np.array_equal(out['joints'], res['joints'].numpy())
    k = out['verts'].shape[0]
    assert 500 < k < 1000 and out['verts'].shape[1:] == (6890, 3)
    rows = torch.randperm(1000, generator=torch.Generator().manual_seed(0))[:k].sort().values
    assert np.array_equal(out['verts'], res['verts'][rows].numpy())


@pytest.mark.gpu
def test_bench_dump_outputs_repeat_exactly(tmp_path):
    B = 512
    out = {}
    for run in ('a', 'b'):
        r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--gpus', '1', '--steps', '2', '--warmup', '1',
                            '--batch', str(B), '--sde-steps', '16', '--no-cpu', '--configs', 'none',
                            '--dump-outputs', str(tmp_path / run)], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-800:]
        line = json.loads([ln for ln in r.stdout.splitlines() if ln.startswith('{')][-1])
        assert line['steps'] == 2
        out[run] = {f[:-4]: np.load(tmp_path / run / f) for f in os.listdir(tmp_path / run)}
    assert sorted(out['a']) == ['joints', 'poses', 'verts']
    assert out['a']['poses'].shape == (B, 63) and out['a']['joints'].shape == (B, 45, 3)
    assert out['a']['verts'].shape == (B, 6890, 3)
    for k, v in out['a'].items():
        assert v.dtype == np.float32 and np.isfinite(v).all(), k
        assert np.array_equal(v, out['b'][k]), k
