"""CPU-side check of bench.py's reference arm (`--impl reference`): it must run without a GPU, time the oracle port on the
headline workload and print ONE JSON line with the contract's keys (the driver computes the speed-up from it)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    env = dict(os.environ, B200REC_REF_SAMPLE='8', CUDA_VISIBLE_DEVICES='')
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0'],
                       capture_output=True, text=True, env=env, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['unit'] == 'pairs/s' and d['value'] > 0 and d['higher_is_better'] is True
    assert d['metric'] == 'scored user-item pairs/sec (NCF fwd)' and d['config']['workload'].startswith('configs[1]')
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1
    assert d['e2e'] == {'value': d['value'], 'unit': 'pairs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}


def test_dump_outputs_writes_one_float_npy_per_array(tmp_path, monkeypatch):
    import bench
    out = tmp_path / 'out'
    scores = torch.linspace(-1.0, 1.0, 12).view(6, 2)
    bench.write_outputs(str(out), {'scores': scores, 'items': torch.tensor([[3, 1 << 40]]), 'half': torch.ones(3, dtype=torch.bfloat16),
                                   'wide': torch.zeros(2, dtype=torch.float64)})
    assert sorted(p.name for p in out.iterdir()) == ['half.npy', 'items.npy', 'scores.npy', 'wide.npy']
    a = np.load(out / 'scores.npy')
    assert a.dtype == np.float32 and np.array_equal(a, scores.numpy())
    a = np.load(out / 'items.npy')
    assert a.dtype == np.float64 and a.tolist() == [[3.0, float(1 << 40)]]
    assert np.load(out / 'half.npy').dtype == np.float32 and np.load(out / 'wide.npy').dtype == np.float64
    monkeypatch.setattr(bench, 'DUMP_LIMIT', 40)
    with pytest.raises(SystemExit, match='more than'):
        bench.write_outputs(str(tmp_path / 'big'), {'scores': scores})
    assert not (tmp_path / 'big').exists()


def test_dump_outputs_is_refused_where_no_leg_is_dumped():
    for extra in (['--impl', 'reference'], ['--workload', 'k3hbm']):
        r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--dump-outputs', 'unused', *extra], capture_output=True, text=True,
                           env=dict(os.environ, CUDA_VISIBLE_DEVICES=''), timeout=120, cwd=ROOT)
        assert r.returncode == 2 and '--dump-outputs covers' in r.stderr and r.stdout == ''


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK='1', WORLD_SIZE='2', CUDA_VISIBLE_DEVICES='')
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2', '--steps', '1', '--warmup', '0'],
                       capture_output=True, text=True, env=env, timeout=120, cwd=ROOT)
    assert r.returncode == 0 and r.stdout.strip() == ''
