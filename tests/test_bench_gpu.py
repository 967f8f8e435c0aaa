"""bench.py --dump-outputs end to end: every dumped leg (attention, basic, allpairs fp32 / bf16, graph fp32 / bf16) writes its arrays under
the expected names and shapes, --steps sets the timed steps of the line, and two runs with the same arguments write identical arrays."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

EXPECTED = {'attention_scores': ((8, 512, 1), np.float32), 'basic_scores': ((512, 1), np.float32),
            'allpairs_fp32_topk_scores': ((4736, 10), np.float32), 'allpairs_fp32_topk_items': ((4736, 10), np.float64),
            'allpairs_bf16_topk_scores': ((4736, 10), np.float32), 'allpairs_bf16_topk_items': ((4736, 10), np.float64),
            'graph_scores': ((512, 1), np.float32), 'graph_bf16_scores': ((512, 1), np.float32)}


def _run(out):
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--gpus', '1', '--steps', '2', '--warmup', '1', '--no-cpu-baseline',
                        '--no-train-step', '--skip-hbm-regime', '--graph-scale', '0.02', '--dump-outputs', str(out)],
                       capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    return json.loads(lines[0]), {f[:-4]: np.load(os.path.join(out, f)) for f in os.listdir(out)}


def test_dump_outputs_of_every_dumped_leg_are_complete_and_repeatable(tmp_path):
    line, first = _run(tmp_path / 'a')
    assert line['steps'] == 2 and line['ms_per_step'] > 0
    assert sorted(first) == sorted(EXPECTED)
    for name, (shape, dtype) in EXPECTED.items():
        a = first[name]
        assert a.shape == shape and a.dtype == dtype and np.isfinite(a).all(), name
    for precision in ('fp32', 'bf16'):
        items = first[f'allpairs_{precision}_topk_items']
        assert (items == np.round(items)).all() and items.min() >= 0 and items.max() < 100_000
    assert np.abs(first['attention_scores']).max() > 0 and not np.array_equal(first['attention_scores'][0], first['attention_scores'][1])
    _, second = _run(tmp_path / 'b')
    for name in EXPECTED:
        assert np.array_equal(first[name], second[name]), name
