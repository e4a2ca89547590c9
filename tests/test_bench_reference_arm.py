"""`bench.py --impl reference` (the CPU arm the driver runs beside the CUDA arm) needs no GPU: run it here for one step and
check the JSON contract of the line it prints."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), '..'))


def test_reference_arm_prints_the_contract_line(tmp_path):
    res = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '1', '--steps', '1',
                          '--warmup', '1', '--dump-outputs', str(tmp_path / 'out')], capture_output=True, text=True, timeout=900,
                         cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.startswith('{')]
    assert len(lines) == 1, res.stdout[-2000:]                       # exactly ONE JSON line
    d = json.loads(lines[0])
    assert d['impl'] == 'reference'
    base = json.load(open(os.path.join(ROOT, 'BASELINE.json')))
    assert d['metric'] == base['metric'] and d['unit'] == 'pairs/s' and d['higher_is_better'] is True
    assert d['n_gpus'] == 1 and d['steps'] == 1 and d['warmup'] >= 1 and d['scaling'] == 'weak' and d['data'] == 'synthetic'
    assert d['vs_baseline'] is None                                   # BASELINE.md holds no published number for this metric
    assert d['value'] > 0 and abs(d['ms_per_step'] * d['value'] - 1000.0) < 1e-3 * 1000.0      # one pair per step
    assert 'workload' in d['config'] and 'model' not in d['config']
    cb = d['cpu_baseline']
    assert cb['kind'] == 'port' and cb['cores'] >= 1 and cb['value'] == d['value'] and 'pair' in cb['sample']
    assert d['e2e'] == {'value': d['value'], 'unit': 'pairs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    # --dump-outputs: the final flow of the timed step, one pair at 448x512
    assert os.listdir(tmp_path / 'out') == ['flow.npy']
    flow = np.load(tmp_path / 'out' / 'flow.npy')
    assert flow.dtype == np.float32 and flow.shape == (1, 448, 512, 2) and np.isfinite(flow).all() and np.abs(flow).max() > 0
