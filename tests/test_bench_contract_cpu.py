"""bench.py's JSON contract: the committed line of the final GPU run carries every key the driver reads, and the reference arm
(`--impl reference`, the CPU ref path through the oracle) prints one line with the same metric / unit / config."""
import importlib.util
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REQUIRED = ('metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling', 'vs_baseline', 'dtype',
            'data', 'config', 'roofline', 'cpu_baseline', 'e2e', 'clocks', 'gpu_launches')


def test_committed_bench_line_has_the_contract_keys():
    line = json.load(open(os.path.join(ROOT, 'profiles', 'r02_bench_v7.json')))
    assert all(k in line for k in REQUIRED), [k for k in REQUIRED if k not in line]
    assert line['metric'] == 'generator_512px_images_per_sec' and line['unit'] == 'images/s' and line['higher_is_better'] is True
    assert line['n_gpus'] == 1 and line['warmup'] >= 3 and line['scaling'] == 'weak' and line['vs_baseline'] is None
    assert 'workload' in line['config'] and 'model' not in line['config']
    roof = line['roofline']
    assert roof['bound'] in ('hbm', 'tensor') and abs(roof['frac'] - roof['achieved'] / roof['peak']) < 1e-9 and roof['traffic']
    assert set(('value', 'unit', 'cores', 'kind', 'sample')) <= set(line['cpu_baseline'])
    e2e = line['e2e']
    assert e2e['h2d_bytes_per_step'] > 0 and e2e['d2h_bytes_per_step'] > 0 and e2e['value'] != line['value']
    assert line['gpu_launches'] > 0 and 'sm_mhz' in line['clocks'] and 'reasons' in line['clocks']
    assert line['eager']['ms_per_step'] > 0 and 'launch' in line['config']          # graph replay is the timed entry; eager figure beside it
    assert set(('modulated_conv2d', 'upfirdn2d', 'bias_act', 'conv2d_gradfix_train')) <= set(line['ops'])       # BASELINE configs[3]
    assert line['train']['ms_per_step'] > 0 and line['train']['batch_per_gpu'] == 8                            # BASELINE configs[4]


def test_reference_arm_prints_one_contract_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '0'],
                       capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    line = json.loads(lines[0])
    assert line['impl'] == 'reference' and line['metric'] == 'generator_512px_images_per_sec' and line['unit'] == 'images/s'
    assert line['value'] > 0 and line['cpu_baseline']['kind'] == 'port' and line['cpu_baseline']['cores'] >= 1
    assert line['e2e'] == {'value': line['value'], 'unit': 'images/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}


def _load_bench():
    spec = importlib.util.spec_from_file_location('pgpp_bench', os.path.join(ROOT, 'bench.py'))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_dump_outputs_writes_float_arrays_and_samples_the_same_rows_within_the_budget(tmp_path, monkeypatch):
    bench = _load_bench()
    g = torch.Generator().manual_seed(0)
    out = {'img': torch.randn(8, 3, 16, 16, generator=g), 'pred_parsing': torch.randn(8, 7, 16, 16, generator=g).half(),
           'Loss/scores': torch.randn(8, generator=g, dtype=torch.float64)}
    bench.dump_outputs(str(tmp_path / 'full'), out)
    full = {n: np.load(tmp_path / 'full' / f'{n}.npy') for n in ('img', 'pred_parsing', 'Loss_scores')}
    assert (full['img'].dtype, full['pred_parsing'].dtype, full['Loss_scores'].dtype) == (np.float32, np.float32, np.float64)
    np.testing.assert_array_equal(full['pred_parsing'], out['pred_parsing'].float().numpy())
    budget = 3 * (3 + 7) * 16 * 16 * 4 + 3 * 8        # room for three of the eight batch rows
    monkeypatch.setattr(bench, 'DUMP_BYTES', budget)
    for run in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / run), out)
    a = {n: np.load(tmp_path / 'a' / f'{n}.npy') for n in full}
    assert sum(v.nbytes for v in a.values()) <= budget and all(v.shape[0] == 3 for v in a.values())
    rows = [i for i in range(8) if any(np.array_equal(full['img'][i], r) for r in a['img'])]
    assert len(rows) == 3
    for n in full:
        np.testing.assert_array_equal(a[n], full[n][rows])
        np.testing.assert_array_equal(a[n], np.load(tmp_path / 'b' / f'{n}.npy'))


def test_steps_below_one_are_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--steps', '0'], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 2 and '--steps must be at least 1' in r.stderr
