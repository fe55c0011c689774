"""The bench.py output contract: the reference arm is run here on the CPU (it only needs the oracle), the product arm is checked
on the bench lines committed under profiles/ (they were produced on a B200 by the same script)."""
import glob
import json
import os
import subprocess
import sys

import numpy as np
import torch

from conftest import ROOT

import bench  # the repository root is on sys.path (conftest.py)

BASE_KEYS = {'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling', 'vs_baseline', 'dtype',
             'data', 'config', 'e2e'}


def test_reference_arm_prints_one_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '1', '--warmup', '1'],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith('{')]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and BASE_KEYS <= set(d) and d['metric'] == 'nav-step decisions/sec' and d['unit'] == 'decisions/s'
    assert d['value'] > 0 and d['higher_is_better'] is True and d['vs_baseline'] is None
    assert d['e2e'] == {'value': d['value'], 'unit': d['unit'], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    cb = d['cpu_baseline']
    assert cb['kind'] in ('reference', 'port') and cb['cores'] >= 1 and cb['value'] == d['value'] and 'sample' in cb
    assert 'workload' in d['config'] and 'model' not in d['config']


def test_reference_arm_dumps_the_logits_of_its_last_step(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--steps', '2', '--warmup', '1',
                          '--dump-outputs', str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.splitlines()[-1])['steps'] == 2
    assert sorted(os.listdir(tmp_path)) == ['fused_logits.npy', 'fused_logits_nonfinite.npy']      # masked logits are -inf
    assert all(np.isfinite(np.load(tmp_path / f)).all() for f in os.listdir(tmp_path))
    got = bench.load_dump(tmp_path)['fused_logits']
    _, shape, _ = bench.workload('duet_cfg2')
    step, _, _ = bench.reference_stepper('duet', shape, 'cpu')
    with torch.no_grad():
        want = step().numpy()
    assert got.dtype == np.float32 and got.shape == want.shape == (shape.batch, shape.n_nodes)
    fin = np.isfinite(want)
    assert (np.isfinite(got) == fin).all()
    assert np.abs(got[fin] - want[fin]).max() <= 1e-4 * np.abs(want[fin]).max()


def test_dump_outputs_writes_finite_float32_within_the_budget(tmp_path, monkeypatch):
    monkeypatch.setattr(bench, 'DUMP_BYTES', 4000)                      # 1000 float32 elements
    outputs = {'masks': torch.tensor([[True, False]]), 'small': torch.arange(6, dtype=torch.float64).view(2, 3),
               'logits': torch.tensor([1.5, -float('inf'), float('inf'), float('nan')]),
               'big': torch.arange(100_000, dtype=torch.int64), 'bigger': -torch.arange(200_000.)}
    bench.dump_outputs(tmp_path / 'a', outputs)
    bench.dump_outputs(tmp_path / 'b', outputs)
    files = sorted(os.listdir(tmp_path / 'a'))
    assert files == sorted([n + '.npy' for n in outputs] + ['logits_nonfinite.npy']) and files == sorted(os.listdir(tmp_path / 'b'))
    stored = [np.load(tmp_path / 'a' / f) for f in files]
    assert all(x.dtype == np.float32 and np.isfinite(x).all() for x in stored)
    assert sum(x.size for x in stored) <= 1000
    a = bench.load_dump(tmp_path / 'a')
    assert set(a) == set(outputs)
    assert a['masks'].tolist() == [[1.0, 0.0]] and a['small'].tolist() == [[0, 1, 2], [3, 4, 5]]    # whole, in shape
    assert a['logits'][:3].tolist() == [1.5, -np.inf, np.inf] and np.isnan(a['logits'][3])
    for n, sign in (('big', 1), ('bigger', -1)):                        # a sorted sample of distinct elements, same each run
        x = a[n]
        assert x.ndim == 1 and 400 <= x.size <= 500 and (np.diff(sign * x) > 0).all()
        assert np.array_equal(x, np.load(tmp_path / 'b' / (n + '.npy')))


def test_committed_product_bench_lines_follow_the_contract():
    files = sorted(glob.glob(os.path.join(ROOT, 'profiles', 'r01b_bench_*.json')))
    assert files
    for f in files:
        d = json.loads(open(f).read().strip().splitlines()[-1])
        assert BASE_KEYS | {'clocks', 'gpu_launches', 'roofline'} <= set(d), f
        assert d['gpu_launches'] > 0 and d['value'] > 0 and d['dtype'] in ('bf16', 'fp32')
        r = d['roofline']
        assert {'bound', 'achieved', 'peak', 'unit', 'frac', 'traffic'} <= set(r) and abs(r['frac'] - r['achieved'] / r['peak']) < 1e-9
        e = d['e2e']
        assert {'value', 'unit', 'h2d_bytes_per_step', 'd2h_bytes_per_step'} <= set(e) and e['value'] != d['value']
        assert not set(d['clocks']['reasons']) & {'hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown'}
        if d['n_gpus'] == 1 and 'train' not in f:
            assert {'value', 'unit', 'cores', 'kind', 'sample'} <= set(d['cpu_baseline'])
