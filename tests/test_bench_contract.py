"""CPU: the reference arm of bench.py (`--impl reference`: the oracle port on the host cores) runs without a GPU and prints
ONE JSON line with the keys the measurement contract names; our arm refuses to run without a CUDA device."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contract_line():
    cp = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--workload', 'lih_paulinet',
                         '--steps', '1', '--warmup', '1', '--cpu-sample', '1'], capture_output=True, text=True, timeout=900)
    assert cp.returncode == 0, cp.stderr[-2000:]
    lines = [l for l in cp.stdout.strip().splitlines() if l.startswith('{')]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d['impl'] == 'reference' and d['metric'] == 'walker.local-energies/sec' and d['higher_is_better'] is True
    assert d['value'] > 0 and d['unit'] == 'walker.local-energies/s' and d['steps'] == 1 and d['warmup'] == 1
    assert d['cpu_baseline']['kind'] == 'port' and d['cpu_baseline']['cores'] >= 1 and d['cpu_baseline']['value'] == d['value']
    assert d['e2e'] == {'value': d['value'], 'unit': d['unit'], 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}
    assert 'workload' in d['config'] and d['data'] == 'synthetic' and d['dtype'] == 'f64'


def test_dump_outputs_writes_float_arrays_and_samples_walkers_over_the_limit(tmp_path, monkeypatch):
    import numpy as np
    import torch

    import bench

    per_walker = {'E_loc': torch.arange(100, dtype=torch.float32), 'walkers': torch.zeros(100, 4, 3, dtype=torch.float64),
                  'hamil_V_el': torch.ones(100, dtype=torch.float32)}
    other = {'stat_energy_count': torch.tensor(100.0, dtype=torch.float64)}
    bench.dump_outputs(str(tmp_path / 'all'), per_walker, other)
    e = np.load(tmp_path / 'all' / 'E_loc.npy')
    assert e.dtype == np.float32 and np.array_equal(e, np.arange(100)) and not (tmp_path / 'all' / 'walker_index.npy').exists()
    assert np.load(tmp_path / 'all' / 'walkers.npy').dtype == np.float64 and np.load(tmp_path / 'all' / 'stat_energy_count.npy') == 100

    monkeypatch.setattr(bench, 'DUMP_LIMIT_BYTES', 4000)
    for d in ('a', 'b'):
        bench.dump_outputs(str(tmp_path / d), per_walker, other)
    files = sorted(os.listdir(tmp_path / 'a'))
    assert files == ['E_loc.npy', 'hamil_V_el.npy', 'stat_energy_count.npy', 'walker_index.npy', 'walkers.npy']
    assert sum(np.load(tmp_path / 'a' / f).nbytes for f in files) <= 4000
    idx = np.load(tmp_path / 'a' / 'walker_index.npy')
    assert 0 < len(idx) < 100 and np.array_equal(np.load(tmp_path / 'a' / 'E_loc.npy'), idx)
    for f in files:  # the sample is fixed: the same walkers every time
        assert np.array_equal(np.load(tmp_path / 'a' / f), np.load(tmp_path / 'b' / f))


def test_other_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK='1', WORLD_SIZE='2')
    cp = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2', '--workload',
                         'lih_paulinet', '--steps', '1', '--warmup', '0'], capture_output=True, text=True, timeout=300, env=env)
    assert cp.returncode == 0 and cp.stdout.strip() == ''
