"""bench.py's reference arm runs on CPU: check the JSON contract (keys, units, reference-arm extras).  No GPU."""
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, str(ROOT / 'bench.py'), '--impl', 'reference', '--size', '16', '--steps', '1', '--warmup', '0'],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ('impl', 'metric', 'value', 'unit', 'n_gpus', 'steps', 'warmup', 'ms_per_step', 'higher_is_better', 'scaling',
                'vs_baseline', 'dtype', 'data', 'config', 'cpu_baseline', 'e2e'):
        assert key in line, key
    assert line['impl'] == 'reference' and line['unit'] == 'matrices/s' and line['higher_is_better'] is True
    assert line['metric'] == 'cmvm_solve_throughput_16x16_int8' and 'workload' in line['config']
    assert line['cpu_baseline']['kind'] in ('reference', 'port') and line['cpu_baseline']['cores'] >= 1
    assert line['e2e']['h2d_bytes_per_step'] == 0 and line['e2e']['d2h_bytes_per_step'] == 0
    assert line['vs_baseline'] is None


def test_default_metric_is_the_baseline_metric():
    sys.path.insert(0, str(ROOT))
    import bench

    assert bench.metric_name(256, 8) == bench.METRIC == 'cmvm_solve_throughput_256x256_int8'
    spec = json.loads((ROOT / 'BASELINE.json').read_text())
    assert '256' in spec['metric'] and 'int8' in spec['metric']


def test_dump_outputs_writes_result_arrays_as_float(tmp_path):
    """--dump-outputs: every result array of the step as float64 (integers) / float32 (ops_f); above the byte limit the
    same seeded sample of rows in every run."""
    sys.path.insert(0, str(ROOT))
    from types import SimpleNamespace

    import bench
    from conftest import load_golden

    _, stages = load_golden('int_32x32_int8_default')
    step = [SimpleNamespace(stages=stages)]
    bench.dump_outputs(tmp_path / 'all', step, '', bench.DUMP_LIMIT)
    for i, st in enumerate(stages):
        for k in bench.STAGE_KEYS:
            a = np.load(tmp_path / 'all' / f'm0_s{i}_{k}.npy')
            assert a.dtype == (np.float32 if k == 'ops_f' else np.float64)
            assert np.array_equal(a, st[k]), k
    limit = sum(np.asarray(st[k]).size * 8 for st in stages for k in bench.STAGE_KEYS) // 4
    for run in ('a', 'b'):
        bench.dump_outputs(tmp_path / run, step, 'x_', limit)
    files = sorted(p.name for p in (tmp_path / 'a').iterdir())
    assert len(files) == 2 * len(bench.STAGE_KEYS) and sum((tmp_path / 'a' / f).stat().st_size for f in files) < limit + 128 * len(files)
    for f in files:
        assert np.array_equal(np.load(tmp_path / 'a' / f), np.load(tmp_path / 'b' / f))
    ops = np.load(tmp_path / 'a' / 'x_m0_s0_ops_i.npy')
    assert 0 < len(ops) < len(stages[0]['ops_i']) and all(any((row == o).all() for o in stages[0]['ops_i']) for row in ops)
