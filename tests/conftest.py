import hashlib
import sys
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

GOLDEN = ROOT / 'tests' / 'golden'
STAGE_KEYS = ['inp_shifts', 'out_idxs', 'out_shifts', 'out_negs', 'ops_i', 'ops_f']


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run on the B200 box with -m gpu)')


def int_matrix(n_in, n_out, bits, seed):
    rng = np.random.default_rng(seed)
    return rng.integers(-(2 ** (bits - 1)), 2 ** (bits - 1), size=(n_in, n_out)).astype(np.float32)


def assert_stage_equal(a, b, tag=''):
    """Bit-exact comparison of two stage dicts (integer arrays and float32 arrays alike)."""
    for k in STAGE_KEYS:
        x, y = np.asarray(a[k]), np.asarray(b[k])
        assert x.shape == y.shape, f'{tag}{k}: shape {x.shape} != {y.shape}'
        if x.dtype.kind == 'f':
            assert np.array_equal(x.view(np.uint32), y.astype(np.float32).view(np.uint32)), f'{tag}{k} differs'
        else:
            assert np.array_equal(x, y), f'{tag}{k} differs'


def digest(named_arrays):
    """SHA-256 over (name, dtype, shape, bytes) of each array: how a golden file stores an answer it does not keep whole."""
    h = hashlib.sha256()
    for name, a in named_arrays:
        a = np.ascontiguousarray(a)
        h.update(f'{name} {a.dtype.str} {a.shape}'.encode())
        h.update(a.tobytes())
    return h.hexdigest()


def stage_digest(stages):
    return digest((f's{i}_{k}', st[k]) for i, st in enumerate(stages) for k in STAGE_KEYS)


def golden_cases(full_only=True):
    import json

    idx = json.loads((GOLDEN / 'index.json').read_text())
    return {k: v for k, v in idx.items() if v['full'] or not full_only}


def load_golden(name):
    z = np.load(GOLDEN / f'{name}.npz')
    n_st = len({k.split('_')[0] for k in z.files if k[0] == 's' and k[1].isdigit()})
    stages = [{k: z[f's{i}_{k}'] for k in STAGE_KEYS} for i in range(n_st)]
    extra = {k: z[k] for k in z.files if not (k[0] == 's' and k[1].isdigit())}
    return extra, stages


@pytest.fixture(scope='session')
def cuda_binary():
    import da4ml_b200._binary as B

    info = B.device_info()
    if info['cuda_devices'] < 1:
        pytest.fail('a test marked gpu is running without a CUDA device')
    return B
