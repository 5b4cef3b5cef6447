"""The CPU checkers against the golden vectors (generated from the reference's own object code by
tests/golden/make_golden.py) and against each other.  No GPU needed."""
import json

import numpy as np
import pytest
from conftest import GOLDEN, assert_stage_equal, digest, golden_cases, int_matrix, load_golden, stage_digest

from oracle import port, ref

FULL = golden_cases()
SOLVE_CASES = sorted(k for k, v in FULL.items() if not v.get('single'))
SINGLE_CASES = sorted(k for k, v in FULL.items() if v.get('single'))


@pytest.mark.parametrize('name', SOLVE_CASES)
def test_port_matches_golden_solve(name):
    extra, stages = load_golden(name)
    got = port.solve(extra['kernel'], **FULL[name]['kwargs'])
    assert len(got) == len(stages) == 2
    for i, (a, b) in enumerate(zip(got, stages)):
        assert_stage_equal(a, b, f'{name} stage{i} ')


@pytest.mark.parametrize('name', SINGLE_CASES)
def test_port_matches_golden_single(name):
    extra, stages = load_golden(name)
    kw = FULL[name]['kwargs']
    got = port.solve_single(extra['kernel'], kw['method'], extra['qint'], extra['lat'], kw['adder_size'], kw['carry_size'])
    assert_stage_equal(got, stages[0], name + ' ')
    assert got['counters']['T'] == len(extra['pairs'])
    assert got['counters']['sum_F'] == int(extra['f_sizes'].sum())


@pytest.mark.skipif(not ref.available(), reason='oracle/_ref not built (it is compiled from the reference sources)')
@pytest.mark.parametrize('name', SOLVE_CASES)
def test_reference_matches_golden(name):
    extra, stages = load_golden(name)
    got = ref.solve(extra['kernel'], **FULL[name]['kwargs'])
    for i, (a, b) in enumerate(zip(got, stages)):
        assert_stage_equal(a, b, f'{name} stage{i} ')


def random_case(seed):
    rng = np.random.default_rng(100 + seed)
    n_in, n_out, bits = int(rng.integers(2, 20)), int(rng.integers(2, 20)), int(rng.integers(2, 9))
    W = int_matrix(n_in, n_out, bits, seed)
    kw = dict(
        method0=str(rng.choice(['mc', 'wmc', 'mc-dc', 'wmc-pdc'])),
        method1=str(rng.choice(['auto', 'mc', 'wmc'])),
        hard_dc=int(rng.choice([-1, 0, 1, 3])),
        decompose_dc=int(rng.choice([-2, -1, 0, 2])),
        adder_size=int(rng.choice([-1, 1, 4])),
        carry_size=int(rng.choice([-1, 2, 8])),
        search_all_decompose_dc=bool(rng.integers(0, 2)),
    )
    return W, kw


@pytest.mark.parametrize('seed', range(6))
def test_port_matches_reference_random(seed):
    """Against the digest of the reference's answer (tests/golden/oracle_digests.json, tests/golden/make_golden_ref_outputs.py)."""
    W, kw = random_case(seed)
    g = json.loads((GOLDEN / 'oracle_digests.json').read_text())[f'random{seed}']
    assert digest([('kernel', W)]) == g['kernel'], 'not the matrix the reference answered for'
    got = port.solve(W, **kw)
    assert len(got) == 2
    assert stage_digest(got) == g['result'], f'{kw}: differs from the reference'


@pytest.mark.parametrize('n,bits', [(2, 2), (4, 4), (8, 8)])
@pytest.mark.parametrize('dc', [-2, -1, 0, 1, 2])
def test_port_kernel_decompose_property(n, bits, dc):
    # reference tests/test_cmvm.py:31-35
    rng = np.random.default_rng(n * 10 + bits)
    kernel = np.round((rng.random((n, n)) - 0.5) * 2 ** (bits + 1)).astype(np.float32)
    m0, m1 = port.kernel_decompose(kernel, dc)
    assert np.all(m0.astype(np.float64) @ m1.astype(np.float64) == kernel)


def test_port_csd_property():
    # reference tests/test_cmvm.py:23-28
    rng = np.random.default_rng(3)
    kernel = np.round((rng.random((8, 8)) - 0.5) * 2**9).astype(np.float32)
    csd, s0, s1 = port.csd_decompose(kernel)
    recon = csd * (2.0 ** s0[:, None, None].astype(np.float64)) * (2.0 ** s1[None, :, None].astype(np.float64)) * (2.0 ** np.arange(csd.shape[-1])[None, None, :])
    assert np.all(recon.sum(-1) == kernel)


def test_golden_index_lists_large_cases():
    idx = json.loads((GOLDEN / 'index.json').read_text())
    for name in ('c2_64x64_int8_default', 'c4_128x128_int6_dc-1', '128x128_int8_dc-1'):
        assert name in idx and len(idx[name]['sha256']) == 64 and idx[name]['n_adders'] > 0
