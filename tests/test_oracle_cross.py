"""The independent restatement (oracle/port) against the reference's own object code (oracle/_ref) on a broad random
family of inputs: ragged shapes, sparse / scaled / wide matrices, heterogeneous intervals and latencies, every
selector.  This is what lets the port stand in as the checker wherever oracle/_ref is absent.  The reference's answers
are stored as digests in tests/golden/oracle_digests.json (written by tests/golden/make_golden_ref_outputs.py).  No GPU."""
import json

import numpy as np
import pytest
from conftest import GOLDEN, digest, stage_digest

from oracle import port

METHODS = ['mc', 'wmc', 'mc-dc', 'mc-pdc', 'wmc-dc', 'wmc-pdc']


def random_matrix(rng, n_in, n_out):
    kind = rng.choice(['dense', 'sparse', 'holes', 'fraction', 'wide', 'constant', 'diag'])
    bits = int(rng.integers(2, 9))
    W = rng.integers(-(2 ** (bits - 1)), 2 ** (bits - 1), size=(n_in, n_out)).astype(np.float64)
    if kind == 'sparse':
        W *= rng.random((n_in, n_out)) < 0.3
    elif kind == 'holes':  # whole rows / columns of zeros
        W[rng.random(n_in) < 0.3, :] = 0
        W[:, rng.random(n_out) < 0.3] = 0
    elif kind == 'fraction':
        W *= 2.0 ** -int(rng.integers(1, 6))
    elif kind == 'wide':
        W = rng.integers(-(2**11), 2**11, size=(n_in, n_out)).astype(np.float64)
    elif kind == 'constant':
        W[:] = float(rng.integers(-7, 8))
    elif kind == 'diag':
        W = np.eye(n_in, n_out) * float(rng.integers(1, 100))
    return np.ascontiguousarray(W, dtype=np.float32), kind


def random_intervals(rng, n_in):
    mode = rng.choice(['none', 'hetero', 'unsigned', 'some_zero'])
    if mode == 'none':
        return None
    q = np.zeros((n_in, 3), np.float32)
    for i in range(n_in):
        step = 2.0 ** int(rng.integers(-3, 3))
        lo, hi = sorted(int(v) for v in rng.integers(-200, 200, size=2))
        if mode == 'unsigned':
            lo = 0
            hi = abs(hi) + 1
        q[i] = (lo * step, hi * step, step)
        if mode == 'some_zero' and rng.random() < 0.3:
            q[i] = (0.0, 0.0, 1.0)
    return [tuple(float(v) for v in r) for r in q]


def random_latencies(rng, n_in):
    if rng.random() < 0.5:
        return None
    return [float(v) for v in rng.integers(0, 4, size=n_in)]


def shapes(rng):
    pick = rng.integers(0, 6)
    if pick == 0:
        return 1, int(rng.integers(1, 12))
    if pick == 1:
        return int(rng.integers(1, 12)), 1
    return int(rng.integers(2, 22)), int(rng.integers(2, 22))


def single_case(seed):
    rng = np.random.default_rng(7000 + seed)
    n_in, n_out = shapes(rng)
    W, kind = random_matrix(rng, n_in, n_out)
    kw = dict(
        method=str(rng.choice(METHODS + ['dummy'])),
        qintervals=random_intervals(rng, n_in),
        latencies=random_latencies(rng, n_in),
        adder_size=int(rng.choice([-1, 1, 3, 8])),
        carry_size=int(rng.choice([-1, 1, 4])),
    )
    return W, kind, kw


def full_case(seed):
    rng = np.random.default_rng(9000 + seed)
    n_in, n_out = shapes(rng)
    W, kind = random_matrix(rng, n_in, n_out)
    kw = dict(
        method0=str(rng.choice(METHODS)),
        method1=str(rng.choice(['auto'] + METHODS)),
        hard_dc=int(rng.choice([-1, 0, 1, 2, 5])),
        decompose_dc=int(rng.choice([-2, -1, 0, 1, 3])),
        qintervals=random_intervals(rng, n_in),
        latencies=random_latencies(rng, n_in),
        adder_size=int(rng.choice([-1, 2])),
        carry_size=int(rng.choice([-1, 3])),
        search_all_decompose_dc=bool(rng.integers(0, 2)),
    )
    return W, kind, kw


def helpers_case(seed):
    rng = np.random.default_rng(11000 + seed)
    n_in, n_out = shapes(rng)
    W, _ = random_matrix(rng, n_in, n_out)
    ints = rng.integers(-(2**20), 2**20, size=(int(rng.integers(1, 40)),)).astype(np.int32)
    Wi = np.round(W * 64).astype(np.float32)  # kernel_decompose works on the integer grid
    return W, ints, Wi


DECOMPOSE_DCS = (-2, -1, 0, 1, 2)


def helpers_outputs(mod, W, ints, Wi):
    """Every helper's arrays for one case, under the names the golden file stores them."""
    out = {}
    for center in (True, False):
        for name, a in zip(('csd', 's0', 's1'), mod.csd_decompose(W, center)):
            out[f'csd{int(center)}_{name}'] = a
    out['int_csd'] = mod.int_arr_to_csd(ints)
    for dc in DECOMPOSE_DCS:
        out[f'kd{dc}_m0'], out[f'kd{dc}_m1'] = mod.kernel_decompose(Wi, dc)
    return out


@pytest.fixture(scope='module')
def gold():
    return json.loads((GOLDEN / 'oracle_digests.json').read_text())


@pytest.mark.parametrize('seed', range(60))
def test_single_stage_random_family(gold, seed):
    W, kind, kw = single_case(seed)
    g = gold[f'single{seed}']
    assert digest([('kernel', W)]) == g['kernel'], 'not the matrix the reference answered for'
    assert stage_digest([port.solve_single(W, **kw)]) == g['result'], f'{kind} {W.shape} {kw["method"]}: differs from the reference'


@pytest.mark.parametrize('seed', range(40))
def test_full_solve_random_family(gold, seed):
    W, kind, kw = full_case(seed)
    g = gold[f'full{seed}']
    assert digest([('kernel', W)]) == g['kernel'], 'not the matrix the reference answered for'
    got = port.solve(W, **kw)
    assert len(got) == 2
    assert stage_digest(got) == g['result'], f'{kind} {W.shape} {kw}: differs from the reference'


@pytest.mark.parametrize('seed', range(20))
def test_helpers_random_family(gold, seed):
    W, ints, Wi = helpers_case(seed)
    g = gold[f'helpers{seed}']
    assert digest([('kernel', W)]) == g['kernel'], 'not the matrix the reference answered for'
    got = helpers_outputs(port, W, ints, Wi)
    assert digest(sorted(got.items())) == g['result'], 'differs from the reference'
    for dc in DECOMPOSE_DCS:
        assert np.array_equal(got[f'kd{dc}_m0'].astype(np.float64) @ got[f'kd{dc}_m1'].astype(np.float64), Wi), dc
