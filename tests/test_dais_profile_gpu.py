"""Profiling and value capture of DAIS programs on the B200 (DaisProgram.profile / .values): every stored case of
tests/golden/dais_profile.npz bit for bit in the default regime and in the global regime with small chunks, CUDA
tensors against host arrays, the reference's lookup error, predict unchanged by profiling, and profile against numpy
reductions of the captured values."""
import hashlib

import numpy as np
import pytest
from test_dais_profile import HEAD, profile_cases, profile_golden, stats_of

pytestmark = pytest.mark.gpu


@pytest.fixture
def dais(cuda_binary):
    from da4ml_b200 import dais as D

    D.set_shared_budget(0, 0)
    yield D
    D.set_shared_budget(0, 0)


def _values_digest(p, x, n_ops, batch):
    """conftest.digest([('v', values)]) of all ops' values, computed in sample batches."""
    h = hashlib.sha256()
    h.update(f'v {np.dtype(np.int64).str} {(len(x), n_ops)}'.encode())
    for b0 in range(0, len(x), batch):
        h.update(np.ascontiguousarray(p.values(x[b0 : b0 + batch], np.arange(n_ops))).tobytes())
    return h.hexdigest()


def _declared_range(signed, w):
    if w <= 0:
        return 0, 0
    if w >= 64:
        return (-(2**63) if signed else 0), 2**63 - 1
    return (-(2 ** (w - 1)), 2 ** (w - 1) - 1) if signed else (0, 2**w - 1)


def _check_case(p, name, prog, x, g, tag):
    n_ops = int(prog[4])
    if f'{name}__error' in g.files:
        for run in (lambda: p.profile(x), lambda: p.values(x, [0])):
            with pytest.raises(RuntimeError) as e:
                run()
            assert str(e.value) == str(g[f'{name}__error']), tag
        return
    stats, first = stats_of(g, name)
    r = p.profile(x)
    assert r.n == len(x)
    got = np.stack([r.min, r.max, r.outside, r.wrapped])
    assert np.array_equal(got, stats) and r.first_outside == first, tag
    assert np.array_equal(r.width_declared, p.dtypes.sum(axis=1))
    from da4ml_b200.dais import width_needed

    assert np.array_equal(r.width_needed, width_needed(stats[0], stats[1])), tag
    if f'{name}__values' in g.files:
        assert np.array_equal(p.values(x, np.arange(n_ops)), g[f'{name}__values']), tag
    else:
        assert _values_digest(p, x, n_ops, max(1, (1 << 27) // (8 * n_ops))) == str(g[f'{name}__values_digest']), tag
        if f'{name}__values_head' in g.files:
            assert np.array_equal(p.values(x[:HEAD], np.arange(n_ops)), g[f'{name}__values_head']), tag


def test_every_stored_case_in_the_default_regime(dais):
    g = profile_golden()
    regimes = set()
    for name, (prog, x) in profile_cases().items():
        p = dais.DaisProgram(prog)
        regimes.add(p.info['regime'])
        _check_case(p, name, prog, x, g, name)
    assert regimes == {'shared', 'global'}


def test_every_stored_case_in_the_global_regime_with_small_chunks(dais):
    dais.set_shared_budget(1, 300)
    g = profile_golden()
    for name, (prog, x) in profile_cases().items():
        p = dais.DaisProgram(prog)
        assert p.info['regime'] == 'global' and p.info['tile'] == 300
        _check_case(p, name, prog, x, g, name + ' (global, chunks of 300)')


def test_cuda_tensor_equals_host_path(dais):
    import torch

    cases = profile_cases()
    for name in ('mlp_wraps', 'mlp_64_128_128_10', 'narrow', 'random5', 'lookup_tables'):
        prog, x = cases[name]
        p = dais.DaisProgram(prog)
        xd = torch.from_numpy(x).cuda()
        a, b = p.profile(x), p.profile(xd)
        for k in ('min', 'max', 'outside', 'wrapped', 'width_needed'):
            assert np.array_equal(getattr(a, k), getattr(b, k)), (name, k)
        assert a.first_outside == b.first_outside and a.n == b.n
        ops = np.array([int(prog[4]) - 1, 0, 3, 0])
        vh = p.values(x, ops)
        vd = p.values(xd, ops)
        assert vd.is_cuda and vd.dtype == torch.int64
        assert np.array_equal(vd.cpu().numpy(), vh), name


def test_lookup_overrun_raises_the_reference_message(dais):
    import torch

    g = profile_golden()
    prog, x = profile_cases()['lookup_overrun']
    want = str(g['lookup_overrun__error'])
    p = dais.DaisProgram(prog)
    for arg in (x, torch.from_numpy(x).cuda()):
        for run in (lambda: p.profile(arg), lambda: p.values(arg, [1, 2])):
            with pytest.raises(RuntimeError) as e:
                run()
            assert str(e.value) == want
    ok = np.zeros((3, 1))
    assert p.profile(ok).n == 3 and p.values(ok, [3]).shape == (3, 1)


def test_predict_is_unchanged_by_profiling(dais):
    from test_dais_full import assert_answer, golden, stored_case

    z, _ = golden()
    for name in ('mlp_16_64_32_32_5', 'mlp_64_128_128_10', 'random7', 'lookup_tables'):
        prog, x, want = stored_case(z, name)
        p = dais.DaisProgram(prog)
        before = p.predict(x)
        assert_answer(before, want, name)
        p.profile(x)
        p.values(x[:100], [0, 1])
        after = p.predict(x)
        assert np.array_equal(before.view(np.uint64), after.view(np.uint64)), name


def test_profile_equals_reductions_of_the_values(dais):
    """numpy reductions of values(x, every op) are profile(x), on the random programs and on fresh inputs."""
    from test_dais_full import N_RANDOM, special_inputs

    from da4ml_b200.dais import width_needed

    g = profile_golden()
    cases = profile_cases()
    for s in range(N_RANDOM):
        name = f'random{s}'
        prog, _ = cases[name]
        if f'{name}__error' in g.files:
            continue
        x = special_inputs(1000 + s, 777, int(prog[2]))
        x[np.isnan(x)] = 0.5  # no lookup error from a NaN wrapped out of range
        p = dais.DaisProgram(prog)
        try:
            v = p.values(x, np.arange(p.n_ops))
        except RuntimeError:
            continue
        r = p.profile(x)
        rng = [_declared_range(sg, i + f + (sg != 0)) for sg, i, f in p.dtypes.tolist()]
        lo, hi = (np.array(c, np.int64) for c in zip(*rng))
        out = (v < lo) | (v > hi)
        assert np.array_equal(r.min, v.min(axis=0)) and np.array_equal(r.max, v.max(axis=0)), name
        assert np.array_equal(r.outside, out.sum(axis=0)), name
        rows = np.flatnonzero(out.any(axis=1))
        assert r.first_outside == ((int(rows[0]), int(np.flatnonzero(out[rows[0]])[0])) if rows.size else (-1, -1)), name
        assert np.array_equal(r.width_needed, width_needed(v.min(axis=0), v.max(axis=0)))
