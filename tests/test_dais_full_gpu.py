"""The complete DAIS interpreter on the B200 (da4ml_b200.dais): every stored reference answer of
tests/golden/dais_full.npz bit for bit, in both slot regimes, at sample counts around the tile and chunk boundaries,
from host arrays and from CUDA tensors, with programs kept resident across calls, and the reference's error for a
lookup out of range.  On the adder graphs of the solver it equals the adder-only replay (dais_interp_run)."""
import numpy as np
import pytest
from conftest import GOLDEN
from test_dais_full import assert_answer, golden, stored_case

pytestmark = pytest.mark.gpu


@pytest.fixture
def dais(cuda_binary):
    from da4ml_b200 import dais as D

    D.set_shared_budget(0, 0)
    yield D
    D.set_shared_budget(0, 0)


def _check(got, want, tag):
    if isinstance(want, tuple) and want[0] == 'error':
        raise AssertionError(f'{tag}: expected the error {want[1]!r}')
    assert_answer(got, want, tag)


def test_every_stored_answer_in_the_default_regime(dais):
    z, names = golden()
    regimes = set()
    for name in names:
        prog, x, want = stored_case(z, name)
        p = dais.DaisProgram(prog)
        regimes.add(p.info['regime'])
        if isinstance(want, tuple) and want[0] == 'error':
            with pytest.raises(RuntimeError) as e:
                p.predict(x)
            assert str(e.value) == want[1], name
            continue
        _check(p.predict(x), want, name)
    assert regimes == {'shared', 'global'}  # the larger MLPs do not fit a CTA's shared memory


def test_every_stored_answer_in_the_global_regime_with_small_chunks(dais):
    dais.set_shared_budget(1, 300)
    z, names = golden()
    for name in names:
        prog, x, want = stored_case(z, name)
        p = dais.DaisProgram(prog)
        assert p.info['regime'] == 'global' and p.info['tile'] == 300
        if isinstance(want, tuple) and want[0] == 'error':
            with pytest.raises(RuntimeError) as e:
                p.predict(x)
            assert str(e.value) == want[1], name
            continue
        _check(p.predict(x), want, name + ' (global)')


@pytest.mark.parametrize('budget,chunk', [(0, 0), (0, 64), (1, 64)])
def test_sample_counts_around_tile_and_chunk_boundaries(dais, budget, chunk):
    dais.set_shared_budget(budget, chunk)
    z, _ = golden()
    for name in ('random0', 'lookup_tables', 'sort'):
        prog, x, want = stored_case(z, name)
        p = dais.DaisProgram(prog)
        T = p.info['tile']
        counts = {1, T - 1, T + 1, 65, 129, len(x)} if p.info['regime'] == 'shared' else {1, 63, 65, 129, len(x)}
        for n in sorted(c for c in counts if 0 < c <= len(x)):
            assert_answer(p.predict(x[:n]), want[:n], f'{name} n={n} {p.info}')
        assert p.predict(x[:0]).shape == (0, p.n_out)


def test_cuda_tensor_equals_host_path(dais):
    import torch

    z, _ = golden()
    for name in ('mlp_16_64_32_32_5', 'mlp_64_128_128_10', 'lookup_tables', 'random5'):
        prog, x, want = stored_case(z, name)
        p = dais.DaisProgram(prog)
        host = p.predict(x)
        xd = torch.from_numpy(x).cuda()
        dev = p.predict(xd)
        assert dev.is_cuda and dev.dtype == torch.float64
        assert np.array_equal(dev.cpu().numpy().view(np.uint64), host.view(np.uint64)), name
        _check(host, want, name)


def test_resident_programs_over_many_calls(dais):
    z, _ = golden()
    pa, xa, wa = stored_case(z, 'mlp_16_64_32_32_5')
    pb, xb, wb = stored_case(z, 'random7')
    a, b = dais.DaisProgram(pa), dais.DaisProgram(pb)  # two programs resident at once
    for _ in range(3):
        _check(a.predict(xa), wa, 'a')
        _check(b.predict(xb), wb, 'b')
    del a
    _check(b.predict(xb), wb, 'b after a was freed')


def test_lookup_overrun_reports_the_first_offending_sample_and_recovers(dais):
    from da4ml_b200.dais import run_interp

    z, _ = golden()
    prog, x, want = stored_case(z, 'lookup_overrun')
    assert want[0] == 'error'
    p = dais.DaisProgram(prog)
    for _ in range(2):
        with pytest.raises(RuntimeError) as e:
            p.predict(x)
        assert str(e.value) == want[1]
    with pytest.raises(RuntimeError) as e:
        run_interp(prog, x)
    assert str(e.value) == want[1]
    ok = np.zeros((3, 1))  # input 0: in range for both tables
    assert p.predict(ok).shape == (3, 2)
    prog2, x2, want2 = stored_case(z, 'lookup_tables')
    _check(run_interp(prog2, x2), want2, 'next program after the error')


def test_adder_graphs_equal_the_adder_only_replay(dais, cuda_binary):
    from test_dais_replay import cuda_replay_inputs

    gold = np.load(GOLDEN / 'dais_ref.npz')
    n = 0
    for tag, sol, x in cuda_replay_inputs():
        prog = sol.to_binary()
        got = dais.DaisProgram(prog).predict(x)
        want = gold['cuda__' + tag.replace('/', '__')]
        assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), tag
        assert np.array_equal(got.view(np.uint64), cuda_binary.dais_interp_run(prog, x).view(np.uint64)), tag
        n += 1
    assert n >= 10
