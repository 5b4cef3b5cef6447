"""Profiling and value capture of DAIS programs (DaisProgram.profile / .values; the every-op variant of
csrc/host_dais.cuh and the observers of csrc/dais_exec.cuh) without a GPU: the variant compiles every op with its
folded dtype range, arguments are checked before any device call, and the kernel source run under the SIMT shim
(tests/simt/sim_dais_profile.cc) equals the reference interpreter's per-op values and the statistics derived from them
(tests/golden/dais_profile.npz, written by tests/golden/make_golden_dais_profile.py) in both slot regimes.  The GPU
half is tests/test_dais_profile_gpu.py."""
import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest
from conftest import GOLDEN, digest
from test_dais_full import golden, program_words, special_inputs, stored_case

SIMT = Path(__file__).resolve().parent / 'simt'
HEAD = 40  # rows of values stored whole for the large cases (what the CPU simulation can afford to run)
I64_MIN, I64_MAX = np.iinfo(np.int64).min, np.iinfo(np.int64).max


# ---- cases (also used by the golden generator) ------------------------------------------------------------------------
def narrow_program():
    """Two signed 4-bit inputs into ops whose declared dtypes are too narrow for their values: an adder (w = 3), an
    unsigned subtraction (w = 4), a multiplication (w = 6), and a quantize (w = 2) that wraps by design."""
    ops = [[-1, 0, -1, 0, 0, 1, 3, 0], [-1, 1, -1, 0, 0, 1, 3, 0], [0, 0, 1, 0, 0, 1, 2, 0], [1, 0, 1, 1, 0, 0, 4, 0],
           [3, 2, -1, 0, 0, 1, 1, 0], [7, 0, 1, 0, 0, 1, 5, 0], [0, 2, 5, 0, 0, 1, 9, 0]]  # fmt: skip
    return program_words([0, 0], [4, 6], [0, 0], [0, 0], ops)


def profile_cases():
    """{name: (program, inputs)}: every program of dais_full.npz with its stored inputs, the narrow program, and the
    smallest traced MLP fed inputs scaled so that its hidden quantize(1, 4, 2) wraps often."""
    z, names = golden()
    cases = {}
    for name in names:
        prog, x, _ = stored_case(z, name)
        cases[name] = (prog, x)
    rng = np.random.default_rng(5)
    cases['narrow'] = (narrow_program(), rng.integers(-8, 8, size=(200, 2)).astype(np.float64))
    prog, _, _ = stored_case(z, 'mlp_16_64_32_32_5')
    cases['mlp_wraps'] = (prog, special_inputs(77, 4096, 16) * 16.0)
    return cases


def profile_golden():
    return np.load(GOLDEN / 'dais_profile.npz')


def stats_of(g, name, head=False):
    k = f'{name}__head_' if head else f'{name}__'
    return g[k + 'stats'], tuple(int(v) for v in g[k + 'first'])


def values_digest(v):
    return digest([('v', v)])


# ---- the kernel source under the SIMT shim --------------------------------------------------------------------------
_sim = None


def sim():
    global _sim
    if _sim is None:
        lib = SIMT / 'libsim_dais_profile.so'
        csrc = SIMT.parents[1] / 'da4ml_b200' / 'csrc'
        srcs = [SIMT / 'sim_dais_profile.cc', SIMT / 'simt.h', csrc / 'dais_exec.cuh', csrc / 'host_dais.cuh']
        if not lib.exists() or lib.stat().st_mtime < max(p.stat().st_mtime for p in srcs):
            tmp = lib.with_name(f'.{lib.name}.{os.getpid()}')
            gxx = '/usr/bin/g++' if Path('/usr/bin/g++').exists() else 'g++'
            subprocess.run([gxx, '-O2', '-std=c++17', '-ffp-contract=off', '-fPIC', '-shared', '-w', str(SIMT / 'sim_dais_profile.cc'), '-o', str(tmp)], check=True)
            os.replace(tmp, lib)
        L = C.CDLL(str(lib))
        L.sim_dais_profile_last_error.restype = C.c_char_p
        L.sim_dais_variant.argtypes = [C.c_void_p, C.c_longlong, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        L.sim_dais_profile.argtypes = [C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_longlong, C.c_longlong, C.c_int, C.c_void_p, C.c_void_p]
        L.sim_dais_capture.argtypes = [C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_void_p, C.c_int, C.c_void_p, C.c_longlong, C.c_longlong, C.c_int]
        _sim = L
    return _sim


def _err():
    return RuntimeError(sim().sim_dais_profile_last_error().decode())


def sim_variant(prog, ops=()):
    prog = np.ascontiguousarray(prog, np.int32)
    ops = np.ascontiguousarray(ops, np.int32)
    info = np.zeros(8, np.int64)
    n_ops = int(prog[4])
    side = np.zeros((max(n_ops, 1), 6), np.int64)
    cols = np.zeros(max(len(ops), 1), np.int32)
    if sim().sim_dais_variant(prog.ctypes.data, prog.size, ops.ctypes.data, len(ops), info.ctypes.data, side.ctypes.data, cols.ctypes.data):
        raise _err()
    n_instr, n_cols = int(info[1]), int(info[3])
    return dict(n_ops=int(info[0]), n_instr=n_instr, n_slots=int(info[2])), side[:n_instr], cols[:n_cols]


def sim_profile(prog, x, shared_bytes=227 * 1024, chunk=1 << 20, cta_threads=32):
    prog = np.ascontiguousarray(prog, np.int32)
    x = np.ascontiguousarray(x, np.float64)
    stats = np.zeros((4, int(prog[4])), np.int64)
    first = np.zeros(2, np.int64)
    rc = sim().sim_dais_profile(prog.ctypes.data, prog.size, x.ctypes.data, x.shape[0], shared_bytes, chunk, cta_threads, stats.ctypes.data, first.ctypes.data)
    if rc < 0:
        raise _err()
    return stats, (int(first[0]), int(first[1])), rc


def sim_values(prog, x, ops, shared_bytes=227 * 1024, chunk=1 << 20, cta_threads=32):
    prog = np.ascontiguousarray(prog, np.int32)
    x = np.ascontiguousarray(x, np.float64)
    ops = np.ascontiguousarray(ops, np.int32)
    out = np.zeros((x.shape[0], len(ops)), np.int64)
    rc = sim().sim_dais_capture(prog.ctypes.data, prog.size, x.ctypes.data, x.shape[0], ops.ctypes.data, len(ops), out.ctypes.data, shared_bytes, chunk, cta_threads)
    if rc < 0:
        raise _err()
    return out, rc


# ---- the compiled variant ---------------------------------------------------------------------------------------------
# (is_signed, integers, fractionals) -> declared range: w <= 0, 1, 63, 64, > 64, signed and unsigned
RANGES = [((1, -3, 1), 0, 0), ((0, 0, 0), 0, 0), ((1, 0, 0), -1, 0), ((0, 1, 0), 0, 1), ((1, 60, 2), -(2**62), 2**62 - 1), ((0, 61, 2), 0, 2**63 - 1),
          ((1, 40, 23), I64_MIN, I64_MAX), ((0, 40, 24), 0, I64_MAX), ((1, 100, 7), I64_MIN, I64_MAX), ((0, 70, 7), 0, I64_MAX),
          ((1, 2**31 - 1, 2**31 - 1), I64_MIN, I64_MAX)]  # fmt: skip


def test_variant_folds_every_dtype_range():
    """w = is_signed + integers + fractionals in 64-bit, the last row overflowing the reference's int32 width."""
    ops = [[5, -1, -1, 0, 0, *dt, ] for dt, _, _ in RANGES]
    prog = program_words([], [0], [0], [0], ops)
    info, side, _ = sim_variant(prog)
    assert info['n_instr'] == len(RANGES)
    for i, (dt, lo, hi) in enumerate(RANGES):
        assert tuple(side[i, [0, 3, 4, 5]]) == (i, 0, lo, hi), dt


def test_variant_compiles_every_op_and_captures_dead_ones():
    """Predict skips ops nobody reads; the every-op variant runs all of them, in program order, with no output
    instructions, and marks the quantizing kinds.  Captured columns follow the request, duplicates included."""
    from test_dais_full import sim_compile

    z, _ = golden()
    prog = z['random3__program']
    _, slots = sim_compile(prog)
    dead = np.flatnonzero(slots < 0)
    assert dead.size  # the random program has ops nobody reads
    n_ops = int(prog[4])
    want_ops = [int(dead[0]), 0, int(dead[0]), n_ops - 1]
    info, side, cols = sim_variant(prog, want_ops)
    assert info['n_instr'] == n_ops and np.array_equal(side[:, 0], np.arange(n_ops))
    opcodes = prog[6 + int(prog[2]) + 3 * int(prog[3]) :][: 8 * n_ops].reshape(-1, 8)[:, 0]
    assert np.array_equal(side[:, 3], np.isin(opcodes, [-1, 2, -2, 3, -3, 6, -6]).astype(np.int64))
    got = {}
    for i in range(n_ops):
        for j in cols[side[i, 1] : side[i, 1] + side[i, 2]]:
            got[int(j)] = i
    assert got == dict(enumerate(want_ops))
    # slots are still assigned by liveness: keeping the dead ops costs at most one slot
    assert info['n_slots'] <= int(slots.max()) + 2
    with pytest.raises(RuntimeError, match='op index -1 out of range'):
        sim_variant(prog, [-1])


# ---- argument validation ------------------------------------------------------------------------------------------------
def _unloaded(prog):
    """A DaisProgram with the info of `prog` and no device handle: a call that reached the library would fail."""
    from da4ml_b200.dais import INFO_FIELDS, DaisProgram

    p = DaisProgram.__new__(DaisProgram)
    p._h, p._words = None, np.ascontiguousarray(prog, np.int32)
    p.info = dict.fromkeys(INFO_FIELDS, 0) | dict(n_in=int(prog[2]), n_out=int(prog[3]), n_ops=int(prog[4]))
    return p


def test_values_rejects_bad_op_indices_before_any_device_call():
    p = _unloaded(narrow_program())
    assert p.dtypes.tolist() == [[1, 3, 0], [1, 3, 0], [1, 2, 0], [0, 4, 0], [1, 1, 0], [1, 5, 0], [1, 9, 0]]
    x = np.zeros((3, 2))
    for ops in ([7], [-1], [0, 99], [[0, 1]], [0.5]):
        with pytest.raises(ValueError):
            p.values(x, ops)
    with pytest.raises(ValueError, match='not divisible'):
        p.profile(np.zeros(5))


def test_abi_rejects_bad_arguments_before_any_device_call():
    import da4ml_b200._binary as B

    L = B._L
    stats, first = np.zeros(8, np.int64), np.zeros(2, np.int64)
    assert L.da4ml_dais_profile(None, None, 1, B._ip(stats), B._ip(first)) == 1
    assert L.da4ml_dais_profile_device(None, None, 1, B._ip(stats), B._ip(first)) == 1
    assert L.da4ml_dais_capture(None, None, 1, None, 0, None) == 1
    assert L.da4ml_dais_capture_device(None, None, 1, None, 0, None) == 1


def test_width_needed():
    from da4ml_b200.dais import width_needed

    lo = np.array([0, 0, 1, -1, -4, -5, 0, I64_MIN, 3, I64_MAX])
    hi = np.array([0, 1, 255, 0, 3, 0, I64_MAX, I64_MAX, -3, I64_MIN])
    assert width_needed(lo, hi).tolist() == [0, 1, 8, 1, 3, 4, 63, 64, 0, 0]


# ---- the kernel source under the SIMT shim -------------------------------------------------------------------------------
SMALL = [f'random{s}' for s in range(24)] + ['relu_quantize', 'neg_quantize', 'const_add', 'const', 'maximum', 'sort', 'multiply', 'bit_and_xor', 'bit_not',
                                              'lookup', 'lookup_tables', 'narrow']  # fmt: skip
REGIMES = ((0, {}), (1, dict(shared_bytes=0, chunk=37, cta_threads=32)), (1, dict(shared_bytes=0, chunk=100, cta_threads=64)))


def test_golden_file_covers_the_semantics():
    g = profile_golden()
    stats, first = stats_of(g, 'narrow')
    assert stats[2].sum() > 0 and first != (-1, -1)
    stats, _ = stats_of(g, 'mlp_wraps')
    assert stats[3].sum() > 1000
    for name in SMALL + ['mlp_16_64_32_32_5', 'mlp_64_128_128_10']:
        assert f'{name}__stats' in g.files or f'{name}__error' in g.files, name
    assert sum(f'{name}__stats' in g.files for name in SMALL) > 30
    assert 'lookup_overrun__error' in g.files


@pytest.mark.parametrize('name', SMALL)
def test_simulated_profile_and_values_equal_the_reference(name):
    """Sample counts of 200: a partial last warp; chunks of 37 and 100 samples in the global regime cross warps."""
    g = profile_golden()
    prog, x = profile_cases()[name]
    if f'{name}__error' in g.files:  # a lookup out of range (NaN inputs wrap to values outside the dtype's range)
        for _, kw in REGIMES:
            for run in (lambda: sim_profile(prog, x, **kw), lambda: sim_values(prog, x, [0], **kw)):
                with pytest.raises(RuntimeError) as e:
                    run()
                assert str(e.value) == str(g[f'{name}__error']), name
        return
    stats, first = stats_of(g, name)
    vals = g[f'{name}__values']
    n_ops = int(prog[4])
    for regime, kw in REGIMES:
        got, got_first, ran = sim_profile(prog, x, **kw)
        assert ran == regime
        assert np.array_equal(got, stats) and got_first == first, f'{name} {kw}'
        v, _ = sim_values(prog, x, np.arange(n_ops), **kw)
        assert np.array_equal(v, vals), f'{name} {kw}'
    sel = np.array([n_ops - 1, 0, n_ops - 1])
    v, _ = sim_values(prog, x[:33], sel)
    assert np.array_equal(v, vals[:33][:, sel])


def test_simulated_profile_on_a_traced_mlp():
    """The head rows of the traced MLP fed wrapping inputs: the shared regime at 32 samples per CTA, and the global one."""
    g = profile_golden()
    prog, x = profile_cases()['mlp_wraps']
    stats, first = stats_of(g, 'mlp_wraps', head=True)
    assert stats[3].sum() > 0
    from test_dais_full import sim_compile

    info, _ = sim_compile(prog)
    n_ops = int(prog[4])
    for kw in (dict(shared_bytes=8 * (info['n_slots'] + 1) * 32), dict(shared_bytes=0, chunk=33)):
        got, got_first, _ = sim_profile(prog, x[:HEAD], **kw)
        assert np.array_equal(got, stats) and got_first == first, kw
    v, _ = sim_values(prog, x[:HEAD], np.arange(n_ops), shared_bytes=0, chunk=64)
    assert np.array_equal(v, g['mlp_wraps__values_head'])


def test_simulated_lookup_overrun_raises_the_reference_message():
    g = profile_golden()
    prog, x = profile_cases()['lookup_overrun']
    want = str(g['lookup_overrun__error'])
    for kw in (dict(), dict(shared_bytes=0, chunk=7)):
        with pytest.raises(RuntimeError) as e:
            sim_profile(prog, x, **kw)
        assert str(e.value) == want
        with pytest.raises(RuntimeError) as e:
            sim_values(prog, x, [0], **kw)
        assert str(e.value) == want


def test_stored_values_agree_with_the_reference_build():
    """The stored values are what the reference interpreter built from its sources (oracle/_ref) gives today."""
    from oracle import dais_ref

    if not dais_ref.available():
        pytest.skip('oracle/_ref is not built')
    import sys

    sys.path.insert(0, str(GOLDEN))
    from make_golden_dais_profile import reference_values

    g = profile_golden()
    for name in ('narrow', 'random0', 'sort'):
        prog, x = profile_cases()[name]
        assert np.array_equal(reference_values(prog, x), g[f'{name}__values']), name
