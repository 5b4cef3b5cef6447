"""The complete DAIS interpreter (da4ml_b200.dais, csrc/host_dais.cuh + csrc/dais_exec.cuh) without a GPU: program
validation and the data-independent errors are raised before any device call, slots are assigned by liveness, and the
kernel source run under the SIMT shim (tests/simt/sim_dais.cc) equals the reference interpreter's stored answers
(tests/golden/dais_full.npz, written by tests/golden/make_golden_dais_full.py) bit for bit in both slot regimes.
The GPU half is tests/test_dais_full_gpu.py."""
import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np
import pytest
from conftest import GOLDEN, digest

SIMT = Path(__file__).resolve().parent / 'simt'
N_RANDOM = 24
MLP_NAMES = ['mlp_16_64_32_32_5', 'mlp_16_64_64_64_5', 'mlp_64_128_128_10']


# ---- programs and inputs (also used by the golden generator) ----------------------------------------------------------
def program_words(inp_shifts, out_idxs, out_shifts, out_negs, ops, tables=()):
    """DAIS int32 words (the CombLogic.to_binary layout) from their parts; ops: [n_ops][8] = (opcode, id0, id1,
    data_low, data_high, is_signed, integers, fractionals)."""
    ops = np.asarray(ops, np.int64).reshape(-1, 8)
    head = [1, 0, len(inp_shifts), len(out_idxs), len(ops), len(tables)]
    parts = [head, inp_shifts, out_idxs, out_shifts, out_negs, ops.ravel(), [len(t) for t in tables], *tables]
    return np.concatenate([np.asarray(p, np.int64).ravel() for p in parts]).astype(np.int32)


def random_program(seed):
    """A program over every opcode with what traced networks rarely contain: -6 and -9, REDUCE_OR / REDUCE_AND, width-1
    and unsigned conditions, negative quantize shifts, 64-bit constants, several lookup tables, unused outputs."""
    rng = np.random.default_rng(seed)
    n_in = int(rng.integers(2, 7))
    ops = []

    def dtype(small=False):
        k = int(rng.integers(0, 2))
        if small:
            return [k, int(rng.integers(0, 5)), int(rng.integers(0, 3))]
        if rng.random() < 0.08:
            return [k, int(rng.choice([0, 1])), 0]  # width 0..2: width-1 unsigned conditions, 1-bit values
        return [k, int(rng.integers(-2, 14)), int(rng.integers(-2, 9))]

    def word():
        return int(rng.integers(-(2**31), 2**31))

    wrapped = []  # ops whose values lie in their dtype's range: what a lookup indexes with
    for j in range(n_in):
        ops.append([-1, j, -1, 0, 0, *dtype(small=rng.random() < 0.4)])
        wrapped.append(j)
    tables = [rng.integers(-(2**31), 2**31, size=int(n)) for n in rng.integers(1, 40, size=int(rng.integers(1, 4)))]
    for _ in range(int(rng.integers(10, 60))):
        i = len(ops)
        pick = lambda: int(rng.integers(0, i))  # noqa: E731
        opc = int(rng.choice([0, 1, 2, -2, 3, -3, 4, 5, 6, -6, 7, 8, 9, -9, 10]))
        if opc in (0, 1):
            ops.append([opc, pick(), pick(), int(rng.integers(-4, 5)), 0, *dtype()])
        elif opc in (2, -2, 3, -3):
            ops.append([opc, pick(), -1, 0, 0, *dtype()])
            wrapped.append(i)
        elif opc in (4, 5):
            hi = int(rng.choice([0, -1, word()]))
            ops.append([opc, pick() if opc == 4 else -1, -1, word(), hi, *dtype()])
        elif opc in (6, -6):
            a, b, c = pick(), pick(), pick()
            dt = dtype()
            if rng.random() < 0.5:  # msb_mux needs shift0 = f_out - f0 or shift1 = f_out - f1 + data_high to be 0
                dt[2] = ops[a][7]
                dh = int(rng.integers(-3, 4))
            else:
                dh = ops[b][7] - dt[2]
            ops.append([opc, a, b, c, dh, *dt])
            wrapped.append(i)
        elif opc == 7:
            ops.append([7, pick(), pick(), 0, 0, *dtype()])
        elif opc == 8:
            cands = [w for w in wrapped if 0 < sum(ops[w][5:8]) <= 5]
            if not cands:
                continue
            a = int(rng.choice(cands))
            size = 2 ** sum(ops[a][5:8])
            t = int(rng.integers(0, len(tables)))
            if len(tables[t]) < size:
                tables.append(rng.integers(-(2**20), 2**20, size=size + int(rng.integers(0, 3))))
                t = len(tables) - 1
            ops.append([8, a, -1, t, -int(rng.integers(0, len(tables[t]) - size + 1)), *dtype()])  # index = v - zero - data_high
        elif opc in (9, -9):
            ops.append([opc, pick(), -1, int(rng.integers(0, 3)), 0, *dtype()])
        else:
            ops.append([10, pick(), pick(), int(rng.integers(-3, 4)), int(rng.integers(0, 4)) | (int(rng.integers(0, 3)) << 24), *dtype()])
    n_out = int(rng.integers(1, 9))
    out_idxs = rng.integers(n_in, len(ops), size=n_out)
    out_idxs[rng.random(n_out) < 0.1] = -1
    return program_words(rng.integers(-3, 4, size=n_in), out_idxs, rng.integers(-4, 5, size=n_out), rng.integers(0, 2, size=n_out), ops, tables)


def lookup_overrun_program():
    """Two lookups of one signed 4-bit input: op 1 runs out of its table for inputs below -6, op 2 for inputs above 3."""
    ops = [[-1, 0, -1, 0, 0, 1, 3, 0], [8, 0, -1, 0, 2, 1, 8, 0], [8, 0, -1, 1, 0, 1, 8, 0], [0, 1, 2, 0, 0, 1, 9, 0]]
    return program_words([0], [3, 1], [0, 0], [0, 1], ops, [np.arange(16) * 3 - 7, np.arange(12) * -5])


def special_inputs(seed, n, n_in):
    """In-range values, values that wrap around, +-0, NaN, +-inf and +-1e300 (and the int64 conversion edges)."""
    rng = np.random.default_rng(seed)
    x = rng.integers(-64, 64, size=(n, n_in)) / 4.0
    x[n // 4 : n // 2] = rng.normal(0, 1e4, size=(n // 2 - n // 4, n_in))
    specials = np.array([0.0, -0.0, np.nan, np.inf, -np.inf, 1e300, -1e300, 2.0**62, -(2.0**63), 2.0**63])
    m = rng.random((n, n_in)) < 0.06
    x[m] = rng.choice(specials, size=int(m.sum()))
    return x


def case_inputs(name, prog):
    """(seed, n_samples) of a stored case's inputs."""
    seed = sum(name.encode()) * 7 + len(name)
    if name.startswith('mlp_'):
        return seed, 8192
    if name == 'lookup_overrun':
        return seed, 40
    return seed, 200


def golden():
    z = np.load(GOLDEN / 'dais_full.npz')
    names = sorted({k.split('__')[0] for k in z.files})
    return z, names


def stored_case(z, name):
    """(program, inputs, expected) with the inputs rebuilt from their seed and checked against the stored digest;
    expected is an array, ('digest', str) or ('error', message)."""
    prog = z[f'{name}__program']
    seed, n = case_inputs(name, prog)
    x = special_inputs(seed, n, int(prog[2]))
    assert digest([('x', x)]) == str(z[f'{name}__input']), f'{name}: the inputs changed since the answers were stored'
    if f'{name}__output' in z.files:
        return prog, x, z[f'{name}__output']
    if f'{name}__digest' in z.files:
        return prog, x, ('digest', str(z[f'{name}__digest']))
    return prog, x, ('error', str(z[f'{name}__error']))


def assert_answer(got, want, tag):
    if isinstance(want, tuple):
        assert want[0] == 'digest', tag
        assert digest([('y', got)]) == want[1], tag
    else:
        assert got.dtype == np.float64 and got.shape == want.shape, tag
        assert np.array_equal(got.view(np.uint64), want.view(np.uint64)), tag


# ---- the kernel source under the SIMT shim --------------------------------------------------------------------------
_sim = None


def sim():
    global _sim
    if _sim is None:
        lib = SIMT / 'libsim_dais.so'
        srcs = [SIMT / 'sim_dais.cc', SIMT / 'simt.h', *sorted((SIMT.parents[1] / 'da4ml_b200' / 'csrc').glob('dais_exec.cuh')),
                SIMT.parents[1] / 'da4ml_b200' / 'csrc' / 'host_dais.cuh']  # fmt: skip
        if not lib.exists() or lib.stat().st_mtime < max(p.stat().st_mtime for p in srcs):
            tmp = lib.with_name(f'.{lib.name}.{os.getpid()}')
            gxx = '/usr/bin/g++' if Path('/usr/bin/g++').exists() else 'g++'
            subprocess.run([gxx, '-O2', '-std=c++17', '-ffp-contract=off', '-fPIC', '-shared', '-w', str(SIMT / 'sim_dais.cc'), '-o', str(tmp)], check=True)
            os.replace(tmp, lib)
        L = C.CDLL(str(lib))
        L.sim_dais_last_error.restype = C.c_char_p
        L.sim_dais_compile.argtypes = [C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p]
        L.sim_dais_run.argtypes = [C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_void_p, C.c_longlong, C.c_longlong, C.c_int]
        _sim = L
    return _sim


def sim_compile(prog):
    prog = np.ascontiguousarray(prog, np.int32)
    info = np.zeros(8, np.int64)
    slots = np.zeros(max(int(prog[4]), 1), np.int32)
    if sim().sim_dais_compile(prog.ctypes.data, prog.size, info.ctypes.data, slots.ctypes.data):
        raise RuntimeError(sim().sim_dais_last_error().decode())
    return dict(zip(['n_in', 'n_out', 'n_ops', 'n_tables', 'n_slots', 'n_instr', 'max_width'], (int(v) for v in info))), slots[: int(prog[4])]


def sim_run(prog, x, shared_bytes=227 * 1024, chunk=1 << 20, cta_threads=32):
    """Outputs of the simulated kernel and the regime it ran in (0 shared, 1 global)."""
    prog = np.ascontiguousarray(prog, np.int32)
    x = np.ascontiguousarray(x, np.float64)
    y = np.zeros((x.shape[0], int(prog[3])), np.float64)
    rc = sim().sim_dais_run(prog.ctypes.data, prog.size, x.ctypes.data, x.shape[0], y.ctypes.data, shared_bytes, chunk, cta_threads)
    if rc < 0:
        raise RuntimeError(sim().sim_dais_last_error().decode())
    return y, rc


# ---- tests ------------------------------------------------------------------------------------------------------------
def test_stored_answers_agree_with_the_reference_build():
    """Every stored answer is what the reference interpreter built from its sources (oracle/_ref) answers today."""
    from oracle import dais_ref

    if not dais_ref.available():
        pytest.skip('oracle/_ref is not built')
    z, names = golden()
    for name in names:
        prog, x, want = stored_case(z, name)
        if isinstance(want, tuple) and want[0] == 'error':
            with pytest.raises(RuntimeError) as e:
                dais_ref.run(prog, x)
            assert str(e.value) == want[1], name
        else:
            assert_answer(dais_ref.run(prog, x), want, name)


def test_golden_file_covers_every_opcode():
    z, names = golden()
    assert set(MLP_NAMES) < set(names) and sum(n.startswith('random') for n in names) == N_RANDOM
    seen = set()
    for name in names:
        prog = z[f'{name}__program']
        n_in, n_out, n_ops = (int(v) for v in prog[2:5])
        seen |= set(prog[6 + n_in + 3 * n_out :][: 8 * n_ops].reshape(-1, 8)[:, 0].tolist())
    assert seen == {-1, 0, 1, 2, -2, 3, -3, 4, 5, 6, -6, 7, 8, 9, -9, 10}
    traced = {-1, 0, 1, 2, -2, 3, -3, 4, 5, 6, 7, 8, 9, 10}  # what the tracing front-end emitted
    seen_traced = set()
    for name in names:
        if not name.startswith('random') and name != 'lookup_overrun':
            prog = z[f'{name}__program']
            n_in, n_out, n_ops = (int(v) for v in prog[2:5])
            seen_traced |= set(prog[6 + n_in + 3 * n_out :][: 8 * n_ops].reshape(-1, 8)[:, 0].tolist())
    assert traced <= seen_traced, traced - seen_traced


GOOD = program_words([0, 1], [2, -1], [0, 0], [0, 0], [[-1, 0, -1, 0, 0, 1, 3, 0], [-1, 1, -1, 0, 0, 1, 3, 0], [0, 0, 1, 0, 0, 1, 4, 0]])


def _mutate(prog, op, field, value):
    p = prog.copy()
    n_in, n_out = int(p[2]), int(p[3])
    p[6 + n_in + 3 * n_out + 8 * op + field] = value
    return p


MALFORMED = [
    (lambda p: p[:5], 'Binary data too small to contain valid DAIS model file'),
    (lambda p: np.concatenate([[2], p[1:]]), 'DAIS version mismatch: expected version 1, got version 2'),
    (lambda p: np.concatenate([p[:2], [-2], p[3:]]), 'Binary data header holds a negative count'),
    (lambda p: p[:-3], 'Binary data size mismatch: expected 152 bytes , got 140 bytes'),
    (lambda p: np.concatenate([p[:5], [1], p[6:], [2, 7]]), 'Binary data size mismatch: expected 164 bytes , got 160 bytes'),
    (lambda p: np.concatenate([p[:5], [1], p[6:], [-3]]), 'negative size for lookup table 0'),
    (lambda p: _mutate(p, 2, 1, 2), 'Operation 2 has id0=2violating causality'),
    (lambda p: _mutate(p, 0, 2, 0), 'Operation 0 has id1=0 violating causality'),
    (lambda p: _mutate(_mutate(p, 2, 0, 6), 2, 3, 2), 'Operation 2 has cond_idx=2 violating causality'),
    (lambda p: _mutate(p, 2, 0, 11), 'Unknown opcode: 11 at index 2'),
    (lambda p: _mutate(p, 2, 0, -7), 'Unknown opcode: -7 at index 2'),
    (lambda p: _mutate(p, 1, 1, 2), 'input index out of range at operation 1'),
    (lambda p: _mutate(p, 2, 1, -1), 'negative operand index at operation 2'),
    (lambda p: _mutate(p, 2, 0, 8), 'lookup table index out of range at operation 2'),
    (lambda p: _mutate(_mutate(p, 2, 0, 9), 2, 3, 3), 'Unknown bit unary operation with data_low=3'),
    (lambda p: _mutate(_mutate(p, 2, 0, -9), 2, 3, -1), 'Unknown bit unary operation with data_low=-1'),
    (lambda p: _mutate(_mutate(p, 2, 0, 10), 2, 4, 3 << 24), 'Unknown bit binary operation with data_low=0'),
    (lambda p: _mutate(_mutate(_mutate(p, 2, 0, 6), 2, 3, 1), 2, 7, 1), 'Unsupported msb_mux shift configuration: shift0=1, shift1=1'),
    (lambda p: np.concatenate([p[:6], [0, 1, 3], p[9:]]), 'output index out of range at output 0'),
]


@pytest.mark.parametrize('case', range(len(MALFORMED)))
def test_load_rejects_before_touching_the_device(case):
    """Header, causality, every index the device would follow and every data-independent runtime error are checked on
    the host when the program is loaded: no GPU is needed to be told, and the reference's wording is kept."""
    from da4ml_b200.dais import DaisProgram

    mutate, msg = MALFORMED[case]
    bad = np.ascontiguousarray(mutate(GOOD.copy()), dtype=np.int32)
    with pytest.raises(RuntimeError) as e:
        DaisProgram(bad)
    assert msg in str(e.value)
    with pytest.raises(RuntimeError) as e:
        sim_compile(bad)
    assert msg in str(e.value)


def _live_ranges(prog):
    n_in, n_out, n_ops = (int(v) for v in prog[2:5])
    ops = prog[6 + n_in + 3 * n_out :][: 8 * n_ops].reshape(-1, 8)
    last = np.full(n_ops, -1)
    for i, (opc, a, b, c) in enumerate(ops[:, :4]):
        if opc not in (-1, 5):
            last[a] = i
        if opc in (0, 1, 6, -6, 7, 10):
            last[b] = i
        if abs(opc) == 6:
            last[c] = i
    return ops, last


# the largest number of values live at once in program order (outputs written through), per traced MLP
MLP_SLOTS = {'mlp_16_64_32_32_5': 409, 'mlp_16_64_64_64_5': 1112, 'mlp_64_128_128_10': 4175}


@pytest.mark.parametrize('name', MLP_NAMES + ['random3', 'lookup_tables', 'sort'])
def test_slots_are_assigned_by_liveness(name):
    z, _ = golden()
    prog = z[f'{name}__program']
    info, slot = sim_compile(prog)
    ops, last = _live_ranges(prog)
    n_ops = len(ops)
    # no slot is given to a second value while the first one may still be read
    owner = {}
    for i in range(n_ops):
        if slot[i] < 0:
            assert last[i] < 0 and ops[i, 0] != 8, f'op {i} is read or is a lookup but got no slot'
            continue
        prev = owner.get(slot[i])
        assert prev is None or last[prev] <= i, f'{name}: slot {slot[i]} of op {prev} (read until {last[prev]}) reused by op {i}'
        owner[slot[i]] = i
    # and no more slots than values live at once (operands read by the op that defines the next value included)
    live_max = 0
    live = 0
    ends = np.bincount(last[last >= 0], minlength=n_ops)
    for i in range(n_ops):
        live -= ends[i]
        if slot[i] >= 0:
            live += 1
            live_max = max(live_max, live)
            if last[i] < 0:
                live -= 1
    assert info['n_slots'] == live_max and slot.max() + 1 == live_max
    if name in MLP_SLOTS:
        assert info['n_slots'] == MLP_SLOTS[name]
    if name.startswith('mlp'):
        assert info['n_slots'] * 4 < n_ops


SIM_CASES = [f'random{s}' for s in range(N_RANDOM)] + ['relu_quantize', 'neg_quantize', 'const_add', 'const', 'maximum', 'sort', 'multiply', 'bit_and_xor',
                                                        'bit_not', 'lookup', 'lookup_tables']  # fmt: skip


@pytest.mark.parametrize('name', SIM_CASES)
def test_simulated_kernel_equals_the_reference_in_both_regimes(name):
    z, _ = golden()
    prog, x, want = stored_case(z, name)
    for regime, kw in ((0, {}), (1, dict(shared_bytes=0, chunk=37, cta_threads=32))):  # global: several launches
        if isinstance(want, tuple):  # a lookup out of range (NaN inputs wrap to values outside the dtype's range)
            with pytest.raises(RuntimeError) as e:
                sim_run(prog, x, **kw)
            assert str(e.value) == want[1], name
            continue
        got, ran = sim_run(prog, x, **kw)
        assert ran == regime
        assert_answer(got, want, f'{name} regime {regime}')


def test_simulated_kernel_on_a_traced_mlp():
    """The first rows of the smallest traced MLP (a CTA's slot file sized for exactly 32 samples), both regimes."""
    z, _ = golden()
    prog, x, _ = stored_case(z, 'mlp_16_64_32_32_5')
    want = z['mlp_16_64_32_32_5__head']
    info, _ = sim_compile(prog)
    got, regime = sim_run(prog, x[: len(want)], shared_bytes=8 * info['n_slots'] * 32)
    assert regime == 0 and np.array_equal(got.view(np.uint64), want.view(np.uint64))
    got, regime = sim_run(prog, x[: len(want)], shared_bytes=8 * info['n_slots'] * 32 - 1, chunk=64)
    assert regime == 1 and np.array_equal(got.view(np.uint64), want.view(np.uint64))


def test_simulated_lookup_overrun_reports_the_first_offending_sample():
    z, _ = golden()
    prog, x, want = stored_case(z, 'lookup_overrun')
    assert want[0] == 'error' and want[1].startswith('Logic lookup index out of bounds: ')
    for kw in (dict(), dict(shared_bytes=0, chunk=7)):
        with pytest.raises(RuntimeError) as e:
            sim_run(prog, x, **kw)
        assert str(e.value) == want[1]
