"""Store the reference DAIS interpreter's per-op values, and the profile statistics derived from them, for
tests/test_dais_profile.py and tests/test_dais_profile_gpu.py:

    dais_profile.npz   per case (tests/test_dais_profile.py:profile_cases): stats [4][n_ops] (min, max, outside,
                       wrapped) and first (sample, op) outside its range; the values [n][n_ops] whole for small cases,
                       else their digest and the first rows; for the MLP run under the CPU simulation, the stats of
                       those rows too; or the reference's error message

The reference interpreter keeps its per-op buffer private, so it runs unmodified (oracle/dais_ref.run) on a widened
copy of each program: every op gets two quantize ops that extract the high and low 32-bit halves of its value (signed
width 32 at f - 32, unsigned width 32 at f; both exact in float64) and every half is an output at scale 1.  The exact
int64 value is hi * 2^32 + (lo mod 2^32); lo is reduced because the reference's % can return a negative remainder when
its left operand wraps.  Needs `make -C oracle`.

    python tests/golden/make_golden_dais_profile.py
"""
import sys
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parents[1]))
sys.path.insert(0, str(HERE.parent))

from conftest import digest  # noqa: E402

from oracle import dais_ref  # noqa: E402

I64_MIN = np.iinfo(np.int64).min
BATCH_BYTES = 1 << 28  # of the widened program's float64 outputs per reference call


def parts(prog):
    prog = np.asarray(prog, np.int64)
    n_in, n_out, n_ops = (int(v) for v in prog[2:5])
    inp_shifts = prog[6 : 6 + n_in]
    ops = prog[6 + n_in + 3 * n_out :][: 8 * n_ops].reshape(-1, 8)
    tables = prog[6 + n_in + 3 * n_out + 8 * n_ops :]
    return n_in, n_ops, inp_shifts, ops, tables


def widened(prog):
    """The program with a high and a low half of every op appended, and those halves as its only outputs."""
    n_in, n_ops, inp_shifts, ops, tables = parts(prog)
    f = ops[:, 7]
    idx = np.arange(n_ops)
    hi = np.stack([np.full(n_ops, 3), idx, np.full(n_ops, -1), 0 * idx, 0 * idx, np.ones(n_ops, np.int64), 63 - f, f - 32], axis=1)
    lo = np.stack([np.full(n_ops, 3), idx, np.full(n_ops, -1), 0 * idx, 0 * idx, 0 * idx, 32 - f, f], axis=1)
    halves = np.stack([hi, lo], axis=1).reshape(-1, 8)
    out_idxs = n_ops + np.arange(2 * n_ops)
    out_shifts = halves[:, 7]
    head = [1, 0, n_in, 2 * n_ops, 3 * n_ops, int(prog[5])]
    words = [head, inp_shifts, out_idxs, out_shifts, np.zeros(2 * n_ops, np.int64), ops.ravel(), halves.ravel(), tables]
    return np.concatenate([np.asarray(w, np.int64).ravel() for w in words]).astype(np.int32)


def reference_values(prog, x):
    """The reference interpreter's buffer[op] for every sample and op: int64 [n][n_ops]."""
    n_ops = int(prog[4])
    wide = widened(prog)
    batch = max(1, BATCH_BYTES // (16 * max(n_ops, 1)))
    out = np.empty((len(x), n_ops), np.int64)
    for b0 in range(0, len(x), batch):
        y = dais_ref.run(wide, x[b0 : b0 + batch])
        hi = y[:, 0::2].astype(np.int64)
        lo = np.mod(y[:, 1::2].astype(np.int64), 2**32)
        out[b0 : b0 + batch] = (hi << 32) + lo
    return out


def check_reconstruction():
    """Values beyond 2^53, INT64_MIN and INT64_MAX included, come back exactly (constants of known value)."""
    import test_dais_full as T

    consts = [I64_MIN, 2**63 - 1, 2**53 + 1, -(2**53) - 3, -1, 0, 2**32 - 1, -(2**32)]
    ops = [[-1, 0, -1, 0, 0, 1, 3, 0]]
    for c in consts:
        u = c & (2**64 - 1)
        lo, hi = u & 0xFFFFFFFF, u >> 32
        ops.append([5, -1, -1, lo - 2**32 if lo >= 2**31 else lo, hi - 2**32 if hi >= 2**31 else hi, 1, 63, 0])
    prog = T.program_words([0], [1], [0], [0], ops)
    got = reference_values(prog, np.zeros((3, 1)))
    assert got[:, 1:].tolist() == [consts] * 3, got


def _w32(v):
    return ((np.asarray(v, np.int64) + 2**31) % 2**32) - 2**31


def pre_wrap(prog, x, vals):
    """A RESTATEMENT in numpy of the value before the wrap step of the four quantizing kinds (-1, +-2, +-3, +-6), from
    the exact operand values: the converted input floor(x * 2^(shift + f)) with NaN and out-of-range inputs giving
    INT64_MIN, the shifted operand of relu / quantize, the selected and shifted operand of msb_mux.  `None` for the
    other ops; relu's negative operands, which give 0 and are not wraps, come as a mask.  Yields (op, (pre, mask))."""
    n_in, n_ops, inp_shifts, ops, _ = parts(prog)
    width = _w32(_w32(ops[:, 6] + ops[:, 7]) + (ops[:, 5] != 0))
    with np.errstate(all='ignore'):
        for i, (opc, a, b, c, dh, sg, ii, f) in enumerate(ops.tolist()):
            if opc == -1:
                v = np.floor(x[:, a] * np.power(2.0, float(_w32(inp_shifts[a] + f))))
                ok = (v >= -(2.0**63)) & (v < 2.0**63)
                yield i, (np.where(ok, np.where(ok, v, 0).astype(np.int64), I64_MIN), None)
            elif abs(opc) in (2, 3):
                v = -vals[:, a] if opc < 0 else vals[:, a]
                p = v >> (int(_w32(ops[a, 7] - f)) & 63)
                yield i, (p, (v < 0) if abs(opc) == 2 else None)
            elif abs(opc) == 6:
                vc = vals[:, c]
                if ops[c, 5]:
                    cond = vc < 0
                else:
                    thr = max(np.int64(1) << np.int64(int(_w32(width[c] - 2)) & 63), 0)
                    cond = vc > thr
                s0 = int(_w32(f - ops[a, 7])) & 63
                s1 = int(_w32(_w32(f - ops[b, 7]) + dh)) & 63
                v1 = -vals[:, b] if opc < 0 else vals[:, b]
                yield i, (np.where(cond, vals[:, a] << s0, v1 << s1), None)


def profile_stats(prog, x, vals):
    """stats [4][n_ops] and first (sample, op), derived from the exact values."""
    n_in, n_ops, _, ops, _ = parts(prog)
    stats = np.zeros((4, n_ops), np.int64)
    stats[0], stats[1] = np.iinfo(np.int64).max, I64_MIN
    if len(vals):
        stats[0], stats[1] = vals.min(axis=0), vals.max(axis=0)
    outside = np.zeros(vals.shape, bool)
    for i, (sg, ii, f) in enumerate(ops[:, 5:8].tolist()):
        w = int(sg != 0) + ii + f
        if w <= 0:
            lo, hi = 0, 0
        elif w >= 64:
            lo, hi = (-(2**63) if sg else 0), 2**63 - 1
        elif sg:
            lo, hi = -(2 ** (w - 1)), 2 ** (w - 1) - 1
        else:
            lo, hi = 0, 2**w - 1
        outside[:, i] = (vals[:, i] < lo) | (vals[:, i] > hi)
    stats[2] = outside.sum(axis=0)
    for i, (p, skip) in pre_wrap(prog, x, vals):
        changed = p != vals[:, i]
        if skip is not None:
            changed &= ~skip
        stats[3, i] = changed.sum()
    rows = np.flatnonzero(outside.any(axis=1))
    first = (int(rows[0]), int(np.flatnonzero(outside[rows[0]])[0])) if rows.size else (-1, -1)
    return stats, np.array(first, np.int64)


def check_outputs(prog, x, vals):
    """The exact values reproduce the original program's outputs, as the reference computes them, bit for bit."""
    prog = np.asarray(prog)
    n_in, n_out, n_ops = (int(v) for v in prog[2:5])
    out_idxs, out_shifts, out_negs = (prog[6 + n_in + k * n_out :][:n_out].astype(np.int64) for k in range(3))
    f = parts(prog)[3][:, 7]
    y = dais_ref.run(prog, x)
    for o in range(n_out):
        if out_idxs[o] < 0:
            assert np.all(y[:, o] == 0)
            continue
        v = vals[:, out_idxs[o]]
        v = -v if out_negs[o] else v
        want = v.astype(np.float64) * np.power(2.0, float(_w32(out_shifts[o] - f[out_idxs[o]])))
        assert np.array_equal(want.view(np.uint64), y[:, o].view(np.uint64)), o


def main():
    import test_dais_profile as TP

    if not dais_ref.available():
        sys.exit('oracle/_ref is not built: run `make -C oracle REF=<da4ml source tree>` first')
    check_reconstruction()
    out = {}
    for name, (prog, x) in TP.profile_cases().items():
        if name in ('narrow', 'mlp_wraps'):
            out[f'{name}__input'] = np.array(digest([('x', x)]))
        if name == 'narrow':
            out[f'{name}__program'] = np.asarray(prog, np.int32)
        try:
            dais_ref.run(prog, x)
        except RuntimeError as e:
            out[f'{name}__error'] = np.array(str(e))
            continue
        with np.errstate(over='ignore'):
            vals = reference_values(prog, x)
            check_outputs(prog, x, vals)
            stats, first = profile_stats(prog, x, vals)
        out[f'{name}__stats'], out[f'{name}__first'] = stats, first
        if vals.size <= 40000:
            out[f'{name}__values'] = vals
        else:
            out[f'{name}__values_digest'] = np.array(TP.values_digest(vals))
            if name == 'mlp_wraps':  # the MLP the CPU simulation runs
                out[f'{name}__values_head'] = vals[: TP.HEAD]
                out[f'{name}__head_stats'], out[f'{name}__head_first'] = profile_stats(prog, x[: TP.HEAD], vals[: TP.HEAD])
        print(name, vals.shape, 'outside', int(stats[2].sum()), 'wrapped', int(stats[3].sum()), 'first', tuple(first), flush=True)
    np.savez_compressed(HERE / 'dais_profile.npz', **out)


if __name__ == '__main__':
    main()
