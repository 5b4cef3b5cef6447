"""Host-side SIMT simulation of the product's CUDA kernel sources -- TEST INFRASTRUCTURE ONLY (see simt.h)."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
LIB = HERE / 'libsim_cmvm.so'
CSRC = HERE.parent.parent / 'da4ml_b200' / 'csrc'


def build(force: bool = False) -> Path:
    """g++ the harness together with the kernel headers (host compilation under the shim)."""
    srcs = [HERE / 'sim_cmvm.cc', HERE / 'simt.h', *sorted(CSRC.glob('*.cuh'))]
    if force or not LIB.exists() or LIB.stat().st_mtime < max(p.stat().st_mtime for p in srcs):
        cmd = ['/usr/bin/g++' if Path('/usr/bin/g++').exists() else 'g++', '-O2', '-std=c++17', '-ffp-contract=off', '-fPIC', '-shared', '-w',
               str(HERE / 'sim_cmvm.cc'), '-o']  # fmt: skip
        tmp = LIB.with_name(f'.{LIB.name}.{os.getpid()}')  # concurrent test workers: build aside, rename atomically
        subprocess.run([*cmd, str(tmp)], check=True)
        os.replace(tmp, LIB)
    return LIB


_lib = None


def lib():
    global _lib
    if _lib is None:
        L = C.CDLL(str(build()))
        L.sim_last_error.restype = C.c_char_p
        L.sim_solve_single.restype = C.c_longlong
        FP, IP = C.POINTER(C.c_float), C.POINTER(C.c_int64)
        L.sim_solve_single.argtypes = [FP, C.c_int, C.c_int, C.c_char_p, FP, FP, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                       IP, IP, IP, IP, IP, IP, FP, C.c_longlong]  # fmt: skip
        PFP, PIP = C.POINTER(FP), C.POINTER(IP)
        L.sim_solve_many.argtypes = [C.c_int, PFP, C.POINTER(C.c_int), C.POINTER(C.c_int), C.c_char_p, PFP, PFP, C.c_int, C.c_int, C.c_int,
                                     PIP, PIP, PIP, PIP, PIP, PIP, PFP, C.POINTER(C.c_longlong), C.POINTER(C.c_longlong)]  # fmt: skip
        L.sim_set_schedule.argtypes = [C.c_int]
        L.sim_set_poison.argtypes = [C.c_int]
        L.sim_set_list_cap.argtypes = [C.c_int]
        L.sim_set_own_caps.argtypes = [C.c_int, C.c_int]
        L.sim_set_wide_rows.argtypes = [C.c_int]
        L.sim_set_segment_cap.argtypes = [C.c_int]
        L.sim_set_caps.argtypes = [C.c_int, C.c_int]
        L.sim_set_first_attempt_caps.argtypes = [C.POINTER(C.c_longlong)]
        L.sim_kernel_decompose.argtypes = [FP, C.c_int, C.c_int, C.c_int, FP, FP]
        _lib = L
    return _lib


def set_schedule(mode: int):
    """Order in which the simulator resumes runnable threads: 0 ascending, 1 descending, >= 2 pseudo-random (seed)."""
    lib().sim_set_schedule(int(mode))


def set_segment_cap(entries: int):
    """Shrink every CTA's histogram segment to `entries` (0 = planner's size): small problems then compact / overflow."""
    lib().sim_set_segment_cap(int(entries))


def set_list_cap(rows: int | None):
    """Shrink the shared-memory owner lists to `rows` rows (None or 0 = planner's size); the rows beyond that spill to
    global memory.  `set_own_caps(list_rows=0)` puts every row there."""
    lib().sim_set_list_cap(int(rows) if rows else -1)


def set_wide_rows(on: bool):
    """Keep three words per shared-memory list row even when 6 bytes would do."""
    lib().sim_set_wide_rows(int(bool(on)))


def set_first_attempt_caps(**caps):
    """The product's first-attempt capacities (``da4ml_b200._binary.FIRST_ATTEMPT_CAPS``; omitted = planner's), applied
    to the plan and the expression table as the host driver applies them on a first attempt (no retry here)."""
    names = ['segment_entries_per_cta', 'list_rows_smem', 'spill_rows', 'log2_pair_counters', 'cells_per_cta', 'extra_expressions']
    arr = (C.c_longlong * 6)(*[int(caps.pop(k, 0)) for k in names])
    assert not caps, f'unknown capacities: {sorted(caps)}'
    lib().sim_set_first_attempt_caps(arr)


def set_own_caps(hash_log: int = 0, spill_rows: int = -1, list_rows: int | None = None):
    """log2 of the pair-counter hash table (0 = planner's), rows an owner list may spill to
    global memory (< 0 = planner's), shared-memory rows per list (None = planner's, 0 = none)."""
    lib().sim_set_own_caps(int(hash_log), int(spill_rows))
    lib().sim_set_list_cap(-1 if list_rows is None else int(list_rows))


def set_poison(on: bool):
    """Fill every buffer the host driver does not clear before a launch with garbage instead of zeros."""
    lib().sim_set_poison(int(bool(on)))


def set_caps(e_cap: int = 0, pool: int = 0):
    """Shrink the expression table (new expressions beyond the inputs) / the cell pool of every CTA."""
    lib().sim_set_caps(int(e_cap), int(pool))


def solve_single(kernel, method='wmc', qintervals=None, latencies=None, adder_size=-1, carry_size=-1, ctas=2, cta_threads=64,
                 accounting=False, list_mul=2):
    """One solve_single executed by the simulated kernels; returns (stage dict like the oracle's, counters[32])."""
    k = np.ascontiguousarray(kernel, dtype=np.float32)
    n_in, n_out = k.shape
    q = np.ascontiguousarray(np.tile(np.array([-128.0, 127.0, 1.0], np.float32), (n_in, 1)) if qintervals is None else np.asarray(qintervals, np.float32))
    l = np.zeros(n_in, np.float32) if latencies is None else np.ascontiguousarray(latencies, dtype=np.float32)
    room = n_in + int(np.count_nonzero(k)) * 34 + 8
    meta = np.zeros(32, np.int64)
    st = dict(inp_shifts=np.zeros(n_in, np.int64), out_idxs=np.zeros(n_out, np.int64), out_shifts=np.zeros(n_out, np.int64), out_negs=np.zeros(n_out, np.int64))
    ops_i = np.zeros((room, 4), np.int64)
    ops_f = np.zeros((room, 5), np.float32)
    p64 = lambda a: a.ctypes.data_as(C.POINTER(C.c_int64))  # noqa: E731
    pf = lambda a: a.ctypes.data_as(C.POINTER(C.c_float))  # noqa: E731
    n = lib().sim_solve_single(pf(k), n_in, n_out, method.encode(), pf(q), pf(l), adder_size, carry_size, ctas, cta_threads, int(accounting),
                               list_mul, p64(meta), p64(st['inp_shifts']), p64(st['out_idxs']), p64(st['out_shifts']), p64(st['out_negs']), p64(ops_i), pf(ops_f), room)  # fmt: skip
    if n == -100:
        raise RuntimeError(lib().sim_last_error().decode())
    if n < 0:
        raise RuntimeError(f'simulated kernel reported capacity status {-n}')
    st['ops_i'] = ops_i[:n].copy()
    st['ops_f'] = ops_f[:n].copy()
    return st, meta


def solve_many(kernels, method='wmc', ctas=2, groups=1, cta_threads=64):
    """Several solve_single jobs (default options) in ONE simulated launch of `groups` groups of `ctas` CTAs: jobs beyond
    the number of groups run one after the other in a group's workspace, as in a batched solve.  Returns the stage dicts."""
    ks = [np.ascontiguousarray(k, dtype=np.float32) for k in kernels]
    n = len(ks)
    qs = [np.ascontiguousarray(np.tile(np.array([-128.0, 127.0, 1.0], np.float32), (k.shape[0], 1))) for k in ks]
    ls = [np.zeros(k.shape[0], np.float32) for k in ks]
    rooms = [k.shape[0] + int(np.count_nonzero(k)) * 34 + 8 for k in ks]
    metas = [np.zeros(32, np.int64) for _ in ks]
    sts = [dict(inp_shifts=np.zeros(k.shape[0], np.int64), out_idxs=np.zeros(k.shape[1], np.int64), out_shifts=np.zeros(k.shape[1], np.int64),
                out_negs=np.zeros(k.shape[1], np.int64)) for k in ks]  # fmt: skip
    ops_i = [np.zeros((r, 4), np.int64) for r in rooms]
    ops_f = [np.zeros((r, 5), np.float32) for r in rooms]
    FP, IP = C.POINTER(C.c_float), C.POINTER(C.c_int64)
    fa = lambda arrs: (FP * n)(*[a.ctypes.data_as(FP) for a in arrs])  # noqa: E731
    ia = lambda arrs: (IP * n)(*[a.ctypes.data_as(IP) for a in arrs])  # noqa: E731
    n_ops = (C.c_longlong * n)()
    rc = lib().sim_solve_many(n, fa(ks), (C.c_int * n)(*[k.shape[0] for k in ks]), (C.c_int * n)(*[k.shape[1] for k in ks]), method.encode(), fa(qs), fa(ls),
                              ctas, groups, cta_threads, ia(metas), ia([s['inp_shifts'] for s in sts]), ia([s['out_idxs'] for s in sts]),
                              ia([s['out_shifts'] for s in sts]), ia([s['out_negs'] for s in sts]), ia(ops_i), fa(ops_f), (C.c_longlong * n)(*rooms), n_ops)  # fmt: skip
    if rc != 0:
        raise RuntimeError(lib().sim_last_error().decode())
    for i, st in enumerate(sts):
        if n_ops[i] < 0:
            raise RuntimeError(f'simulated kernel reported capacity status {-n_ops[i]} for job {i}')
        st['ops_i'] = ops_i[i][: n_ops[i]].copy()
        st['ops_f'] = ops_f[i][: n_ops[i]].copy()
    return sts


def kernel_decompose(kernel, dc=-2):
    """``kernel_decompose`` executed by the simulated centre / distance / MST kernels -> (m0, m1)."""
    k = np.ascontiguousarray(kernel, dtype=np.float32)
    m0 = np.zeros(k.shape, np.float32)
    m1 = np.zeros((k.shape[1], k.shape[1]), np.float32)
    FP = C.POINTER(C.c_float)
    if lib().sim_kernel_decompose(k.ctypes.data_as(FP), k.shape[0], k.shape[1], int(dc), m0.ctypes.data_as(FP), m1.ctypes.data_as(FP)) != 0:
        raise RuntimeError(lib().sim_last_error().decode())
    return m0, m1
