"""ctypes binding of libda4ml_b200_cmvm.so (C ABI: include/da4ml_b200_cmvm.h).

Mirror of the reference's ``da4ml._binary`` re-exports (``src/da4ml/_binary/__init__.py:4,19``;
nanobind module ``_binary/cmvm/bindings.cc:227-263``): ``solve, csd_decompose, int_arr_to_csd,
kernel_decompose, get_lsb_loc, iceil_log2, cost_add`` with the same signatures, defaults and exception
types.  Added on top: ``solve_batch`` (many independent problems in one launch) and ``solve_single``.

The shared library is the product's only compute path; importing this module without it raises.
"""

from __future__ import annotations

import ctypes as C
from pathlib import Path

import numpy as np

from ..types import pipeline_from_arrays, stage_to_binary, stages_to_json

_LIB_PATH = Path(__file__).resolve().parent / 'libda4ml_b200_cmvm.so'
if not _LIB_PATH.exists():
    raise ImportError(
        f'{_LIB_PATH} not found: build it with `python -c "import __graft_entry__ as g; g.build()"` '
        '(nvcc, sm_100a). The CMVM solver has no CPU fallback.'
    )
_L = C.CDLL(str(_LIB_PATH))

_f32p = C.POINTER(C.c_float)
_i64p = C.POINTER(C.c_int64)
_i32p = C.POINTER(C.c_int32)
_i8p = C.POINTER(C.c_int8)
_vp = C.c_void_p

_L.da4ml_cmvm_last_error.restype = C.c_char_p
_L.da4ml_cmvm_device_info.argtypes = [_i32p]
_L.da4ml_cmvm_set_stream.argtypes = [_vp]
_L.da4ml_cmvm_plan.argtypes = [_i64p, C.c_int64, C.c_int, C.c_int, _i64p]
_L.da4ml_cmvm_set_group_size.argtypes = [C.c_int]
_L.da4ml_cmvm_set_accounting.argtypes = [C.c_int]
_L.da4ml_cmvm_set_job_sharing.argtypes = [C.c_int]
_L.da4ml_cmvm_set_first_attempt_caps.argtypes = [_i64p]
_L.da4ml_cmvm_solve.argtypes = [_f32p, C.c_int64, C.c_int64, C.c_char_p, C.c_char_p, C.c_int, C.c_int, _f32p, _f32p, C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]
_L.da4ml_cmvm_solve_batch.argtypes = [C.c_int64, C.POINTER(_f32p), _i64p, _i64p, C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.POINTER(_f32p), C.POINTER(_f32p), C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]
_L.da4ml_cmvm_solve_batch_device.argtypes = [C.c_int64, C.POINTER(_vp), _i64p, _i64p, C.c_char_p, C.c_char_p, C.c_int, C.c_int, C.POINTER(_f32p), C.POINTER(_f32p), C.c_int, C.c_int, C.c_int, C.POINTER(_vp)]
_L.da4ml_cmvm_solve_single.argtypes = [_f32p, C.c_int64, C.c_int64, C.c_char_p, _f32p, _f32p, C.c_int, C.c_int, _i32p, C.c_int64, C.POINTER(_vp)]
_L.da4ml_pipeline_free.argtypes = [_vp]
_L.da4ml_pipeline_n_stages.restype = C.c_int64
_L.da4ml_pipeline_n_stages.argtypes = [_vp]
_L.da4ml_pipeline_stage_meta.argtypes = [_vp, C.c_int64, _i64p]
_L.da4ml_pipeline_stage_copy.argtypes = [_vp, C.c_int64, _i64p, _i64p, _i64p, _i64p, _i64p, _f32p]
_L.da4ml_pipeline_stage_counters.argtypes = [_vp, C.c_int64, _i64p]
_L.da4ml_pipeline_stage_milestones.argtypes = [_vp, C.c_int64, _i64p]
_L.da4ml_pipeline_stage_words.argtypes = [_vp, C.c_int64, _i64p]
_L.da4ml_pipeline_device_ms.restype = C.c_double
_L.da4ml_pipeline_device_ms.argtypes = [_vp]
_L.da4ml_pipeline_launches.restype = C.c_int64
_L.da4ml_pipeline_launches.argtypes = [_vp]
_L.da4ml_pipeline_profile.argtypes = [_vp, C.POINTER(C.c_double)]
_L.da4ml_cmvm_csd_decompose.argtypes = [_f32p, C.c_int64, C.c_int64, C.c_int, _i8p, _i8p, _i8p, _i64p]
_L.da4ml_cmvm_int_arr_to_csd.argtypes = [_i32p, C.c_int64, _i8p, _i64p]
_L.da4ml_cmvm_kernel_decompose.argtypes = [_f32p, C.c_int64, C.c_int64, C.c_int, _f32p, _f32p]
_L.da4ml_dais_run.argtypes = [_i32p, C.c_int64, C.POINTER(C.c_double), C.c_int64, C.POINTER(C.c_double)]
_L.da4ml_dais_load.argtypes = [_i32p, C.c_int64, C.POINTER(_vp)]
_L.da4ml_dais_info.argtypes = [_vp, _i64p]
_L.da4ml_dais_infer.argtypes = [_vp, _vp, C.c_int64, _vp]
_L.da4ml_dais_infer_device.argtypes = [_vp, _vp, C.c_int64, _vp]
_L.da4ml_dais_free.argtypes = [_vp]
_L.da4ml_dais_free.restype = None
_L.da4ml_dais_set_shared_budget.argtypes = [C.c_int64, C.c_int64]
_L.da4ml_dais_profile.argtypes = [_vp, _vp, C.c_int64, _i64p, _i64p]
_L.da4ml_dais_profile_device.argtypes = [_vp, _vp, C.c_int64, _i64p, _i64p]
_L.da4ml_dais_capture.argtypes = [_vp, _vp, C.c_int64, _i32p, C.c_int32, _vp]
_L.da4ml_dais_capture_device.argtypes = [_vp, _vp, C.c_int64, _i32p, C.c_int32, _vp]
_L.da4ml_cmvm_get_lsb_loc.argtypes = [C.c_float]
_L.da4ml_cmvm_iceil_log2.argtypes = [C.c_float]
_L.da4ml_cmvm_cost_add.argtypes = [_f32p, _f32p, C.c_int64, C.c_int, C.c_int, C.c_int, _f32p]

EXPORTED_SYMBOLS = [
    'da4ml_cmvm_last_error', 'da4ml_cmvm_device_info', 'da4ml_cmvm_set_stream', 'da4ml_cmvm_set_group_size',
    'da4ml_cmvm_set_accounting', 'da4ml_cmvm_set_job_sharing', 'da4ml_cmvm_set_first_attempt_caps', 'da4ml_pipeline_profile',
    'da4ml_cmvm_release', 'da4ml_cmvm_plan', 'da4ml_cmvm_solve', 'da4ml_cmvm_solve_batch', 'da4ml_cmvm_solve_batch_device',
    'da4ml_cmvm_solve_single', 'da4ml_pipeline_free', 'da4ml_pipeline_n_stages', 'da4ml_pipeline_stage_meta', 'da4ml_pipeline_stage_copy',
    'da4ml_pipeline_stage_counters', 'da4ml_pipeline_stage_milestones', 'da4ml_pipeline_stage_words', 'da4ml_pipeline_device_ms',
    'da4ml_pipeline_launches',
    'da4ml_cmvm_csd_decompose', 'da4ml_cmvm_int_arr_to_csd', 'da4ml_cmvm_kernel_decompose',
    'da4ml_cmvm_get_lsb_loc', 'da4ml_cmvm_iceil_log2', 'da4ml_cmvm_cost_add', 'da4ml_dais_run',
    'da4ml_dais_load', 'da4ml_dais_info', 'da4ml_dais_infer', 'da4ml_dais_infer_device', 'da4ml_dais_free',
    'da4ml_dais_set_shared_budget', 'da4ml_dais_profile', 'da4ml_dais_profile_device', 'da4ml_dais_capture', 'da4ml_dais_capture_device',
]  # fmt: skip

COUNTER_NAMES = ['status', 'n_ops', 'T', 'sum_F', 'sum_R', 'F0', 'R0', 'D_final', 'F_max', 'compactions', 'D0', 'n_bits', 'group_ctas',
                 'rescanned', 'list_max', 'smem_list_cap']


def lib_path() -> Path:
    return _LIB_PATH


def _check(rc: int):
    if rc == 0:
        return
    msg = _L.da4ml_cmvm_last_error().decode()
    if rc == 1:
        raise ValueError(msg)  # nanobind maps std::invalid_argument -> ValueError
    raise RuntimeError(msg)  # std::runtime_error -> RuntimeError (e.g. "Unknown method: ...")


def device_info() -> dict:
    out = (C.c_int32 * 5)()
    _L.da4ml_cmvm_device_info(out)
    return dict(abi_version=out[0], cuda_devices=out[1], sm_count=out[2], cc=(out[3], out[4]))


PLAN_FIELDS = ['ctas_per_problem', 'concurrent_groups', 'columns_per_cta', 'list_rows_smem', 'log2_chunk', 'chunk_slots',
               'segment_entries_per_cta', 'log2_pair_counters', 'shared_bytes', 'shared_budget', 'narrow_rows', 'spill_rows']


def plan(jobs, co_resident_ctas: int = 148, group_override: int = 0) -> dict:
    """Launch geometry the solver would pick for ``jobs`` (no device needed).  Each job is a dict with ``n_in, n_out,
    nbits, digits`` (CSD digits of the matrix) and optionally ``dcol_max`` (digits of the densest column, default
    digits / n_out), ``col_cap`` (bound on rows per column list, default n_in + dcol_max), ``f_mul, list_mul``
    (retry multipliers, default 1, 2)."""
    rows = np.zeros((len(jobs), 8), np.int64)
    for r, j in zip(rows, jobs):
        dcol = int(j.get('dcol_max', -(-int(j['digits']) // int(j['n_out']))))
        r[:] = [j['n_in'], j['n_out'], j['nbits'], j['digits'], dcol, j.get('col_cap', int(j['n_in']) + dcol), j.get('f_mul', 1), j.get('list_mul', 2)]
    out = np.zeros(12, np.int64)
    _check(_L.da4ml_cmvm_plan(_ip(rows), len(jobs), int(co_resident_ctas), int(group_override), _ip(out)))
    return dict(zip(PLAN_FIELDS, (int(v) for v in out)))


def set_stream(cuda_stream: int | None):
    """Run every later call on this CUDA stream (``torch.cuda.current_stream().cuda_stream``)."""
    _L.da4ml_cmvm_set_stream(_vp(cuda_stream or 0))


def set_group_size(n: int):
    _L.da4ml_cmvm_set_group_size(int(n))


def release():
    """Free the device / pinned work buffers cached between calls."""
    _check(_L.da4ml_cmvm_release())


def set_job_sharing(on: bool):
    """Solve byte-identical solve_single jobs of one call once (default on; results are the same either way)."""
    _L.da4ml_cmvm_set_job_sharing(int(bool(on)))


def set_accounting(on: bool):
    """Exact work counters (sum over iterations of the live histogram size); slower, identical results."""
    _L.da4ml_cmvm_set_accounting(int(bool(on)))


FIRST_ATTEMPT_CAPS = ['segment_entries_per_cta', 'list_rows_smem', 'spill_rows', 'log2_pair_counters', 'cells_per_cta', 'extra_expressions']


def set_first_attempt_caps(**caps):
    """Development switch: force capacities below the planner's choice on the first attempt of every round of
    solve_single jobs (keywords from ``FIRST_ATTEMPT_CAPS``; omitted or 0 = the planner's value, no keywords = all
    back to the planner).  Overflows are retried with the planner's sizes (``profile['retried_jobs']``); results do not
    change.  ``plan()`` shows the first attempt's plan."""
    unknown = set(caps) - set(FIRST_ATTEMPT_CAPS)
    if unknown:
        raise TypeError(f'unknown capacities: {sorted(unknown)}')
    arr = np.asarray([int(caps.get(k, 0)) for k in FIRST_ATTEMPT_CAPS], np.int64)
    _check(_L.da4ml_cmvm_set_first_attempt_caps(_ip(arr)))


def _fp(a):
    return a.ctypes.data_as(_f32p) if a is not None else None


def _ip(a):
    return a.ctypes.data_as(_i64p)


def _kernel_arg(kernel) -> np.ndarray:
    # the reference binds `kernel` as noconvert float ndarray (bindings.cc:238): no silent dtype casts
    if not isinstance(kernel, np.ndarray) or kernel.dtype != np.float32:
        raise TypeError('kernel must be a numpy float32 ndarray')
    if kernel.ndim != 2:
        raise RuntimeError('csd_decompose only supports 2D arrays.')
    return np.ascontiguousarray(kernel)


def _qint_arg(qintervals, n_in):
    # an empty sequence means "defaults", as in the reference (bindings.cc extract_qintervals -> api.cc:161-174)
    if qintervals is None or len(qintervals) == 0:
        return None
    q = np.ascontiguousarray(np.asarray([tuple(map(float, qi)) for qi in qintervals], dtype=np.float32).reshape(-1, 3))
    if q.shape[0] != n_in:
        raise ValueError(f'expected {n_in} qintervals, got {q.shape[0]}')
    return q


def _lat_arg(latencies, n_in):
    if latencies is None or len(latencies) == 0:
        return None
    l = np.ascontiguousarray(np.asarray(list(latencies), dtype=np.float32).reshape(-1))
    if l.shape[0] != n_in:
        raise ValueError(f'expected {n_in} latencies, got {l.shape[0]}')
    return l


class RawPipeline:
    """Flat-array view of one solver result (what the C ABI hands back)."""

    def __init__(self, handle=None):
        self.stages = []
        self.counters = []
        self.device_ms = 0.0
        self.launches = 0
        self.profile = {}
        if handle is None:
            return
        try:
            for s in range(_L.da4ml_pipeline_n_stages(handle)):
                meta = np.zeros(5, np.int64)
                _check(_L.da4ml_pipeline_stage_meta(handle, s, _ip(meta)))
                n_in, n_out, n_ops = int(meta[0]), int(meta[1]), int(meta[2])
                st = dict(
                    shape=(n_in, n_out),
                    inp_shifts=np.zeros(n_in, np.int64),
                    out_idxs=np.zeros(n_out, np.int64),
                    out_shifts=np.zeros(n_out, np.int64),
                    out_negs=np.zeros(n_out, np.int64),
                    ops_i=np.zeros((n_ops, 4), np.int64),
                    ops_f=np.zeros((n_ops, 5), np.float32),
                    carry_size=int(meta[3]),
                    adder_size=int(meta[4]),
                )
                _check(_L.da4ml_pipeline_stage_copy(handle, s, _ip(st['inp_shifts']), _ip(st['out_idxs']), _ip(st['out_shifts']), _ip(st['out_negs']), _ip(st['ops_i']), _fp(st['ops_f'])))
                cnt = np.zeros(32, np.int64)
                _check(_L.da4ml_pipeline_stage_counters(handle, s, _ip(cnt)))
                self.stages.append(st)
                cd = dict(zip(COUNTER_NAMES, (int(v) for v in cnt)))
                cd['phase_cycles'] = [int(v) for v in cnt[16:24]]
                cd['phase_cycles_max'] = [int(v) for v in cnt[24:32]]
                ms = np.zeros(63, np.int64)
                _check(_L.da4ml_pipeline_stage_milestones(handle, s, _ip(ms)))
                cd['milestones'] = {250 << k: [int(v) for v in ms[9 * k : 9 * k + 9]] for k in range(7) if ms[9 * k + 8] > 0}
                words = np.zeros(96, np.int64)
                _check(_L.da4ml_pipeline_stage_words(handle, s, _ip(words)))
                cd['split_passes'] = int(words[95])
                self.counters.append(cd)
            self.device_ms = float(_L.da4ml_pipeline_device_ms(handle))
            self.launches = int(_L.da4ml_pipeline_launches(handle))
            prof = (C.c_double * 8)()
            _L.da4ml_pipeline_profile(handle, prof)
            self.profile = dict(device_ms=prof[0], launches=int(prof[1]), solve_kernel_ms=prof[2], solve_kernel_launches=int(prof[3]), algo_bytes=prof[4], jobs_total=int(prof[5]), jobs_run=int(prof[6]),
                                retried_jobs=int(prof[7]))
        finally:
            _L.da4ml_pipeline_free(handle)

    @property
    def n_adders(self) -> int:
        return int(sum(int(np.count_nonzero(st['ops_i'][:, 2] >= 0)) for st in self.stages))

    @classmethod
    def from_stages(cls, stages):
        """Wrap per-stage flat arrays that did not come from a solver handle (fixtures, results received from
        another rank)."""
        r = cls()
        r.stages = list(stages)
        return r

    def to_pipeline(self, types_module=None):
        return pipeline_from_arrays(self.stages, types_module)

    # ---- serialisation straight from the flat arrays (SURVEY 8f N3): no per-op Python objects
    def to_binary(self, version: int = 0) -> list:
        """One DAIS int32 program per stage (reference ``CombLogic.to_binary``, types.py:500-541)."""
        return [stage_to_binary(st, version) for st in self.stages]

    def save_binary(self, path, version: int = 0):
        """Write stage ``i`` to ``<path>.<i>`` (a single-stage result goes to ``path`` itself), the layout
        ``CombLogic.save_binary`` uses per stage."""
        progs = self.to_binary(version)
        if len(progs) == 1:
            progs[0].tofile(path)
        else:
            for i, b in enumerate(progs):
                b.tofile(f'{path}.{i}')

    def to_json(self) -> str:
        """The text ``Pipeline.save`` writes (reference types.py:678-693)."""
        return stages_to_json(self.stages)

    def save(self, path):
        with open(path, 'w') as f:
            f.write(self.to_json())

    def predict_stage(self, i: int, data, n_threads: int = 0):
        """Bit-exact replay of stage ``i`` on a batch of inputs through the GPU DAIS interpreter (reference
        ``CombLogic.predict``, types.py:549-581).  Stages are replayed one at a time: the reference hands stage 1 the
        *unshifted* intervals of stage 0's output ops (api.cc:101-110), so feeding stage 0's outputs into stage 1 under
        fixed-point semantics would wrap -- the reference's ``Pipeline`` has no ``predict`` either."""
        return dais_interp_run(stage_to_binary(self.stages[i]), data, n_threads)

    def stage_kernel(self, i: int):
        """Constant matrix of stage ``i`` (reference ``CombLogic.kernel``, types.py:373-378), recovered on the GPU: input
        ``j`` is probed with one quantum of its declared interval (always representable and in range, unlike 1.0) and
        the response is divided by it -- exact, every factor is a power of two."""
        st = self.stages[i]
        n_in = int(st['shape'][0])
        oi = np.asarray(st['ops_i']).reshape(-1, 4)
        q = np.asarray(st['ops_f'], dtype=np.float32).reshape(-1, 5)[oi[:, 2] == -1][:, :3].astype(np.float64)
        probe = np.where(q[:, 1] >= q[:, 2], q[:, 2], np.where(q[:, 0] <= -q[:, 2], -q[:, 2], 0.0))
        out = self.predict_stage(i, np.diag(probe))
        with np.errstate(divide='ignore', invalid='ignore'):
            k = np.where(probe[:, None] != 0, out / probe[:, None], 0.0)
        assert k.shape[0] == n_in
        return k.astype(np.float32)

    @property
    def kernel(self):
        """The constant matrix this cascade implements = product of the stage kernels (reference ``Pipeline.kernel``,
        types.py:627-629), computed from GPU replays instead of the interpreted float replay."""
        k = self.stage_kernel(0)
        for i in range(1, len(self.stages)):
            k = k @ self.stage_kernel(i)
        return k


def solve_raw(kernel, method0='wmc', method1='auto', hard_dc=-1, decompose_dc=-2, qintervals=None, latencies=None,
              adder_size=-1, carry_size=-1, search_all_decompose_dc=True) -> RawPipeline:
    k = _kernel_arg(kernel)
    q = _qint_arg(qintervals, k.shape[0])
    l = _lat_arg(latencies, k.shape[0])
    h = _vp()
    _check(_L.da4ml_cmvm_solve(_fp(k), k.shape[0], k.shape[1], method0.encode(), method1.encode(), hard_dc, decompose_dc, _fp(q), _fp(l), adder_size, carry_size, int(bool(search_all_decompose_dc)), C.byref(h)))
    return RawPipeline(h)


def solve(kernel, method0='wmc', method1='auto', hard_dc=-1, decompose_dc=-2, qintervals=None, latencies=None,
          adder_size=-1, carry_size=-1, search_all_decompose_dc=True):
    """``da4ml._binary.cmvm_bin.solve`` (bindings.cc:235-248): returns a ``Pipeline`` of two ``CombLogic`` stages."""
    return solve_raw(kernel, method0, method1, hard_dc, decompose_dc, qintervals, latencies, adder_size, carry_size, search_all_decompose_dc).to_pipeline()


def solve_batch_raw(kernels, method0='wmc', method1='auto', hard_dc=-1, decompose_dc=-2, qintervals=None, latencies=None,
                    adder_size=-1, carry_size=-1, search_all_decompose_dc=True) -> list[RawPipeline]:
    ks = [_kernel_arg(k) for k in kernels]
    n = len(ks)
    if n == 0:
        return []
    qs = [_qint_arg(qintervals[i], ks[i].shape[0]) if qintervals is not None else None for i in range(n)]
    ls = [_lat_arg(latencies[i], ks[i].shape[0]) if latencies is not None else None for i in range(n)]
    kp = (_f32p * n)(*[_fp(k) for k in ks])
    qp = (_f32p * n)(*[_fp(q) for q in qs])
    lp = (_f32p * n)(*[_fp(l) for l in ls])
    n_in = np.asarray([k.shape[0] for k in ks], np.int64)
    n_out = np.asarray([k.shape[1] for k in ks], np.int64)
    hs = (_vp * n)()
    _check(_L.da4ml_cmvm_solve_batch(n, kp, _ip(n_in), _ip(n_out), method0.encode(), method1.encode(), hard_dc, decompose_dc, qp, lp, adder_size, carry_size, int(bool(search_all_decompose_dc)), hs))
    return [RawPipeline(_vp(h)) for h in hs]


def solve_batch_device_raw(dev_ptrs, shapes, method0='wmc', method1='auto', hard_dc=-1, decompose_dc=-2, adder_size=-1,
                           carry_size=-1, search_all_decompose_dc=True) -> list[RawPipeline]:
    """Batch solve of matrices already resident in device memory: ``dev_ptrs[i]`` is the address of a dense
    float32 ``shapes[i] = (n_in, n_out)`` array on the current CUDA device (e.g. ``tensor.data_ptr()``)."""
    n = len(dev_ptrs)
    kp = (_vp * n)(*[_vp(int(p)) for p in dev_ptrs])
    n_in = np.asarray([s[0] for s in shapes], np.int64)
    n_out = np.asarray([s[1] for s in shapes], np.int64)
    hs = (_vp * n)()
    _check(_L.da4ml_cmvm_solve_batch_device(n, kp, _ip(n_in), _ip(n_out), method0.encode(), method1.encode(), hard_dc, decompose_dc, None, None, adder_size, carry_size, int(bool(search_all_decompose_dc)), hs))
    return [RawPipeline(_vp(h)) for h in hs]


def solve_batch(kernels, **kw):
    """Solve many independent constant matrices in one GPU pass; list of ``Pipeline``."""
    return [r.to_pipeline() for r in solve_batch_raw(kernels, **kw)]


def solve_single_raw(kernel, method='wmc', qintervals=None, latencies=None, adder_size=-1, carry_size=-1, trace_cap=0):
    """One CSE stage (reference ``solve_single``, cmvm_core.cc:227).  Returns (RawPipeline, trace[n,5] or None)."""
    k = _kernel_arg(kernel)
    q = _qint_arg(qintervals, k.shape[0])
    l = _lat_arg(latencies, k.shape[0])
    tr = np.zeros((max(trace_cap, 1), 5), np.int32)
    h = _vp()
    _check(_L.da4ml_cmvm_solve_single(_fp(k), k.shape[0], k.shape[1], method.encode(), _fp(q), _fp(l), adder_size, carry_size, tr.ctypes.data_as(_i32p) if trace_cap > 0 else None, trace_cap, C.byref(h)))
    raw = RawPipeline(h)
    return raw, (tr[: min(trace_cap, raw.counters[0]['T'])] if trace_cap > 0 else None)


def csd_decompose(inp, center=True):
    """(csd int8[n_in,n_out,N], shift0 int8[n_in], shift1 int8[n_out])  (bindings.cc:63-103)."""
    k = _kernel_arg(inp)
    csd = np.zeros(k.size * 32, np.int8)
    s0 = np.zeros(k.shape[0], np.int8)
    s1 = np.zeros(k.shape[1], np.int8)
    nb = C.c_int64(0)
    _check(_L.da4ml_cmvm_csd_decompose(_fp(k), k.shape[0], k.shape[1], int(bool(center)), csd.ctypes.data_as(_i8p), s0.ctypes.data_as(_i8p), s1.ctypes.data_as(_i8p), C.byref(nb)))
    return csd[: k.size * nb.value].reshape(k.shape[0], k.shape[1], nb.value).copy(), s0, s1


def int_arr_to_csd(inp):
    """int32 ndarray -> int8[..., N] CSD digits (bindings.cc:43-61)."""
    if not isinstance(inp, np.ndarray) or inp.dtype != np.int32:
        raise TypeError('inp must be a numpy int32 ndarray')
    a = np.ascontiguousarray(inp)
    out = np.zeros(a.size * 32, np.int8)
    nb = C.c_int64(0)
    _check(_L.da4ml_cmvm_int_arr_to_csd(a.ctypes.data_as(_i32p), a.size, out.ctypes.data_as(_i8p), C.byref(nb)))
    return out[: a.size * nb.value].reshape(*a.shape, nb.value).copy()


def kernel_decompose(kernel, dc=-2):
    """W = m0 @ m1 graph decomposition (bindings.cc:232-234 -> mat_decompose.cc:62-137)."""
    k = _kernel_arg(kernel)
    m0 = np.zeros(k.shape, np.float32)
    m1 = np.zeros((k.shape[1], k.shape[1]), np.float32)
    _check(_L.da4ml_cmvm_kernel_decompose(_fp(k), k.shape[0], k.shape[1], int(dc), _fp(m0), _fp(m1)))
    return m0, m1


def dais_interp_run(bin_logic, data, n_threads: int = 1):
    """``da4ml._binary.dais_interp_run`` (reference _binary/__init__.py:8-16): run a DAIS program (int32 words of
    ``CombLogic.to_binary``) on a batch of inputs; float64 ``[n_samples, n_out]``.  Runs on the GPU (``n_threads`` is
    accepted for signature compatibility); programs are limited to what the CMVM path emits (opcodes -1/0/1)."""
    prog = np.ascontiguousarray(np.ravel(bin_logic), dtype=np.int32)
    x = np.ascontiguousarray(np.ravel(data), dtype=np.float64)
    if prog.size < 6 or prog[0] != 1 or min(prog[2:5]) < 0:  # let the library word the header error
        inp_size, out_size, n = 0, 0, 0
    else:
        inp_size, out_size = int(prog[2]), int(prog[3])
        assert inp_size == 0 or x.size % inp_size == 0, f'Input size {x.size} is not divisible by {inp_size}'
        n = x.size // inp_size if inp_size else 0
    out = np.zeros((n, out_size), np.float64)
    _check(_L.da4ml_dais_run(prog.ctypes.data_as(_i32p), prog.size, x.ctypes.data_as(C.POINTER(C.c_double)), n, out.ctypes.data_as(C.POINTER(C.c_double))))
    return out


def get_lsb_loc(x: float) -> int:
    return int(_L.da4ml_cmvm_get_lsb_loc(float(x)))


def iceil_log2(x: float) -> int:
    return int(_L.da4ml_cmvm_iceil_log2(float(x)))


def cost_add(q0, q1, shift: int, sub: bool, adder_size: int, carry_size: int):
    a = np.asarray(tuple(q0), np.float32)
    b = np.asarray(tuple(q1), np.float32)
    out = np.zeros(2, np.float32)
    _L.da4ml_cmvm_cost_add(_fp(a), _fp(b), int(shift), int(bool(sub)), int(adder_size), int(carry_size), _fp(out))
    return float(out[0]), float(out[1])


__all__ = [
    'solve', 'solve_batch', 'solve_raw', 'solve_batch_raw', 'solve_batch_device_raw', 'solve_single_raw', 'csd_decompose', 'int_arr_to_csd',
    'kernel_decompose', 'get_lsb_loc', 'iceil_log2', 'cost_add', 'dais_interp_run', 'device_info', 'plan', 'set_stream', 'set_group_size', 'set_accounting',
]  # fmt: skip
