"""Import the reference's pure-Python ``da4ml.trace`` package (from the da4ml source tree oracle/_ref was built from, as
recorded in oracle/_ref/source_tree by `make -C oracle`) with its native module ``da4ml._binary`` replaced by a stand-in
built from callables the test supplies -- the way an integration would point the tracing front-end at another solver.
TEST INFRASTRUCTURE."""
import importlib
import os
import sys
import types
from pathlib import Path

_RECORD = Path(__file__).resolve().parents[1] / 'oracle' / '_ref' / 'source_tree'
REF = os.path.join(_RECORD.read_text().strip(), 'src', 'da4ml') if _RECORD.is_file() else None


def available() -> bool:
    """The reference's Python sources can be read (isdir is False for a missing or unreadable tree)."""
    return REF is not None and os.path.isdir(os.path.join(REF, 'trace'))


def load(solve, get_lsb_loc, iceil_log2, cost_add, kernel_decompose=None, csd_decompose=None, int_arr_to_csd=None):
    for name in [m for m in sys.modules if m == 'da4ml' or m.startswith('da4ml.')]:
        del sys.modules[name]
    pkg = types.ModuleType('da4ml')
    pkg.__path__ = [REF]
    sys.modules['da4ml'] = pkg
    binary = types.ModuleType('da4ml._binary')
    binary.__path__ = []
    cmvm_bin = types.ModuleType('da4ml._binary.cmvm_bin')
    for mod in (binary, cmvm_bin):
        mod.solve = solve
        mod.get_lsb_loc = get_lsb_loc
        mod.iceil_log2 = iceil_log2
        mod.cost_add = cost_add
        mod.kernel_decompose = kernel_decompose
        mod.csd_decompose = csd_decompose
        mod.int_arr_to_csd = int_arr_to_csd
    binary.dais_interp_run = lambda *a, **k: (_ for _ in ()).throw(RuntimeError('not available in this stand-in'))
    binary.cmvm_bin = cmvm_bin
    sys.modules['da4ml._binary'] = binary
    sys.modules['da4ml._binary.cmvm_bin'] = cmvm_bin
    if 'quantizers' not in sys.modules:  # third-party dependency of trace/ops/quantization.py (absent here; matmul does not use it)
        q0 = types.ModuleType('quantizers')
        q1 = types.ModuleType('quantizers.fixed_point')
        q2 = types.ModuleType('quantizers.fixed_point.fixed_point_ops_np')
        q2.get_fixed_quantizer_np = lambda *a, **k: (_ for _ in ()).throw(RuntimeError('quantizers is not installed'))
        q0.fixed_point, q1.fixed_point_ops_np = q1, q2
        sys.modules.update({'quantizers': q0, 'quantizers.fixed_point': q1, 'quantizers.fixed_point.fixed_point_ops_np': q2})
    T = importlib.import_module('da4ml.types')
    trace = importlib.import_module('da4ml.trace')
    return T, trace
