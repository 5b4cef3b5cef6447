"""DAIS binary golden vectors from the reference's own ``da4ml.types.CombLogic.to_binary`` (types.py:500-541).

Imports types.py of the da4ml source tree oracle/_ref is built from (tests/ref_trace.py) with a stub standing in for its
native module (the reference package itself needs meson/nanobind/xtensor to install).  Writes tests/golden/dais_binary.npz.
"""
import importlib.util
import sys
import types
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parents[1]))
sys.path.insert(0, str(HERE.parent))


def reference_types():
    from ref_trace import REF

    pkg = types.ModuleType('da4ml')
    pkg.__path__ = [REF]
    sys.modules['da4ml'] = pkg
    stub = types.ModuleType('da4ml._binary')
    stub.dais_interp_run = lambda *a, **k: None
    sys.modules['da4ml._binary'] = stub
    spec = importlib.util.spec_from_file_location('da4ml.types', f'{REF}/types.py')
    T = importlib.util.module_from_spec(spec)
    sys.modules['da4ml.types'] = T
    spec.loader.exec_module(T)
    return T


def main():
    from conftest import golden_cases, load_golden

    from da4ml_b200.types import pipeline_from_arrays

    T = reference_types()
    out = {}
    for name, meta in golden_cases().items():
        _, stages = load_golden(name)
        for st in stages:
            st['shape'] = (len(st['inp_shifts']), len(st['out_idxs']))
            st['carry_size'] = meta['kwargs'].get('carry_size', -1)
            st['adder_size'] = meta['kwargs'].get('adder_size', -1)
        pipe = pipeline_from_arrays(stages, types_module=T)  # the reference's own NamedTuples
        assert type(pipe).__module__ == 'da4ml.types'
        for i, sol in enumerate(pipe.solutions):
            out[f'{name}__s{i}'] = sol.to_binary(version=3)
    np.savez_compressed(HERE / 'dais_binary.npz', **out)
    print(len(out), 'programs')


if __name__ == '__main__':
    main()
