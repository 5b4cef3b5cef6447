"""Result containers: replay, cost/latency accessors and the JSON layout.  No GPU."""
import numpy as np
import pytest
from conftest import golden_cases, load_golden

from da4ml_b200.types import CombLogic, Pipeline, pipeline_from_arrays


def test_pipeline_reproduces_kernel_and_roundtrips(tmp_path):
    for name, meta in golden_cases().items():
        extra, stages = load_golden(name)
        for st in stages:
            n_out = len(st['out_idxs'])
            st['shape'] = (len(st['inp_shifts']), n_out)
            st['carry_size'] = meta['kwargs'].get('carry_size', -1)
            st['adder_size'] = meta['kwargs'].get('adder_size', -1)
        pipe = pipeline_from_arrays(stages)
        want = extra['kernel'].copy()
        if 'qint' in extra:  # inputs whose interval is {0, 0} are dropped by the solver (state_opr.cc:92-97)
            want[(extra['qint'][:, 0] == 0) & (extra['qint'][:, 1] == 0)] = 0
        assert np.array_equal(pipe.kernel, want), name
        assert pipe.n_adders == meta['n_adders']
        x = np.random.default_rng(0).integers(-8, 8, size=(5, pipe.shape[0])).astype(np.float64)
        assert np.array_equal(pipe(x), x @ want.astype(np.float64))
        p = tmp_path / f'{name}.json'
        pipe.save(p)
        again = Pipeline.load(p)
        assert again == pipe
        assert isinstance(again.solutions[0], CombLogic)
        assert again.cost == pipe.cost and again.latency == pipe.latency


def test_dais_binary_matches_reference_serialiser():
    """SURVEY 8f N3: the DAIS int32 program written from the flat op table equals what the reference's
    ``CombLogic.to_binary`` produces (golden file made by tests/golden/make_golden_binary.py)."""
    from conftest import GOLDEN

    z = np.load(GOLDEN / 'dais_binary.npz')
    seen = 0
    for name, meta in golden_cases().items():
        _, stages = load_golden(name)
        for st in stages:
            st['shape'] = (len(st['inp_shifts']), len(st['out_idxs']))
            st['carry_size'] = meta['kwargs'].get('carry_size', -1)
            st['adder_size'] = meta['kwargs'].get('adder_size', -1)
        pipe = pipeline_from_arrays(stages)
        for i, sol in enumerate(pipe.solutions):
            want = z[f'{name}__s{i}']
            got = sol.to_binary(version=3)
            assert got.dtype == np.int32 and np.array_equal(got, want), f'{name} stage {i}'
            seen += 1
    assert seen == len(z.files)


def test_serialisers_from_flat_arrays_match_the_container_path(tmp_path):
    """SURVEY 8f N3: the DAIS program and the JSON text written straight from the per-stage arrays (no Op objects)
    equal the golden reference serialisation and the NamedTuple path byte for byte."""
    import json

    from conftest import GOLDEN

    from da4ml_b200.types import stage_to_binary, stages_to_json

    z = np.load(GOLDEN / 'dais_binary.npz')
    for name, meta in golden_cases().items():
        _, stages = load_golden(name)
        for st in stages:
            st['shape'] = (len(st['inp_shifts']), len(st['out_idxs']))
            st['carry_size'] = meta['kwargs'].get('carry_size', -1)
            st['adder_size'] = meta['kwargs'].get('adder_size', -1)
        for i, st in enumerate(stages):
            got = stage_to_binary(st, version=3)
            assert got.dtype == np.int32 and np.array_equal(got, z[f'{name}__s{i}']), f'{name} stage {i}'
        pipe = pipeline_from_arrays(stages)
        text = stages_to_json(stages)
        assert text == json.dumps(pipe, separators=(',', ':')), name
        p = tmp_path / f'{name}.json'
        p.write_text(text)
        assert Pipeline.load(p) == pipe


def test_results_build_the_reference_own_containers():
    """Drop-in check (needs the reference tree): with ``types_module=da4ml.types`` the result is made of the reference's
    own NamedTuples, as its nanobind glue does (bindings.cc:106-151), and its serialiser accepts them."""
    import pytest
    import ref_trace

    if not ref_trace.available():
        pytest.skip('needs the da4ml source tree oracle/_ref is built from')
    import sys

    sys.path.insert(0, str(__import__('pathlib').Path(__file__).resolve().parent / 'golden'))
    from make_golden_binary import reference_types

    T = reference_types()
    _, stages = load_golden('c1_8x8_int4_default')
    for st in stages:
        st['shape'] = (len(st['inp_shifts']), len(st['out_idxs']))
        st['carry_size'] = st['adder_size'] = -1
    pipe = pipeline_from_arrays(stages, types_module=T)
    assert type(pipe) is T.Pipeline and type(pipe.solutions[0]) is T.CombLogic and type(pipe.solutions[0].ops[0]) is T.Op
    mine = pipeline_from_arrays(stages)
    assert pipe.cost == mine.cost and tuple(pipe.latency) == tuple(mine.latency)
    assert np.array_equal(pipe.solutions[0].to_binary(), mine.solutions[0].to_binary())
    for m in ('da4ml', 'da4ml._binary', 'da4ml.types'):
        sys.modules.pop(m, None)


def test_fast_op_builder_equals_python_construction():
    """csrc_py/fastbuild.c builds the same list of Op / QInterval NamedTuples as the Python comprehension, for this
    repository's containers and for foreign tuple subclasses; other classes take the Python path."""
    from typing import NamedTuple

    import da4ml_b200.types as T

    rng = np.random.default_rng(0)
    oi = rng.integers(-3, 1000, (500, 4)).astype(np.int64)
    of = rng.random((500, 5)).astype(np.float32)
    want = [T.Op(int(a[0]), int(a[1]), int(a[2]), int(a[3]), T.QInterval(float(b[0]), float(b[1]), float(b[2])), float(b[3]), float(b[4])) for a, b in zip(oi, of)]
    got = T._build_ops(oi, of, T.Op, T.QInterval)
    assert got == want and type(got[0]) is T.Op and type(got[0].qint) is T.QInterval and isinstance(got[0].id0, int)

    class Q2(NamedTuple):
        min: float
        max: float
        step: float

    class Op2(NamedTuple):
        id0: int
        id1: int
        opcode: int
        data: int
        qint: Q2
        latency: float
        cost: float

    got2 = T._build_ops(oi, of, Op2, Q2)
    assert [tuple(o) for o in got2] == [tuple(o) for o in want] and type(got2[7]) is Op2 and type(got2[7].qint) is Q2
    got3 = T._build_ops(oi[:5], of[:5], lambda *a: list(a), lambda *a: list(a))  # not tuple classes: plain Python path
    assert got3[0][:4] == [int(v) for v in oi[0]]
    assert T._build_ops(np.zeros((0, 4), np.int64), np.zeros((0, 5), np.float32), T.Op, T.QInterval) == []


def test_inp_qint_is_indexed_by_input_and_empty_option_lists_mean_defaults():
    """reference types.py:428-435 (inp_qint scatters by id0, default (0, 0, 1)); bindings: empty qintervals / latencies
    sequences mean the defaults (api.cc:161-174)."""
    import da4ml_b200._binary as B
    from da4ml_b200.types import CombLogic, Op, QInterval

    ops = [Op(2, -1, -1, 0, QInterval(-4.0, 3.0, 1.0), 0.0, 0.0), Op(0, -1, -1, 0, QInterval(-8.0, 7.0, 0.5), 1.0, 0.0)]
    cl = CombLogic((3, 1), [0, 0, 0], [1], [0], [False], ops, -1, -1)
    assert cl.inp_qint == [QInterval(-8.0, 7.0, 0.5), QInterval(0.0, 0.0, 1.0), QInterval(-4.0, 3.0, 1.0)]
    assert B._qint_arg([], 4) is None and B._lat_arg((), 4) is None
    with pytest.raises(ValueError):
        B._qint_arg([(0.0, 1.0, 1.0)], 4)
