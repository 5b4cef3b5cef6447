"""SURVEY 8f N4: register pipelining (``to_pipeline``, retiming off) and the Verilog / VHDL / HLS emitters of
``da4ml_b200.emit``, which work from the solver's flat result arrays, against texts produced by the reference's own
``trace/pipeline.py`` and ``codegen`` modules (tests/golden/codegen.json.gz, tests/golden/make_golden_codegen.py)."""
import gzip
import json

import numpy as np
import pytest
from conftest import GOLDEN, golden_cases, load_golden

from da4ml_b200 import emit
from da4ml_b200.types import pipeline_from_arrays


@pytest.fixture(scope='module')
def gold():
    with gzip.open(GOLDEN / 'codegen.json.gz', 'rb') as f:
        return json.loads(f.read())


def _stages(name, gold=None):
    if name.startswith('custom_'):  # solved by the reference's object code when the golden file was made; arrays inside it
        stages = []
        for a in gold[name]['arrays']:
            st = {k: np.asarray(a[k], dtype=np.int64) for k in ('inp_shifts', 'out_idxs', 'out_shifts', 'out_negs')}
            st['ops_i'] = np.asarray(a['ops_i'], dtype=np.int64).reshape(-1, 4)
            st['ops_f'] = np.asarray(a['ops_f_bits'], dtype=np.uint32).view(np.float32).reshape(-1, 5)
            st['shape'] = (len(st['inp_shifts']), len(st['out_idxs']))
            st['adder_size'], st['carry_size'] = a['adder_size'], a['carry_size']
            stages.append(st)
        return stages
    meta = golden_cases()[name]
    _, stages = load_golden(name)
    for st in stages:
        st['shape'] = (len(st['inp_shifts']), len(st['out_idxs']))
        st['carry_size'] = meta['kwargs'].get('carry_size', -1)
        st['adder_size'] = meta['kwargs'].get('adder_size', -1)
    return stages


CASES = ['c1_8x8_int4_default', 'int_16x16_int8_default', 'pytest_8_b4_harddc2_add1', 'single_16x12_hetero_wmc', 'int_12x20_int6_harddc1', 'int_17x5_int8_mcpdc',
         'pytest_4_b2_mc_wmc', 'custom_neg_zero_6x7', 'custom_neg_frac_9x6', 'custom_dead_input_7x6']  # fmt: skip


def _ok(v):
    return not (isinstance(v, dict) and 'error' in v)


@pytest.mark.parametrize('name', CASES)
def test_combinational_emitters_match_the_reference_text(gold, name):
    for i, (st, g) in enumerate(zip(_stages(name, gold), gold[name]['stages'])):
        assert emit.verilog_comb_logic_gen(st, f'm{i}') == g['verilog']
        assert emit.verilog_comb_logic_gen(st, f'm{i}', print_latency=True, timescale='`timescale 1ns/1ps') == g['verilog_lat']
        assert emit.vhdl_comb_logic_gen(st, f'm{i}', print_latency=(i == 1)) == g['vhdl']
        assert emit.verilog_generate_io_wrapper(st, f'm{i}', False) == g['verilog_io']
        assert emit.vhdl_generate_io_wrapper(st, f'm{i}', False) == g['vhdl_io']
        assert emit.rtl_binder_gen(st, f'm{i}_wrapper') == g['binder']
        for fl, (code, bridge) in g['hls'].items():
            got = emit.hls_logic_and_bridge_gen(st, f'f{i}', fl, pragmas=['#pragma HLS INLINE'] if fl == 'vitis' else None, print_latency=(fl == 'hlslib'),
                                                namespace='ns' if fl == 'oneapi' else '', n_base_indent=1 if fl == 'oneapi' else 0)  # fmt: skip
            assert got[0] == code and got[1] == bridge, fl


@pytest.mark.parametrize('name', CASES)
def test_two_stage_result_as_register_pipeline(gold, name):
    stages, g = _stages(name, gold), gold[name]['pipeline']
    assert emit.verilog_pipeline_logic_gen(stages, 'top') == g['verilog']
    assert emit.vhdl_pipeline_logic_gen(stages, 'top') == g['vhdl']
    assert emit.verilog_generate_io_wrapper(stages, 'top', True) == g['verilog_io']
    assert emit.vhdl_generate_io_wrapper(stages, 'top', True) == g['vhdl_io']
    assert emit.rtl_binder_gen(stages, 'top_wrapper') == g['binder']


@pytest.mark.parametrize('name', CASES)
def test_to_pipeline_matches_the_reference(gold, name):
    n_checked = 0
    for st, g in zip(_stages(name, gold), gold[name]['stages']):
        for cut, want in g['to_pipeline'].items():
            if not _ok(want):
                with pytest.raises(Exception):  # (a stage without ops: KeyError in the reference, too)
                    emit.to_pipeline(st, float(cut))
                continue
            got = emit.to_pipeline(st, float(cut))
            assert len(got) == len(want['stages'])
            for a, b in zip(got, want['stages']):
                assert list(a['shape']) == b['shape']
                assert a['inp_shifts'].tolist() == b['inp_shifts'] and a['out_idxs'].tolist() == b['out_idxs']
                assert a['out_shifts'].tolist() == b['out_shifts'] and a['out_negs'].tolist() == b['out_negs']
                assert a['ops_i'].tolist() == [o[:4] for o in b['ops']]
                assert a['ops_f'].tolist() == [[*o[4], o[5], o[6]] for o in b['ops']]  # exact doubles
            n_checked += 1
            if _ok(want['verilog']):
                assert emit.verilog_pipeline_logic_gen(got, 'pm', register_layers=1) == want['verilog']
                assert emit.verilog_pipeline_logic_gen(got, 'pm', print_latency=True, register_layers=3)['pm'] == want['verilog_r3']
                assert emit.vhdl_pipeline_logic_gen(got, 'pm', register_layers=2) == want['vhdl']
                assert emit.verilog_generate_io_wrapper(got, 'pm', True) == want['verilog_io']
                assert emit.vhdl_generate_io_wrapper(got, 'pm', True) == want['vhdl_io']
                assert emit.rtl_binder_gen(got, 'pm_wrapper', 1, 2) == want['binder']
    assert n_checked > 0


def test_pipelined_stages_compute_the_same_function():
    """Replaying the register stages one after the other reproduces the constant matrix of the combinational graph."""
    st = _stages('int_16x16_int8_default')[0]
    comb = pipeline_from_arrays([st]).solutions[0]
    for cut in (1.0, 2.0, 5.0):
        parts = emit.to_pipeline(st, cut)
        x = np.identity(st['shape'][0])
        for s in pipeline_from_arrays(parts).solutions:
            x = s(x)
        assert np.array_equal(x.astype(np.float32), comb.kernel)


def test_containers_and_arrays_are_interchangeable():
    st = _stages('c1_8x8_int4_default')[0]
    comb = pipeline_from_arrays([st]).solutions[0]
    assert emit.verilog_comb_logic_gen(comb, 'm') == emit.verilog_comb_logic_gen(st, 'm')
    assert emit.hls_logic_and_bridge_gen(comb, 'f', 'vitis') == emit.hls_logic_and_bridge_gen(st, 'f', 'vitis')
    a, b = emit.to_pipeline(comb, 2.0), emit.to_pipeline(st, 2.0)
    assert all(np.array_equal(x['ops_i'], y['ops_i']) and np.array_equal(x['ops_f'], y['ops_f']) for x, y in zip(a, b))


def test_foreign_opcodes_are_rejected():
    st = _stages('c1_8x8_int4_default')[0]
    st['ops_i'] = st['ops_i'].copy()
    st['ops_i'][-1, 2] = 7  # a multiplier: not an adder graph
    with pytest.raises(ValueError, match='outside the CMVM path'):
        emit.verilog_comb_logic_gen(st, 'm')
    with pytest.raises(ValueError, match='outside the CMVM path'):
        emit.to_pipeline(st, 2.0)
    with pytest.raises(ValueError, match='Unsupported flavor'):
        emit.hls_logic_and_bridge_gen(_stages('c1_8x8_int4_default')[0], 'f', 'quartus')


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['c1_8x8_int4_default', 'int_16x16_int8_default', 'pytest_8_b4_harddc2_add1', 'int_12x20_int6_harddc1'])
def test_gpu_result_arrays_emit_the_reference_text(cuda_binary, gold, name):
    """The whole chain on the B200: CUDA solve -> flat arrays -> pipelining / emitters, no Op objects in between; the text
    equals what the reference's emitters write for the reference's own solve of the same matrix."""
    meta = golden_cases()[name]
    extra, _ = load_golden(name)
    raw = cuda_binary.solve_raw(extra['kernel'], **meta['kwargs'])
    g = gold[name]
    assert emit.verilog_pipeline_logic_gen(raw, 'top') == g['pipeline']['verilog']
    assert emit.vhdl_generate_io_wrapper(raw, 'top', True) == g['pipeline']['vhdl_io']
    for i, (st, gs) in enumerate(zip(raw.stages, g['stages'])):
        assert emit.hls_logic_and_bridge_gen(st, f'f{i}', 'vitis', pragmas=['#pragma HLS INLINE'])[0] == gs['hls']['vitis'][0]
        assert emit.vhdl_comb_logic_gen(st, f'm{i}', print_latency=(i == 1)) == gs['vhdl']
    for cut, want in g['stages'][0]['to_pipeline'].items():
        if _ok(want) and _ok(want['verilog']):
            assert emit.verilog_pipeline_logic_gen(emit.to_pipeline(raw.stages[0], float(cut)), 'pm') == want['verilog']


def _same_stages(got, want):
    assert len(got) == len(want)
    for a, b in zip(got, want):
        assert list(a['shape']) == b['shape'] and a['inp_shifts'].tolist() == b['inp_shifts'] and a['out_idxs'].tolist() == b['out_idxs']
        assert a['out_shifts'].tolist() == b['out_shifts'] and a['out_negs'].tolist() == b['out_negs']
        assert a['ops_i'].tolist() == [o[:4] for o in b['ops']]
        assert a['ops_f'].tolist() == [[*o[4], o[5], o[6]] for o in b['ops']]  # exact doubles


def _has_constants(stages):
    """Would the reference tracer see a constant (an input with min == max, an output that reads no op)?"""
    q = np.asarray(stages[0]['ops_f'])[np.asarray(stages[0]['ops_i'])[:, 2] == -1][:, :2]
    n_inputs = int(np.count_nonzero(np.asarray(stages[0]['ops_i'])[:, 2] == -1))
    return bool((q[:, 0] == q[:, 1]).any()) or n_inputs < stages[0]['shape'][0] or any((np.asarray(st['out_idxs']) < 0).any() for st in stages)


@pytest.mark.parametrize('name', CASES)
def test_retiming_matches_the_reference_tracer(gold, name):
    """``retime_pipeline`` (bisection of the cutoff, re-tracing the adder graph for every cutoff tried) against what the
    reference's own ``retime_pipeline`` -- FixedVariable replay + comb_trace -- returned when the golden file was made:
    the solver's two-stage result retimed as it is, and stage 0 split at several cutoffs with ``retiming=True``."""
    stages, g = _stages(name, gold), gold[name]
    n_checked = 0
    if _ok(g['pipeline_retimed']):
        got = emit.retime_pipeline(stages)
        _same_stages(got, g['pipeline_retimed'])
        n_checked += 1
        if 'pipeline_retimed_text' in g:  # ... and the emitters on the retimed stages (a dead output is a constant-0 op there)
            txt = g['pipeline_retimed_text']
            assert emit.verilog_pipeline_logic_gen(got, 'rt') == txt['verilog']
            assert emit.vhdl_pipeline_logic_gen(got, 'rt') == txt['vhdl']
            assert [list(emit.hls_logic_and_bridge_gen(s, f'rt{k}', 'vitis')) for k, s in enumerate(got)] == txt['hls']
            assert emit.verilog_generate_io_wrapper(got, 'rt', True) == txt['verilog_io']
    for cut, want in g['stages'][0]['to_pipeline'].items():
        if not _ok(want) or not _ok(want['retimed']):
            continue
        _same_stages(emit.to_pipeline(stages[0], float(cut), retiming=True), want['retimed'])
        n_checked += 1
    assert n_checked > 0


@pytest.mark.skipif(not __import__('ref_trace').available(), reason='needs the da4ml source tree oracle/_ref is built from')
def test_retiming_is_delegated_to_the_reference_tracer():
    """``retiming=True, da4ml=<package>`` hands the split to the reference's own ``retime_pipeline`` and returns flat stages
    (the route for graphs in which the tracer produces constants); equal to the reference's ``to_pipeline(..., retiming=True)``
    and, for this constant-free graph, to the native retiming."""
    import importlib
    import sys

    import ref_trace
    from oracle import port

    T, _ = ref_trace.load(None, port.get_lsb_loc, port.iceil_log2, port.cost_add)
    P = importlib.import_module('da4ml.trace.pipeline')
    st = _stages('pytest_8_b4_harddc2_add1')[0]
    comb = pipeline_from_arrays([st], types_module=T).solutions[0]
    for cut in (2.0, 3.0):
        want = P.to_pipeline(comb, cut, retiming=True, verbose=False)
        got = emit.to_pipeline(st, cut, retiming=True, da4ml=sys.modules['da4ml'])
        native = emit.to_pipeline(st, cut, retiming=True)
        assert len(got) == len(want.solutions) == len(native)
        assert all(np.array_equal(a['ops_i'], b['ops_i']) and np.array_equal(a['ops_f'], b['ops_f']) for a, b in zip(got, native))
        for a, b in zip(got, want.solutions):
            assert a['ops_i'].tolist() == [[o.id0, o.id1, o.opcode, o.data] for o in b.ops]
            assert a['ops_f'].tolist() == [[*o.qint, o.latency, o.cost] for o in b.ops]
            assert a['out_idxs'].tolist() == list(b.out_idxs) and tuple(a['shape']) == tuple(b.shape)
