"""SURVEY 8f N2: replay of the adder graphs with the DAIS int64 semantics.  CPU: the compiled reference interpreter
(oracle/_ref/libdais_ref.so) agrees with the float replay on in-range inputs.  GPU: the CUDA replay equals the reference
interpreter bit for bit, including the wrap-around of out-of-range inputs.  The interpreter's answers (a digest for the
largest) are stored in tests/golden/dais_ref.npz (written by tests/golden/make_golden_ref_outputs.py)."""
import hashlib

import numpy as np
import pytest
from conftest import GOLDEN, digest, golden_cases, int_matrix, load_golden

from da4ml_b200.types import pipeline_from_arrays


@pytest.fixture(scope='module')
def gold():
    return np.load(GOLDEN / 'dais_ref.npz')


def golden_stage_programs():
    out = []
    for name, meta in golden_cases().items():
        _, stages = load_golden(name)
        for st in stages:
            st['shape'] = (len(st['inp_shifts']), len(st['out_idxs']))
            st['carry_size'] = st['adder_size'] = -1
        for i, sol in enumerate(pipeline_from_arrays(stages).solutions):
            out.append((f'{name}/s{i}', sol))
    return out


def float_replay_inputs():
    """(tag, program, samples): stage-0 graphs with the default 8-bit inputs, every sample in range."""
    rng = np.random.default_rng(0)
    for tag, sol in golden_stage_programs():
        if '/s0' not in tag or 'hetero' in tag:
            continue
        yield tag, sol, rng.integers(-128, 128, size=(9, sol.shape[0])).astype(np.float64)


def cuda_replay_inputs():
    """(tag, program, samples): every golden stage, in-range samples and out-of-range ones that wrap around."""
    rng = np.random.default_rng(1)
    for tag, sol in golden_stage_programs():
        n_in = sol.shape[0]
        yield tag, sol, np.concatenate([rng.integers(-128, 128, size=(33, n_in)), rng.integers(-5000, 5000, size=(8, n_in)) / 8.0]).astype(np.float64)


SOLVED_KW = dict(search_all_decompose_dc=False, decompose_dc=-1)


def solved_matrix_case():
    return int_matrix(64, 48, 8, 21), np.random.default_rng(2).integers(-128, 128, size=(5000, 64)).astype(np.float64)


def call_key(prog, x):
    """Name under which the interpreter's answer to one call (program, samples) is stored."""
    h = hashlib.sha256(np.ascontiguousarray(prog, dtype=np.int32).tobytes())
    h.update(np.ascontiguousarray(x, dtype=np.float64).tobytes())
    return 'call_' + h.hexdigest()[:32]


def test_reference_interpreter_agrees_with_float_replay(gold):
    for tag, sol, x in float_replay_inputs():
        assert np.array_equal(gold['float__' + tag.replace('/', '__')], sol(x)), tag


@pytest.mark.gpu
def test_cuda_replay_matches_reference_interpreter(cuda_binary, gold):
    for tag, sol, x in cuda_replay_inputs():
        want = gold['cuda__' + tag.replace('/', '__')]
        got = sol.predict(x)
        assert got.dtype == np.float64 and np.array_equal(got.view(np.uint64), want.view(np.uint64)), tag


@pytest.mark.gpu
def test_cuda_replay_of_a_solved_matrix(cuda_binary, gold):
    W, x = solved_matrix_case()
    pipe = cuda_binary.solve(W, **SOLVED_KW)
    sol = pipe.solutions[0]
    assert digest([('program', sol.to_binary())]) == str(gold['solved_program'])  # the program the stored answer belongs to
    got = sol.predict(x)
    assert digest([('out', got)]) == str(gold['solved_out'])
    assert np.array_equal(got, sol(x))  # in-range inputs: fixed-point replay == exact arithmetic
    with pytest.raises(RuntimeError, match='Unknown opcode'):
        bad = sol.to_binary()
        bad[6 + 64 + 3 * 48 + 8 * 70] = 7  # turn one op into a multiplication
        cuda_binary.dais_interp_run(bad, x[:4])


def _raw_from_golden(name):
    import da4ml_b200._binary as B

    extra, stages = load_golden(name)
    for st in stages:
        st['shape'] = (len(st['inp_shifts']), len(st['out_idxs']))
        st['carry_size'] = st['adder_size'] = -1
    want = extra['kernel'].copy()
    if 'qint' in extra:  # inputs whose interval is {0, 0} are dropped by the solver (state_opr.cc:92-97)
        want[(extra['qint'][:, 0] == 0) & (extra['qint'][:, 1] == 0)] = 0
    return B.RawPipeline.from_stages(stages), want


def test_kernel_from_fixed_point_probes(monkeypatch, gold):
    """``RawPipeline.kernel`` probes every stage with one quantum per input under the DAIS fixed-point semantics; with
    the reference interpreter standing in for the CUDA one (its stored answers to exactly these probes), it reproduces
    the matrix of every golden case."""
    import da4ml_b200._binary as B

    def reference_answer(prog, x, n_threads=1):
        key = call_key(prog, x)
        assert key in gold.files, 'a probe the reference interpreter was not asked when the golden file was made'
        return gold[key].copy()

    monkeypatch.setattr(B, 'dais_interp_run', reference_answer)
    for name in golden_cases():
        raw, want = _raw_from_golden(name)
        assert np.array_equal(raw.kernel, want), name
        for i, sol in enumerate(raw.to_pipeline().solutions):
            assert np.array_equal(raw.stage_kernel(i), sol.kernel), (name, i)


@pytest.mark.gpu
def test_raw_result_replays_and_serialises_without_containers(cuda_binary, tmp_path):
    """SURVEY 8f N3: the flat result of a default two-stage solve is replayed on the GPU stage by stage, reproduces
    the matrix, and writes the same JSON / DAIS words as the container path."""
    import json

    from da4ml_b200.types import Pipeline

    W = int_matrix(48, 40, 8, 5)
    raw = cuda_binary.solve_raw(W)
    assert len(raw.stages) == 2
    assert np.array_equal(raw.kernel, W)
    pipe = raw.to_pipeline()
    x = np.random.default_rng(3).integers(-128, 128, size=(257, 48)).astype(np.float64)
    assert np.array_equal(raw.predict_stage(0, x), pipe.solutions[0](x))
    assert raw.to_json() == json.dumps(pipe, separators=(',', ':'))
    for b, sol in zip(raw.to_binary(), pipe.solutions):
        assert np.array_equal(b, sol.to_binary())
    raw.save(tmp_path / 'p.json')
    assert Pipeline.load(tmp_path / 'p.json') == pipe
    raw.save_binary(tmp_path / 'p.bin')
    assert np.array_equal(np.fromfile(tmp_path / 'p.bin.1', dtype=np.int32), pipe.solutions[1].to_binary())
    for name in golden_cases():  # reference results replayed by the CUDA interpreter
        gold, want = _raw_from_golden(name)
        assert np.array_equal(gold.kernel, want), name


def test_replay_rejects_malformed_headers_before_touching_the_device():
    """Header validation of a foreign DAIS file happens on the host (reference DAISInterpreter.cc:11-42: size and version
    checks) -- no GPU is needed to be told the file is bad."""
    import da4ml_b200._binary as B

    x = np.zeros((1, 2))
    good = np.array([1, 0, 2, 1, 2, 0, 0, 0, 1, 0, 0] + [-1, 0, 0, 0, 0, 0, 0, 0] + [-1, 1, 0, 0, 0, 0, 0, 0], dtype=np.int32)
    for mutate, msg in (
        (lambda p: p[:4], 'too small'),
        (lambda p: np.concatenate([[2], p[1:]]).astype(np.int32), 'version mismatch'),
        (lambda p: np.concatenate([p[:2], [-2], p[3:]]).astype(np.int32), 'negative count'),
        (lambda p: p[:-3], 'size mismatch'),
        (lambda p: np.concatenate([p[:5], [1], p[6:]]).astype(np.int32), 'size mismatch'),
    ):
        with pytest.raises(RuntimeError, match=msg):
            B.dais_interp_run(np.ascontiguousarray(mutate(good.copy())), x)
