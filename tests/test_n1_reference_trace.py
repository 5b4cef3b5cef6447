"""SURVEY 8f N1, reference side (CPU, build container only): the reference's own ``da4ml.trace.FixedVariableArray.matmul``
(trace/fixed_variable_array.py:333-373) is imported from the reference tree with its native module replaced by a stand-in
(tests/ref_trace.py) and pointed at ``SolveBatcher.solve``.  Checks that the two-pass batching is transparent to the real
front-end: the same calls in the same order in both passes, one batched solve, and the traced result of the second pass
equals what the front-end builds call by call.  The solver here is the CPU checker (the CUDA solver needs a GPU; the GPU
suite checks the batched CUDA path against the checker, tests/test_n1_traced_matmul_gpu.py)."""
import numpy as np
import pytest
import ref_trace
from conftest import int_matrix

pytestmark = pytest.mark.skipif(not ref_trace.available(), reason='needs the da4ml source tree oracle/_ref is built from')


def _checker_batch(types_module):
    from oracle import port

    from da4ml_b200._binary import RawPipeline

    def solver(kernels, qintervals=None, latencies=None, **opts):
        out = []
        for i, k in enumerate(kernels):
            stages = port.solve(k, qintervals=None if qintervals is None else qintervals[i], latencies=None if latencies is None else latencies[i], **opts)
            for st in stages:
                st.setdefault('shape', (len(st['inp_shifts']), len(st['out_idxs'])))
                st.setdefault('carry_size', opts.get('carry_size', -1))
                st.setdefault('adder_size', opts.get('adder_size', -1))
            out.append(RawPipeline.from_stages(stages))
        return out

    return solver


def test_reference_matmul_through_the_batcher():
    import da4ml_b200._binary as B
    from da4ml_b200.batching import SolveBatcher

    batcher = SolveBatcher()
    T, trace = ref_trace.load(batcher.solve, B.get_lsb_loc, B.iceil_log2, B.cost_add)
    batcher.types_module = T
    batcher.solver = _checker_batch(T)
    hw = trace.HWConfig(1, -1, -1)
    rng = np.random.default_rng(0)
    hi = 2.0 ** rng.integers(2, 6, (4, 6))
    hi[2] = hi[0]  # two identical rows
    x = trace.FixedVariableArray.from_lhs(low=-hi, high=hi - 1.0, step=np.ones((4, 6)), hwconf=hw)
    W = int_matrix(6, 5, 5, 9)
    y = batcher.run(lambda: x @ W)
    assert y.shape == (4, 5)
    assert len(batcher.calls) == 4 and batcher.raw[0] is batcher.raw[2]
    for c in batcher.calls:
        assert np.array_equal(c.kernel, W) and len(c.qintervals) == 6 and set(c.options) >= {'adder_size', 'carry_size'}
    # the same front-end, call by call (no batcher): identical traced outputs (intervals and latencies of every element)
    from oracle import port

    from da4ml_b200._binary import RawPipeline

    def one(kernel, **kw):
        stages = port.solve(kernel, **{k: v for k, v in kw.items()})
        for st in stages:
            st.setdefault('shape', (len(st['inp_shifts']), len(st['out_idxs'])))
            st.setdefault('carry_size', kw.get('carry_size', -1))
            st.setdefault('adder_size', kw.get('adder_size', -1))
        return RawPipeline.from_stages(stages).to_pipeline(T)

    T2, trace2 = ref_trace.load(one, B.get_lsb_loc, B.iceil_log2, B.cost_add)
    x2 = trace2.FixedVariableArray.from_lhs(low=-hi, high=hi - 1.0, step=np.ones((4, 6)), hwconf=trace2.HWConfig(1, -1, -1))
    y2 = x2 @ W
    for a, b in zip(y._vars.ravel(), y2._vars.ravel(), strict=True):
        assert (a.low, a.high, a.step, a.latency) == (b.low, b.high, b.step, b.latency)
