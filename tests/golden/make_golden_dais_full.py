"""Store the reference DAIS interpreter's answers for tests/test_dais_full.py and tests/test_dais_full_gpu.py, so that
they run wherever the reference is absent (the GPU machine included):

    dais_full.npz   for every case: the program (int32 words), the seed and digest of its inputs, and the reference's
                    output (whole for small cases, a digest for large ones) or its error message

Programs come from the reference's own tracing front-end (tests/ref_trace.py, with the reference's compiled solver
behind it): three relu + quantize MLPs, one small program per opcode family, one with several lookup tables.  The
random programs of tests/test_dais_full.py cover what the tracer does not emit reliably.  Needs `make -C oracle`.

    python tests/golden/make_golden_dais_full.py
"""
import sys
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parents[1]))
sys.path.insert(0, str(HERE.parent))

from conftest import digest  # noqa: E402

from oracle import dais_ref, ref  # noqa: E402

MLPS = {'mlp_16_64_32_32_5': [16, 64, 32, 32, 5], 'mlp_16_64_64_64_5': [16, 64, 64, 64, 5], 'mlp_64_128_128_10': [64, 128, 128, 10]}


def tracer():
    import ref_trace

    import da4ml_b200._binary as B

    T = None

    def solver(kernel, **kw):
        stages = ref.solve(kernel, **kw)
        for st in stages:
            st.setdefault('shape', (len(st['inp_shifts']), len(st['out_idxs'])))
            st.setdefault('carry_size', kw.get('carry_size', -1))
            st.setdefault('adder_size', kw.get('adder_size', -1))
        return B.RawPipeline.from_stages(stages).to_pipeline(T)

    T, trace = ref_trace.load(solver, B.get_lsb_loc, B.iceil_log2, B.cost_add)
    return trace


def mlp(trace, sizes, seed):
    """Dense layers of 3-bit-fraction weights; hidden layers relu (i=5, f=3) then wrap to signed (i=4, f=2)."""
    rng = np.random.default_rng(seed)
    n0 = sizes[0]
    x = trace.FixedVariableArray.from_kif(np.ones(n0, int), np.full(n0, 3), np.full(n0, 3))
    h = x
    for l, (a, b) in enumerate(zip(sizes[:-1], sizes[1:])):
        h = h @ (rng.integers(-16, 16, size=(a, b)) / 8.0)
        if l < len(sizes) - 2:
            h = h.relu(i=np.full(b, 5), f=np.full(b, 3)).quantize(1, 4, 2)
    return trace.comb_trace(x, h)


def family_programs(trace):
    """One small traced program per opcode family of the tracing front-end."""
    FVA = trace.FixedVariableArray
    rng = np.random.default_rng(11)

    def inp(n=8, k=1, i=3, f=2):
        return FVA.from_kif(np.full(n, k), np.full(n, i), np.full(n, f))

    def layer(x, n_out=8):
        return x @ (rng.integers(-8, 8, size=(x.shape[0], n_out)) / 4.0)

    out = {}
    x = inp()
    out['relu_quantize'] = trace.comb_trace(x, layer(x).relu(i=np.full(8, 4), f=np.full(8, 1)).quantize(1, 3, 1))
    x = inp()
    out['neg_quantize'] = trace.comb_trace(x, (-layer(x)).quantize(1, 3, 1))
    x = inp()
    out['const_add'] = trace.comb_trace(x, layer(x) + 1.25)
    x = inp()
    h = layer(x)
    out['const'] = trace.comb_trace(x, FVA(np.concatenate([h._vars[:7], [trace.FixedVariable.from_const(2.75, hwconf=h.hwconf)]]), h.solver_options))
    x = inp()
    h = layer(x)
    out['maximum'] = trace.comb_trace(x, np.maximum(h[:4], h[4:]))
    x = inp()
    from da4ml.trace.ops import sort

    out['sort'] = trace.comb_trace(x, sort(layer(x)))
    x = inp()
    h = layer(x)
    out['multiply'] = trace.comb_trace(x, h[:3] * h[3:6])
    x = inp(k=0, i=4, f=0)
    h = layer(x).quantize(0, 4, 0)
    out['bit_and_xor'] = trace.comb_trace(x, FVA(np.concatenate([(h[:4] & h[4:])._vars, (h[:4] ^ h[4:])._vars]), h.solver_options))
    x = inp(k=0, i=4, f=0)
    out['bit_not'] = trace.comb_trace(x, ~layer(x).quantize(0, 4, 0))
    x = inp(n=4, k=1, i=2, f=1)
    h = x.quantize(1, 2, 1)
    table = rng.integers(-100, 100, size=16) / 4.0
    out['lookup'] = trace.comb_trace(x, FVA(np.array([v.lookup(table) for v in h._vars]), h.solver_options))
    x = inp(n=6, k=1, i=2, f=1)
    h = layer(x, 6).quantize(1, 2, 1)
    tables = [rng.integers(-1000, 1000, size=16) / 8.0 for _ in range(3)]
    out['lookup_tables'] = trace.comb_trace(x, FVA(np.array([v.lookup(tables[j % 3]) for j, v in enumerate(h._vars)]), h.solver_options))
    return out


def main():
    import test_dais_full as T

    if not (dais_ref.available() and ref.available()):
        sys.exit('oracle/_ref is not built: run `make -C oracle REF=<da4ml source tree>` first')
    trace = tracer()
    progs = {}
    for name, sizes in MLPS.items():
        progs[name] = mlp(trace, sizes, 0).to_binary()
        print(name, progs[name][4], 'ops', flush=True)
    for name, comb in family_programs(trace).items():
        progs[name] = comb.to_binary()
    for seed in range(T.N_RANDOM):
        progs[f'random{seed}'] = T.random_program(seed)
    progs['lookup_overrun'] = T.lookup_overrun_program()
    out = {}
    for name, prog in progs.items():
        seed, n = T.case_inputs(name, prog)
        x = T.special_inputs(seed, n, int(prog[2]))
        out[f'{name}__program'] = np.asarray(prog, np.int32)
        out[f'{name}__input'] = np.array(digest([('x', x)]))
        try:
            y = dais_ref.run(prog, x)
        except RuntimeError as e:
            out[f'{name}__error'] = np.array(str(e))
            continue
        if y.size <= 4096:
            out[f'{name}__output'] = y
        else:
            out[f'{name}__digest'] = np.array(digest([('y', y)]))
            if name == 'mlp_16_64_32_32_5':
                out[f'{name}__head'] = y[:96]  # what the CPU simulation of the kernel can afford to run
    np.savez_compressed(HERE / 'dais_full.npz', **out)


if __name__ == '__main__':
    main()
