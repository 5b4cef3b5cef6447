"""Store what the reference's own object code (oracle/_ref, built by `make -C oracle` from a da4ml source tree) answers
for the inputs of the tests that compare with it, so that those tests run wherever the reference is absent:

    oracle_digests.json   tests/test_oracle.py::test_port_matches_reference_random and tests/test_oracle_cross.py
                          (ref.solve / solve_single / helpers): a digest of every answer, as conftest.digest computes it
    dais_ref.npz          tests/test_dais_replay.py (the reference DAIS interpreter): the answers, a digest for the largest

Every input is rebuilt by the test module's own case builder; a digest of each input matrix is stored next to the
answer so that a test can tell it still asks the question the answer belongs to.

    python tests/golden/make_golden_ref_outputs.py
"""
import json
import sys
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
sys.path.insert(0, str(HERE.parents[1]))
sys.path.insert(0, str(HERE.parent))

from conftest import digest, golden_cases, stage_digest  # noqa: E402

from oracle import dais_ref, ref  # noqa: E402


def case(W, result):
    return {'kernel': digest([('kernel', W)]), 'result': result}


def oracle_digests():
    import test_oracle
    import test_oracle_cross as T

    out = {}
    for seed in range(6):
        W, kw = test_oracle.random_case(seed)
        out[f'random{seed}'] = case(W, stage_digest(ref.solve(W, **kw)))
    for seed in range(60):
        W, _, kw = T.single_case(seed)
        out[f'single{seed}'] = case(W, stage_digest([ref.solve_single(W, **kw)]))
    for seed in range(40):
        W, _, kw = T.full_case(seed)
        out[f'full{seed}'] = case(W, stage_digest(ref.solve(W, **kw)))
    for seed in range(20):
        W, ints, Wi = T.helpers_case(seed)
        out[f'helpers{seed}'] = case(W, digest(sorted(T.helpers_outputs(ref, W, ints, Wi).items())))
    return out


def dais():
    import test_dais_replay as T

    import da4ml_b200._binary as B
    from da4ml_b200.types import pipeline_from_arrays

    out = {}
    for tag, sol, x in T.float_replay_inputs():
        out['float__' + tag.replace('/', '__')] = dais_ref.run(sol.to_binary(), x)
    for tag, sol, x in T.cuda_replay_inputs():
        out['cuda__' + tag.replace('/', '__')] = dais_ref.run(sol.to_binary(), x)
    W, x = T.solved_matrix_case()
    sol = pipeline_from_arrays(ref.solve(W, **T.SOLVED_KW)).solutions[0]
    out['solved_program'] = np.array(digest([('program', sol.to_binary())]))
    out['solved_out'] = np.array(digest([('out', dais_ref.run(sol.to_binary(), x))]))

    def record(prog, x, n_threads=1):  # the probes RawPipeline.kernel / stage_kernel send to the interpreter
        y = dais_ref.run(prog, x)
        out[T.call_key(prog, x)] = y
        return y

    B.dais_interp_run = record
    for name in golden_cases():
        raw, _ = T._raw_from_golden(name)
        raw.kernel
        for i in range(len(raw.stages)):
            raw.stage_kernel(i)
    return out


def main():
    if not (ref.available() and dais_ref.available()):
        sys.exit('oracle/_ref is not built: run `make -C oracle REF=<da4ml source tree>` first')
    (HERE / 'oracle_digests.json').write_text(json.dumps(oracle_digests(), indent=0) + '\n')
    np.savez_compressed(HERE / 'dais_ref.npz', **dais())


if __name__ == '__main__':
    main()
