"""Throughput of the complete DAIS interpreter (da4ml_b200.dais) on one GPU; prints one JSON line.

Workloads (programs from tests/golden/dais_full.npz and the solver goldens, traced by the reference front-end):
  mlp_16_64_32_32_5    relu + quantize MLP whose value slots fit a CTA's shared memory (shared regime)
  mlp_64_128_128_10    the same family, too many live values for shared memory (global regime)
  adder_stage          the largest golden adder graph of the solver, new engine against dais_interp_run
Per workload and sample count: device time from CUDA events around the launches on device-resident inputs
(samples/s, op-samples/s), and end to end from host arrays.  The reference's CPU interpreter (oracle/_ref/libdais_ref.so,
built by `make -C oracle`) runs a bounded number of samples with one thread per sample chunk as the baseline.

    python scripts/dais_bench.py [--samples 20,22,24] [--reps 3] [--ref-samples 65536]
"""
import argparse
import json
import os
import subprocess
import sys
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / 'tests'))


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'], capture_output=True, text=True, timeout=30).stdout
        name, power, clock = (s.strip() for s in out.splitlines()[0].split(','))
        return dict(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:  # noqa: BLE001
        return dict(error=str(e))


def inputs(n, n_in, seed=0):
    rng = np.random.default_rng(seed)
    return (rng.integers(-64, 64, size=(n, n_in), dtype=np.int8) / 8.0).astype(np.float64)


def device_rate(p, x_host, reps):
    """ms per call from CUDA events over `reps` calls on device-resident data (after one warm-up call)."""
    import torch

    xd = torch.from_numpy(x_host).cuda()
    y = p.predict(xd)
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        y = p.predict(xd)
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps, y


def host_rate(fn, x, reps):
    fn(x[:1024])
    t = time.perf_counter()
    for _ in range(reps):
        y = fn(x)
    return (time.perf_counter() - t) * 1e3 / reps, y


def reference_rate(prog, x, threads):
    """The reference interpreter on the CPU, sample chunks over `threads` threads (ctypes releases the GIL)."""
    from oracle import dais_ref

    if not dais_ref.available():
        return None
    chunks = np.array_split(x, threads)
    dais_ref.run(prog, x[:64])
    t = time.perf_counter()
    with ThreadPoolExecutor(threads) as ex:
        y = np.concatenate(list(ex.map(lambda c: dais_ref.run(prog, c), chunks)))
    return (time.perf_counter() - t) * 1e3, y


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--samples', default='20,22,24', help='log2 of the sample counts')
    ap.add_argument('--reps', type=int, default=3)
    ap.add_argument('--ref-samples', type=int, default=65536)
    ap.add_argument('--ref-threads', type=int, default=os.cpu_count() or 1)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit('dais_bench.py needs a CUDA device')
    import da4ml_b200._binary as B
    from conftest import GOLDEN, golden_cases
    from da4ml_b200.dais import DaisProgram
    from test_dais_replay import golden_stage_programs

    z = np.load(GOLDEN / 'dais_full.npz')
    progs = {name: z[f'{name}__program'] for name in ('mlp_16_64_32_32_5', 'mlp_64_128_128_10')}
    assert golden_cases()
    stage_tag, stage = max(golden_stage_programs(), key=lambda ts: int(ts[1].to_binary()[4]))
    progs['adder_stage'] = stage.to_binary()
    result = dict(card=card(), workloads=[])
    for name, prog in progs.items():
        p = DaisProgram(prog)
        n_ops = p.info['n_ops']
        ref = reference_rate(prog, inputs(args.ref_samples, p.n_in, 1), args.ref_threads)
        for lg in (int(s) for s in args.samples.split(',')):
            n = 1 << lg
            if n * (p.n_in + p.n_out) * 8 * 2 > 24 << 30:  # keep inputs and outputs of one call under 24 GB
                continue
            x = inputs(n, p.n_in)
            dev_ms, yd = device_rate(p, x, args.reps)
            e2e_ms, yh = host_rate(p.predict, x, max(1, args.reps // 2))
            row = dict(workload=name, info=p.info, samples=n, device_ms=dev_ms, samples_per_s=n / dev_ms * 1e3, op_samples_per_s=n * n_ops / dev_ms * 1e3,
                       end_to_end_ms=e2e_ms, end_to_end_samples_per_s=n / e2e_ms * 1e3,
                       device_equals_host=bool(np.array_equal(yd.cpu().numpy().view(np.uint64), yh.view(np.uint64))))  # fmt: skip
            if name == 'adder_stage':
                row['stage'] = stage_tag
                old_ms, yo = host_rate(lambda a: B.dais_interp_run(prog, a), x, max(1, args.reps // 2))
                row.update(adder_only_end_to_end_ms=old_ms, adder_only_samples_per_s=n / old_ms * 1e3, equals_adder_only=bool(np.array_equal(yo.view(np.uint64), yh.view(np.uint64))))
            if ref is not None:
                m = args.ref_samples
                row['equals_reference'] = bool(np.array_equal(p.predict(inputs(m, p.n_in, 1)).view(np.uint64), ref[1].view(np.uint64)))
            result['workloads'].append(row)
            del x, yd, yh
            torch.cuda.empty_cache()
        if ref is not None:
            result['workloads'].append(dict(workload=name, arm='reference_cpu', samples=args.ref_samples, threads=args.ref_threads, ms=ref[0],
                                            samples_per_s=args.ref_samples / ref[0] * 1e3, op_samples_per_s=args.ref_samples * n_ops / ref[0] * 1e3))  # fmt: skip
        del p
    print(json.dumps(result))


if __name__ == '__main__':
    main()
