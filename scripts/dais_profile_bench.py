"""Throughput of DaisProgram.profile against DaisProgram.predict on one GPU; prints one JSON line.

Workloads (programs from tests/golden/dais_full.npz, traced by the reference front-end):
  mlp_16_64_32_32_5    relu + quantize MLP whose value slots fit a CTA's shared memory (shared regime)
  mlp_64_128_128_10    the same family, too many live values for shared memory (global regime)
Per workload and sample count: device time from CUDA events around `reps` calls on device-resident float64 inputs,
for predict, for profile (one pass over every op with per-warp reductions, totals copied back once per call), and for
values of 8 ops.  The card's name, power limit and clocks are read in the same run.

    python scripts/dais_profile_bench.py [--samples 20,22] [--reps 3]
"""
import argparse
import json
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / 'tests'))


def card():
    try:
        q = 'name,power.limit,clocks.max.sm,clocks.sm'
        out = subprocess.run(['nvidia-smi', f'--query-gpu={q}', '--format=csv,noheader'], capture_output=True, text=True, timeout=30).stdout
        name, power, max_clock, clock = (s.strip() for s in out.splitlines()[0].split(','))
        return dict(name=name, power_limit=power, max_sm_clock=max_clock, sm_clock_at_start=clock)
    except Exception as e:  # noqa: BLE001
        return dict(error=str(e))


def timed(fn, reps):
    import torch

    out = fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--samples', default='20,22', help='log2 of the sample counts')
    ap.add_argument('--reps', type=int, default=3)
    args = ap.parse_args()
    import torch

    if not torch.cuda.is_available():
        sys.exit('dais_profile_bench.py needs a CUDA device')
    from conftest import GOLDEN
    from da4ml_b200.dais import DaisProgram

    z = np.load(GOLDEN / 'dais_full.npz')
    result = dict(card=card(), workloads=[])
    for name in ('mlp_16_64_32_32_5', 'mlp_64_128_128_10'):
        p = DaisProgram(z[f'{name}__program'])
        ops = np.linspace(0, p.n_ops - 1, 8).astype(np.int64)
        for lg in (int(s) for s in args.samples.split(',')):
            n = 1 << lg
            rng = np.random.default_rng(lg)
            x = torch.from_numpy(rng.integers(-64, 64, size=(n, p.n_in)) / 8.0).cuda()
            pred_ms, _ = timed(lambda: p.predict(x), args.reps)
            prof_ms, r = timed(lambda: p.profile(x), args.reps)
            val_ms, v = timed(lambda: p.values(x, ops), args.reps)
            vh = v.cpu().numpy()
            row = dict(workload=name, info=p.info, samples=n, predict_ms=pred_ms, profile_ms=prof_ms, values8_ms=val_ms,
                       predict_samples_per_s=n / pred_ms * 1e3, profile_samples_per_s=n / prof_ms * 1e3,
                       profile_over_predict=pred_ms / prof_ms, values8_samples_per_s=n / val_ms * 1e3,
                       profile_op_samples_per_s=n * p.n_ops / prof_ms * 1e3,
                       values_agree_with_profile=bool(np.array_equal(vh.min(axis=0), r.min[ops]) and np.array_equal(vh.max(axis=0), r.max[ops])),
                       wrapped_total=int(r.wrapped.sum()), outside_total=int(r.outside.sum()))  # fmt: skip
            result['workloads'].append(row)
            del x, v
            torch.cuda.empty_cache()
        del p
    result['card_after'] = card()
    print(json.dumps(result))


if __name__ == '__main__':
    main()
