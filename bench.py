"""bench.py -- CMVM solve throughput on B200 (BASELINE.json metric: 256x256 int8 matrices/s).

    python bench.py --gpus N --steps K --warmup W            # CUDA path (this repository)
    python bench.py --impl reference --gpus N ...            # the reference's own CPU code (oracle/_ref)
    python bench.py ... --dump-outputs DIR                    # also write the last timed step's result arrays to DIR

A "step" = one pass of the hot path over one batch: every rank solves ``--batch`` synthetic 256x256 int8 constant
matrices with the reference's default call (``solve(W)``: search over all decompose_dc candidates, two CSE stages each).
Every step takes NEW matrices (seed + step); the steps whose matrices have a golden answer from the reference's own object
code (tests/golden/index.json) are checked against it.  Matrices are independent, so ranks shard them with no data-path
collective (weak scaling).  The line also carries a `c4` sub-record: BASELINE config 4, a fixed job of 64 128x128 int6
matrices split over the ranks (strong scaling).  Prints ONE JSON line on rank 0.  Writes nothing into the repository:
figures it has to count at run time are cached in the temporary directory.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
sys.dont_write_bytecode = True  # no __pycache__ in the tree for the modules imported from here on

ALGO_BYTES = ROOT / 'profiles' / 'algo_bytes.json'  # committed figures
ALGO_BYTES_RUN = Path(tempfile.gettempdir()) / 'da4ml_b200_bench' / 'algo_bytes.json'  # figures counted by earlier runs
DUMP_LIMIT = 64 << 20  # bytes of --dump-outputs
STAGE_KEYS = ('inp_shifts', 'out_idxs', 'out_shifts', 'out_negs', 'ops_i', 'ops_f')

METRIC = 'cmvm_solve_throughput_256x256_int8'  # BASELINE.json metric (default workload)
UNIT = 'matrices/s'


def metric_name(n: int, bits: int) -> str:
    return f'cmvm_solve_throughput_{n}x{n}_int{bits}'


def workload_name(n: int, bits: int, batch: int) -> str:
    """One string for both arms (the driver compares them)."""
    return f'{n}x{n} int{bits} uniform random constant matrix, default solve() (search over all decompose_dc candidates, 2 CSE stages each), batch {batch}/rank, new matrices every step (seed + step)'


def make_matrix(n: int, bits: int, seed: int) -> np.ndarray:
    rng = np.random.default_rng(seed)
    return rng.integers(-(2 ** (bits - 1)), 2 ** (bits - 1), size=(n, n)).astype(np.float32)


def golden_default(n: int, bits: int, seed: int):
    """Reference answer of the default solve of make_matrix(n, bits, seed), if the golden index has one."""
    idx_path = ROOT / 'tests' / 'golden' / 'index.json'
    if not idx_path.exists():
        return None
    idx = json.loads(idx_path.read_text())
    for name, v in idx.items():
        if v.get('spec') == ['int', n, n, bits, seed] and v.get('kwargs') == {}:
            return dict(name=name, **v)
    return None


def stage_digest(stages) -> str:
    import hashlib

    h = hashlib.sha256()
    for st in stages:
        for k in STAGE_KEYS:
            a = np.ascontiguousarray(st[k])
            h.update(k.encode())
            h.update(str(a.shape).encode())
            h.update(a.tobytes())
    return h.hexdigest()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    QUERY = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'

    def __init__(self, index: int):
        self.index = index
        self.rows: list[list[str]] = []
        self._stop = threading.Event()
        self._thr = None

    def _run(self):
        while not self._stop.is_set():
            try:
                out = subprocess.run(['nvidia-smi', f'--query-gpu={self.QUERY}', '--format=csv,noheader,nounits', '-i', str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([v.strip() for v in out.split(',')])
            except Exception:
                pass
            self._stop.wait(0.2)

    def __enter__(self):
        self._thr = threading.Thread(target=self._run, daemon=True)
        self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._thr.join(timeout=6)

    def summary(self) -> dict:
        if not self.rows:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace('.', '').isdigit())
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith('active') for r in self.rows if len(r) > 3 + i)]
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': float(self.rows[0][1]) if self.rows[0][1].replace('.', '').isdigit() else None,
                'power_w_max': max((float(r[2]) for r in self.rows if r[2].replace('.', '').isdigit()), default=None), 'reasons': reasons, 'samples': len(self.rows)}


def dist_env():
    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    return rank, world, local


def cached_algo_bytes(key: str):
    for cache in (ALGO_BYTES, ALGO_BYTES_RUN):
        value = json.loads(cache.read_text()).get(key) if cache.exists() else None
        if value is not None:
            return value
    return None


def store_algo_bytes(key: str, value: float):
    cache = ALGO_BYTES_RUN
    try:
        known = json.loads(cache.read_text()) if cache.exists() else {}
        known[key] = value
        cache.parent.mkdir(parents=True, exist_ok=True)
        tmp = cache.with_suffix(f'.{os.getpid()}')
        tmp.write_text(json.dumps(known, indent=1, sort_keys=True))
        tmp.replace(cache)
    except (OSError, ValueError):
        pass


def dump_outputs(out_dir: Path, results, prefix: str, limit: int) -> None:
    """The result arrays of one step (what solve_batch_device_raw hands its caller) as <out_dir>/<prefix>m<j>_s<i>_<key>.npy:
    integers as float64 (exact), ops_f as float32.  Above ``limit`` bytes in all, every array keeps the same fraction of its
    rows, drawn with a fixed seed."""
    arrays = {}
    for j, r in enumerate(results):
        for i, st in enumerate(r.stages):
            for k in STAGE_KEYS:
                a = np.asarray(st[k])
                arrays[f'{prefix}m{j}_s{i}_{k}'] = a.astype(np.float32 if a.dtype.kind == 'f' else np.float64)
    total = sum(a.nbytes for a in arrays.values())
    out_dir.mkdir(parents=True, exist_ok=True)
    rng = np.random.default_rng(0)
    for name, a in arrays.items():
        if total > limit and len(a):
            keep = max(1, int(len(a) * limit / total))
            a = a[np.sort(rng.choice(len(a), keep, replace=False))]
        np.save(out_dir / f'{name}.npy', a)


def full_cpu_run(n: int, bits: int, seed: int = 0):
    """The reference's default solve of this workload executed in full, once, by tests/golden/make_golden_large.py
    (wall time, threads, host CPU): the real CPU figure next to the bounded samples taken in the bench run."""
    g = golden_default(n, bits, seed)
    if not g or 'cpu_seconds' not in g:
        return None
    return {'seconds': g['cpu_seconds'], 'threads': g.get('cpu_threads'), 'host': g.get('cpu_model', 'build container'), 'adders': g['n_adders'],
            'matrices_per_s': 1.0 / g['cpu_seconds'], 'what': f'{g["name"]}: oracle/_ref (the reference translation units) run to completion in the build container'}


# ------------------------------------------------------------------------------------------------
def cpu_sample(n: int, bits: int, seed: int, a_total: float | None, seconds: float, threads: int):
    """Bounded sample of the reference CPU path on the same workload.

    The reference cannot finish one 256x256 default solve in bench time (~1.2 h per decompose_dc candidate, single
    threaded; it parallelises only over the <= 10 candidates).  Each of ``threads`` workers runs the reference's own
    greedy loop (create_state / idx_wmc / update_state) on one candidate's stage-0 matrix for ``seconds`` and the
    algorithmic bytes it got through are counted; throughput in matrices/s = bytes/s / (algorithmic bytes of one
    full default solve as the reference executes it, from the CUDA path's exact counters with job sharing off).
    """
    import oracle
    from oracle import port

    mod, kind = oracle.best()
    W = make_matrix(n, bits, seed)
    max_dc = int(np.ceil(np.log2(n)))
    dcs = list(range(-1, max_dc + 1))[: max(1, threads)]
    mats = [port.kernel_decompose(W, dc)[0] for dc in dcs]  # stage-0 matrices of the candidates (CPU restatement)
    results = [None] * len(mats)

    def work(i):
        method = 'wmc-dc' if dcs[i] == -1 else 'wmc'
        if kind == 'reference':
            tr = mod.trace(mats[i], method, max_iters=-1, time_limit_s=seconds, counters=True)
            a = 8.0 * n * n + 12.0 * tr['f0'] + 2.0 * tr['r0'] + 12.0 * float(tr['f_sizes'].sum()) + 10.0 * float(tr['r_sizes'].sum())
            results[i] = (a, tr['seconds'], len(tr['pairs']))
        else:
            r = mod.partial(mats[i], method, -1, seconds)
            a = 8.0 * n * n + 12.0 * r['F0'] + 2.0 * r['R0'] + 12.0 * r['sum_F'] + 10.0 * r['sum_R']
            results[i] = (a, r['seconds'], r['iters'])

    t0 = time.time()
    ths = [threading.Thread(target=work, args=(i,)) for i in range(len(mats))]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    wall = time.time() - t0
    a_sum = sum(r[0] for r in results)
    rate = a_sum / wall  # algorithmic bytes per second over all workers
    iters = [r[2] for r in results]
    info = {
        'kind': kind, 'cores': len(mats), 'algo_bytes_per_s': rate, 'wall_s': wall,
        'sample': f'{len(mats)} thread(s), each: create_state + the first {seconds:.0f} s of the reference greedy loop (idx_* + update_state) on one '
                  f'decompose_dc candidate of the same {n}x{n} int{bits} matrix (iterations done: {iters}); matrices/s = algorithmic bytes/s over '
                  f'the algorithmic bytes of one full default solve (all candidates, as the reference executes them)',
    }
    if a_total:
        info['value'] = rate / a_total
        info['unit'] = UNIT
    return info


# ------------------------------------------------------------------------------------------------
def run_reference(args):
    rank, world, _ = dist_env()
    if rank != 0:
        return 0
    a_total = cached_algo_bytes(f'{args.size}x{args.size}_int{args.bits}_default_seed{args.seed}_reference')
    threads = min(os.cpu_count() or 1, int(np.ceil(np.log2(args.size))) + 2)
    per_step = max(2.0, min(12.0, 72.0 / max(1, args.steps)))  # greedy-loop budget per worker per step (create_state comes on top)
    vals = []
    info = None
    for i in range(args.warmup + args.steps):
        info = cpu_sample(args.size, args.bits, args.seed + max(0, i - args.warmup), a_total, per_step if i >= args.warmup else 1.0, threads)
        if i >= args.warmup:
            vals.append(info.get('value'))
    value = float(np.mean([v for v in vals if v is not None])) if a_total else None
    line = {
        'impl': 'reference', 'metric': metric_name(args.size, args.bits), 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup,
        'ms_per_step': 1e3 * args.batch / value if value else None, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None,
        'dtype': 'int32/f32', 'data': 'synthetic', 'config': {'workload': workload_name(args.size, args.bits, args.batch)},
        'extrapolated': True,
        'extrapolation': 'value = (algorithmic bytes/s of a bounded sample of the reference greedy loop on this box) / (algorithmic bytes of one full reference solve); '
                         'the reference needs hours per matrix, see full_run_cached for the one complete run',
        'full_run_cached': full_cpu_run(args.size, args.bits, 0),
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': info['cores'], 'kind': info['kind'], 'sample': info['sample']},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    if a_total is None:
        line['note'] = 'algorithmic bytes of the full solve unknown (run the CUDA arm once to cache profiles/algo_bytes.json); reporting bytes/s only'
        line['cpu_baseline']['algo_bytes_per_s'] = info['algo_bytes_per_s']
    print(json.dumps(line), flush=True)
    return 0


# ------------------------------------------------------------------------------------------------
def accounting_bytes(B, dev_ptr, shape, share: bool) -> float:
    """Exact algorithmic bytes (SURVEY 8d) of the default solve of one device-resident matrix: one pass in accounting mode."""
    B.set_accounting(True)
    B.set_job_sharing(share)
    try:
        r = B.solve_batch_device_raw([dev_ptr], [shape])[0]
    finally:
        B.set_accounting(False)
        B.set_job_sharing(True)
    return float(r.profile['algo_bytes'])


def run_cuda(args):
    import torch
    import torch.distributed as dist

    import da4ml_b200._binary as B
    from da4ml_b200 import cmvm
    from da4ml_b200.distributed import solve_sharded

    rank, world, local = dist_env()
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', rank=rank, world_size=world)
    if not torch.cuda.is_available():
        raise SystemExit('bench.py needs a CUDA device (the CMVM solver has no CPU fallback)')
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    stream = torch.cuda.current_stream()
    B.set_stream(stream.cuda_stream)

    n, bits = args.size, args.bits
    # per-rank batch of distinct matrices, new ones every step.  Default: weak scaling (fixed work per GPU).  --total T: a
    # fixed job of T matrices split over the ranks (strong scaling, e.g. BASELINE config 4: --size 128 --bits 6 --total 64).
    if args.total > 0:
        mine = [i for i in range(args.total) if i % world == rank]
        args.batch = len(mine)
        if not mine:
            raise SystemExit('--total must be at least the number of ranks')
    else:
        mine = [rank * args.batch + i for i in range(args.batch)]
    stride = max(args.total, world * args.batch)

    def step_seeds(step):  # timed step s uses seeds seed + s * stride + (this rank's slots); warm-up steps use seeds far away
        base = args.seed + step * stride if step >= 0 else 100000 + (-step) * stride
        return [base + i for i in mine]

    shapes = [(n, n)] * args.batch

    def stage(seeds):
        mats = [make_matrix(n, bits, s) for s in seeds]
        pinned = [torch.from_numpy(m).pin_memory() for m in mats]
        dmats = [p.to(dev, non_blocking=True) for p in pinned]
        return mats, dmats

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    timed = [stage(step_seeds(s)) for s in range(args.steps)]
    warm = [stage(step_seeds(-1 - s)) for s in range(args.warmup)]
    torch.cuda.synchronize()

    # ---- exact algorithmic bytes of the workload (a deterministic function of the input): accounting passes, cached
    a_run = a_ref = None
    if rank == 0:
        key = f'{n}x{n}_int{bits}_default_seed{args.seed}'
        a_run, a_ref = cached_algo_bytes(key), cached_algo_bytes(key + '_reference')
        if a_run is None or a_ref is None or args.recount:
            d0 = torch.from_numpy(make_matrix(n, bits, args.seed)).to(dev)
            a_run = accounting_bytes(B, d0.data_ptr(), (n, n), share=True)    # what this path executes (identical jobs shared)
            a_ref = accounting_bytes(B, d0.data_ptr(), (n, n), share=False)   # every solve_single the reference executes
            store_algo_bytes(key, a_run)
            store_algo_bytes(key + '_reference', a_ref)
    # ---- warm-up
    for _, dmats in warm:
        B.solve_batch_device_raw([t.data_ptr() for t in dmats], shapes)
    barrier()

    # ---- timed region 1: inputs resident in HBM, CUDA events on the launching stream
    # (per-step working set: histogram segments, cell pools and op tables of the concurrent candidates, several hundred
    #  MB, i.e. larger than the 126 MB L2, and every step solves NEW matrices: nothing of one step survives into the next)
    launches = 0
    solve_ms = 0.0
    solve_launches = 0
    jobs_total = jobs_run = 0
    results = []
    with ClockSampler(local) as clocks:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record(stream)
        for _, dmats in timed:
            res = B.solve_batch_device_raw([t.data_ptr() for t in dmats], shapes)
            launches += res[0].launches
            solve_ms += res[0].profile['solve_kernel_ms']
            solve_launches += res[0].profile['solve_kernel_launches']
            jobs_total += res[0].profile['jobs_total']
            jobs_run += res[0].profile['jobs_run']
            results.append(res)
        e1.record(stream)
        barrier()
        dev_ms = e0.elapsed_time(e1)
    # ---- parity: every timed result whose matrix has a golden answer from the reference's object code
    checked, mismatches = [], []
    for s, res in enumerate(results):
        for seed, r in zip(step_seeds(s), res):
            g = golden_default(n, bits, seed)
            if g is None:
                continue
            ok = r.n_adders == g['n_adders'] and stage_digest(r.stages) == g['sha256']
            checked.append({'seed': seed, 'golden': g['name'], 'adders': r.n_adders, 'ok': bool(ok)})
            if not ok:
                mismatches.append(seed)
    adders = [[r.n_adders for r in res] for res in results]
    # ---- timed region 2 (end to end): host numpy in -> the reference's result type (Pipeline of CombLogic / Op) out,
    # through the public call a user makes (da4ml_b200.cmvm.solve / solve_batch); and the same down to flat arrays only
    barrier()
    t0 = time.perf_counter()
    d2h = 0
    for mats, _ in timed:
        pipes = cmvm.solve_batch(mats) if len(mats) > 1 else [cmvm.solve(mats[0])]
        assert all(len(p.solutions) == 2 for p in pipes)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    barrier()
    t0 = time.perf_counter()
    for mats, _ in timed:
        res = B.solve_batch_raw(mats)
        d2h = sum(sum(a.nbytes for k, a in st.items() if hasattr(a, 'nbytes')) for r in res for st in r.stages)
    torch.cuda.synchronize()
    e2e_raw_s = time.perf_counter() - t0
    h2d = sum(m.nbytes for m in timed[0][0])

    # ---- BASELINE config 4 as a sub-record: a fixed job of 64 128x128 int6 matrices over the ranks (strong scaling)
    c4 = None
    if args.c4 > 0:
        c4_mats = [make_matrix(128, 6, s) for s in range(args.c4)]
        solve_sharded(c4_mats, gather=False)  # warm-up: the same job once, untimed (the grow-only work buffers reach their final size)
        barrier()
        t0 = time.perf_counter()
        part = solve_sharded(c4_mats, gather=False)  # this rank's {index: RawPipeline}; no collective in the timed path
        torch.cuda.synchronize()
        c4_s = time.perf_counter() - t0
        c4_local = part if isinstance(part, dict) else dict(enumerate(part))
        c4_ok = []
        for i, r in c4_local.items():
            g = golden_default(128, 6, i)
            if g is not None:
                c4_ok.append(bool(r.n_adders == g['n_adders'] and stage_digest(r.stages) == g['sha256']))
        t_c4 = torch.tensor([c4_s, float(len(c4_ok)), float(sum(c4_ok))], dtype=torch.float64, device=dev)
        if world > 1:
            mx = t_c4.clone()
            dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            dist.all_reduce(t_c4, op=dist.ReduceOp.SUM)
            c4_time = float(mx[0])
        else:
            c4_time = c4_s
        c4 = {'workload': f'{args.c4} x 128x128 int6 default solve(), one fixed job sharded over {world} rank(s) by da4ml_b200.distributed.solve_sharded (host arrays in, flat result arrays out)',
              'value': args.c4 / c4_time, 'unit': UNIT, 'seconds': c4_time, 'scaling': 'strong', 'warmup': 'the same job once, untimed', 'parity_checked': int(t_c4[1]), 'parity_ok': int(t_c4[2])}
        if world > 1:  # the same job on ONE GPU, in the same run: the denominator of the strong-scaling efficiency
            barrier()
            if rank == 0:
                B.solve_batch_raw(c4_mats)  # (untimed: buffers for the 64-matrix batch, as for the sharded job above)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                B.solve_batch_raw(c4_mats)
                torch.cuda.synchronize()
                c4['seconds_one_gpu'] = time.perf_counter() - t0
                c4['strong_efficiency'] = c4['seconds_one_gpu'] / (world * c4_time)
            barrier()
        elif rank == 0:
            a4 = cached_algo_bytes('128x128_int6_default_seed0')
            if a4 is None or args.recount:
                d4 = torch.from_numpy(c4_mats[0]).to(dev)
                a4 = accounting_bytes(B, d4.data_ptr(), (128, 128), share=True)
                store_algo_bytes('128x128_int6_default_seed0', a4)
            peaks = json.loads((ROOT / 'MEASURED_PEAKS.json').read_text()) if (ROOT / 'MEASURED_PEAKS.json').exists() else {}
            pk = float(peaks.get('hbm_gbs', 6650.0))
            ach = a4 * args.c4 / c4_time / 1e9
            c4['roofline'] = {'bound': 'hbm', 'achieved': ach, 'peak': pk, 'unit': 'GB/s', 'frac': ach / pk,
                              'note': 'algorithmic bytes of seed 0 (exact, accounting mode) x 64 matrices / end-to-end wall time of the job'}

    t_dev = torch.tensor([dev_ms, 1e3 * e2e_s, 1e3 * e2e_raw_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_dev, op=dist.ReduceOp.MAX)
    dev_ms_max, e2e_ms_max, e2e_raw_ms_max = (float(v) for v in t_dev.cpu())
    total = (args.total if args.total > 0 else args.batch * world) * args.steps
    value = total / (dev_ms_max * 1e-3)

    if rank == 0:
        peaks = {}
        pk = ROOT / 'MEASURED_PEAKS.json'
        if pk.exists():
            peaks = json.loads(pk.read_text())
        peak_gbs = float(peaks.get('hbm_gbs', 6650.0))
        peak_src = 'measured (MEASURED_PEAKS.json hbm_gbs)' if 'hbm_gbs' in peaks else 'fallback 6.65 TB/s'
        # dominant kernel: the persistent solve kernel.  Algorithmic bytes of everything those launches solved / their CUDA-event time.
        a_step = (a_run or 0.0) * args.batch
        achieved = (a_step * args.steps) / (solve_ms * 1e-3) / 1e9 if solve_ms > 0 else None
        traffic = None
        tj = ROOT / 'profiles' / 'traffic.json'
        if tj.exists():
            traffic = json.loads(tj.read_text()).get('solve_kernel_dram_bytes_per_launch')
        cpu = cpu_sample(n, bits, args.seed, a_ref, args.cpu_seconds, 1) if args.cpu_seconds > 0 else None
        line = {
            'metric': metric_name(n, bits), 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps, 'warmup': args.warmup,
            'ms_per_step': dev_ms_max / args.steps, 'higher_is_better': True, 'scaling': 'strong' if args.total > 0 else 'weak', 'vs_baseline': None,
            'dtype': 'u32 sign planes / f32 intervals', 'data': 'synthetic',
            'config': {
                'workload': workload_name(n, bits, args.batch) if args.total <= 0 else f'{n}x{n} int{bits} default solve(), fixed job of {args.total} matrices over {world} rank(s)',
                'timing': 'every step solves new matrices and the per-step working set (histogram segments, cell pools, op tables of the concurrent candidates) exceeds the 126 MB L2',
                'adders_rank0': adders,
                'jobs': {'reference_solve_single_calls': jobs_total, 'executed': jobs_run,
                         'note': 'byte-identical solve_single jobs of one call (decompose_dc candidates with the same stage matrix) are solved once'},
            },
            'parity_checked': bool(checked) and not mismatches,
            'parity': {'checked': checked, 'against': 'tests/golden/index.json: sha256 over all result arrays + adder count, produced by oracle/_ref (the reference translation units)'},
            'solve_ms_per_matrix': dev_ms_max / args.steps / args.batch,
            'gpu_launches': launches,
            'clocks': clocks.summary(),
            'e2e': {'value': total / (e2e_ms_max * 1e-3), 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h, 'ms_per_step': e2e_ms_max / args.steps,
                    'what': 'da4ml_b200.cmvm.solve(host float32 ndarray) -> Pipeline of CombLogic / Op objects (the reference call and result type)'},
            'e2e_raw': {'value': total / (e2e_raw_ms_max * 1e-3), 'unit': UNIT, 'ms_per_step': e2e_raw_ms_max / args.steps, 'what': 'the same down to the flat result arrays of the C ABI (no Python containers)'},
            'roofline': {
                'bound': 'hbm', 'kernel': 'cmvm_solve_kernel', 'achieved': achieved, 'peak': peak_gbs, 'unit': 'GB/s',
                'frac': (achieved / peak_gbs) if achieved else None, 'traffic': traffic, 'traffic_source': 'static: one ncu --set full capture (profiles/traffic.json), not measured in this run',
                'peak_source': peak_src, 'algo_bytes_per_step': a_step, 'algo_bytes_per_step_reference': (a_ref or 0.0) * args.batch,
                'launches_per_step': solve_launches / max(1, args.steps), 'kernel_ms_per_step': solve_ms / max(1, args.steps),
                # SURVEY 8d defines A over every solve_single the REFERENCE executes for the call; `frac` above is the stricter figure
                # (only the jobs actually executed after sharing identical candidates)
                'frac_reference_job_list': ((a_ref * args.batch / 1e9) / (solve_ms / max(1, args.steps) * 1e-3) / peak_gbs) if (a_ref and solve_ms) else None,
                'note': 'achieved = algorithmic bytes (SURVEY 8d: full-histogram scans + pair recounts) of the solve_single jobs EXECUTED (seed-0 matrix, exact counters) / CUDA-event time of the '
                        'solve-kernel launches; algo_bytes_per_step_reference counts every job the reference executes (no sharing).  The kernel touches far fewer bytes than either '
                        '(chunk-cached argmax), the path is a chain of dependent greedy steps',
            },
        }
        if c4 is not None:
            line['c4'] = c4
        if mismatches:
            line['parity_mismatch_seeds'] = mismatches
        full = full_cpu_run(n, bits, 0)
        if cpu is not None:
            line['cpu_baseline'] = {'value': cpu.get('value'), 'unit': UNIT, 'cores': cpu['cores'], 'kind': cpu['kind'], 'sample': cpu['sample'], 'algo_bytes_per_s': cpu['algo_bytes_per_s'], 'full_run_cached': full}
    if args.dump_outputs:
        dump_outputs(Path(args.dump_outputs), results[-1], f'rank{rank}_' if world > 1 else '', DUMP_LIMIT // world)
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=3)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='cuda', choices=['cuda', 'reference'])
    ap.add_argument('--size', type=int, default=256)
    ap.add_argument('--bits', type=int, default=8)
    ap.add_argument('--batch', type=int, default=1, help='matrices per rank per step')
    ap.add_argument('--total', type=int, default=0, help='fixed total number of matrices split over the ranks (strong scaling); 0 = weak scaling with --batch per rank')
    ap.add_argument('--seed', type=int, default=0)
    ap.add_argument('--c4', type=int, default=64, help='matrices of the BASELINE config 4 sub-record (128x128 int6, fixed job over the ranks); 0 disables')
    ap.add_argument('--cpu-seconds', type=float, default=15.0, help='bounded CPU-baseline sample (0 disables)')
    ap.add_argument('--recount', action='store_true', help='recompute the cached algorithmic-byte figures')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the result arrays of the last timed step to DIR/<name>.npy (CUDA arm)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.impl == 'reference':
        return run_reference(args)
    return run_cuda(args)


if __name__ == '__main__':
    sys.exit(main())
