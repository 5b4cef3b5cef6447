"""The solver's capacity paths on the GPU: owner lists that spill to global memory, pair-counting passes that run out of
counters and are split, histogram-segment compaction, every overflow status and the host's relaunch of the failed jobs,
and batches with more jobs than concurrent groups.  The planner sizes buffers generously, so ordinary solves take none of
these paths; ``set_first_attempt_caps`` forces small capacities on the first attempt of each round of jobs.  Every test
checks its results against the CPU checker or the stored reference digests, and asserts the counter that shows its path
ran.  The forced values are ones the kernel sources are shown to survive under the CPU simulation (here and in
tests/test_kernel_sim.py): they end in a result or in a capacity status.

The first tests need no GPU: they check the switch's argument handling, the plan it produces, and the forced values
under the simulation."""
import numpy as np
import pytest
from conftest import assert_stage_equal, golden_cases, int_matrix, load_golden
from test_cmvm_gpu import digest

import oracle
from oracle import port

from da4ml_b200 import _binary as Bin

ALL = golden_cases(full_only=False)
SINGLE_CASES = sorted(k for k, v in ALL.items() if v['full'] and v.get('single'))
C4 = sorted((ALL[k]['spec'][4], k) for k in ALL if k.startswith('c4_128x128_int6_default'))

# the 16x16 int6 matrix (seed 11) on two CTAs, with the capacities tests/test_kernel_sim.py runs it under
SIM_W = (16, 16, 6, 11)
SIM_G = 2


@pytest.fixture
def B(cuda_binary):
    """The library with every development switch restored afterwards."""
    try:
        yield cuda_binary
    finally:
        cuda_binary.set_first_attempt_caps()
        cuda_binary.set_group_size(0)
        cuda_binary.set_accounting(False)
        cuda_binary.set_job_sharing(True)


@pytest.fixture
def B_host():
    try:
        yield Bin
    finally:
        Bin.set_first_attempt_caps()


def job(n_in, n_out, nbits, density=0.36):
    return dict(n_in=n_in, n_out=n_out, nbits=nbits, digits=int(n_in * n_out * nbits * density))


def single(B, W, method='wmc', trace=True, **kw):
    raw, tr = B.solve_single_raw(W, method, trace_cap=1 << 14 if trace else 0, **kw)
    return raw, tr


# ---- no GPU: the switch and the plan ---------------------------------------------------------------------------------


def test_setter_rejects_bad_capacities_and_keeps_the_old_ones(B_host):
    j = [job(48, 40, 8)]
    free = B_host.plan(j, group_override=1)
    B_host.set_first_attempt_caps(list_rows_smem=6)
    forced = B_host.plan(j, group_override=1)
    for bad in (dict(spill_rows=-1), dict(log2_pair_counters=9), dict(log2_pair_counters=17), dict(cells_per_cta=-5), dict(extra_expressions=2**31)):
        with pytest.raises(ValueError):
            B_host.set_first_attempt_caps(**bad)
        assert B_host.plan(j, group_override=1) == forced, bad
    with pytest.raises(TypeError):
        B_host.set_first_attempt_caps(list_rows=4)
    B_host.set_first_attempt_caps()
    assert B_host.plan(j, group_override=1) == free


def test_caps_shrink_the_first_plan_only_where_smaller(B_host):
    j = [job(48, 40, 8)]
    free = B_host.plan(j, group_override=1)
    assert free['log2_pair_counters'] == 13 and free['list_rows_smem'] > 7
    B_host.set_first_attempt_caps(list_rows_smem=7, log2_pair_counters=10, segment_entries_per_cta=5000)
    p = B_host.plan(j, group_override=1)
    assert p['list_rows_smem'] == 6  # (even: the 32-bit plane arrays of 6-byte rows stay aligned)
    assert p['list_rows_smem'] + p['spill_rows'] == free['list_rows_smem'] + free['spill_rows']  # the rows moved to global memory
    assert p['log2_pair_counters'] == 10 and p['segment_entries_per_cta'] == 5000
    assert (p['segment_entries_per_cta'] >> p['log2_chunk']) + 2 == p['chunk_slots']
    assert p['shared_bytes'] < free['shared_bytes'] and p['ctas_per_problem'] == 1
    B_host.set_first_attempt_caps(spill_rows=3, list_rows_smem=4)
    p = B_host.plan(j, group_override=1)
    assert (p['list_rows_smem'], p['spill_rows']) == (4, 3)
    # caps above the planner's values change nothing, and neither does the group size the planner picks
    B_host.set_first_attempt_caps(list_rows_smem=10**6, log2_pair_counters=16, segment_entries_per_cta=2**30, spill_rows=10**6, cells_per_cta=2**30)
    assert B_host.plan(j, group_override=1) == free
    jobs = [job(128, 128, 6)] * 384
    want = B_host.plan(jobs)
    B_host.set_first_attempt_caps(list_rows_smem=2, log2_pair_counters=10)
    got = B_host.plan(jobs)
    assert (got['ctas_per_problem'], got['concurrent_groups']) == (want['ctas_per_problem'], want['concurrent_groups'])
    assert got['list_rows_smem'] == 2 and got['log2_pair_counters'] == 10


FORCED = {
    'segment': dict(segment_entries_per_cta=700),  # ST_FSEG_OVERFLOW
    'lists': dict(list_rows_smem=4, spill_rows=1),  # ST_LIST_OVERFLOW: owner lists
    'cells': dict(cells_per_cta=150),  # ST_LIST_OVERFLOW: cell pool
    'expressions': dict(extra_expressions=19),  # ST_EXPR_OVERFLOW
}
FORCED_STATUS = {'segment': 2, 'lists': 5, 'cells': 5, 'expressions': 1}


def test_forced_capacities_under_the_cpu_simulation():
    """The capacities the GPU tests below force, applied by the product's planner to the kernel sources under the CPU
    SIMT shim (one attempt, no retry): the overflows end in their status, the others in the reference graph with the
    path taken."""
    import simt

    W = int_matrix(*SIM_W)
    want = port.solve_single(W, 'wmc')
    try:
        for what, caps in FORCED.items():
            simt.set_first_attempt_caps(**caps)
            with pytest.raises(RuntimeError, match=f'capacity status {FORCED_STATUS[what]}'):
                simt.solve_single(W, 'wmc', ctas=SIM_G, cta_threads=128)
        for caps, check in (
            (dict(segment_entries_per_cta=2000), lambda m: m[9] > 0),  # compactions
            (dict(list_rows_smem=2), lambda m: m[15] == 2 and m[14] > 2),  # spilled owner lists
            (dict(log2_pair_counters=10), lambda m: m[0] == 0),  # (the split count is not in the 32 words the shim returns)
        ):
            simt.set_first_attempt_caps(**caps)
            got, meta = simt.solve_single(W, 'wmc', ctas=SIM_G, cta_threads=128)
            assert_stage_equal(got, want, f'{caps} ')
            assert check(meta), (caps, list(meta[:16]))
    finally:
        simt.set_first_attempt_caps()


# ---- GPU ---------------------------------------------------------------------------------------------------------------


@pytest.mark.gpu
def test_config4_as_one_batch(B):
    """64 x 128x128 int6 (BASELINE config 4) in one call: hundreds of stage-0 jobs on a few dozen groups, each group's
    workspace reused by one job after another.  Host arrays in, and again device arrays in."""
    torch = pytest.importorskip('torch')
    assert [s for s, _ in C4] == list(range(64))
    mats = [int_matrix(128, 128, 6, s) for s, _ in C4]
    dev = [torch.from_numpy(m).cuda() for m in mats]
    torch.cuda.synchronize()
    sm = B.device_info()['sm_count']
    for how, res in (('host', B.solve_batch_raw(mats)), ('device', B.solve_batch_device_raw([t.data_ptr() for t in dev], [m.shape for m in mats]))):
        for (s, name), r in zip(C4, res, strict=True):
            meta = ALL[name]
            assert r.n_adders == meta['n_adders'], f'{how} {name}'
            assert [len(st['ops_i']) for st in r.stages] == meta['stage_ops'], f'{how} {name}'
            assert digest(r.stages) == meta['sha256'], f'{how} {name}'
        # the first round's stage-0 launch has at least one job per matrix; more jobs than groups means several waves
        G = res[0].counters[0]['group_ctas']
        assert len(mats) > sm // G, (how, G)
        assert res[0].profile['jobs_run'] > sm // G and res[0].profile['retried_jobs'] == 0


def small_family(n=200, seed=0):
    rng = np.random.default_rng(seed)
    mats, qs, ls = [], [], []
    for i in range(n):
        n_in, n_out, bits = int(rng.integers(1, 41)), int(rng.integers(1, 41)), int(rng.integers(2, 13))
        W = int_matrix(n_in, n_out, bits, 9000 + i)
        if i % 5 == 1:
            W = W * np.float32(0.125)  # fractional weights
        if i % 7 == 2:
            W[:, int(rng.integers(0, n_out))] = 0  # an all-zero column
        q = np.stack([-(2.0 ** rng.integers(0, 9, n_in)), 2.0 ** rng.integers(0, 9, n_in) - 0.25, np.full(n_in, 0.25)], axis=1)
        mats.append(np.ascontiguousarray(W, dtype=np.float32))
        qs.append([tuple(map(float, r)) for r in q.astype(np.float32)])
        ls.append([float(v) for v in rng.integers(0, 4, n_in)])
    return mats, qs, ls


@pytest.mark.gpu
def test_multi_wave_batch_at_group_size_one(B):
    """About 200 small problems of mixed shapes, widths and intervals at one CTA per job: more jobs than the GPU has
    groups, so every group's workspace is reused by problems of other sizes.  Reversed, every workspace sees a different
    predecessor."""
    mod, _ = oracle.best()
    mats, qs, ls = small_family()
    want = [mod.solve(W, qintervals=q, latencies=l) for W, q, l in zip(mats, qs, ls)]
    sm = B.device_info()['sm_count']
    B.set_group_size(1)
    for order in (range(len(mats)), range(len(mats) - 1, -1, -1)):
        order = list(order)
        res = B.solve_batch_raw([mats[i] for i in order], qintervals=[qs[i] for i in order], latencies=[ls[i] for i in order])
        for i, r in zip(order, res, strict=True):
            assert all(c['group_ctas'] == 1 for c in r.counters)
            for k, (a, b) in enumerate(zip(r.stages, want[i], strict=True)):
                assert_stage_equal(a, b, f'problem {i} {mats[i].shape} stage{k} ')
        assert len(mats) > sm and res[0].profile['retried_jobs'] == 0  # one stage-0 job per problem at least: several waves


SPILL_CASES = {
    '48x40_int8': lambda: int_matrix(48, 40, 8, 9),
    '24x130_int6': lambda: int_matrix(24, 130, 6, 4),  # five bitmap words per row
    '24x20_20bit': lambda: int_matrix(24, 20, 20, 4),  # more than 16 CSD bits: 12-byte list rows
}


@pytest.mark.gpu
@pytest.mark.parametrize('name', sorted(SPILL_CASES))
def test_spilled_owner_lists(B, name):
    """Two rows per owner list in shared memory, the rest in the spill rows in global memory (same total capacity, so
    nothing is retried), at 1, 2 and 7 CTAs per problem."""
    mod, _ = oracle.best()
    W = SPILL_CASES[name]()
    want = mod.solve_single(W, 'wmc')
    B.set_first_attempt_caps(list_rows_smem=2)
    for G in (1, 2, 7):
        B.set_group_size(G)
        raw, _ = single(B, W, trace=False)
        c = raw.counters[0]
        assert_stage_equal(raw.stages[0], want, f'{name} G={G} ')
        assert c['group_ctas'] == G and c['smem_list_cap'] == 2 and c['list_max'] > 2, (G, c['list_max'])
        assert raw.profile['retried_jobs'] == 0
        if name.endswith('20bit'):
            assert c['n_bits'] > 16  # (the planner's narrow rows need at most 16)


@pytest.mark.gpu
def test_split_counting_passes(B):
    """The smallest pair-counter table the kernel supports (2^10 counters): passes that run out of counters are abandoned
    and split.  Graphs and step traces equal the stored single-stage answers and the unforced run."""
    mod, _ = oracle.best()
    splits = 0
    B.set_group_size(1)
    cases = [(name, *load_golden(name)) for name in SINGLE_CASES]
    for name, extra, stages in cases:
        kw = ALL[name]['kwargs']
        B.set_first_attempt_caps(log2_pair_counters=10)
        raw, tr = B.solve_single_raw(extra['kernel'], kw['method'], extra['qint'], extra['lat'], kw['adder_size'], kw['carry_size'], trace_cap=4096)
        assert_stage_equal(raw.stages[0], stages[0], name + ' ')
        assert np.array_equal(tr[:, :4], extra['pairs']) and np.array_equal(tr[:, 4], extra['f_sizes']), name
        assert raw.profile['retried_jobs'] == 0
        splits += raw.counters[0]['split_passes']
    W = int_matrix(48, 40, 8, 9)
    B.set_first_attempt_caps()
    free, free_tr = single(B, W)
    B.set_first_attempt_caps(log2_pair_counters=10)
    raw, tr = single(B, W)
    assert_stage_equal(raw.stages[0], mod.solve_single(W, 'wmc'), '48x40 ')
    assert np.array_equal(tr, free_tr) and raw.profile['retried_jobs'] == 0
    assert raw.counters[0]['split_passes'] > 0
    splits += raw.counters[0]['split_passes']
    assert splits > 0


@pytest.mark.gpu
def test_segment_compaction(B):
    """A histogram segment small enough to be compacted during the run (and, at 2000 entries, too small for the hot
    regions), never so small that it overflows: same graph, and in accounting mode the exact work counters of the
    reference algorithm."""
    W = int_matrix(*SIM_W)
    want = port.solve_single(W, 'wmc')
    B.set_group_size(SIM_G)
    free, free_tr = single(B, W)
    assert free.counters[0]['compactions'] == 0
    B.set_first_attempt_caps(segment_entries_per_cta=2000)
    raw, tr = single(B, W)
    assert raw.counters[0]['compactions'] > 0 and raw.profile['retried_jobs'] == 0
    assert_stage_equal(raw.stages[0], want, 'compacted ')
    assert np.array_equal(tr, free_tr)
    B.set_accounting(True)
    raw, _ = single(B, W, trace=False)
    c, r = raw.counters[0], want['counters']
    assert c['compactions'] > 0 and raw.profile['retried_jobs'] == 0
    assert_stage_equal(raw.stages[0], want, 'compacted, accounting ')
    for k in ('T', 'sum_F', 'sum_R', 'F0', 'R0'):
        assert c[k] == r[k], k


@pytest.mark.gpu
@pytest.mark.parametrize('what', sorted(FORCED))
def test_every_overflow_status_is_retried(B, what):
    """A capacity forced below what the job needs: the kernel reports the status, the host relaunches the job with the
    planner's escalated sizes, and the graph and step trace are those of the unforced run and of the checker."""
    W = int_matrix(*SIM_W)
    want = port.solve_single(W, 'wmc')
    B.set_group_size(SIM_G)
    free, free_tr = single(B, W)
    assert free.profile['retried_jobs'] == 0
    B.set_first_attempt_caps(**FORCED[what])
    raw, tr = single(B, W)
    assert raw.profile['retried_jobs'] >= 1
    assert_stage_equal(raw.stages[0], want, f'{what} ')
    assert_stage_equal(raw.stages[0], free.stages[0], f'{what} vs unforced ')
    assert np.array_equal(tr, free_tr)


@pytest.mark.gpu
def test_retry_relaunches_only_the_failed_jobs(B):
    """A cap on the expressions a job may create that only the larger problems of a batch exceed (a 3x3 int3 matrix has
    at most 18 digits, so at most 18 steps): some jobs are relaunched, not all, and every problem gets its own answer."""
    mod, _ = oracle.best()
    mats = [int_matrix(3, 3, 3, 70 + i) if i % 2 else int_matrix(24, 20, 8, 70 + i) for i in range(12)]
    want = [mod.solve(W) for W in mats]
    B.set_first_attempt_caps(extra_expressions=30)
    res = B.solve_batch_raw(mats)
    prof = res[0].profile
    assert 0 < prof['retried_jobs'] < prof['jobs_run'], prof
    for i, (r, w) in enumerate(zip(res, want, strict=True)):
        for k, (a, b) in enumerate(zip(r.stages, w, strict=True)):
            assert_stage_equal(a, b, f'problem {i} {mats[i].shape} stage{k} ')


@pytest.mark.gpu
@pytest.mark.parametrize('name', ['c2_64x64_int8_default', '128x128_int8_dc-1'])
def test_full_solves_under_forced_capacities(B, name):
    """Whole solves through the candidate rounds with every stage job's first attempt under forced spills and under a
    segment that overflows, with identical jobs shared and not shared: the stored digests."""
    meta = ALL[name]
    W = int_matrix(*meta['spec'][1:])
    for caps in (dict(list_rows_smem=2), dict(segment_entries_per_cta=700)):
        for share in (True, False):
            B.set_job_sharing(share)
            B.set_first_attempt_caps(**caps)
            raw = B.solve_raw(W, **meta['kwargs'])
            tag = f'{name} {caps} share={share}'
            assert raw.n_adders == meta['n_adders'], tag
            assert [len(st['ops_i']) for st in raw.stages] == meta['stage_ops'], tag
            assert digest(raw.stages) == meta['sha256'], tag
            if 'list_rows_smem' in caps:
                assert raw.profile['retried_jobs'] == 0, tag
                assert all(c['smem_list_cap'] == 2 for c in raw.counters), tag
                assert raw.counters[0]['list_max'] > 2, tag
            else:
                assert raw.profile['retried_jobs'] >= 1, tag
