// cmvm_kernel_own.cuh -- the persistent solve kernel (owner-partitioned formulation, solve_owned.cuh): per greedy step ONE
// group exchange (the argmax), no cross-CTA counters and no L2 atomics.  The per-CTA context lives in shared memory
// (nothing of it is passed around by value).
#pragma once
#include "cmvm_kernels.cuh"
#include "solve_owned.cuh"
#ifdef DA_RECOUNT_PROF
#include <cstdio>
#endif

namespace da {

// shared-memory plan of one CTA of the owner-partitioned kernel (host and device agree through this function)
struct OwnPlan {
    OwnLayout lay;
    size_t bytes;
};
__host__ __device__ inline OwnPlan own_plan(int nchunk_cap, int n_out_max, int e_cap_max, int lcap, int hlog, int narrow) {
    OwnPlan P;
    size_t o = ((size_t)nchunk_cap * 17 + 15) & ~size_t(15); // chunk caches: 3 x u32 + dirty list (int) + dirty flag (u8)
    auto take = [&](size_t bytes) {
        const size_t at = o;
        o += (bytes + 15) & ~size_t(15);
        return (uint32_t)at;
    };
    const int words = (n_out_max + 31) / 32;
    for (int r = 0; r < 3; ++r)
        P.lay.D[r] = take(sizeof(uint2) * (size_t)n_out_max);
    for (int r = 0; r < 3; ++r)
        P.lay.B[r] = take(sizeof(uint32_t) * (size_t)words);
    P.lay.A = take(sizeof(uint32_t) * (size_t)words);
    P.lay.pre = take(sizeof(uint32_t) * (size_t)words);
    P.lay.ver = take(sizeof(uint32_t) * (size_t)((e_cap_max + 31) / 32));
    P.lay.col_len = take(sizeof(int) * (size_t)n_out_max);
    P.lay.tcol = take(sizeof(uint16_t) * (size_t)n_out_max);
    P.lay.tpre = take(sizeof(int) * ((size_t)n_out_max + 1));
    P.lay.hkey = take(sizeof(uint32_t) << hlog);
    P.lay.hval = take(sizeof(uint32_t) << hlog);
    P.lay.hins = take(sizeof(uint16_t) << hlog);
    P.lay.lists = take((narrow ? 6 : 12) * (size_t)n_out_max * (size_t)lcap); // (lcap is even: the 32-bit plane arrays stay aligned)
    P.lay.narrow = narrow;
    P.lay.lcap = lcap;
    P.lay.hlog = hlog;
    P.lay.words = words;
    P.bytes = o;
    return P;
}

__device__ void solve_problem_own(const ProblemDesc &p, const Ctx &cx, const OwnCtx &ox) {
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
    const int n_in = p.n_in, n_out = p.n_out, nbits = p.nbits, G = cx.cfg.G;
    const uint32_t thresh = method_threshold(p.method);
    BlockCtx &b = *cx.b;
    OwnBlock &ob = *ox.ob;

    if (tid == 0) {
        b.seg_len = 0;
        {
            // hot regions for the first expressions this CTA owns: its inputs and the earliest new expressions, the dense
            // rows that are rewritten again and again (not worth it when a region would be only a few chunks long)
            const int n_own = (p.e_cap - cx.rank + G - 1) / G, H = min(n_own, DA_HOT_MAX), ch = 1 << cx.cfg.chunk_log;
            b.cap0 = cx.ws.fseg_cap;
            b.hot_n = 0;
            b.hot_cap = 0;
            if (H > 0) {
                const int half = (cx.ws.fseg_cap / 4) & ~(ch - 1), hc = ((cx.ws.fseg_cap - half) / H) & ~(ch - 1); // a quarter for the common log
                if (hc >= 4 * ch)
                    b.cap0 = half, b.hot_n = H, b.hot_cap = hc;
            }
            for (int k = 0; k < DA_HOT_MAX; ++k)
                b.hot_len[k] = b.hot_snap[k] = 0;
        }
        b.n_new = 0;
        b.live_old = 0;
        b.n_dirty = 0;
        b.status = ST_OK;
        b.list_max = 0;
        b.r_count = 0ull;
        b.rescanned = 0ull;
        b.r_step = 0;
        b.rescan_step = 0;
        b.chosen = Best{0u, 0u, 0u};
        for (int k = 0; k < 8; ++k) {
            b.phase[k] = 0;
            b.peak[k] = 0;
            b.nslow[k] = 0;
        }
        b.poll_iters = 0;
        ob.pool_used = 0;
        ob.pass_bits = 0;
        ob.splits = 0;
        ob.n_ins = 0;
        ob.overflow = 0;
#ifdef DA_RECOUNT_PROF
        for (int k = 0; k < 4; ++k)
            ob.xphase[k] = 0;
#endif
    }
    for (int c = tid; c < cx.cfg.nchunk_cap; c += nt) {
        cx.cb_score[c] = 0u;
        cx.cb_khi[c] = 0u;
        cx.cb_klo[c] = 0u;
        cx.cb_dirty[c] = 0;
    }
    {
        DA_DYN_SHARED(da_smem);
        uint32_t *hkey = DA_SM(uint32_t, ox.lay.hkey), *hval = DA_SM(uint32_t, ox.lay.hval);
        for (int k = tid; k < (1 << ox.lay.hlog); k += nt) {
            hkey[k] = 0u;
            hval[k] = 0u;
        }
    }
    for (int i = cx.rank * nt + tid; i < p.e_cap; i += G * nt)
        cx.ws.mod_step[i] = 0u;
    group_sync(cx); // every CTA's share of the stamps is zero before anybody judges an entry by them
    own_init(p, cx, ox);
    // ---- input ops (state_opr.cc:146-149)
    for (int i = cx.rank * nt + tid; i < n_in; i += G * nt) {
        p.op_misc[i] = make_int4(i, -1, -1, 0);
        p.op_q[i] = make_float4(p.qint[3 * i], p.qint[3 * i + 1], p.qint[3 * i + 2], p.lat[i]);
        p.op_cost[i] = 0.0f;
    }

    Best best{0u, 0u, 0u};
    unsigned long long r0 = 0;
    if (p.method != M_DUMMY)
        r0 = initial_histogram(p, cx, thresh, best);
    if (r0)
        atomicAdd(&b.r_count, r0);
    __syncthreads();
    const unsigned long long r0_cta = b.r_count;
    if (tid == 0) {
        b.seg_len = min(b.seg_len, b.cap0);
        b.n_new = 0;
    }
    __syncthreads();
    int seg_cur = b.seg_len; // entries of this CTA's segment (every thread keeps a copy: team R must not read the live counter)
    refresh_chunks(cx, team_all(), seg_cur, 0u, 0u, false, true, thresh);
    publish_best(cx, Best{0u, 0u, 0u}); // the exchange also orders the cells / input ops written above
    if (tid == 0) { // (thread 0 has published; nobody touches these before the barrier inside the collect)
        b.live_old = 0;
        b.n_new = 0;
    }
    int f_live = collect_best(cx);
    const int f0 = f_live;
    int f_max = f_live;

    // ---- greedy loop (cmvm_core.cc:36-70)
    // Two teams of warps work side by side in a step: the first warps substitute, update and recount (team C, barrier 1),
    // the last quarter brings the argmax caches up to date for the rewritten expressions (team R, barrier 2) -- which
    // chunks a substitution invalidates varies wildly from CTA to CTA and step to step, and the group waits for its slowest
    // CTA.  (A CTA of a single warp does both one after the other.)
    const int rw = nw >= 4 ? nw / 4 : (nw >= 2 ? 1 : 0);
    const bool split = rw > 0;
    const int nt_c = nt - 32 * rw;
    const bool in_c = tid < nt_c;
    const Team tm_c = split ? Team{tid, nt_c, 1} : team_all(), tm_r = Team{tid - nt_c, 32 * rw, 2};
    int t = 0;
    unsigned long long sum_f = 0;
    int status = b.scratch_i[1];
    const long long t_start = clock64();
    while (status == ST_OK) {
        const Best ch = b.chosen;
        if (ch.score == 0u || p.method == M_DUMMY)
            break;
        if (n_in + t >= p.e_cap) {
            status = ST_EXPR_OVERFLOW;
            break;
        }
        const uint64_t key = ((uint64_t)ch.khi << 32) | ch.klo;
        const uint32_t c0 = key_id0(key), c1 = key_id1(key);
        const int shift = key_shift(key), sub = key_sub(key);
        const uint32_t newid = (uint32_t)(n_in + t);
        const uint32_t stamp = (uint32_t)(t + 1);
        sum_f += (unsigned long long)f_live;
        f_max = max(f_max, f_live);
        if (tid == nt_c - 1) {
            // pair_to_op (state_opr.cc:211-225): every CTA needs the new record for the entries it emits in this step;
            // CTA 0 also publishes it (with the rewrite stamps) for the later steps
            QInt q0, q1;
            float l0, l1;
            load_op(p, c0, q0, l0);
            load_op(p, c1, q1, l1);
            float dlat, cost;
            cost_add(q0, q1, shift, sub != 0, p.adder_size, p.carry_size, dlat, cost);
            const QInt q = qint_add(q0, q1, shift, false, sub != 0);
            const float lat = fadd(fmaxf_std(l0, l1), dlat);
            int r = 0;
            ob.mid[r] = c0, ob.mq[r] = q0, ob.ml[r] = l0, ++r;
            if (c1 != c0)
                ob.mid[r] = c1, ob.mq[r] = q1, ob.ml[r] = l1, ++r;
            ob.mid[r] = newid, ob.mq[r] = q, ob.ml[r] = lat, ++r;
            ob.n_mods = r;
            if (cx.rank == 0) {
                p.op_misc[newid] = make_int4((int)c0, (int)c1, sub, shift);
                p.op_q[newid] = make_float4(q.min, q.max, q.step, lat);
                p.op_cost[newid] = cost;
                st_racy(&cx.ws.mod_step[c0], stamp);
                st_racy(&cx.ws.mod_step[c1], stamp);
                st_racy(&cx.ws.mod_step[newid], stamp);
                if (p.trace && t < p.trace_cap) {
                    int *tr = p.trace + 5 * (size_t)t;
                    tr[0] = (int)c0;
                    tr[1] = (int)c1;
                    tr[2] = shift;
                    tr[3] = sub;
                    tr[4] = f_live;
                }
            }
        }
        if (tid == 0)
            b.t_last = clock64();
        const bool compacting = b.scratch_i[3] != 0; // agreed by the whole group in the last exchange
        if (compacting) {
            compact_segment(cx, c0, c1, true, thresh, cx.rank == 0 ? &p.result_meta[META_COMPACTIONS] : nullptr);
            seg_cur = b.seg_len;
            __syncthreads(); // (every thread has its copy before team C appends)
        }
        const int seg0 = seg_cur; // what the argmax caches have to cover; this step's entries are appended behind it
        {
            // a hot input of this CTA is rewritten: every entry of its region dies with it (uniform over the CTA)
            const bool k0 = (int)(c0 % (uint32_t)G) == cx.rank && (int)(c0 / (uint32_t)G) < b.hot_n;
            const bool k1 = c1 != c0 && (int)(c1 % (uint32_t)G) == cx.rank && (int)(c1 / (uint32_t)G) < b.hot_n;
            if (k0 || k1) {
                for (int w = 0; w < 2; ++w) {
                    if (!(w == 0 ? k0 : k1))
                        continue;
                    const int k = (int)((w == 0 ? c0 : c1) / (uint32_t)G), cpr = b.hot_cap >> cx.cfg.chunk_log, cb = (b.cap0 >> cx.cfg.chunk_log) + k * cpr;
                    for (int c = tid; c < cpr; c += nt) {
                        cx.cb_score[cb + c] = 0u;
                        cx.cb_khi[cb + c] = 0u;
                        cx.cb_klo[cb + c] = 0u;
                        cx.cb_dirty[cb + c] = 0;
                    }
                    if (tid == 0)
                        b.hot_len[k] = b.hot_snap[k] = 0;
                }
                __syncthreads();
            }
        }
        best = Best{0u, 0u, 0u};
        if (in_c) {
            // A. substitution in every column (redundantly on every CTA), B. the owners update their cells and lists,
            // C. the recount appends this step's entries
            own_substitute(p, cx, ox, tm_c, c0, c1, shift, sub);
            DA_LAP(0)
            own_update(p, cx, ox, tm_c, c0, c1, newid);
            DA_LAP(3)
            if (!split && !compacting)
                refresh_chunks(cx, tm_c, seg0, c0, c1, true, cx.cfg.accounting != 0, thresh);
            own_recount(p, cx, ox, tm_c, newid, stamp, thresh, best);
            // maxima of the entries each log received in this step (their chunks' caches are updated behind the join)
            for (int r = wid; r <= b.hot_n; r += nt_c >> 5) {
                const int base = r == 0 ? 0 : b.cap0 + (r - 1) * b.hot_cap, l0 = r == 0 ? seg0 : b.hot_snap[r - 1];
                const int l1 = r == 0 ? min(b.seg_len, b.cap0) : min(b.hot_len[r - 1], b.hot_cap);
                if (l1 > l0) // (uniform over the warp; most logs receive nothing in a step)
                    merge_appended_scan(cx, r, base, l0, l1, thresh);
            }
            DA_LAP(1)
        }
        else if (!compacting) {
            // the argmax caches: entries touching c0 / c1 die
            const long long r0c = clock64();
            refresh_chunks(cx, tm_r, seg0, c0, c1, true, cx.cfg.accounting != 0, thresh);
            if (tid == nt_c)
                b.phase[2] += clock64() - r0c;
        }
        __syncthreads();
        DA_LAP(4)
        {
            // this step's entries -> the cached maxima of the chunks that received them
            const int seg1 = min(b.seg_len, b.cap0);
            seg_cur = seg1; // (nothing is appended before the next step's team C starts, two exchanges' barriers away)
            for (int r = tid; r <= b.hot_n; r += nt) {
                if (r == 0)
                    merge_appended_apply(cx, 0, 0, seg0, seg1);
                else {
                    const int k = r - 1, l1 = min(b.hot_len[k], b.hot_cap);
                    merge_appended_apply(cx, r, b.cap0 + k * b.hot_cap, b.hot_snap[k], l1);
                    b.hot_len[k] = l1; // the region's fill becomes the next step's snapshot
                    b.hot_snap[k] = l1;
                }
            }
            __syncthreads();
        }
        publish_best(cx, best);
        if (tid == 0) { // (thread 0 has published; nobody touches these before the barrier inside the collect)
            b.live_old = 0;
            b.n_new = 0;
            b.r_count += (unsigned long long)b.r_step;
            b.r_step = 0;
            b.rescanned += (unsigned long long)b.rescan_step;
            b.rescan_step = 0;
        }
        DA_LAP(5)
        f_live = collect_best(cx);
        DA_LAP(7)
        ++t;
        if (cx.rank == 0 && tid == 0 && t >= 250 && t % 250 == 0 && ((t / 250) & (t / 250 - 1)) == 0 && t / 250 <= 64) {
            long long *ms = &p.result_meta[META_MILESTONES + 9 * (31 - __clz(t / 250))]; // (diagnostic: where the time of a stage goes)
            for (int k = 0; k < 8; ++k)
                ms[k] = b.phase[k];
            ms[8] = clock64() - t_start;
#ifdef DA_RECOUNT_PROF
            printf("  recount parts after %d steps (cumulative ms at 1.9 GHz): setup %.2f counting %.2f harvest %.2f\n", t, ob.xphase[0] / 1.9e6, ob.xphase[1] / 1.9e6, ob.xphase[2] / 1.9e6);
#endif
        }
        if (b.scratch_i[1] != ST_OK) {
            status = b.scratch_i[1];
            break;
        }
    }

    // ---- to_solution: column lists from the owner lists, then one warp per column
    own_scatter_columns(p, cx, ox);
    finish_columns(p, cx, t);
    // ---- bookkeeping
    __syncthreads();
    if (tid == 0) {
        b.r_count += (unsigned long long)b.r_step;
        b.rescanned += (unsigned long long)b.rescan_step;
        atomicAdd((unsigned long long *)&p.result_meta[META_SUM_R], b.r_count - r0_cta);
        atomicAdd((unsigned long long *)&p.result_meta[META_R0], r0_cta);
        atomicAdd((unsigned long long *)&p.result_meta[META_RESCANNED], b.rescanned);
        atomicMax((long long *)&p.result_meta[META_LIST_MAX], (long long)b.list_max);
        if (ob.splits)
            atomicAdd((unsigned long long *)&p.result_meta[META_SPLITS], (unsigned long long)ob.splits);
        for (int k = 0; k < 8; ++k)
            atomicMax((long long *)&p.result_meta[META_PHASEMAX + k], b.phase[k]); // the slowest CTA's total per phase
        if (b.status != ST_OK)
            atomicMax((int *)&p.result_meta[META_STATUS], b.status);
    }
    if (cx.rank == 0 && tid == 0) {
        long long tree = 0, dfin = 0;
        for (int o = 0; o < n_out; ++o) {
            const int k = __ldcg(&cx.ws.col_k[o]);
            tree += k > 1 ? k - 1 : 0;
            dfin += k;
        }
        const long long n_ops = (long long)n_in + t + tree;
        p.result_meta[META_N_OPS] = n_ops;
        p.result_meta[META_T] = t;
        p.result_meta[META_SUM_F] = (long long)sum_f;
        p.result_meta[META_F0] = f0;
        p.result_meta[META_D_FINAL] = dfin;
        p.result_meta[META_F_MAX] = f_max;
        for (int k = 0; k < 8; ++k)
            p.result_meta[META_PHASE0 + k] = b.phase[k];
        p.result_meta[15] = b.poll_iters;
        if (status != ST_OK)
            atomicMax((int *)&p.result_meta[META_STATUS], status);
        if (n_ops > p.ops_cap)
            atomicMax((int *)&p.result_meta[META_STATUS], (int)ST_OPS_OVERFLOW);
    }
    group_sync(cx); // the workspace may be reused by the next problem of this group
    (void)lane;
    (void)wid;
    (void)nw;
    (void)nbits;
}

// grid = n_groups * G CTAs; group i solves problems i, i + n_groups, ...
__device__ __forceinline__ void solve_own_kernel_body(const ProblemDesc *probs, int n_probs, const GroupWs *wss, const OwnWs *ows, const LaunchCfg &cfg, int n_out_max, int e_cap_max, int lcap, int hlog, int narrow) {
    DA_DYN_SHARED(smem);
    DA_SHARED_VAR(BlockCtx, bctx);
    DA_SHARED_VAR(OwnBlock, oblk);
    DA_SHARED_VAR(Ctx, cxs);
    DA_SHARED_VAR(OwnCtx, oxs);
    if (threadIdx.x == 0) {
        Ctx &cx = cxs;
        cx.cfg = cfg;
        cx.rank = blockIdx.x % cfg.G;
        const int group = blockIdx.x / cfg.G;
        cx.ws = wss[group];
        cx.seg = cx.ws.fseg + (size_t)cx.rank * cx.ws.fseg_cap;
        cx.b = &bctx;
        unsigned char *sp = smem;
        cx.cb_score = (uint32_t *)sp;
        sp += sizeof(uint32_t) * cfg.nchunk_cap;
        cx.cb_khi = (uint32_t *)sp;
        sp += sizeof(uint32_t) * cfg.nchunk_cap;
        cx.cb_klo = (uint32_t *)sp;
        sp += sizeof(uint32_t) * cfg.nchunk_cap;
        cx.dirty_list = (int *)sp;
        sp += sizeof(int) * cfg.nchunk_cap;
        cx.cb_dirty = sp;
        OwnCtx &ox = oxs;
        ox.ws = ows[group];
        ox.lay = own_plan(cfg.nchunk_cap, n_out_max, e_cap_max, lcap, hlog, narrow).lay;
        ox.ob = &oblk;
        ox.ovf = ox.ws.ovf + (size_t)cx.rank * (size_t)n_out_max * 3 * (size_t)ox.ws.ovf_cap;
        bctx.bar_target = 0u; // the host zeroes the arrive counter and the exchange slots before every launch
        bctx.epoch = 0u;
    }
    __syncthreads();
    const int group = blockIdx.x / cfg.G, n_groups = gridDim.x / cfg.G;
    for (int pi = group; pi < n_probs; pi += n_groups)
        solve_problem_own(probs[pi], cxs, oxs);
}
__global__ void __launch_bounds__(512, 1) cmvm_solve_kernel(const ProblemDesc *probs, int n_probs, const GroupWs *wss, const OwnWs *ows, LaunchCfg cfg, int n_out_max, int e_cap_max, int lcap, int hlog, int narrow) {
    solve_own_kernel_body(probs, n_probs, wss, ows, cfg, n_out_max, e_cap_max, lcap, hlog, narrow);
}

} // namespace da
