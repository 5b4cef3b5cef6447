// host_stage.cuh -- one round of solve_single jobs on the device: prep launch, capacity planning, the persistent
// cooperative solve launch, retries on capacity overflow, result download (reference cmvm_core.cc:227-237 per job).
#pragma once
#include "host_common.cuh"
#include "host_plan.cuh"
#include <deque>

namespace da {

// ------------------------------------------------------------------------------------------------
// one CSE stage = one solve_single job

struct StageResult {
    int64_t n_in = 0, n_out = 0;
    int carry_size = -1, adder_size = -1;
    std::vector<int64_t> inp_shifts, out_idxs, out_shifts, out_negs;
    std::vector<float4> out_q; // per output: (qmin, qmax, qstep, latency) of its op; (0, 0, inf, 0) for dead outputs
    float cost_sum = 0.0f;     // cost_init + sum of op costs in op order (float, device)
    int64_t n_ops_dev = 0;
    // op records in device layout: they stay on the device until somebody needs them (only the winning candidate's are
    // ever copied back); expanded to the ABI's int64 / float32 tables when a caller asks for them
    const int4 *d_misc = nullptr;
    const float4 *d_q = nullptr;
    const float *d_cost = nullptr;
    bool have_ops = false;
    std::vector<int4> op_misc;   // id0, id1, opcode, data
    std::vector<float4> op_q;    // qmin, qmax, qstep, latency
    std::vector<float> op_cost;
    int64_t counters[META_WORDS] = {0};
    int64_t n_ops() const { return n_ops_dev; }
};

struct StageJob {
    int n_in = 0, n_out = 0, method = M_WMC, adder_size = -1, carry_size = -1;
    const float *d_kernel = nullptr; // device, [n_in][n_out]
    std::vector<float> qint, lat;    // host
    float cost_init = 0.0f; // float cost accumulated by the earlier stage(s) of the same candidate
    int32_t *trace = nullptr;
    int64_t trace_cap = 0;
    StageResult res;
    // capacity escalation after an overflow status
    bool full_expr = false;
    int f_mul = 1, list_mul = 2;
};

// Device memory for per-job outputs that must outlive one run_stage_jobs call (op tables of every candidate until the
// winner is known): bump allocation over a list of chunks, recycled by the next API call.
struct OutArena {
    std::deque<DevBuf> chunks; // (a deque: the buffers register their address, which must stay put; chunks are only ever added)
    size_t cur = 0, off = 0;
    void reset() {
        cur = 0;
        off = 0;
    }
    char *take(size_t bytes) {
        bytes = (bytes + 255) & ~size_t(255);
        while (true) {
            if (cur < chunks.size() && off + bytes <= chunks[cur].cap) {
                char *p = (char *)chunks[cur].p + off;
                off += bytes;
                return p;
            }
            if (cur < chunks.size() && off == 0 && chunks[cur].cap < bytes) { // empty chunk too small: regrow it
                chunks[cur].ensure(bytes, false);
                continue;
            }
            if (cur + 1 < chunks.size() || (cur < chunks.size() && off > 0)) {
                if (cur + 1 >= chunks.size())
                    chunks.emplace_back();
                ++cur;
                off = 0;
                if (chunks[cur].cap < bytes)
                    chunks[cur].ensure(std::max<size_t>(bytes, size_t(256) << 20), false);
                continue;
            }
            chunks.emplace_back();
            cur = chunks.size() - 1;
            off = 0;
            chunks[cur].ensure(std::max<size_t>(bytes, size_t(256) << 20), false);
        }
    }
};
static OutArena g_out_arena2;

static void release_device_buffers() {
    for (DevBuf *b : devbuf_registry())
        b->drop();
    g_out_arena2.reset(); // (its chunks were dropped with the rest and are re-grown on demand)
}

// copy one stage's op table back (device layout)
static void fetch_ops(StageResult &r) {
    if (r.have_ops)
        return;
    const size_t n = (size_t)r.n_ops_dev;
    r.op_misc.resize(n);
    r.op_q.resize(n);
    r.op_cost.resize(n);
    if (n) {
        CK(cudaMemcpyAsync(r.op_misc.data(), r.d_misc, sizeof(int4) * n, cudaMemcpyDeviceToHost, g_stream));
        CK(cudaMemcpyAsync(r.op_q.data(), r.d_q, sizeof(float4) * n, cudaMemcpyDeviceToHost, g_stream));
        CK(cudaMemcpyAsync(r.op_cost.data(), r.d_cost, sizeof(float) * n, cudaMemcpyDeviceToHost, g_stream));
        CK(cudaStreamSynchronize(g_stream));
    }
    r.have_ops = true;
}

static int ilog2_ceil(int v) {
    int l = 0;
    while ((1 << l) < v)
        ++l;
    return l;
}

// Solve all jobs concurrently (one prep launch + one persistent solve launch per attempt).
static void run_stage_jobs(std::vector<StageJob *> &jobs, Timing &tm, bool want_ops) {
    if (jobs.empty())
        return;
    init_device();
    const int nj = (int)jobs.size();
    std::vector<StageJob *> todo(jobs.begin(), jobs.end());
    for (int attempt = 0; attempt < 6 && !todo.empty(); ++attempt) {
        const int n = (int)todo.size();
        // ---- job arena: inputs + prep outputs
        Carver cj;
        struct Off {
            size_t qint, lat, masks, s0, s1, cold, pmeta;
        };
        std::vector<Off> off(n);
        for (int i = 0; i < n; ++i) {
            StageJob &j = *todo[i];
            off[i].qint = cj.take(sizeof(float) * 3 * j.n_in);
            off[i].lat = cj.take(sizeof(float) * j.n_in);
            off[i].masks = cj.take(sizeof(uint2) * (size_t)j.n_in * j.n_out);
            off[i].s0 = cj.take(j.n_in);
            off[i].s1 = cj.take(j.n_out);
            off[i].cold = cj.take(sizeof(int) * j.n_out);
            off[i].pmeta = cj.take(sizeof(int) * PM_WORDS);
        }
        const size_t job_in_bytes = cj.off;
        g_job_arena.ensure(job_in_bytes, false);
        char *ja = (char *)g_job_arena.p;
        // upload qint/lat through one pinned staging buffer
        {
            size_t up = 0;
            for (int i = 0; i < n; ++i)
                up += sizeof(float) * 4 * todo[i]->n_in;
            g_pin_up.ensure(up + sizeof(ProblemDesc) * n);
            char *hp = (char *)g_pin_up.p;
            size_t o = 0;
            for (int i = 0; i < n; ++i) {
                StageJob &j = *todo[i];
                memcpy(hp + o, j.qint.data(), sizeof(float) * 3 * j.n_in);
                CK(cudaMemcpyAsync(ja + off[i].qint, hp + o, sizeof(float) * 3 * j.n_in, cudaMemcpyHostToDevice, g_stream));
                o += sizeof(float) * 3 * j.n_in;
                memcpy(hp + o, j.lat.data(), sizeof(float) * j.n_in);
                CK(cudaMemcpyAsync(ja + off[i].lat, hp + o, sizeof(float) * j.n_in, cudaMemcpyHostToDevice, g_stream));
                o += sizeof(float) * j.n_in;
            }
        }
        std::vector<ProblemDesc> desc(n);
        for (int i = 0; i < n; ++i) {
            StageJob &j = *todo[i];
            ProblemDesc &d = desc[i];
            memset(&d, 0, sizeof(d));
            d.n_in = j.n_in;
            d.n_out = j.n_out;
            d.method = j.method;
            d.adder_size = j.adder_size;
            d.carry_size = j.carry_size;
            d.kernel = j.d_kernel;
            d.qint = (const float *)(ja + off[i].qint);
            d.lat = (const float *)(ja + off[i].lat);
            d.masks0 = (uint2 *)(ja + off[i].masks);
            d.shift0 = (int8_t *)(ja + off[i].s0);
            d.shift1 = (int8_t *)(ja + off[i].s1);
            d.col_digits = (int *)(ja + off[i].cold);
            d.prep_meta = (int *)(ja + off[i].pmeta);
        }
        g_desc_arena.ensure(sizeof(ProblemDesc) * n + sizeof(GroupWs) * 256 + 4096, false);
        ProblemDesc *d_desc = (ProblemDesc *)g_desc_arena.p;
        CK(cudaMemcpyAsync(d_desc, desc.data(), sizeof(ProblemDesc) * n, cudaMemcpyHostToDevice, g_stream));
        tm.begin();
        cmvm_prep_kernel<<<n, 256, 0, g_stream>>>(d_desc);
        tm.end(1);
        CK(cudaGetLastError());
        std::vector<int> pmeta((size_t)n * PM_WORDS);
        for (int i = 0; i < n; ++i)
            CK(cudaMemcpyAsync(&pmeta[(size_t)i * PM_WORDS], desc[i].prep_meta, sizeof(int) * PM_WORDS, cudaMemcpyDeviceToHost, g_stream));
        CK(cudaStreamSynchronize(g_stream));
        tm.collect();

        // ---- capacities, group geometry
        bool accounting = g_accounting != 0;
        for (int i = 0; i < n; ++i)
            accounting = accounting || todo[i]->trace_cap > 0;
        const int coop = g_max_coop, cta_threads = 512; // one persistent 512-thread CTA per SM
        // ---- per-job quantities that do not depend on the group size
        Carver co;
        co.off = job_in_bytes;
        struct OOff {
            size_t oi, os, on, meta, trace;
        };
        std::vector<OOff> oo(n);
        long long max_cols = 0, max_colcap = 0, max_heap = 0, max_ecap = 0;
        const long long *caps = attempt == 0 ? g_first_caps : nullptr; // forced capacities (set_first_attempt_caps): first attempt only
        for (int i = 0; i < n; ++i) {
            StageJob &j = *todo[i];
            const int *pm = &pmeta[(size_t)i * PM_WORDS];
            ProblemDesc &d = desc[i];
            const long long d0 = pm[PM_D0];
            d.nbits = pm[PM_NBITS];
            long long t_cap = j.full_expr ? d0 : std::min<long long>(d0, d0 / 2 + 1024);
            if (caps && caps[CAP_EXPR] > 0)
                t_cap = std::min(t_cap, caps[CAP_EXPR]);
            d.e_cap = (int)(j.n_in + t_cap + 1);
            d.ops_cap = (int)(j.n_in + d0 + 1);
            d.col_cap = pm[PM_COLCAP] + 1;
            d.heap_lane_cap = (std::min(d.nbits, 32) + 1) * ((d.col_cap + 31) / 32) + 2;
            if (d.e_cap >= (1 << 28) || d.nbits > 32)
                throw ApiError(DA4ML_E_CAPACITY, "problem too large for the packed histogram keys");
            d.op_misc = (int4 *)g_out_arena2.take(sizeof(int4) * d.ops_cap);
            d.op_q = (float4 *)g_out_arena2.take(sizeof(float4) * d.ops_cap);
            d.op_cost = (float *)g_out_arena2.take(sizeof(float) * d.ops_cap);
            d.out_q = (float4 *)g_out_arena2.take(sizeof(float4) * j.n_out);
            d.cost_init = j.cost_init;
            oo[i].oi = co.take(sizeof(int) * j.n_out);
            oo[i].os = co.take(sizeof(int) * j.n_out);
            oo[i].on = co.take(sizeof(int) * j.n_out);
            oo[i].meta = co.take(sizeof(long long) * META_WORDS);
            d.trace_cap = (int)std::min<long long>(j.trace_cap, t_cap + 1);
            oo[i].trace = co.take(sizeof(int) * 5 * (size_t)std::max(d.trace_cap, 1));
            max_cols = std::max<long long>(max_cols, j.n_out);
            max_colcap = std::max<long long>(max_colcap, d.col_cap);
            max_ecap = std::max<long long>(max_ecap, d.e_cap);
            max_heap = std::max<long long>(max_heap, (long long)j.n_out * 32 * d.heap_lane_cap);
        }
        // ---- launch geometry (host_plan.cuh)
        std::vector<PlanJob> pj(n);
        for (int i = 0; i < n; ++i) {
            const StageJob &j = *todo[i];
            const int *pm = &pmeta[(size_t)i * PM_WORDS];
            pj[i].n_in = j.n_in;
            pj[i].n_out = j.n_out;
            pj[i].nbits = desc[i].nbits;
            pj[i].d0 = pm[PM_D0];
            pj[i].dcol_max = pm[PM_DCOL_MAX];
            pj[i].col_cap = desc[i].col_cap;
            pj[i].f_mul = j.f_mul;
            pj[i].list_mul = j.list_mul;
            pj[i].e_cap = desc[i].e_cap;
        }
        PlanEnv penv;
        penv.coop = coop;
        penv.accounting = accounting;
        penv.own_budget = g_own_smem_max - 1024;
        penv.group_override = g_group_override;
        if (caps)
            std::copy(caps, caps + CAP_WORDS, penv.caps);
        const LaunchPlan plan = plan_launch(pj, penv);
        const LaunchCfg cfg = plan.cfg;
        const int G = cfg.G, n_groups = plan.n_groups;
        const long long max_fcap = plan.max_fcap;
        const size_t smem_bytes = plan.smem_bytes;
        for (int i = 0; i < n; ++i)
            if (((long long)(desc[i].e_cap / G + 1) << 9) >= (1LL << 32))
                throw ApiError(DA4ML_E_CAPACITY, "problem too large for the 32-bit pair-counter keys");
        if (smem_bytes > (size_t)g_own_smem_max)
            throw ApiError(DA4ML_E_CAPACITY, "the solve kernel's shared-memory plan does not fit (" + std::to_string(smem_bytes) + " bytes)");
        static DevBuf g_out_arena;
        g_out_arena.ensure(co.off - job_in_bytes, false);
        char *oa = (char *)g_out_arena.p - job_in_bytes;
        for (int i = 0; i < n; ++i) {
            ProblemDesc &d = desc[i];
            d.out_idx = (int *)(oa + oo[i].oi);
            d.out_shift = (int *)(oa + oo[i].os);
            d.out_neg = (int *)(oa + oo[i].on);
            d.result_meta = (long long *)(oa + oo[i].meta);
            d.trace = todo[i]->trace_cap > 0 ? (int *)(oa + oo[i].trace) : nullptr;
            CK(cudaMemsetAsync(d.result_meta, 0, sizeof(long long) * META_WORDS, g_stream));
        }
        // ---- group workspaces
        Carver cw;
        struct WOff {
            size_t ents, len, colk, mod, fseg, heap, bar, xchg, e_col, e_pl0, e_pl1, e_dir, e_ovf;
        };
        std::vector<WOff> wo(n_groups);
        for (int gi = 0; gi < n_groups; ++gi) {
            wo[gi].ents = cw.take(sizeof(uint32_t) * 3 * max_cols * max_colcap);
            wo[gi].len = cw.take(sizeof(int) * max_cols);
            wo[gi].colk = cw.take(sizeof(int) * max_cols);
            wo[gi].mod = cw.take(sizeof(uint32_t) * max_ecap);
            wo[gi].fseg = cw.take(sizeof(FEnt) * (size_t)G * max_fcap);
            wo[gi].heap = cw.take(sizeof(uint4) * 2 * max_heap);
            wo[gi].bar = cw.take(256);
            wo[gi].xchg = cw.take(sizeof(unsigned long long) * 2 * 4 * G);
            wo[gi].e_col = cw.take(sizeof(uint32_t) * (size_t)G * plan.pool_cap);
            wo[gi].e_pl0 = cw.take(sizeof(uint2) * (size_t)G * plan.pool_cap);
            wo[gi].e_pl1 = cw.take(sizeof(uint2) * (size_t)G * plan.pool_cap);
            wo[gi].e_dir = cw.take(sizeof(uint2) * (size_t)max_ecap);
            wo[gi].e_ovf = cw.take(sizeof(uint32_t) * 3 * (size_t)G * (size_t)max_cols * (size_t)std::max<long long>(plan.ovf_cap, 1));
        }
        g_ws_arena.ensure(cw.off, false);
        std::vector<GroupWs> gws(n_groups);
        std::vector<OwnWs> ows(n_groups);
        char *wa = (char *)g_ws_arena.p;
        for (int gi = 0; gi < n_groups; ++gi) {
            GroupWs &w = gws[gi];
            memset(&w, 0, sizeof(w));
            w.col_u32 = (uint32_t *)(wa + wo[gi].ents);
            w.col_len = (int *)(wa + wo[gi].len);
            w.col_k = (int *)(wa + wo[gi].colk);
            w.mod_step = (uint32_t *)(wa + wo[gi].mod);
            w.fseg = (FEnt *)(wa + wo[gi].fseg);
            w.heap = (uint4 *)(wa + wo[gi].heap);
            w.barrier = (unsigned *)(wa + wo[gi].bar);
            w.fseg_cap = (int)max_fcap;
            w.heap_cap = max_heap;
            w.xchg = (unsigned long long *)(wa + wo[gi].xchg);
            CK(cudaMemsetAsync(w.barrier, 0, 256, g_stream));
            CK(cudaMemsetAsync(w.xchg, 0, sizeof(unsigned long long) * 2 * 4 * G, g_stream));
            OwnWs &e = ows[gi];
            memset(&e, 0, sizeof(e));
            e.cell_col = (uint32_t *)(wa + wo[gi].e_col);
            e.cell_pl[0] = (uint2 *)(wa + wo[gi].e_pl0);
            e.cell_pl[1] = (uint2 *)(wa + wo[gi].e_pl1);
            e.cell_dir = (uint2 *)(wa + wo[gi].e_dir);
            e.ovf = (uint32_t *)(wa + wo[gi].e_ovf);
            e.pool_cap = (int)plan.pool_cap;
            e.e_cap = (int)max_ecap;
            e.ovf_cap = (int)plan.ovf_cap;
            e.n_out_max = (int)max_cols;
        }
        const size_t desc_bytes = (sizeof(ProblemDesc) * n + 255) & ~size_t(255), gws_bytes = (sizeof(GroupWs) * n_groups + 255) & ~size_t(255);
        g_desc_arena.ensure(desc_bytes + gws_bytes + sizeof(OwnWs) * n_groups + 4096, false);
        ProblemDesc *d_desc2 = (ProblemDesc *)g_desc_arena.p;
        GroupWs *d_gws = (GroupWs *)((char *)g_desc_arena.p + desc_bytes);
        OwnWs *d_ows = (OwnWs *)((char *)g_desc_arena.p + desc_bytes + gws_bytes);
        // biggest problems first so that the groups finish together
        std::vector<int> order(n);
        for (int i = 0; i < n; ++i)
            order[i] = i;
        std::stable_sort(order.begin(), order.end(), [&](int a, int b) { return pmeta[(size_t)a * PM_WORDS + PM_D0] > pmeta[(size_t)b * PM_WORDS + PM_D0]; });
        std::vector<ProblemDesc> sorted(n);
        for (int i = 0; i < n; ++i)
            sorted[i] = desc[order[i]];
        {
            g_pin_up.ensure(sizeof(ProblemDesc) * n + sizeof(GroupWs) * n_groups + sizeof(OwnWs) * n_groups);
            char *hp = (char *)g_pin_up.p; // (the earlier uploads from this buffer have completed: the stream was synced)
            memcpy(hp, sorted.data(), sizeof(ProblemDesc) * n);
            memcpy(hp + sizeof(ProblemDesc) * n, gws.data(), sizeof(GroupWs) * n_groups);
            memcpy(hp + sizeof(ProblemDesc) * n + sizeof(GroupWs) * n_groups, ows.data(), sizeof(OwnWs) * n_groups);
            CK(cudaMemcpyAsync(d_desc2, hp, sizeof(ProblemDesc) * n, cudaMemcpyHostToDevice, g_stream));
            CK(cudaMemcpyAsync(d_gws, hp + sizeof(ProblemDesc) * n, sizeof(GroupWs) * n_groups, cudaMemcpyHostToDevice, g_stream));
            CK(cudaMemcpyAsync(d_ows, hp + sizeof(ProblemDesc) * n + sizeof(GroupWs) * n_groups, sizeof(OwnWs) * n_groups, cudaMemcpyHostToDevice, g_stream));
        }
        // ---- persistent solve kernel (cooperative launch: all CTAs must be co-resident for the group exchanges)
        {
            const ProblemDesc *a0 = d_desc2;
            int a1 = n;
            const GroupWs *a2 = d_gws;
            const OwnWs *a3 = d_ows;
            LaunchCfg a4 = cfg;
            int a5 = (int)max_cols, a6 = (int)max_ecap, a7 = plan.lcap, a8 = plan.hlog, a9 = plan.narrow;
            void *args[] = {(void *)&a0, (void *)&a1, (void *)&a2, (void *)&a3, (void *)&a4, (void *)&a5, (void *)&a6, (void *)&a7, (void *)&a8, (void *)&a9};
            tm.begin();
            CK(cudaLaunchCooperativeKernel((void *)cmvm_solve_kernel, dim3(n_groups * G), dim3(cta_threads), args, smem_bytes, g_stream));
            tm.end(1);
            tm.solve_launches += 1;
            tm.mark_solve();
        }
        // ---- results
        std::vector<long long> meta((size_t)n * META_WORDS);
        for (int i = 0; i < n; ++i)
            CK(cudaMemcpyAsync(&meta[(size_t)i * META_WORDS], desc[i].result_meta, sizeof(long long) * META_WORDS, cudaMemcpyDeviceToHost, g_stream));
        CK(cudaStreamSynchronize(g_stream));
        tm.collect();
        std::vector<StageJob *> again;
        size_t down = 0;
        for (int i = 0; i < n; ++i) {
            const long long *m = &meta[(size_t)i * META_WORDS];
            if (m[META_STATUS] == ST_OK)
                down += (want_ops ? (size_t)m[META_N_OPS] * 36 : 0) + (size_t)todo[i]->n_out * 28 + todo[i]->n_in + todo[i]->n_out + 5 * 4 * (size_t)desc[i].trace_cap + 1024;
        }
        g_pin_down.ensure(down + 4096);
        char *dp = (char *)g_pin_down.p;
        struct DOff {
            size_t misc, q, cost, oi, os, on, oq, s0, tr;
        };
        std::vector<DOff> dof(n);
        size_t dofs = 0;
        auto dtake = [&](size_t b) {
            size_t o = dofs;
            dofs += (b + 15) & ~size_t(15);
            return o;
        };
        for (int i = 0; i < n; ++i) {
            StageJob &j = *todo[i];
            const long long *m = &meta[(size_t)i * META_WORDS];
            if (m[META_STATUS] != ST_OK) {
                switch ((int)m[META_STATUS]) {
                case ST_EXPR_OVERFLOW:
                    if (j.full_expr)
                        throw ApiError(DA4ML_E_CAPACITY, "expression table overflow");
                    j.full_expr = true;
                    break;
                case ST_FSEG_OVERFLOW:
                    j.f_mul *= 4;
                    break;
                case ST_LIST_OVERFLOW: // owner lists (shared memory + spill rows) or the cell pool ran out
                    if (j.list_mul >= 64)
                        throw ApiError(DA4ML_E_CAPACITY, "expression list overflow");
                    j.list_mul *= 2;
                    break;
                default:
                    throw ApiError(DA4ML_E_CAPACITY, "internal capacity overflow, status " + std::to_string((int)m[META_STATUS]));
                }
                again.push_back(&j);
                continue;
            }
            const size_t n_ops = (size_t)m[META_N_OPS];
            if (want_ops) {
                dof[i].misc = dtake(sizeof(int4) * n_ops);
                dof[i].q = dtake(sizeof(float4) * n_ops);
                dof[i].cost = dtake(sizeof(float) * n_ops);
            }
            dof[i].oq = dtake(sizeof(float4) * j.n_out);
            dof[i].oi = dtake(sizeof(int) * j.n_out);
            dof[i].os = dtake(sizeof(int) * j.n_out);
            dof[i].on = dtake(sizeof(int) * j.n_out);
            dof[i].s0 = dtake(j.n_in);
            dof[i].tr = dtake(sizeof(int) * 5 * (size_t)std::max(desc[i].trace_cap, 1));
            if (want_ops) {
                CK(cudaMemcpyAsync(dp + dof[i].misc, desc[i].op_misc, sizeof(int4) * n_ops, cudaMemcpyDeviceToHost, g_stream));
                CK(cudaMemcpyAsync(dp + dof[i].q, desc[i].op_q, sizeof(float4) * n_ops, cudaMemcpyDeviceToHost, g_stream));
                CK(cudaMemcpyAsync(dp + dof[i].cost, desc[i].op_cost, sizeof(float) * n_ops, cudaMemcpyDeviceToHost, g_stream));
            }
            CK(cudaMemcpyAsync(dp + dof[i].oq, desc[i].out_q, sizeof(float4) * j.n_out, cudaMemcpyDeviceToHost, g_stream));
            CK(cudaMemcpyAsync(dp + dof[i].oi, desc[i].out_idx, sizeof(int) * j.n_out, cudaMemcpyDeviceToHost, g_stream));
            CK(cudaMemcpyAsync(dp + dof[i].os, desc[i].out_shift, sizeof(int) * j.n_out, cudaMemcpyDeviceToHost, g_stream));
            CK(cudaMemcpyAsync(dp + dof[i].on, desc[i].out_neg, sizeof(int) * j.n_out, cudaMemcpyDeviceToHost, g_stream));
            CK(cudaMemcpyAsync(dp + dof[i].s0, desc[i].shift0, j.n_in, cudaMemcpyDeviceToHost, g_stream));
            if (desc[i].trace)
                CK(cudaMemcpyAsync(dp + dof[i].tr, desc[i].trace, sizeof(int) * 5 * (size_t)desc[i].trace_cap, cudaMemcpyDeviceToHost, g_stream));
        }
        CK(cudaStreamSynchronize(g_stream));
        for (int i = 0; i < n; ++i) {
            StageJob &j = *todo[i];
            const long long *m = &meta[(size_t)i * META_WORDS];
            if (m[META_STATUS] != ST_OK)
                continue;
            StageResult &r = j.res;
            const size_t n_ops = (size_t)m[META_N_OPS];
            r.n_in = j.n_in;
            r.n_out = j.n_out;
            r.carry_size = j.carry_size;
            r.adder_size = j.adder_size;
            for (int w = 0; w < META_WORDS; ++w)
                r.counters[w] = m[w];
            // algorithmic bytes of this solve_single (SURVEY.md section 8d); sum_F is exact only in accounting mode
            tm.algo_bytes += 8.0 * j.n_in * j.n_out + 12.0 * (double)m[META_F0] + 2.0 * (double)m[META_R0] + 12.0 * (double)m[META_SUM_F] +
                             10.0 * (double)m[META_SUM_R] + 2.0 * (double)m[META_D_FINAL] + 56.0 * (double)m[META_N_OPS];
            r.counters[10] = pmeta[(size_t)i * PM_WORDS + PM_D0];
            r.counters[11] = pmeta[(size_t)i * PM_WORDS + PM_NBITS];
            r.counters[12] = G;
            r.counters[15] = plan.lcap;
            r.counters[12] = G;
            r.inp_shifts.resize(j.n_in);
            const int8_t *s0 = (const int8_t *)(dp + dof[i].s0);
            for (int k = 0; k < j.n_in; ++k)
                r.inp_shifts[k] = s0[k];
            r.out_idxs.resize(j.n_out);
            r.out_shifts.resize(j.n_out);
            r.out_negs.resize(j.n_out);
            const int *oi = (const int *)(dp + dof[i].oi), *os = (const int *)(dp + dof[i].os), *on = (const int *)(dp + dof[i].on);
            for (int k = 0; k < j.n_out; ++k) {
                r.out_idxs[k] = oi[k];
                r.out_shifts[k] = os[k];
                r.out_negs[k] = on[k];
            }
            r.n_ops_dev = (int64_t)n_ops;
            r.d_misc = desc[i].op_misc;
            r.d_q = desc[i].op_q;
            r.d_cost = desc[i].op_cost;
            r.have_ops = false;
            r.out_q.assign((const float4 *)(dp + dof[i].oq), (const float4 *)(dp + dof[i].oq) + j.n_out);
            {
                const uint32_t bits = (uint32_t)m[META_COST_BITS];
                memcpy(&r.cost_sum, &bits, 4);
            }
            if (want_ops) {
                r.op_misc.assign((const int4 *)(dp + dof[i].misc), (const int4 *)(dp + dof[i].misc) + n_ops);
                r.op_q.assign((const float4 *)(dp + dof[i].q), (const float4 *)(dp + dof[i].q) + n_ops);
                r.op_cost.assign((const float *)(dp + dof[i].cost), (const float *)(dp + dof[i].cost) + n_ops);
                r.have_ops = true;
            }
            if (j.trace && j.trace_cap > 0) {
                int64_t rows = std::min<int64_t>(std::min<int64_t>(j.trace_cap, desc[i].trace_cap), m[META_T]);
                memcpy(j.trace, dp + dof[i].tr, sizeof(int) * 5 * (size_t)rows);
            }
        }
        tm.retried_jobs += (int64_t)again.size();
        todo.swap(again);
    }
    if (!todo.empty())
        throw ApiError(DA4ML_E_CAPACITY, "could not size the solver buffers after repeated attempts");
    (void)nj;
}


} // namespace da
