// sim_cmvm.cc -- TEST INFRASTRUCTURE ONLY: runs the product's CUDA kernel sources (cmvm_prep_kernel, cmvm_solve_kernel;
// da4ml_b200/csrc/*.cuh, unmodified) on the CPU under the SIMT shim of simt.h, for one solve_single job, so that their
// logic can be compared with the oracle in the CPU test suite.  The buffer sizing mirrors run_stage_jobs
// (da4ml_b200/csrc/host_stage.cuh) and uses the product's own planner (host_plan.cuh).  Never linked into the product.
#include "simt.h"

#include "../../da4ml_b200/csrc/cmvm_kernel_own.cuh"
#include "../../da4ml_b200/csrc/cmvm_decompose.cuh"
#include "../../da4ml_b200/csrc/host_plan.cuh"

#include <string>

using namespace da;

namespace {
std::string g_err;
int method_id(const std::string &m) {
    const char *names[] = {"mc", "mc-dc", "mc-pdc", "wmc", "wmc-dc", "wmc-pdc", "dummy"};
    for (int i = 0; i < 7; ++i)
        if (m == names[i])
            return i;
    throw std::runtime_error("Unknown method: " + m);
}
int ilog2_ceil(int v) {
    int l = 0;
    while ((1 << l) < v)
        ++l;
    return l;
}
template <class T> T *zalloc(std::vector<std::unique_ptr<unsigned char[]>> &keep, size_t n) {
    const size_t bytes = std::max<size_t>(n, 1) * sizeof(T) + 64;
    keep.emplace_back(new unsigned char[bytes]());
    uintptr_t a = ((uintptr_t)keep.back().get() + 63) & ~(uintptr_t)63;
    return (T *)a;
}
// like zalloc, but filled with garbage when poisoning is on: for every buffer the host driver does NOT clear before a
// launch (run_stage_jobs zeroes only the counter slab, the barrier / exchange words and result_meta)
static bool g_poison = false;
template <class T> T *palloc(std::vector<std::unique_ptr<unsigned char[]>> &keep, size_t n) {
    T *p = zalloc<T>(keep, n);
    if (g_poison)
        memset((void *)p, 0xA5, std::max<size_t>(n, 1) * sizeof(T));
    return p;
}
} // namespace

extern "C" {

const char *sim_last_error() { return g_err.c_str(); }
void sim_set_schedule(int mode) { simt::schedule_mode() = mode; }
void sim_set_poison(int on) { g_poison = on != 0; }
static int g_fcap_override = 0, g_ecap_override = 0, g_pool_override = 0, g_lcap_override = 0, g_hlog_override = 0, g_ovf_override = -1;
static bool g_lcap_set = false;
static int g_wide_rows = 0;
// shrink capacities (0 = the planner's size) so that small problems reach the compaction / overflow paths: histogram
// segment entries per CTA, expression table entries, cells per CTA
void sim_set_segment_cap(int entries) { g_fcap_override = entries; }
void sim_set_caps(int e_cap, int pool) {
    g_ecap_override = e_cap;
    g_pool_override = pool;
}
// rows per shared-memory owner list; < 0 = the planner's size, 0 = every row in global memory
void sim_set_list_cap(int rows) {
    g_lcap_override = rows < 0 ? 0 : rows;
    g_lcap_set = rows >= 0;
}
// the product's first-attempt capacities (host_plan.cuh FirstCap; 0 = planner's), applied where run_stage_jobs applies them
static long long g_first_caps[CAP_WORDS] = {0};
void sim_set_first_attempt_caps(const long long *caps) {
    for (int k = 0; k < CAP_WORDS; ++k)
        g_first_caps[k] = caps[k];
}
// log2 of the pair-counter hash table (0 = planner's), spill rows per owner list (< 0 = planner's)
void sim_set_wide_rows(int on) { g_wide_rows = on; } // 12-byte list rows even when 6 bytes would do
void sim_set_own_caps(int hlog, int ovf_rows) {
    g_hlog_override = hlog;
    g_ovf_override = ovf_rows;
}

// Self-test of the shim: warp collectives, block barrier, shared variables, inter-CTA polling, deadlock detection.
// Returns 0 when every check passes, else the number of the failing check.
int sim_selftest() {
    try {
        std::vector<int> out(2 * 64, -1);
        std::vector<unsigned> flag(1, 0u);
        simt::launch(dim3(2), dim3(64), 128, [&] {
            DA_SHARED_VAR(int, total);
            DA_DYN_SHARED(dyn);
            const int tid = threadIdx.x, lane = tid & 31;
            if (tid == 0)
                total = 0;
            __syncthreads();
            int v = lane;
            for (int off = 16; off > 0; off >>= 1)
                v += __shfl_xor_sync(0xffffffffu, v, off); // 496 on every lane
            const unsigned b = __ballot_sync(0xffffffffu, (lane & 1) != 0);
            const int up = __shfl_up_sync(0xffffffffu, lane, 1);
            if (v == 496 && b == 0xaaaaaaaau && up == (lane ? lane - 1 : 0) && __shfl_sync(0xffffffffu, tid, 5) == (tid & ~31) + 5)
                atomicAdd(&total, 1);
            ((int *)dyn)[tid & 31] = tid; // touch dynamic shared memory
            __syncthreads();
            // CTA 1 waits for CTA 0 through a polled global flag
            if (blockIdx.x == 0 && tid == 0)
                flag[0] = 1u;
            if (blockIdx.x == 1 && tid == 0)
                while (ld_acquire_u32(&flag[0]) == 0u) {
                }
            __syncthreads();
            out[blockIdx.x * 64 + tid] = total;
        });
        for (int v : out)
            if (v != 64)
                return 1;
        bool caught = false;
        try {
            simt::launch(dim3(1), dim3(32), 0, [&] {
                if (threadIdx.x != 3)
                    __syncthreads(); // thread 3 never arrives
            });
        } catch (const std::runtime_error &e) {
            caught = std::string(e.what()).find("deadlock") != std::string::npos;
        }
        if (!caught)
            return 2;
        caught = false;
        try {
            simt::launch(dim3(1), dim3(32), 0, [&] {
                if (threadIdx.x < 16)
                    (void)__ballot_sync(0xffffffffu, true); // half of the warp skips a full-mask collective
            });
        } catch (const std::runtime_error &) {
            caught = true;
        }
        return caught ? 0 : 3;
    } catch (const std::exception &e) {
        g_err = e.what();
        return 100;
    }
}

} // extern "C"

struct SimJob {
    const float *kernel, *qint, *lat;
    int n_in, n_out, method, adder_size, carry_size;
    // outputs (caller-owned)
    int64_t *meta, *inp_shifts, *out_idxs, *out_shifts, *out_negs, *ops_i;
    float *ops_f;
    long long ops_room, n_ops;
};

// solve_single jobs on `n_groups` groups of `G` simulated CTAs (jobs beyond the number of groups reuse a group's
// workspace one after the other, as in a batched launch).  Mirrors run_stage_jobs.
static void run_jobs(std::vector<SimJob> &jobs, int G, int n_groups, int cta_threads, bool accounting, int list_mul) {
    std::vector<std::unique_ptr<unsigned char[]>> keep;
    const int n = (int)jobs.size();
    std::vector<ProblemDesc> desc(n);
    std::vector<PlanJob> pj(n);
    long long max_cols = 0, max_colcap = 0, max_heap = 0, max_ecap = 0;
    for (int i = 0; i < n; ++i) {
        SimJob &j = jobs[i];
        ProblemDesc &d = desc[i];
        memset(&d, 0, sizeof(d));
        d.n_in = j.n_in;
        d.n_out = j.n_out;
        d.method = j.method;
        d.adder_size = j.adder_size;
        d.carry_size = j.carry_size;
        float *k = zalloc<float>(keep, (size_t)j.n_in * j.n_out);
        memcpy(k, j.kernel, sizeof(float) * (size_t)j.n_in * j.n_out);
        d.kernel = k;
        float *q = zalloc<float>(keep, 3 * (size_t)j.n_in), *l = zalloc<float>(keep, j.n_in);
        memcpy(q, j.qint, sizeof(float) * 3 * j.n_in);
        memcpy(l, j.lat, sizeof(float) * j.n_in);
        d.qint = q;
        d.lat = l;
        d.masks0 = palloc<uint2>(keep, (size_t)j.n_in * j.n_out);
        d.shift0 = palloc<int8_t>(keep, j.n_in);
        d.shift1 = palloc<int8_t>(keep, j.n_out);
        d.col_digits = palloc<int>(keep, j.n_out);
        d.prep_meta = palloc<int>(keep, PM_WORDS);
    }
    simt::launch(dim3(n), dim3(256), 0, [&] { cmvm_prep_kernel(desc.data()); });
    for (int i = 0; i < n; ++i) {
        SimJob &j = jobs[i];
        ProblemDesc &d = desc[i];
        const int *pm = d.prep_meta;
        const long long d0 = pm[PM_D0];
        d.nbits = pm[PM_NBITS];
        long long t_cap = std::min<long long>(d0, d0 / 2 + 1024);
        if (g_first_caps[CAP_EXPR] > 0)
            t_cap = std::min(t_cap, g_first_caps[CAP_EXPR]);
        d.e_cap = (int)(j.n_in + t_cap + 1);
        d.ops_cap = (int)(j.n_in + d0 + 1);
        d.col_cap = pm[PM_COLCAP] + 1;
        d.heap_lane_cap = (std::min(d.nbits, 32) + 1) * ((d.col_cap + 31) / 32) + 2;
        d.op_misc = palloc<int4>(keep, d.ops_cap);
        d.op_q = palloc<float4>(keep, d.ops_cap);
        d.op_cost = palloc<float>(keep, d.ops_cap);
        d.out_q = palloc<float4>(keep, j.n_out);
        d.out_idx = palloc<int>(keep, j.n_out);
        d.out_shift = palloc<int>(keep, j.n_out);
        d.out_neg = palloc<int>(keep, j.n_out);
        d.result_meta = zalloc<long long>(keep, META_WORDS);
        pj[i].n_in = j.n_in;
        pj[i].n_out = j.n_out;
        pj[i].nbits = d.nbits;
        pj[i].d0 = d0;
        pj[i].dcol_max = pm[PM_DCOL_MAX];
        pj[i].col_cap = d.col_cap;
        pj[i].list_mul = list_mul > 0 ? list_mul : 2;
        pj[i].e_cap = d.e_cap;
        max_cols = std::max<long long>(max_cols, j.n_out);
        max_colcap = std::max<long long>(max_colcap, d.col_cap);
        max_ecap = std::max<long long>(max_ecap, d.e_cap);
        max_heap = std::max<long long>(max_heap, (long long)j.n_out * 32 * d.heap_lane_cap);
    }
    if (g_ecap_override > 0) // (buffers keep their full size)
        for (int i = 0; i < n; ++i)
            desc[i].e_cap = std::min(desc[i].e_cap, jobs[i].n_in + g_ecap_override);
    // launch geometry from the product's planner, with the group size pinned
    PlanEnv env;
    env.coop = G * n_groups;
    env.group_override = G;
    env.accounting = accounting;
    std::copy(g_first_caps, g_first_caps + CAP_WORDS, env.caps);
    LaunchPlan plan = plan_launch(pj, env);
    if (g_lcap_set) { // shrink the shared-memory part of the owner lists: rows spill to global memory
        plan.ovf_cap += std::max(0, plan.lcap - g_lcap_override);
        plan.lcap = std::min(plan.lcap, g_lcap_override) & ~1;
    }
    if (g_hlog_override > 0)
        plan.hlog = g_hlog_override;
    if (g_wide_rows)
        plan.narrow = 0;
    if (g_ovf_override >= 0)
        plan.ovf_cap = g_ovf_override;
    plan.smem_bytes = own_plan_bytes(plan.cfg.nchunk_cap, plan.n_out_max, plan.e_cap_max, plan.lcap, plan.hlog, plan.narrow);
    if (own_plan(plan.cfg.nchunk_cap, plan.n_out_max, plan.e_cap_max, plan.lcap, plan.hlog, plan.narrow).bytes != plan.smem_bytes)
        throw std::runtime_error("own_plan_bytes (host planner) and own_plan (kernel layout) disagree");
    const LaunchCfg cfg = plan.cfg;
    std::vector<GroupWs> gws(n_groups);
    std::vector<OwnWs> ows(n_groups);
    for (int gi = 0; gi < n_groups; ++gi) {
        GroupWs &w = gws[gi];
        memset(&w, 0, sizeof(w));
        w.col_u32 = palloc<uint32_t>(keep, (size_t)3 * max_cols * max_colcap);
        w.col_len = palloc<int>(keep, max_cols);
        w.col_k = palloc<int>(keep, max_cols);
        w.mod_step = palloc<uint32_t>(keep, max_ecap);
        w.fseg = palloc<FEnt>(keep, (size_t)G * plan.max_fcap);
        w.heap = palloc<uint4>(keep, 2 * (size_t)max_heap);
        w.barrier = zalloc<unsigned>(keep, 64);
        w.xchg = zalloc<unsigned long long>(keep, 2 * 4 * (size_t)G);
        w.fseg_cap = g_fcap_override > 0 ? std::min<int>(g_fcap_override, (int)plan.max_fcap) : (int)plan.max_fcap;
        w.heap_cap = max_heap;
        OwnWs &e = ows[gi];
        memset(&e, 0, sizeof(e));
        e.pool_cap = g_pool_override > 0 ? std::min<int>(g_pool_override, (int)plan.pool_cap) : (int)plan.pool_cap;
        e.e_cap = (int)max_ecap;
        e.ovf_cap = (int)plan.ovf_cap;
        e.n_out_max = (int)max_cols;
        e.cell_col = palloc<uint32_t>(keep, (size_t)G * e.pool_cap);
        e.cell_pl[0] = palloc<uint2>(keep, (size_t)G * e.pool_cap);
        e.cell_pl[1] = palloc<uint2>(keep, (size_t)G * e.pool_cap);
        e.cell_dir = palloc<uint2>(keep, (size_t)max_ecap);
        e.ovf = palloc<uint32_t>(keep, 3 * (size_t)G * (size_t)max_cols * (size_t)std::max(e.ovf_cap, 1));
    }
    simt::launch(dim3(G * n_groups), dim3(cta_threads), plan.smem_bytes,
                 [&] { cmvm_solve_kernel(desc.data(), n, gws.data(), ows.data(), cfg, (int)max_cols, (int)max_ecap, plan.lcap, plan.hlog, plan.narrow); });
    for (int i = 0; i < n; ++i) {
        SimJob &j = jobs[i];
        const ProblemDesc &d = desc[i];
        for (int w = 0; w < 32; ++w) // (the caller's array holds the 32 counter words, not the milestone snapshots)
            j.meta[w] = d.result_meta[w];
        j.meta[10] = d.prep_meta[PM_D0];
        j.meta[11] = d.nbits;
        j.meta[12] = cfg.G;
        j.meta[15] = plan.lcap;
        if (d.result_meta[META_STATUS] != ST_OK) {
            j.n_ops = -(long long)d.result_meta[META_STATUS];
            continue;
        }
        j.n_ops = d.result_meta[META_N_OPS];
        if (j.n_ops > j.ops_room)
            throw std::runtime_error("ops_room too small");
        for (int k = 0; k < j.n_in; ++k)
            j.inp_shifts[k] = d.shift0[k];
        for (int o = 0; o < j.n_out; ++o) {
            j.out_idxs[o] = d.out_idx[o];
            j.out_shifts[o] = d.out_shift[o];
            j.out_negs[o] = d.out_neg[o];
        }
        for (long long k = 0; k < j.n_ops; ++k) {
            j.ops_i[4 * k + 0] = d.op_misc[k].x;
            j.ops_i[4 * k + 1] = d.op_misc[k].y;
            j.ops_i[4 * k + 2] = d.op_misc[k].z;
            j.ops_i[4 * k + 3] = d.op_misc[k].w;
            j.ops_f[5 * k + 0] = d.op_q[k].x;
            j.ops_f[5 * k + 1] = d.op_q[k].y;
            j.ops_f[5 * k + 2] = d.op_q[k].z;
            j.ops_f[5 * k + 3] = d.op_q[k].w;
            j.ops_f[5 * k + 4] = d.op_cost[k];
        }
    }
}

extern "C" {

// One solve_single on `G` simulated CTAs of `cta_threads` threads.  Returns the number of ops (>= 0) or -(status) when a
// capacity was exceeded, -100 on an exception (sim_last_error()).  meta_out: the kernel's 32 result words.
long long sim_solve_single(const float *kernel, int n_in, int n_out, const char *method, const float *qint, const float *lat, int adder_size, int carry_size,
                           int G, int cta_threads, int accounting, int list_mul, int64_t *meta_out, int64_t *inp_shifts, int64_t *out_idxs,
                           int64_t *out_shifts, int64_t *out_negs, int64_t *ops_i, float *ops_f, long long ops_room) {
    try {
        std::vector<SimJob> jobs(1);
        jobs[0] = SimJob{kernel, qint, lat, n_in, n_out, method_id(method), adder_size, carry_size, meta_out, inp_shifts, out_idxs, out_shifts, out_negs, ops_i, ops_f, ops_room, 0};
        run_jobs(jobs, G, 1, cta_threads, accounting != 0, list_mul);
        return jobs[0].n_ops;
    } catch (const std::exception &e) {
        g_err = e.what();
        return -100;
    }
}

// `n` jobs described by arrays of pointers / sizes (default options otherwise) on n_groups groups; n_ops_out[i] as above.
int sim_solve_many(int n, const float **kernels, const int *n_in, const int *n_out, const char *method, const float **qints, const float **lats, int G, int n_groups,
                   int cta_threads, int64_t **metas, int64_t **inp_shifts, int64_t **out_idxs, int64_t **out_shifts, int64_t **out_negs, int64_t **ops_i,
                   float **ops_f, const long long *ops_room, long long *n_ops_out) {
    try {
        std::vector<SimJob> jobs(n);
        for (int i = 0; i < n; ++i)
            jobs[i] = SimJob{kernels[i], qints[i], lats[i], n_in[i], n_out[i], method_id(method), -1, -1, metas[i], inp_shifts[i], out_idxs[i], out_shifts[i], out_negs[i], ops_i[i], ops_f[i], ops_room[i], 0};
        run_jobs(jobs, G, n_groups, cta_threads, false, 2);
        for (int i = 0; i < n; ++i)
            n_ops_out[i] = jobs[i].n_ops;
        return 0;
    } catch (const std::exception &e) {
        g_err = e.what();
        return -100;
    }
}

// kernel_decompose (mat_decompose.cc:62-137) through center_kernel, dist_kernel and mst_build_kernel, launched as
// solve_many does (host_solve.cuh).  m0: [n_in][n_out], m1: [n_out][n_out].
int sim_kernel_decompose(const float *kernel, int n_in, int n_out, int dc, float *m0, float *m1) {
    try {
        std::vector<std::unique_ptr<unsigned char[]>> keep;
        const int n = n_out + 1;
        float *k = zalloc<float>(keep, (size_t)n_in * n_out);
        memcpy(k, kernel, sizeof(float) * (size_t)n_in * n_out);
        float *aug = zalloc<float>(keep, (size_t)n_in * n);
        int8_t *s0 = zalloc<int8_t>(keep, n_in), *s1 = zalloc<int8_t>(keep, n_out);
        int *dist = zalloc<int>(keep, (size_t)n * n);
        int8_t *sign = zalloc<int8_t>(keep, (size_t)n * n);
        DecompJob job;
        job.dc = dc;
        job.m0 = zalloc<float>(keep, (size_t)n_in * n_out);
        job.m1 = zalloc<float>(keep, (size_t)n_out * n_out);
        job.mapping = zalloc<int>(keep, 2 * (size_t)n);
        simt::launch(dim3(1), dim3(256), 0, [&] { center_kernel(k, n_in, n_out, aug, s0, s1); });
        simt::launch(dim3((unsigned)(((long long)n * n + 255) / 256)), dim3(256), 0, [&] { dist_kernel(aug, n_in, n, dist, sign); });
        const int threads = std::min(1024, std::max(64, (n + 31) / 32 * 32));
        simt::launch(dim3(1), dim3(threads), (size_t)n * 17 + 64, [&] { mst_build_kernel(aug, dist, sign, s0, s1, n_in, n_out, &job); });
        memcpy(m0, job.m0, sizeof(float) * (size_t)n_in * n_out);
        memcpy(m1, job.m1, sizeof(float) * (size_t)n_out * n_out);
        return 0;
    } catch (const std::exception &e) {
        g_err = e.what();
        return -100;
    }
}
}
