// host_plan.cuh -- launch geometry of the persistent solve kernel: CTAs per problem (G), concurrent groups, and the
// shared-memory layout of one CTA.  Pure host arithmetic (no CUDA calls) so that it can be exercised without a GPU
// (da4ml_cmvm_plan, tests/test_planner.py).
#pragma once
#include <algorithm>
#include <cstring>
#include <vector>

#include "cmvm_types.cuh"

namespace da {

// what the planner needs to know about one solve_single job (after cmvm_prep_kernel has counted its digits)
struct PlanJob {
    int n_in = 0, n_out = 0, nbits = 0;
    long long d0 = 0;   // CSD digits of the matrix
    int dcol_max = 0;   // digits of the densest output column
    int col_cap = 0;    // hard bound on the rows of one column list
    int f_mul = 1, list_mul = 2; // capacity multipliers raised by retries
    int e_cap = 0;               // expression ids the job may use
};
// Capacities a development switch may force below the planner's choice on the first attempt of a round of jobs
// (da4ml_cmvm_set_first_attempt_caps): small problems then take the spill, split-pass, compaction and retry paths.
enum FirstCap : int { CAP_FSEG = 0, CAP_LCAP = 1, CAP_OVF = 2, CAP_HLOG = 3, CAP_POOL = 4, CAP_EXPR = 5, CAP_WORDS = 6 };
// log2 of the pair-counter table: one owned expression has at most 3 rows x 63 shifts x 2 signs = 378 counters, which
// must fit the 5/8 of the table one pass may claim (so a split always ends); slot indices are 16-bit
constexpr int HLOG_MIN = 10, HLOG_MAX = 16;

struct PlanEnv {
    int coop = 148;      // co-resident CTAs of the launch (one persistent 512-thread CTA per SM)
    bool accounting = false;
    int group_override = 0; // > 0: fixed group size (set_group_size)
    long long own_budget = 208 * 1024; // dynamic shared memory one CTA of the solve kernel may use
    long long caps[CAP_WORDS] = {0};   // > 0: upper bound on that capacity of the final plan (the group size is chosen without them)
};

// shared-memory bytes of one CTA of the owner-partitioned kernel (mirrors own_plan in cmvm_kernel_own.cuh, which is the
// layout the kernel uses; tests/test_planner.py checks the two against each other through da4ml_cmvm_plan)
inline size_t own_plan_bytes(int nchunk_cap, int n_out_max, int e_cap_max, int lcap, int hlog, int narrow) {
    auto up = [](size_t b) { return (b + 15) & ~size_t(15); };
    const size_t words = (size_t)(n_out_max + 31) / 32;
    size_t o = up((size_t)nchunk_cap * 17);
    o += 3 * up(8 * (size_t)n_out_max) + 5 * up(4 * words) + up(4 * (size_t)((e_cap_max + 31) / 32)) + up(4 * (size_t)n_out_max) + up(2 * (size_t)n_out_max) + up(4 * ((size_t)n_out_max + 1));
    o += 2 * up((size_t)4 << hlog) + up((size_t)2 << hlog) + up((narrow ? 6 : 12) * (size_t)n_out_max * (size_t)lcap);
    return o;
}

// ---- launch plan ---------------------------------------------------------------------------------------------------
struct LaunchPlan {
    LaunchCfg cfg;
    long long max_fcap = 0; // histogram-segment entries per CTA
    int n_groups = 1;
    int lcap = 0, hlog = 12;       // rows per owner list in shared memory, log2 of the pair-counter hash table
    int nbits_max = 1, narrow = 0; // narrow: list rows of 6 bytes
    int n_out_max = 0, e_cap_max = 0;
    long long pool_cap = 0, ovf_cap = 0; // cells per CTA; rows per owner list that may spill to global memory
    size_t smem_bytes = 0;
    bool lists_fit = false; // every owner list has its target capacity in shared memory
    bool roomy = false;     // ... next to a pair-counter table of at least 4096 counters
};

inline LaunchPlan plan_for_group(const std::vector<PlanJob> &jobs, const PlanEnv &env, int G) {
    LaunchPlan P;
    memset(&P.cfg, 0, sizeof(P.cfg));
    long long rows_target = 0, rows_hard = 0;
    for (const PlanJob &j : jobs) {
        // (half of a segment is the common log, half the hot regions; a log that is still 3/4 full after a compaction would
        // compact every step, so the capacity is generous.  A job that needs more reports it and is retried with f_mul x 4.)
        const long long fcap_total = (128 * j.d0 + 65536) * j.f_mul;
        P.max_fcap = std::max(P.max_fcap, fcap_total / G + fcap_total / (2 * G) + 8192);
        // ... and never small: with many CTAs per problem a CTA's share of the initial histogram plus what spills out of its
        // (then tiny) hot regions must not keep the common log above its compaction threshold (12 MB per CTA at most)
        P.max_fcap = std::max(P.max_fcap, std::min<long long>(768 * 1024, 16 * j.d0 + 65536) * j.f_mul);
        P.n_out_max = std::max(P.n_out_max, j.n_out);
        P.e_cap_max = std::max(P.e_cap_max, j.e_cap);
        P.nbits_max = std::max(P.nbits_max, j.nbits);
        const long long own_in = (j.n_in + G - 1) / G; // inputs one CTA owns
        // observed: a column holds up to ~1.6 x n_in rows; an owner's share of them fluctuates around 1 / G of that
        rows_target = std::max(rows_target, own_in + own_in / 2 + 8);
        rows_hard = std::max(rows_hard, std::min<long long>(j.col_cap, (long long)j.list_mul * 2 * own_in + 64));
        P.pool_cap = std::max(P.pool_cap, ((long long)j.n_in * j.n_out + j.d0) / G * j.list_mul + j.n_out + 64);
    }
    if (P.max_fcap >= (1LL << 27))
        P.max_fcap = (1LL << 27) - 1;
    const long long *caps = env.caps;
    if (caps[CAP_FSEG] > 0)
        P.max_fcap = std::min(P.max_fcap, caps[CAP_FSEG]);
    if (caps[CAP_POOL] > 0)
        P.pool_cap = std::min(P.pool_cap, caps[CAP_POOL]);
    LaunchCfg &cfg = P.cfg;
    cfg.G = G;
    cfg.cpc = (P.n_out_max + G - 1) / G;
    cfg.accounting = env.accounting ? 1 : 0;
    cfg.chunk_log = 6;
    while ((((P.max_fcap >> cfg.chunk_log) + 2) * 17) > 44 * 1024) // (small chunks: what a dead cached winner costs is one chunk re-read)
        ++cfg.chunk_log;
    cfg.nchunk_cap = (int)((P.max_fcap >> cfg.chunk_log) + 2);
    const long long budget = env.own_budget;
    P.narrow = (P.nbits_max <= 16 && (P.e_cap_max + G - 1) / G + 1 <= 65535) ? 1 : 0;
    // pair-counter hash table: as large as the target list capacity leaves room for (2^13 ... 2^11 counters)
    const int hlog_top = caps[CAP_HLOG] > 0 ? (int)std::min<long long>(13, caps[CAP_HLOG]) : 13;
    for (int hlog = hlog_top; hlog >= std::min(11, hlog_top); --hlog) {
        const long long fixed = (long long)own_plan_bytes(cfg.nchunk_cap, P.n_out_max, P.e_cap_max, 0, hlog, P.narrow);
        long long lcap = (budget - fixed) / ((P.narrow ? 6LL : 12LL) * P.n_out_max);
        lcap = std::max<long long>(0, std::min(lcap, rows_hard)) & ~1LL;
        P.hlog = hlog;
        P.lcap = (int)lcap;
        P.lists_fit = lcap >= std::min(rows_target, rows_hard);
        if (P.lists_fit)
            break;
    }
    P.roomy = P.lists_fit && P.hlog >= 12; // (a 2048-counter table means many counting passes per step while the rows are dense)
    if (caps[CAP_LCAP] > 0) // (the rows taken out of shared memory become spill rows)
        P.lcap = (int)(std::min<long long>(P.lcap, caps[CAP_LCAP]) & ~1LL);
    P.ovf_cap = std::max<long long>(0, rows_hard - P.lcap);
    if (caps[CAP_OVF] > 0)
        P.ovf_cap = std::min(P.ovf_cap, caps[CAP_OVF]);
    P.smem_bytes = own_plan_bytes(cfg.nchunk_cap, P.n_out_max, P.e_cap_max, P.lcap, P.hlog, P.narrow);
    return P;
}

// Group size: as many concurrent problems as possible, but with the owner lists in shared memory -- the jobs then run
// in equal waves over coop / G groups.
inline LaunchPlan plan_launch(const std::vector<PlanJob> &jobs, const PlanEnv &env_caps) {
    PlanEnv env = env_caps; // (forced capacities apply to the final plan only: they do not change the group size)
    for (long long &c : env.caps)
        c = 0;
    const int n = (int)jobs.size(), coop = env.coop;
    long long want = 1; // CTAs one problem can keep busy
    for (const PlanJob &j : jobs) {
        want = std::max(want, std::min<long long>(coop, std::max<long long>(1, j.d0 / 384)));
        // the initial histogram streams n_in^2 / 2 row pairs over n_out columns whatever the density (stage-1 matrices)
        want = std::max(want, std::min<long long>(coop, ((long long)j.n_in * j.n_in * j.n_out) >> 21));
    }
    int G = (int)std::min<long long>(want, std::max(1, coop / std::max(n, 1)));
    while (G < std::min<long long>(want, coop) && !plan_for_group(jobs, env, G).roomy)
        ++G;
    const int waves = (n + (coop / G) - 1) / (coop / G);
    const int groups = (n + waves - 1) / waves;
    G = (int)std::min<long long>(want, std::max(G, coop / groups));
    if (waves > 1) {
        // Several waves of (nearly) equal jobs: a job's time is ~ 1 / G in this range (measured: 128x128 int6 stage, G = 2, 3,
        // 4 -> 67.6, 46.7, 34.2 us per step), so the launch costs ceil(n / floor(coop / G)) / G job-times: pick the group size
        // that wastes the least of the last wave (64 x config 4: 384 jobs, G = 2 -> 6 waves on 74 groups = 0.865 of the
        // CTAs busy; G = 3 -> 8 waves on 49 groups = 0.973).  Ties go to the smaller group.
        const int g_lo = G, g_hi = (int)std::min<long long>(want, 2LL * G + 2);
        double best_u = 0.0;
        for (int g = g_lo; g <= g_hi; ++g) {
            const int gr = coop / g;
            if (gr < 1 || (g != g_lo && !plan_for_group(jobs, env, g).roomy))
                continue;
            const int wv = (n + gr - 1) / gr;
            const double u = (double)n * g / ((double)wv * coop);
            if (u > best_u + 0.01) {
                best_u = u;
                G = g;
            }
        }
    }
    if (env.group_override > 0)
        G = std::min(env.group_override, coop);
    LaunchPlan P = plan_for_group(jobs, env_caps, G);
    P.n_groups = std::max(1, std::min(n, coop / G));
    return P;
}

} // namespace da
