// host_solve.cuh -- the reference's candidate search and two-stage driver on the host (api.cc:28-250): every pending
// solve_single of every candidate of every problem goes into one launch per round.
#pragma once
#include "host_stage.cuh"

namespace da {

// ------------------------------------------------------------------------------------------------
// kernel_decompose on the device: results stay on the device for the stage jobs

// ------------------------------------------------------------------------------------------------
// _solve state machine (api.cc:28-145), one per decompose_dc candidate

struct PipelineImpl {
    std::vector<StageResult> stages;
    double device_ms = 0, solve_ms = 0, algo_bytes = 0;
    int64_t launches = 0, solve_launches = 0;
    int64_t jobs_total = 0, jobs_run = 0; // solve_single jobs the reference would execute / executed after sharing identical ones
    int64_t retried_jobs = 0;             // jobs relaunched after a capacity overflow
};

struct Candidate {
    // fixed
    int problem = 0;
    std::string method0, method1;
    int hard_dc = -1;
    int decompose_dc = -2; // current value (after the api.cc:74-80 clamp)
    int adder_size = -1, carry_size = -1;
    float latency_allowed = std::numeric_limits<float>::infinity();
    // state
    int phase = 0; // 0: needs stage 0, 1: needs stage 1, 2: done
    StageJob job0, job1;
    float *d_m0 = nullptr, *d_m1 = nullptr;
    int *d_map = nullptr;
};

struct Problem {
    const float *h_kernel = nullptr;
    int n_in = 0, n_out = 0;
    std::vector<float> qint, lat;
    // device
    float *d_kernel = nullptr, *d_aug = nullptr;
    int *d_dist = nullptr;
    int8_t *d_sign = nullptr, *d_s0 = nullptr, *d_s1 = nullptr;
    bool need_min_lat = false;
    StageJob min_lat_job;
    float min_lat = std::numeric_limits<float>::infinity();
    std::vector<int> cand; // indices into the candidate vector
};

static bool ends_with(const std::string &s, const std::string &suf) {
    return s.size() >= suf.size() && s.compare(s.size() - suf.size(), suf.size(), suf) == 0;
}

// Candidates of one problem often decompose to the very same stage matrix (a dense random matrix gives identical M0 for
// decompose_dc = -1, 0, 1 and for every dc beyond the unconstrained spanning tree's depth).  A solve_single job is a pure
// function of its inputs, so identical jobs are solved once and the result shared.  `mats[i]` are device matrices of
// `words[i]` 32-bit words; `key[i]` collects everything else that defines job i (method, sizes, intervals, ...): jobs
// with different keys are never compared.  Returns rep[i] = first job identical to i.
static std::vector<int> identical_jobs(const std::vector<const float *> &mats, const std::vector<long long> &words, const std::vector<std::string> &key, Timing &tm) {
    const int n = (int)mats.size();
    std::vector<int> rep(n);
    for (int i = 0; i < n; ++i)
        rep[i] = i;
    std::vector<MatPair> pairs;
    std::vector<std::pair<int, int>> who;
    for (int i = 0; i < n; ++i)
        for (int j = 0; j < i; ++j)
            if (key[i] == key[j] && words[i] == words[j]) {
                pairs.push_back(MatPair{(const uint32_t *)mats[j], (const uint32_t *)mats[i], words[i]});
                who.push_back({j, i});
            }
    if (pairs.empty())
        return rep;
    static DevBuf buf;
    static PinBuf pin;
    const size_t pb = sizeof(MatPair) * pairs.size(), ob = sizeof(int) * pairs.size();
    const size_t pb_al = (pb + 255) & ~size_t(255);
    buf.ensure(pb_al + ob, false);
    pin.ensure(pb + ob);
    CK(cudaStreamSynchronize(g_stream)); // (the pinned buffer may still be in use by the previous call's copies)
    memcpy(pin.p, pairs.data(), pb);
    CK(cudaMemcpyAsync(buf.p, pin.p, pb, cudaMemcpyHostToDevice, g_stream));
    int *d_out = (int *)((char *)buf.p + pb_al);
    tm.begin();
    mat_equal_kernel<<<(unsigned)pairs.size(), 256, 0, g_stream>>>((const MatPair *)buf.p, d_out);
    tm.end(1);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync((char *)pin.p + pb, d_out, ob, cudaMemcpyDeviceToHost, g_stream));
    CK(cudaStreamSynchronize(g_stream));
    tm.collect();
    const int *eq = (const int *)((char *)pin.p + pb);
    for (size_t k = 0; k < pairs.size(); ++k) // (pairs are ordered by i, then j ascending: the first identical j wins)
        if (eq[k] && rep[who[k].second] == who[k].second && rep[who[k].first] == who[k].first)
            rep[who[k].second] = who[k].first;
    return rep;
}

static float stage_max_latency(const StageResult &r) {
    float m = 0.0f;
    for (size_t k = 0; k < r.out_idxs.size(); ++k) {
        float lat = r.out_idxs[k] >= 0 ? r.out_q[k].w : 0.0f;
        m = std::max(m, lat);
    }
    return m;
}

static void solve_many(
    int64_t n_problems, const float *const *kernels, const int64_t *n_in, const int64_t *n_out, const std::string &method0_in,
    const std::string &method1_in, int hard_dc, int decompose_dc, const float *const *qints, const float *const *lats,
    int adder_size, int carry_size, bool search_all, std::vector<std::unique_ptr<PipelineImpl>> &out, bool kernels_on_device = false
) {
    init_device();
    g_out_arena2.reset();
    Timing tm;
    int64_t jobs_total = 0, jobs_run = 0;
    // validate methods up front (the reference throws from the worker, api.cc:231-240)
    parse_method(method0_in);
    if (method1_in != "auto")
        parse_method(method1_in);

    std::vector<Problem> probs(n_problems);
    std::vector<Candidate> cands;
    // ---- device residency of the inputs + decomposition scratch
    static DevBuf g_base, g_pool;
    Carver cb;
    struct BOff {
        size_t k, aug, dist, sign, s0, s1;
    };
    std::vector<BOff> bo(n_problems);
    size_t up_bytes = 0;
    for (int64_t pi = 0; pi < n_problems; ++pi) {
        Problem &P = probs[pi];
        if (n_in[pi] <= 0 || n_out[pi] <= 0)
            throw ApiError(DA4ML_E_INVALID, "kernel must be a non-empty 2D array");
        P.n_in = (int)n_in[pi];
        P.n_out = (int)n_out[pi];
        P.h_kernel = kernels[pi];
        const float *q = qints ? qints[pi] : nullptr;
        const float *l = lats ? lats[pi] : nullptr;
        P.qint.resize(3 * (size_t)P.n_in);
        P.lat.resize(P.n_in);
        for (int i = 0; i < P.n_in; ++i) { // api.cc:161-174 defaults
            P.qint[3 * i + 0] = q ? q[3 * i + 0] : -128.0f;
            P.qint[3 * i + 1] = q ? q[3 * i + 1] : 127.0f;
            P.qint[3 * i + 2] = q ? q[3 * i + 2] : 1.0f;
            P.lat[i] = l ? l[i] : 0.0f;
        }
        const size_t n = (size_t)P.n_out + 1;
        bo[pi].k = cb.take(sizeof(float) * (size_t)P.n_in * P.n_out);
        bo[pi].aug = cb.take(sizeof(float) * (size_t)P.n_in * n);
        bo[pi].dist = cb.take(sizeof(int) * n * n);
        bo[pi].sign = cb.take(n * n);
        bo[pi].s0 = cb.take(P.n_in);
        bo[pi].s1 = cb.take(P.n_out);
        up_bytes += sizeof(float) * (size_t)P.n_in * P.n_out;
    }
    g_base.ensure(cb.off, false);
    static PinBuf g_pin_k;
    g_pin_k.ensure(up_bytes);
    {
        size_t o = 0;
        for (int64_t pi = 0; pi < n_problems; ++pi) {
            Problem &P = probs[pi];
            char *b = (char *)g_base.p;
            P.d_kernel = (float *)(b + bo[pi].k);
            P.d_aug = (float *)(b + bo[pi].aug);
            P.d_dist = (int *)(b + bo[pi].dist);
            P.d_sign = (int8_t *)(b + bo[pi].sign);
            P.d_s0 = (int8_t *)(b + bo[pi].s0);
            P.d_s1 = (int8_t *)(b + bo[pi].s1);
            size_t bytes = sizeof(float) * (size_t)P.n_in * P.n_out;
            if (kernels_on_device) // inputs already resident in HBM
                CK(cudaMemcpyAsync(P.d_kernel, P.h_kernel, bytes, cudaMemcpyDeviceToDevice, g_stream));
            else {
                memcpy((char *)g_pin_k.p + o, P.h_kernel, bytes);
                CK(cudaMemcpyAsync(P.d_kernel, (char *)g_pin_k.p + o, bytes, cudaMemcpyHostToDevice, g_stream));
            }
            o += bytes;
        }
    }
    // ---- candidates (api.cc:176-201)
    for (int64_t pi = 0; pi < n_problems; ++pi) {
        Problem &P = probs[pi];
        std::vector<std::pair<int, int>> tries; // (hard_dc passed to _solve, decompose_dc passed to _solve)
        if (!search_all)
            tries.push_back({hard_dc, decompose_dc});
        else {
            int _hard_dc = hard_dc < 0 ? 1000000000 : hard_dc;
            int max_dc = std::min(_hard_dc, (int)std::ceil(std::log2((float)P.n_in)));
            for (int d = -1; d <= max_dc; ++d)
                tries.push_back({_hard_dc, d});
        }
        // latency_allowed = hard_dc + minimal latency (api.cc:72) is only ever COMPARED with stage latencies (api.cc:117,133).
        // With search_all the reference passes hard_dc = 1e9 when the caller gave none: as long as every latency of the graph
        // stays far below that (input latencies < 1e6; an adder adds at most 64 and there are < 1e6 of them), no comparison
        // can come out differently whatever the minimal latency is, so its adder trees need not be built.
        bool latencies_small = true;
        for (float v : P.lat)
            latencies_small = latencies_small && std::isfinite(v) && std::fabs(v) < 1e6f;
        for (auto &tr : tries) {
            Candidate c;
            c.problem = (int)pi;
            c.method0 = method0_in;
            c.method1 = method1_in;
            c.hard_dc = tr.first;
            c.adder_size = adder_size;
            c.carry_size = carry_size;
            // api.cc:41-51
            if (c.method1 == "auto")
                c.method1 = (c.hard_dc >= 6 || ends_with(c.method0, "dc")) ? c.method0 : c.method0 + "-dc";
            if (c.hard_dc == 0 && !ends_with(c.method0, "dc"))
                c.method0 = c.method0 + "-dc";
            // api.cc:74-80
            int log2_n = (int)std::ceil(std::log2((float)P.n_in));
            c.decompose_dc = tr.second == -2 ? std::min(c.hard_dc, log2_n) : std::min({c.hard_dc, tr.second, log2_n});
            if (c.hard_dc >= 0 && !(c.hard_dc >= 100000000 && latencies_small))
                P.need_min_lat = true; // (see below: a delay bound of 1e9 can never bind)
            P.cand.push_back((int)cands.size());
            cands.push_back(std::move(c));
        }
    }
    // ---- decomposition scratch: one (m0, m1, mapping) triple per candidate
    Carver cp;
    struct POff {
        size_t m0, m1, map;
    };
    std::vector<POff> po(cands.size());
    for (size_t ci = 0; ci < cands.size(); ++ci) {
        Problem &P = probs[cands[ci].problem];
        po[ci].m0 = cp.take(sizeof(float) * (size_t)P.n_in * P.n_out);
        po[ci].m1 = cp.take(sizeof(float) * (size_t)P.n_out * P.n_out);
        po[ci].map = cp.take(sizeof(int) * 2 * (size_t)(P.n_out + 1));
    }
    g_pool.ensure(cp.off + sizeof(DecompJob) * cands.size() + 4096, false);
    for (size_t ci = 0; ci < cands.size(); ++ci) {
        char *b = (char *)g_pool.p;
        cands[ci].d_m0 = (float *)(b + po[ci].m0);
        cands[ci].d_m1 = (float *)(b + po[ci].m1);
        cands[ci].d_map = (int *)(b + po[ci].map);
    }
    DecompJob *d_djobs = (DecompJob *)((char *)g_pool.p + ((cp.off + 255) & ~size_t(255)));
    // centre + all-pairs distance once per problem (mat_decompose.cc:64-93)
    tm.begin();
    int n_l = 0;
    for (auto &P : probs) {
        const int n = P.n_out + 1;
        center_kernel<<<1, 256, 0, g_stream>>>(P.d_kernel, P.n_in, P.n_out, P.d_aug, P.d_s0, P.d_s1);
        long long tot = (long long)n * n;
        dist_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, g_stream>>>(P.d_aug, P.n_in, n, P.d_dist, P.d_sign);
        n_l += 2;
    }
    tm.end(n_l);
    CK(cudaGetLastError());

    // minimal_latency (api.cc:11-26, :68-72): to_solution of the un-optimised state
    std::vector<StageJob *> jobs;
    for (auto &P : probs) {
        if (!P.need_min_lat)
            continue;
        StageJob &j = P.min_lat_job;
        j.n_in = P.n_in;
        j.n_out = P.n_out;
        j.method = M_DUMMY;
        j.adder_size = adder_size;
        j.carry_size = carry_size;
        j.d_kernel = P.d_kernel;
        j.qint = P.qint;
        j.lat = P.lat;
        jobs.push_back(&j);
    }
    run_stage_jobs(jobs, tm, false);
    for (auto &P : probs)
        P.min_lat = P.need_min_lat ? stage_max_latency(P.min_lat_job.res) : 0.0f;
    for (auto &c : cands)
        if (c.hard_dc >= 0)
            c.latency_allowed = (float)c.hard_dc + probs[c.problem].min_lat; // api.cc:72

    // ---- rounds: every unfinished candidate contributes its next solve_single
    for (int round = 0; round < 4096; ++round) {
        // (re)decompose the candidates that need a stage-0 solve
        std::vector<int> dec;
        for (size_t ci = 0; ci < cands.size(); ++ci)
            if (cands[ci].phase == 0)
                dec.push_back((int)ci);
        bool any_left = !dec.empty();
        for (auto &c : cands)
            any_left = any_left || c.phase == 1;
        if (!any_left)
            break;
        if (!dec.empty()) {
            // api.cc:84-93: once decompose_dc < 0 under a finite hard_dc, both methods are forced
            for (int ci : dec) {
                Candidate &c = cands[ci];
                if (c.decompose_dc < 0 && c.hard_dc >= 0) {
                    if (c.method0 != "dummy") {
                        c.method0 = "wmc-dc";
                        c.method1 = "wmc-dc";
                    }
                    else {
                        c.method0 = "dummy";
                        c.method1 = "dummy";
                    }
                }
            }
            // group by problem: one launch per problem, one CTA per candidate
            std::vector<DecompJob> dj(cands.size());
            for (int ci : dec)
                dj[ci] = DecompJob{cands[ci].decompose_dc, cands[ci].d_m0, cands[ci].d_m1, cands[ci].d_map};
            static PinBuf pin_dj;
            pin_dj.ensure(sizeof(DecompJob) * cands.size());
            CK(cudaStreamSynchronize(g_stream));
            tm.begin();
            int nl = 0;
            size_t run0 = 0;
            // candidates of one problem are contiguous in `cands`
            std::vector<DecompJob> packed;
            for (auto &P : probs) {
                packed.clear();
                for (int ci : P.cand)
                    if (cands[ci].phase == 0)
                        packed.push_back(dj[ci]);
                if (packed.empty())
                    continue;
                memcpy((char *)pin_dj.p + sizeof(DecompJob) * run0, packed.data(), sizeof(DecompJob) * packed.size());
                CK(cudaMemcpyAsync(d_djobs + run0, (char *)pin_dj.p + sizeof(DecompJob) * run0, sizeof(DecompJob) * packed.size(), cudaMemcpyHostToDevice, g_stream));
                const int n = P.n_out + 1;
                const int threads = std::min(1024, std::max(64, (n + 31) / 32 * 32));
                const size_t smem = (size_t)n * 17 + 64;
                if (smem > 48 * 1024)
                    CK(cudaFuncSetAttribute(mst_build_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                mst_build_kernel<<<(unsigned)packed.size(), threads, smem, g_stream>>>(P.d_aug, P.d_dist, P.d_sign, P.d_s0, P.d_s1, P.n_in, P.n_out, d_djobs + run0);
                run0 += packed.size();
                ++nl;
            }
            tm.end(nl);
            CK(cudaGetLastError());
        }
        for (auto &c : cands) {
            Problem &P = probs[c.problem];
            if (c.phase == 0) {
                StageJob &j = c.job0;
                j = StageJob();
                j.n_in = P.n_in;
                j.n_out = P.n_out;
                j.method = parse_method(c.method0);
                j.adder_size = c.adder_size;
                j.carry_size = c.carry_size;
                j.d_kernel = c.d_m0;
                j.qint = P.qint;
                j.lat = P.lat;
            }
            else if (c.phase == 1) {
                StageJob &j = c.job1;
                j = StageJob();
                j.n_in = P.n_out;
                j.n_out = P.n_out;
                j.method = parse_method(c.method1);
                j.adder_size = c.adder_size;
                j.carry_size = c.carry_size;
                j.d_kernel = c.d_m1;
                j.cost_init = c.job0.res.cost_sum; // the float cost keeps accumulating across the two stages (api.cc:222-227)
                // api.cc:100-115: stage-1 inputs are the RAW op qint/latency of the stage-0 outputs
                const StageResult &r0 = c.job0.res;
                j.qint.resize(3 * (size_t)P.n_out);
                j.lat.resize(P.n_out);
                for (int k = 0; k < P.n_out; ++k) {
                    int64_t idx = r0.out_idxs[k];
                    if (idx >= 0) {
                        j.qint[3 * k + 0] = r0.out_q[k].x;
                        j.qint[3 * k + 1] = r0.out_q[k].y;
                        j.qint[3 * k + 2] = r0.out_q[k].z;
                        j.lat[k] = r0.out_q[k].w;
                    }
                    else {
                        j.qint[3 * k + 0] = 0.0f;
                        j.qint[3 * k + 1] = 0.0f;
                        j.qint[3 * k + 2] = std::numeric_limits<float>::infinity();
                        j.lat[k] = 0.0f;
                    }
                }
            }
        }
        // stage-0 and stage-1 jobs differ wildly in size: run them as separate launches; identical jobs are solved once
        for (int stage = 0; stage < 2; ++stage) {
            std::vector<int> idx;
            for (size_t ci = 0; ci < cands.size(); ++ci)
                if (cands[ci].phase == stage)
                    idx.push_back((int)ci);
            if (idx.empty())
                continue;
            std::vector<const float *> mats;
            std::vector<long long> words;
            std::vector<std::string> keys;
            for (int ci : idx) {
                const Candidate &c = cands[ci];
                const StageJob &j = stage == 0 ? c.job0 : c.job1;
                mats.push_back(j.d_kernel);
                words.push_back((long long)j.n_in * j.n_out);
                std::string k;
                auto put = [&](const void *p, size_t n) { k.append((const char *)p, n); };
                const int head[6] = {c.problem, j.n_in, j.n_out, j.method, j.adder_size, j.carry_size};
                put(head, sizeof(head));
                put(&j.cost_init, sizeof(float));
                put(j.qint.data(), sizeof(float) * j.qint.size());
                put(j.lat.data(), sizeof(float) * j.lat.size());
                keys.push_back(std::move(k));
            }
            const std::vector<int> rep = g_share_jobs ? identical_jobs(mats, words, keys, tm) : [&] {
                std::vector<int> r(idx.size());
                for (size_t i = 0; i < r.size(); ++i)
                    r[i] = (int)i;
                return r;
            }();
            std::vector<StageJob *> run;
            for (size_t i = 0; i < idx.size(); ++i)
                if (rep[i] == (int)i)
                    run.push_back(stage == 0 ? &cands[idx[i]].job0 : &cands[idx[i]].job1);
            jobs_total += (int64_t)idx.size();
            jobs_run += (int64_t)run.size();
            run_stage_jobs(run, tm, false);
            for (size_t i = 0; i < idx.size(); ++i)
                if (rep[i] != (int)i) { // (op tables stay on the device and are shared; the host-side vectors are copied)
                    if (stage == 0)
                        cands[idx[i]].job0.res = cands[idx[rep[i]]].job0.res;
                    else
                        cands[idx[i]].job1.res = cands[idx[rep[i]]].job1.res;
                }
        }
        for (auto &c : cands) {
            const bool both_wmc_dc = c.method0 == "wmc-dc" && c.method1 == "wmc-dc";
            if (c.phase == 0) {
                float max_lat0 = stage_max_latency(c.job0.res);
                if (max_lat0 > c.latency_allowed && (!both_wmc_dc || c.decompose_dc >= 0)) {
                    c.decompose_dc--; // api.cc:117-122
                    if (c.decompose_dc < -64)
                        throw ApiError(DA4ML_E_RUNTIME, "latency constraint cannot be met");
                    continue;
                }
                c.phase = 1;
            }
            else if (c.phase == 1) {
                float max_lat1 = stage_max_latency(c.job1.res);
                if (max_lat1 > c.latency_allowed && (!both_wmc_dc || c.decompose_dc >= 0)) {
                    c.decompose_dc--; // api.cc:133-138
                    if (c.decompose_dc < -64)
                        throw ApiError(DA4ML_E_RUNTIME, "latency constraint cannot be met");
                    c.phase = 0;
                    continue;
                }
                c.phase = 2;
            }
        }
    }
    // ---- argmin over candidates, first minimum wins (api.cc:243-249); cost summed in float in op order (api.cc:222-227)
    out.clear();
    for (auto &P : probs) {
        int best = -1;
        float best_cost = 0;
        for (int ci : P.cand) {
            Candidate &c = cands[ci];
            const float cost = c.job1.res.cost_sum; // stage-0 sum carried into stage 1 on the device
            if (best < 0 || cost < best_cost) {
                best = ci;
                best_cost = cost;
            }
        }
        fetch_ops(cands[best].job0.res); // only the winner's op tables leave the device
        fetch_ops(cands[best].job1.res);
        auto pl = std::make_unique<PipelineImpl>();
        pl->stages.push_back(std::move(cands[best].job0.res));
        pl->stages.push_back(std::move(cands[best].job1.res));
        out.push_back(std::move(pl));
    }
    for (auto &pl : out) {
        pl->device_ms = tm.device_ms;
        pl->launches = tm.launches;
        pl->solve_ms = tm.solve_ms;
        pl->solve_launches = tm.solve_launches;
        pl->algo_bytes = tm.algo_bytes;
        pl->jobs_total = jobs_total;
        pl->jobs_run = jobs_run;
        pl->retried_jobs = tm.retried_jobs;
    }
}

// small export kernels for the helper entry points ------------------------------------------------

} // namespace da
