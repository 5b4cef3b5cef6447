// cmvm_lib.cu -- host driver and C ABI (include/da4ml_b200_cmvm.h) of the B200-native CMVM solver.
//
// Host-side control mirrors the reference's api.cc: `solve` (candidate search over decompose_dc,
// api.cc:147-250) and `_solve` (two-stage driver with the latency-retry loop, api.cc:28-145).  The
// reference parallelises the candidates with OpenMP; here all pending solve_single jobs of all
// candidates (and of all problems of a batch) are solved concurrently by one persistent kernel
// launch per round.  All arithmetic of the path runs in the kernels of cmvm_kernels.cuh /
// cmvm_decompose.cuh; nothing here falls back to the CPU.
#include "host_dais.cuh"
#include "host_solve.cuh"

namespace da {

// small export kernels for the helper entry points ------------------------------------------------
__global__ void csd_export_kernel(const uint2 *masks, int n, int nbits, int8_t *csd) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n)
        return;
    uint2 m = masks[idx];
    for (int k = 0; k < nbits; ++k)
        csd[(size_t)idx * nbits + k] = (int8_t)(((m.x >> k) & 1) - ((m.y >> k) & 1));
}
// plain digits without centring: the matrix is interpreted as already integer (bit_decompose.cc:22-42)
__global__ void int_csd_kernel(const int *x, int n, int nbits, int8_t *csd) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n)
        return;
    int v = x[idx];
    for (int k = nbits - 1; k >= 0; --k) {
        int p2 = (int)(1u << k);
        int thres = (int)(((long long)p2 * 2) / 3);
        int d = (v > thres) - (v < -thres);
        csd[(size_t)idx * nbits + k] = (int8_t)d;
        v -= p2 * d;
    }
}
__global__ void int_absmax_kernel(const int *x, int n, int *out) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    int v = idx < n ? abs(x[idx]) : 0;
    for (int off = 16; off > 0; off >>= 1)
        v = max(v, __shfl_xor_sync(0xffffffffu, v, off));
    if ((threadIdx.x & 31) == 0 && v)
        atomicMax(out, v);
}
__global__ void float_to_int_kernel(const float *x, int n, int *out) {
    int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx < n)
        out[idx] = (int)x[idx];
}

} // namespace da

// ================================================================================================
using namespace da;

struct da4ml_pipeline {
    std::unique_ptr<PipelineImpl> impl;
};

// The every-op variant of a program (dais_compile with every_op) on the device: the profile variant is compiled once,
// lazily, and kept; a capture variant is compiled per call into the same kind of buffer, reused while it is big enough.
struct DaisVariant {
    DaisCompiled P;
    int tile = 0;
    long long chunk = 0;
    void *mem = nullptr; // instructions | side table | capture columns | totals [4][n_ops] | first-outside key
    size_t cap = 0;
    DaisInstr *d_prog = nullptr;
    DaisObsEntry *d_obs = nullptr;
    int32_t *d_cols = nullptr;
    long long *d_totals = nullptr;
    unsigned long long *d_first = nullptr;
    ~DaisVariant() {
        if (mem)
            cudaFree(mem);
    }
};

// A DAIS program compiled for the device and kept resident (host_dais.cuh, dais_exec.cuh).
struct da4ml_dais {
    DaisCompiled P;
    std::vector<int32_t> words; // the program, for the variants
    int device = -1;
    int tile = 0;           // samples per CTA in the shared regime; 0 = global regime
    long long chunk = 0;    // samples per launch
    long long budget = 0;   // shared memory a CTA's slot file may use, as fixed at load
    long long forced_chunk = 0;
    int optin = 0;
    bool has_lookup = false;
    void *mem = nullptr;    // instructions | tables | error word, v0 word
    DaisInstr *d_prog = nullptr;
    int32_t *d_tables = nullptr;
    unsigned long long *d_err = nullptr;
    long long *d_v0 = nullptr;
    std::unique_ptr<DaisVariant> profile, capture;
    ~da4ml_dais() {
        if (mem)
            cudaFree(mem);
    }
};

namespace {
long long g_dais_shared_budget = 0; // bytes of shared memory for one CTA's slot file; 0 = what the device allows
long long g_dais_chunk = 0;         // samples per launch; 0 = automatic
DevBuf g_dais_arena, g_dais_io, g_dais_rec;

// One compiled stream on the device: predict's, or a variant's.
struct DaisStream {
    const DaisCompiled &P;
    const DaisInstr *prog;
    int tile;
    const int32_t *tables;
};
DaisStream dais_stream(const da4ml_dais *h) { return {h->P, h->d_prog, h->tile, h->d_tables}; }
DaisStream dais_stream(const da4ml_dais *h, const DaisVariant &V) { return {V.P, V.d_prog, V.tile, h->d_tables}; }

template <class Obs = DaisNoObserver>
void dais_launch(const DaisStream &D, const double *x, double *y, long long n, long long sample0, unsigned long long *err, long long *err_v0, Obs obs = Obs()) {
    const DaisCompiled &P = D.P;
    const int n_instr = (int)P.prog.size();
    if (D.tile > 0) {
        const size_t smem = (size_t)8 * std::max(P.n_slots, 1) * D.tile;
        dais_exec_kernel<true, Obs><<<(unsigned)((n + D.tile - 1) / D.tile), D.tile, smem, g_stream>>>(D.prog, n_instr, x, P.n_in, y, P.n_out, n, nullptr, 0, D.tables, err, sample0, err_v0, obs);
    }
    else {
        // an observer runs whole warps, so the lanes past n need arena columns too
        const long long stride = Obs::kActive ? (n + 255) / 256 * 256 : n;
        g_dais_arena.ensure((size_t)8 * std::max(P.n_slots, 1) * std::max(stride, 1LL), false);
        dais_exec_kernel<false, Obs><<<(unsigned)((n + 255) / 256), 256, 0, g_stream>>>(D.prog, n_instr, x, P.n_in, y, P.n_out, n, (long long *)g_dais_arena.p, stride, D.tables, err, sample0, err_v0, obs);
    }
    CK(cudaGetLastError());
}

// After the launches of a call: raise the reference's message for the first (sample, op) whose lookup was out of range.
// That sample is run once more on its own to recover the operand.  `row(s)` is a device pointer to input row s.
template <class Row> void dais_check(const da4ml_dais *h, const DaisStream &D, Row row, double *y_scratch) {
    if (!h->has_lookup)
        return;
    unsigned long long key = 0;
    CK(cudaMemcpyAsync(&key, h->d_err, sizeof(key), cudaMemcpyDeviceToHost, g_stream));
    CK(cudaStreamSynchronize(g_stream));
    if (key == ~0ull)
        return;
    const unsigned long long n_instr = D.P.prog.size();
    const long long s = (long long)(key / n_instr);
    const int pc = (int)(key % n_instr);
    dais_launch(D, row(s), y_scratch, 1, 0, h->d_err + 1, h->d_v0);
    long long v0 = 0;
    CK(cudaMemcpyAsync(&v0, h->d_v0, sizeof(v0), cudaMemcpyDeviceToHost, g_stream));
    CK(cudaStreamSynchronize(g_stream));
    throw ApiError(DA4ML_E_RUNTIME, dais_lookup_message(D.P, pc, v0));
}

// Compiles the every-op variant of h's program into V (capturing ops[0..k), if any) and uploads it; V's buffer is
// reused while it is big enough.  A profile's launches are sized so that the per-warp records stay within 1 GB.
void dais_variant_build(const da4ml_dais *h, DaisVariant &V, const int32_t *ops, int k, bool profile) {
    try {
        V.P = dais_compile(h->words.data(), (long long)h->words.size(), true, ops, k);
    }
    catch (const std::runtime_error &e) {
        throw ApiError(DA4ML_E_INVALID, e.what());
    }
    const DaisCompiled &P = V.P;
    V.tile = dais_shared_tile(P.n_slots, h->budget);
    if (V.tile > 0) {
        V.chunk = 1LL << 24;
        CK(cudaFuncSetAttribute(dais_exec_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->optin));
        CK(cudaFuncSetAttribute(dais_exec_kernel<true, DaisProfileObserver>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->optin));
        CK(cudaFuncSetAttribute(dais_exec_kernel<true, DaisCaptureObserver>, cudaFuncAttributeMaxDynamicSharedMemorySize, h->optin));
    }
    else
        V.chunk = std::max<long long>(256, ((1LL << 31) / (8LL * std::max(P.n_slots, 1))) / 256 * 256);
    V.chunk = std::min<long long>(V.chunk, std::max<long long>(256, ((1LL << 28) / (8LL * std::max(1, P.n_in + k))) / 256 * 256));
    if (profile)
        V.chunk = dais_profile_chunk((long long)P.prog.size(), V.chunk, 1LL << 30);
    if (h->forced_chunk > 0)
        V.chunk = h->forced_chunk;
    Carver c;
    const size_t o_prog = c.take(sizeof(DaisInstr) * P.prog.size()), o_obs = c.take(sizeof(DaisObsEntry) * P.obs.size()), o_cols = c.take(sizeof(int32_t) * P.cap_cols.size()),
                 o_tot = c.take(sizeof(long long) * (4 * (size_t)P.n_ops + 1));
    if (c.off > V.cap) {
        if (V.mem)
            CK(cudaFree(V.mem));
        V.mem = nullptr;
        V.cap = 0;
        CK(cudaMalloc(&V.mem, c.off));
        V.cap = c.off;
    }
    char *b = (char *)V.mem;
    V.d_prog = (DaisInstr *)(b + o_prog);
    V.d_obs = (DaisObsEntry *)(b + o_obs);
    V.d_cols = (int32_t *)(b + o_cols);
    V.d_totals = (long long *)(b + o_tot);
    V.d_first = (unsigned long long *)(V.d_totals + 4 * (size_t)P.n_ops);
    if (!P.prog.empty()) {
        CK(cudaMemcpyAsync(V.d_prog, P.prog.data(), sizeof(DaisInstr) * P.prog.size(), cudaMemcpyHostToDevice, g_stream));
        CK(cudaMemcpyAsync(V.d_obs, P.obs.data(), sizeof(DaisObsEntry) * P.obs.size(), cudaMemcpyHostToDevice, g_stream));
    }
    if (!P.cap_cols.empty())
        CK(cudaMemcpyAsync(V.d_cols, P.cap_cols.data(), sizeof(int32_t) * P.cap_cols.size(), cudaMemcpyHostToDevice, g_stream));
}

// The profile of n > 0 samples into stats [4][n_ops] (min, max, outside, wrapped) and first {sample, op}.
// `stage(s0, m)` gives a device pointer to input rows [s0, s0 + m), valid until the next call; `row(s)` one row.
// Totals stay on the device across the launches and come back once.
template <class Stage, class Row> void dais_profile_run(da4ml_dais *h, long long n, Stage stage, Row row, int64_t *stats, int64_t *first) {
    if (!h->profile) {
        auto V = std::make_unique<DaisVariant>();
        dais_variant_build(h, *V, nullptr, 0, true);
        h->profile = std::move(V);
    }
    const DaisVariant &V = *h->profile;
    const DaisCompiled &P = V.P;
    const DaisStream D = dais_stream(h, V);
    const int n_instr = (int)P.prog.size();
    const size_t n_tot = 4 * (size_t)P.n_ops + 1;
    std::vector<long long> tot(n_tot, 0);
    std::fill(tot.begin(), tot.begin() + P.n_ops, (long long)0x7fffffffffffffffll);
    std::fill(tot.begin() + P.n_ops, tot.begin() + 2 * P.n_ops, (long long)0x8000000000000000ull);
    tot[n_tot - 1] = -1;
    CK(cudaMemcpyAsync(V.d_totals, tot.data(), sizeof(long long) * n_tot, cudaMemcpyHostToDevice, g_stream));
    CK(cudaMemsetAsync(h->d_err, 0xff, 2 * sizeof(unsigned long long), g_stream));
    const long long C = std::min<long long>(V.chunk, n);
    g_dais_rec.ensure((size_t)32 * std::max(n_instr, 1) * ((C + 31) / 32), false);
    for (long long s0 = 0; s0 < n; s0 += C) {
        const long long Sc = std::min<long long>(C, n - s0);
        const double *xs = stage(s0, Sc);
        DaisProfileObserver obs{};
        obs.side = V.d_obs, obs.rec = (long long *)g_dais_rec.p, obs.n_warps = (Sc + 31) / 32, obs.first = V.d_first, obs.n_ops = P.n_ops;
        dais_launch(D, xs, nullptr, Sc, s0, h->d_err, nullptr, obs);
        if (n_instr > 0) {
            dais_profile_merge_kernel<<<(unsigned)(((long long)n_instr * 32 + 255) / 256), 256, 0, g_stream>>>(obs.rec, n_instr, obs.n_warps, V.d_obs, V.d_totals, P.n_ops);
            CK(cudaGetLastError());
        }
        dais_check(h, D, row, nullptr);
    }
    CK(cudaMemcpyAsync(tot.data(), V.d_totals, sizeof(long long) * n_tot, cudaMemcpyDeviceToHost, g_stream));
    CK(cudaStreamSynchronize(g_stream));
    std::copy(tot.begin(), tot.end() - 1, stats);
    const unsigned long long key = (unsigned long long)tot[n_tot - 1];
    first[0] = key == ~0ull ? -1 : (int64_t)(key / (unsigned long long)P.n_ops);
    first[1] = key == ~0ull ? -1 : (int64_t)(key % (unsigned long long)P.n_ops);
}

// The values of ops[0..k) for n > 0 samples: `stage` / `row` as above; `dst(s0, m)` gives the device rows [s0, s0 + m)
// of the [n][k] int64 result, and `flush(s0, m)` is called once they are written.
template <class Stage, class Row, class Dst, class Flush>
void dais_capture_run(da4ml_dais *h, long long n, const int32_t *ops, int k, Stage stage, Row row, Dst dst, Flush flush) {
    if (!h->capture)
        h->capture = std::make_unique<DaisVariant>();
    DaisVariant &V = *h->capture;
    dais_variant_build(h, V, ops, k, false);
    const DaisStream D = dais_stream(h, V);
    CK(cudaMemsetAsync(h->d_err, 0xff, 2 * sizeof(unsigned long long), g_stream));
    for (long long s0 = 0; s0 < n; s0 += V.chunk) {
        const long long Sc = std::min<long long>(V.chunk, n - s0);
        const double *xs = stage(s0, Sc); // (before dst: the host path carves both from one staging buffer)
        DaisCaptureObserver obs{};
        obs.side = V.d_obs, obs.cols = V.d_cols, obs.out = dst(s0, Sc), obs.k = k;
        dais_launch(D, xs, nullptr, Sc, s0, h->d_err, nullptr, obs);
        dais_check(h, D, row, nullptr);
        flush(s0, Sc);
    }
}

// The op list of a capture call, checked before any device call.
void dais_check_ops(const da4ml_dais *h, const int32_t *ops, int k) {
    for (int j = 0; j < k; ++j)
        if (ops[j] < 0 || ops[j] >= h->P.n_ops)
            throw ApiError(DA4ML_E_INVALID, "op index " + std::to_string(ops[j]) + " out of range [0, " + std::to_string(h->P.n_ops) + ")");
}

void dais_check_device(const da4ml_dais *h) {
    int dev = 0;
    CK(cudaGetDevice(&dev));
    if (dev != h->device)
        throw ApiError(DA4ML_E_INVALID, "the DAIS program was loaded on CUDA device " + std::to_string(h->device) + ", the current device is " + std::to_string(dev));
}
} // namespace

template <class F> static int guarded(F &&f) {
    try {
        std::lock_guard<std::mutex> lock(g_mutex);
        f();
        return DA4ML_OK;
    }
    catch (const ApiError &e) {
        g_err = e.what();
        return e.code;
    }
    catch (const std::exception &e) {
        g_err = e.what();
        return DA4ML_E_RUNTIME;
    }
}

extern "C" {

const char *da4ml_cmvm_last_error(void) { return g_err.c_str(); }

int da4ml_cmvm_device_info(int32_t out[5]) {
    out[0] = 1;
    out[1] = out[2] = out[3] = out[4] = 0;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess) {
        cudaGetLastError();
        return DA4ML_OK;
    }
    out[1] = ndev;
    if (ndev > 0) {
        int dev = 0;
        cudaDeviceProp prop;
        if (cudaGetDevice(&dev) == cudaSuccess && cudaGetDeviceProperties(&prop, dev) == cudaSuccess) {
            out[2] = prop.multiProcessorCount;
            out[3] = prop.major;
            out[4] = prop.minor;
        }
    }
    return DA4ML_OK;
}

int da4ml_cmvm_plan(const int64_t *jobs, int64_t n_jobs, int coop, int group_override, int64_t out[12]) {
    return guarded([&]() -> int {
        if (!jobs || !out || n_jobs <= 0 || coop <= 0)
            throw ApiError(DA4ML_E_INVALID, "da4ml_cmvm_plan: bad arguments");
        std::vector<PlanJob> pj((size_t)n_jobs);
        for (int64_t i = 0; i < n_jobs; ++i) {
            const int64_t *r = jobs + 8 * i;
            if (r[0] <= 0 || r[1] <= 0 || r[2] <= 0 || r[6] <= 0 || r[7] <= 0)
                throw ApiError(DA4ML_E_INVALID, "da4ml_cmvm_plan: bad job row");
            pj[i].n_in = (int)r[0];
            pj[i].n_out = (int)r[1];
            pj[i].nbits = (int)r[2];
            pj[i].d0 = r[3];
            pj[i].dcol_max = (int)r[4];
            pj[i].col_cap = (int)r[5];
            pj[i].f_mul = (int)r[6];
            pj[i].list_mul = (int)r[7];
            pj[i].e_cap = (int)(r[0] + std::min<long long>(r[3], r[3] / 2 + 1024) + 1); // as run_stage_jobs sizes it
        }
        PlanEnv env;
        env.coop = coop;
        env.group_override = group_override;
        std::copy(g_first_caps, g_first_caps + CAP_WORDS, env.caps); // (the first attempt's plan)
        const LaunchPlan P = plan_launch(pj, env);
        out[0] = P.cfg.G;
        out[1] = P.n_groups;
        out[2] = P.cfg.cpc;
        out[3] = P.lcap;
        out[4] = P.cfg.chunk_log;
        out[5] = P.cfg.nchunk_cap;
        out[6] = P.max_fcap;
        out[7] = P.hlog;
        out[8] = (int64_t)P.smem_bytes;
        out[9] = env.own_budget;
        out[10] = P.narrow;
        out[11] = P.ovf_cap;
        return DA4ML_OK;
    });
}

int da4ml_cmvm_set_stream(void *s) {
    g_stream = (cudaStream_t)s;
    return DA4ML_OK;
}
int da4ml_cmvm_set_group_size(int g) {
    g_group_override = g;
    return DA4ML_OK;
}
// Free every device / pinned buffer the library keeps between calls (they are re-grown on demand).
int da4ml_cmvm_release(void) {
    return guarded([&] {
        release_device_buffers();
        for (PinBuf *b : {&g_pin_up, &g_pin_down}) {
            if (b->p)
                cudaFreeHost(b->p);
            b->p = nullptr;
            b->cap = 0;
        }
    });
}
int da4ml_cmvm_set_job_sharing(int on) {
    g_share_jobs = on != 0;
    return DA4ML_OK;
}
int da4ml_cmvm_set_accounting(int on) {
    g_accounting = on;
    return DA4ML_OK;
}
int da4ml_cmvm_set_first_attempt_caps(const int64_t caps[6]) {
    return guarded([&] {
        if (!caps)
            throw ApiError(DA4ML_E_INVALID, "da4ml_cmvm_set_first_attempt_caps: null caps");
        for (int k = 0; k < CAP_WORDS; ++k)
            if (caps[k] < 0 || caps[k] > INT32_MAX)
                throw ApiError(DA4ML_E_INVALID, "da4ml_cmvm_set_first_attempt_caps: capacity " + std::to_string(k) + " out of range");
        if (caps[CAP_HLOG] != 0 && (caps[CAP_HLOG] < HLOG_MIN || caps[CAP_HLOG] > HLOG_MAX))
            throw ApiError(DA4ML_E_INVALID, "da4ml_cmvm_set_first_attempt_caps: log2_pair_counters must be 0 or " + std::to_string(HLOG_MIN) + ".." +
                                                std::to_string(HLOG_MAX));
        std::copy(caps, caps + CAP_WORDS, g_first_caps);
    });
}

int da4ml_cmvm_solve_batch(
    int64_t n_problems, const float *const *kernels, const int64_t *n_in, const int64_t *n_out, const char *method0,
    const char *method1, int hard_dc, int decompose_dc, const float *const *qintervals, const float *const *latencies,
    int adder_size, int carry_size, int search_all, da4ml_pipeline_t **out
) {
    return guarded([&] {
        if (n_problems <= 0 || !kernels || !n_in || !n_out || !out || !method0 || !method1)
            throw ApiError(DA4ML_E_INVALID, "invalid argument");
        std::vector<std::unique_ptr<PipelineImpl>> res;
        solve_many(n_problems, kernels, n_in, n_out, method0, method1, hard_dc, decompose_dc, qintervals, latencies, adder_size, carry_size, search_all != 0, res);
        for (int64_t i = 0; i < n_problems; ++i) {
            out[i] = new da4ml_pipeline();
            out[i]->impl = std::move(res[i]);
        }
    });
}

int da4ml_cmvm_solve_batch_device(
    int64_t n_problems, const float *const *kernels_dev, const int64_t *n_in, const int64_t *n_out, const char *method0,
    const char *method1, int hard_dc, int decompose_dc, const float *const *qintervals, const float *const *latencies,
    int adder_size, int carry_size, int search_all, da4ml_pipeline_t **out
) {
    return guarded([&] {
        if (n_problems <= 0 || !kernels_dev || !n_in || !n_out || !out || !method0 || !method1)
            throw ApiError(DA4ML_E_INVALID, "invalid argument");
        std::vector<std::unique_ptr<PipelineImpl>> res;
        solve_many(n_problems, kernels_dev, n_in, n_out, method0, method1, hard_dc, decompose_dc, qintervals, latencies, adder_size, carry_size, search_all != 0, res, true);
        for (int64_t i = 0; i < n_problems; ++i) {
            out[i] = new da4ml_pipeline();
            out[i]->impl = std::move(res[i]);
        }
    });
}

int da4ml_cmvm_solve(
    const float *kernel, int64_t n_in, int64_t n_out, const char *method0, const char *method1, int hard_dc, int decompose_dc,
    const float *qintervals, const float *latencies, int adder_size, int carry_size, int search_all, da4ml_pipeline_t **out
) {
    const float *ks[1] = {kernel};
    const float *qs[1] = {qintervals};
    const float *ls[1] = {latencies};
    return da4ml_cmvm_solve_batch(1, ks, &n_in, &n_out, method0, method1, hard_dc, decompose_dc, qs, ls, adder_size, carry_size, search_all, out);
}

int da4ml_cmvm_solve_single(
    const float *kernel, int64_t n_in, int64_t n_out, const char *method, const float *qintervals, const float *latencies,
    int adder_size, int carry_size, int32_t *trace, int64_t trace_cap, da4ml_pipeline_t **out
) {
    return guarded([&] {
        if (!kernel || n_in <= 0 || n_out <= 0 || !method || !out)
            throw ApiError(DA4ML_E_INVALID, "invalid argument");
        init_device();
        static DevBuf kbuf;
        static PinBuf kpin;
        size_t bytes = sizeof(float) * (size_t)n_in * n_out;
        kbuf.ensure(bytes, false);
        kpin.ensure(bytes);
        memcpy(kpin.p, kernel, bytes);
        CK(cudaMemcpyAsync(kbuf.p, kpin.p, bytes, cudaMemcpyHostToDevice, g_stream));
        StageJob j;
        j.n_in = (int)n_in;
        j.n_out = (int)n_out;
        j.method = parse_method(method);
        j.adder_size = adder_size;
        j.carry_size = carry_size;
        j.d_kernel = (const float *)kbuf.p;
        j.qint.resize(3 * (size_t)n_in);
        j.lat.resize(n_in);
        for (int64_t i = 0; i < n_in; ++i) { // cmvm_core.cc:18-32 defaults
            j.qint[3 * i + 0] = qintervals ? qintervals[3 * i + 0] : -128.0f;
            j.qint[3 * i + 1] = qintervals ? qintervals[3 * i + 1] : 127.0f;
            j.qint[3 * i + 2] = qintervals ? qintervals[3 * i + 2] : 1.0f;
            j.lat[i] = latencies ? latencies[i] : 0.0f;
        }
        j.trace = trace;
        j.trace_cap = trace ? trace_cap : 0;
        Timing tm;
        std::vector<StageJob *> jobs{&j};
        g_out_arena2.reset();
        run_stage_jobs(jobs, tm, true);
        auto pl = std::make_unique<PipelineImpl>();
        pl->stages.push_back(std::move(j.res));
        pl->device_ms = tm.device_ms;
        pl->launches = tm.launches;
        pl->solve_ms = tm.solve_ms;
        pl->solve_launches = tm.solve_launches;
        pl->algo_bytes = tm.algo_bytes;
        pl->retried_jobs = tm.retried_jobs;
        *out = new da4ml_pipeline();
        (*out)->impl = std::move(pl);
    });
}

void da4ml_pipeline_free(da4ml_pipeline_t *p) { delete p; }
int64_t da4ml_pipeline_n_stages(const da4ml_pipeline_t *p) { return p ? (int64_t)p->impl->stages.size() : 0; }
int da4ml_pipeline_stage_meta(const da4ml_pipeline_t *p, int64_t s, int64_t meta[5]) {
    if (!p || s < 0 || s >= (int64_t)p->impl->stages.size())
        return DA4ML_E_INVALID;
    const StageResult &r = p->impl->stages[s];
    meta[0] = r.n_in;
    meta[1] = r.n_out;
    meta[2] = r.n_ops();
    meta[3] = r.carry_size;
    meta[4] = r.adder_size;
    return DA4ML_OK;
}
int da4ml_pipeline_stage_copy(
    const da4ml_pipeline_t *p, int64_t s, int64_t *inp_shifts, int64_t *out_idxs, int64_t *out_shifts, int64_t *out_negs,
    int64_t *ops_i, float *ops_f
) {
    if (!p || s < 0 || s >= (int64_t)p->impl->stages.size())
        return DA4ML_E_INVALID;
    const StageResult &r = p->impl->stages[s];
    if (inp_shifts)
        std::copy(r.inp_shifts.begin(), r.inp_shifts.end(), inp_shifts);
    if (out_idxs)
        std::copy(r.out_idxs.begin(), r.out_idxs.end(), out_idxs);
    if (out_shifts)
        std::copy(r.out_shifts.begin(), r.out_shifts.end(), out_shifts);
    if (out_negs)
        std::copy(r.out_negs.begin(), r.out_negs.end(), out_negs);
    const size_t n_ops = r.op_misc.size();
    if (ops_i)
        for (size_t k = 0; k < n_ops; ++k) {
            ops_i[4 * k + 0] = r.op_misc[k].x;
            ops_i[4 * k + 1] = r.op_misc[k].y;
            ops_i[4 * k + 2] = r.op_misc[k].z;
            ops_i[4 * k + 3] = r.op_misc[k].w;
        }
    if (ops_f)
        for (size_t k = 0; k < n_ops; ++k) {
            ops_f[5 * k + 0] = r.op_q[k].x;
            ops_f[5 * k + 1] = r.op_q[k].y;
            ops_f[5 * k + 2] = r.op_q[k].z;
            ops_f[5 * k + 3] = r.op_q[k].w;
            ops_f[5 * k + 4] = r.op_cost[k];
        }
    return DA4ML_OK;
}
int da4ml_pipeline_stage_counters(const da4ml_pipeline_t *p, int64_t s, int64_t counters[32]) {
    if (!p || s < 0 || s >= (int64_t)p->impl->stages.size())
        return DA4ML_E_INVALID;
    std::copy(p->impl->stages[s].counters, p->impl->stages[s].counters + 32, counters);
    return DA4ML_OK;
}
int da4ml_pipeline_stage_milestones(const da4ml_pipeline_t *p, int64_t s, int64_t out[63]) {
    if (!p || s < 0 || s >= (int64_t)p->impl->stages.size())
        return DA4ML_E_INVALID;
    std::copy(p->impl->stages[s].counters + META_MILESTONES, p->impl->stages[s].counters + META_MILESTONES + 63, out);
    return DA4ML_OK;
}
int da4ml_pipeline_stage_words(const da4ml_pipeline_t *p, int64_t s, int64_t out[96]) {
    if (!p || s < 0 || s >= (int64_t)p->impl->stages.size())
        return DA4ML_E_INVALID;
    std::copy(p->impl->stages[s].counters, p->impl->stages[s].counters + META_WORDS, out);
    return DA4ML_OK;
}
double da4ml_pipeline_device_ms(const da4ml_pipeline_t *p) { return p ? p->impl->device_ms : 0.0; }
int64_t da4ml_pipeline_launches(const da4ml_pipeline_t *p) { return p ? p->impl->launches : 0; }
int da4ml_pipeline_profile(const da4ml_pipeline_t *p, double out[8]) {
    if (!p)
        return DA4ML_E_INVALID;
    out[0] = p->impl->device_ms;
    out[1] = (double)p->impl->launches;
    out[2] = p->impl->solve_ms;
    out[3] = (double)p->impl->solve_launches;
    out[4] = p->impl->algo_bytes;
    out[5] = (double)p->impl->jobs_total;
    out[6] = (double)p->impl->jobs_run;
    out[7] = (double)p->impl->retried_jobs;
    return DA4ML_OK;
}

// ---- helpers -------------------------------------------------------------------------------------
int da4ml_cmvm_csd_decompose(const float *kernel, int64_t n_in, int64_t n_out, int center, int8_t *csd, int8_t *shift0, int8_t *shift1, int64_t *n_bits) {
    return guarded([&] {
        if (!kernel || n_in <= 0 || n_out <= 0 || !csd || !shift0 || !shift1 || !n_bits)
            throw ApiError(DA4ML_E_INVALID, "csd_decompose only supports 2D arrays."); // bit_decompose.cc:48
        init_device();
        const size_t ne = (size_t)n_in * n_out;
        static DevBuf buf;
        Carver c;
        size_t ok = c.take(sizeof(float) * ne), oq = c.take(sizeof(float) * 3 * n_in), ol = c.take(sizeof(float) * n_in), om = c.take(sizeof(uint2) * ne),
               os0 = c.take(n_in), os1 = c.take(n_out), ocd = c.take(sizeof(int) * n_out), opm = c.take(sizeof(int) * PM_WORDS), od = c.take(sizeof(ProblemDesc)),
               ocsd = c.take(ne * 32), oint = c.take(sizeof(int) * (ne + 1));
        buf.ensure(c.off, false);
        char *b = (char *)buf.p;
        CK(cudaMemcpyAsync(b + ok, kernel, sizeof(float) * ne, cudaMemcpyHostToDevice, g_stream));
        int nbits = 0;
        if (center) {
            std::vector<float> q(3 * (size_t)n_in, 1.0f); // non-zero ranges: no row is blanked
            CK(cudaMemcpyAsync(b + oq, q.data(), sizeof(float) * 3 * n_in, cudaMemcpyHostToDevice, g_stream));
            ProblemDesc d;
            memset(&d, 0, sizeof(d));
            d.n_in = (int)n_in;
            d.n_out = (int)n_out;
            d.kernel = (const float *)(b + ok);
            d.qint = (const float *)(b + oq);
            d.lat = (const float *)(b + ol);
            d.masks0 = (uint2 *)(b + om);
            d.shift0 = (int8_t *)(b + os0);
            d.shift1 = (int8_t *)(b + os1);
            d.col_digits = (int *)(b + ocd);
            d.prep_meta = (int *)(b + opm);
            CK(cudaMemcpyAsync(b + od, &d, sizeof(d), cudaMemcpyHostToDevice, g_stream));
            cmvm_prep_kernel<<<1, 256, 0, g_stream>>>((ProblemDesc *)(b + od));
            CK(cudaGetLastError());
            int pm[PM_WORDS];
            CK(cudaMemcpyAsync(pm, b + opm, sizeof(pm), cudaMemcpyDeviceToHost, g_stream));
            CK(cudaStreamSynchronize(g_stream));
            nbits = pm[PM_NBITS];
            csd_export_kernel<<<(unsigned)((ne + 255) / 256), 256, 0, g_stream>>>((const uint2 *)(b + om), (int)ne, nbits, (int8_t *)(b + ocsd));
            CK(cudaMemcpyAsync(shift0, b + os0, n_in, cudaMemcpyDeviceToHost, g_stream));
            CK(cudaMemcpyAsync(shift1, b + os1, n_out, cudaMemcpyDeviceToHost, g_stream));
        }
        else {
            int *xi = (int *)(b + oint);
            float_to_int_kernel<<<(unsigned)((ne + 255) / 256), 256, 0, g_stream>>>((const float *)(b + ok), (int)ne, xi);
            CK(cudaMemsetAsync(xi + ne, 0, sizeof(int), g_stream));
            int_absmax_kernel<<<(unsigned)((ne + 255) / 256), 256, 0, g_stream>>>(xi, (int)ne, xi + ne);
            int mx = 0;
            CK(cudaMemcpyAsync(&mx, xi + ne, sizeof(int), cudaMemcpyDeviceToHost, g_stream));
            CK(cudaStreamSynchronize(g_stream));
            nbits = std::max(1, ceil_log2_pos((double)std::max((float)mx, 1.0f) * 1.5));
            int_csd_kernel<<<(unsigned)((ne + 255) / 256), 256, 0, g_stream>>>(xi, (int)ne, nbits, (int8_t *)(b + ocsd));
            memset(shift0, 0, n_in);
            memset(shift1, 0, n_out);
        }
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(csd, b + ocsd, ne * nbits, cudaMemcpyDeviceToHost, g_stream));
        CK(cudaStreamSynchronize(g_stream));
        *n_bits = nbits;
    });
}

int da4ml_cmvm_int_arr_to_csd(const int32_t *x, int64_t n, int8_t *csd, int64_t *n_bits) {
    return guarded([&] {
        if (!x || n <= 0 || !csd || !n_bits)
            throw ApiError(DA4ML_E_INVALID, "invalid argument");
        init_device();
        static DevBuf buf;
        Carver c;
        size_t ox = c.take(sizeof(int) * (n + 1)), oc = c.take((size_t)n * 32);
        buf.ensure(c.off, false);
        char *b = (char *)buf.p;
        int *xi = (int *)(b + ox);
        CK(cudaMemcpyAsync(xi, x, sizeof(int) * n, cudaMemcpyHostToDevice, g_stream));
        CK(cudaMemsetAsync(xi + n, 0, sizeof(int), g_stream));
        int_absmax_kernel<<<(unsigned)((n + 255) / 256), 256, 0, g_stream>>>(xi, (int)n, xi + n);
        int mx = 0;
        CK(cudaMemcpyAsync(&mx, xi + n, sizeof(int), cudaMemcpyDeviceToHost, g_stream));
        CK(cudaStreamSynchronize(g_stream));
        int nbits = std::max(1, ceil_log2_pos((double)std::max((float)mx, 1.0f) * 1.5));
        int_csd_kernel<<<(unsigned)((n + 255) / 256), 256, 0, g_stream>>>(xi, (int)n, nbits, (int8_t *)(b + oc));
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(csd, b + oc, (size_t)n * nbits, cudaMemcpyDeviceToHost, g_stream));
        CK(cudaStreamSynchronize(g_stream));
        *n_bits = nbits;
    });
}

int da4ml_cmvm_kernel_decompose(const float *kernel, int64_t n_in, int64_t n_out, int dc, float *m0, float *m1) {
    return guarded([&] {
        if (!kernel || n_in <= 0 || n_out <= 0 || !m0 || !m1)
            throw ApiError(DA4ML_E_INVALID, "csd_decompose only supports 2D arrays.");
        init_device();
        const size_t n = (size_t)n_out + 1;
        static DevBuf buf;
        Carver c;
        size_t ok = c.take(sizeof(float) * n_in * n_out), oa = c.take(sizeof(float) * n_in * n), od = c.take(sizeof(int) * n * n), os = c.take(n * n), os0 = c.take(n_in),
               os1 = c.take(n_out), om0 = c.take(sizeof(float) * n_in * n_out), om1 = c.take(sizeof(float) * n_out * n_out), omap = c.take(sizeof(int) * 2 * n), oj = c.take(sizeof(DecompJob));
        buf.ensure(c.off, false);
        char *b = (char *)buf.p;
        CK(cudaMemcpyAsync(b + ok, kernel, sizeof(float) * n_in * n_out, cudaMemcpyHostToDevice, g_stream));
        center_kernel<<<1, 256, 0, g_stream>>>((const float *)(b + ok), (int)n_in, (int)n_out, (float *)(b + oa), (int8_t *)(b + os0), (int8_t *)(b + os1));
        long long tot = (long long)n * n;
        dist_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, g_stream>>>((const float *)(b + oa), (int)n_in, (int)n, (int *)(b + od), (int8_t *)(b + os));
        DecompJob j{dc, (float *)(b + om0), (float *)(b + om1), (int *)(b + omap)};
        CK(cudaMemcpyAsync(b + oj, &j, sizeof(j), cudaMemcpyHostToDevice, g_stream));
        const int threads = std::min(1024, std::max(64, (int)((n + 31) / 32 * 32)));
        const size_t smem = n * 17 + 64;
        if (smem > 48 * 1024)
            CK(cudaFuncSetAttribute(mst_build_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        mst_build_kernel<<<1, threads, smem, g_stream>>>((const float *)(b + oa), (const int *)(b + od), (const int8_t *)(b + os), (const int8_t *)(b + os0), (const int8_t *)(b + os1), (int)n_in, (int)n_out, (const DecompJob *)(b + oj));
        CK(cudaGetLastError());
        CK(cudaMemcpyAsync(m0, b + om0, sizeof(float) * n_in * n_out, cudaMemcpyDeviceToHost, g_stream));
        CK(cudaMemcpyAsync(m1, b + om1, sizeof(float) * n_out * n_out, cudaMemcpyDeviceToHost, g_stream));
        CK(cudaStreamSynchronize(g_stream));
    });
}

// ---- DAIS program replay (reference dais/bindings.cc `run_interp`), opcodes -1/0/1 -------------------------------
int da4ml_dais_run(const int32_t *program, int64_t n_words, const double *inputs, int64_t n_samples, double *outputs) {
    return guarded([&] {
        if (!program || n_words < 6 || !inputs || !outputs || n_samples < 0)
            throw ApiError(DA4ML_E_RUNTIME, "Binary data too small to contain valid DAIS model file"); // DAISInterpreter.cc:11-15
        if (program[0] != 1)
            throw ApiError(DA4ML_E_RUNTIME, "DAIS version mismatch: expected version 1, got version " + std::to_string(program[0]));
        const int n_in = program[2], n_out = program[3], n_ops = program[4], n_tables = program[5];
        if (n_in < 0 || n_out < 0 || n_ops < 0)
            throw ApiError(DA4ML_E_RUNTIME, "Binary data header holds a negative count");
        if (n_tables != 0 || n_words != 6 + (int64_t)n_in + 3LL * n_out + 8LL * n_ops)
            throw ApiError(DA4ML_E_RUNTIME, "Binary data size mismatch (lookup tables are not produced by the CMVM path)");
        if (n_samples == 0)
            return;
        init_device();
        const int32_t *inp_shifts = program + 6, *out_idxs = inp_shifts + n_in, *out_shifts = out_idxs + n_out, *out_negs = out_shifts + n_out;
        const DaisOp *hops = reinterpret_cast<const DaisOp *>(out_negs + n_out);
        for (int i = 0; i < n_out; ++i) // (the reference interpreter indexes its buffer unchecked; a foreign file must not fault the device)
            if (out_idxs[i] < -1 || out_idxs[i] >= n_ops)
                throw ApiError(DA4ML_E_RUNTIME, "output index out of range at output " + std::to_string(i));
        for (int i = 0; i < n_in; ++i)
            if (inp_shifts[i] < -1023 || inp_shifts[i] > 1023)
                throw ApiError(DA4ML_E_RUNTIME, "input shift out of range at input " + std::to_string(i));
        for (int i = 0; i < n_out; ++i)
            if (out_shifts[i] < -1023 || out_shifts[i] > 1023)
                throw ApiError(DA4ML_E_RUNTIME, "output shift out of range at output " + std::to_string(i));
        // causality + supported opcodes (DAISInterpreter::validate), levels
        std::vector<int> level(n_ops, 0);
        int n_levels = 1;
        for (int i = 0; i < n_ops; ++i) {
            const DaisOp &op = hops[i];
            if (op.opcode == -1) {
                if (op.id0 < 0 || op.id0 >= n_in)
                    throw ApiError(DA4ML_E_RUNTIME, "input index out of range at operation " + std::to_string(i));
                continue;
            }
            if (op.opcode != 0 && op.opcode != 1)
                throw ApiError(DA4ML_E_RUNTIME, "Unknown opcode: " + std::to_string(op.opcode) + " at index " + std::to_string(i) + " (only adder graphs are replayed on this path)");
            if (op.id0 < 0 || op.id0 >= i || op.id1 < 0 || op.id1 >= i)
                throw ApiError(DA4ML_E_RUNTIME, "Operation " + std::to_string(i) + " violating causality");
            level[i] = 1 + std::max(level[op.id0], level[op.id1]);
            n_levels = std::max(n_levels, level[i] + 1);
        }
        std::vector<int> lvl_begin(n_levels + 1, 0), order(n_ops);
        for (int i = 0; i < n_ops; ++i)
            lvl_begin[level[i] + 1]++;
        for (int l = 0; l < n_levels; ++l)
            lvl_begin[l + 1] += lvl_begin[l];
        {
            std::vector<int> fill(lvl_begin.begin(), lvl_begin.end() - 1);
            for (int i = 0; i < n_ops; ++i)
                order[fill[level[i]]++] = i;
        }
        // samples per chunk: keep the [n_ops][S] int64 buffer around 1 GB
        const long long S_max = std::max<long long>(256, (1LL << 27) / std::max(1, n_ops));
        const long long S = std::min<long long>(n_samples, S_max);
        static DevBuf buf;
        Carver c;
        size_t o_ops = c.take(sizeof(DaisOp) * n_ops), o_ord = c.take(sizeof(int) * n_ops), o_hdr = c.take(sizeof(int) * (n_in + 3 * n_out)),
               o_in = c.take(sizeof(double) * S * n_in), o_out = c.take(sizeof(double) * S * n_out), o_buf = c.take(sizeof(long long) * S * n_ops);
        buf.ensure(c.off, false);
        char *b = (char *)buf.p;
        CK(cudaMemcpyAsync(b + o_ops, hops, sizeof(DaisOp) * n_ops, cudaMemcpyHostToDevice, g_stream));
        CK(cudaMemcpyAsync(b + o_ord, order.data(), sizeof(int) * n_ops, cudaMemcpyHostToDevice, g_stream));
        CK(cudaMemcpyAsync(b + o_hdr, inp_shifts, sizeof(int) * (n_in + 3 * n_out), cudaMemcpyHostToDevice, g_stream));
        const int *d_inp_shifts = (const int *)(b + o_hdr), *d_out_idxs = d_inp_shifts + n_in, *d_out_shifts = d_out_idxs + n_out, *d_out_negs = d_out_shifts + n_out;
        for (int64_t s0 = 0; s0 < n_samples; s0 += S) {
            const long long Sc = std::min<long long>(S, n_samples - s0);
            CK(cudaMemcpyAsync(b + o_in, inputs + s0 * n_in, sizeof(double) * Sc * n_in, cudaMemcpyHostToDevice, g_stream));
            for (int l = 0; l < n_levels; ++l) {
                const int n_l = lvl_begin[l + 1] - lvl_begin[l];
                if (!n_l)
                    continue;
                const long long threads = (long long)n_l * Sc;
                dais_level_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, g_stream>>>((const DaisOp *)(b + o_ops), (const int *)(b + o_ord) + lvl_begin[l], n_l, d_inp_shifts, (const double *)(b + o_in), n_in, Sc, (long long *)(b + o_buf));
            }
            const long long threads = (long long)n_out * Sc;
            dais_output_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, g_stream>>>((const DaisOp *)(b + o_ops), d_out_idxs, d_out_shifts, d_out_negs, n_out, Sc, (const long long *)(b + o_buf), (double *)(b + o_out));
            CK(cudaGetLastError());
            CK(cudaMemcpyAsync(outputs + s0 * n_out, b + o_out, sizeof(double) * Sc * n_out, cudaMemcpyDeviceToHost, g_stream));
            CK(cudaStreamSynchronize(g_stream));
        }
    });
}

// ---- complete DAIS interpreter: programs loaded once and kept on the device -----------------------------------------
int da4ml_dais_set_shared_budget(int64_t shared_bytes, int64_t chunk_samples) {
    g_dais_shared_budget = std::max<int64_t>(shared_bytes, 0);
    g_dais_chunk = std::max<int64_t>(chunk_samples, 0);
    return DA4ML_OK;
}

int da4ml_dais_load(const int32_t *program, int64_t n_words, da4ml_dais_t **out) {
    return guarded([&] {
        if (!out)
            throw ApiError(DA4ML_E_INVALID, "invalid argument");
        auto h = std::make_unique<da4ml_dais>();
        try {
            h->P = dais_compile(program, n_words);
        }
        catch (const std::runtime_error &e) {
            throw ApiError(DA4ML_E_RUNTIME, e.what());
        }
        init_device();
        h->device = g_device;
        h->words.assign(program, program + n_words);
        const DaisCompiled &P = h->P;
        for (const DaisInstr &I : P.prog)
            h->has_lookup |= I.kind == DK_LOOKUP;
        int optin = 0;
        CK(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, g_device));
        const long long budget = g_dais_shared_budget > 0 ? std::min<long long>(g_dais_shared_budget, optin) : optin;
        h->budget = budget;
        h->forced_chunk = g_dais_chunk;
        h->optin = optin;
        h->tile = dais_shared_tile(P.n_slots, budget);
        if (h->tile > 0) {
            CK(cudaFuncSetAttribute(dais_exec_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
            h->chunk = 1LL << 24; // (bounds the staging buffers of host arrays)
        }
        else
            h->chunk = std::max<long long>(256, ((1LL << 31) / (8LL * P.n_slots)) / 256 * 256); // a 2 GB slot arena
        h->chunk = std::min<long long>(h->chunk, std::max<long long>(256, ((1LL << 28) / (8LL * std::max(1, P.n_in + P.n_out))) / 256 * 256));
        if (g_dais_chunk > 0)
            h->chunk = g_dais_chunk;
        Carver c;
        const size_t o_prog = c.take(sizeof(DaisInstr) * P.prog.size()), o_tab = c.take(sizeof(int32_t) * P.tables.size()), o_err = c.take(4 * sizeof(long long));
        CK(cudaMalloc(&h->mem, c.off));
        h->d_prog = (DaisInstr *)((char *)h->mem + o_prog);
        h->d_tables = (int32_t *)((char *)h->mem + o_tab);
        h->d_err = (unsigned long long *)((char *)h->mem + o_err);
        h->d_v0 = (long long *)(h->d_err + 2);
        CK(cudaMemcpyAsync(h->d_prog, P.prog.data(), sizeof(DaisInstr) * P.prog.size(), cudaMemcpyHostToDevice, g_stream));
        if (!P.tables.empty())
            CK(cudaMemcpyAsync(h->d_tables, P.tables.data(), sizeof(int32_t) * P.tables.size(), cudaMemcpyHostToDevice, g_stream));
        CK(cudaStreamSynchronize(g_stream));
        *out = h.release();
    });
}

int da4ml_dais_info(const da4ml_dais_t *h, int64_t out[8]) {
    if (!h || !out)
        return DA4ML_E_INVALID;
    const DaisCompiled &P = h->P;
    out[0] = P.n_in;
    out[1] = P.n_out;
    out[2] = P.n_ops;
    out[3] = P.n_tables;
    out[4] = P.n_slots;
    out[5] = h->tile > 0 ? 0 : 1;
    out[6] = h->tile > 0 ? h->tile : h->chunk;
    out[7] = P.max_width;
    return DA4ML_OK;
}

int da4ml_dais_infer(da4ml_dais_t *h, const double *x, int64_t n_samples, double *y) {
    return guarded([&] {
        if (!h || n_samples < 0 || (n_samples > 0 && ((!x && h->P.n_in) || (!y && h->P.n_out))))
            throw ApiError(DA4ML_E_INVALID, "invalid argument");
        if (n_samples == 0)
            return;
        init_device();
        dais_check_device(h);
        const DaisCompiled &P = h->P;
        const long long C = std::min<long long>(h->chunk, n_samples);
        Carver c;
        const size_t o_x = c.take(sizeof(double) * std::max<long long>(C * P.n_in, 1)), o_y = c.take(sizeof(double) * std::max<long long>(C * P.n_out, 1));
        g_dais_io.ensure(c.off, false);
        double *dx = (double *)((char *)g_dais_io.p + o_x), *dy = (double *)((char *)g_dais_io.p + o_y);
        CK(cudaMemsetAsync(h->d_err, 0xff, 2 * sizeof(unsigned long long), g_stream));
        for (long long s0 = 0; s0 < n_samples; s0 += C) {
            const long long Sc = std::min<long long>(C, n_samples - s0);
            if (P.n_in)
                CK(cudaMemcpyAsync(dx, x + s0 * P.n_in, sizeof(double) * Sc * P.n_in, cudaMemcpyHostToDevice, g_stream));
            dais_launch(dais_stream(h), dx, dy, Sc, s0, h->d_err, nullptr);
            dais_check(h, dais_stream(h), [&](long long s) {
                CK(cudaMemcpyAsync(dx, x + s * P.n_in, sizeof(double) * P.n_in, cudaMemcpyHostToDevice, g_stream));
                return (const double *)dx;
            }, dy);
            if (P.n_out)
                CK(cudaMemcpyAsync(y + s0 * P.n_out, dy, sizeof(double) * Sc * P.n_out, cudaMemcpyDeviceToHost, g_stream));
            CK(cudaStreamSynchronize(g_stream));
        }
    });
}

int da4ml_dais_infer_device(da4ml_dais_t *h, const double *x_dev, int64_t n_samples, double *y_dev) {
    return guarded([&] {
        if (!h || n_samples < 0 || (n_samples > 0 && ((!x_dev && h->P.n_in) || (!y_dev && h->P.n_out))))
            throw ApiError(DA4ML_E_INVALID, "invalid argument");
        if (n_samples == 0)
            return;
        init_device();
        dais_check_device(h);
        const DaisCompiled &P = h->P;
        g_dais_io.ensure(sizeof(double) * std::max(P.n_out, 1), false);
        CK(cudaMemsetAsync(h->d_err, 0xff, 2 * sizeof(unsigned long long), g_stream));
        for (long long s0 = 0; s0 < n_samples; s0 += h->chunk) {
            const long long Sc = std::min<long long>(h->chunk, n_samples - s0);
            dais_launch(dais_stream(h), x_dev + s0 * P.n_in, y_dev + s0 * P.n_out, Sc, s0, h->d_err, nullptr);
        }
        dais_check(h, dais_stream(h), [&](long long s) { return x_dev + s * P.n_in; }, (double *)g_dais_io.p);
    });
}

namespace {
void dais_profile_args(const da4ml_dais *h, const double *x, int64_t n_samples, int64_t *stats, int64_t *first) {
    if (!h || n_samples < 0 || !stats || !first || (n_samples > 0 && !x && h->P.n_in))
        throw ApiError(DA4ML_E_INVALID, "invalid argument");
    const int n_ops = h->P.n_ops;
    std::fill(stats, stats + n_ops, (int64_t)0x7fffffffffffffffll);
    std::fill(stats + n_ops, stats + 2LL * n_ops, (int64_t)0x8000000000000000ull);
    std::fill(stats + 2LL * n_ops, stats + 4LL * n_ops, (int64_t)0);
    first[0] = first[1] = -1;
}
void dais_capture_args(const da4ml_dais *h, const double *x, int64_t n_samples, const int32_t *ops, int32_t k, int64_t *out) {
    if (!h || n_samples < 0 || k < 0 || (k > 0 && !ops) || (n_samples > 0 && ((!x && h->P.n_in) || (!out && k))))
        throw ApiError(DA4ML_E_INVALID, "invalid argument");
    dais_check_ops(h, ops, k);
}
} // namespace

int da4ml_dais_profile(da4ml_dais_t *h, const double *x, int64_t n_samples, int64_t *stats, int64_t first[2]) {
    return guarded([&] {
        dais_profile_args(h, x, n_samples, stats, first);
        if (n_samples == 0)
            return;
        init_device();
        dais_check_device(h);
        const int n_in = h->P.n_in;
        double *dx = nullptr;
        dais_profile_run(h, n_samples, [&](long long s0, long long m) {
            g_dais_io.ensure(sizeof(double) * std::max<long long>(m * n_in, 1), false);
            dx = (double *)g_dais_io.p;
            if (n_in)
                CK(cudaMemcpyAsync(dx, x + s0 * n_in, sizeof(double) * m * n_in, cudaMemcpyHostToDevice, g_stream));
            return (const double *)dx;
        }, [&](long long s) {
            CK(cudaMemcpyAsync(dx, x + s * n_in, sizeof(double) * n_in, cudaMemcpyHostToDevice, g_stream));
            return (const double *)dx;
        }, stats, first);
    });
}

int da4ml_dais_profile_device(da4ml_dais_t *h, const double *x_dev, int64_t n_samples, int64_t *stats, int64_t first[2]) {
    return guarded([&] {
        dais_profile_args(h, x_dev, n_samples, stats, first);
        if (n_samples == 0)
            return;
        init_device();
        dais_check_device(h);
        const int n_in = h->P.n_in;
        dais_profile_run(h, n_samples, [&](long long s0, long long) { return x_dev + s0 * n_in; }, [&](long long s) { return x_dev + s * n_in; }, stats, first);
    });
}

int da4ml_dais_capture(da4ml_dais_t *h, const double *x, int64_t n_samples, const int32_t *ops, int32_t k, int64_t *out) {
    return guarded([&] {
        dais_capture_args(h, x, n_samples, ops, k, out);
        if (n_samples == 0)
            return;
        init_device();
        dais_check_device(h);
        const int n_in = h->P.n_in;
        double *dx = nullptr;
        long long *dout = nullptr;
        dais_capture_run(h, n_samples, ops, k, [&](long long s0, long long m) {
            Carver c;
            const size_t o_x = c.take(sizeof(double) * std::max<long long>(m * n_in, 1)), o_out = c.take(sizeof(long long) * std::max<long long>(m * k, 1));
            g_dais_io.ensure(c.off, false);
            dx = (double *)((char *)g_dais_io.p + o_x);
            dout = (long long *)((char *)g_dais_io.p + o_out);
            if (n_in)
                CK(cudaMemcpyAsync(dx, x + s0 * n_in, sizeof(double) * m * n_in, cudaMemcpyHostToDevice, g_stream));
            return (const double *)dx;
        }, [&](long long s) {
            CK(cudaMemcpyAsync(dx, x + s * n_in, sizeof(double) * n_in, cudaMemcpyHostToDevice, g_stream));
            return (const double *)dx;
        }, [&](long long, long long) { return dout; }, [&](long long s0, long long m) {
            if (k)
                CK(cudaMemcpyAsync(out + s0 * k, dout, sizeof(long long) * m * k, cudaMemcpyDeviceToHost, g_stream));
            CK(cudaStreamSynchronize(g_stream));
        });
    });
}

int da4ml_dais_capture_device(da4ml_dais_t *h, const double *x_dev, int64_t n_samples, const int32_t *ops, int32_t k, int64_t *out_dev) {
    return guarded([&] {
        dais_capture_args(h, x_dev, n_samples, ops, k, out_dev);
        if (n_samples == 0)
            return;
        init_device();
        dais_check_device(h);
        const int n_in = h->P.n_in;
        dais_capture_run(h, n_samples, ops, k, [&](long long s0, long long) { return x_dev + s0 * n_in; }, [&](long long s) { return x_dev + s * n_in; },
                         [&](long long s0, long long) { return (long long *)out_dev + s0 * k; }, [](long long, long long) {});
    });
}

void da4ml_dais_free(da4ml_dais_t *h) {
    std::lock_guard<std::mutex> lock(g_mutex);
    delete h;
}

int da4ml_cmvm_get_lsb_loc(float x) { return get_lsb_loc(x); }
int da4ml_cmvm_iceil_log2(float x) { return iceil_log2(x); }
int da4ml_cmvm_cost_add(const float q0[3], const float q1[3], int64_t shift, int sub, int adder_size, int carry_size, float out[2]) {
    cost_add(QInt{q0[0], q0[1], q0[2]}, QInt{q1[0], q1[1], q1[2]}, shift, sub != 0, adder_size, carry_size, out[0], out[1]);
    return DA4ML_OK;
}

} // extern "C"
