// host_common.cuh -- host-side plumbing shared by the driver pieces: error type, grow-only device / pinned buffers,
// bump carving, CUDA-event timing, device bring-up.  (Split out of cmvm_lib.cu; no path logic here.)
#pragma once
#include "../../include/da4ml_b200_cmvm.h"
#include "cmvm_decompose.cuh"
#include "cmvm_kernels.cuh"
#include "cmvm_kernel_own.cuh"
#include "dais_replay.cuh"

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <limits>
#include <memory>
#include <mutex>
#include <stdexcept>
#include <string>
#include <vector>

namespace da {

thread_local std::string g_err;
static std::mutex g_mutex;
static cudaStream_t g_stream = nullptr;
static int g_group_override = 0;
static int g_accounting = 0;
static int g_share_jobs = 1;  // solve byte-identical solve_single jobs of one call once (host_solve.cuh)
static long long g_first_caps[6] = {0}; // capacities forced on the first attempt of a round of jobs (host_plan.cuh FirstCap)

struct ApiError : std::runtime_error {
    int code;
    ApiError(int c, const std::string &m) : std::runtime_error(m), code(c) {}
};

#define CK(expr)                                                                                                  \
    do {                                                                                                          \
        cudaError_t _e = (expr);                                                                                  \
        if (_e != cudaSuccess)                                                                                    \
            throw ApiError(DA4ML_E_CUDA, std::string("CUDA error: ") + cudaGetErrorString(_e) + " at " #expr);    \
    } while (0)

// grow-only device buffer, reused across calls.  Every instance (globals and function-local statics alike) registers
// itself so that a change of the current CUDA device can drop them all (init_device).
struct DevBuf;
static std::vector<DevBuf *> &devbuf_registry() {
    static std::vector<DevBuf *> r;
    return r;
}
struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    bool fresh = false; // true right after (re)allocation: contents were zeroed
    bool registered = false;
    void drop() {
        if (p)
            cudaFree(p); // (valid whatever the current device is: unified addressing)
        p = nullptr;
        cap = 0;
    }
    void ensure(size_t bytes, bool zero_on_alloc) {
        if (!registered) {
            devbuf_registry().push_back(this);
            registered = true;
        }
        fresh = false;
        if (bytes <= cap)
            return;
        if (p)
            CK(cudaFree(p));
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 4 + 4096;
        CK(cudaMalloc(&p, want));
        cap = want;
        if (zero_on_alloc)
            CK(cudaMemsetAsync(p, 0, want, g_stream));
        fresh = true;
    }
};
struct PinBuf {
    void *p = nullptr;
    size_t cap = 0;
    void ensure(size_t bytes) {
        if (bytes <= cap)
            return;
        if (p)
            CK(cudaFreeHost(p));
        p = nullptr;
        cap = 0;
        CK(cudaMallocHost(&p, bytes + bytes / 4 + 4096));
        cap = bytes + bytes / 4 + 4096;
    }
};

struct Carver { // bump allocator over a byte range (256 B aligned pieces)
    size_t off = 0;
    size_t take(size_t bytes) {
        size_t o = off;
        off += (bytes + 255) & ~size_t(255);
        return o;
    }
};

static DevBuf g_job_arena, g_ws_arena, g_desc_arena;
static PinBuf g_pin_up, g_pin_down;
static int g_sm_count = 0, g_max_coop = 0;
static long long g_own_smem_max = 212 * 1024; // dynamic shared memory one CTA of the solve kernel may use
static int g_device = -1;       // CUDA device the cached buffers / kernel attributes belong to

struct Timing {
    double device_ms = 0;
    double solve_ms = 0;       // time inside cmvm_solve_kernel launches
    int64_t launches = 0;
    int64_t solve_launches = 0;
    double algo_bytes = 0;     // algorithmic bytes (SURVEY.md 8d) of every solve_single executed
    int64_t retried_jobs = 0;  // jobs relaunched after a capacity overflow
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> pending;
    std::vector<char> is_solve;
    void mark_solve() { is_solve.back() = 1; }
    void begin() {
        cudaEvent_t a, b;
        CK(cudaEventCreate(&a));
        CK(cudaEventCreate(&b));
        CK(cudaEventRecord(a, g_stream));
        pending.push_back({a, b});
        is_solve.push_back(0);
    }
    void end(int n_launch) {
        CK(cudaEventRecord(pending.back().second, g_stream));
        launches += n_launch;
    }
    void collect() { // call after a stream sync
        for (size_t i = 0; i < pending.size(); ++i) {
            auto &pr = pending[i];
            float ms = 0;
            if (cudaEventElapsedTime(&ms, pr.first, pr.second) == cudaSuccess) {
                device_ms += ms;
                if (is_solve[i])
                    solve_ms += ms;
            }
            cudaEventDestroy(pr.first);
            cudaEventDestroy(pr.second);
        }
        pending.clear();
        is_solve.clear();
    }
};

static void release_device_buffers(); // host_stage.cuh (needs the arenas declared there)

// Every call runs on the CURRENT CUDA device.  Cached device buffers and the kernels' shared-memory opt-ins belong to
// one device: when the caller has switched devices since the last call, everything cached is dropped and set up again.
static void init_device() {
    int dev = 0;
    if (g_sm_count) {
        CK(cudaGetDevice(&dev));
        if (dev == g_device)
            return;
        release_device_buffers();
        g_sm_count = 0;
    }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        throw ApiError(DA4ML_E_CUDA, "no CUDA device available (the CMVM solver has no CPU fallback)");
    CK(cudaGetDevice(&dev));
    g_device = dev;
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, dev));
    {
        // dynamic shared memory the solve kernel may ask for: what the SM offers minus the kernel's static part
        cudaFuncAttributes fa;
        CK(cudaFuncGetAttributes(&fa, cmvm_solve_kernel));
        int optin = 0;
        CK(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
        g_own_smem_max = std::min<long long>(216 * 1024, (long long)optin - (long long)fa.sharedSizeBytes);
        CK(cudaFuncSetAttribute(cmvm_solve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)g_own_smem_max));
        int per_sm = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, cmvm_solve_kernel, 512, (size_t)g_own_smem_max));
        if (per_sm < 1)
            throw ApiError(DA4ML_E_CUDA, "cmvm_solve_kernel cannot be made resident on this device");
    }
    g_sm_count = prop.multiProcessorCount;
    g_max_coop = g_sm_count; // one persistent CTA per SM
}

static int parse_method(const std::string &m) {
    if (m == "mc")
        return M_MC;
    if (m == "mc-dc")
        return M_MC_DC;
    if (m == "mc-pdc")
        return M_MC_PDC;
    if (m == "wmc")
        return M_WMC;
    if (m == "wmc-dc")
        return M_WMC_DC;
    if (m == "wmc-pdc")
        return M_WMC_PDC;
    if (m == "dummy")
        return M_DUMMY;
    throw ApiError(DA4ML_E_RUNTIME, "Unknown method: " + m); // cmvm_core.cc:63
}


} // namespace da
