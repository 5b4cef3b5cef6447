// sim_dais_profile.cc -- TEST INFRASTRUCTURE ONLY: the product's every-op DAIS variant (host_dais.cuh) and its profile
// and capture observers (dais_exec.cuh, unmodified) run on the CPU under the SIMT shim of simt.h, in either slot
// regime, so that the CPU test suite can compare them with the reference interpreter's stored values.  The launch
// sequence mirrors da4ml_dais_profile / da4ml_dais_capture (da4ml_b200/csrc/cmvm_lib.cu).  Never linked into the product.
#include "simt.h"

#include "../../da4ml_b200/csrc/host_dais.cuh"

#include <string>

using namespace da;

namespace {
std::string g_err;

// Runs the variant over x in chunks with observer `make_obs(s0, m)`, `after(s0, m)` after each launch; raises the
// reference's message for a lookup out of range as the library does.  Returns the regime (0 shared, 1 global).
template <class MakeObs, class After>
int run(const DaisCompiled &P, const double *x, long long n, long long shared_bytes, long long chunk, int cta_threads, MakeObs make_obs, After after) {
    const int n_instr = (int)P.prog.size();
    const int tile = dais_shared_tile(P.n_slots, shared_bytes);
    const long long pad = (chunk + 255) / 256 * 256;
    std::vector<long long> arena((size_t)std::max(P.n_slots, 1) * pad);
    auto launch = [&](const double *xs, long long m, long long sample0, unsigned long long *err, long long *v0, auto obs) {
        using Obs = decltype(obs);
        if (tile > 0) {
            const size_t smem = (size_t)8 * std::max(P.n_slots, 1) * tile;
            simt::launch(dim3((unsigned)((m + tile - 1) / tile)), dim3(tile), smem, [&] {
                dais_exec_kernel<true, Obs>(P.prog.data(), n_instr, xs, P.n_in, nullptr, P.n_out, m, nullptr, 0, P.tables.data(), err, sample0, v0, obs);
            }, 64 * 1024);
        }
        else {
            const long long stride = Obs::kActive ? (m + cta_threads - 1) / cta_threads * cta_threads : m;
            simt::launch(dim3((unsigned)((m + cta_threads - 1) / cta_threads)), dim3(cta_threads), 0, [&] {
                dais_exec_kernel<false, Obs>(P.prog.data(), n_instr, xs, P.n_in, nullptr, P.n_out, m, arena.data(), stride, P.tables.data(), err, sample0, v0, obs);
            }, 64 * 1024);
        }
    };
    unsigned long long err = ~0ull;
    for (long long s0 = 0; s0 < n; s0 += chunk) {
        const long long m = std::min(chunk, n - s0);
        launch(x + s0 * P.n_in, m, s0, &err, nullptr, make_obs(s0, m));
        if (err != ~0ull) {
            const long long s = (long long)(err / n_instr);
            const int pc = (int)(err % n_instr);
            unsigned long long err1 = ~0ull;
            long long v0 = 0;
            launch(x + s * P.n_in, 1, 0, &err1, &v0, DaisNoObserver{});
            throw std::runtime_error(dais_lookup_message(P, pc, v0));
        }
        after(s0, m);
    }
    return tile > 0 ? 0 : 1;
}
} // namespace

extern "C" {

const char *sim_dais_profile_last_error() { return g_err.c_str(); }

// The every-op variant: info {n_ops, n_instr, n_slots, n_cols, 0...}; side [n_instr][6] {op, cap_begin, cap_count,
// quant, lo, hi}; cols [n_cols] (either may be NULL).  0, or -1 on an error.
int sim_dais_variant(const int32_t *words, long long n_words, const int32_t *ops, int k, long long *info, long long *side, int *cols) {
    try {
        const DaisCompiled P = dais_compile(words, n_words, true, ops, k);
        const long long v[8] = {P.n_ops, (long long)P.prog.size(), P.n_slots, (long long)P.cap_cols.size(), 0, 0, 0, 0};
        std::copy(v, v + 8, info);
        for (size_t i = 0; side && i < P.obs.size(); ++i) {
            const DaisObsEntry &e = P.obs[i];
            const long long r[6] = {e.op, e.cap_begin, e.cap_count, e.quant, e.lo, e.hi};
            std::copy(r, r + 6, side + 6 * i);
        }
        if (cols)
            std::copy(P.cap_cols.begin(), P.cap_cols.end(), cols);
        return 0;
    }
    catch (const std::exception &e) {
        g_err = e.what();
        return -1;
    }
}

// stats [4][n_ops] and first[2] of x [n][n_in], as da4ml_dais_profile computes them.  Returns the regime or -1.
int sim_dais_profile(const int32_t *words, long long n_words, const double *x, long long n, long long shared_bytes, long long chunk, int cta_threads, long long *stats, long long *first) {
    try {
        const DaisCompiled P = dais_compile(words, n_words, true);
        const int n_instr = (int)P.prog.size(), n_ops = P.n_ops;
        std::vector<long long> tot(4 * (size_t)n_ops, 0), rec((size_t)4 * std::max(n_instr, 1) * ((chunk + 31) / 32));
        std::fill(tot.begin(), tot.begin() + n_ops, (long long)0x7fffffffffffffffll);
        std::fill(tot.begin() + n_ops, tot.begin() + 2 * n_ops, (long long)0x8000000000000000ull);
        unsigned long long key = ~0ull;
        int regime = dais_shared_tile(P.n_slots, shared_bytes) > 0 ? 0 : 1;
        if (n > 0)
            regime = run(P, x, n, shared_bytes, chunk, cta_threads, [&](long long, long long m) {
                DaisProfileObserver o{};
                o.side = P.obs.data(), o.rec = rec.data(), o.n_warps = (m + 31) / 32, o.first = &key, o.n_ops = n_ops;
                return o;
            }, [&](long long, long long m) {
                if (n_instr > 0)
                    simt::launch(dim3((unsigned)(((long long)n_instr * 32 + 255) / 256)), dim3(256), 0, [&] {
                        dais_profile_merge_kernel(rec.data(), n_instr, (m + 31) / 32, P.obs.data(), tot.data(), n_ops);
                    }, 64 * 1024);
            });
        std::copy(tot.begin(), tot.end(), stats);
        first[0] = key == ~0ull ? -1 : (long long)(key / (unsigned long long)n_ops);
        first[1] = key == ~0ull ? -1 : (long long)(key % (unsigned long long)n_ops);
        return regime;
    }
    catch (const std::exception &e) {
        g_err = e.what();
        return -1;
    }
}

// out [n][k]: the values of ops[0..k), as da4ml_dais_capture computes them.  Returns the regime or -1.
int sim_dais_capture(const int32_t *words, long long n_words, const double *x, long long n, const int32_t *ops, int k, long long *out, long long shared_bytes, long long chunk, int cta_threads) {
    try {
        const DaisCompiled P = dais_compile(words, n_words, true, ops, k);
        if (n == 0)
            return dais_shared_tile(P.n_slots, shared_bytes) > 0 ? 0 : 1;
        return run(P, x, n, shared_bytes, chunk, cta_threads, [&](long long s0, long long) {
            DaisCaptureObserver o{};
            o.side = P.obs.data(), o.cols = P.cap_cols.data(), o.out = out + s0 * k, o.k = k;
            return o;
        }, [](long long, long long) {});
    }
    catch (const std::exception &e) {
        g_err = e.what();
        return -1;
    }
}

} // extern "C"
