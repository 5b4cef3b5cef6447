// sim_dais.cc -- TEST INFRASTRUCTURE ONLY: the product's DAIS compiler and interpreter kernel (host_dais.cuh,
// dais_exec.cuh, unmodified) run on the CPU under the SIMT shim of simt.h, in either slot regime, so that the CPU
// test suite can compare them with the reference interpreter's stored answers.  The launch sequence mirrors
// da4ml_dais_infer (da4ml_b200/csrc/cmvm_lib.cu).  Never linked into the product.
#include "simt.h"

#include "../../da4ml_b200/csrc/host_dais.cuh"

#include <string>

using namespace da;

namespace {
std::string g_err;
}

extern "C" {

const char *sim_dais_last_error() { return g_err.c_str(); }

// info: {n_in, n_out, n_ops, n_tables, L, n_instr, max_width, 0}; op_slot[n_ops] (may be NULL).  0, or -1 on a load
// error (sim_dais_last_error()).
int sim_dais_compile(const int32_t *words, long long n_words, long long *info, int *op_slot) {
    try {
        const DaisCompiled P = dais_compile(words, n_words);
        const long long v[8] = {P.n_in, P.n_out, P.n_ops, P.n_tables, P.n_slots, (long long)P.prog.size(), P.max_width, 0};
        std::copy(v, v + 8, info);
        if (op_slot)
            std::copy(P.op_slot.begin(), P.op_slot.end(), op_slot);
        return 0;
    }
    catch (const std::exception &e) {
        g_err = e.what();
        return -1;
    }
}

// x [n][n_in] -> y [n][n_out] through the simulated kernel.  shared_bytes: slot budget of one CTA (the shared regime
// when 32 samples fit); chunk: samples per launch; cta_threads: CTA size of the global regime.  Returns the regime
// (0 shared, 1 global), or -1 on an error (load error or lookup out of range, sim_dais_last_error()).
int sim_dais_run(const int32_t *words, long long n_words, const double *x, long long n, double *y, long long shared_bytes, long long chunk, int cta_threads) {
    try {
        const DaisCompiled P = dais_compile(words, n_words);
        const int n_instr = (int)P.prog.size();
        const int tile = dais_shared_tile(P.n_slots, shared_bytes);
        std::vector<long long> arena((size_t)std::max(P.n_slots, 1) * std::max<long long>(chunk, 1));
        auto launch = [&](const double *xs, double *ys, long long m, long long sample0, unsigned long long *err, long long *v0) {
            if (tile > 0) {
                const size_t smem = (size_t)8 * std::max(P.n_slots, 1) * tile;
                simt::launch(dim3((unsigned)((m + tile - 1) / tile)), dim3(tile), smem, [&] {
                    dais_exec_kernel<true>(P.prog.data(), n_instr, xs, P.n_in, ys, P.n_out, m, nullptr, 0, P.tables.data(), err, sample0, v0);
                }, 64 * 1024);
            }
            else
                simt::launch(dim3((unsigned)((m + cta_threads - 1) / cta_threads)), dim3(cta_threads), 0, [&] {
                    dais_exec_kernel<false>(P.prog.data(), n_instr, xs, P.n_in, ys, P.n_out, m, arena.data(), m, P.tables.data(), err, sample0, v0);
                }, 64 * 1024);
        };
        unsigned long long err = ~0ull;
        for (long long s0 = 0; s0 < n; s0 += chunk) {
            const long long m = std::min(chunk, n - s0);
            launch(x + s0 * P.n_in, y + s0 * P.n_out, m, s0, &err, nullptr);
        }
        if (err != ~0ull) {
            const long long s = (long long)(err / n_instr);
            const int pc = (int)(err % n_instr);
            std::vector<double> y1(std::max(P.n_out, 1));
            unsigned long long err1 = ~0ull;
            long long v0 = 0;
            launch(x + s * P.n_in, y1.data(), 1, 0, &err1, &v0);
            throw std::runtime_error(dais_lookup_message(P, pc, v0));
        }
        return tile > 0 ? 0 : 1;
    }
    catch (const std::exception &e) {
        g_err = e.what();
        return -1;
    }
}

} // extern "C"
