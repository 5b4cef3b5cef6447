// cmvm_types.cuh -- device-side data layout of the CMVM solver (see DESIGN.md "Data layout in HBM").
#pragma once
#include <cstdint>
#ifndef DA_CPU_SIM
#include <cuda_runtime.h>
// shared-memory declarations go through these two macros so that the host-side SIMT shim of the tests (tests/simt) can
// give every simulated CTA its own copy
#define DA_SHARED_VAR(type, name) __shared__ type name
#define DA_DYN_SHARED(name) extern __shared__ __align__(16) unsigned char name[]
#endif

namespace da {

// One live row of one output column: expression id + the two packed sign planes of its CSD digits
// in that column (bit j of P: digit +2^j present, bit j of N: digit -2^j present).  Replaces the
// reference's SparseExpr::rows[i_out] vector<int8_t> (types.hh:104-141).
struct ColEnt {
    uint32_t e, P, N, pad;
};

// One histogram entry (replaces FreqMap::value_type = pair<Pair,uint32_t>, types.hh:39-41):
//   x = sortable selector score, y = count (0 = tombstone), z/w = low/high word of the packed key.
typedef uint4 FEnt;

enum Status : int { ST_OK = 0, ST_EXPR_OVERFLOW = 1, ST_FSEG_OVERFLOW = 2, ST_TOUCH_OVERFLOW = 3 /* internal: pair-counter passes */, ST_OPS_OVERFLOW = 4, ST_LIST_OVERFLOW = 5 };

// result_meta layout (int64 words)
enum Meta : int {
    META_STATUS = 0,
    META_N_OPS = 1,
    META_T = 2,      // greedy iterations
    META_SUM_F = 3,  // sum over iterations of live histogram entries seen by the selector
    META_SUM_R = 4,  // sum over iterations of digit pairs enumerated (update_stats)
    META_F0 = 5,     // initial histogram entries
    META_R0 = 6,     // digit pairs behind the initial histogram (sum of counts incl. count==1)
    META_D_FINAL = 7,
    META_F_MAX = 8,
    META_COMPACTIONS = 9,
    META_COST_BITS = 11, // float bits: cost_init + sum of op costs in op order
    META_RESCANNED = 13, // histogram entries re-read by the chunked argmax (all steps)
    META_LIST_MAX = 14,  // longest column list seen
    META_PHASE0 = 16, // 8 words: cycles spent by CTA rank 0 in substitute, recount, refresh, wait1, harvest, publish, wait2, collect
    META_PHASEMAX = 24, // 8 words: the same, maximum over the CTAs of the group
    META_MILESTONES = 32, // 7 x 9 words: cumulative phase cycles of CTA rank 0 (8 words) + cycles since the problem started, after 250 * 2^k greedy steps (k = 0..6)
    META_SPLITS = 95,     // pair-counting passes abandoned for a full counter table and split in two (sum over the CTAs)
    META_WORDS = 96
};

// prep_meta layout (int32 words) written by the prep kernel
enum PrepMeta : int { PM_NBITS = 0, PM_D0 = 1, PM_COLCAP = 2, PM_DCOL_MAX = 3, PM_ROWS_MAX = 4, PM_WORDS = 8 };

struct ProblemDesc {
    // ---- inputs
    int n_in, n_out;
    int method;
    int adder_size, carry_size;
    const float *kernel; // [n_in, n_out] row-major, device
    const float *qint;   // [n_in, 3]
    const float *lat;    // [n_in]
    // ---- prep outputs
    uint2 *masks0; // [n_in][n_out] (P, N)
    int8_t *shift0; // [n_in]
    int8_t *shift1; // [n_out]
    int *col_digits; // [n_out]
    int *prep_meta;  // [PM_WORDS]
    // ---- solve outputs
    int4 *op_misc;  // [ops_cap] id0, id1, opcode, data
    float4 *op_q;   // [ops_cap] qmin, qmax, qstep, latency
    float *op_cost; // [ops_cap]
    int *out_idx, *out_shift, *out_neg; // [n_out]
    float4 *out_q;                      // [n_out] (qmin, qmax, qstep, latency) of each output's op, (0, 0, inf, 0) for dead outputs
    float cost_init;                    // running float cost the sequential sum over this stage's ops starts from (api.cc:222-227)
    long long *result_meta;             // [META_WORDS]
    int *trace;                         // optional [trace_cap][5]: id0,id1,shift,sub,|F| per iteration
    int trace_cap;
    // ---- capacities chosen by the host after prep
    int nbits;          // CSD width
    int e_cap;          // expression ids the problem may use (n_in + T_cap)
    int ops_cap;        // n_in + D0
    int col_cap;        // capacity of each global column list (adder-tree phase)
    int heap_lane_cap;  // to_solution: private heap entries per lane (32 lanes per column)
};

// Per-group scratch ("group slot"): one group of G CTAs solves one problem at a time.
struct GroupWs {
    uint32_t *col_u32; // column lists handed to the adder trees: [n_out_max][3][col_cap_max] (e[], P[], N[])
    int *col_len;      // [n_out_max]
    int *col_k;        // [n_out_max] digits per column at to_solution time
    uint32_t *mod_step; // [e_cap_max] step at which an expression was last rewritten (lazy histogram purge)
    FEnt *fseg;        // [G][fseg_cap]
    uint4 *heap;       // [n_out_max][32 lanes][heap_lane_cap][2] to_solution scratch (lane-private)
    unsigned *barrier; // monotonically increasing arrive counter
    unsigned long long *xchg; // [2][G][4] stamped all-gather slots (barrier + payload in one round trip)
    int fseg_cap;
    long long heap_cap;
};

// Launch-wide configuration of the persistent solve kernel (uniform over all groups / problems of a launch).
struct LaunchCfg {
    int G;          // CTAs per group
    int cpc;        // output columns per CTA in the adder-tree phase
    int chunk_log;  // log2(histogram entries per argmax chunk)
    int nchunk_cap; // chunk-cache slots per CTA
    int accounting; // 1: exact live-histogram size every step (re-reads every chunk), for traces / counters
};

} // namespace da
