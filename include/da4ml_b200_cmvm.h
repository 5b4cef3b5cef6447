/* da4ml_b200_cmvm.h -- C ABI of the B200-native CMVM solver (libda4ml_b200_cmvm.so).
 *
 * Drop-in boundary for the reference's nanobind module `da4ml._binary.cmvm_bin`
 * (reference src/da4ml/_binary/cmvm/bindings.cc:227-263).  Each entry point names the reference
 * interface it replaces.  Plain pointers and sizes only; all arrays are host memory unless noted,
 * dense C order.  Every compute entry point runs on the current CUDA device (cudaSetDevice /
 * torch.cuda.set_device) on the stream set with da4ml_cmvm_set_stream (default: stream 0) and
 * returns 0 on success; on failure it returns a non-zero DA4ML_E_* code and
 * da4ml_cmvm_last_error() describes it.  There is no CPU fallback: without a usable CUDA device the
 * compute calls fail with DA4ML_E_CUDA.
 */
#ifndef DA4ML_B200_CMVM_H
#define DA4ML_B200_CMVM_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum {
    DA4ML_OK = 0,
    DA4ML_E_INVALID = 1, /* bad argument; reference raises ValueError / std::invalid_argument  */
    DA4ML_E_RUNTIME = 2, /* e.g. "Unknown method: ..." (cmvm_core.cc:63), reference RuntimeError */
    DA4ML_E_CUDA = 3,    /* CUDA runtime failure or no device                                    */
    DA4ML_E_CAPACITY = 4 /* internal buffer could not be grown                                  */
};

typedef struct da4ml_pipeline da4ml_pipeline_t; /* opaque result, mirrors PipelineResult (types.hh:164-166) */

/* Message of the last failure on the calling thread. */
const char *da4ml_cmvm_last_error(void);

/* Library / device information: writes {abi_version, cuda_device_count, sm_count, sm_major, sm_minor}. */
int da4ml_cmvm_device_info(int32_t out[5]);

/* Stream (cudaStream_t as void*) used for every subsequent launch and copy issued by this library. */
int da4ml_cmvm_set_stream(void *cuda_stream);

/* Tuning knob: CTAs cooperating on one problem (0 = automatic). */
int da4ml_cmvm_set_group_size(int ctas_per_problem);

/* Launch geometry the solver would choose for a set of solve_single jobs on `co_resident_ctas` CTAs (148 on a B200),
 * without touching a device.  jobs: [n][8] int64 = {n_in, n_out, nbits, csd_digits, max_digits_per_column,
 * column_list_bound, f_mul, list_mul}; out: [12] int64 = {ctas_per_problem, concurrent_groups, columns_per_cta (adder
 * trees), list_rows_in_shared_memory, log2_chunk, chunk_slots, segment_entries_per_cta, log2_pair_counters,
 * dynamic_shared_bytes, shared_budget_bytes, narrow_rows (6-byte list rows), spill_rows}.  Diagnostic; the reference has
 * no counterpart. */
int da4ml_cmvm_plan(const int64_t *jobs, int64_t n_jobs, int co_resident_ctas, int group_override, int64_t out[12]);

/* Free the large device / pinned work buffers the library caches between calls (re-grown on demand; function-local
 * scratch of the small helper entry points is kept). */
int da4ml_cmvm_release(void);

/* Exact work accounting (sum over iterations of the live histogram size, needed for the algorithmic-bytes
 * figure): when on, every iteration re-reads the whole histogram instead of only the chunks whose cached
 * maximum was invalidated.  Results are identical; only the counters and the speed change.  Off by default;
 * implied by a trace request. */
int da4ml_cmvm_set_accounting(int on);
/* The decompose_dc candidates of one call often decompose to byte-identical stage matrices; a solve_single job is a
 * pure function of its inputs, so by default identical jobs are solved once and the result shared (identical output to
 * the reference, which solves each candidate separately).  0 switches the sharing off. */
int da4ml_cmvm_set_job_sharing(int on);

/* ---- solve -------------------------------------------------------------------------------------
 * Replaces `solve` (bindings.cc:184-225 -> api.cc:147-250).
 *   kernel       [n_in, n_out] float32
 *   method0/1    "mc" "mc-dc" "mc-pdc" "wmc" "wmc-dc" "wmc-pdc" "dummy"; method1 may be "auto"
 *   qintervals   [n_in, 3] (min, max, step) or NULL  -> (-128, 127, 1)      (api.cc:161-167)
 *   latencies    [n_in] or NULL                     -> 0                   (api.cc:168-174)
 * Result: two stages (CombLogicResult, types.hh:153-162).  Free with da4ml_pipeline_free.          */
int da4ml_cmvm_solve(
    const float *kernel, int64_t n_in, int64_t n_out, const char *method0, const char *method1,
    int hard_dc, int decompose_dc, const float *qintervals, const float *latencies, int adder_size,
    int carry_size, int search_all_decompose_dc, da4ml_pipeline_t **out
);

/* Batched form of da4ml_cmvm_solve: n independent problems solved concurrently on one GPU (the
 * reference has no batch API; its caller loops, trace/fixed_variable_array.py:368-371).  Per-problem
 * arrays of pointers; qintervals[i] / latencies[i] (or the arrays themselves) may be NULL.        */
int da4ml_cmvm_solve_batch(
    int64_t n_problems, const float *const *kernels, const int64_t *n_in, const int64_t *n_out,
    const char *method0, const char *method1, int hard_dc, int decompose_dc,
    const float *const *qintervals, const float *const *latencies, int adder_size, int carry_size,
    int search_all_decompose_dc, da4ml_pipeline_t **out /* [n_problems] */
);

/* Same as da4ml_cmvm_solve_batch but kernels_dev[i] are DEVICE pointers ([n_in, n_out] float32, dense): the
 * constant matrices are already resident in HBM (qintervals / latencies stay small host arrays). */
int da4ml_cmvm_solve_batch_device(
    int64_t n_problems, const float *const *kernels_dev, const int64_t *n_in, const int64_t *n_out,
    const char *method0, const char *method1, int hard_dc, int decompose_dc,
    const float *const *qintervals, const float *const *latencies, int adder_size, int carry_size,
    int search_all_decompose_dc, da4ml_pipeline_t **out /* [n_problems] */
);

/* One CSE stage on its own: `solve_single` (cmvm_core.cc:227-237).  One-stage pipeline.  When
 * trace_cap > 0, trace receives up to trace_cap rows of (id0, id1, shift, sub, |F|) per greedy
 * iteration (the reference's loop cmvm_core.cc:36-70) for step-level parity checks.              */
int da4ml_cmvm_solve_single(
    const float *kernel, int64_t n_in, int64_t n_out, const char *method, const float *qintervals,
    const float *latencies, int adder_size, int carry_size, int32_t *trace, int64_t trace_cap,
    da4ml_pipeline_t **out
);

/* ---- result access (mirrors make_py_comblogic, bindings.cc:106-139) ---------------------------- */
void da4ml_pipeline_free(da4ml_pipeline_t *p);
int64_t da4ml_pipeline_n_stages(const da4ml_pipeline_t *p);
/* meta: {n_in, n_out, n_ops, carry_size, adder_size} */
int da4ml_pipeline_stage_meta(const da4ml_pipeline_t *p, int64_t stage, int64_t meta[5]);
/* inp_shifts[n_in], out_idxs/out_shifts/out_negs[n_out] int64;
 * ops_i [n_ops,4] int64 (id0,id1,opcode,data); ops_f [n_ops,5] float32 (qmin,qmax,qstep,latency,cost).
 * Any pointer may be NULL to skip that array. */
int da4ml_pipeline_stage_copy(
    const da4ml_pipeline_t *p, int64_t stage, int64_t *inp_shifts, int64_t *out_idxs,
    int64_t *out_shifts, int64_t *out_negs, int64_t *ops_i, float *ops_f
);
/* Work counters of one stage, int64[32]: see enum Meta in csrc/cmvm_types.cuh
 * (status, n_ops, T, sum|F_t|, sum R_t, F0, R0, D_final, F_max, compactions, ..., per-phase SM cycles). */
int da4ml_pipeline_stage_counters(const da4ml_pipeline_t *p, int64_t stage, int64_t counters[32]);
/* Diagnostic: 7 x 9 words, one group per milestone of 250 * 2^k greedy steps (k = 0..6): cumulative cycles CTA 0 of the
 * problem's group spent in each of the 8 phases of a greedy step, and the cycles since the loop started (zero for
 * milestones the stage did not reach). */
int da4ml_pipeline_stage_milestones(const da4ml_pipeline_t *p, int64_t stage, int64_t out[63]);
/* Device milliseconds spent in this library's kernels for the call that produced p (CUDA events). */
double da4ml_pipeline_device_ms(const da4ml_pipeline_t *p);
/* Number of kernel launches issued for the call that produced p. */
int64_t da4ml_pipeline_launches(const da4ml_pipeline_t *p);
/* Profile of the call that produced p: {device_ms, launches, solve_kernel_ms, solve_kernel_launches,
 * algorithmic_bytes (all solve_single jobs of the call, exact in accounting mode), 0, 0, 0}. */
int da4ml_pipeline_profile(const da4ml_pipeline_t *p, double out[8]);

/* ---- DAIS replay (SURVEY 8f N2) -------------------------------------------------------------------
 * Replaces `run_interp` of the reference's second native module (dais/bindings.cc:32-110 -> DAISInterpreter.cc) for
 * the programs the CMVM path produces (opcodes -1, 0, 1; no lookup tables): `program` = int32 words of
 * CombLogic.to_binary (types.py:500-541), inputs [n_samples, n_in] float64, outputs [n_samples, n_out] float64.
 * Bit-exact int64 fixed-point semantics of the reference interpreter. */
int da4ml_dais_run(const int32_t *program, int64_t n_words, const double *inputs, int64_t n_samples, double *outputs);

/* ---- complete DAIS interpreter ---------------------------------------------------------------------
 * Every opcode of the reference's DAISInterpreter.cc, lookup tables included, bit-exact.  A program is loaded once:
 * parsed, validated (with the reference's messages, before any device call), compiled into device instructions with
 * value slots assigned by liveness, and kept resident until da4ml_dais_free.  A lookup index out of range is reported
 * as the reference reports it with one thread: the first offending sample, then its first offending op. */
typedef struct da4ml_dais da4ml_dais_t;
int da4ml_dais_load(const int32_t *program, int64_t n_words, da4ml_dais_t **out);
/* {n_in, n_out, n_ops, n_tables, value slots L, regime (0 shared memory, 1 global memory), samples per CTA (shared) or
 * per launch (global), widest dtype in bits} */
int da4ml_dais_info(const da4ml_dais_t *h, int64_t out[8]);
/* x [n_samples, n_in], y [n_samples, n_out] float64 in host memory */
int da4ml_dais_infer(da4ml_dais_t *h, const double *x, int64_t n_samples, double *y);
/* the same with x and y in device memory (on the device the program was loaded on), on the library's stream */
int da4ml_dais_infer_device(da4ml_dais_t *h, const double *x_dev, int64_t n_samples, double *y_dev);
/* Profile of n_samples samples, every op (dead ones included) run as the reference runs them.  stats [4][n_ops]:
 * min and max of each op's int64 value (INT64_MAX / INT64_MIN for no samples), the number of samples whose value lies
 * outside the op's declared dtype range, and, for the wrapping ops (-1, +-2, +-3, +-6), the number of samples whose
 * value the wrap step changed.  first = {sample, op} of the first value outside its range (sample order, then op
 * order), {-1, -1} when there is none.  x in host memory; stats and first in host memory. */
int da4ml_dais_profile(da4ml_dais_t *h, const double *x, int64_t n_samples, int64_t *stats, int64_t first[2]);
/* the same with x in device memory, on the library's stream; stats and first are still host memory */
int da4ml_dais_profile_device(da4ml_dais_t *h, const double *x_dev, int64_t n_samples, int64_t *stats, int64_t first[2]);
/* The raw int64 values of ops[0..k) (each in [0, n_ops), duplicates allowed) for every sample: out [n_samples][k],
 * the reference interpreter's buffer[op].  x and out in host memory. */
int da4ml_dais_capture(da4ml_dais_t *h, const double *x, int64_t n_samples, const int32_t *ops, int32_t k, int64_t *out);
/* the same with x and out in device memory (ops in host memory), on the library's stream */
int da4ml_dais_capture_device(da4ml_dais_t *h, const double *x_dev, int64_t n_samples, const int32_t *ops, int32_t k, int64_t *out_dev);
void da4ml_dais_free(da4ml_dais_t *h);
/* Development switch, read by da4ml_dais_load: shared memory one CTA's slot file may use (a budget below 32 samples'
 * worth selects the global-memory regime) and samples per launch.  0 = automatic for either. */
int da4ml_dais_set_shared_budget(int64_t shared_bytes, int64_t chunk_samples);

/* ---- helpers exported by the reference module -------------------------------------------------- */
/* `csd_decompose` (bindings.cc:63-103 -> bit_decompose.cc:44-62).  csd must hold n_in*n_out*32 int8;
 * *n_bits receives N, the caller reads csd as [n_in, n_out, N].  shift0[n_in], shift1[n_out] int8. */
int da4ml_cmvm_csd_decompose(
    const float *kernel, int64_t n_in, int64_t n_out, int center, int8_t *csd, int8_t *shift0,
    int8_t *shift1, int64_t *n_bits
);
/* `int_arr_to_csd` (bindings.cc:43-61 -> bit_decompose.cc:22-42): flat int32[n] -> int8[n, N]. */
int da4ml_cmvm_int_arr_to_csd(const int32_t *x, int64_t n, int8_t *csd, int64_t *n_bits);
/* `kernel_decompose` (mat_decompose.cc:62-137): m0 [n_in,n_out], m1 [n_out,n_out]. */
int da4ml_cmvm_kernel_decompose(const float *kernel, int64_t n_in, int64_t n_out, int dc, float *m0, float *m1);
/* scalar helpers (bit_decompose.cc:10-20, indexers.hh:12-18, state_opr.cc:31-67) */
int da4ml_cmvm_get_lsb_loc(float x);
int da4ml_cmvm_iceil_log2(float x);
int da4ml_cmvm_cost_add(
    const float q0[3], const float q1[3], int64_t shift, int sub, int adder_size, int carry_size,
    float out[2] /* (latency increment, cost) */
);

#ifdef __cplusplus
}
#endif
#endif
