// dais_exec.cuh -- the complete DAIS interpreter on the device: every opcode of the reference's DAISInterpreter.cc
// (exec_ops :291-388, inference :390-401), lookup tables included, over programs compiled once by host_dais.cuh.
//
// One thread runs one sample through the whole compiled instruction stream.  Every thread of a CTA executes the same
// instruction at the same time, so dispatch never diverges; only the data-dependent selects do.  Values live in int64
// slots assigned by liveness on the host (L slots, not n_ops), in one of two places (the template argument):
//   shared: the CTA's [L][T] slot file in dynamic shared memory, T = blockDim.x samples; HBM sees only inputs, outputs
//           and the instruction stream
//   global: an [L][S] arena in HBM, sample fastest so that a warp's accesses to one slot are coalesced
// Arithmetic is two's-complement int64, done in uint64 where C++ would overflow.  Shift counts that come from dtypes
// are taken modulo 64 explicitly (the reference's x86 build shifts int64 by count & 63); the host folds the int32
// parts (widths, int_min, shift sums) in the reference's int32 arithmetic.
#pragma once
#include <cstdint>
#include <cstring>
#ifndef DA_CPU_SIM
#include <cuda_runtime.h>
#define DA_DYN_SHARED(name) extern __shared__ __align__(16) unsigned char name[]
#else
// the CPU simulation of the kernels (tests/simt) has no redux.sync: the same 32-bit warp reductions on its shuffles
template <class T, class F> T da_sim_reduce(unsigned m, T v, F f) {
    for (int o = 16; o > 0; o >>= 1)
        v = f(v, __shfl_xor_sync(m, v, o));
    return v;
}
inline int __reduce_min_sync(unsigned m, int v) { return da_sim_reduce(m, v, [](int a, int b) { return a < b ? a : b; }); }
inline unsigned __reduce_min_sync(unsigned m, unsigned v) { return da_sim_reduce(m, v, [](unsigned a, unsigned b) { return a < b ? a : b; }); }
inline int __reduce_max_sync(unsigned m, int v) { return da_sim_reduce(m, v, [](int a, int b) { return a > b ? a : b; }); }
inline unsigned __reduce_max_sync(unsigned m, unsigned v) { return da_sim_reduce(m, v, [](unsigned a, unsigned b) { return a > b ? a : b; }); }
inline unsigned __reduce_add_sync(unsigned m, unsigned v) { return da_sim_reduce(m, v, [](unsigned a, unsigned b) { return a + b; }); }
#endif

namespace da {

enum DaisKind : int32_t {
    DK_INPUT = 0,  // opcode -1
    DK_SHIFT_ADD,  // 0 / 1
    DK_RELU,       // +-2
    DK_QUANT,      // +-3
    DK_CONST_ADD,  // 4
    DK_CONST,      // 5
    DK_MUX,        // +-6
    DK_MUL,        // 7
    DK_LOOKUP,     // 8
    DK_NOT,        // +-9 with data_low 0
    DK_REDUCE_OR,  // +-9 with data_low 1
    DK_REDUCE_AND, // +-9 with data_low 2
    DK_BITBIN,     // 10
    DK_OUTPUT,     // output column `dst` <- slot `a` (a < 0: the column is 0.0), negated if `neg`, times the scale in k2
};

// One compiled instruction.  Field use per kind:
//   dst      result slot (DK_OUTPUT: output column)
//   a, b, c  operand slots: id0, id1, condition (DK_INPUT: input column in a)
//   neg      negate operand a (+-2, +-3, +-9), operand b (opcode 1, -6); bits 0 / 1 negate a / b (10)
//   s0, s1   shift counts: quantize shift (2, 3), actual / global shift (0, 1, 10: s0), const_add shift, shift0 / shift1 (6)
//   aux0     6: the condition's dtype is signed; 8: table offset; 9 NOT: the result dtype is signed; 10: AND / OR / XOR
//   aux1     1 when the masked fast path of dx_wrap is exact for the dtype (2, 3, 6, -1); 8: table size
//   k0, k1   wrap int_min / mod (-1, 2, 3, 6); 4, 5: constant; 9: mask; 8: zero + data_high
//   k2       -1 and outputs: bits of the power-of-two scale (double); 6: unsigned-condition threshold
struct DaisInstr {
    int32_t kind, dst, a, b, c, neg, s0, s1, aux0, aux1;
    long long k0, k1, k2;
};
static_assert(sizeof(DaisInstr) == 64, "DaisInstr is 64 bytes");

__device__ __forceinline__ long long dx_shl(long long v, int s) { return (long long)((unsigned long long)v << (s & 63)); }
__device__ __forceinline__ long long dx_sar(long long v, int s) { return v >> (s & 63); }
__device__ __forceinline__ long long dx_add(long long a, long long b) { return (long long)((unsigned long long)a + (unsigned long long)b); }
__device__ __forceinline__ long long dx_sub(long long a, long long b) { return (long long)((unsigned long long)a - (unsigned long long)b); }
__device__ __forceinline__ long long dx_neg(long long a) { return (long long)(0ull - (unsigned long long)a); }
__device__ __forceinline__ long long dx_mul(long long a, long long b) { return (long long)((unsigned long long)a * (unsigned long long)b); }
__device__ __forceinline__ double dx_bits_to_double(long long b) {
    double d;
    memcpy(&d, &b, sizeof(d));
    return d;
}

// DAISInterpreter::quantize after its shift (:148-150): ((v - int_min + (|v| / mod + 1) * mod) % mod) + int_min with
// int64 wrap-around.  `fast`: the host proved mod = 2^m with 1 <= m <= 60 and -2^31 <= int_min <= 0; then for |v| < 2^61
// nothing overflows, the left operand of % is non-negative and the remainder is a mask: the same value without the
// 64-bit division.
__device__ __forceinline__ long long dx_wrap(long long v, long long int_min, long long mod, bool fast) {
    if (fast && (unsigned long long)v + (1ull << 61) < (1ull << 62))
        return ((v - int_min) & (mod - 1)) + int_min;
    const long long av = v < 0 ? dx_neg(v) : v;
    const long long t = dx_add(dx_sub(v, int_min), dx_mul(av / mod + 1, mod));
    return dx_add(t % mod, int_min);
}

// double -> int64 as the reference's x86 build converts it (cvttsd2si): NaN and everything outside [-2^63, 2^63) give
// INT64_MIN.  (cvt.rzi.s64.f64 would saturate instead.)
__device__ __forceinline__ long long dx_f2i(double f) {
    if (!(f >= -9223372036854775808.0 && f < 9223372036854775808.0))
        return (long long)0x8000000000000000ull;
    return (long long)f;
}

// Per-instruction side table of the profile / capture variants (host_dais.cuh, dais_compile_variant), read only by the
// observers below; the instruction stream itself is the one predict runs.
//   op         the op this instruction computes
//   cap_begin  its capture columns are cols[cap_begin .. cap_begin + cap_count) (duplicates in the request included)
//   quant      1 for the ops whose value passes a wrap step (-1, +-2, +-3, +-6)
//   lo, hi     the declared dtype's range, folded on the host
struct DaisObsEntry {
    int32_t op, cap_begin, cap_count, quant;
    long long lo, hi;
};
static_assert(sizeof(DaisObsEntry) == 32, "DaisObsEntry is 32 bytes");

// The observer of predict: sees nothing, costs nothing.
struct DaisNoObserver {
    static constexpr bool kActive = false;
    __device__ __forceinline__ void begin(long long, long long, bool) {}
    __device__ __forceinline__ void operator()(int, long long, long long) {}
    __device__ __forceinline__ void end() {}
};

// Runs the compiled program for one sample.  `S(k)` is a reference to the sample's slot k.  Returns the index of the
// first instruction whose table index was out of range (its result is 0), or -1; `*err_v0` receives that operand.
// `obs(pc, r, pre)` sees every result r; for the kinds with a wrap step, `pre` is the value before it (the converted
// input, the shifted operand; equal to r where relu clamps a negative operand to 0).
template <class Slots, class Obs>
__device__ __forceinline__ int dais_exec_sample(const DaisInstr *__restrict__ prog, int n_instr, const double *__restrict__ x, double *__restrict__ y, const int32_t *__restrict__ tables, Slots S, long long *err_v0, Obs &obs) {
    int first_err = -1;
    for (int pc = 0; pc < n_instr; ++pc) {
        const DaisInstr I = prog[pc];
        long long r = 0, pre = 0;
        switch (I.kind) {
        case DK_INPUT:
            pre = dx_f2i(floor(x[I.a] * dx_bits_to_double(I.k2)));
            r = dx_wrap(pre, I.k0, I.k1, I.aux1 != 0);
            break;
        case DK_SHIFT_ADD: {
            const long long v1 = S(I.a);
            const long long v2 = I.neg ? dx_neg(S(I.b)) : S(I.b);
            r = I.s0 > 0 ? dx_add(v1, dx_shl(v2, I.s0)) : dx_add(dx_shl(v1, -I.s0), v2);
            if (I.s1 > 0)
                r = dx_sar(r, I.s1);
            break;
        }
        case DK_RELU:
        case DK_QUANT: {
            const long long v = I.neg ? dx_neg(S(I.a)) : S(I.a);
            r = (I.kind == DK_RELU && v < 0) ? 0 : dx_wrap(dx_sar(v, I.s0), I.k0, I.k1, I.aux1 != 0);
            pre = (I.kind == DK_RELU && v < 0) ? 0 : dx_sar(v, I.s0);
            break;
        }
        case DK_CONST_ADD:
            r = dx_add(dx_shl(S(I.a), I.s0), I.k0);
            break;
        case DK_CONST:
            r = I.k0;
            break;
        case DK_MUX: {
            const long long vc = S(I.c);
            const bool cond = I.aux0 ? vc < 0 : vc > I.k2;
            pre = cond ? dx_shl(S(I.a), I.s0) : dx_shl(I.neg ? dx_neg(S(I.b)) : S(I.b), I.s1);
            r = dx_wrap(pre, I.k0, I.k1, I.aux1 != 0);
            break;
        }
        case DK_MUL:
            r = dx_mul(S(I.a), S(I.b));
            break;
        case DK_LOOKUP: {
            const long long v0 = S(I.a);
            const long long idx = dx_sub(v0, I.k0);
            if (idx >= 0 && idx < (long long)I.aux1)
                r = tables[(long long)I.aux0 + idx];
            else if (first_err < 0) {
                first_err = pc;
                if (err_v0)
                    *err_v0 = v0;
            }
            break;
        }
        case DK_NOT: {
            const long long v = I.neg ? dx_neg(S(I.a)) : S(I.a);
            r = I.aux0 ? ~v : (~v & I.k0);
            break;
        }
        case DK_REDUCE_OR:
            r = (I.neg ? dx_neg(S(I.a)) : S(I.a)) != 0;
            break;
        case DK_REDUCE_AND:
            r = ((I.neg ? dx_neg(S(I.a)) : S(I.a)) & I.k0) == I.k0;
            break;
        case DK_BITBIN: {
            long long v1 = (I.neg & 1) ? dx_neg(S(I.a)) : S(I.a);
            long long v2 = (I.neg & 2) ? dx_neg(S(I.b)) : S(I.b);
            if (I.s0 > 0)
                v2 = dx_shl(v2, I.s0);
            else
                v1 = dx_shl(v1, -I.s0);
            r = I.aux0 == 0 ? (v1 & v2) : I.aux0 == 1 ? (v1 | v2) : (v1 ^ v2);
            break;
        }
        case DK_OUTPUT:
            if (I.a < 0)
                y[I.dst] = 0.0;
            else {
                const long long v = I.neg ? dx_neg(S(I.a)) : S(I.a);
                y[I.dst] = (double)v * dx_bits_to_double(I.k2);
            }
            continue;
        }
        S(I.dst) = r;
        obs(pc, r, pre);
    }
    return first_err;
}

// Error word of a launch: the smallest (sample, instruction) key of a lookup out of range, ~0 when there was none.
// key = (sample0 + sample) * n_instr + pc: sample order first, then program order, as the reference with one thread
// reports it.
__device__ __forceinline__ void dais_report(unsigned long long *err, long long sample, int n_instr, int pc) {
    if (pc >= 0)
        atomicMin(err, (unsigned long long)sample * (unsigned long long)n_instr + (unsigned long long)pc);
}

// 64-bit warp minimum / maximum on the 32-bit reduction unit: the extreme high word first, then the extreme low word
// among the lanes that hold it.  Every lane gets the result.
__device__ __forceinline__ long long dx_warp_min(long long v) {
    const int hi = (int)(v >> 32);
    const int mh = __reduce_min_sync(0xffffffffu, hi);
    const unsigned ml = __reduce_min_sync(0xffffffffu, hi == mh ? (unsigned)v : 0xffffffffu);
    return (long long)(((unsigned long long)(unsigned)mh << 32) | ml);
}
__device__ __forceinline__ long long dx_warp_max(long long v) {
    const int hi = (int)(v >> 32);
    const int mh = __reduce_max_sync(0xffffffffu, hi);
    const unsigned ml = __reduce_max_sync(0xffffffffu, hi == mh ? (unsigned)v : 0u);
    return (long long)(((unsigned long long)(unsigned)mh << 32) | ml);
}

// Profile observer: per instruction, one warp's samples reduced to a 32-byte record {min, max, outside, wrapped} in
// rec[pc][warp] (`n_warps` warps in this launch), merged per op afterwards by dais_profile_merge_kernel.  Dispatch is
// warp-uniform, so every lane of a warp reaches every reduction; lanes past the launch's samples contribute nothing.
// The first value outside its range is kept per warp as the key sample * n_ops + op (sample order first, then op
// order) and folded into `*first` with one atomicMin when the warp is done.
struct DaisProfileObserver {
    static constexpr bool kActive = true;
    const DaisObsEntry *__restrict__ side;
    long long *__restrict__ rec;
    long long n_warps;
    unsigned long long *first;
    long long n_ops;
    // this thread
    long long warp, sample; // warp index in the launch; sample (in the whole call) of the warp's lane 0
    int lane;
    bool valid;
    unsigned long long key;

    __device__ __forceinline__ void begin(long long sample0, long long s, bool v) {
        lane = (int)(s & 31);
        warp = s >> 5;
        sample = sample0 + (s - lane);
        valid = v;
        key = ~0ull;
    }
    __device__ __forceinline__ void operator()(int pc, long long r, long long pre) {
        const DaisObsEntry e = side[pc];
        const long long mn = dx_warp_min(valid ? r : (long long)0x7fffffffffffffffll);
        const long long mx = dx_warp_max(valid ? r : (long long)0x8000000000000000ull);
        const unsigned out = __ballot_sync(0xffffffffu, valid && (r < e.lo || r > e.hi));
        const unsigned wr = e.quant ? __ballot_sync(0xffffffffu, valid && pre != r) : 0u;
        if (out) {
            const unsigned long long k = (unsigned long long)(sample + __ffs((int)out) - 1) * (unsigned long long)n_ops + (unsigned long long)e.op;
            key = k < key ? k : key;
        }
        if (lane < 4)
            rec[((long long)pc * n_warps + warp) * 4 + lane] = lane == 0 ? mn : lane == 1 ? mx : lane == 2 ? (long long)__popc(out) : (long long)__popc(wr);
    }
    __device__ __forceinline__ void end() {
        if (lane == 0 && key != ~0ull)
            atomicMin(first, key);
    }
};

// Capture observer: the values of the ops marked in the side table, written through to out[s][col] when they run.
struct DaisCaptureObserver {
    static constexpr bool kActive = true;
    const DaisObsEntry *__restrict__ side;
    const int32_t *__restrict__ cols;
    long long *__restrict__ out; // [n][k] of this launch
    int k;
    long long *row;

    __device__ __forceinline__ void begin(long long, long long s, bool v) { row = v ? out + s * k : nullptr; }
    __device__ __forceinline__ void operator()(int pc, long long r, long long) {
        if (!row)
            return;
        const DaisObsEntry e = side[pc];
        for (int j = 0; j < e.cap_count; ++j)
            row[cols[e.cap_begin + j]] = r;
    }
    __device__ __forceinline__ void end() {}
};

// SHARED: the CTA's slot file is [L][blockDim.x] int64 in dynamic shared memory.  Otherwise slot k of sample s is
// arena[k * stride + s] (s counted within this launch).  x / y: [n][n_in] / [n][n_out] of this launch; `sample0` is the
// index of its first sample in the whole call (error keys only).
// With an active observer every warp that holds a sample of the launch runs whole (its reductions are full-mask
// collectives): the lanes past n run the last sample, write nothing and report no lookup error.  The arena then needs
// stride >= the launch's threads.
template <bool SHARED, class Obs = DaisNoObserver>
__global__ void __launch_bounds__(256) dais_exec_kernel(const DaisInstr *__restrict__ prog, int n_instr, const double *__restrict__ x, int n_in, double *__restrict__ y, int n_out, long long n,
                                                        long long *__restrict__ arena, long long stride, const int32_t *__restrict__ tables, unsigned long long *err, long long sample0, long long *err_v0,
                                                        Obs obs = Obs()) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (Obs::kActive ? (s & ~31LL) >= n : s >= n)
        return;
    const bool valid = s < n;
    const long long sx = valid ? s : n - 1;
    Obs o = obs; // (a register copy: a reference to the parameter itself would put it in local memory)
    o.begin(sample0, s, valid);
    int pc;
    if (SHARED) {
        DA_DYN_SHARED(dais_smem);
        long long *base = reinterpret_cast<long long *>(dais_smem) + threadIdx.x;
        const int T = (int)blockDim.x;
        pc = dais_exec_sample(prog, n_instr, x + sx * n_in, y + sx * n_out, tables, [=](int k) -> long long & { return base[(long long)k * T]; }, err_v0, o);
    }
    else {
        long long *base = arena + s;
        pc = dais_exec_sample(prog, n_instr, x + sx * n_in, y + sx * n_out, tables, [=](int k) -> long long & { return base[(long long)k * stride]; }, err_v0, o);
    }
    o.end();
    if (valid)
        dais_report(err, sample0 + s, n_instr, pc);
}

// Folds the records of one profile launch (rec[n_instr][n_warps][4]) into the per-op totals [4][n_ops]: min, max,
// outside, wrapped.  One warp per instruction; each op has exactly one instruction in the profile variant, so no two
// warps touch the same total, and launches on one stream follow each other.
__global__ void __launch_bounds__(256) dais_profile_merge_kernel(const long long *__restrict__ rec, int n_instr, long long n_warps, const DaisObsEntry *__restrict__ side, long long *__restrict__ totals, int n_ops) {
    const int pc = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = (int)(threadIdx.x & 31);
    if (pc >= n_instr)
        return;
    long long mn = 0x7fffffffffffffffll, mx = (long long)0x8000000000000000ull;
    unsigned out = 0, wr = 0; // at most one launch's samples
    for (long long w = lane; w < n_warps; w += 32) {
        const long long *r = rec + ((long long)pc * n_warps + w) * 4;
        mn = r[0] < mn ? r[0] : mn;
        mx = r[1] > mx ? r[1] : mx;
        out += (unsigned)r[2];
        wr += (unsigned)r[3];
    }
    mn = dx_warp_min(mn);
    mx = dx_warp_max(mx);
    out = __reduce_add_sync(0xffffffffu, out);
    wr = __reduce_add_sync(0xffffffffu, wr);
    if (lane == 0) {
        long long *t = totals + side[pc].op;
        t[0] = mn < t[0] ? mn : t[0];
        t[n_ops] = mx > t[n_ops] ? mx : t[n_ops];
        t[2LL * n_ops] += out;
        t[3LL * n_ops] += wr;
    }
}

} // namespace da
