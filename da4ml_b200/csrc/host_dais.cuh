// host_dais.cuh -- load, validate and compile a DAIS program (the int32 words of CombLogic.to_binary) for the device
// interpreter of dais_exec.cuh.  Plain C++, no CUDA calls: everything here happens before the device is touched, and
// the CPU test harness runs it as it is.
//
// Parsing follows DAISInterpreter::load_from_binary (:10-91) and the causality check DAISInterpreter::validate
// (:429-448), with the reference's messages.  On top, everything the reference indexes unchecked and that could make
// the device read out of bounds is rejected, and the runtime errors that do not depend on the data (unknown opcode,
// bit_unary / bit_binary operation, msb_mux shift configuration) are raised here, at load time.
#pragma once
#include "dais_exec.cuh"

#include <algorithm>
#include <cmath>
#include <stdexcept>
#include <string>
#include <vector>

namespace da {

struct DaisCompiled {
    int n_in = 0, n_out = 0, n_ops = 0, n_tables = 0;
    int n_slots = 0;   // L: most values live at once
    int max_width = 0; // widest dtype of any op (the reference's max_ops_width)
    std::vector<DaisInstr> prog;
    std::vector<int32_t> tables;  // every lookup table, concatenated
    std::vector<int> op_slot;     // slot of op i, -1 for an op whose value nobody reads (not compiled)
    std::vector<int> instr_op;    // op of each instruction (-1 for outputs)
    std::vector<int32_t> table_size;
    // profile / capture variants only (dais_compile with every_op): one entry per instruction, and the capture columns
    std::vector<DaisObsEntry> obs;
    std::vector<int32_t> cap_cols;
};

namespace dais_detail {
// the reference computes these in int32; C++ overflow there is the x86 wrap-around
inline int32_t wadd(int32_t a, int32_t b) { return (int32_t)((uint32_t)a + (uint32_t)b); }
inline int32_t wsub(int32_t a, int32_t b) { return (int32_t)((uint32_t)a - (uint32_t)b); }
inline int32_t wneg(int32_t a) { return (int32_t)(0u - (uint32_t)a); }
struct Op {
    int32_t opcode, id0, id1, data_low, data_high, is_signed, integers, fractionals;
    int32_t width() const { return wadd(wadd(integers, fractionals), is_signed ? 1 : 0); }
    long long int_min() const { return is_signed ? (long long)wneg((int32_t)(1u << ((uint32_t)wsub(width(), 1) & 31))) : 0; }
    long long mod() const { return (long long)(1ull << ((uint32_t)width() & 63)); }
    bool fast_wrap() const {
        const int32_t w = width();
        return w >= 1 && w <= 60; // mod = 2^w, |int_min| <= 2^31: see dx_wrap
    }
};
inline std::string s(long long v) { return std::to_string(v); }
inline bool reads_id0(int opc) { return opc != -1 && opc != 5; }
inline bool reads_id1(int opc) { return opc == 0 || opc == 1 || opc == 6 || opc == -6 || opc == 7 || opc == 10; }
inline bool wraps(int opc) { return opc == -1 || std::abs(opc) == 2 || std::abs(opc) == 3 || std::abs(opc) == 6; }
} // namespace dais_detail

// The range of a declared dtype, with w = is_signed + integers + fractionals in 64-bit (not the reference's int32):
// w <= 0 holds only 0; 1 <= w <= 63 the usual two's-complement or unsigned range; w >= 64 is unbounded (unsigned: >= 0).
inline void dais_dtype_range(int32_t is_signed, int32_t integers, int32_t fractionals, long long &lo, long long &hi) {
    const long long w = (is_signed ? 1LL : 0LL) + integers + fractionals;
    if (w <= 0)
        lo = hi = 0;
    else if (w >= 64) {
        lo = is_signed ? (long long)0x8000000000000000ull : 0;
        hi = 0x7fffffffffffffffll;
    }
    else if (is_signed) {
        lo = -(1LL << (w - 1));
        hi = (1LL << (w - 1)) - 1;
    }
    else {
        lo = 0;
        hi = (long long)((1ull << w) - 1);
    }
}

// Parse, validate and compile.  Throws std::runtime_error with the reference's message where it has one.
// `every_op` compiles the profile / capture variant: every op runs, as in the reference (none is skipped for want of
// a reader), no output instructions are emitted, and each instruction gets a side-table entry (P.obs).  The ops listed
// in `capture` (duplicates allowed) are marked for the capture observer, column j for capture[j]; like outputs, they
// are written through when they run and do not lengthen any slot's lifetime.
inline DaisCompiled dais_compile(const int32_t *w, long long n_words, bool every_op = false, const int32_t *capture = nullptr, int n_capture = 0) {
    using namespace dais_detail;
    if (!w || n_words < 6)
        throw std::runtime_error("Binary data too small to contain valid DAIS model file");
    if (w[0] != 1)
        throw std::runtime_error("DAIS version mismatch: expected version 1, got version " + s(w[0]));
    DaisCompiled P;
    P.n_in = w[2], P.n_out = w[3], P.n_ops = w[4], P.n_tables = w[5];
    if (P.n_in < 0 || P.n_out < 0 || P.n_ops < 0 || P.n_tables < 0)
        throw std::runtime_error("Binary data header holds a negative count");
    const long long table_offset = 6 + (long long)P.n_in + 3LL * P.n_out + 8LL * P.n_ops;
    long long expect = table_offset;
    if (P.n_tables > 0 && table_offset + P.n_tables > n_words) // (the reference reads the table sizes past the end)
        throw std::runtime_error("Binary data size mismatch: expected at least " + s((table_offset + P.n_tables) * 4) + " bytes , got " + s(n_words * 4) + " bytes");
    for (int t = 0; t < P.n_tables; ++t) {
        if (w[table_offset + t] < 0)
            throw std::runtime_error("Binary data holds a negative size for lookup table " + s(t));
        expect += 1 + (long long)w[table_offset + t];
    }
    if (expect != n_words)
        throw std::runtime_error("Binary data size mismatch: expected " + s(expect * 4) + " bytes , got " + s(n_words * 4) + " bytes");
    const int32_t *inp_shifts = w + 6, *out_idxs = inp_shifts + P.n_in, *out_shifts = out_idxs + P.n_out, *out_negs = out_shifts + P.n_out;
    const Op *ops = reinterpret_cast<const Op *>(out_negs + P.n_out);
    std::vector<long long> table_begin(P.n_tables + 1, 0);
    for (int t = 0; t < P.n_tables; ++t) {
        P.table_size.push_back(w[table_offset + t]);
        table_begin[t + 1] = table_begin[t] + w[table_offset + t];
    }
    if (table_begin[P.n_tables] > 0x7fffffffLL)
        throw std::runtime_error("lookup tables larger than 2^31 entries are not supported");
    P.tables.assign(w + table_offset + P.n_tables, w + n_words);
    const int n = P.n_ops;
    for (int i = 0; i < n; ++i) { // DAISInterpreter::validate (:429-448)
        const Op &op = ops[i];
        P.max_width = std::max(P.max_width, op.width());
        if (op.id0 >= i && op.opcode != -1)
            throw std::runtime_error("Operation " + s(i) + " has id0=" + s(op.id0) + "violating causality");
        if (op.id1 >= i)
            throw std::runtime_error("Operation " + s(i) + " has id1=" + s(op.id1) + " violating causality");
        if (std::abs(op.opcode) == 6 && (unsigned)op.data_low >= (unsigned)i)
            throw std::runtime_error("Operation " + s(i) + " has cond_idx=" + s(op.data_low) + " violating causality");
    }
    // what the reference indexes unchecked, and the runtime errors that do not depend on the data
    for (int i = 0; i < n; ++i) {
        const Op &op = ops[i];
        const int opc = op.opcode;
        switch (opc) {
        case -1: case 0: case 1: case 2: case -2: case 3: case -3: case 4: case 5: case 6: case -6: case 7: case 8: case 9: case -9: case 10:
            break;
        default:
            throw std::runtime_error("Unknown opcode: " + s(opc) + " at index " + s(i));
        }
        if (opc == -1 && (op.id0 < 0 || op.id0 >= P.n_in))
            throw std::runtime_error("input index out of range at operation " + s(i));
        if ((reads_id0(opc) && op.id0 < 0) || (reads_id1(opc) && op.id1 < 0))
            throw std::runtime_error("negative operand index at operation " + s(i));
        if (opc == 8 && (op.data_low < 0 || op.data_low >= P.n_tables))
            throw std::runtime_error("lookup table index out of range at operation " + s(i));
        if ((opc == 9 || opc == -9) && (op.data_low < 0 || op.data_low > 2))
            throw std::runtime_error("Unknown bit unary operation with data_low=" + s(op.data_low));
        if (opc == 10 && (op.data_high >> 24 < 0 || op.data_high >> 24 > 2))
            throw std::runtime_error("Unknown bit binary operation with data_low=" + s(op.data_low));
        if (opc == 6 || opc == -6) {
            const int32_t shift1 = wadd(wsub(op.fractionals, ops[op.id1].fractionals), op.data_high);
            const int32_t shift0 = wsub(op.fractionals, ops[op.id0].fractionals);
            if (shift1 != 0 && shift0 != 0)
                throw std::runtime_error("Unsupported msb_mux shift configuration: shift0=" + s(shift0) + ", shift1=" + s(shift1));
        }
    }
    for (int o = 0; o < P.n_out; ++o)
        if (out_idxs[o] < -1 || out_idxs[o] >= n)
            throw std::runtime_error("output index out of range at output " + s(o));
    if (n_capture > 0 && !every_op)
        throw std::logic_error("ops are captured by the every-op variant only");
    std::vector<std::vector<int>> cols_of(every_op ? n : 0);
    for (int j = 0; j < n_capture; ++j) {
        if (capture[j] < 0 || capture[j] >= n)
            throw std::runtime_error("op index " + s(capture[j]) + " out of range [0, " + s(n) + ")");
        cols_of[capture[j]].push_back(j);
    }

    // liveness: last reader of every value; outputs are written through when their op runs and do not extend it
    std::vector<int> last_use(n, -1);
    std::vector<char> is_out(n, 0);
    for (int i = 0; i < n; ++i) {
        const Op &op = ops[i];
        if (reads_id0(op.opcode))
            last_use[op.id0] = i;
        if (reads_id1(op.opcode))
            last_use[op.id1] = i;
        if (std::abs(op.opcode) == 6)
            last_use[op.data_low] = i;
    }
    std::vector<std::vector<int>> outs_of(n);
    for (int o = 0; o < P.n_out; ++o)
        if (out_idxs[o] >= 0) {
            is_out[out_idxs[o]] = 1;
            outs_of[out_idxs[o]].push_back(o);
        }
    P.op_slot.assign(n, -1);
    std::vector<int> free_slots;
    auto release = [&](int v, int i) {
        if (v >= 0 && v < n && P.op_slot[v] >= 0 && last_use[v] == i) {
            free_slots.push_back(P.op_slot[v]);
            last_use[v] = -2; // (an op may read one value twice)
        }
    };
    for (int o = 0; o < P.n_out && !every_op; ++o)
        if (out_idxs[o] < 0) {
            DaisInstr I{};
            I.kind = DK_OUTPUT, I.dst = o, I.a = -1;
            P.prog.push_back(I);
            P.instr_op.push_back(-1);
        }
    for (int i = 0; i < n; ++i) {
        const Op &op = ops[i];
        const int opc = op.opcode;
        // a value nobody reads is not computed; a lookup still is (its index check is observable)
        if (!every_op && last_use[i] < 0 && !is_out[i] && opc != 8)
            continue;
        DaisInstr I{};
        auto slot = [&](int v) { return P.op_slot[v]; };
        auto set_wrap = [&](const Op &to) {
            I.k0 = to.int_min();
            I.k1 = to.mod();
            I.aux1 = to.fast_wrap() ? 1 : 0;
        };
        switch (opc) {
        case -1: {
            I.kind = DK_INPUT;
            I.a = op.id0;
            const double scale = std::pow(2.0, (double)wadd(inp_shifts[op.id0], op.fractionals));
            memcpy(&I.k2, &scale, 8);
            set_wrap(op);
            break;
        }
        case 0: case 1: {
            const Op &o0 = ops[op.id0], &o1 = ops[op.id1];
            I.kind = DK_SHIFT_ADD;
            I.a = slot(op.id0), I.b = slot(op.id1), I.neg = opc == 1;
            I.s0 = wsub(wadd(op.data_low, o0.fractionals), o1.fractionals);
            I.s1 = wsub(std::max(o0.fractionals, wsub(o1.fractionals, op.data_low)), op.fractionals);
            break;
        }
        case 2: case -2: case 3: case -3:
            I.kind = std::abs(opc) == 2 ? DK_RELU : DK_QUANT;
            I.a = slot(op.id0), I.neg = opc < 0;
            I.s0 = wsub(ops[op.id0].fractionals, op.fractionals);
            set_wrap(op);
            break;
        case 4:
            I.kind = DK_CONST_ADD;
            I.a = slot(op.id0);
            I.s0 = wsub(op.fractionals, ops[op.id0].fractionals);
            I.k0 = (long long)(((unsigned long long)(uint32_t)op.data_high << 32) | (uint32_t)op.data_low);
            break;
        case 5:
            I.kind = DK_CONST;
            I.k0 = (long long)(((unsigned long long)(uint32_t)op.data_high << 32) | (uint32_t)op.data_low);
            break;
        case 6: case -6: {
            const Op &oc = ops[op.data_low];
            I.kind = DK_MUX;
            I.a = slot(op.id0), I.b = slot(op.id1), I.c = slot(op.data_low), I.neg = opc < 0;
            I.s0 = wsub(op.fractionals, ops[op.id0].fractionals);
            I.s1 = wadd(wsub(op.fractionals, ops[op.id1].fractionals), op.data_high);
            I.aux0 = oc.is_signed ? 1 : 0;
            I.k2 = std::max((long long)(1ull << ((uint32_t)wsub(oc.width(), 2) & 63)), 0LL); // get_msb :180, as written
            set_wrap(op);
            break;
        }
        case 7:
            I.kind = DK_MUL;
            I.a = slot(op.id0), I.b = slot(op.id1);
            break;
        case 8: {
            const Op &o0 = ops[op.id0];
            I.kind = DK_LOOKUP;
            I.a = slot(op.id0);
            const long long zero = (long long)((unsigned long long)(long long)wneg(o0.is_signed) * (1ull << ((uint32_t)wsub(o0.width(), 1) & 63)));
            I.k0 = (long long)((unsigned long long)zero + (unsigned long long)(long long)op.data_high);
            I.k1 = zero;
            I.aux0 = (int32_t)table_begin[op.data_low];
            I.aux1 = P.table_size[op.data_low];
            break;
        }
        case 9: case -9:
            I.kind = op.data_low == 0 ? DK_NOT : op.data_low == 1 ? DK_REDUCE_OR : DK_REDUCE_AND;
            I.a = slot(op.id0), I.neg = opc < 0;
            I.aux0 = op.is_signed ? 1 : 0;
            I.k0 = (long long)((1ull << ((uint32_t)ops[op.id0].width() & 63)) - 1);
            break;
        case 10:
            I.kind = DK_BITBIN;
            I.a = slot(op.id0), I.b = slot(op.id1), I.neg = op.data_high & 3;
            I.s0 = wsub(wadd(op.data_low, ops[op.id0].fractionals), ops[op.id1].fractionals);
            I.aux0 = op.data_high >> 24;
            break;
        }
        // operands whose last reader this is give their slots back before the result takes one
        if (reads_id0(opc))
            release(op.id0, i);
        if (reads_id1(opc))
            release(op.id1, i);
        if (std::abs(opc) == 6)
            release(op.data_low, i);
        if (free_slots.empty())
            free_slots.push_back(P.n_slots++);
        P.op_slot[i] = I.dst = free_slots.back();
        free_slots.pop_back();
        P.prog.push_back(I);
        P.instr_op.push_back(i);
        if (every_op) {
            DaisObsEntry E{};
            E.op = i, E.cap_begin = (int32_t)P.cap_cols.size(), E.cap_count = (int32_t)cols_of[i].size(), E.quant = wraps(opc) ? 1 : 0;
            dais_dtype_range(op.is_signed, op.integers, op.fractionals, E.lo, E.hi);
            P.obs.push_back(E);
            P.cap_cols.insert(P.cap_cols.end(), cols_of[i].begin(), cols_of[i].end());
            if (last_use[i] < 0)
                free_slots.push_back(P.op_slot[i]);
            continue;
        }
        for (int o : outs_of[i]) {
            DaisInstr O{};
            O.kind = DK_OUTPUT, O.dst = o, O.a = P.op_slot[i], O.neg = out_negs[o] != 0;
            const double scale = std::pow(2.0, (double)wsub(out_shifts[o], op.fractionals));
            memcpy(&O.k2, &scale, 8);
            P.prog.push_back(O);
            P.instr_op.push_back(-1);
        }
        if (last_use[i] < 0) // written through to the outputs, or a lookup nobody reads
            free_slots.push_back(P.op_slot[i]);
    }
    return P;
}

// "Logic lookup index out of bounds: ..." of DAISInterpreter::logic_lookup (:228-234) for instruction `pc`, operand v0
inline std::string dais_lookup_message(const DaisCompiled &P, int pc, long long v0) {
    const DaisInstr &I = P.prog[pc];
    const long long zero = I.k1, data_high = (long long)((unsigned long long)I.k0 - (unsigned long long)zero);
    const long long index = (long long)((unsigned long long)v0 - (unsigned long long)I.k0);
    return "Logic lookup index out of bounds: index=" + std::to_string(index) + ", table_size=" + std::to_string(I.aux1) + ", zero=" + std::to_string(zero) +
           ", data_high=" + std::to_string(data_high) + ", v0=" + std::to_string(v0);
}

// Samples per CTA in the shared regime: the largest multiple of 32 (at most 256) whose [L][T] int64 slot file fits
// `budget` bytes; 0 selects the global regime.
inline int dais_shared_tile(int n_slots, long long budget) {
    const long long per_sample = 8LL * std::max(n_slots, 1);
    const long long t = std::min<long long>(256, budget / per_sample / 32 * 32);
    return (int)std::max<long long>(t, 0);
}

// Samples per launch of a profile run: at most `chunk`, a multiple of 256, and few enough that the per-warp records
// (32 bytes per instruction and warp of 32 samples: n_instr bytes per sample) fit `record_bytes`.
inline long long dais_profile_chunk(long long n_instr, long long chunk, long long record_bytes) {
    return std::max<long long>(256, std::min(chunk, record_bytes / std::max(n_instr, 1LL) / 256 * 256));
}

} // namespace da
