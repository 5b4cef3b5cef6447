// solve_owned.cuh -- the greedy step in the owner-partitioned formulation.
//
// Expression e is owned by CTA e mod G of its group.  Two views of the live digits are kept:
//   * cells (global memory): per expression, the list of (column, P, N) of its digits.  Written by the owner, read by
//     every CTA of the group when the expression is chosen: each CTA rebuilds the dense rows of c0 and c1 in shared
//     memory and computes the substitution for all columns itself (update_expr, state_opr.cc:227-283).
//   * owner lists (shared memory of the owner, private): for every output column the rows (e / G, P, N) of the owned
//     expressions that have digits there.  The recount (update_stats, state_opr.cc:307-340) walks the lists of the
//     columns the rewritten rows touch -- work proportional to the rows of those columns -- and counts digit pairs in
//     a shared-memory hash table keyed by (owned expression, rewritten row, shift, sub).  A pair count is a sum over
//     columns, and all columns of an owned expression are in its owner's lists, so the counts are complete inside one
//     CTA: no cross-CTA counters, no L2 atomics, no harvest exchange.  Entries with count >= 2 go to the CTA's own
//     histogram segment.
// One group exchange per step (the argmax).
#pragma once
#include "solve_common.cuh"

namespace da {

// global workspace of one group
struct OwnWs {
    // cells of the expressions a CTA owns, bump-allocated from its slice [rank * pool_cap, (rank + 1) * pool_cap):
    // column + two versions of the sign planes.  Other CTAs read the cells of c0 / c1 at the start of a step while the
    // owner rewrites them later in the same step, so a rewrite goes to the other version; which version is current is
    // the parity of the number of rewrites of the expression, which every CTA tracks in a private shared-memory bitmap.
    uint32_t *cell_col; // [G * pool_cap]
    uint2 *cell_pl[2];  // [G * pool_cap] each
    uint2 *cell_dir;    // [e_cap] (first cell (absolute index), cells allocated; dead cells keep empty planes)
    uint32_t *ovf;      // [G][n_out_max][3][ovf_cap] rows of an owner list beyond its shared-memory capacity
    int *col_len_g;     // [n_out_max] lengths of the global column lists handed to the adder trees
    int pool_cap, e_cap, ovf_cap, n_out_max;
};

#define DA_OWN_STACK 48
// per-CTA scalars of the step (static shared memory)
struct OwnBlock {
    int pool_used;   // cells handed out of this CTA's pool slice
    int n_mods;      // rewritten rows of this step: 2 (self pair) or 3
    uint32_t mid[3]; // their ids, ascending: c0, (c1,) new
    QInt mq[3];      // their op records
    float ml[3];
    int new_cells;   // nonzero columns of the new row
    int n_tcol;      // columns touched by the rewritten rows
    int n_ins;       // hash slots claimed in the current pass
    int overflow;    // the current pass ran out of hash slots
    int pass_bits;   // the owned expressions are counted in 2^pass_bits subsets (adapted from step to step)
    int grew;        // a subset had to be split in this step
    int ins_max;     // most slots claimed by one pass of this step
    int sub_top;
    int splits;      // counting passes abandoned and split in two (whole problem)
#ifdef DA_RECOUNT_PROF
    long long xphase[4], xt; // development build: cycles of thread 0 in the parts of the recount (setup, counting, harvest)
#endif
    uint32_t sub_stack[DA_OWN_STACK]; // pending subsets: (bits << 16) | value -> expressions with (e / G) mod 2^bits == value
};

// shared-memory layout of one CTA, as byte offsets into the dynamic shared memory (so that accesses compile to LDS / STS)
struct OwnLayout {
    uint32_t D[3];    // uint2[n_out_max] dense rows of the rewritten expressions after the substitution (D[1] = new row for a self pair)
    uint32_t B[3];    // uint32[words] their column bitmaps
    uint32_t A;       // uint32[words] union of the three
    uint32_t pre;     // uint32[words] exclusive prefix of popc(B[new])
    uint32_t ver;     // uint32[ceil(e_cap / 32)] rewrite parity of every expression
    uint32_t col_len; // int[n_out_max] rows of each owner list
    uint32_t tcol;    // uint16[n_out_max] touched columns of the step
    uint32_t tpre;    // int[n_out_max + 1] exclusive prefix of their list lengths
    uint32_t lists;   // [n_out_max][lcap] rows: 6 bytes each when `narrow` (u16 index array, then u32 P | N << 16), else three uint32 arrays
    uint32_t hkey;    // uint32[1 << hlog] key + 1 (0 = empty)
    uint32_t hval;    // uint32[1 << hlog] count
    uint32_t hins;    // uint16[1 << hlog] claimed slots of the pass
    int lcap, hlog, words;
    int narrow;       // shared-memory list rows are 6 bytes (owned index and planes fit 16 bits each)
};

struct OwnCtx {
    OwnWs ws;
    OwnLayout lay;
    OwnBlock *ob;
    uint32_t *ovf; // this CTA's overflow rows
};

#define DA_SM(type, off) ((type *)(da_smem + (off)))
// development build (-DDA_RECOUNT_PROF, scripts/dev_prof_variant.sh): thread 0 of the counting team times the parts of
// the recount; the kernel prints them at the milestones of CTA 0
#ifdef DA_RECOUNT_PROF
#define DA_XLAP(k)                                 \
    if (tm.tid == 0) {                             \
        const long long _n = clock64();            \
        ox.ob->xphase[k] += _n - ox.ob->xt;        \
        ox.ob->xt = _n;                            \
    }
#else
#define DA_XLAP(k)
#endif

struct OwnRow {
    uint32_t j, P, N; // owned expression j * G + rank, sign planes
};
// Rows of an owner list: the first lcap in shared memory -- 6 bytes each (16-bit owned index, two 16-bit planes) when the
// problem allows it (`narrow`), else three words --, the rest in this CTA's spill area in global memory (three words).
__device__ __forceinline__ OwnRow own_row_load(const OwnCtx &ox, int o, int k) {
    DA_DYN_SHARED(da_smem);
    OwnRow r;
    const int lcap = ox.lay.lcap;
    if (k < lcap) {
        if (ox.lay.narrow) {
            const unsigned char *b = da_smem + ox.lay.lists + (size_t)o * 6 * lcap;
            r.j = ((const uint16_t *)b)[k];
            const uint32_t pn = ((const uint32_t *)(b + 2 * lcap))[k];
            r.P = pn & 0xffffu, r.N = pn >> 16;
        }
        else {
            const uint32_t *b = DA_SM(uint32_t, ox.lay.lists) + (size_t)o * 3 * lcap;
            r.j = b[k], r.P = b[lcap + k], r.N = b[2 * lcap + k];
        }
    }
    else {
        const int oc = ox.ws.ovf_cap;
        const uint32_t *b = ox.ovf + (size_t)o * 3 * oc;
        r.j = b[k - lcap], r.P = b[oc + k - lcap], r.N = b[2 * oc + k - lcap];
    }
    return r;
}
__device__ __forceinline__ void own_row_store(const OwnCtx &ox, int o, int k, uint32_t j, uint32_t P, uint32_t N) {
    DA_DYN_SHARED(da_smem);
    const int lcap = ox.lay.lcap;
    if (k < lcap) {
        if (ox.lay.narrow) {
            unsigned char *b = da_smem + ox.lay.lists + (size_t)o * 6 * lcap;
            ((uint16_t *)b)[k] = (uint16_t)j;
            ((uint32_t *)(b + 2 * lcap))[k] = P | (N << 16);
        }
        else {
            uint32_t *b = DA_SM(uint32_t, ox.lay.lists) + (size_t)o * 3 * lcap;
            b[k] = j, b[lcap + k] = P, b[2 * lcap + k] = N;
        }
    }
    else {
        const int oc = ox.ws.ovf_cap;
        uint32_t *b = ox.ovf + (size_t)o * 3 * oc;
        b[k - lcap] = j, b[oc + k - lcap] = P, b[2 * oc + k - lcap] = N;
    }
}
__device__ __forceinline__ void own_row_planes(const OwnCtx &ox, int o, int k, uint32_t P, uint32_t N) {
    DA_DYN_SHARED(da_smem);
    const int lcap = ox.lay.lcap;
    if (k < lcap) {
        if (ox.lay.narrow) {
            unsigned char *b = da_smem + ox.lay.lists + (size_t)o * 6 * lcap;
            ((uint32_t *)(b + 2 * lcap))[k] = P | (N << 16);
        }
        else {
            uint32_t *b = DA_SM(uint32_t, ox.lay.lists) + (size_t)o * 3 * lcap;
            b[lcap + k] = P, b[2 * lcap + k] = N;
        }
    }
    else {
        const int oc = ox.ws.ovf_cap;
        uint32_t *b = ox.ovf + (size_t)o * 3 * oc;
        b[oc + k - lcap] = P, b[2 * oc + k - lcap] = N;
    }
}

// update_expr for one column on sign planes (state_opr.cc:227-283); planes are updated in place, the new row returned
__device__ __forceinline__ void substitute_planes(uint32_t &P0, uint32_t &N0, uint32_t &P1, uint32_t &N1, bool self, int shift, int sub, int nbits, uint32_t &Pn, uint32_t &Nn) {
    Pn = 0u, Nn = 0u;
    if (!self) {
        const bool flip = shift < 0;
        const int rel = flip ? -shift : shift;
        const uint32_t AP = flip ? P1 : P0, AN = flip ? N1 : N0; // expr0 after the reference's swap
        const uint32_t BP = flip ? P0 : P1, BN = flip ? N0 : N1;
        const uint32_t M = sub ? ((AP & (BN >> rel)) | (AN & (BP >> rel))) : ((AP & (BP >> rel)) | (AN & (BN >> rel)));
        const uint32_t MB = M << rel;
        if (!flip) { // the new digit takes position and sign of id0's digit
            Pn = AP & M, Nn = AN & M;
            P0 = AP & ~M, N0 = AN & ~M, P1 = BP & ~MB, N1 = BN & ~MB;
        }
        else {
            Pn = BP & MB, Nn = BN & MB;
            P1 = AP & ~M, N1 = AN & ~M, P0 = BP & ~MB, N0 = BN & ~MB;
        }
    }
    else { // self pair (always shift < 0): order-dependent greedy matching with tombstones
        const int rel = -shift;
        const uint32_t live = P0 | N0;
        uint32_t tomb = 0u;
        for (uint32_t m = live; m; m &= m - 1) {
            const int pl = __ffs(m) - 1;
            if ((tomb >> pl) & 1u)
                continue;
            const int q = pl + rel;
            if (q >= nbits || q >= 32)
                continue;
            if (!((live >> q) & 1u) || ((tomb >> q) & 1u))
                continue;
            if ((int)(((N0 >> pl) ^ (N0 >> q)) & 1u) != sub)
                continue;
            if ((N0 >> q) & 1u)
                Nn |= 1u << q;
            else
                Pn |= 1u << q;
            tomb |= (1u << pl) | (1u << q);
        }
        P0 &= ~tomb, N0 &= ~tomb;
        P1 = P0, N1 = N0;
    }
}

// ---- initial state (state_opr.cc:100-112): owner lists (warp per column) and cells (warp per owned input) ----------
__device__ void own_init(const ProblemDesc &p, const Ctx &cx, const OwnCtx &ox) {
    DA_DYN_SHARED(da_smem);
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, wid = tid >> 5, nw = nt >> 5, G = cx.cfg.G;
    OwnBlock &ob = *ox.ob;
    int *col_len = DA_SM(int, ox.lay.col_len);
    uint32_t *ver = DA_SM(uint32_t, ox.lay.ver);
    for (int i = tid; i < (p.e_cap + 31) / 32; i += nt)
        ver[i] = 0u;
    const int n_own = p.n_in > cx.rank ? (p.n_in - cx.rank + G - 1) / G : 0; // owned inputs: rank, rank + G, ...
    const int cap = ox.lay.lcap + ox.ws.ovf_cap;
    for (int o = wid; o < p.n_out; o += nw) {
        int cnt = 0;
        for (int j0 = 0; j0 < n_own; j0 += 32) {
            const int j = j0 + lane;
            uint2 m = make_uint2(0u, 0u);
            if (j < n_own)
                m = p.masks0[(size_t)(j * G + cx.rank) * p.n_out + o];
            const bool on = (m.x | m.y) != 0u;
            const unsigned bal = __ballot_sync(0xffffffffu, on);
            const int pos = cnt + __popc(bal & ((1u << lane) - 1u));
            if (on) {
                if (pos < cap)
                    own_row_store(ox, o, pos, (uint32_t)j, m.x, m.y);
                else
                    cx.b->status = ST_LIST_OVERFLOW;
            }
            cnt += __popc(bal);
        }
        if (lane == 0) {
            col_len[o] = min(cnt, cap);
            atomicMax(&cx.b->list_max, min(cnt, cap));
        }
    }
    const size_t pool = (size_t)cx.rank * ox.ws.pool_cap;
    for (int i = cx.rank + G * wid; i < p.n_in; i += G * nw) {
        const uint2 *row = p.masks0 + (size_t)i * p.n_out;
        int cnt = 0;
        for (int o0 = 0; o0 < p.n_out; o0 += 32) {
            const int o = o0 + lane;
            const uint2 m = o < p.n_out ? row[o] : make_uint2(0u, 0u);
            cnt += __popc(__ballot_sync(0xffffffffu, (m.x | m.y) != 0u));
        }
        int off = 0;
        if (lane == 0) {
            off = smem_add(&ob.pool_used, cnt);
            if (off + cnt > ox.ws.pool_cap) {
                cx.b->status = ST_LIST_OVERFLOW;
                cnt = 0;
            }
            ox.ws.cell_dir[i] = make_uint2((uint32_t)(pool + off), (uint32_t)cnt);
        }
        off = __shfl_sync(0xffffffffu, off, 0);
        cnt = __shfl_sync(0xffffffffu, cnt, 0);
        int k = 0;
        for (int o0 = 0; o0 < p.n_out; o0 += 32) {
            const int o = o0 + lane;
            const uint2 m = o < p.n_out ? row[o] : make_uint2(0u, 0u);
            const bool on = (m.x | m.y) != 0u && cnt > 0;
            const unsigned bal = __ballot_sync(0xffffffffu, on);
            if (on) {
                const size_t ci = pool + off + k + __popc(bal & ((1u << lane) - 1u));
                ox.ws.cell_col[ci] = (uint32_t)o;
                ox.ws.cell_pl[0][ci] = m; // version 0
            }
            k += __popc(bal);
        }
    }
}

// ---- A. dense rows of c0 / c1 from their cells, the substitution in every column, bitmaps of the three new rows -----
__device__ void own_substitute(const ProblemDesc &p, const Ctx &cx, const OwnCtx &ox, const Team &tm, uint32_t c0, uint32_t c1, int shift, int sub) {
    DA_DYN_SHARED(da_smem);
    const int tid = tm.tid, nt = tm.nt, lane = tid & 31, wid = tid >> 5, nw = nt >> 5;
    const bool self = c0 == c1;
    uint2 *D0 = DA_SM(uint2, ox.lay.D[0]), *D1 = self ? D0 : DA_SM(uint2, ox.lay.D[1]), *Dn = DA_SM(uint2, ox.lay.D[self ? 1 : 2]);
    uint32_t *ver = DA_SM(uint32_t, ox.lay.ver);
    // (the directory entries and the first cells are requested before the rows are cleared: their latency overlaps)
    const uint2 dir0 = __ldcg(&ox.ws.cell_dir[c0]);
    const uint2 dir1 = self ? dir0 : __ldcg(&ox.ws.cell_dir[c1]);
    const uint2 *pl0 = ox.ws.cell_pl[(ver[c0 >> 5] >> (c0 & 31)) & 1u];
    const uint2 *pl1 = ox.ws.cell_pl[(ver[c1 >> 5] >> (c1 & 31)) & 1u];
    uint2 a0 = make_uint2(0u, 0u), a1 = make_uint2(0u, 0u);
    uint32_t k0 = 0u, k1 = 0u;
    if ((uint32_t)tid < dir0.y) {
        a0 = __ldcg(&pl0[dir0.x + tid]);
        k0 = __ldcg(&ox.ws.cell_col[dir0.x + tid]);
    }
    if (!self && (uint32_t)tid < dir1.y) {
        a1 = __ldcg(&pl1[dir1.x + tid]);
        k1 = __ldcg(&ox.ws.cell_col[dir1.x + tid]);
    }
    for (int o = tid; o < p.n_out; o += nt) {
        DA_SM(uint2, ox.lay.D[0])[o] = make_uint2(0u, 0u);
        DA_SM(uint2, ox.lay.D[1])[o] = make_uint2(0u, 0u);
        DA_SM(uint2, ox.lay.D[2])[o] = make_uint2(0u, 0u);
    }
    team_sync(tm);
    if ((uint32_t)tid < dir0.y)
        D0[k0] = a0;
    if (!self && (uint32_t)tid < dir1.y)
        D1[k1] = a1;
    for (uint32_t i = tid + nt; i < dir0.y; i += nt)
        D0[__ldcg(&ox.ws.cell_col[dir0.x + i])] = __ldcg(&pl0[dir0.x + i]);
    if (!self)
        for (uint32_t i = tid + nt; i < dir1.y; i += nt)
            D1[__ldcg(&ox.ws.cell_col[dir1.x + i])] = __ldcg(&pl1[dir1.x + i]);
    team_sync(tm);
    const int n_pad = (p.n_out + 31) & ~31;
    for (int o0 = wid * 32; o0 < n_pad; o0 += nw * 32) {
        const int o = o0 + lane;
        uint32_t P0 = 0u, N0 = 0u, P1 = 0u, N1 = 0u, Pn = 0u, Nn = 0u;
        if (o < p.n_out) {
            const uint2 a = D0[o], c = D1[o];
            P0 = a.x, N0 = a.y, P1 = c.x, N1 = c.y;
            if ((P0 | N0) != 0u && (P1 | N1) != 0u)
                substitute_planes(P0, N0, P1, N1, self, shift, sub, p.nbits, Pn, Nn);
            D0[o] = make_uint2(P0, N0);
            if (!self)
                D1[o] = make_uint2(P1, N1);
            Dn[o] = make_uint2(Pn, Nn);
        }
        const unsigned b0 = __ballot_sync(0xffffffffu, (P0 | N0) != 0u);
        const unsigned b1 = __ballot_sync(0xffffffffu, (P1 | N1) != 0u);
        const unsigned bn = __ballot_sync(0xffffffffu, (Pn | Nn) != 0u);
        if (lane == 0) {
            const int w = o0 >> 5;
            DA_SM(uint32_t, ox.lay.B[0])[w] = b0;
            if (!self)
                DA_SM(uint32_t, ox.lay.B[1])[w] = b1;
            DA_SM(uint32_t, ox.lay.B[self ? 1 : 2])[w] = bn;
            DA_SM(uint32_t, ox.lay.A)[w] = b0 | b1 | bn;
        }
    }
    team_sync(tm);
    if (wid == 0) {
        // exclusive prefix over the new row's bitmap words (cell positions of the new expression) and the compact list
        // of touched columns; this CTA's view of the versions: c0 and c1 have now been rewritten once more (everybody
        // read the old ones above)
        const uint32_t *Bn = DA_SM(uint32_t, ox.lay.B[self ? 1 : 2]), *A = DA_SM(uint32_t, ox.lay.A);
        uint32_t *pre = DA_SM(uint32_t, ox.lay.pre);
        uint16_t *tcol = DA_SM(uint16_t, ox.lay.tcol);
        const int words = (p.n_out + 31) >> 5;
        int acc = 0, nt_col = 0;
        for (int w0 = 0; w0 < words; w0 += 32) {
            const int w = w0 + lane;
            const uint32_t bw = w < words ? Bn[w] : 0u, aw = w < words ? A[w] : 0u;
            int cn = __popc(bw), ca = __popc(aw);
            int in = cn, ia = ca;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const int vn = __shfl_up_sync(0xffffffffu, in, off), va = __shfl_up_sync(0xffffffffu, ia, off);
                if (lane >= off)
                    in += vn, ia += va;
            }
            if (w < words)
                pre[w] = (uint32_t)(acc + in - cn);
            int pos = nt_col + ia - ca;
            for (uint32_t m = aw; m; m &= m - 1)
                tcol[pos++] = (uint16_t)((w << 5) + __ffs(m) - 1);
            acc += __shfl_sync(0xffffffffu, in, 31);
            nt_col += __shfl_sync(0xffffffffu, ia, 31);
        }
        if (lane == 0) {
            ox.ob->new_cells = acc;
            ox.ob->n_tcol = nt_col;
            ver[c0 >> 5] ^= 1u << (c0 & 31);
            if (!self)
                ver[c1 >> 5] ^= 1u << (c1 & 31);
        }
    }
    team_sync(tm);
}

// ---- B. the owners write the rewritten rows back (cells + owner lists) and create the new expression -------------------
__device__ void own_update(const ProblemDesc &p, const Ctx &cx, const OwnCtx &ox, const Team &tm, uint32_t c0, uint32_t c1, uint32_t newid) {
    DA_DYN_SHARED(da_smem);
    const int tid = tm.tid, nt = tm.nt, G = cx.cfg.G;
    const bool self = c0 == c1;
    const uint32_t *ver = DA_SM(uint32_t, ox.lay.ver);
    int *col_len = DA_SM(int, ox.lay.col_len);
    const bool own0 = (int)(c0 % (uint32_t)G) == cx.rank, own1 = !self && (int)(c1 % (uint32_t)G) == cx.rank, ownn = (int)(newid % (uint32_t)G) == cx.rank;
    if (!(own0 || own1 || ownn))
        return; // (uniform over the CTA)
    for (int r = 0; r < (self ? 1 : 2); ++r) {
        if (r == 1)
            team_sync(tm); // (uniform) the two rows of one column are rewritten one after the other
        if (!(r == 0 ? own0 : own1))
            continue;
        const uint32_t e = r == 0 ? c0 : c1, j = e / (uint32_t)G;
        const uint2 dir = ox.ws.cell_dir[e];
        uint2 *pl = ox.ws.cell_pl[(ver[e >> 5] >> (e & 31)) & 1u]; // the version that has just become current
        const uint2 *old = ox.ws.cell_pl[((ver[e >> 5] >> (e & 31)) & 1u) ^ 1u];
        const uint2 *D = DA_SM(uint2, ox.lay.D[r]);
        for (uint32_t i = tid; i < dir.y; i += nt) {
            const uint32_t o = ox.ws.cell_col[dir.x + i];
            const uint2 was = old[dir.x + i], now = D[o];
            pl[dir.x + i] = now;
            if ((was.x | was.y) == 0u || (was.x == now.x && was.y == now.y))
                continue; // dead cell, or a column the substitution did not change
            // the row of e in this column's owner list (one thread per column: nobody else touches the list now)
            const int len = col_len[o];
            for (int k = 0; k < len; ++k) {
                const OwnRow row = own_row_load(ox, (int)o, k);
                if (row.j == j && (row.P | row.N) != 0u) {
                    own_row_planes(ox, (int)o, k, now.x, now.y);
                    break;
                }
            }
        }
    }
    team_sync(tm); // rows that just died may be recycled by the new expression below
    if (ownn) {
        const int r = self ? 1 : 2;
        const uint2 *D = DA_SM(uint2, ox.lay.D[r]);
        const uint32_t *Bn = DA_SM(uint32_t, ox.lay.B[r]), *pre = DA_SM(uint32_t, ox.lay.pre);
        const int M = ox.ob->new_cells;
        const int off = ox.ob->pool_used; // (read by every thread before thread 0 advances it behind the barrier below)
        const bool fits = off + M <= ox.ws.pool_cap;
        const size_t pool = (size_t)cx.rank * ox.ws.pool_cap;
        const uint32_t jn = newid / (uint32_t)G;
        const int cap = ox.lay.lcap + ox.ws.ovf_cap;
        for (int o = tid; o < p.n_out; o += nt) {
            const uint2 v = D[o];
            if ((v.x | v.y) == 0u)
                continue;
            if (fits) {
                const int w = o >> 5;
                const size_t ci = pool + off + pre[w] + __popc(Bn[w] & ((1u << (o & 31)) - 1u));
                ox.ws.cell_col[ci] = (uint32_t)o;
                ox.ws.cell_pl[0][ci] = v; // a new expression starts at version 0
            }
            // owner list of column o: recycle a dead row, else append
            const int len = col_len[o];
            int pos = -1;
            for (int k = 0; k < len; ++k) {
                const OwnRow row = own_row_load(ox, o, k);
                if ((row.P | row.N) == 0u) {
                    pos = k;
                    break;
                }
            }
            if (pos < 0) {
                if (len < cap) {
                    pos = len;
                    col_len[o] = len + 1;
                    atomicMax(&cx.b->list_max, len + 1);
                }
                else
                    cx.b->status = ST_LIST_OVERFLOW;
            }
            if (pos >= 0)
                own_row_store(ox, o, pos, jn, v.x, v.y);
        }
        team_sync(tm); // (uniform: the condition depends on newid and the CTA rank only)
        if (tid == 0) {
            ox.ws.cell_dir[newid] = make_uint2((uint32_t)(pool + off), fits ? (uint32_t)M : 0u);
            if (fits)
                ox.ob->pool_used = off + M;
            else
                cx.b->status = ST_LIST_OVERFLOW;
        }
    }
    team_sync(tm);
}

// ---- C. recount -------------------------------------------------------------------------------------------------------
// Pair counters: a shared-memory hash table keyed by (owned expression, rewritten row, shift, sub) -- open addressing, a
// key claims an empty slot with a CAS, counts are added with reductions nobody waits for.
__device__ __forceinline__ void smem_red_add(uint32_t *p, uint32_t v) {
#if !defined(DA_CPU_SIM)
    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"((unsigned)__cvta_generic_to_shared(p)), "r"(v) : "memory");
#else
    atomicAdd(p, v);
#endif
}
template <int U> __device__ __forceinline__ void own_count_keys(const OwnCtx &ox, const uint32_t (&key)[U], const bool (&on)[U]) {
    DA_DYN_SHARED(da_smem);
    uint32_t *hkey = DA_SM(uint32_t, ox.lay.hkey), *hval = DA_SM(uint32_t, ox.lay.hval);
    const int hlog = ox.lay.hlog;
    const uint32_t mask = (1u << hlog) - 1u;
    const int cap = (int)((mask + 1u) >> 1) + (int)((mask + 1u) >> 3); // 5/8 of the slots
    uint32_t h[U], cur[U];
#pragma unroll
    for (int u = 0; u < U; ++u) { // (the first probes of all U keys are issued together)
        h[u] = (key[u] * 0x9E3779B1u) >> (32 - hlog);
        cur[u] = on[u] ? ld_racy(&hkey[h[u]]) : 0u;
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
        if (!on[u])
            continue;
        const uint32_t k1 = key[u] + 1u;
        uint32_t c = cur[u], hh = h[u], probes = 0u;
        while (true) {
            if (c == 0u) {
                if (ld_racy(&ox.ob->overflow))
                    break; // this pass is being abandoned
                c = atomicCAS(&hkey[hh], 0u, k1);
                if (c == 0u) {
                    const int pos = smem_add(&ox.ob->n_ins, 1);
                    if (pos < cap)
                        DA_SM(uint16_t, ox.lay.hins)[pos] = (uint16_t)hh;
                    else
                        st_racy(&ox.ob->overflow, 1);
                    c = k1;
                }
            }
            if (c == k1) {
                smem_red_add(&hval[hh], 1u);
                break;
            }
            if (++probes > mask) { // every slot is taken by other keys (threads racing past the overflow flag filled the table)
                st_racy(&ox.ob->overflow, 1);
                break;
            }
            hh = (hh + 1u) & mask;
            c = ld_racy(&hkey[hh]);
        }
    }
}

// Per-lane enumeration state of the digit pairs of one list row against the rewritten rows (dedup and ordering rules
// of state_opr.cc:307-340): a small state machine that always points at the next pair (mh != 0) or is exhausted, so that
// the lanes of a warp -- rows of different expressions, each with its own number of pairs -- stay converged.
struct OwnPairs {
    uint32_t P, N;   // the row's planes
    uint32_t flags;  // bit r: rewritten row r pairs with this row; bit 4 + r: the row is the smaller id of pair (row, m_r);
                     // bit 8 + r: the row IS m_r (pairs inside one row); bit 12: the current source is such a self pair
    uint32_t kbase;  // owned index << 9
    int o;           // the row's column (the rewritten rows' planes there are re-read when the source changes)
    int r;           // current rewritten row (3 = done)
    uint32_t Pl, Nl, Ph, Nh; // planes of the smaller / larger id of the current source
    uint32_t ml, mh; // digits of the smaller id still to do (lowest = current), digits of the larger id still to pair with it
};
__device__ __forceinline__ void own_pairs_source(const OwnCtx &ox, OwnPairs &s) { // load source s.r (if any is left)
    DA_DYN_SHARED(da_smem);
    while (s.r < 3 && !((s.flags >> s.r) & 1u))
        ++s.r;
    if (s.r >= 3) {
        s.ml = s.mh = 0u;
        return;
    }
    const uint2 d = DA_SM(uint2, ox.lay.D[s.r])[s.o];
    const bool x_lo = (s.flags >> (4 + s.r)) & 1u, self = (s.flags >> (8 + s.r)) & 1u;
    s.flags = (s.flags & ~0x1000u) | (self ? 0x1000u : 0u);
    s.Pl = x_lo ? s.P : d.x, s.Nl = x_lo ? s.N : d.y;
    s.Ph = x_lo ? d.x : s.P, s.Nh = x_lo ? d.y : s.N;
    s.ml = s.Pl | s.Nl;
    // pairs inside one row (state_opr.cc:323-330): v0 = higher digit, v1 = lower -> the partners of a digit are the digits below it
    s.mh = self ? 0u : (s.Ph | s.Nh);
}
// when the current digit of the smaller id has no partner left: next digit, else next source (a few iterations at most;
// the lanes of the warp re-converge behind the loop)
__device__ __forceinline__ void own_pairs_advance(const OwnCtx &ox, OwnPairs &s) {
    while (s.mh == 0u && s.r < 3) {
        s.ml &= s.ml - 1u;
        if (s.ml != 0u) {
            const int pl = __ffs(s.ml) - 1;
            s.mh = (s.flags & 0x1000u) ? ((s.Ph | s.Nh) & ((1u << pl) - 1u)) : (s.Ph | s.Nh);
        }
        else {
            ++s.r;
            own_pairs_source(ox, s);
        }
    }
}
// the lane's current pair -> key (precondition: s.mh != 0), then on to the next one
__device__ __forceinline__ uint32_t own_pairs_take(const OwnCtx &ox, OwnPairs &s, int nb1) {
    const int pl = __ffs(s.ml) - 1, ph = __ffs(s.mh) - 1;
    const uint32_t key = s.kbase | ((uint32_t)s.r << 7) | ((uint32_t)(ph - pl + nb1) << 1) | (((s.Nl >> pl) ^ (s.Nh >> ph)) & 1u);
    s.mh &= s.mh - 1u;
    own_pairs_advance(ox, s);
    return key;
}

// Pairs of the rows of one subset of the owned expressions (those with (e / G) mod 2^bits == val) with the rewritten rows,
// over the touched columns.  The (column, row) items of all touched columns are flattened over the threads of the CTA
// (tpre = exclusive prefix of the list lengths); the lanes of a warp then draw pairs from their rows in lock step, U at a
// time.  Returns this thread's digit pairs.
#ifndef DA_OWN_UNROLL
#define DA_OWN_UNROLL 2
#endif
__device__ int own_count_subset(const ProblemDesc &p, const Ctx &cx, const OwnCtx &ox, const Team &tm, int bits, uint32_t val) {
    DA_DYN_SHARED(da_smem);
    const int tid = tm.tid, nt = tm.nt, G = cx.cfg.G;
    const uint16_t *tcol = DA_SM(uint16_t, ox.lay.tcol);
    const int *tpre = DA_SM(int, ox.lay.tpre);
    const OwnBlock &ob = *ox.ob;
    const int n_mods = ob.n_mods, n_tcol = ob.n_tcol, nb1 = p.nbits - 1, total = tpre[n_tcol];
    const uint32_t smask = (1u << bits) - 1u;
    const uint32_t m0 = ob.mid[0], m1 = ob.mid[1], m2 = n_mods > 2 ? ob.mid[2] : 0xffffffffu;
    constexpr int U = DA_OWN_UNROLL;
    int pairs = 0;
    const int total_pad = (total + 31) & ~31; // whole warps enter the loop together
    for (int item = tid; item < total_pad; item += nt) {
        OwnPairs s;
        s.flags = 0u, s.r = 3, s.ml = s.mh = 0u, s.kbase = 0u, s.o = 0;
        s.P = s.N = s.Pl = s.Nl = s.Ph = s.Nh = 0u;
        if (item < total) {
            int lo = 0, hi = n_tcol; // largest ti with tpre[ti] <= item
            while (hi - lo > 1) {
                const int mid = (lo + hi) >> 1;
                if (tpre[mid] <= item)
                    lo = mid;
                else
                    hi = mid;
            }
            const int o = tcol[lo];
            const OwnRow row = own_row_load(ox, o, item - tpre[lo]);
            if ((row.P | row.N) != 0u && (row.j & smask) == val) {
                const uint32_t x = row.j * (uint32_t)G + (uint32_t)cx.rank;
                const bool xmod = x == m0 || x == m1 || x == m2;
                s.P = row.P, s.N = row.N;
                s.kbase = row.j << 9;
                s.o = o;
#pragma unroll
                for (int r = 0; r < 3; ++r) {
                    const uint32_t m = r == 0 ? m0 : (r == 1 ? m1 : m2);
                    const uint2 d = DA_SM(uint2, ox.lay.D[r])[o];
                    if (r < n_mods && (d.x | d.y) != 0u && !(xmod && m > x)) // pairs among the rewritten rows are counted once, at the larger id
                        s.flags |= 1u << r;
                    if (x <= m)
                        s.flags |= 1u << (4 + r);
                    if (x == m)
                        s.flags |= 1u << (8 + r);
                }
                s.r = 0;
                own_pairs_source(ox, s);
                own_pairs_advance(ox, s);
            }
        }
        while (__any_sync(0xffffffffu, s.mh != 0u)) {
            uint32_t key[U];
            bool on[U];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                on[u] = s.mh != 0u;
                key[u] = 0u;
                if (on[u]) {
                    key[u] = own_pairs_take(ox, s, nb1);
                    ++pairs;
                }
            }
            own_count_keys<U>(ox, key, on);
        }
    }
    return pairs;
}

// counters of the pass -> histogram entries (count >= 2); leaves the table empty
__device__ void own_harvest(const ProblemDesc &p, const Ctx &cx, const OwnCtx &ox, const Team &tm, uint32_t newid, uint32_t stamp, uint32_t thresh, Best &best) {
    DA_DYN_SHARED(da_smem);
    const int tid = tm.tid, nt = tm.nt, G = cx.cfg.G;
    uint32_t *hkey = DA_SM(uint32_t, ox.lay.hkey), *hval = DA_SM(uint32_t, ox.lay.hval);
    const uint16_t *hins = DA_SM(uint16_t, ox.lay.hins);
    const OwnBlock &ob = *ox.ob;
    const int n = ob.n_ins, rn = ob.n_mods - 1;
    for (int i = tid; i < n; i += nt) {
        const int s = hins[i];
        const uint32_t key = hkey[s] - 1u, cnt = hval[s];
        hkey[s] = 0u;
        hval[s] = 0u;
        if (cnt < 2u)
            continue;
        const int r = (int)((key >> 7) & 3u);
        const uint32_t x = (key >> 9) * (uint32_t)G + (uint32_t)cx.rank, m = ob.mid[r];
        const int shift = (int)((key >> 1) & 63u) - (p.nbits - 1), sub = (int)(key & 1u);
        QInt qx, qm = ob.mq[r];
        float lx, lm = ob.ml[r];
        if (x == newid) // (its record reaches the op table only with this step's exchange)
            qx = ob.mq[rn], lx = ob.ml[rn];
        else
            load_op(p, x, qx, lx);
        const bool x_lo = x <= m;
        const int hot = (int)(key >> 9) < cx.b->hot_n ? (int)(key >> 9) : -1; // x's own region, if it has one
        emit_entry(p, cx, x_lo ? x : m, x_lo ? m : x, shift, sub, cnt, x_lo ? qx : qm, x_lo ? lx : lm, x_lo ? qm : qx, x_lo ? lm : lx, stamp, thresh, best, false, hot);
    }
}

// The whole recount of one step: the owned expressions are processed in subsets small enough for the hash table; a subset
// that runs out of slots is abandoned (nothing of it has been emitted), the table cleared and the subset split in two.
__device__ void own_recount(const ProblemDesc &p, const Ctx &cx, const OwnCtx &ox, const Team &tm, uint32_t newid, uint32_t stamp, uint32_t thresh, Best &best) {
    DA_DYN_SHARED(da_smem);
    const int tid = tm.tid, nt = tm.nt, lane = tid & 31;
    OwnBlock &ob = *ox.ob;
    if (tid < 32) { // the (column, row) items of the touched columns, flattened: exclusive prefix of the list lengths
        const uint16_t *tcol = DA_SM(uint16_t, ox.lay.tcol);
        const int *col_len = DA_SM(int, ox.lay.col_len);
        int *tpre = DA_SM(int, ox.lay.tpre);
        const int n_tcol = ob.n_tcol;
        int carry = 0;
        for (int i0 = 0; i0 < n_tcol; i0 += 32) {
            const int i = i0 + lane;
            const int v = i < n_tcol ? col_len[tcol[i]] : 0;
            int incl = v;
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const int u = __shfl_up_sync(0xffffffffu, incl, off);
                if (lane >= off)
                    incl += u;
            }
            if (i < n_tcol)
                tpre[i] = carry + incl - v;
            carry += __shfl_sync(0xffffffffu, incl, 31);
        }
        if (lane == 0)
            tpre[n_tcol] = carry;
    }
    if (tid == 0) {
        const int b = ob.pass_bits;
        ob.sub_top = 0;
        for (int v = (1 << b) - 1; v >= 0; --v)
            ob.sub_stack[ob.sub_top++] = ((uint32_t)b << 16) | (uint32_t)v;
        ob.n_ins = 0;
        ob.overflow = 0;
        ob.grew = 0;
        ob.ins_max = 0;
#ifdef DA_RECOUNT_PROF
        ob.xt = clock64();
#endif
    }
    team_sync(tm);
    DA_XLAP(0)
    int nr = 0;
    while (ob.sub_top > 0) { // (uniform: sub_top only changes between the barriers below)
        const uint32_t sv = ob.sub_stack[ob.sub_top - 1];
        const int bits = (int)(sv >> 16);
        const uint32_t val = sv & 0xffffu;
        const int mine = own_count_subset(p, cx, ox, tm, bits, val);
        team_sync(tm);
        DA_XLAP(1)
        const bool over = ob.overflow != 0;
        if (!over) {
            nr += mine;
            own_harvest(p, cx, ox, tm, newid, stamp, thresh, best);
        }
        else {
            uint32_t *hkey = DA_SM(uint32_t, ox.lay.hkey), *hval = DA_SM(uint32_t, ox.lay.hval);
            for (int k = tid; k < (1 << ox.lay.hlog); k += nt) {
                hkey[k] = 0u;
                hval[k] = 0u;
            }
        }
        team_sync(tm);
        if (tid == 0) {
            ob.sub_top -= 1;
            if (over) {
                if (bits >= 16 || ob.sub_top + 2 > DA_OWN_STACK)
                    cx.b->status = ST_TOUCH_OVERFLOW; // (cannot happen: one expression has fewer than 400 counters)
                else {
                    ob.sub_stack[ob.sub_top++] = ((uint32_t)(bits + 1) << 16) | (val | (1u << bits));
                    ob.sub_stack[ob.sub_top++] = ((uint32_t)(bits + 1) << 16) | val;
                    ob.grew = 1;
                    ob.splits += 1;
                }
            }
            else
                ob.ins_max = max(ob.ins_max, ob.n_ins);
            ob.n_ins = 0;
            ob.overflow = 0;
        }
        team_sync(tm);
        DA_XLAP(2)
    }
    if (tid == 0) { // next step's first split: finer after an overflow, coarser when the table stayed almost empty
        if (ob.grew)
            ob.pass_bits = min(ob.pass_bits + 1, 5);
        else if (ob.pass_bits > 0 && ob.ins_max < (1 << ox.lay.hlog) / 16)
            ob.pass_bits -= 1;
    }
#pragma unroll
    for (int off = 16; off > 0; off >>= 1)
        nr += __shfl_xor_sync(0xffffffffu, nr, off);
    if (lane == 0 && nr)
        smem_add(&cx.b->r_step, nr);
}

// ---- D. before the adder trees: the owner lists of all CTAs -> per-column lists in global memory ---------------------
__device__ void own_scatter_columns(const ProblemDesc &p, const Ctx &cx, const OwnCtx &ox) {
    DA_DYN_SHARED(da_smem);
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, wid = tid >> 5, nw = nt >> 5, G = cx.cfg.G;
    const int *col_len = DA_SM(int, ox.lay.col_len);
    for (int o = cx.rank * nt + tid; o < p.n_out; o += G * nt)
        cx.ws.col_len[o] = 0;
    group_sync(cx);
    for (int o = wid; o < p.n_out; o += nw) {
        const int len = col_len[o];
        for (int k0 = 0; k0 < len; k0 += 32) {
            const int k = k0 + lane;
            OwnRow row{0u, 0u, 0u};
            if (k < len)
                row = own_row_load(ox, o, k);
            const bool on = (row.P | row.N) != 0u;
            const unsigned bal = __ballot_sync(0xffffffffu, on);
            int base = 0;
            if (lane == 0 && bal)
                base = atomicAdd(&cx.ws.col_len[o], __popc(bal));
            base = __shfl_sync(0xffffffffu, base, 0);
            if (on) {
                const int pos = base + __popc(bal & ((1u << lane) - 1u));
                if (pos >= p.col_cap)
                    cx.b->status = ST_LIST_OVERFLOW;
                else {
                    uint32_t *col = cx.ws.col_u32 + (size_t)o * 3 * p.col_cap;
                    col[pos] = row.j * (uint32_t)G + (uint32_t)cx.rank;
                    col[p.col_cap + pos] = row.P;
                    col[2 * p.col_cap + pos] = row.N;
                }
            }
        }
    }
    group_sync(cx);
}

} // namespace da
