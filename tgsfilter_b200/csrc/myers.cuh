// K3 building blocks: Myers/Hyyro bit-vector edit distance, multi-word in registers.
//
// Replaces include/edlib.cpp's calculateBlock (E.cpp:409-444), myersCalcEditDistanceSemiGlobal
// (E.cpp:547-704, HW and SHW modes), myersCalcEditDistanceNW (E.cpp:730-931) and
// obtainAlignmentTraceback (E.cpp:945-1144) with the equivalent specification validated in
// SURVEY.md §3.5 / tests/test_oracle.py: plain semi-global DP semantics, all end columns
// with the best distance, smallest start per end, traceback priority Up > Left > Diagonal.
//
// Layouts.  HW scans use a TOP-padded pattern: the 64*NW-bit column holds W = 64*NW - q wildcard
// rows in bits [0,W) (they match every byte and start with vertical delta 0, i.e. "the target has
// an unbounded prefix that only wildcards can consume") followed by the q query rows, so the
// bottom row of the query is always bit 63 of the last word: the per-column score update is two
// shifts by a constant and there is no column shift or tail fix-up as in edlib's bottom padding
// (E.cpp:658-693).  SHW / NW passes (start search, traceback) are tiny and use the unpadded layout
// with the bottom row at a run-time bit.
#pragma once
#include "common.cuh"

template <int NW>
struct Myers {
    u64 Pv[NW];
    u64 Mv[NW];
    int score;
};

// State "before column 0" of an HW scan in the top-padded layout.  W = 64*NW - qlen wildcard rows (vertical
// delta 0) sit below the query; W >= 64 when NW is a rounded-up word count (adapters > 256 bp run with
// NW = 8, 16 or 32).
template <int NW>
static __device__ __forceinline__ void myers_init_hw(Myers<NW> &s, int qlen) {
    const int W = 64 * NW - qlen;
#pragma unroll
    for (int w = 0; w < NW; ++w) {
        const int below = W - 64 * w; // wildcard rows in this word and above it
        s.Pv[w] = below >= 64 ? 0ull : (below <= 0 ? ~0ull : (~0ull << below));
        s.Mv[w] = 0;
    }
    s.score = qlen;
}

// State before column 0 of an SHW / NW pass (unpadded): H[i][-1] = i.
template <int NW>
static __device__ __forceinline__ void myers_init_plain(Myers<NW> &s, int qlen) {
#pragma unroll
    for (int w = 0; w < NW; ++w) {
        s.Pv[w] = ~0ull;
        s.Mv[w] = 0;
    }
    s.score = qlen;
}

// One column.  HIN = horizontal delta entering the top row: 0 for HW (free leading gap), +1 for
// SHW / NW.  TOPBIT: the query's bottom row is bit 63 of the last word (HW layout); otherwise it is
// row `lastbit` = qlen - 1 counted from bit 0 of word 0 (word lastbit >> 6, which is NW - 1 unless NW is a
// rounded-up word count).  Same recurrences as calculateBlock (E.cpp:409-444).
template <int NW, int HIN, bool TOPBIT>
static __device__ __forceinline__ void myers_step(Myers<NW> &s, const u64 *__restrict__ eq,
                                                  int lastbit) {
    int hin = HIN;
#pragma unroll
    for (int w = 0; w < NW; ++w) {
        u64 Eq = eq[w];
        const u64 Pv = s.Pv[w], Mv = s.Mv[w];
        const u64 hinNeg = (hin < 0) ? 1ull : 0ull;
        const u64 Xv = Eq | Mv;
        Eq |= hinNeg;
        const u64 Xh = (((Eq & Pv) + Pv) ^ Pv) | Eq;
        u64 Ph = Mv | ~(Xh | Pv);
        u64 Mh = Pv & Xh;
        const int hout = (int)(Ph >> 63) - (int)(Mh >> 63);
        if (TOPBIT) {
            if (w == NW - 1) s.score += hout;
        } else if (NW <= 4) { // exact word count: the bottom row is in the last word
            if (w == NW - 1) s.score += (int)((Ph >> (lastbit & 63)) & 1ull) - (int)((Mh >> (lastbit & 63)) & 1ull);
        } else {
            if (w == (lastbit >> 6)) s.score += (int)((Ph >> (lastbit & 63)) & 1ull) - (int)((Mh >> (lastbit & 63)) & 1ull);
        }
        Ph = (Ph << 1) | ((hin > 0) ? 1ull : 0ull);
        Mh = (Mh << 1) | hinNeg;
        s.Pv[w] = Mh | ~(Xv | Ph);
        s.Mv[w] = Ph & Xv;
        hin = hout;
    }
}

// HW column for the hot scan loop: state only.  The bottom-row score is never carried along: in the
// top-padded HW layout the top boundary is 0 and the wildcard rows have zero vertical deltas, so
// H[q][j] = popc(Pv_j) - popc(Mv_j) can be read off the state whenever it is needed
// (myers_score); k_mid_scan does that once per 16 columns.
template <int NW, bool HIST = false>
static __device__ __forceinline__ void myers_step_state(u64 (&sPv)[NW], u64 (&sMv)[NW],
                                                        const u64 *__restrict__ eq, u32 *hM = nullptr) {
    int hin = 0;
#pragma unroll
    for (int w = 0; w < NW; ++w) {
        u64 Eq = eq[w];
        const u64 Pv = sPv[w], Mv = sMv[w];
        const u64 hinNeg = (hin < 0) ? 1ull : 0ull;
        const u64 Xv = Eq | Mv;
        if (w > 0) Eq |= hinNeg;
        const u64 Xh = (((Eq & Pv) + Pv) ^ Pv) | Eq;
        u64 Ph = Mv | ~(Xh | Pv);
        u64 Mh = Pv & Xh;
        // optional history of the bottom row's -1 steps (bit 63 of the last word of Mh)
        if (HIST && w == NW - 1) *hM = __funnelshift_l((u32)(Mh >> 32), *hM, 1);
        const int hout = (w == NW - 1) ? 0 : (int)(Ph >> 63) - (int)(Mh >> 63);
        Ph <<= 1;
        Mh <<= 1;
        if (w > 0) {
            Ph |= (hin > 0) ? 1ull : 0ull;
            Mh |= hinNeg;
        }
        sPv[w] = Mh | ~(Xv | Ph);
        sMv[w] = Ph & Xv;
        hin = hout;
    }
}
template <int NW>
static __device__ __forceinline__ int myers_score(const u64 (&Pv)[NW], const u64 (&Mv)[NW]) {
    int s = 0;
#pragma unroll
    for (int w = 0; w < NW; ++w) s += __popcll(Pv[w]) - __popcll(Mv[w]);
    return s;
}

// 96-bit add through the carry flag (IADD3, IADD3.X, and IMAD.X on the FMA pipe for the top word).
static __device__ __forceinline__ void add96(u32 (&r)[3], const u32 (&a)[3], const u32 (&b)[3]) {
    asm("add.cc.u32 %0, %3, %6;\n\taddc.cc.u32 %1, %4, %7;\n\taddc.u32 %2, %5, %8;"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(b[0]), "r"(b[1]), "r"(b[2]));
}

// HW column of a PACKED PAIR (k_mid_scan_packed): two independent 48-row top-padded HW fields in one 96-bit vector of
// three 32-bit words, field a in bits [0, 48), field b in bits [48, 96).  Field b's top row (bit 48) must see the HW
// boundary (horizontal delta 0), not field a's bottom row (bit 47 = bit 15 of word 1), so nothing may cross from bit
// 47 into bit 48:
//   - bit 47 of Ph and Mh is cleared before the shifts, so 0 comes in at bit 48 (the Mh mask folds into its LOP3);
//   - the add (Eq & Pv) + Pv runs with bit 47 of both addends cleared, so it carries nothing into bit 48.  Its sum bit
//     47 is then wrong, and so is Xh's, but bit 47 of Xh only reaches bit 47 of Ph and Mh, which are cleared anyway.
// Shifts are adds of a vector to itself, so they carry between the words like the add.
static __device__ __forceinline__ void myers_step_pair96(u32 (&Pv)[3], u32 (&Mv)[3], const u32 (&Eq)[3]) {
    constexpr u32 H = ~(1u << 15);
    const u32 Pm[3] = {Pv[0], Pv[1] & H, Pv[2]};
    const u32 t[3] = {Eq[0] & Pv[0], Eq[1] & Pv[1] & H, Eq[2] & Pv[2]};
    u32 sum[3], Ph[3], Mh[3];
    add96(sum, t, Pm);
#pragma unroll
    for (int w = 0; w < 3; ++w) {
        const u32 Xh = (sum[w] ^ Pv[w]) | Eq[w];
        Ph[w] = Mv[w] | ~(Xh | Pv[w]);
        Mh[w] = Pv[w] & Xh;
    }
    Ph[1] &= H;
    Mh[1] &= H;
    add96(Ph, Ph, Ph);
    add96(Mh, Mh, Mh);
#pragma unroll
    for (int w = 0; w < 3; ++w) {
        const u32 Xv = Eq[w] | Mv[w];
        Pv[w] = Mh[w] | ~(Xv | Ph[w]);
        Mv[w] = Ph[w] & Xv;
    }
}

// Bottom-row scores of the two fields of a packed pair (vertical deltas of the top-padded rows, as myers_score).
// Field a's rows in word 1 are counted once and moved from b's sum to a's.
static __device__ __forceinline__ void pair96_scores(const u32 (&Pv)[3], const u32 (&Mv)[3], int &sa, int &sb) {
    const int a_hi = __popc(Pv[1] << 16) - __popc(Mv[1] << 16);
    sa = __popc(Pv[0]) - __popc(Mv[0]) + a_hi;
    sb = __popc(Pv[1]) - __popc(Mv[1]) + __popc(Pv[2]) - __popc(Mv[2]) - a_hi;
}

// Measured and rejected (round 1): moving the 64-bit add and the two 1-bit shifts onto the FMA pipe
// with mad.wide.u32 (IMAD.WIDE) made k_mid_scan 21 % slower (12.0 -> 14.6 ms on config[1]): ALU-pipe
// instructions fell from 20.2 to 17.5 per column but IMAD.WIDE.U32 issues at about a quarter of the
// IMAD rate, so the FMA pipe became the limiter.  The plain C form below already compiles to the
// 32-bit IADD3 + IMAD.X pairs that split each add/shift one ALU op + one FMA op.
// Also replaced (round 1): per-column Ph/Mh top-bit histories (2 SHF per column) by myers_score.

// Bounds on the match count of ANY optimal global alignment of a q-long query against a tl-long
// target with edit distance d: with X mismatches, I insertions, D deletions and M matches,
// q = M+X+I, tl = M+X+D, d = X+I+D  =>  X + 2I = d - (tl - q) =: c  and  M = q - X - I is in
// [q - c, q - ceil(c/2)].  Lets the resolve kernels skip the traceback whenever the threshold is
// outside that interval (SURVEY.md §7 "Hard parts").
static __device__ __forceinline__ int mlen_decision(int q, int tl, int d, int thr) {
    const int c = d - (tl - q);
    if (q - ((c + 1) >> 1) < thr) return 0;  // cannot reach the threshold
    if (q - c >= thr) return 1;              // always reaches it
    return -1;                               // traceback decides
}

// ---------------------------------------------------------------------------------------------
// Small-window helpers used by the resolve kernels (one thread per window; byte loads).
// ---------------------------------------------------------------------------------------------

struct AdapterTables {
    const u64 *hw; // [256][NW] top-padded
    const u64 *fw; // [256][NW] forward, unpadded
    const u64 *rv; // [256][NW] reversed query, unpadded
    int qlen;
};

// Best HW distance <= k over target[lo, hi) (absolute byte offsets); INT_MAX if none.
template <int NW>
static __device__ int hw_best(const AdapterTables &T, const uint8_t *__restrict__ bases, u64 lo,
                              u64 hi, int k) {
    Myers<NW> s;
    myers_init_hw<NW>(s, T.qlen);
    int best = 0x7fffffff;
    for (u64 p = lo; p < hi; ++p) {
        const u64 *eq = T.hw + (u32)__ldg(bases + p) * NW;
        myers_step<NW, 0, true>(s, eq, 0);
        best = min(best, s.score);
    }
    return best <= k ? best : 0x7fffffff;
}

// Smallest start s (absolute) with NW(query, target[s..e]) == d, for a window starting at wlo.
// Reversed-query SHW over target[e], target[e-1], ...; last column whose score is d
// (E.cpp:246-256).
template <int NW>
static __device__ u64 shw_start(const AdapterTables &T, const uint8_t *__restrict__ bases, u64 wlo,
                                u64 e, int d) {
    Myers<NW> s;
    myers_init_plain<NW>(s, T.qlen);
    const int lastbit = T.qlen - 1;
    u64 avail = e - wlo + 1;
    int ncols = (int)min(avail, (u64)(T.qlen + d));
    int last = 0;
    for (int j = 0; j < ncols; ++j) {
        const u64 *eq = T.rv + (u32)__ldg(bases + (e - (u64)j)) * NW;
        myers_step<NW, 1, false>(s, eq, lastbit);
        if (s.score == d) last = j;
    }
    return e - (u64)last;
}

// Cell value H(i, j) of the stored NW matrix, j >= 1 (1-based prefix lengths), 0 <= i <= q.
template <int NW>
static __device__ __forceinline__ int nw_cell(const u64 *Pv, const u64 *Mv, int bottom, int i,
                                              int qlen) {
    // rows i+1..q  <->  bits i..q-1
    int v = bottom;
#pragma unroll
    for (int w = 0; w < NW; ++w) {
        const int lo = max(i - 64 * w, 0);
        const int hi = min(qlen - 64 * w, 64);
        if (lo < hi) {
            u64 m = (hi == 64 ? ~0ull : ((1ull << hi) - 1ull)) & ~((lo == 0) ? 0ull : ((1ull << lo) - 1ull));
            v -= __popcll(Pv[w] & m);
            v += __popcll(Mv[w] & m);
        }
    }
    return v;
}

// Rows [off, off + len) of a table row (NW words) as the Peq words of that SUB-query (bits beyond len are 0).
template <int NW>
static __device__ __forceinline__ void eq_extract(const u64 *__restrict__ full, int off, int len, u64 *out) {
    const int w0 = off >> 6, r = off & 63;
#pragma unroll
    for (int w = 0; w < NW; ++w) {
        const u64 lo = (w0 + w < NW) ? full[w0 + w] : 0ull;
        const u64 hi = (w0 + w + 1 < NW) ? full[w0 + w + 1] : 0ull;
        u64 v = r ? ((lo >> r) | (hi << (64 - r))) : lo;
        const int rem = len - 64 * w;
        if (rem < 64) v = rem <= 0 ? 0ull : (v & ((1ull << rem) - 1ull));
        out[w] = v;
    }
}

// alignmentLength of NW(query[qoff .. qoff+q), target[s0..e0]) traced back Up > Left > Diagonal
// (E.cpp:1023/1057/1088).  scratch: per-thread column store, element (col, k) at
// scratch[(col * (2*NW+1) + k) * stride + tid]; must hold tl = e0 - s0 + 1 columns.
// SUB: the query is a sub-range of the adapter (Hirschberg parts); its Peq words are cut out of the table rows.
template <int NW, bool SUB>
static __device__ int nw_traceback_len_impl(const AdapterTables &T, const uint8_t *__restrict__ bases, int qoff, int q,
                                            u64 s0, u64 e0, u64 *scratch, u64 stride) {
    const int tl = (int)(e0 - s0 + 1);
    const int lastbit = q - 1;
    const int REC = 2 * NW + 1;
    Myers<NW> s;
    myers_init_plain<NW>(s, q);
    for (int j = 0; j < tl; ++j) {
        const u64 *eq = T.fw + (u32)__ldg(bases + s0 + (u64)j) * NW;
        if (SUB) {
            u64 eb[NW];
            eq_extract<NW>(eq, qoff, q, eb);
            myers_step<NW, 1, false>(s, eb, lastbit);
        } else {
            myers_step<NW, 1, false>(s, eq, lastbit);
        }
        u64 *rec = scratch + (u64)j * REC * stride;
#pragma unroll
        for (int w = 0; w < NW; ++w) {
            rec[(u64)(2 * w) * stride] = s.Pv[w];
            rec[(u64)(2 * w + 1) * stride] = s.Mv[w];
        }
        rec[(u64)(2 * NW) * stride] = (u64)(u32)s.score;
    }
    // walk
    int i = q, j = tl, len = 0;
    u64 cP[NW], cM[NW], lP[NW], lM[NW];
    int cBottom, lBottom = 0;
    auto load_col = [&](int col1, u64 *P, u64 *M, int &bottom) { // col1: 1-based column
        const u64 *rec = scratch + (u64)(col1 - 1) * REC * stride;
#pragma unroll
        for (int w = 0; w < NW; ++w) {
            P[w] = rec[(u64)(2 * w) * stride];
            M[w] = rec[(u64)(2 * w + 1) * stride];
        }
        bottom = (int)(u32)rec[(u64)(2 * NW) * stride];
    };
    load_col(j, cP, cM, cBottom);
    if (j >= 2) load_col(j - 1, lP, lM, lBottom);
    int cur = cBottom;
    while (true) {
        if (i == 0) { len += j; break; }
        if (j == 0) { len += i; break; }
        // vertical delta of row i in column j = bit i-1
        const int w = (i - 1) >> 6, b = (i - 1) & 63;
        int dv = 0;
#pragma unroll
        for (int ww = 0; ww < NW; ++ww)
            if (ww == w) dv = (int)((cP[ww] >> b) & 1ull) - (int)((cM[ww] >> b) & 1ull);
        if (dv == 1) { // up + 1 == cur
            cur -= 1;
            i -= 1;
            len += 1;
            continue;
        }
        const int left = (j == 1) ? i : nw_cell<NW>(lP, lM, lBottom, i, q);
        int ni = i, ncur;
        if (left + 1 == cur) {
            ncur = left;
        } else {
            int dl;
            if (j == 1) {
                dl = 1; // H(i,0) - H(i-1,0)
            } else {
                dl = 0;
#pragma unroll
                for (int ww = 0; ww < NW; ++ww)
                    if (ww == w) dl = (int)((lP[ww] >> b) & 1ull) - (int)((lM[ww] >> b) & 1ull);
            }
            ncur = left - dl;
            ni = i - 1;
        }
        // move one column to the left
        j -= 1;
        i = ni;
        cur = ncur;
        len += 1;
        if (j >= 1) {
#pragma unroll
            for (int ww = 0; ww < NW; ++ww) { cP[ww] = lP[ww]; cM[ww] = lM[ww]; }
            cBottom = lBottom;
            if (j >= 2) load_col(j - 1, lP, lM, lBottom);
        }
    }
    return len;
}

template <int NW>
static __device__ int nw_traceback_len(const AdapterTables &T, const uint8_t *__restrict__ bases,
                                       u64 s0, u64 e0, u64 *scratch, u64 stride) {
    return nw_traceback_len_impl<NW, false>(T, bases, 0, T.qlen, s0, e0, scratch, stride);
}

// alignmentLength the way obtainAlignment decides it (E.cpp:1164-1215): the traceback while the matrix edlib would
// store stays below 1 MiB, otherwise Hirschberg's divide and conquer (E.cpp:1232-1390).  Only adapters above
// ~1 250 bp can get there ((20 * ceil(q/64) + 8) * tl >= 2^20 with tl < 2q), so only the 32-word instantiation carries
// the code.  The split: cut the target in the middle; the alignment passes between row i of the last left column
// and row i + 1 of the first right column for the SMALLEST i (then the top, then the bottom boundary) whose scores
// add up to the optimum; both parts are solved the same way (explicit stack instead of recursion).
// `best` = the optimal distance of the whole problem (edlib passes it down as k).
template <int NW>
static __device__ int nw_alignment_len(const AdapterTables &T, const uint8_t *__restrict__ bases, u64 s0, u64 e0,
                                       int best, u64 *scratch, u64 stride) {
    if constexpr (NW < 32) {
        return nw_traceback_len<NW>(T, bases, s0, e0, scratch, stride);
    } else {
        {   // the common case first: no split at all
            const long long nb = (T.qlen + 63) / 64, tl = (long long)(e0 - s0 + 1);
            if ((20 * nb + 8) * tl < (1ll << 20)) return nw_traceback_len<NW>(T, bases, s0, e0, scratch, stride);
        }
        struct Frame { int qoff, ql; u64 s, e1; int best; }; // target [s, e1)
        Frame st[16];
        int sp = 0, total = 0;
        st[sp++] = Frame{0, T.qlen, s0, e0 + 1, best};
        while (sp) {
            const Frame f = st[--sp];
            const int tl = (int)(f.e1 - f.s);
            if (f.ql == 0 || tl == 0) { total += f.ql + tl; continue; } // E.cpp:1171-1178
            const long long nb = (f.ql + 63) / 64;
            if ((20 * nb + 8) * (long long)tl < (1ll << 20) || sp + 2 > 16) {
                total += nw_traceback_len_impl<NW, true>(T, bases, f.qoff, f.ql, f.s, f.e1 - 1, scratch, stride);
                continue;
            }
            const int lw = tl / 2, rw = tl - lw;
            u64 eb[NW];
            Myers<NW> a, b; // a: sub-query vs the left half; b: reversed sub-query vs the reversed right half
            myers_init_plain<NW>(a, f.ql);
            for (int j = 0; j < lw; ++j) {
                eq_extract<NW>(T.fw + (u32)__ldg(bases + f.s + (u64)j) * NW, f.qoff, f.ql, eb);
                myers_step<NW, 1, false>(a, eb, f.ql - 1);
            }
            myers_init_plain<NW>(b, f.ql);
            const int roff = T.qlen - f.qoff - f.ql; // the same rows in the reversed-query table
            for (int j = 0; j < rw; ++j) {
                eq_extract<NW>(T.rv + (u32)__ldg(bases + (f.e1 - 1 - (u64)j)) * NW, roff, f.ql, eb);
                myers_step<NW, 1, false>(b, eb, f.ql - 1);
            }
            // L[i] = lw + sum_{r <= i} da(r);  R[i + 1] = Rrev[ql - 2 - i] with Rrev[x] = rw + sum_{r <= x} db(r)
            auto delta = [](const Myers<NW> &m, int r) {
                return (int)((m.Pv[r >> 6] >> (r & 63)) & 1ull) - (int)((m.Mv[r >> 6] >> (r & 63)) & 1ull);
            };
            int idx = -2, ls = 0, rs = 0;
            int Lc = lw, Rc = b.score; // before the loop: L[-1] = lw, Rrev[ql - 1] = b.score
            for (int i = 0; i + 1 < f.ql; ++i) {
                Lc += delta(a, i);
                Rc -= delta(b, f.ql - 1 - i);
                if (Lc + Rc == f.best) { idx = i; ls = Lc; rs = Rc; break; }
            }
            if (idx == -2 && lw + b.score == f.best) { idx = -1; ls = lw; rs = b.score; }
            if (idx == -2 && a.score + rw == f.best) { idx = f.ql - 1; ls = a.score; rs = rw; }
            if (idx == -2) { // cannot happen for a correct optimum: fall back to the traceback
                total += nw_traceback_len_impl<NW, true>(T, bases, f.qoff, f.ql, f.s, f.e1 - 1, scratch, stride);
                continue;
            }
            const int ul = idx + 1;
            st[sp++] = Frame{f.qoff + ul, f.ql - ul, f.s + (u64)lw, f.e1, rs};
            st[sp++] = Frame{f.qoff, ul, f.s, f.s + (u64)lw, ls};
        }
        return total;
    }
}
