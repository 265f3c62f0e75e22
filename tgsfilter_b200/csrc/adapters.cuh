// K3: adapter search kernels.  Replaces GetEditDistance (T.cpp:1218-1322) = three edlibAlign
// (HW, PATH) calls per (read, adapter): middle window, 5' window, 3' window.
//
//   k_mid_scan    one thread per run of consecutive 1024-column absolute chunks of a read's middle window and
//                 adapter: HW scan with a q+k-1 column halo before the run, chunk minima + atomicMin per
//                 (read, adapter).
//                 This is the kernel that dominates the pipeline (INT-ALU bound).
//   k_mid_count   one thread per (read, adapter) whose best distance is <= k: enumerates the end
//                 columns (only chunks whose minimum equals the best), runs edlib's PATH step on
//                 the first location (start search + traceback -> mlen) and the two thresholds.
//   k_mid_emit    same walk, writes one region per location into the pool.
//   k_ends        one thread per (read, adapter, end): whole window in one thread.
#pragma once
#include "common.cuh"
#include "myers.cuh"

#define MID_THREADS 128
#define RES_THREADS 128

struct AdapterCtx {
    const DevAdapter *ad; // [n_adapters]
    const u64 *peq_pool;
};

static __device__ __forceinline__ AdapterTables adapter_tables(const AdapterCtx &C, int a) {
    const DevAdapter A = C.ad[a];
    AdapterTables T;
    T.hw = C.peq_pool + A.peq_off;
    T.fw = T.hw + 256 * A.nw;
    T.rv = T.fw + 256 * A.nw;
    T.qlen = A.qlen;
    return T;
}

// ---------------------------------------------------------------------------------------------
// k_mid_scan
// ---------------------------------------------------------------------------------------------
// One thread per run: up to 2^run_shift consecutive chunks of a read's middle window (the absolute block
// [run << (chunk_shift + run_shift), +2^(chunk_shift + run_shift)) clipped to the window).  The thread restarts a
// q+k-1 column halo before the run's first chunk only and carries the Myers state across the later chunk
// boundaries, where the state is the exact DP column; at each boundary it closes the finished chunk and starts
// the next one's minimum.  The per-chunk results are what a halo restart per chunk gives: a chunk minimum is only
// reported when it is <= k, and every column scoring <= k is exact after a halo of q+k-1 columns.
//
// The thread scans the run for AP adapters of the same word count at once: one LDS (64*AP*NW bits) per column
// serves all of them and the independent Myers chains interleave.  The bottom-row score is not kept per column:
// it is read off the state (popcounts) every 8 columns; the exact per-column minimum is only evaluated for a
// group when score - popc(minus bits) could reach k (otherwise no column of the group can score <= k, and scores
// > k are never reported).
//
// chunk_min : [n_adapters][chunk_stride] u8 (255 = nothing <= min(k,254) / window too short)
// chunk_cnt / chunk_first : [n_adapters][chunk_stride], written only where chunk_min != 255:
//             number of columns of the chunk scoring chunk_min and the first of them (offset from
//             the start of the bases stream, low 48 bits; the chunk minimum sits in the top 16)
// best_mid  : [n_reads][n_adapters] u32, pre-set to 0xffffffff
struct MidScanArgs {
    int a[2];            // adapter indices handled by this launch (a[1] unused when AP == 1)
    int end_len;
    int chunk_shift;     // log2(chunk length)
    int run_shift;       // log2(chunks per run)
    u32 chunk_stride;
    int n_adapters;
    u32 byte_mul[4];     // {2^24, 2^16, 2^8, 8 * AP * NW}: see mid_row_off
};

template <int NW>
static __device__ void mid_chunk_record(const u64 *__restrict__ tab, int tab_stride, int qlen,
                                        const uint8_t *__restrict__ bases, u64 sb, u64 ob, u64 oe,
                                        int d, u32 &cnt, u64 &first) {
    Myers<NW> s;
    myers_init_hw<NW>(s, qlen);
    cnt = 0;
    first = 0;
    for (u64 p = sb; p < oe; ++p) {
        myers_step<NW, 0, true>(s, tab + (u32)bases[p] * tab_stride, 0);
        if (p >= ob && s.score == d) {
            if (cnt == 0) first = p;
            ++cnt;
        }
    }
}

// Rare path of k_mid_scan: exact column-by-column minimum of one 8-column group, replayed from the state saved at
// the group start, folded into the replay threshold (see k_mid_scan_dyn).  Kept out of line so that it costs the
// hot loop no registers.
template <int NW>
static __device__ __noinline__ int mid_replay_group(const u64 *P0, const u64 *M0, u32 w0, u32 w1,
                                                    const u64 *tab, int tab_stride, int thr) {
    int best = 0x7fffffff;
    u64 tP[NW], tM[NW];
#pragma unroll
    for (int w = 0; w < NW; ++w) { tP[w] = P0[w]; tM[w] = M0[w]; }
    const u32 wd[2] = {w0, w1};
#pragma unroll 1
    for (int j = 0; j < 8; ++j) {
        const u32 byte = (wd[j >> 2] >> (8 * (j & 3))) & 0xffu;
        myers_step_state<NW>(tP, tM, tab + byte * tab_stride);
        best = min(best, myers_score<NW>(tP, tM));
    }
    return min(thr, 2 * best + 6);
}

// Byte offset of the table row of base j of a 16-byte group, computed on the FMA pipe: the ALU pipe is the limiter
// of the scan, and a shift-and-mask costs it two instructions per base.  w * 2^(24-8j) puts byte j at the top,
// mulhi(., 2^8) brings it down alone and * row_bytes scales it.  The multipliers come from the kernel arguments
// (MidScanArgs::byte_mul = {2^24, 2^16, 2^8, row bytes}) so that ptxas cannot turn the multiplies back into shifts.
static __device__ __forceinline__ u32 mid_row_off(const u32 (&wd)[4], int j, const u32 (&mul)[4]) {
    const u32 w = wd[j >> 2];
    const u32 top = (j & 3) == 3 ? w : w * mul[j & 3];
    return __umulhi(top, mul[2]) * mul[3];
}

template <int NW, int AP>
__global__ void __launch_bounds__(MID_THREADS, (NW * AP <= 2) ? 6 : 3)
k_mid_scan_dyn(DevBatch B, AdapterCtx C, MidScanArgs M, const u32 *__restrict__ chunk_off,
               const ChunkEntry *__restrict__ runs, const u32 *__restrict__ perm,
               const u32 *__restrict__ n_runs_ptr, uint8_t *__restrict__ chunk_min,
               u32 *__restrict__ chunk_cnt, u64 *__restrict__ chunk_first,
               u32 *__restrict__ best_mid, u32 *__restrict__ work_ctr) {
    const u32 n_runs = *n_runs_ptr; // device-side total (run_off[n_reads])
    extern __shared__ __align__(16) u64 s_peq_smem[]; // [256][AP][NW] top-padded tables
    DevAdapter A[AP];
#pragma unroll
    for (int x = 0; x < AP; ++x) A[x] = C.ad[M.a[x]];
    // adapters > 256 bp (NW > 4, always launched one per thread) read their table from global memory / L1: 256 x NW
    // words do not fit the shared memory of several resident CTAs, and they are rare
    const u64 *s_peq = s_peq_smem;
    if (NW > 4) {
        s_peq = C.peq_pool + A[0].peq_off;
    } else {
#pragma unroll
        for (int x = 0; x < AP; ++x) {
            const u64 *src = C.peq_pool + A[x].peq_off;
            for (int i = threadIdx.x; i < 256 * NW; i += MID_THREADS)
                s_peq_smem[(i / NW) * (AP * NW) + x * NW + (i % NW)] = src[i];
        }
        __syncthreads();
    }
    constexpr int TS = AP * NW; // table stride per byte value (in u64)
    const int cs = M.chunk_shift;
    const u64 chunk_len = 1ull << cs;
    int halo = 0, qmin = 0x7fffffff;
#pragma unroll
    for (int x = 0; x < AP; ++x) {
        halo = max(halo, A[x].halo_mid);
        qmin = min(qmin, A[x].qlen);
    }
    const uint4 *__restrict__ b16 = (const uint4 *)B.bases;
    // The chunk minimum so far is kept as the replay threshold thr = 2 * min(k, best - 1) + 8 = min(2k + 8,
    // 2 * best + 6).  An 8-column group that starts at score s_0 and ends at s_8 has a minimum
    // >= floor((s_0 + s_8 - 7) / 2) (adjacent columns differ by at most 1), which can only reach min(k, best - 1)
    // when s_0 + s_8 <= thr: one add and one compare per group.  The chunk minimum is <= k exactly when
    // thr < thr0 = 2k + 8, and it is then (thr - 6) / 2; a larger one is never reported.
    int thr0[AP];
#pragma unroll
    for (int x = 0; x < AP; ++x) thr0[x] = 2 * A[x].k_mid + 8;

    // Work is handed out dynamically, 32 consecutive entries of the length-descending order per warp and fetch
    // (zeroed counter per launch): longest runs first, and CTAs that become resident late (another batch's
    // kernels occupied the SM when this launch started) simply take fewer runs instead of stretching the tail.
    const u32 lane = threadIdx.x & 31u;
    for (;;) {
        u32 it = 0;
        if (lane == 0) it = atomicAdd(work_ctr, 32u);
        it = __shfl_sync(0xffffffffu, it, 0);
        if (it >= n_runs) break;
        it += lane;
        if (it >= n_runs) continue; // (the warp's next fetch ends the loop)
        const ChunkEntry re = runs[perm[it]]; // length-descending order: a warp's 32 runs have the same length
        const u64 rs = B.offsets[re.read];
        const i64 tsm = (i64)(B.offsets[re.read + 1] - rs) - 2 * (i64)M.end_len;
        const u64 mb = rs + (u64)M.end_len, me = B.offsets[re.read + 1] - (u64)M.end_len; // middle window
        const u32 c_first = (u32)(mb >> cs);                                               // window's first chunk
        u32 c = max(re.chunk << M.run_shift, c_first);                                     // run's first chunk
        const u32 c_last = min(((re.chunk + 1) << M.run_shift) - 1u, (u32)((me - 1) >> cs));
        u32 ci = chunk_off[re.read] + (c - c_first);                                       // its chunk table index

        u64 Pv[AP][NW], Mv[AP][NW];
        int score[AP], thr[AP];
        bool on[AP];
#pragma unroll
        for (int x = 0; x < AP; ++x) {
            Myers<NW> s0;
            myers_init_hw<NW>(s0, A[x].qlen);
#pragma unroll
            for (int w = 0; w < NW; ++w) { Pv[x][w] = s0.Pv[w]; Mv[x][w] = s0.Mv[w]; }
            score[x] = A[x].qlen;
            thr[x] = thr0[x];
            on[x] = A[x].k_mid > 0 && tsm >= (i64)A[x].qlen; // tsmLen >= qLen, T.cpp:1237
        }
        const bool scan = tsm >= (i64)qmin;
        u64 ob = max((u64)c << cs, mb);                               // first column the run reports
        u64 sb = ob > (u64)halo ? ob - (u64)halo : 0;                  // restart point
        if (sb < mb) sb = mb;
        u64 p = sb;
        if (scan) {
            // head: single bytes up to the next 16-byte boundary (first chunk of a window only)
            const u64 oe0 = min(((u64)c << cs) + chunk_len, me);
            while (p < oe0 && (p & 15ull)) {
                const u64 *eq = s_peq + (u32)B.bases[p] * TS;
#pragma unroll
                for (int x = 0; x < AP; ++x) {
                    myers_step_state<NW>(Pv[x], Mv[x], eq + x * NW);
                    score[x] = myers_score<NW>(Pv[x], Mv[x]);
                    if (p >= ob) thr[x] = min(thr[x], 2 * score[x] + 6);
                }
                ++p;
            }
            // halo: whole 16-byte groups up to ob (16-aligned whenever a halo exists), nothing tracked
            for (; p < ob; p += 16) {
                const uint4 v = __ldg(b16 + (p >> 4));
                const u32 wd[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    const u64 *eq = s_peq + ((wd[j >> 2] >> (8 * (j & 3))) & 0xffu) * TS;
#pragma unroll
                    for (int x = 0; x < AP; ++x) myers_step_state<NW>(Pv[x], Mv[x], eq + x * NW);
                }
            }
#pragma unroll
            for (int x = 0; x < AP; ++x) score[x] = myers_score<NW>(Pv[x], Mv[x]);
        }
        for (;;) { // the run's chunks; p >= ob here
            const u64 cb = (u64)c << cs;
            const u64 oe = min(cb + chunk_len, me); // the chunk reports [max(cb, mb), oe)
            if (scan && p < oe) {
                // whole 16-byte groups (p is 16-aligned: the head only stops short of a boundary at oe)
                const uint4 *q = b16 + (p >> 4);
                for (u32 g = (u32)((oe - p) >> 4); g; --g, ++q) {
                    const uint4 v = __ldg(q);
                    const u32 wd[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                    for (int h = 0; h < 2; ++h) { // two 8-column groups per 16-byte load
                        u64 Pv0[AP][NW], Mv0[AP][NW]; // state at the group start (only read on the rare path)
#pragma unroll
                        for (int x = 0; x < AP; ++x)
#pragma unroll
                            for (int w = 0; w < NW; ++w) { Pv0[x][w] = Pv[x][w]; Mv0[x][w] = Mv[x][w]; }
#pragma unroll
                        for (int j = 8 * h; j < 8 * h + 8; ++j) {
                            const char *row = (const char *)s_peq + mid_row_off(wd, j, M.byte_mul);
                            u64 eq[TS]; // 16-byte loads when rows are 16-byte multiples (the offset hides that)
                            if constexpr (TS % 2 == 0) {
#pragma unroll
                                for (int i = 0; i < TS; i += 2) {
                                    const ulonglong2 v = *(const ulonglong2 *)(row + 8 * i);
                                    eq[i] = v.x;
                                    eq[i + 1] = v.y;
                                }
                            } else {
#pragma unroll
                                for (int i = 0; i < TS; ++i) eq[i] = *(const u64 *)(row + 8 * i);
                            }
#pragma unroll
                            for (int x = 0; x < AP; ++x) myers_step_state<NW>(Pv[x], Mv[x], eq + x * NW);
                        }
#pragma unroll
                        for (int x = 0; x < AP; ++x) {
                            const int s_end = myers_score<NW>(Pv[x], Mv[x]);
                            if (score[x] + s_end <= thr[x])
                                thr[x] = mid_replay_group<NW>(Pv0[x], Mv0[x], wd[2 * h], wd[2 * h + 1],
                                                              s_peq + x * NW, TS, thr[x]);
                            score[x] = s_end;
                        }
                    }
                }
                p = oe & ~15ull;
                // tail (the window's last chunk only)
                for (; p < oe; ++p) {
                    const u64 *eq = s_peq + (u32)B.bases[p] * TS;
#pragma unroll
                    for (int x = 0; x < AP; ++x) {
                        myers_step_state<NW>(Pv[x], Mv[x], eq + x * NW);
                        score[x] = myers_score<NW>(Pv[x], Mv[x]);
                        thr[x] = min(thr[x], 2 * score[x] + 6);
                    }
                }
            }
            // close chunk ci
#pragma unroll
            for (int x = 0; x < AP; ++x) {
                uint8_t result = 255;
                const u64 slot = (u64)M.a[x] * M.chunk_stride + ci;
                if (on[x] && thr[x] < thr0[x]) {
                    const int best = (thr[x] - 6) >> 1; // <= k
                    result = (uint8_t)min(best, 254);
                    atomicMin(best_mid + (u64)re.read * M.n_adapters + M.a[x], (u32)best);
                    // rare: this chunk holds a candidate; record how many columns reach the chunk
                    // minimum and the first of them so that k_mid_count never has to rescan.
                    const u64 cob = max(cb, mb);
                    u64 csb = cob > (u64)halo ? cob - (u64)halo : 0;
                    if (csb < mb) csb = mb;
                    u32 cnt;
                    u64 first;
                    mid_chunk_record<NW>(s_peq + x * NW, TS, A[x].qlen, B.bases, csb, cob, oe, best, cnt, first);
                    chunk_cnt[slot] = cnt;
                    chunk_first[slot] = first | ((u64)best << 48);
                }
                chunk_min[slot] = result;
                thr[x] = thr0[x];
            }
            if (c == c_last) break;
            ++c;
            ++ci;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Enumerate, in ascending order, the end columns of the middle window of read r whose HW score
// equals d, visiting only the chunks whose minimum is d.  f(p) is called with the absolute byte
// offset of each such column; return false from f to stop.
// ---------------------------------------------------------------------------------------------
template <int NW, typename F>
static __device__ void mid_for_each_end(const DevBatch &B, const AdapterTables &T,
                                        const DevAdapter &A, int a, int end_len, int chunk_shift,
                                        u32 r, int d, const u32 *__restrict__ chunk_off,
                                        const ChunkEntry *__restrict__ chunks, u32 chunk_stride,
                                        const uint8_t *__restrict__ chunk_min,
                                        const u32 *__restrict__ chunk_hits,
                                        const u64 *__restrict__ chunk_first, F f) {
    const u64 rs = B.offsets[r], re = B.offsets[r + 1];
    const u64 mb = rs + (u64)end_len, me = re - (u64)end_len;
    for (u32 ci = chunk_off[r]; ci < chunk_off[r + 1]; ++ci) {
        const u64 slot = (u64)a * chunk_stride + ci;
        if (chunk_min[slot] != (uint8_t)min(d, 254)) continue;
        const u64 rec = chunk_first[slot]; // first column scoring the chunk minimum | minimum << 48
        if ((int)(rec >> 48) != d) continue;
        const u64 first = rec & ((1ull << 48) - 1);
        u32 left = chunk_hits[slot];
        const u64 cb = (u64)chunks[ci].chunk << chunk_shift;
        const u64 oe = min(cb + (1ull << chunk_shift), me);
        // restart a halo before the first location (exact from `first` on), stop after the last
        u64 sb = first > (u64)A.halo_mid ? first - (u64)A.halo_mid : 0;
        if (sb < mb) sb = mb;
        Myers<NW> s;
        myers_init_hw<NW>(s, T.qlen);
        for (u64 p = sb; p < oe && left; ++p) {
            myers_step<NW, 0, true>(s, T.hw + (u32)__ldg(B.bases + p) * NW, 0);
            if (p >= first && s.score == d) {
                --left;
                if (!f(p)) return;
            }
        }
    }
}

// One thread per (read, adapter) whose best middle distance is <= k: number of locations (sum of
// the per-chunk records), PATH step of the first location, thresholds (T.cpp:1241-1250).
// mid_n: [n_reads][n_adapters] number of regions (0 if the thresholds fail)
template <int NW>
__global__ void __launch_bounds__(RES_THREADS)
k_mid_count(DevBatch B, AdapterCtx C, int a, int end_len, int n_adapters,
            const u32 *__restrict__ best_mid, const u32 *__restrict__ chunk_off, u32 chunk_stride,
            const uint8_t *__restrict__ chunk_min, const u32 *__restrict__ chunk_cnt,
            const u64 *__restrict__ chunk_first, u32 *__restrict__ mid_n, u64 *scratch,
            u64 scratch_stride) {
    const DevAdapter A = C.ad[a];
    const AdapterTables T = adapter_tables(C, a);
    const u64 tid = (u64)blockIdx.x * RES_THREADS + threadIdx.x;
    for (u32 r = (u32)tid; r < B.n_reads; r += gridDim.x * RES_THREADS) {
        const u32 bd = best_mid[(u64)r * n_adapters + a];
        if (bd == 0xffffffffu) continue;
        const int d = (int)bd;
        const uint8_t tag = (uint8_t)min(d, 254);
        u32 count = 0;
        u64 first = 0;
        for (u32 ci = chunk_off[r]; ci < chunk_off[r + 1]; ++ci) {
            const u64 slot = (u64)a * chunk_stride + ci;
            if (chunk_min[slot] != tag) continue;
            const u64 rec = chunk_first[slot]; // first column | chunk minimum << 48
            if ((int)(rec >> 48) != d) continue;
            if (count == 0) first = rec & ((1ull << 48) - 1);
            count += chunk_cnt[slot];
        }
        const u64 mb = B.offsets[r] + (u64)end_len;
        const u64 s0 = shw_start<NW>(T, B.bases, mb, first, d);
        int ok = mlen_decision(T.qlen, (int)(first - s0 + 1), d, A.thr_mid);
        if (ok < 0) {
            const int alen = nw_alignment_len<NW>(T, B.bases, s0, first, d, scratch + tid, scratch_stride);
            ok = (alen - d >= A.thr_mid) ? 1 : 0;
        }
        mid_n[(u64)r * n_adapters + a] = ok ? count : 0u;
    }
}

// pool: Region {ts, te} per location (T.cpp:1247-1258), at mid_off[r*A+a] .. + mid_n
template <int NW>
__global__ void __launch_bounds__(RES_THREADS)
k_mid_emit(DevBatch B, AdapterCtx C, int a, int end_len, int chunk_shift, int extra_len,
           int n_adapters, const u32 *__restrict__ best_mid, const u32 *__restrict__ chunk_off,
           const ChunkEntry *__restrict__ chunks, u32 chunk_stride,
           const uint8_t *__restrict__ chunk_min, const u32 *__restrict__ chunk_hits,
           const u64 *__restrict__ chunk_first, const u32 *__restrict__ mid_n,
           const u32 *__restrict__ mid_off, Region *__restrict__ pool,
           const u32 *__restrict__ dev_status) {
    if (*dev_status != DEV_STATUS_OK) return;
    const DevAdapter A = C.ad[a];
    const AdapterTables T = adapter_tables(C, a);
    for (u32 r = blockIdx.x * RES_THREADS + threadIdx.x; r < B.n_reads;
         r += gridDim.x * RES_THREADS) {
        const u64 key = (u64)r * n_adapters + a;
        const u32 n = mid_n[key];
        if (n == 0) continue;
        const int d = (int)best_mid[key];
        const u64 rs = B.offsets[r];
        const int tLen = (int)(B.offsets[r + 1] - rs);
        const u64 mb = rs + (u64)end_len;
        Region *out = pool + mid_off[key];
        u32 i = 0;
        mid_for_each_end<NW>(B, T, A, a, end_len, chunk_shift, r, d, chunk_off, chunks, chunk_stride,
                             chunk_min, chunk_hits, chunk_first, [&](u64 p) {
                                 const u64 s0 = shw_start<NW>(T, B.bases, mb, p, d);
                                 int ts = (int)(s0 - rs) - extra_len;       // T.cpp:1248,1253
                                 int te = (int)(p - rs) + 1 + extra_len;    // T.cpp:1249,1254
                                 if (ts < 0) ts = 0;
                                 if (te > tLen) te = tLen;
                                 out[i].s = ts;
                                 out[i].e = te;
                                 ++i;
                                 return i < n;
                             });
    }
}

// ---------------------------------------------------------------------------------------------
// k_ends: 5' and 3' windows (T.cpp:1266-1321).  One thread per (read, side); all tasks of one side
// are contiguous so a warp runs one side.  Every phase is a flat loop of nearly the same trip
// count in all lanes (no per-location nested searches), so warps stay converged:
//   1. forward HW scan: best distance d, number of end columns with that distance, first / last
//   2. start of the first location (reversed-query SHW) and its traceback -> mlen thresholds
//   3. 3' only: HW scan of the REVERSED query from the right end of the window; the left-most
//      column scoring d is min_i startLocations[i] (a column s scores d in the reversed scan iff
//      NW(query, window[s..e]) == d for some e, and every such e is one of the forward end
//      locations), which is all the merge of the {start_i, tLen} regions needs.
// out: end_n [n_reads][n_adapters][2] location counts (0 if the thresholds fail),
//      end_pos[n_reads][n_adapters][2]: side 0 -> max te (region {0, te}), side 1 -> min ts.
// ---------------------------------------------------------------------------------------------
// AP adapters (same word count) per thread: the forward scan of phase 1 is one serial chain per adapter, so two
// chains fed by the same byte loads double the instruction-level parallelism (as in k_mid_scan).
template <int NW, int AP>
__global__ void __launch_bounds__(RES_THREADS)
k_ends(DevBatch B, AdapterCtx C, int a0, int a1, int end_len, int n_adapters,
       const int *__restrict__ read_active, int *__restrict__ end_n, int *__restrict__ end_pos,
       u64 *scratch, u64 scratch_stride) {
    extern __shared__ u64 s_tab_smem[]; // per adapter: hw | fw | rv | rvhw tables (NW <= 4; longer adapters: global memory)
    const int aidx[2] = {a0, a1};
    DevAdapter A[AP];
    AdapterTables T[AP];
    const u64 *rvhw[AP];
#pragma unroll
    for (int x = 0; x < AP; ++x) {
        A[x] = C.ad[aidx[x]];
        const u64 *tab = C.peq_pool + A[x].peq_off;
        if (NW <= 4) {
            u64 *dst = s_tab_smem + (size_t)x * 4 * 256 * NW;
            for (int i = threadIdx.x; i < 4 * 256 * NW; i += RES_THREADS) dst[i] = tab[i];
            tab = dst;
        }
        T[x].hw = tab;
        T[x].fw = tab + 256 * NW;
        T[x].rv = tab + 512 * NW;
        T[x].qlen = A[x].qlen;
        rvhw[x] = tab + 768 * NW;
    }
    if (NW <= 4) __syncthreads();
    const u64 tid = (u64)blockIdx.x * RES_THREADS + threadIdx.x;
    const u64 total = (u64)B.n_reads * 2;
    for (u64 w = tid; w < total; w += (u64)gridDim.x * RES_THREADS) {
        const int side = w >= B.n_reads ? 1 : 0;
        const u32 r = (u32)(side ? w - B.n_reads : w);
        const bool active = read_active[r] != 0;
        const u64 rs = B.offsets[r];
        const int tLen = (int)(B.offsets[r + 1] - rs);
        u64 lo[AP], hi[AP];
        Myers<NW> s[AP];
        int d[AP], cnt[AP];
        u64 first[AP], last[AP];
        u64 lo_min = ~0ull, hi_max = 0;
#pragma unroll
        for (int x = 0; x < AP; ++x) {
            int checkLen = end_len + A[x].end_extra; // T.cpp:1267
            if (checkLen > tLen) checkLen = tLen;
            const bool on = active && A[x].k_end > 0 && checkLen >= 5;
            lo[x] = side == 0 ? rs : rs + (u64)(tLen - checkLen);
            hi[x] = on ? lo[x] + (u64)checkLen : lo[x]; // empty window: nothing to scan
            if (on) { lo_min = min(lo_min, lo[x]); hi_max = max(hi_max, hi[x]); }
            myers_init_hw<NW>(s[x], T[x].qlen);
            d[x] = 0x7fffffff;
            cnt[x] = 0;
            first[x] = last[x] = 0;
        }
        // phase 1 (all adapters of the thread off the same byte)
#pragma unroll 4
        for (u64 p = lo_min; p < hi_max; ++p) {
            const u32 byte = (u32)__ldg(B.bases + p);
#pragma unroll
            for (int x = 0; x < AP; ++x) {
                if (AP == 1 || (p >= lo[x] && p < hi[x])) {
                    myers_step<NW, 0, true>(s[x], T[x].hw + byte * NW, 0);
                    if (s[x].score < d[x]) { d[x] = s[x].score; cnt[x] = 1; first[x] = p; last[x] = p; }
                    else if (s[x].score == d[x]) { ++cnt[x]; last[x] = p; }
                }
            }
        }
#pragma unroll
        for (int x = 0; x < AP; ++x) {
            if (AP == 2 && x == 1 && a1 == a0) break; // odd adapter out: the second lane of the pair is a copy
            const u64 oidx = ((u64)r * n_adapters + aidx[x]) * 2 + side;
            int n_loc = 0, pos = 0;
            if (hi[x] > lo[x] && d[x] <= A[x].k_end) {
                // phase 2
                const u64 s0 = shw_start<NW>(T[x], B.bases, lo[x], first[x], d[x]);
                int ok = mlen_decision(T[x].qlen, (int)(first[x] - s0 + 1), d[x], A[x].thr_end);
                if (ok < 0) {
                    const int alen = nw_alignment_len<NW>(T[x], B.bases, s0, first[x], d[x], scratch + tid, scratch_stride);
                    ok = (alen - d[x] >= A[x].thr_end) ? 1 : 0;
                }
                if (ok) {
                    n_loc = cnt[x];
                    if (side == 0) {
                        pos = (int)(last[x] - rs) + 1; // te of the last location, T.cpp:1286
                    } else {
                        // phase 3
                        Myers<NW> sr;
                        myers_init_hw<NW>(sr, T[x].qlen);
                        u64 leftmost = s0;
#pragma unroll 4
                        for (u64 p = hi[x]; p-- > lo[x];) {
                            myers_step<NW, 0, true>(sr, rvhw[x] + (u32)__ldg(B.bases + p) * NW, 0);
                            if (sr.score == d[x]) leftmost = p;
                        }
                        pos = (int)(leftmost - rs); // min ts, T.cpp:1310
                    }
                }
            }
            end_n[oidx] = n_loc;
            end_pos[oidx] = pos;
        }
    }
}
