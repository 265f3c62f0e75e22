// Fold-back screen (tgsf_set_foldback): a piece X·rc(X') that read through a junction without adapter is cut at the
// junction and only its longer arm is kept.
//
// Rules (include/tgsf.h, DESIGN §4): window i = s[i, i+15) of a piece, valid when all 15 bytes are A/C/G/T in either
// case (the contaminant screen's rolling code, ContamRoll); key = min(forward, reverse-complement code), orientation o
// = 0 when the forward code is the smaller.  A window is sampled iff (fmix32(key) & 7) == 0.  A key that occurs among
// the sampled windows exactly once with o = 0 (at p0) and exactly once with o = 1 (at p1) is an anchor with
// d = p0 + p1 + 15 (twice the fold centre) and g = |p1 - p0| - 15.  Anchors vote into bins d >> 7; the peak is the
// b maximising n[b] + n[b+1] (smallest b on ties); V = its count, c = floor(sum d / 2V).  Cut iff V >= 8,
// min g <= 500, 400 V >= min(c, L - c) and 0 < c < L.
//
// Layout: one CTA per piece.  The CTA rolls over the piece (one contiguous run of windows per thread), inserts every
// sampled key into an open-addressing table (key, two saturating 16-bit orientation counts, p0, p1), then walks the
// table and votes the anchors into the d histogram, then reduces the peak.  k_fold_smem keeps table and histogram in
// shared memory and takes pieces of at most FOLD_SMEM_MAX_LEN bases; a piece that is longer, or whose distinct sampled
// keys fill 3/4 of the table, goes to a list that k_fold_global works through with a per-CTA table and histogram in
// global memory (L2).  There the key space is split into passes by hash so that each pass fits the table; a pass that
// overflows doubles the pass count and restarts the piece, up to FOLD_MAX_PASSES.  Which table a key lands in does
// not change which keys are anchors, so both paths give the same result.
#pragma once
#include "common.cuh"
#include "contam.cuh"

#define FOLD_K 15
#define FOLD_SAMPLE_MASK 7u
#define FOLD_BIN_SHIFT 7
#define FOLD_MIN_ANCHORS 8
#define FOLD_MAX_GAP 500
#define FOLD_DENSITY 400

#define FOLD_THREADS 512
#define FOLD_EMPTY 0xFFFFFFFFu                // keys are 30-bit
#define FOLD_ANCHOR 0x00010001u               // one o = 0 and one o = 1 occurrence
#define FOLD_SMEM_SLOTS 8192u
#define FOLD_SMEM_MAX_LEN 40960               // ~5 100 sampled keys expected: 5/8 of the table
#define FOLD_SMEM_BINS ((((2 * FOLD_SMEM_MAX_LEN - FOLD_K) >> FOLD_BIN_SHIFT) + 2 + 1) & ~1)
#define FOLD_SMEM_BYTES (FOLD_SMEM_SLOTS * 16u + FOLD_SMEM_BINS * 16u)
#define FOLD_GLOBAL_SLOTS 65536u              // 1 MB table per CTA of k_fold_global
#define FOLD_GLOBAL_WINDOWS_PER_PASS (3u * FOLD_GLOBAL_SLOTS) // ~3/8 of the table sampled per pass
// fmix32 is a bijection, so a pass over 1/2^14 of the hash range holds at most 2^15 sampled keys and fits: a pass
// that overflows at this many passes means the constants above were changed, and the batch fails
#define FOLD_MAX_PASSES (1u << 14)

struct FoldTable {
    u32 *key, *cnt, *p0, *p1;
    u32 slots; // power of two
};
struct FoldBins {
    u32 *n;
    int *min_g;
    u64 *sum_d;
};

// Per-CTA workspace of k_fold_global: the table, then the histogram (bins_cap bins).
static __host__ __device__ __forceinline__ size_t fold_ws_bytes(u32 bins_cap) {
    return (size_t)FOLD_GLOBAL_SLOTS * 16u + (size_t)bins_cap * 16u;
}

// Bins a piece of L >= FOLD_K bases can vote into, plus one empty bin so that n[b + 1] is always defined.
static __host__ __device__ __forceinline__ u32 fold_bins(u32 L) { return ((2u * L - FOLD_K) >> FOLD_BIN_SHIFT) + 2u; }

static __device__ __forceinline__ u32 fold_fmix32(u32 h) { // murmur3 finaliser
    h ^= h >> 16;
    h *= 0x85ebca6bu;
    h ^= h >> 13;
    h *= 0xc2b2ae35u;
    h ^= h >> 16;
    return h;
}

struct FoldShared {
    u32 fill, over, piece;
    unsigned long long best;
};

// The fold decision of one piece, as tgsf_fold_detect reports it (fold = c when cut, else -1).
static __device__ __forceinline__ tgsf_fold_result fold_decide(u32 L, u32 V, u64 sum_d, int min_g) {
    tgsf_fold_result r;
    r.anchors = (int32_t)V;
    r.fold = -1;
    if (V == 0) {
        r.centre = -1;
        r.min_gap = -1;
        return r;
    }
    const u64 c = sum_d / (2ull * V);
    r.centre = (int32_t)c;
    r.min_gap = min_g;
    const u64 shorter = c < (u64)L - c ? c : (u64)L - c;
    if (V >= FOLD_MIN_ANCHORS && min_g <= FOLD_MAX_GAP && (u64)FOLD_DENSITY * V >= shorter && c > 0 && c < (u64)L)
        r.fold = (int32_t)c;
    return r;
}

// Table passes + votes + peak for seq[0, L), L >= FOLD_K.  Returns false (and leaves the result undefined) when a
// pass overflowed the table.  On success thread 0 gets the decision in *res.  Every thread of the CTA calls it.
static __device__ bool fold_piece(const uint8_t *__restrict__ seq, u32 L, FoldTable T, u32 passes, FoldBins Bn,
                                  FoldShared &sh, tgsf_fold_result *res) {
    const u32 nb = fold_bins(L);
    const u32 limit = T.slots / 4u * 3u;
    for (u32 b = threadIdx.x; b < nb; b += blockDim.x) {
        Bn.n[b] = 0;
        Bn.min_g[b] = 0x7fffffff;
        Bn.sum_d[b] = 0;
    }
    const u32 windows = L - (FOLD_K - 1);
    const u32 per = (windows + blockDim.x - 1) / blockDim.x;
    const u32 w0 = min(windows, threadIdx.x * per), w1 = min(windows, w0 + per);
    const u64 kmask = (1ull << (2 * FOLD_K)) - 1ull;
    for (u32 pass = 0; pass < passes; ++pass) {
        for (u32 i = threadIdx.x; i < T.slots; i += blockDim.x) {
            T.key[i] = FOLD_EMPTY;
            T.cnt[i] = 0;
        }
        if (threadIdx.x == 0) {
            sh.fill = 0;
            sh.over = 0;
        }
        __syncthreads();
        if (w0 < w1) {
            ContamRoll roll;
            const u32 end = w1 + (FOLD_K - 1);
            for (u32 j = w0; j < end; ++j) {
                if (!roll.push(__ldg(seq + j), FOLD_K, kmask)) continue;
                const u32 key = (u32)roll.key();
                const u32 h = fold_fmix32(key);
                if (h & FOLD_SAMPLE_MASK) continue;
                if (passes > 1 && (u32)(((u64)h * passes) >> 32) != pass) continue;
                if (*(volatile u32 *)&sh.over) break;
                u32 s = (h >> 3) & (T.slots - 1u);
                bool placed = false;
                for (u32 probe = 0; probe < T.slots; ++probe, s = (s + 1u) & (T.slots - 1u)) {
                    const u32 old = atomicCAS(T.key + s, FOLD_EMPTY, key);
                    if (old == FOLD_EMPTY) {
                        if (atomicAdd(&sh.fill, 1u) >= limit) sh.over = 1;
                        placed = true;
                        break;
                    }
                    if (old == key) {
                        placed = true;
                        break;
                    }
                }
                if (!placed) {
                    sh.over = 1;
                    break;
                }
                // saturating count: an orientation seen twice is no anchor, so stop counting it (bounded by the
                // threads that raced past the check: < 2^16)
                const u32 shift = roll.fwd < roll.rev ? 0u : 16u;
                if (((*(volatile u32 *)(T.cnt + s) >> shift) & 0xFFFFu) < 2u) {
                    atomicAdd(T.cnt + s, 1u << shift);
                    (shift ? T.p1 : T.p0)[s] = j - (FOLD_K - 1); // read only when this was the sole occurrence
                }
            }
        }
        __syncthreads();
        if (*(volatile u32 *)&sh.over) return false;
        for (u32 i = threadIdx.x; i < T.slots; i += blockDim.x) {
            if (T.cnt[i] != FOLD_ANCHOR) continue;
            const u32 p0 = T.p0[i], p1 = T.p1[i];
            const u32 d = p0 + p1 + FOLD_K;
            const int g = (int)(p1 > p0 ? p1 - p0 : p0 - p1) - FOLD_K;
            const u32 b = d >> FOLD_BIN_SHIFT;
            atomicAdd(Bn.n + b, 1u);
            atomicAdd((unsigned long long *)(Bn.sum_d + b), (unsigned long long)d);
            atomicMin(Bn.min_g + b, g);
        }
        __syncthreads();
    }
    // peak: max n[b] + n[b+1], smallest b on ties (key = count << 32 | ~b)
    unsigned long long best = 0;
    for (u32 b = threadIdx.x; b + 1 < nb; b += blockDim.x) {
        const unsigned long long v = ((unsigned long long)(Bn.n[b] + Bn.n[b + 1]) << 32) | (u32)~b;
        best = v > best ? v : best;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long x = __shfl_xor_sync(0xffffffffu, best, o);
        best = x > best ? x : best;
    }
    if (threadIdx.x == 0) sh.best = 0;
    __syncthreads();
    if ((threadIdx.x & 31) == 0 && best) atomicMax(&sh.best, best);
    __syncthreads();
    if (threadIdx.x == 0) {
        const u32 V = (u32)(sh.best >> 32), b = ~(u32)sh.best;
        u64 sum_d = 0;
        int min_g = 0x7fffffff;
        if (V) {
            sum_d = Bn.sum_d[b] + Bn.sum_d[b + 1];
            min_g = min(Bn.min_g[b], Bn.min_g[b + 1]);
        }
        *res = fold_decide(L, V, sum_d, min_g);
    }
    return true;
}

// Thread 0: detect-only output, or the cut (longer arm, the 5' one on a tie) and the statistics
// {pieces cut, bases removed, pieces dropped as TGSF_PIECE_FOLDBACK, their kept-arm bases}.
static __device__ void fold_apply(tgsf_piece *pieces, u32 pi, const tgsf_fold_result &r, int min_len,
                                  unsigned long long *stats, tgsf_fold_result *out) {
    if (out) {
        out[pi] = r;
        return;
    }
    if (r.fold < 0) return;
    tgsf_piece p = pieces[pi];
    const int c = r.fold, L = p.len;
    const int arm = c >= L - c ? c : L - c;
    if (arm != c) p.start += c;
    p.len = arm;
    atomicAdd(stats + 0, 1ull);
    atomicAdd(stats + 1, (unsigned long long)(L - arm));
    if (arm < min_len) {
        p.status = TGSF_PIECE_FOLDBACK;
        p.sum_q = 0;
        p.repeat_len = -1;
        atomicAdd(stats + 2, 1ull);
        atomicAdd(stats + 3, (unsigned long long)arm);
    }
    pieces[pi] = p;
}

static __device__ __forceinline__ bool fold_takes(const tgsf_piece &p) {
    return p.status == TGSF_PIECE_EMIT && p.len >= FOLD_K;
}

// Shared-memory path.  Pieces are taken from a work counter; those longer than FOLD_SMEM_MAX_LEN or whose table
// overflows are appended to long_list for k_fold_global.  Launched over the SMs; the piece count is device-side.
__global__ void __launch_bounds__(FOLD_THREADS, 1)
k_fold_smem(DevBatch B, tgsf_piece *pieces, const u32 *__restrict__ n_pieces_ptr, u32 *work, u32 *long_list,
            u32 *n_long, int min_len, unsigned long long *stats, tgsf_fold_result *out, const u32 *__restrict__ dev_status) {
    extern __shared__ __align__(16) uint8_t fmem[];
    __shared__ FoldShared sh;
    if (*dev_status != DEV_STATUS_OK) return;
    FoldTable T;
    T.slots = FOLD_SMEM_SLOTS;
    T.key = (u32 *)fmem;
    T.cnt = T.key + FOLD_SMEM_SLOTS;
    T.p0 = T.cnt + FOLD_SMEM_SLOTS;
    T.p1 = T.p0 + FOLD_SMEM_SLOTS;
    FoldBins Bn;
    Bn.sum_d = (u64 *)(T.p1 + FOLD_SMEM_SLOTS);
    Bn.n = (u32 *)(Bn.sum_d + FOLD_SMEM_BINS);
    Bn.min_g = (int *)(Bn.n + FOLD_SMEM_BINS);
    const u32 n_pieces = *n_pieces_ptr;
    while (true) {
        if (threadIdx.x == 0) sh.piece = atomicAdd(work, 1u);
        __syncthreads();
        const u32 pi = sh.piece;
        __syncthreads();
        if (pi >= n_pieces) return;
        const tgsf_piece p = pieces[pi];
        if (!fold_takes(p)) {
            if (out && threadIdx.x == 0) out[pi] = fold_decide((u32)max(p.len, 0), 0, 0, 0);
            continue;
        }
        tgsf_fold_result r;
        const bool ok = p.len <= FOLD_SMEM_MAX_LEN &&
                        fold_piece(B.bases + B.offsets[p.read] + (u64)p.start, (u32)p.len, T, 1, Bn, sh, &r);
        if (threadIdx.x == 0) {
            if (ok) fold_apply(pieces, pi, r, min_len, stats, out);
            else long_list[atomicAdd(n_long, 1u)] = pi;
        }
        __syncthreads();
    }
}

// Global-memory path over the long list: CTA b owns workspace ws + b * fold_ws_bytes(bins_cap).
__global__ void __launch_bounds__(FOLD_THREADS, 1)
k_fold_global(DevBatch B, tgsf_piece *pieces, const u32 *__restrict__ long_list, const u32 *__restrict__ n_long_ptr,
              u32 *work, uint8_t *ws, u32 bins_cap, int min_len, unsigned long long *stats, tgsf_fold_result *out,
              u32 *dev_status) {
    __shared__ FoldShared sh;
    if (*dev_status != DEV_STATUS_OK) return;
    uint8_t *mine = ws + (size_t)blockIdx.x * fold_ws_bytes(bins_cap);
    FoldTable T;
    T.slots = FOLD_GLOBAL_SLOTS;
    T.key = (u32 *)mine;
    T.cnt = T.key + FOLD_GLOBAL_SLOTS;
    T.p0 = T.cnt + FOLD_GLOBAL_SLOTS;
    T.p1 = T.p0 + FOLD_GLOBAL_SLOTS;
    FoldBins Bn;
    Bn.sum_d = (u64 *)(T.p1 + FOLD_GLOBAL_SLOTS);
    Bn.n = (u32 *)(Bn.sum_d + bins_cap);
    Bn.min_g = (int *)(Bn.n + bins_cap);
    const u32 n_long = *n_long_ptr;
    while (true) {
        if (threadIdx.x == 0) sh.piece = atomicAdd(work, 1u);
        __syncthreads();
        const u32 li = sh.piece;
        __syncthreads();
        if (li >= n_long) return;
        const u32 pi = long_list[li];
        const tgsf_piece p = pieces[pi];
        const u32 L = (u32)p.len;
        if (fold_bins(L) > bins_cap) { // longer than the per-100 bp tables allow: the batch fails as such
            if (threadIdx.x == 0) atomicExch(dev_status, DEV_STATUS_BIN_OVERFLOW);
            return;
        }
        const uint8_t *seq = B.bases + B.offsets[p.read] + (u64)p.start;
        u32 passes = (L - (FOLD_K - 1) + FOLD_GLOBAL_WINDOWS_PER_PASS - 1) / FOLD_GLOBAL_WINDOWS_PER_PASS;
        tgsf_fold_result r;
        while (!fold_piece(seq, L, T, passes, Bn, sh, &r)) {
            __syncthreads();
            if (passes >= FOLD_MAX_PASSES) {
                if (threadIdx.x == 0) atomicExch(dev_status, DEV_STATUS_HASH_OVERFLOW);
                return;
            }
            passes *= 2;
        }
        if (threadIdx.x == 0) fold_apply(pieces, pi, r, min_len, stats, out);
        __syncthreads();
    }
}
