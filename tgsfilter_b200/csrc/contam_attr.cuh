// Per-record attribution of the contaminant screen (tgsf_set_contaminants_labelled).  The first-pass screen
// (k_contam_screen) stays as it is; k_contam_decide<true> lists the pieces it marks, and k_contam_attr re-rolls only
// those, so the attribution costs work in proportion to the contaminated bases.
//
// k_contam_attr: a persistent grid takes listed pieces from a device work counter, one CTA per piece.  Each thread
// rolls a contiguous run of the piece's windows and probes like the screen (the prefilter bitmap for small sets, then
// the table); a hit whose label is a record adds 1 to that label's count in a shared-memory (label -> count) table.
// A block reduction picks (largest count, smallest label).  A pass that would fill the table past 3/4 is dropped and
// the piece restarts with twice the passes, pass p taking the labels with label mod P == p: with P >= the record count
// a pass holds at most one label, so the split ends, and the result is exact however many records one piece hits.
#pragma once
#include "contam.cuh"

#define ATTR_THREADS 512
#define ATTR_SLOTS_LOG2 12
#define ATTR_SLOTS (1u << ATTR_SLOTS_LOG2) // shared (label, count) table: 32 KB
#define ATTR_FILL_MAX (ATTR_SLOTS / 4u * 3u)

// One pass over the labelled table: record_kmers[label] (shared keys: row n_seqs) += 1 per key, one atomic per
// distinct row in a warp.
__global__ void k_contam_label_count(const u64 *__restrict__ table, const u32 *__restrict__ labels, u64 cap,
                                     u32 n_seqs, unsigned long long *record_kmers) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += (u64)gridDim.x * blockDim.x) {
        if (table[i] == CONTAM_EMPTY) continue;
        const u32 l = labels[i];
        const u32 row = l == CONTAM_LABEL_SHARED ? n_seqs : l;
        const u32 peers = __match_any_sync(__activemask(), row);
        if ((u32)(threadIdx.x & 31) == (u32)(__ffs(peers) - 1)) atomicAdd(record_kmers + row, (unsigned long long)__popc(peers));
    }
}

// Slot of a key in the table, or ~0 when it is not there.
static __device__ __forceinline__ u64 contam_find(const u64 *__restrict__ table, u64 mask, u64 key, u64 h) {
    for (u64 i = h & mask;; i = (i + 1) & mask) {
        const u64 v = __ldg(table + i);
        if (v == key) return i;
        if (v == CONTAM_EMPTY) return ~0ull;
    }
}

// Attribution of the listed pieces.  Per piece: record = the label with the most windows (smallest on a tie) and
// record_hits = that count, or record = n_seqs and record_hits = 0 when every hit has a shared key.  tally (2 x
// (n_seqs + 1) u64: reads, then bases) gets 1 and the piece's length in the record's row; out (per piece index:
// record, record_hits) gets the pair instead when it is given.
template <bool PREFILTER>
__global__ void __launch_bounds__(ATTR_THREADS, 1)
k_contam_attr(DevBatch B, const tgsf_piece *__restrict__ pieces, const u32 *__restrict__ list,
              const u32 *__restrict__ list_n, u32 *work, int k, const u64 *__restrict__ table, u64 mask,
              const u32 *__restrict__ labels, const u32 *__restrict__ pf_bits, u32 n_seqs,
              unsigned long long *tally, int2 *out, const u32 *__restrict__ dev_status) {
    extern __shared__ u32 s_bits[];
    __shared__ u32 s_key[ATTR_SLOTS], s_cnt[ATTR_SLOTS];
    __shared__ unsigned long long s_red[ATTR_THREADS / 32];
    __shared__ u32 s_task, s_fill;
    __shared__ volatile u32 s_over;
    if (*dev_status != DEV_STATUS_OK) return;
    if (PREFILTER) {
        const uint4 *src = (const uint4 *)pf_bits;
        uint4 *dst = (uint4 *)s_bits;
        for (u32 i = threadIdx.x; i < CONTAM_PF_WORDS / 4; i += ATTR_THREADS) dst[i] = __ldg(src + i);
    }
    const u32 n_list = *list_n;
    const u64 kmask = (1ull << (2 * k)) - 1ull;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (;;) {
        if (threadIdx.x == 0) s_task = atomicAdd(work, 1u);
        __syncthreads();
        const u32 t = s_task;
        if (t >= n_list) return;
        const u32 pi = list[t];
        const tgsf_piece p = pieces[pi];
        const uint8_t *seq = B.bases + B.offsets[p.read] + (u64)p.start;
        const u32 windows = (u32)(p.len - k + 1);
        const u32 span = (windows + ATTR_THREADS - 1) / ATTR_THREADS;
        const u32 w0 = min(windows, threadIdx.x * span), w1 = min(windows, w0 + span);
        unsigned long long best = 0; // (count << 32) | ~label: the max is the largest count, then the smallest label
        u32 passes = 1;
        for (u32 pass = 0; pass < passes;) {
            for (u32 j = threadIdx.x; j < ATTR_SLOTS; j += ATTR_THREADS) {
                s_key[j] = CONTAM_LABEL_EMPTY;
                s_cnt[j] = 0;
            }
            if (threadIdx.x == 0) {
                s_fill = 0;
                s_over = 0;
            }
            __syncthreads();
            if (w0 < w1) {
                const uint8_t *q = seq + w0;
                const u32 n_bytes = (w1 - w0) + (u32)(k - 1);
                ContamRoll roll;
                for (u32 j = 0; j < n_bytes; ++j) {
                    if (!roll.push(__ldg(q + j), k, kmask)) continue;
                    if (s_over) break;
                    const u64 key = roll.key();
                    const u64 h = contam_mix(key);
                    if (PREFILTER && !contam_pf_test(s_bits, h)) continue;
                    const u64 i = contam_find(table, mask, key, h);
                    if (i == ~0ull) continue;
                    const u32 label = __ldg(labels + i);
                    if (label == CONTAM_LABEL_SHARED || (passes > 1 && label % passes != pass)) continue;
                    u32 s = (label * 0x9E3779B1u) >> (32 - ATTR_SLOTS_LOG2);
                    bool over = false;
                    for (;; s = (s + 1) & (ATTR_SLOTS - 1)) {
                        u32 o = s_key[s];
                        if (o == CONTAM_LABEL_EMPTY) {
                            o = atomicCAS(&s_key[s], CONTAM_LABEL_EMPTY, label);
                            if (o == CONTAM_LABEL_EMPTY) {
                                // each thread places at most one key after the limit: the table never fills up
                                over = atomicAdd(&s_fill, 1u) >= ATTR_FILL_MAX;
                                break;
                            }
                        }
                        if (o == label) break;
                    }
                    atomicAdd(&s_cnt[s], 1u);
                    if (over) {
                        s_over = 1;
                        break;
                    }
                }
            }
            __syncthreads();
            const bool overflow = s_over != 0;
            if (overflow) { // drop this pass's counts and split the labels over twice the passes
                passes *= 2;
                pass = 0;
                best = 0;
                __syncthreads(); // every thread has read s_over before it is cleared
                continue;
            }
            unsigned long long mine = 0;
            for (u32 j = threadIdx.x; j < ATTR_SLOTS; j += ATTR_THREADS) {
                const u32 l = s_key[j];
                if (l != CONTAM_LABEL_EMPTY) mine = max(mine, ((unsigned long long)s_cnt[j] << 32) | (u32)~l);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) mine = max(mine, __shfl_xor_sync(0xffffffffu, mine, o));
            if (lane == 0) s_red[warp] = mine;
            __syncthreads();
            if (warp == 0) {
                mine = lane < ATTR_THREADS / 32 ? s_red[lane] : 0ull;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) mine = max(mine, __shfl_xor_sync(0xffffffffu, mine, o));
                best = max(best, mine);
            }
            ++pass;
            __syncthreads(); // the table and s_red are reused by the next pass or piece
        }
        if (threadIdx.x == 0) {
            const u32 record = best ? ~(u32)best : n_seqs;
            const u32 record_hits = (u32)(best >> 32);
            if (out) {
                out[pi] = make_int2((int)record, (int)record_hits);
            } else {
                atomicAdd(tally + record, 1ull);
                atomicAdd(tally + (n_seqs + 1) + record, (unsigned long long)p.len);
            }
        }
    }
}
