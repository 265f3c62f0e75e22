// Contaminant screen (tgsf_set_contaminants): every canonical k-mer of a contaminant set sits in an open-addressing
// u64 table in HBM; every window of every emitted piece is looked up once.  A piece whose share of hit windows reaches
// the threshold gets TGSF_PIECE_CONTAM.
//
// Codes: A0 C1 G2 T3, case-insensitive; a window with any other byte is not a k-mer (never inserted, never a hit).
// Canonical key = min(forward code, reverse-complement code), 2 bits per base, k <= 31, so no key has all 64 bits set
// and ~0 marks an empty slot.  Membership does not depend on the order of insertion, so the screen is deterministic.
//
// Screen: the windows of the screened pieces are cut into chunks of CONTAM_CHUNK windows (count + exclusive scan +
// fill, like the scan tiles); one warp takes a chunk, each lane a contiguous run of windows with its k - 1 bases of
// look-back, one rolling canonical code per lane, one atomic per chunk into the piece's contam_hits.  For sets of at
// most CONTAM_PF_MAX_KEYS keys every CTA first tests a 2^20-bit two-hash bitmap of the set in shared memory, so a
// window whose k-mer is not in the set (almost all of them) costs no L2 probe.
#pragma once
#include "common.cuh"

#define CONTAM_EMPTY (~0ull)
#define CONTAM_K_MIN 11
#define CONTAM_K_MAX 31
#define CONTAM_THREADS 512
#define CONTAM_CHUNK 2048u             // windows per warp task (64 per lane)
#define CONTAM_BUILD_SEG 256u          // window end positions per thread of the build
#define CONTAM_PF_LOG2 20              // prefilter: 2^20 bits = 128 KB of shared memory per CTA
#define CONTAM_PF_WORDS ((1u << CONTAM_PF_LOG2) / 32u)
#define CONTAM_PF_SMEM_BYTES (CONTAM_PF_WORDS * 4u)
#define CONTAM_PF_MAX_KEYS (1ull << 17) // <= 2^17 keys: <= 5 % false positives with two bits per key

struct __align__(16) ContamChunk {
    u64 start; // absolute byte offset of the chunk's first window
    u32 piece;
    u32 n_win; // windows in the chunk (1 .. CONTAM_CHUNK)
};

static __device__ __forceinline__ u64 contam_mix(u64 x) { // splitmix64 finaliser
    x ^= x >> 30;
    x *= 0xbf58476d1ce4e5b9ull;
    x ^= x >> 27;
    x *= 0x94d049bb133111ebull;
    x ^= x >> 31;
    return x;
}

static __device__ __forceinline__ int contam_code(u32 b) {
    b &= 0xDFu; // upper case; only 'a'/'c'/'g'/'t' map onto 'A'/'C'/'G'/'T'
    return b == 'A' ? 0 : b == 'C' ? 1 : b == 'G' ? 2 : b == 'T' ? 3 : -1;
}

// Rolling forward / reverse-complement codes; returns true when the last k bytes are a valid window.
struct ContamRoll {
    u64 fwd = 0, rev = 0;
    int run = 0;
    __device__ __forceinline__ bool push(u32 byte, int k, u64 mask) {
        const int c = contam_code(byte);
        if (c < 0) {
            run = 0;
            return false;
        }
        fwd = ((fwd << 2) | (u64)c) & mask;
        rev = (rev >> 2) | ((u64)(3 - c) << (2 * (k - 1)));
        return ++run >= k;
    }
    __device__ __forceinline__ u64 key() const { return fwd < rev ? fwd : rev; }
};

static __device__ __forceinline__ bool contam_pf_test(const u32 *bits, u64 h) {
    const u32 b1 = (u32)(h >> (64 - CONTAM_PF_LOG2)), b2 = (u32)(h >> 24) & ((1u << CONTAM_PF_LOG2) - 1u);
    return ((bits[b1 >> 5] >> (b1 & 31)) & (bits[b2 >> 5] >> (b2 & 31)) & 1u) != 0;
}

static __device__ __forceinline__ bool contam_lookup(const u64 *__restrict__ table, u64 mask, u64 key, u64 h) {
    for (u64 i = h & mask;; i = (i + 1) & mask) {
        const u64 v = __ldg(table + i);
        if (v == key) return true;
        if (v == CONTAM_EMPTY) return false;
    }
}

// Build: thread t owns the window END positions [t*SEG, (t+1)*SEG) of the concatenated records and rolls in from k - 1
// bytes before (clamped to its record); windows never span two records.  *n_inserted += successful inserts.
__global__ void __launch_bounds__(256)
k_contam_build(const uint8_t *__restrict__ seq, const u64 *__restrict__ offs, u32 n_seqs, int k, u64 *table, u64 mask,
               unsigned long long *n_inserted) {
    const u64 n_bytes = offs[n_seqs];
    const u64 kmask = (1ull << (2 * k)) - 1ull;
    unsigned long long mine = 0;
    for (u64 e0 = ((u64)blockIdx.x * blockDim.x + threadIdx.x) * CONTAM_BUILD_SEG; e0 < n_bytes;
         e0 += (u64)gridDim.x * blockDim.x * CONTAM_BUILD_SEG) {
        const u64 e1 = min(e0 + CONTAM_BUILD_SEG, n_bytes);
        u32 lo = 0, hi = n_seqs; // record r with offs[r] <= e0 < offs[r + 1]
        while (hi - lo > 1) {
            const u32 mid = (lo + hi) >> 1;
            if (offs[mid] <= e0) lo = mid; else hi = mid;
        }
        u32 r = lo;
        u64 p = e0 >= (u64)(k - 1) ? e0 - (u64)(k - 1) : 0;
        if (p < offs[r]) p = offs[r];
        ContamRoll roll;
        for (; p < e1; ++p) {
            if (p >= offs[r + 1]) {
                while (p >= offs[r + 1]) ++r;
                roll.run = 0;
            }
            if (!roll.push(seq[p], k, kmask) || p < e0) continue;
            const u64 key = roll.key();
            for (u64 i = contam_mix(key) & mask;; i = (i + 1) & mask) {
                const u64 old = atomicCAS((unsigned long long *)(table + i), CONTAM_EMPTY, key);
                if (old == CONTAM_EMPTY) { ++mine; break; }
                if (old == key) break;
            }
        }
    }
    if (mine) atomicAdd(n_inserted, mine);
}

// Prefilter bitmap of a built table (small sets only).
__global__ void k_contam_bitmap(const u64 *__restrict__ table, u64 cap, u32 *bits) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < cap; i += (u64)gridDim.x * blockDim.x) {
        const u64 key = table[i];
        if (key == CONTAM_EMPTY) continue;
        const u64 h = contam_mix(key);
        const u32 b1 = (u32)(h >> (64 - CONTAM_PF_LOG2)), b2 = (u32)(h >> 24) & ((1u << CONTAM_PF_LOG2) - 1u);
        atomicOr(bits + (b1 >> 5), 1u << (b1 & 31));
        atomicOr(bits + (b2 >> 5), 1u << (b2 & 31));
    }
}

// Chunks per piece: only pieces still emitted and at least k long are screened.  Launched over the piece capacity; the
// live count is device-side.
__global__ void k_contam_count(const tgsf_piece *__restrict__ pieces, const u32 *__restrict__ n_pieces_ptr, u32 cap,
                               int k, u32 *__restrict__ n_chunks, const u32 *__restrict__ dev_status) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= cap) return;
    u32 n = 0;
    if (*dev_status == DEV_STATUS_OK && i < *n_pieces_ptr) {
        const tgsf_piece p = pieces[i];
        if (p.status == TGSF_PIECE_EMIT && p.len >= k) n = ((u32)(p.len - k) + CONTAM_CHUNK) / CONTAM_CHUNK;
    }
    n_chunks[i] = n;
}

__global__ void k_contam_fill(DevBatch B, const tgsf_piece *__restrict__ pieces, const u32 *__restrict__ chunk_off,
                              u32 cap, int k, ContamChunk *__restrict__ chunks) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= cap) return;
    const u32 b = chunk_off[i], e = chunk_off[i + 1];
    if (b == e) return;
    const tgsf_piece p = pieces[i];
    const u64 s0 = B.offsets[p.read] + (u64)p.start;
    const u32 windows = (u32)(p.len - k + 1);
    for (u32 c = b; c < e; ++c) {
        const u32 w0 = (c - b) * CONTAM_CHUNK;
        ContamChunk ch;
        ch.start = s0 + w0;
        ch.piece = i;
        ch.n_win = min(CONTAM_CHUNK, windows - w0);
        chunks[c] = ch;
    }
}

// One warp per chunk (grid-stride over the device-side chunk total); lane l rolls over windows
// [l*span, min((l+1)*span, n_win)) of the chunk, span = ceil(n_win / 32).
template <bool PREFILTER>
__global__ void __launch_bounds__(CONTAM_THREADS)
k_contam_screen(const uint8_t *__restrict__ bases, const ContamChunk *__restrict__ chunks,
                const u32 *__restrict__ n_chunks_ptr, int k, const u64 *__restrict__ table, u64 mask,
                const u32 *__restrict__ pf_bits, tgsf_piece *pieces, const u32 *__restrict__ dev_status) {
    extern __shared__ u32 s_bits[];
    if (*dev_status != DEV_STATUS_OK) return;
    if (PREFILTER) {
        const uint4 *src = (const uint4 *)pf_bits;
        uint4 *dst = (uint4 *)s_bits;
        for (u32 i = threadIdx.x; i < CONTAM_PF_WORDS / 4; i += CONTAM_THREADS) dst[i] = __ldg(src + i);
        __syncthreads();
    }
    const u32 n_chunks = *n_chunks_ptr;
    const int lane = threadIdx.x & 31;
    const u32 warps = gridDim.x * (CONTAM_THREADS / 32);
    const u64 kmask = (1ull << (2 * k)) - 1ull;
    for (u32 c = blockIdx.x * (CONTAM_THREADS / 32) + (threadIdx.x >> 5); c < n_chunks; c += warps) {
        const ContamChunk ch = chunks[c];
        const u32 span = (ch.n_win + 31) / 32;
        const u32 w0 = min(ch.n_win, (u32)lane * span), w1 = min(ch.n_win, w0 + span);
        u32 hits = 0;
        if (w0 < w1) {
            const uint8_t *p = bases + ch.start + w0;
            const u32 n_bytes = (w1 - w0) + (u32)(k - 1);
            ContamRoll roll;
            for (u32 j = 0; j < n_bytes; ++j) {
                if (!roll.push(__ldg(p + j), k, kmask)) continue;
                const u64 key = roll.key();
                const u64 h = contam_mix(key);
                if (PREFILTER && !contam_pf_test(s_bits, h)) continue;
                hits += contam_lookup(table, mask, key, h) ? 1u : 0u;
            }
        }
        hits = warp_sum_u32(hits);
        if (lane == 0 && hits) atomicAdd(&pieces[ch.piece].contam_hits, (int)hits);
    }
}

// Threshold: contaminant iff hits * 10^6 >= ppm * windows (u64).
__global__ void k_contam_decide(tgsf_piece *pieces, const u32 *__restrict__ n_pieces_ptr, u32 cap, int k, u64 ppm,
                                const u32 *__restrict__ dev_status) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= cap || *dev_status != DEV_STATUS_OK || i >= *n_pieces_ptr) return;
    const tgsf_piece p = pieces[i];
    if (p.status != TGSF_PIECE_EMIT || p.len < k) return;
    const u64 windows = (u64)(p.len - k + 1);
    if ((u64)p.contam_hits * 1000000ull >= ppm * windows) pieces[i].status = TGSF_PIECE_CONTAM;
}
