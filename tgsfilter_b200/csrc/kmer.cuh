// K4: k-mer repeat length of a kept piece = (L - k + 1) - #distinct k-mers.
// Replaces GetKmerCount (T.cpp:1703-1753): rolling 2-bit code A0 C1 G2 T3, every other byte
// (lower case, N) contributes 00, mask (1 << 2k) - 1, std::unordered_set of the codes.
//
// Which pieces reach which kernel: for k <= 16, k_kmer_tag16 (kmer16.cuh) takes every piece and leaves
// those with more than KMER16_MAX_KMERS k-mers in a long list, which k_kmer_smem (k <= 12) or k_kmer
// (k = 13 .. 16) then works through; for k > 16, k_kmer takes every piece.
//
// k_kmer: one CTA per piece; the set is an open-addressing hash table in shared memory (atomicCAS).
// Pieces with more k-mers than half the table are processed in several passes over disjoint
// hash partitions of the key space, so any piece length is exact with the same 128 KB table.
// Nothing bounds how many distinct keys one partition gets (a piece can be built to crowd one), so a
// pass counts its new keys and stops once they pass 3/4 of the table; the pass is then split in two
// (twice the passes: partition p of P is exactly partitions 2p and 2p + 1 of 2P, so the passes already
// done stay counted) and the piece goes on from the first half.  A pass that still overflows at
// KMER_MAX_PASSES fails the batch with DEV_STATUS_HASH_OVERFLOW.
#pragma once
#include "common.cuh"

#define KMER_THREADS 512
#define KMER_SMEM_BYTES (128 * 1024)
#define KMER_MAX_PASSES (1u << 24) // the partition is taken from 24 hash bits: more passes separate no more keys

static __device__ __forceinline__ u32 mix32(u64 x) {
    x ^= x >> 33;
    x *= 0xff51afd7ed558ccdull;
    x ^= x >> 33;
    x *= 0xc4ceb9fe1a85ec53ull;
    x ^= x >> 33;
    return (u32)x;
}

static __device__ __forceinline__ u32 base_code(uint8_t b) { // T.cpp:1709-1724
    return b == 'C' ? 1u : b == 'G' ? 2u : b == 'T' ? 3u : 0u;
}

template <typename KEY>
__global__ void __launch_bounds__(KMER_THREADS, 1)
k_kmer(DevBatch B, DevParams P, tgsf_piece *pieces, const u32 *__restrict__ n_pieces_ptr,
       u64 *__restrict__ counters, u32 *__restrict__ dev_status,
       const u32 *__restrict__ piece_list, // null (k > 16): all pieces; else the long list k_kmer_tag16 left, n_pieces_ptr counts it
       u32 fill_cap) { // new keys one pass may hold, below the table's 3/4 (smaller: tests of the split)
    if (*dev_status != DEV_STATUS_OK) return;
    extern __shared__ __align__(16) uint8_t kmem[];
    KEY *table = (KEY *)kmem;
    constexpr u32 SLOTS = KMER_SMEM_BYTES / sizeof(KEY);
    constexpr KEY EMPTY = (KEY)~(KEY)0;
    // At most `limit` + KMER_THREADS keys get in before every thread has seen s_over: the table never fills.
    const u32 limit = min(SLOTS / 4u * 3u, fill_cap);
    __shared__ u32 s_distinct, s_fill, s_over;
    const int k = P.kmer;
    const u64 mask = (k >= 32) ? ~0ull : ((1ull << (2 * k)) - 1ull);
    const u32 n_pieces = *n_pieces_ptr;

    for (u32 li = blockIdx.x; li < n_pieces; li += gridDim.x) {
        const u32 pi = piece_list ? piece_list[li] : li;
        tgsf_piece pc = pieces[pi];
        if (pc.status != TGSF_PIECE_EMIT) continue;
        const int L = pc.len;
        const int total = L - k + 1;
        int repeat = 0;
        if (total <= 0) {
            repeat = total - 1; // see oracle/tgsf_oracle.c kmer_repeat_len
        } else {
            const uint8_t *seq = B.bases + B.offsets[pc.read] + (u64)pc.start;
            u32 passes = ((u32)total + SLOTS / 2 - 1) / (SLOTS / 2);
            if (threadIdx.x == 0) s_distinct = 0;
            const int per = (total + KMER_THREADS - 1) / KMER_THREADS;
            const int i0 = min((int)threadIdx.x * per, total), i1 = min(i0 + per, total);
            u32 mine = 0;
            for (u32 pass = 0; pass < passes;) {
                __syncthreads(); // every thread has read s_over and is done with the table
                for (u32 i = threadIdx.x; i < SLOTS; i += KMER_THREADS) table[i] = EMPTY;
                if (threadIdx.x == 0) {
                    s_fill = 0;
                    s_over = 0;
                }
                __syncthreads();
                u32 got = 0;
                if (i0 < i1) {
                    u64 km = 0;
                    for (int j = 0; j < k - 1; ++j) km = (km << 2) | base_code(seq[i0 + j]);
                    for (int i = i0; i < i1; ++i) {
                        km = ((km << 2) | base_code(seq[i + k - 1])) & mask;
                        const u32 h = mix32(km);
                        if (passes > 1 && (u32)(((u64)(h >> 8) * passes) >> 24) != pass) continue;
                        if (*(volatile u32 *)&s_over) break;
                        u32 slot = h & (SLOTS - 1);
                        const KEY key = (KEY)km;
                        while (true) {
                            const KEY old = atomicCAS(&table[slot], EMPTY, key);
                            if (old == EMPTY) {
                                ++got;
                                if (atomicAdd(&s_fill, 1u) >= limit) *(volatile u32 *)&s_over = 1;
                                break;
                            }
                            if (old == key) break;
                            slot = (slot + 1) & (SLOTS - 1);
                        }
                    }
                }
                __syncthreads();
                if (!s_over) { // the pass is complete
                    mine += got;
                    ++pass;
                    continue;
                }
                if (passes >= KMER_MAX_PASSES) { // every thread takes this branch: the batch fails
                    if (threadIdx.x == 0) atomicExch(dev_status, DEV_STATUS_HASH_OVERFLOW);
                    return;
                }
                passes *= 2;
                pass *= 2;
            }
            atomicAdd(&s_distinct, mine);
            __syncthreads();
        }
        if (threadIdx.x == 0) {
            if (total > 0) repeat = total - (int)*(volatile u32 *)&s_distinct; // thread 0 alone reads and resets it
            pc.repeat_len = repeat;
            if (repeat < P.min_repeat) { // T.cpp:1984-1988
                pc.status = TGSF_PIECE_SHORT_REPEAT;
                atomic_add_u64(counters + P.L.drop_info + 15, 1ull);
                atomic_add_u64(counters + P.L.drop_info + 16, (u64)pc.len);
            }
            pieces[pi] = pc;
        }
    }
}

// k_kmer_smem, k <= 12, pieces of the long list (more k-mers than k_kmer_tag16 takes).  A piece that fits one
// staged tile is counted by tag rounds (kmer_tag_count below); a longer one by a bitmap over the key space.
// The 4^k-bit map lives in SHARED memory, split into ceil(4^k / KMER_SB_BITS) key ranges that
// are handled in successive passes (k <= 10: one pass, k = 11: three, k = 12: twelve).  The piece is
// staged once as a big-endian 2-bit stream (16 bases per word, first base in the top bits; coalesced
// 16-byte loads from the 16-byte-aligned address at or below the piece start), so a k-mer is a funnel
// shift of two neighbouring words and each thread walks 16 consecutive k-mers from two LDS.  One
// shared-memory atomicOr per k-mer in the pass that owns its key; its return value says whether the
// k-mer is new.  No global traffic beyond reading the piece.
#define KMER_SB_THREADS 1024
#define KMER_SB_BITMAP_BYTES 176128                 // 172 KB; 3 x 176128 x 8 >= 4^11
#define KMER_SB_BITS (KMER_SB_BITMAP_BYTES * 8u)
#define KMER_SB_TILE_WORDS 12288                    // 48 KB of codes = 196 608 bases per tile
#define KMER_SB_SMEM_BYTES (KMER_SB_BITMAP_BYTES + (KMER_SB_TILE_WORDS + 2) * 4)

static __device__ __forceinline__ u32 pack_codes4(u32 x) { // 4 bytes -> 8 bits, lowest address in the top 2 bits
    const u32 y = base_code((uint8_t)x) | (base_code((uint8_t)(x >> 8)) << 8) | (base_code((uint8_t)(x >> 16)) << 16) |
                  (base_code((uint8_t)(x >> 24)) << 24);
    return (y * 0x40100401u) >> 24;
}

// Stage bases [abase, abase + 16 * n_words) as 2-bit codes into tile[0..n_words), tile[n_words] = 0.
static __device__ __forceinline__ void kmer_stage_tile(const DevBatch &B, u64 n_total, u64 abase, u32 n_words, u32 *tile) {
    for (u32 w = threadIdx.x; w < n_words + 1; w += blockDim.x) {
        u32 v = 0;
        if (w < n_words) {
            const u64 a = abase + 16ull * w;
            uint4 q;
            if (a + 16 <= n_total) {
                q = __ldg((const uint4 *)(B.bases + a));
            } else { // last, partial group of the batch: bytes beyond the stream are not touched
                __align__(16) uint8_t tmp[16];
                // bytes left in the stream (< 16 here); comparing in 32 bits keeps k_kmer_smem free of spills
                const u32 avail = a < n_total ? (u32)(n_total - a) : 0u;
#pragma unroll
                for (u32 j = 0; j < 16; ++j) tmp[j] = j < avail ? B.bases[a + j] : (uint8_t)0;
                q = *(uint4 *)tmp;
            }
            v = (pack_codes4(q.x) << 24) | (pack_codes4(q.y) << 16) | (pack_codes4(q.z) << 8) | pack_codes4(q.w);
        }
        tile[w] = v; // tile[n_words] = 0: the window of the last word reads one word past it
    }
}

// Atomics-free distinct count of the k-mers of ONE staged tile ("last writer wins" tags).
// Shared-memory atomics run at ~2 cycles per lane per SM, plain shared stores at 32 lanes per cycle, so
// the set is built without any read-modify-write: in each round every pending k-mer stores the tag
// (remainder bits of its mixed key | its position) into slot = low 15 bits of the mixed key (a bijection
// of the 2k-bit key, so slot + remainder identify the key exactly).  After a barrier each k-mer reads its
// slot back: tag equal to its own -> it is the one representative of its key (count 1); same remainder ->
// duplicate of the representative; otherwise its key lost the slot to another key and stays pending for
// the next round (new multiplier).  All instances of a key share the slot and see the same winner, so
// keys are resolved as a whole; a k-mer only reads a slot it has just written, so the table is never
// cleared.  pend[w]: 16-bit mask of the unresolved positions of word w.
#define KMER_TAG_SLOTS 32768u
#define KMER_TAG_IDX_BITS 18
static __device__ __forceinline__ u32 kmer_tag_of(u32 mixed, u32 pos) { // remainder bits above the position
    return ((mixed << (KMER_TAG_IDX_BITS - 15)) & ~((1u << KMER_TAG_IDX_BITS) - 1u)) | pos;
}

static __device__ __forceinline__ u32 kmer_mix(u32 key, u32 mult, u32 keymask, u32 half) {
    const u32 p = (key * mult) & keymask;
    return p ^ (p >> half);
}
// x: 32 stream bits whose top 2k bits are the key.  Round 0 uses a plain xor-shift (a bijection of the key:
// the bits shifted in from above are zero), later rounds a multiplicative mix with a per-round multiplier.
template <bool R0>
static __device__ __forceinline__ u32 kmer_mix_x(u32 x, u32 sh, u32 mult, u32 keymask, u32 half) {
    if (R0) return (x ^ (x >> 11)) >> sh;
    return kmer_mix(x >> sh, mult, keymask, half);
}

template <bool R0>
static __device__ __forceinline__ void kmer_dense_store(const u32 *tile, u32 *table, const uint16_t *pend, u32 n_scan,
                                                        u32 sh, u32 mult, u32 keymask, u32 half) {
    for (u32 w = threadIdx.x; w < n_scan; w += blockDim.x) {
        const u32 m = pend[w];
        if (!m) continue;
        const u32 w0 = tile[w], w1 = tile[w + 1], pw = w << 4;
        if (m == 0xFFFFu) {
#pragma unroll
            for (u32 j = 0; j < 16; ++j) {
                const u32 mixed = kmer_mix_x<R0>(__funnelshift_l(w1, w0, 2 * j), sh, mult, keymask, half);
                table[mixed & (KMER_TAG_SLOTS - 1)] = kmer_tag_of(mixed, pw + j);
            }
        } else {
#pragma unroll 4
            for (u32 j = 0; j < 16; ++j) {
                if ((m >> j) & 1u) {
                    const u32 mixed = kmer_mix_x<R0>(__funnelshift_l(w1, w0, 2 * j), sh, mult, keymask, half);
                    table[mixed & (KMER_TAG_SLOTS - 1)] = kmer_tag_of(mixed, pw + j);
                }
            }
        }
    }
}

// returns (#representatives found by this thread) and adds its still-pending count to `left`
template <bool R0>
static __device__ __forceinline__ u32 kmer_dense_read(const u32 *tile, const u32 *table, uint16_t *pend, u32 n_scan, u32 sh,
                                                      u32 mult, u32 keymask, u32 half, u32 &left) {
    u32 mine = 0;
    for (u32 w = threadIdx.x; w < n_scan; w += blockDim.x) {
        u32 m = pend[w];
        if (!m) continue;
        const u32 w0 = tile[w], w1 = tile[w + 1], pw = w << 4;
        if (m == 0xFFFFu) {
#pragma unroll
            for (u32 j = 0; j < 16; ++j) {
                const u32 mixed = kmer_mix_x<R0>(__funnelshift_l(w1, w0, 2 * j), sh, mult, keymask, half);
                const u32 tag = kmer_tag_of(mixed, pw + j);
                const u32 v = table[mixed & (KMER_TAG_SLOTS - 1)];
                mine += (v == tag) ? 1u : 0u;
                if (((v ^ tag) >> KMER_TAG_IDX_BITS) == 0) m &= ~(1u << j); // representative or its duplicate
            }
        } else {
#pragma unroll 4
            for (u32 j = 0; j < 16; ++j) {
                if ((m >> j) & 1u) {
                    const u32 mixed = kmer_mix_x<R0>(__funnelshift_l(w1, w0, 2 * j), sh, mult, keymask, half);
                    const u32 tag = kmer_tag_of(mixed, pw + j);
                    const u32 v = table[mixed & (KMER_TAG_SLOTS - 1)];
                    mine += (v == tag) ? 1u : 0u;
                    if (((v ^ tag) >> KMER_TAG_IDX_BITS) == 0) m &= ~(1u << j);
                }
            }
        }
        pend[w] = (uint16_t)m;
        left += __popc(m);
    }
    return mine;
}

// s_cnt: two u32 counters in shared memory.  Dense rounds walk the per-word masks; as soon as the pending
// k-mers fit list_a (cap_a entries) they are compacted into a position list and the remaining rounds only
// touch those (a round over the masks costs the same issue slots however few lanes are still pending).
// The second list aliases pend[], which is dead once the first list is built.
static __device__ u32 kmer_tag_count(const u32 *tile, u32 *table, uint16_t *pend, u32 *list_a, u32 cap_a,
                                     u32 *s_cnt, u32 shift, u32 p_end, int k) {
    const u32 kbits = 2u * (u32)k, sh = 32u - kbits, keymask = (1u << kbits) - 1u, half = max(kbits >> 1, 1u);
    const u32 n_scan = (p_end + 15) >> 4; // words holding the start of at least one k-mer
    const u32 lane = threadIdx.x & 31u;
    for (u32 w = threadIdx.x; w < n_scan; w += blockDim.x) {
        const u32 pw = w << 4;
        u32 m = 0xFFFFu;
        if (pw < shift) m &= 0xFFFFu << (shift - pw);
        if (pw + 16 > p_end) m &= 0xFFFFu >> (pw + 16 - p_end);
        pend[w] = (uint16_t)m;
    }
    if (threadIdx.x == 0) s_cnt[1] = 0;
    u32 mine = 0, round = 0, n_list = 0;
    for (;; ++round) { // ---- dense rounds ----
        const u32 mult = 0x9E3779B1u + 0x3C6EF372u * round; // odd for every round
        __syncthreads(); // pend / tile ready; everyone is done with the table and with s_cnt[0]
        if (threadIdx.x == 0) s_cnt[0] = 0;
        if (round == 0) kmer_dense_store<true>(tile, table, pend, n_scan, sh, mult, keymask, half);
        else kmer_dense_store<false>(tile, table, pend, n_scan, sh, mult, keymask, half);
        __syncthreads();
        u32 left = 0;
        if (round == 0) mine += kmer_dense_read<true>(tile, table, pend, n_scan, sh, mult, keymask, half, left);
        else mine += kmer_dense_read<false>(tile, table, pend, n_scan, sh, mult, keymask, half, left);
        left = __reduce_add_sync(0xffffffffu, left);
        if (lane == 0 && left) atomicAdd(&s_cnt[0], left);
        __syncthreads();
        const u32 total = s_cnt[0];
        if (total == 0) return mine;
        if (total <= cap_a) { // compact the pending positions into list_a
            for (u32 w0 = (threadIdx.x & ~31u); w0 < n_scan; w0 += KMER_SB_THREADS) { // warp-uniform trip count
                const u32 w = w0 + lane;
                u32 m = (w < n_scan) ? pend[w] : 0u;
                const u32 c = __popc(m);
                u32 incl = c;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const u32 t = __shfl_up_sync(0xffffffffu, incl, d);
                    if ((int)lane >= d) incl += t;
                }
                const u32 wtot = __shfl_sync(0xffffffffu, incl, 31);
                u32 base = 0;
                if (lane == 0 && wtot) base = atomicAdd(&s_cnt[1], wtot);
                base = __shfl_sync(0xffffffffu, base, 0);
                u32 off = base + incl - c;
                while (m) {
                    const u32 j = (u32)__ffs((int)m) - 1u;
                    m &= m - 1u;
                    list_a[off++] = (w << 4) + j;
                }
            }
            n_list = total;
            break;
        }
    }
    // ---- list rounds ----
    u32 *cur = list_a, *nxt = (u32 *)pend;
    u32 ci = 0;
    __syncthreads(); // list_a complete; pend[] is dead from here on
    while (n_list) {
        if (n_list <= 64) {
            // tail: the few keys left are compared pairwise (a round costs ~100 issue slots in every warp of
            // the CTA however short the list is, and each round only resolves ~80 % of it)
            u32 key = 0;
            if (threadIdx.x < n_list) {
                const u32 pos = cur[threadIdx.x], w = pos >> 4;
                key = __funnelshift_l(tile[w + 1], tile[w], 2 * (pos & 15u)) >> sh;
                nxt[threadIdx.x] = key;
            }
            __syncthreads();
            if (threadIdx.x < n_list) {
                bool dup = false;
                for (u32 j = 0; j < threadIdx.x; ++j) dup |= nxt[j] == key;
                mine += dup ? 0u : 1u;
            }
            break;
        }
        ++round;
        const u32 mult = 0x9E3779B1u + 0x3C6EF372u * round;
        if (threadIdx.x == 0) s_cnt[ci] = 0;
        for (u32 i = threadIdx.x; i < n_list; i += KMER_SB_THREADS) {
            const u32 pos = cur[i], w = pos >> 4;
            const u32 mixed = kmer_mix(__funnelshift_l(tile[w + 1], tile[w], 2 * (pos & 15u)) >> sh, mult, keymask, half);
            table[mixed & (KMER_TAG_SLOTS - 1)] = kmer_tag_of(mixed, pos);
        }
        __syncthreads();
        for (u32 i0 = (threadIdx.x & ~31u); i0 < n_list; i0 += KMER_SB_THREADS) { // warp-uniform trip count
            const u32 i = i0 + lane;
            bool lost = false;
            u32 pos = 0;
            if (i < n_list) {
                pos = cur[i];
                const u32 w = pos >> 4;
                const u32 mixed = kmer_mix(__funnelshift_l(tile[w + 1], tile[w], 2 * (pos & 15u)) >> sh, mult, keymask, half);
                const u32 tag = kmer_tag_of(mixed, pos);
                const u32 v = table[mixed & (KMER_TAG_SLOTS - 1)];
                mine += (v == tag) ? 1u : 0u;
                lost = ((v ^ tag) >> KMER_TAG_IDX_BITS) != 0;
            }
            const u32 bal = __ballot_sync(0xffffffffu, lost);
            if (bal) {
                u32 base = 0;
                if (lane == 0) base = atomicAdd(&s_cnt[ci], (u32)__popc(bal));
                base = __shfl_sync(0xffffffffu, base, 0);
                if (lost) nxt[base + __popc(bal & ((1u << lane) - 1u))] = pos;
            }
        }
        __syncthreads();
        n_list = s_cnt[ci];
        u32 *t = cur; cur = nxt; nxt = t;
        ci ^= 1u;
    }
    return mine;
}

__global__ void __launch_bounds__(KMER_SB_THREADS, 1)
k_kmer_smem(DevBatch B, DevParams P, tgsf_piece *pieces, const u32 *__restrict__ n_pieces_ptr,
            u64 *__restrict__ counters, const u32 *__restrict__ dev_status,
            const u32 *__restrict__ piece_list) { // the long list k_kmer_tag16 left; n_pieces_ptr counts its entries
    if (*dev_status != DEV_STATUS_OK) return;
    extern __shared__ __align__(16) uint8_t kmem[];
    u32 *bm = (u32 *)kmem;
    u32 *tile = (u32 *)(kmem + KMER_SB_BITMAP_BYTES);
    __shared__ u32 s_distinct;
    __shared__ u32 s_cnt[2];
    const int k = P.kmer;
    const u32 keyspace = 1u << (2 * k);                       // k <= 12
    const u32 passes = (keyspace + KMER_SB_BITS - 1) / KMER_SB_BITS;
    const u32 clear_vec = (min(keyspace, KMER_SB_BITS) / 8 + 15) / 16; // uint4 stores per pass
    const u32 n_pieces = *n_pieces_ptr;
    const u64 n_total = B.offsets[B.n_reads];
    const u32 tile_kmers = KMER_SB_TILE_WORDS * 16 - 16 - (u32)(k - 1); // k-mers one staged tile can hold (15 bases of slack for the alignment shift)

    for (u32 li = blockIdx.x; li < n_pieces; li += gridDim.x) {
        const u32 pi = piece_list[li];
        tgsf_piece pc = pieces[pi];
        if (pc.status != TGSF_PIECE_EMIT) continue;
        const int total = pc.len - k + 1;
        int repeat = 0;
        if (total <= 0) {
            repeat = total - 1; // see oracle/tgsf_oracle.c kmer_repeat_len
        } else {
            const u64 seq0 = B.offsets[pc.read] + (u64)pc.start; // absolute offset of the piece
            const u32 n_tiles = ((u32)total + tile_kmers - 1) / tile_kmers;
            if (threadIdx.x == 0) s_distinct = 0;
            u32 mine = 0;
            if (n_tiles == 1) { // the whole piece fits one staged tile: tag rounds, no atomics
                const u64 abase = seq0 & ~15ull;
                const u32 shift = (u32)(seq0 - abase);
                __syncthreads(); // the previous piece is done with tile / table
                kmer_stage_tile(B, n_total, abase, (shift + (u32)total + (u32)k - 1 + 15) / 16, tile);
                // shared layout of this path: table 128 KB | pend masks 24 KB (later: second list) | first list 20 KB | tile
                mine = kmer_tag_count(tile, bm, (uint16_t *)(kmem + KMER_TAG_SLOTS * 4),
                                      (u32 *)(kmem + KMER_TAG_SLOTS * 4 + KMER_SB_TILE_WORDS * 2),
                                      (KMER_SB_BITMAP_BYTES - KMER_TAG_SLOTS * 4 - KMER_SB_TILE_WORDS * 2) / 4, s_cnt, shift,
                                      shift + (u32)total, k);
            } else
            for (u32 pass = 0; pass < passes; ++pass) {
                const u32 lo = pass * KMER_SB_BITS;
                __syncthreads(); // previous pass / piece is done with the bitmap
                for (u32 i = threadIdx.x; i < clear_vec; i += KMER_SB_THREADS) ((uint4 *)bm)[i] = make_uint4(0, 0, 0, 0);
                for (u32 t = 0; t < n_tiles; ++t) {
                    const u32 km0 = t * tile_kmers, cnt = min(tile_kmers, (u32)total - km0);
                    const u64 first = seq0 + km0;            // first base of the tile
                    const u64 abase = first & ~15ull;        // staged from the aligned address below it
                    const u32 shift = (u32)(first - abase);  // position of k-mer 0 in the staged stream
                    __syncthreads(); // readers of the previous tile are done
                    kmer_stage_tile(B, n_total, abase, (shift + cnt + (u32)k - 1 + 15) / 16, tile);
                    __syncthreads(); // bitmap cleared, tile staged
                    // each thread: 16 consecutive stream positions of one word.  x = the 32 stream bits from
                    // position p on; its top 2k bits are the k-mer, so the pass's key range is tested on x itself.
                    const u32 p_end = shift + cnt; // stream positions [shift, p_end) start a k-mer
                    const u32 sh = 32u - 2u * (u32)k;
                    // used when passes > 1 (k >= 11).  The last range is cut at the key space so that
                    // lo_s + span_s never passes 2^32 (the unsigned compare below would wrap around)
                    const u32 lo_s = lo << sh, span_s = min(KMER_SB_BITS, keyspace - lo) << sh;
                    for (u32 w = threadIdx.x; (w << 4) < p_end; w += KMER_SB_THREADS) {
                        const u32 w0 = tile[w], w1 = tile[w + 1];
                        const u32 pw = w << 4;
                        const bool interior = pw >= shift && pw + 16 <= p_end;
                        if (interior) {
#pragma unroll
                            for (u32 j = 0; j < 16; ++j) {
                                const u32 x = __funnelshift_l(w1, w0, 2 * j);
                                if (passes == 1 || x - lo_s < span_s) {
                                    const u32 rel = (x >> sh) - lo;
                                    const u32 bit = 1u << (rel & 31u);
                                    const u32 old = atomicOr(bm + (rel >> 5), bit);
                                    mine += (old & bit) ? 0u : 1u;
                                }
                            }
                        } else {
#pragma unroll 4
                            for (u32 j = 0; j < 16; ++j) {
                                const u32 pp = pw + j;
                                const u32 x = __funnelshift_l(w1, w0, 2 * j);
                                if (pp >= shift && pp < p_end && (passes == 1 || x - lo_s < span_s)) {
                                    const u32 rel = (x >> sh) - lo;
                                    const u32 bit = 1u << (rel & 31u);
                                    const u32 old = atomicOr(bm + (rel >> 5), bit);
                                    mine += (old & bit) ? 0u : 1u;
                                }
                            }
                        }
                    }
                }
            }
            atomicAdd(&s_distinct, mine);
            __syncthreads();
        }
        if (threadIdx.x == 0) {
            if (total > 0) repeat = total - (int)*(volatile u32 *)&s_distinct; // thread 0 alone reads and resets it
            pc.repeat_len = repeat;
            if (repeat < P.min_repeat) { // T.cpp:1984-1988
                pc.status = TGSF_PIECE_SHORT_REPEAT;
                atomic_add_u64(counters + P.L.drop_info + 15, 1ull);
                atomic_add_u64(counters + P.L.drop_info + 16, (u64)pc.len);
            }
            pieces[pi] = pc;
        }
    }
}
