// K1: per-segment quality sum + per-100 bp x {A,T,G,C,all} count / quality-sum bins, the read-end
// (5'/3') per-position tables and the mean-quality decisions.
//
// Replaces CalcAvgQuality (T.cpp:1436-1479), Get_5p/3p_base_qual (T.cpp:1481-1575), the FASTA
// variants Get_base_counts / Get_5p/3p_base_counts (T.cpp:1577-1678, typos included) and the
// quality-band checks + histograms of filter_sequence (T.cpp:1942-1952, 1994-2002).
//
// HBM-bound by design: 2 algorithmic bytes per base.  One warp owns one 3200-base tile; the two
// byte streams of the tile are brought into shared memory with one bulk-async (TMA) copy each,
// double-buffered per warp; lane l then owns bin l of the tile (100 bases = 25 words at a lane
// stride of 25 words: bank-conflict free), classifies 4 bases per 32-bit word with SWAR masks and
// accumulates counts / quality sums with dp4a.  Bins below SCAN_SMEM_BINS are privatised per CTA in
// shared memory and flushed once; deeper bins (reads > 102 kb) go to L2 atomics.
//
// The privatised quality sums are 32-bit when no CTA can reach 2^31 in one bin: a tile adds at most
// 100 x (128 + |qtype|) to a bin, and the host knows how many tiles a CTA can take (scan_needs_wide).
// Otherwise (few CTAs over very many reads: one CTA, 100-bp reads at Q93 pass 2^31 after ~230 k
// reads) the WIDE kernel keeps them in 64 bits.  The counts stay 32-bit: at most 100 per tile, so
// they hold for < 42.9 M tiles per CTA, more than any batch has.
#pragma once
#include "common.cuh"

#define SCAN_WARPS 12
#define SCAN_THREADS (SCAN_WARPS * 32)
#define SCAN_STAGES 2
#define SCAN_BUF (SCAN_TILE + 32) /* aligned superset of one tile of one stream */
#define SCAN_SMEM_BINS 1024
#define SCAN_SMEM_BYTES \
    (SCAN_WARPS * SCAN_STAGES * 2 * SCAN_BUF + SCAN_SMEM_BINS * 10 * 4 + SCAN_WARPS * SCAN_STAGES * 8)
#define SCAN_SMEM_BYTES_WIDE (SCAN_SMEM_BYTES + SCAN_SMEM_BINS * 5 * 4) /* quality sums in 64 bits */

// Whether k_scan_tiles_dyn must keep its shared quality sums in 64 bits for a launch of `grid` CTAs over
// at most `max_tiles` tiles.
static inline bool scan_needs_wide(u64 max_tiles, int grid, int qtype) {
    const u64 per_cta = max_tiles / (u64)grid + SCAN_WARPS; // tiles are dealt to warps round-robin
    const u64 per_tile = (u64)SCAN_BIN * (u64)(128 + (qtype < 0 ? -(i64)qtype : (i64)qtype));
    return per_cta * per_tile >= (1ull << 31);
}

static __device__ __forceinline__ u32 smem_u32(const void *p) {
    return (u32)__cvta_generic_to_shared(p);
}
static __device__ __forceinline__ void mbar_init(u32 bar, u32 count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
static __device__ __forceinline__ void mbar_expect_tx(u32 bar, u32 bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
                 : "memory");
}
static __device__ __forceinline__ void mbar_wait(u32 bar, u32 parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra WAIT_DONE;\n"
        "bra WAIT_LOOP;\n"
        "WAIT_DONE:\n"
        "}\n" ::"r"(bar),
        "r"(parity)
        : "memory");
}
// 1-D bulk async copy global -> shared (TMA engine, SASS UBLKCP), completion on an mbarrier.
static __device__ __forceinline__ void bulk_g2s(u32 dst, const void *src, u32 bytes, u32 bar) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
        "l"(src), "r"(bytes), "r"(bar)
        : "memory");
}

// 0x80 in every byte of x that is zero.
static __device__ __forceinline__ u32 zero_bytes80(u32 x) {
    return ~(((x & 0x7f7f7f7fu) + 0x7f7f7f7fu) | x) & 0x80808080u;
}
// signed bytes of a times unsigned bytes of b, accumulated.
static __device__ __forceinline__ int dp4a_su(u32 a, u32 b, int c) {
    int d;
    asm("dp4a.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
static __device__ __forceinline__ u32 dp4a_uu(u32 a, u32 b, u32 c) {
    u32 d;
    asm("dp4a.u32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}

struct BinAcc {
    u32 c128[4]; // 128 x count of A,T,G,C
    int q128[4]; // 128 x sum of raw quality bytes per category
    int qall;    // sum of raw quality bytes
};

template <bool HAS_QUAL>
static __device__ __forceinline__ void scan_word(BinAcc &a, u32 bw, u32 qw) {
    const u32 u = bw & 0xdfdfdfdfu; // fold case: 'a'..'z' -> 'A'..'Z'
    const u32 mA = zero_bytes80(u ^ 0x41414141u);
    const u32 mT = zero_bytes80(u ^ 0x54545454u);
    const u32 mG = zero_bytes80(u ^ 0x47474747u);
    const u32 mC = zero_bytes80(u ^ 0x43434343u);
    a.c128[0] = dp4a_uu(mA, 0x01010101u, a.c128[0]);
    a.c128[1] = dp4a_uu(mT, 0x01010101u, a.c128[1]);
    a.c128[2] = dp4a_uu(mG, 0x01010101u, a.c128[2]);
    a.c128[3] = dp4a_uu(mC, 0x01010101u, a.c128[3]);
    if (HAS_QUAL) {
        a.q128[0] = dp4a_su(qw, mA, a.q128[0]);
        a.q128[1] = dp4a_su(qw, mT, a.q128[1]);
        a.q128[2] = dp4a_su(qw, mG, a.q128[2]);
        a.q128[3] = dp4a_su(qw, mC, a.q128[3]);
        a.qall = dp4a_su(qw, 0x01010101u, a.qall);
    }
}

// bases/quals: whole batch streams (16-byte aligned, readable up to the next 16-byte boundary
// past the last segment).  tiles: self-contained records (reads in the raw pass, kept pieces in
// the clean pass).  seg_sum[seg] += sum(q - qtype).
template <bool HAS_QUAL, bool WIDE>
__global__ void __launch_bounds__(SCAN_THREADS, 1)
k_scan_tiles_dyn(const uint8_t *__restrict__ bases, const uint8_t *__restrict__ quals,
                 const TileEntry *__restrict__ tiles, const u32 *__restrict__ n_tiles_ptr,
                 u64 *__restrict__ seg_sum, u64 *__restrict__ bin_cnt, u64 *__restrict__ bin_qual,
                 int qtype, u32 max_bins, u32 *__restrict__ dev_status) {
    extern __shared__ __align__(128) uint8_t smem[];
    const u32 n_tiles = *n_tiles_ptr; // device-side total (tile_off[n_seg])
    uint8_t *stage_base = smem;
    // narrow: [bin][10] u32 = 5 counts, 5 quality sums.  WIDE: [bin][5] u32 counts, then [bin][5] u64 sums.
    u32 *sbins = (u32 *)(smem + SCAN_WARPS * SCAN_STAGES * 2 * SCAN_BUF);
    u64 *squal = (u64 *)(sbins + SCAN_SMEM_BINS * 5);
    u64 *bars = (u64 *)(sbins + SCAN_SMEM_BINS * (WIDE ? 15 : 10));

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = threadIdx.x; i < SCAN_SMEM_BINS * (WIDE ? 15 : 10); i += SCAN_THREADS) sbins[i] = 0;
    if (threadIdx.x < SCAN_WARPS * SCAN_STAGES) mbar_init(smem_u32(&bars[threadIdx.x]), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    __syncthreads();

    const u32 warps_total = gridDim.x * SCAN_WARPS;
    const u32 gwarp = blockIdx.x * SCAN_WARPS + warp;
    uint8_t *wbuf = stage_base + (size_t)warp * SCAN_STAGES * 2 * SCAN_BUF;
    u64 *wbar = bars + warp * SCAN_STAGES;
    const uint4 *__restrict__ tile4 = (const uint4 *)tiles;

    auto load_entry = [&](u32 t) -> TileEntry {
        TileEntry te;
        te.start = 0; te.seg = 0; te.tile = 0;
        if (t < n_tiles) {
            const uint4 v = __ldg(tile4 + t);
            te.start = ((u64)v.y << 32) | v.x;
            te.seg = v.z;
            te.tile = v.w;
        }
        return te;
    };
    // issue the two bulk copies of a tile into stage st (lane 0 only)
    auto issue = [&](const TileEntry &te, int st) {
        const u64 a0 = te.start;
        const int n = (int)(te.tile & ((1u << TILE_N_BITS) - 1u));
        const u64 al = a0 & ~15ull;
        const u32 bytes = (u32)(((a0 - al) + (u64)n + 15ull) & ~15ull);
        const u32 bar = smem_u32(&wbar[st]);
        uint8_t *dst = wbuf + (size_t)st * 2 * SCAN_BUF;
        mbar_expect_tx(bar, HAS_QUAL ? 2 * bytes : bytes);
        bulk_g2s(smem_u32(dst), bases + al, bytes, bar);
        if (HAS_QUAL) bulk_g2s(smem_u32(dst + SCAN_BUF), quals + al, bytes, bar);
    };

    u32 t = gwarp;
    int st = 0;
    u32 phase = 0;
    TileEntry cur = load_entry(t);
    TileEntry nxt = load_entry(t + warps_total);
    if (t < n_tiles && lane == 0) issue(cur, 0);
    for (; t < n_tiles; t += warps_total) {
        if (t + warps_total < n_tiles && lane == 0) issue(nxt, st ^ 1);
        const TileEntry nxt2 = load_entry(t + 2 * warps_total); // metadata two tiles ahead
        const TileEntry te = cur;
        const u64 a0 = te.start;
        const int n = (int)(te.tile & ((1u << TILE_N_BITS) - 1u));
        const u32 tile_idx = te.tile >> TILE_N_BITS;
        const u32 a = (u32)(a0 & 15ull);
        mbar_wait(smem_u32(&wbar[st]), phase);

        const int nvalid = min(max(n - SCAN_BIN * lane, 0), SCAN_BIN);
        BinAcc acc;
#pragma unroll
        for (int c = 0; c < 4; ++c) { acc.c128[c] = 0; acc.q128[c] = 0; }
        acc.qall = 0;
        if (nvalid > 0) {
            const uint8_t *sb = wbuf + (size_t)st * 2 * SCAN_BUF;
            const u32 off = a + SCAN_BIN * lane;
            const u32 *bwp = (const u32 *)(sb + (off & ~3u));
            const u32 *qwp = (const u32 *)(sb + SCAN_BUF + (off & ~3u));
            const u32 sh = (off & 3u) * 8u;
            if (nvalid == SCAN_BIN) {
                u32 b0 = bwp[0], q0 = HAS_QUAL ? qwp[0] : 0u;
#pragma unroll
                for (int w = 0; w < SCAN_BIN / 4; ++w) {
                    const u32 b1 = bwp[w + 1];
                    const u32 q1 = HAS_QUAL ? qwp[w + 1] : 0u;
                    scan_word<HAS_QUAL>(acc, __funnelshift_r(b0, b1, sh), __funnelshift_r(q0, q1, sh));
                    b0 = b1;
                    q0 = q1;
                }
            } else {
                u32 b0 = bwp[0], q0 = HAS_QUAL ? qwp[0] : 0u;
                for (int w = 0; w * 4 < nvalid; ++w) {
                    const u32 b1 = bwp[w + 1];
                    const u32 q1 = HAS_QUAL ? qwp[w + 1] : 0u;
                    const int v = nvalid - w * 4;
                    const u32 m = v >= 4 ? 0xffffffffu : ((1u << (8 * v)) - 1u);
                    scan_word<HAS_QUAL>(acc, __funnelshift_r(b0, b1, sh) & m,
                                        __funnelshift_r(q0, q1, sh) & m);
                    b0 = b1;
                    q0 = q1;
                }
            }
        }
        // fold the x128 scaling and the Phred offset: sum(q - qtype) = sum(q) - qtype * count
        u32 cnt[5];
        int qs[5];
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            cnt[c] = acc.c128[c] >> 7;
            qs[c] = (acc.q128[c] >> 7) - qtype * (int)cnt[c];
        }
        cnt[4] = (u32)nvalid;
        qs[4] = acc.qall - qtype * nvalid;
        if (nvalid > 0) {
            const u32 gb = tile_idx * SCAN_TILE_BINS + lane;
            if (gb < SCAN_SMEM_BINS) {
                u32 *p = sbins + gb * (WIDE ? 5 : 10);
#pragma unroll
                for (int c = 0; c < 5; ++c) {
                    if (cnt[c]) atomicAdd(p + c, cnt[c]);
                    if (HAS_QUAL && qs[c]) {
                        if constexpr (WIDE) atomicAdd(squal + gb * 5 + c, (u64)(i64)qs[c]);
                        else atomicAdd(p + 5 + c, (u32)qs[c]);
                    }
                }
            } else if (gb < max_bins) {
#pragma unroll
                for (int c = 0; c < 5; ++c) {
                    if (cnt[c]) atomic_add_u64(bin_cnt + (u64)gb * 5 + c, (u64)cnt[c]);
                    if (HAS_QUAL && qs[c]) atomic_add_u64(bin_qual + (u64)gb * 5 + c, (u64)(i64)qs[c]);
                }
            } else {
                *dev_status = DEV_STATUS_BIN_OVERFLOW;
            }
        }
        if (HAS_QUAL) {
            const i64 ws = warp_sum_i64((i64)qs[4]);
            if (lane == 0) atomic_add_u64(seg_sum + te.seg, (u64)ws);
        }
        __syncwarp();
        st ^= 1;
        if (st == 0) phase ^= 1;
        cur = nxt;
        nxt = nxt2;
    }
    __syncthreads();
    for (int i = threadIdx.x; i < SCAN_SMEM_BINS * 5; i += SCAN_THREADS) {
        const int b = i / 5, c = i % 5;
        if ((u32)b >= max_bins) continue;
        const u32 vc = sbins[b * (WIDE ? 5 : 10) + c];
        if (vc) atomic_add_u64(bin_cnt + (u64)b * 5 + c, (u64)vc);
        if (HAS_QUAL) {
            const u64 vq = WIDE ? squal[i] : (u64)(i64)(int)sbins[b * 10 + 5 + c];
            if (vq) atomic_add_u64(bin_qual + (u64)b * 5 + c, vq);
        }
    }
}

// ---------------------------------------------------------------------------------------------
// Read-end tables.  One warp per segment; lanes stride over the first / last min(bc_len, len)
// positions; per-CTA shared tables when bc_len <= ENDS_SMEM_ROWS.
// ---------------------------------------------------------------------------------------------
#define ENDS_THREADS 256
#define ENDS_SMEM_ROWS 256

static __device__ __forceinline__ int base_cat(uint8_t b) { // T.cpp:1462-1474
    const uint8_t u = b & 0xdf;
    return u == 'A' ? 0 : u == 'T' ? 1 : u == 'G' ? 2 : u == 'C' ? 3 : -1;
}

// tables: cnt5, qual5, cnt3, qual3 -> each [bc_len][5] u64 in the counter block.
// seg_flag (may be null): only segments with flag != 0 are counted.
template <bool HAS_QUAL>
__global__ void __launch_bounds__(ENDS_THREADS)
k_ends_qc(const uint8_t *__restrict__ bases, const uint8_t *__restrict__ quals, u32 n_seg,
          const u64 *__restrict__ seg_start, const int *__restrict__ seg_len,
          const int *__restrict__ seg_flag, int bc_len, int qtype, u64 *cnt5, u64 *qual5, u64 *cnt3,
          u64 *qual3) {
    extern __shared__ u32 sm[]; // [2][rows][10] when rows <= ENDS_SMEM_ROWS
    const bool use_smem = bc_len <= ENDS_SMEM_ROWS;
    if (use_smem) {
        for (int i = threadIdx.x; i < 2 * bc_len * 10; i += ENDS_THREADS) sm[i] = 0;
        __syncthreads();
    }
    const int lane = threadIdx.x & 31;
    const u32 wpb = ENDS_THREADS / 32;
    for (u32 sgi = blockIdx.x * wpb + (threadIdx.x >> 5); sgi < n_seg; sgi += gridDim.x * wpb) {
        const int len = seg_len[sgi];
        if (len <= 0 || (seg_flag && !seg_flag[sgi])) continue;
        const u64 s0 = seg_start[sgi];
        const int n = min(bc_len, len);
        for (int i = lane; i < n; i += 32) {
#pragma unroll
            for (int side = 0; side < 2; ++side) {
                const u64 p = side == 0 ? s0 + (u64)i : s0 + (u64)(len - 1 - i);
                const uint8_t b = bases[p];
                int c = base_cat(b);
                if (!HAS_QUAL) { // typos of the FASTA path: T.cpp:1634 ('g') and T.cpp:1669 ('t')
                    if (side == 0 && b == 'g') c = -1;
                    if (side == 1 && b == 't') c = -1;
                }
                const int qv = HAS_QUAL ? (int)(signed char)quals[p] - qtype : 0;
                if (use_smem) {
                    u32 *row = sm + (side * bc_len + i) * 10;
                    if (c >= 0) {
                        atomicAdd(row + c, 1u);
                        if (HAS_QUAL) atomicAdd(row + 5 + c, (u32)qv);
                    }
                    atomicAdd(row + 4, 1u);
                    if (HAS_QUAL) atomicAdd(row + 9, (u32)qv);
                } else {
                    u64 *ct = side == 0 ? cnt5 : cnt3;
                    u64 *qt = side == 0 ? qual5 : qual3;
                    if (c >= 0) {
                        atomic_add_u64(ct + (u64)i * 5 + c, 1ull);
                        if (HAS_QUAL) atomic_add_u64(qt + (u64)i * 5 + c, (u64)(i64)qv);
                    }
                    atomic_add_u64(ct + (u64)i * 5 + 4, 1ull);
                    if (HAS_QUAL) atomic_add_u64(qt + (u64)i * 5 + 4, (u64)(i64)qv);
                }
            }
        }
    }
    // The shared sums are 32-bit, which is enough: one CTA takes every (4 x sm_count)-th segment of a launch,
    // and a row adds at most |qv| <= 192 per segment, so a sum stays below 2^31 up to 11.1 M segments per CTA,
    // i.e. 44.7 M x sm_count segments per launch (a batch has at most 2^24 reads).
    if (use_smem) {
        __syncthreads();
        for (int i = threadIdx.x; i < 2 * bc_len * 5; i += ENDS_THREADS) {
            const int side = i / (bc_len * 5), r = (i / 5) % bc_len, c = i % 5;
            const u32 vc = sm[(side * bc_len + r) * 10 + c];
            const int vq = (int)sm[(side * bc_len + r) * 10 + 5 + c];
            u64 *ct = side == 0 ? cnt5 : cnt3;
            u64 *qt = side == 0 ? qual5 : qual3;
            if (vc) atomic_add_u64(ct + (u64)r * 5 + c, (u64)vc);
            if (HAS_QUAL && vq) atomic_add_u64(qt + (u64)r * 5 + c, (u64)(i64)vq);
        }
    }
}

static __device__ __forceinline__ int qual_hist_index(double q) { // int(rawQuality), T.cpp:1943
    if (!(q >= 0.0)) return 0;
    if (q >= 255.0) return 255;
    return (int)q;
}
