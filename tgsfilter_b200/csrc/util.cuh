// Plumbing kernels: segment / tile / chunk tables and the exclusive scan they are built with.
#pragma once
#include "common.cuh"

#define UTIL_THREADS 256
#define SCANB_ITEMS 8
#define SCANB_TILE (UTIL_THREADS * SCANB_ITEMS)

// Block-level exclusive scan of in[0..n) into out[0..n); block totals into sums[blockIdx].
__global__ void __launch_bounds__(UTIL_THREADS)
k_scan_block(const u32 *__restrict__ in, u32 *__restrict__ out, u32 n, u32 *__restrict__ sums) {
    __shared__ u32 warp_tot[UTIL_THREADS / 32];
    const u32 base = blockIdx.x * SCANB_TILE + threadIdx.x * SCANB_ITEMS;
    u32 v[SCANB_ITEMS];
    u32 tsum = 0;
#pragma unroll
    for (int i = 0; i < SCANB_ITEMS; ++i) {
        v[i] = (base + i < n) ? in[base + i] : 0u;
        tsum += v[i];
    }
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    u32 inc = tsum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const u32 t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) warp_tot[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        u32 w = lane < UTIL_THREADS / 32 ? warp_tot[lane] : 0u;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const u32 t = __shfl_up_sync(0xffffffffu, w, o);
            if (lane >= o) w += t;
        }
        if (lane < UTIL_THREADS / 32) warp_tot[lane] = w; // inclusive
    }
    __syncthreads();
    u32 excl = inc - tsum + (warp ? warp_tot[warp - 1] : 0u);
#pragma unroll
    for (int i = 0; i < SCANB_ITEMS; ++i) {
        if (base + i < n) out[base + i] = excl;
        excl += v[i];
    }
    if (threadIdx.x == UTIL_THREADS - 1) sums[blockIdx.x] = excl;
}

// out[i] += sums_scanned[block]; also writes the grand total to out[n].
__global__ void __launch_bounds__(UTIL_THREADS)
k_scan_add(u32 *__restrict__ out, u32 n, const u32 *__restrict__ sums_scanned,
           const u32 *__restrict__ total) {
    const u32 i = blockIdx.x * UTIL_THREADS + threadIdx.x;
    if (i < n) out[i] += sums_scanned[i / SCANB_TILE];
    if (i == 0) out[n] = *total;
}

// Raw pass segments = reads.  Also validates the read length against the bin capacity.
__global__ void k_read_segments(DevBatch B, u64 *__restrict__ seg_start, int *__restrict__ seg_len,
                                u64 *__restrict__ seg_sum, u32 *__restrict__ n_tiles, u32 max_bins,
                                u32 *__restrict__ dev_status) {
    const u32 r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= B.n_reads) return;
    const u64 s = B.offsets[r];
    const u64 len = B.offsets[r + 1] - s;
    if (len / SCAN_BIN + 1 > (u64)max_bins || len > 0x7fffffffull) {
        *dev_status = DEV_STATUS_BIN_OVERFLOW;
        seg_len[r] = 0;
        n_tiles[r] = 0;
        seg_start[r] = s;
        seg_sum[r] = 0;
        return;
    }
    seg_start[r] = s;
    seg_len[r] = (int)len;
    seg_sum[r] = 0;
    n_tiles[r] = (u32)((len + SCAN_TILE - 1) / SCAN_TILE);
}

// Self-contained tile records (start, length, owner) so that the scan kernel needs exactly one
// 16-byte load per tile, prefetched a tile ahead.
__global__ void k_fill_tiles(const u32 *__restrict__ tile_off, u32 n_seg,
                             const u64 *__restrict__ seg_start, const int *__restrict__ seg_len,
                             TileEntry *__restrict__ tiles) {
    const u32 s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_seg) return;
    const u32 b = tile_off[s], e = tile_off[s + 1];
    const u64 s0 = seg_start[s];
    const int len = seg_len[s];
    for (u32 t = b; t < e; ++t) {
        const u32 ti = t - b;
        TileEntry te;
        te.start = s0 + (u64)ti * SCAN_TILE;
        te.seg = s;
        te.tile = (ti << TILE_N_BITS) | (u32)min(len - (int)(ti * SCAN_TILE), SCAN_TILE);
        tiles[t] = te;
    }
}

// Number of absolute 2^chunk_shift blocks (chunks) and 2^(chunk_shift + run_shift) blocks (runs of the middle scan)
// overlapping the middle window of each active read (0 when the window is shorter than the shortest adapter:
// tsmLen >= qLen, T.cpp:1237).
__global__ void k_count_chunks(DevBatch B, const int *__restrict__ read_active, int end_len,
                               int chunk_shift, int run_shift, int min_qlen, u32 *__restrict__ chunk_cnt,
                               u32 *__restrict__ run_cnt, u32 *__restrict__ best_mid, u32 *__restrict__ mid_n,
                               int n_adapters) {
    const u32 r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= B.n_reads) return;
    for (int a = 0; a < n_adapters; ++a) {
        best_mid[(u64)r * n_adapters + a] = 0xffffffffu;
        mid_n[(u64)r * n_adapters + a] = 0;
    }
    u32 c = 0, n = 0;
    if (read_active[r]) {
        const u64 rs = B.offsets[r], re = B.offsets[r + 1];
        const i64 tsm = (i64)(re - rs) - 2 * (i64)end_len;
        if (tsm >= (i64)min_qlen && tsm > 0) {
            const u64 mb = rs + (u64)end_len, me = re - (u64)end_len;
            c = (u32)(((me - 1) >> chunk_shift) - (mb >> chunk_shift) + 1);
            n = (u32)(((me - 1) >> (chunk_shift + run_shift)) - (mb >> (chunk_shift + run_shift)) + 1);
        }
    }
    chunk_cnt[r] = c;
    run_cnt[r] = n;
}

__global__ void k_fill_chunks(DevBatch B, const u32 *__restrict__ chunk_off, int end_len,
                              int block_shift, ChunkEntry *__restrict__ chunks) {
    const u32 r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= B.n_reads) return;
    const u32 b = chunk_off[r], e = chunk_off[r + 1];
    if (b == e) return;
    const u32 first = (u32)((B.offsets[r] + (u64)end_len) >> block_shift);
    for (u32 t = b; t < e; ++t) {
        ChunkEntry ce;
        ce.read = r;
        ce.chunk = first + (t - b);
        chunks[t] = ce;
    }
}

// k_fill_chunks fills the chunk table (block_shift = chunk_shift) or the run table (block_shift = chunk_shift +
// run_shift).
//
// Length-descending permutation of the run table (counting sort over 64 length buckets, block aggregated;
// block_shift = chunk_shift + run_shift).  k_mid_scan walks the runs in this order so that the
// 32 lanes of a warp (and the CTAs of a wave) work on runs of the same length: the first and last run of a
// read's window are partial and would otherwise idle their warp for part of a run.
#define CHUNK_BUCKETS 64
static __device__ __forceinline__ u32 chunk_bucket(const DevBatch &B, u32 r, u32 chunk, int end_len,
                                                   int block_shift) {
    const u64 mb = B.offsets[r] + (u64)end_len, me = B.offsets[r + 1] - (u64)end_len;
    const u64 cb = (u64)chunk << block_shift;
    const u64 ob = max(cb, mb), oe = min(cb + (1ull << block_shift), me);
    const u32 len = (u32)(oe - ob);
    return (CHUNK_BUCKETS - 1) - ((len - 1) >> (block_shift - 6)); // bucket 0 = longest
}

__global__ void __launch_bounds__(UTIL_THREADS)
k_chunk_hist(DevBatch B, const u32 *__restrict__ chunk_off, const ChunkEntry *__restrict__ chunks,
             int end_len, int block_shift, u32 *__restrict__ hist) {
    __shared__ u32 h[CHUNK_BUCKETS];
    if (threadIdx.x < CHUNK_BUCKETS) h[threadIdx.x] = 0;
    __syncthreads();
    const u32 r = blockIdx.x * UTIL_THREADS + threadIdx.x;
    if (r < B.n_reads)
        for (u32 t = chunk_off[r]; t < chunk_off[r + 1]; ++t)
            atomicAdd(&h[chunk_bucket(B, r, chunks[t].chunk, end_len, block_shift)], 1u);
    __syncthreads();
    if (threadIdx.x < CHUNK_BUCKETS && h[threadIdx.x]) atomicAdd(&hist[threadIdx.x], h[threadIdx.x]);
}

// hist[64] -> exclusive prefix in place (cursor of each bucket)
__global__ void k_chunk_base(u32 *__restrict__ hist) {
    if (threadIdx.x == 0) {
        u32 acc = 0;
        for (int b = 0; b < CHUNK_BUCKETS; ++b) {
            const u32 c = hist[b];
            hist[b] = acc;
            acc += c;
        }
    }
}

__global__ void __launch_bounds__(UTIL_THREADS)
k_chunk_scatter(DevBatch B, const u32 *__restrict__ chunk_off, const ChunkEntry *__restrict__ chunks,
                int end_len, int block_shift, u32 *__restrict__ cursor, u32 *__restrict__ perm) {
    __shared__ u32 cnt[CHUNK_BUCKETS], base[CHUNK_BUCKETS];
    if (threadIdx.x < CHUNK_BUCKETS) cnt[threadIdx.x] = 0;
    __syncthreads();
    const u32 r = blockIdx.x * UTIL_THREADS + threadIdx.x;
    const u32 b0 = r < B.n_reads ? chunk_off[r] : 0, b1 = r < B.n_reads ? chunk_off[r + 1] : 0;
    for (u32 t = b0; t < b1; ++t) atomicAdd(&cnt[chunk_bucket(B, r, chunks[t].chunk, end_len, block_shift)], 1u);
    __syncthreads();
    if (threadIdx.x < CHUNK_BUCKETS) {
        const u32 c = cnt[threadIdx.x];
        base[threadIdx.x] = c ? atomicAdd(&cursor[threadIdx.x], c) : 0u;
        cnt[threadIdx.x] = 0;
    }
    __syncthreads();
    for (u32 t = b0; t < b1; ++t) {
        const u32 k = chunk_bucket(B, r, chunks[t].chunk, end_len, block_shift);
        perm[base[k] + atomicAdd(&cnt[k], 1u)] = t;
    }
}

__global__ void k_check_pool(const u32 *__restrict__ pool_total, u32 pool_cap,
                             u32 *__restrict__ dev_status) {
    if (*pool_total > pool_cap) *dev_status = DEV_STATUS_POOL_OVERFLOW;
}

// dst[i] += src[i]: the reduction step of tgsf_allreduce (counter blocks of peer GPUs).
__global__ void k_add_u64(u64 *__restrict__ dst, const u64 *__restrict__ src, u32 n) {
    for (u32 i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) dst[i] += src[i];
}

// 2-bit packed bases (A0 C1 G2 T3, base i in bits 2*(i%4) of byte i/4) -> ASCII bytes.  One thread
// expands 4 packed bytes into one 16-byte store.  Bytes that are not upper-case ACGT travel as an
// exception list and are patched in afterwards, so the reconstructed stream is byte-identical to
// what the host parsed (edlib compares raw bytes, the QC counts fold case: SURVEY.md D5).
__global__ void k_unpack_bases(const u32 *__restrict__ packed, u64 n_words, uint4 *__restrict__ out) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n_words; i += (u64)gridDim.x * blockDim.x) {
        const u32 w = packed[i];
        u32 o[4];
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const u32 byte = (w >> (8 * b)) & 0xffu;
            // selector nibbles = the four 2-bit codes; table bytes = 'A','C','G','T'
            const u32 sel = (byte & 3u) | ((byte & 0xcu) << 2) | ((byte & 0x30u) << 4) | ((byte & 0xc0u) << 6);
            o[b] = __byte_perm(0x54474341u, 0u, sel);
        }
        out[i] = make_uint4(o[0], o[1], o[2], o[3]);
    }
}

__global__ void k_apply_exceptions(uint8_t *__restrict__ bases, const u64 *__restrict__ pos,
                                   const uint8_t *__restrict__ val, u64 n) {
    for (u64 i = (u64)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (u64)gridDim.x * blockDim.x)
        bases[pos[i]] = val[i];
}
