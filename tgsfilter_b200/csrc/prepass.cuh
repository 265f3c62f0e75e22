// K2 + pre-pass adapter search + the stand-alone alignment entry point.
//
// k_base_content : counting loop of CheckBaseContent (T.cpp:1080-1095)
// k_lib_search   : edlib loop of adapterSearch (T.cpp:1156-1176): maps[i] += mlen
// k_end_kmers    : k-mer counts of the sampled ends for the de novo adapter assembly (extension, tgsf_end_kmer_counts)
// k_align_pairs  : edlibAlign(HW, PATH) for independent (query, target) pairs (tgsf_align_hw)
#pragma once
#include "adapters.cuh"
#include "scan.cuh"

#define PRE_THREADS 256
// Columns per k_base_content tile: a [3072][4] u32 table is 48 KB, the dynamic shared memory a launch gets without
// an opt-in, so any row length is counted with the same table.
#define PRE_TILE_COLS 3072

// rows: [n][row_len] bytes; out: [row_len][4] int32 (A,T,G,C).  blockIdx.y picks a tile of PRE_TILE_COLS columns
// (the last one shorter); each CTA counts its rows over that tile in a shared-memory table and adds it to out.
__global__ void __launch_bounds__(PRE_THREADS)
k_base_content(const uint8_t *__restrict__ rows, u32 n, u32 row_len, int *__restrict__ out) {
    extern __shared__ u32 hist[]; // [cols][4]
    const u32 col0 = blockIdx.y * PRE_TILE_COLS;
    const u32 cols = min(row_len - col0, (u32)PRE_TILE_COLS);
    for (u32 i = threadIdx.x; i < cols * 4; i += PRE_THREADS) hist[i] = 0;
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const u32 wpb = PRE_THREADS / 32;
    for (u32 r = blockIdx.x * wpb + (threadIdx.x >> 5); r < n; r += gridDim.x * wpb) {
        const uint8_t *row = rows + (u64)r * row_len + col0;
        for (u32 i = lane; i < cols; i += 32) {
            const int c = base_cat(row[i]);
            if (c >= 0) atomicAdd(&hist[i * 4 + c], 1u);
        }
    }
    __syncthreads();
    int *tile_out = out + (u64)col0 * 4;
    for (u32 i = threadIdx.x; i < cols * 4; i += PRE_THREADS)
        if (hist[i]) atomicAdd(tile_out + i, (int)hist[i]);
}

// One thread per (row, library adapter).  k per adapter is DevAdapter::k_end (the host stores
// int((1 - minSim) * qLen) + 1 there for the library set).  maps: [n_lib] i64.
template <int NW>
__global__ void __launch_bounds__(RES_THREADS)
k_lib_search(const uint8_t *__restrict__ rows, u32 n, u32 row_len, AdapterCtx C, int a,
             long long *__restrict__ maps, u64 *scratch, u64 scratch_stride) {
    const DevAdapter A = C.ad[a];
    const AdapterTables T = adapter_tables(C, a);
    const u64 tid = (u64)blockIdx.x * RES_THREADS + threadIdx.x;
    long long acc = 0;
    for (u64 r = tid; r < n; r += (u64)gridDim.x * RES_THREADS) {
        const u64 lo = r * row_len, hi = lo + row_len;
        const int d = hw_best<NW>(T, rows, lo, hi, A.k_end);
        if (d == 0x7fffffff) continue;
        Myers<NW> s;
        myers_init_hw<NW>(s, T.qlen);
        for (u64 p = lo; p < hi; ++p) {
            myers_step<NW, 0, true>(s, T.hw + (u32)__ldg(rows + p) * NW, 0);
            if (s.score == d) {
                const u64 s0 = shw_start<NW>(T, rows, lo, p, d);
                const int alen = nw_alignment_len<NW>(T, rows, s0, p, d, scratch + tid, scratch_stride);
                acc += alen - d;
                break;
            }
        }
    }
    acc = warp_sum_i64(acc);
    if ((threadIdx.x & 31) == 0 && acc) atomicAdd((u64 *)maps, (u64)acc);
}

// k-mer counts of the sampled ends for the de novo adapter assembly (tgsf_end_kmer_counts).  One warp per row, grid
// stride; the windows [w_lo, w_hi) of a row (window j = row[j, j+k)) are cut into 32 contiguous runs, one per lane,
// and each lane rolls a 2-bit code (A0 C1 G2 T3, first base most significant) over its run.  A window counts only
// when its k bytes are all upper-case A/C/G/T.  table: [4^k] u32, one band (outer or inner) per launch.
__global__ void __launch_bounds__(PRE_THREADS)
k_end_kmers(const uint8_t *__restrict__ rows, u32 n, u32 row_len, int k, u32 w_lo, u32 w_hi,
            u32 *__restrict__ table) {
    const int lane = threadIdx.x & 31;
    const u32 wpb = PRE_THREADS / 32;
    const u32 per_lane = (w_hi - w_lo + 31) / 32;
    const u32 j0 = min(w_lo + lane * per_lane, w_hi), j1 = min(j0 + per_lane, w_hi);
    if (j0 == j1) return; // no barrier below: idle lanes may leave
    const u32 mask = (1u << (2 * k)) - 1u; // k <= 13
    for (u32 r = blockIdx.x * wpb + (threadIdx.x >> 5); r < n; r += gridDim.x * wpb) {
        const uint8_t *row = rows + (u64)r * row_len;
        u32 code = 0;
        int run = 0; // valid bases ending at column c, counted from j0
        for (u32 c = j0; c < j1 + k - 1; ++c) {
            const uint8_t b = __ldg(row + c);
            const int v = b == 'A' ? 0 : b == 'C' ? 1 : b == 'G' ? 2 : b == 'T' ? 3 : -1;
            if (v < 0) { run = 0; continue; }
            code = ((code << 2) | (u32)v) & mask;
            run = min(run + 1, k);
            if (run == k) atomicAdd(table + code, 1u);
        }
    }
}

static __device__ __forceinline__ void fnv_mix(u32 &h, u32 v) {
#pragma unroll
    for (int b = 0; b < 4; ++b) {
        h ^= (v >> (8 * b)) & 0xffu;
        h *= 16777619u;
    }
}

// Pair i uses adapter entry i (tables built from its query) and target [t_off[i], t_off[i+1]).
template <int NW>
__global__ void __launch_bounds__(RES_THREADS)
k_align_pairs(const uint8_t *__restrict__ targets, const u32 *__restrict__ t_off,
              const int *__restrict__ kk, AdapterCtx C, u32 n, int nw_filter,
              tgsf_align_result *__restrict__ out, u64 *scratch, u64 scratch_stride) {
    const u64 tid = (u64)blockIdx.x * RES_THREADS + threadIdx.x;
    for (u64 i = tid; i < n; i += (u64)gridDim.x * RES_THREADS) {
        const DevAdapter A = C.ad[i];
        if (A.nw != nw_filter) continue;
        const AdapterTables T = adapter_tables(C, (int)i);
        const int q = A.qlen;
        const u64 lo = t_off[i], hi = t_off[i + 1];
        tgsf_align_result R;
        R.edit_distance = -1;
        R.n_locations = 0;
        R.align_len = 0;
        R.first_start = R.first_end = R.last_start = R.last_end = 0;
        R.loc_hash = 2166136261u;
        int k = kk[i];
        if (k < 0) k = q;   // E.cpp:194-212
        k = min(k, q);      // E.cpp:565-567
        int d = hw_best<NW>(T, targets, lo, hi, min(k, q - 1));
        bool minus_one = false;
        if (d == 0x7fffffff && k >= q) { // every column scores <= q; column -1 only via W > 0
            d = q;
            minus_one = (q % 64) != 0;
        }
        if (d != 0x7fffffff) {
            R.edit_distance = d;
            int nloc = 0;
            auto add = [&](int st, int en) {
                if (nloc == 0) { R.first_start = st; R.first_end = en; }
                R.last_start = st;
                R.last_end = en;
                fnv_mix(R.loc_hash, (u32)st);
                fnv_mix(R.loc_hash, (u32)en);
                ++nloc;
            };
            if (minus_one) {
                add(0, -1);
                R.align_len = q; // E.cpp:1171-1178
            }
            Myers<NW> s;
            myers_init_hw<NW>(s, q);
            for (u64 p = lo; p < hi; ++p) {
                myers_step<NW, 0, true>(s, T.hw + (u32)__ldg(targets + p) * NW, 0);
                if (s.score != d) continue;
                const u64 s0 = shw_start<NW>(T, targets, lo, p, d);
                if (nloc == 0)
                    R.align_len = nw_alignment_len<NW>(T, targets, s0, p, d, scratch + tid, scratch_stride);
                add((int)(s0 - lo), (int)(p - lo));
            }
            R.n_locations = nloc;
        }
        out[i] = R;
    }
}
