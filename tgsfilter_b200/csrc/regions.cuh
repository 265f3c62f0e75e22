// K5: trim-region merge, middle-adapter split, length filter, DropInfo counters and the compaction
// of the kept pieces.  Replaces adapterMap (T.cpp:1324-1434) and the control flow of
// filter_sequence around it (T.cpp:1946-1965, 1976-2000).
#pragma once
#include "common.cuh"
#include "scan.cuh"

#define REG_THREADS 128

// Per read: mean quality, histogram, the -q/-Q band (T.cpp:1942-1952).  One thread per read.
// Writes res[r] (status, sum_q; counts zeroed) and read_active[r] (goes on to adapterMap).
template <bool HAS_QUAL>
__global__ void __launch_bounds__(REG_THREADS)
k_finalize_raw(DevBatch B, DevParams P, const u64 *__restrict__ seg_sum, tgsf_read_result *res,
               int *__restrict__ read_active, u32 *__restrict__ piece_cnt,
               u64 *__restrict__ counters) {
    const u32 r = blockIdx.x * REG_THREADS + threadIdx.x;
    u64 lowq_reads = 0, lowq_bases = 0;
    if (r < B.n_reads) {
        const u64 len = B.offsets[r + 1] - B.offsets[r];
        tgsf_read_result R;
        R.sum_q = 0;
        R.status = TGSF_READ_EVALUATED;
        R.n_mid = R.n_5p = R.n_3p = 0;
        R.piece_begin = 0;
        R.n_pieces = 0;
        int active = 1;
        if (len == 0) {
            R.status = TGSF_READ_EMPTY;
            active = 0;
        } else if (HAS_QUAL) {
            const u64 sum = seg_sum[r];
            R.sum_q = sum;
            const double q = __ull2double_rn(sum) / __ull2double_rn(len); // T.cpp:1478
            atomic_add_u64(counters + P.L.raw_hist + qual_hist_index(q), len);
            if ((P.flags & TGSF_FLAG_FILTER) && (q < P.min_q || q > P.max_q)) {
                R.status = TGSF_READ_LOWQ;
                active = 0;
                lowq_reads = 1;
                lowq_bases = len;
            }
        }
        res[r] = R;
        read_active[r] = active;
        piece_cnt[r] = 0;
    }
    lowq_reads = (u64)warp_sum_i64((i64)lowq_reads);
    lowq_bases = (u64)warp_sum_i64((i64)lowq_bases);
    if ((threadIdx.x & 31) == 0 && lowq_reads) {
        atomic_add_u64(counters + P.L.drop_info + 0, lowq_reads);
        atomic_add_u64(counters + P.L.drop_info + 1, lowq_bases);
    }
}

// Small in-place insertion sort by (s, e) — region lists are short (<= 4 + middle hits).
static __device__ void sort_regions(Region *v, int n) {
    for (int i = 1; i < n; ++i) {
        const Region x = v[i];
        int j = i - 1;
        while (j >= 0 && (v[j].s > x.s || (v[j].s == x.s && v[j].e > x.e))) {
            v[j + 1] = v[j];
            --j;
        }
        v[j + 1] = x;
    }
}

// adapterMap for one read per thread.  Emits TmpPiece records through an atomic cursor (order is
// restored by k_place_pieces) and per-read counts into res[r].
__global__ void __launch_bounds__(REG_THREADS)
k_regions(DevBatch B, DevParams P, const int *__restrict__ read_active,
          const int *__restrict__ end_n, const int *__restrict__ end_pos,
          const u32 *__restrict__ mid_n, const u32 *__restrict__ mid_off,
          const Region *__restrict__ pool, Region *__restrict__ sortbuf, u32 sortbuf_cap,
          u32 *__restrict__ sort_cursor, tgsf_read_result *res, u32 *__restrict__ piece_cnt,
          TmpPiece *__restrict__ tmp, u32 tmp_cap, u32 *__restrict__ tmp_cursor,
          u64 *__restrict__ counters,
          u32 *__restrict__ dev_status) {
    if (*dev_status != DEV_STATUS_OK) return;
    const u32 r = blockIdx.x * REG_THREADS + threadIdx.x;
    if (r >= B.n_reads || !read_active[r]) return;
    u64 *DropInfo = counters + P.L.drop_info;
    const int rawLen = (int)(B.offsets[r + 1] - B.offsets[r]);
    const int A = P.n_adapters;
    int n_pieces = 0;

    auto keep = [&](int start, int len) { // length filter, T.cpp:1406-1411
        if (len >= P.min_len && len <= P.max_len) {
            const u32 slot = atomicAdd(tmp_cursor, 1u);
            if (slot < tmp_cap) {
                TmpPiece t;
                t.read = (int)r;
                t.idx = n_pieces;
                t.start = start;
                t.len = len;
                tmp[slot] = t;
            } else {
                *dev_status = DEV_STATUS_POOL_OVERFLOW;
            }
            ++n_pieces;
        } else {
            atomic_add_u64(DropInfo + 11, 1ull);
            atomic_add_u64(DropInfo + 12, (u64)len);
        }
    };

    if (!(P.flags & TGSF_FLAG_FILTER)) { // T.cpp:1963-1965
        const u32 slot = atomicAdd(tmp_cursor, 1u);
        if (slot < tmp_cap) {
            TmpPiece t;
            t.read = (int)r; t.idx = 0; t.start = 0; t.len = rawLen;
            tmp[slot] = t;
        } else {
            *dev_status = DEV_STATUS_POOL_OVERFLOW;
        }
        res[r].n_pieces = 1;
        piece_cnt[r] = 1;
        return;
    }

    int num5p = 0, num3p = 0, numMid = 0;
    int te5 = 0, ts3 = 0x7fffffff;
    for (int a = 0; a < A; ++a) {
        const u64 k2 = ((u64)r * A + a) * 2;
        if (end_n[k2] > 0) { num5p += end_n[k2]; te5 = max(te5, end_pos[k2]); }
        if (end_n[k2 + 1] > 0) { num3p += end_n[k2 + 1]; ts3 = min(ts3, end_pos[k2 + 1]); }
        numMid += (int)mid_n[(u64)r * A + a];
    }
    res[r].n_mid = numMid;
    res[r].n_5p = num5p;
    res[r].n_3p = num3p;
    {
        const int m = numMid > 0, f = num5p > 0, t = num3p > 0; // T.cpp:1354-1370
        const int cls = m ? (f ? (t ? 2 : 3) : (t ? 4 : 6)) : (f ? (t ? 5 : 7) : (t ? 8 : 9));
        atomic_add_u64(DropInfo + cls, 1ull);
    }
    if (numMid > 0 && (P.flags & TGSF_FLAG_DISCARD_MID)) { // T.cpp:1372-1373
        atomic_add_u64(DropInfo + 10, (u64)rawLen);
        res[r].n_pieces = 0;
        return;
    }

    // region list: fixed trims (T.cpp:1334-1348), one collapsed region per read end (all 5'
    // regions start at 0, all 3' regions end at rawLen, so their union is what the merge would
    // produce), every middle region.
    Region local[4];
    Region *v = local;
    int n = 0;
    if (numMid > 0) {
        const u32 need = (u32)numMid + 4u;
        const u32 off = atomicAdd(sort_cursor, need);
        if (off + need > sortbuf_cap) {
            *dev_status = DEV_STATUS_POOL_OVERFLOW;
            return;
        }
        v = sortbuf + off;
        for (int a = 0; a < A; ++a) {
            const u64 key = (u64)r * A + a;
            const u32 c = mid_n[key];
            for (u32 i = 0; i < c; ++i) v[n++] = pool[mid_off[key] + i];
        }
    }
    if (P.head_trim > 0) { v[n].s = 0; v[n].e = P.head_trim >= rawLen ? rawLen : P.head_trim; ++n; }
    if (P.tail_trim > 0) {
        if (P.tail_trim >= rawLen) { v[n].s = 0; v[n].e = rawLen; }
        else { v[n].s = rawLen - P.tail_trim; v[n].e = rawLen; }
        ++n;
    }
    if (num5p > 0) { v[n].s = 0; v[n].e = te5; ++n; }
    if (num3p > 0) { v[n].s = ts3; v[n].e = rawLen; ++n; }
    sort_regions(v, n);

    // merge (T.cpp:1383-1390) fused with the keep/drop walk (T.cpp:1393-1432)
    u64 trimmed = 0;
    if (n >= 1) {
        int currentStart = 0;
        int ms = v[0].s, me = v[0].e;
        for (int i = 1; i <= n; ++i) {
            if (i < n && me >= v[i].s) {
                me = max(me, v[i].e);
                continue;
            }
            const int dropLen = me - ms;
            trimmed += (u64)(i64)dropLen;
            if (dropLen == rawLen) atomic_add_u64(DropInfo + 11, 1ull);
            if (ms > currentStart) keep(currentStart, ms - currentStart);
            currentStart = me;
            if (i < n) { ms = v[i].s; me = v[i].e; }
        }
        if (currentStart < rawLen) keep(currentStart, rawLen - currentStart);
    } else {
        keep(0, rawLen);
    }
    if (trimmed) atomic_add_u64(DropInfo + 10, trimmed);
    res[r].n_pieces = n_pieces;
    piece_cnt[r] = (u32)n_pieces;
}

// n_pieces -> piece_begin was produced by an exclusive scan; scatter the tmp records to their
// final (read, start) order and initialise the piece records.
__global__ void k_place_pieces(const TmpPiece *__restrict__ tmp, const u32 *__restrict__ tmp_cursor,
                               const u32 *__restrict__ piece_begin, tgsf_read_result *res,
                               tgsf_piece *pieces, u32 n_reads, int only_qc,
                               const u32 *__restrict__ dev_status) {
    if (*dev_status != DEV_STATUS_OK) return;
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n_reads) res[i].piece_begin = (int)piece_begin[i];
    if (i >= *tmp_cursor) return;
    const TmpPiece t = tmp[i];
    tgsf_piece p;
    p.sum_q = 0;
    p.read = t.read;
    p.start = t.start;
    p.len = t.len;
    p.repeat_len = -1;
    p.status = only_qc ? TGSF_PIECE_QC_ONLY : TGSF_PIECE_EMIT;
    p.contam_hits = 0;
    pieces[piece_begin[t.read] + (u32)t.idx] = p;
}

// Segment arrays of the clean pass: piece i -> absolute start + length (0 if not scanned).
// Launched over the piece capacity; the live count is device-side.
__global__ void k_piece_segments_dyn(DevBatch B, const tgsf_piece *__restrict__ pieces,
                                     const u32 *__restrict__ n_pieces_ptr, u32 cap,
                                     u64 *__restrict__ seg_start, int *__restrict__ seg_len,
                                     u64 *__restrict__ seg_sum, u32 *__restrict__ n_tiles,
                                     const u32 *__restrict__ dev_status) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= cap) return;
    int len = 0;
    u64 start = 0;
    if (*dev_status == DEV_STATUS_OK && i < *n_pieces_ptr) {
        const tgsf_piece p = pieces[i];
        len = p.status == TGSF_PIECE_EMIT ? p.len : 0;
        start = B.offsets[p.read] + (u64)p.start;
    }
    seg_start[i] = start;
    seg_len[i] = len;
    seg_sum[i] = 0;
    n_tiles[i] = (u32)((len + SCAN_TILE - 1) / SCAN_TILE);
}

// Clean-side decisions (T.cpp:1994-2002): quality band after the clean bins were updated,
// DropInfo[13]/[14], clean histogram; seg_flag = piece still emitted (drives the clean 5'/3' pass).
template <bool HAS_QUAL>
__global__ void __launch_bounds__(REG_THREADS)
k_finalize_clean_dyn(DevParams P, tgsf_piece *pieces, const u32 *__restrict__ n_pieces_ptr, u32 cap,
                     const u64 *__restrict__ seg_sum, int *__restrict__ seg_flag,
                     u64 *__restrict__ counters, const u32 *__restrict__ dev_status) {
    const u32 i = blockIdx.x * REG_THREADS + threadIdx.x;
    if (i >= cap) return;
    if (*dev_status != DEV_STATUS_OK || i >= *n_pieces_ptr) {
        seg_flag[i] = 0;
        return;
    }
    tgsf_piece p = pieces[i];
    int flag = 0;
    if (p.status == TGSF_PIECE_EMIT) {
        flag = 1;
        if (HAS_QUAL) {
            const u64 sum = seg_sum[i];
            p.sum_q = sum;
            const double q = __ull2double_rn(sum) / __ull2double_rn((u64)p.len);
            if ((P.flags & TGSF_FLAG_FILTER) && (q < P.min_q || q > P.max_q)) {
                p.status = TGSF_PIECE_LOWQ;
                flag = 0;
                atomic_add_u64(counters + P.L.drop_info + 13, 1ull);
                atomic_add_u64(counters + P.L.drop_info + 14, (u64)p.len);
            } else {
                atomic_add_u64(counters + P.L.clean_hist + qual_hist_index(q), (u64)p.len);
            }
            pieces[i] = p;
        }
    }
    seg_flag[i] = flag;
}
