// Shared device-side types of libtgsf_cuda (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/tgsf.h"
#include "../../include/tgsf_layout.h"

typedef unsigned long long u64;
typedef long long i64;
typedef unsigned int u32;

#define TGSF_SM_COUNT_FALLBACK 148

// ---- tunables -------------------------------------------------------------------------------
// K1: one warp owns one tile of 32 bins x 100 bases; lane l owns bin l (T.cpp:1460 index = i/100).
#define SCAN_BIN 100
#define SCAN_TILE_BINS 32
#define SCAN_TILE (SCAN_BIN * SCAN_TILE_BINS) /* 3200 bases */
// K3: the middle window is cut into 16-byte-aligned absolute chunks of 2^chunk_shift columns
// (1024..4096, chosen per batch), the unit of the per-chunk minima.  k_mid_scan works through runs of consecutive
// chunks, absolute blocks of 2^MID_RUN_BLOCK_SHIFT columns, and re-starts a halo of q+k-1 columns before each run
// (exact for scores <= k, see DESIGN.md).
#define MID_CHUNK_SHIFT_MIN 10
#define MID_CHUNK_SHIFT_MAX 12
#define MID_RUN_BLOCK_SHIFT 12

// Per-adapter constants precomputed on the host (tgsf_create), replacing the float expressions of
// GetEditDistance (T.cpp:1233, 1250, 1267, 1271, 1287).
struct DevAdapter {
    int qlen;
    int nw;        // 64-bit Myers words = ceil(qlen/64)
    int k_mid;     // min(qlen - MidMatchLen + 1, qlen - 1); <= 0: middle search can never hit
    int k_end;     // min(qlen - EndMatchLen + 1, qlen - 1)
    int thr_mid;   // smallest mlen with mlen >= MidMatchLen && float(mlen)/qlen >= MidSim
    int thr_end;
    int end_extra; // int(qlen / EndSim)
    int halo_mid;  // round_up(qlen + k_mid - 1, 16)
    u32 peq_off;   // offset (in u64) of this adapter's three tables in the Peq pool
};
// Peq pool layout per adapter (nw words per byte value, 256 byte values each):
//   [0]            hw : top-padded (W = 64*nw - qlen wildcard rows below bit W), HW scans
//   [256*nw]       fw : forward query, unpadded, NW pass of the traceback
//   [512*nw]       rv : reversed query, unpadded, SHW start search
//   [768*nw]       rvhw : reversed query, top-padded, right-to-left HW scan (3' window starts)

struct DevParams {
    int min_len, max_len;
    double min_q, max_q; // float thresholds promoted exactly like `rawQuality < P2In->MinQ`
    int bc_len, head_trim, tail_trim, end_len, extra_len;
    int kmer, min_repeat, qtype;
    u32 flags;
    int n_adapters;
    int has_qual;
    tgsf_counter_layout L;
};

// One batch resident in HBM.
struct DevBatch {
    const uint8_t *bases;
    const uint8_t *quals; // may be null
    const u64 *offsets;   // n_reads + 1
    u32 n_reads;
};

struct __align__(16) TileEntry {
    u64 start; // absolute byte offset of the tile's first base in the batch streams
    u32 seg;   // read index (raw pass) or piece index (clean pass)
    u32 tile;  // tile index inside the segment (high 20 bits) | valid bases in the tile (low 12)
};
#define TILE_N_BITS 12

struct __align__(8) ChunkEntry {
    u32 read;
    u32 chunk; // absolute chunk index: covers bytes [chunk << chunk_shift, (chunk+1) << chunk_shift)
};

struct __align__(8) Region {
    int s, e;
};

struct __align__(16) TmpPiece {
    int read, idx, start, len;
};

#define DEV_STATUS_OK 0u
#define DEV_STATUS_POOL_OVERFLOW 1u
#define DEV_STATUS_BIN_OVERFLOW 2u

static __device__ __forceinline__ void atomic_add_u64(u64 *p, u64 v) { atomicAdd(p, v); }

static __device__ __forceinline__ u32 warp_sum_u32(u32 v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
static __device__ __forceinline__ i64 warp_sum_i64(i64 v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
