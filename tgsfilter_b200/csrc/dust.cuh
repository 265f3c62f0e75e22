// Low-complexity screen (tgsf_set_dust): the original windowed DUST score over the pieces still emitted after the
// repeat check and the contaminant screen.  A piece whose masked bases reach the threshold gets TGSF_PIECE_LOWCOMPLEX.
//
// Rules (include/tgsf.h, DESIGN §4), on piece-relative positions of s[0, L): codes A0 C1 G2 T3, case-insensitive;
// triplet i = s[i, i+3), code 16a + 4b + c.  Window j = s[j, j+64) (0 <= j <= L - 64) is valid iff all 64 bytes are
// ACGT/acgt; c_t counts its 62 triplets by code and S_j = sum_t c_t (c_t - 1) / 2.  Window j is masked iff it is valid
// and S_j > 61 level.  M = |union of [j, j+64) over the masked windows|: each masked start adds min(64, j - previous
// masked start), the first one 64.  The piece is dropped iff L >= 64 and M 10^6 >= ppm L (u64).
//
// Layout: the pieces' windows are cut into chunks of DUST_CHUNK windows by the contaminant screen's k_contam_count /
// k_contam_fill (window length 64).  One warp takes a chunk; each lane a contiguous run of windows.  A lane keeps its 64
// u8 triplet counts in shared memory, word (t >> 2) * 32 + lane, byte t & 3, so every lane stays in its own bank, and
// updates S as it rolls: adding triplet t adds c_t and then increments it, removing one decrements c_t and subtracts it.
// The outgoing triplet is recomputed from the bytes 62 positions back.  Only valid triplets are counted, so in a valid
// window the counts are exactly its triplets and an N needs no reset.  A chunk that is not its piece's first also
// scores the 63 windows before it, spread over its lanes: the masked start before its first masked window is then known
// within the chunk, which makes each chunk self-contained.  The last masked start of the lanes below comes from a warp
// max-scan; one atomic per chunk adds the chunk's share of M into the piece's u32 slot, and k_dust_decide applies the
// threshold.
//
// Chunk length: a lane first rolls 63 bytes through its counters before it scores its first window.  With the
// contaminant screen's 2 048-window chunks (64 windows a lane) that warm-up would double the work; with 16 384 windows
// (512 a lane, 514 with the halo) it adds 12 %.  Longer chunks would not help the common case: a piece of up to
// 16 447 bases is a single chunk already.
#pragma once
#include "common.cuh"
#include "contam.cuh"

#define DUST_WINDOW 64
#define DUST_TRIPLETS 62 // triplets per window (l - 1 = 61 in DUST's S / (l - 1))
#define DUST_LEVEL_MIN 1
#define DUST_LEVEL_MAX 30
#define DUST_CHUNK 16384u
#define DUST_THREADS 256
#define DUST_NONE (-128) // "no masked start yet": any start j >= -63 then adds min(64, j - DUST_NONE) = 64

// Rolling triplet code over a byte stream; valid() once the last 3 bytes were ACGT/acgt.
struct DustRoll {
    u32 code = 0;
    int run = 0;
    __device__ __forceinline__ void push(u32 byte) {
        const int c = contam_code(byte);
        run = c < 0 ? 0 : run + 1;
        code = ((code << 2) | (u32)(c & 3)) & 63u;
    }
    __device__ __forceinline__ bool valid() const { return run >= 3; }
};

// One warp per chunk (grid-stride over the device-side chunk total).  thr = 61 level.  masked[piece] += the chunk's
// share of M.
__global__ void __launch_bounds__(DUST_THREADS)
k_dust_screen(const uint8_t *__restrict__ bases, const ContamChunk *__restrict__ chunks,
              const u32 *__restrict__ n_chunks_ptr, u32 thr, u32 *__restrict__ masked,
              const u32 *__restrict__ dev_status) {
    __shared__ u32 s_cnt[DUST_THREADS / 32][16][32];
    if (*dev_status != DEV_STATUS_OK) return;
    const u32 n_chunks = *n_chunks_ptr;
    const int lane = threadIdx.x & 31;
    const u32 warps = gridDim.x * (DUST_THREADS / 32);
    uint8_t *cnt = (uint8_t *)&s_cnt[threadIdx.x >> 5][0][lane];
    for (u32 c = blockIdx.x * (DUST_THREADS / 32) + (threadIdx.x >> 5); c < n_chunks; c += warps) {
        const ContamChunk ch = chunks[c];
        // chunks of a piece are consecutive and DUST_CHUNK > 63 windows apart: only a piece's first chunk has no halo
        const int halo = (c > 0 && chunks[c - 1].piece == ch.piece) ? DUST_WINDOW - 1 : 0;
        const int n_ext = (int)ch.n_win + halo; // windows [-halo, n_win) relative to the chunk's first window
        const int span = (n_ext + 31) / 32;
        const int x0 = min(n_ext, lane * span) - halo, x1 = min(n_ext, (lane + 1) * span) - halo;
        int first = DUST_NONE, last = DUST_NONE, prev = DUST_NONE;
        u32 add = 0; // M share of this lane's masked windows after its first one
        if (x0 < x1) {
            for (int t = 0; t < 16; ++t) s_cnt[threadIdx.x >> 5][t][lane] = 0;
            const uint8_t *p = bases + ((i64)ch.start + x0);
            const int n_bytes = (x1 - x0) + DUST_WINDOW - 1;
            DustRoll in, out;
            u32 S = 0;
            for (int q = 0; q < n_bytes; ++q) {
                in.push(__ldg(p + q));
                if (q >= DUST_TRIPLETS) out.push(__ldg(p + q - DUST_TRIPLETS));
                if (in.valid()) { // add triplet q - 2
                    uint8_t *ct = cnt + ((in.code >> 2) << 7) + (in.code & 3);
                    const u32 v = *ct;
                    S += v;
                    *ct = (uint8_t)(v + 1);
                }
                if (q >= DUST_WINDOW && out.valid()) { // remove triplet q - 64
                    uint8_t *ct = cnt + ((out.code >> 2) << 7) + (out.code & 3);
                    const u32 v = *ct - 1u;
                    *ct = (uint8_t)v;
                    S -= v;
                }
                if (q >= DUST_WINDOW - 1 && in.run >= DUST_WINDOW && S > thr) { // window x0 + q - 63
                    const int j = x0 + q - (DUST_WINDOW - 1);
                    if (first == DUST_NONE) first = j;
                    else if (j >= 0) add += (u32)min(DUST_WINDOW, j - prev);
                    prev = j;
                }
            }
            last = prev;
        }
        // masked start before this lane's first one: the last one of the lanes below
        int below = last;
        for (int o = 1; o < 32; o <<= 1) {
            const int v = __shfl_up_sync(0xffffffffu, below, o);
            if (lane >= o) below = max(below, v);
        }
        below = __shfl_up_sync(0xffffffffu, below, 1);
        if (lane == 0) below = DUST_NONE;
        if (first >= 0) add += (u32)min(DUST_WINDOW, first - below);
        add = warp_sum_u32(add);
        if (lane == 0 && add) atomicAdd(masked + ch.piece, add);
    }
}

// Threshold: low complexity iff L >= 64 and M 10^6 >= ppm L (u64).
__global__ void k_dust_decide(tgsf_piece *pieces, const u32 *__restrict__ n_pieces_ptr, u32 cap,
                              const u32 *__restrict__ masked, u64 ppm, const u32 *__restrict__ dev_status) {
    const u32 i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= cap || *dev_status != DEV_STATUS_OK || i >= *n_pieces_ptr) return;
    const tgsf_piece p = pieces[i];
    if (p.status != TGSF_PIECE_EMIT || p.len < DUST_WINDOW) return;
    if ((u64)masked[i] * 1000000ull >= ppm * (u64)p.len) pieces[i].status = TGSF_PIECE_LOWCOMPLEX;
}
