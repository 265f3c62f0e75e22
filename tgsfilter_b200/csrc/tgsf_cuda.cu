// libtgsf_cuda: C-ABI (include/tgsf.h) over the sm_100a kernels.  Host side = context, slot ring,
// buffer management and the launch sequence that replaces one batch worth of
// TGSFilterTask::filter_sequence iterations (T.cpp:1939-2061).
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <new>
#include <string>
#include <type_traits>
#include <utility>
#include <vector>

#include "adapters.cuh"
#include "common.cuh"
#include "contam.cuh"
#include "contam_attr.cuh"
#include "dust.cuh"
#include "foldback.cuh"
#include "kmer.cuh"
#include "kmer16.cuh"
#include "gzenc.cuh"
#include "prepass.cuh"
#include "regions.cuh"
#include "scan.cuh"
#include "util.cuh"

namespace {

thread_local char g_err[512] = "";

void set_err(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

#define CU(call)                                                                          \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess) {                                                          \
            set_err("%s:%d %s: %s", __FILE__, __LINE__, #call, cudaGetErrorString(e_));   \
            return TGSF_ERR_CUDA;                                                         \
        }                                                                                 \
    } while (0)

#define TRY(call)              \
    do {                       \
        int rc_ = (call);      \
        if (rc_ != TGSF_OK) return rc_; \
    } while (0)

// A growable buffer that owns its memory: device memory (DBuf) or pinned host memory (HBuf).  Move-only; the
// destructor frees.  Destructors of owned CUDA resources (this, Stream, Event) never call cudaSetDevice: the entry
// point that owns a resource has made its device current, and tgsf_destroy makes the context's device current
// before it deletes the context.
template <bool Pinned>
struct Buf {
    void *p = nullptr;
    size_t cap = 0;
    Buf() = default;
    Buf(Buf &&o) noexcept : p(std::exchange(o.p, nullptr)), cap(std::exchange(o.cap, 0)) {}
    Buf &operator=(Buf &&o) noexcept {
        if (this != &o) {
            reset();
            p = std::exchange(o.p, nullptr);
            cap = std::exchange(o.cap, 0);
        }
        return *this;
    }
    ~Buf() { reset(); }
    int ensure(size_t bytes) {
        if (bytes <= cap) return TGSF_OK;
        reset();
        size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = Pinned ? cudaHostAlloc(&p, want, cudaHostAllocDefault) : cudaMalloc(&p, want);
        if (e != cudaSuccess) {
            set_err("%s(%zu): %s", Pinned ? "cudaHostAlloc" : "cudaMalloc", want, cudaGetErrorString(e));
            return TGSF_ERR_NOMEM;
        }
        cap = want;
        return TGSF_OK;
    }
    void reset() {
        if (p) Pinned ? cudaFreeHost(p) : cudaFree(p);
        p = nullptr;
        cap = 0;
    }
    template <typename T> T *as() const { return (T *)p; }
};
using DBuf = Buf<false>;
using HBuf = Buf<true>;

struct StreamDestroy { void operator()(cudaStream_t s) const { cudaStreamDestroy(s); } };
struct EventDestroy { void operator()(cudaEvent_t e) const { cudaEventDestroy(e); } };
using Stream = std::unique_ptr<std::remove_pointer_t<cudaStream_t>, StreamDestroy>;
using Event = std::unique_ptr<std::remove_pointer_t<cudaEvent_t>, EventDestroy>;

int create(Stream &s) {
    cudaStream_t h;
    CU(cudaStreamCreateWithFlags(&h, cudaStreamNonBlocking));
    s.reset(h);
    return TGSF_OK;
}

int create(Event &e, unsigned flags = cudaEventDefault) {
    cudaEvent_t h;
    CU(cudaEventCreateWithFlags(&h, flags));
    e.reset(h);
    return TGSF_OK;
}

inline int round_nw(int nw);

// Adapter tables on the device (shared by the context, the pre-pass and tgsf_align_hw).
struct AdapterSet {
    std::vector<DevAdapter> host;
    DBuf d_ad, d_peq;
    int max_q = 0, min_q = 0x7fffffff, max_nw = 1;
    int max_cols = 0; // traceback scratch columns: max(q + k)

    // k_mid/k_end/thr_* are filled by the caller in `host` before upload().
    int build(const uint8_t *const *seq, const int32_t *len, int n) {
        host.resize((size_t)n);
        size_t words = 0;
        for (int a = 0; a < n; ++a) {
            DevAdapter &A = host[(size_t)a];
            memset(&A, 0, sizeof(A));
            A.qlen = len[a];
            A.nw = round_nw((len[a] + 63) / 64);
            A.peq_off = (u32)words;
            words += (size_t)4 * 256 * (size_t)std::max(A.nw, 1);
            if (A.qlen > 0) {
                max_q = std::max(max_q, A.qlen);
                min_q = std::min(min_q, A.qlen);
                max_nw = std::max(max_nw, A.nw);
            }
        }
        std::vector<u64> peq(words, 0);
        for (int a = 0; a < n; ++a) {
            const DevAdapter &A = host[(size_t)a];
            const int q = A.qlen, nw = A.nw;
            if (q <= 0) continue;
            const int W = 64 * nw - q;
            u64 *hw = peq.data() + A.peq_off, *fw = hw + 256 * nw, *rv = fw + 256 * nw, *rvhw = rv + 256 * nw;
            for (int b = 0; b < 256; ++b)
                for (int i = 0; i < W; ++i) { // wildcards
                    hw[b * nw + (i >> 6)] |= 1ull << (i & 63);
                    rvhw[b * nw + (i >> 6)] |= 1ull << (i & 63);
                }
            for (int i = 0; i < q; ++i) {
                const int b = seq[a][i];
                hw[b * nw + ((W + i) >> 6)] |= 1ull << ((W + i) & 63);
                fw[b * nw + (i >> 6)] |= 1ull << (i & 63);
                const int br = seq[a][q - 1 - i];
                rv[br * nw + (i >> 6)] |= 1ull << (i & 63);
                rvhw[br * nw + ((W + i) >> 6)] |= 1ull << ((W + i) & 63);
            }
        }
        TRY(d_peq.ensure(std::max<size_t>(words, 1) * sizeof(u64)));
        if (words) {
            cudaError_t e = cudaMemcpy(d_peq.p, peq.data(), words * sizeof(u64), cudaMemcpyHostToDevice);
            if (e != cudaSuccess) { set_err("peq upload: %s", cudaGetErrorString(e)); return TGSF_ERR_CUDA; }
        }
        return TGSF_OK;
    }
    int upload() {
        max_cols = 16;
        for (auto &A : host) max_cols = std::max(max_cols, 2 * A.qlen + 2);
        TRY(d_ad.ensure(std::max<size_t>(host.size(), 1) * sizeof(DevAdapter)));
        if (!host.empty()) {
            cudaError_t e = cudaMemcpy(d_ad.p, host.data(), host.size() * sizeof(DevAdapter), cudaMemcpyHostToDevice);
            if (e != cudaSuccess) { set_err("adapter upload: %s", cudaGetErrorString(e)); return TGSF_ERR_CUDA; }
        }
        return TGSF_OK;
    }
    AdapterCtx ctx() const {
        AdapterCtx c;
        c.ad = d_ad.as<DevAdapter>();
        c.peq_pool = d_peq.as<u64>();
        return c;
    }
};

// Per-thread traceback scratch (nw_traceback_len: one (2*nw+1)-word record per target column and thread).  The
// resolve kernels run grid-stride loops, so the grid of a launch is chosen per adapter such that its column store
// stays within a budget: the default 4 CTAs per SM for ordinary adapters, fewer for very long ones.
#define TGSF_SCRATCH_BUDGET (2ull << 30)
struct Scratch {
    DBuf buf;
    static size_t per_thread(int cols, int nw) { return (size_t)cols * (size_t)(2 * nw + 1) * sizeof(u64); }
    static int grid_for(int default_grid, int threads_per_cta, int cols, int nw) {
        const u64 fit = TGSF_SCRATCH_BUDGET / ((u64)per_thread(cols, nw) * (u64)threads_per_cta);
        return (int)std::max<u64>(1, std::min<u64>((u64)default_grid, fit));
    }
    // size for the largest launch over `ads` with `default_grid` CTAs of `threads_per_cta` threads
    template <typename ADS>
    int ensure(const ADS &ads, int default_grid, int threads_per_cta) {
        size_t need = 0;
        for (const auto &A : ads) {
            if (A.qlen <= 0 || A.nw <= 0) continue;
            const int cols = 2 * A.qlen + 2;
            need = std::max(need, (size_t)grid_for(default_grid, threads_per_cta, cols, A.nw) * threads_per_cta * per_thread(cols, A.nw));
        }
        return buf.ensure(std::max<size_t>(need, 256));
    }
};

// what a batch that ended with DEV_STATUS_HASH_OVERFLOW reports
#define HASH_OVERFLOW_MSG "a piece crowds more distinct keys into one hash pass than the repeat check or the fold-back screen can split"

struct DevHeader { // small block mirrored to the host with every batch
    u32 status;
    u32 tmp_cursor;  // total pieces
    u32 sort_cursor;
    u32 gz_overflow; // k_gz_encode ran out of blob space
    unsigned long long gz_cursor; // bytes of deflate blocks produced
    u32 kmer_work;   // k_kmer_tag16: next piece to take
    u32 kmer_long;   // pieces it left for k_kmer_smem (too long for 16-bit positions)
    u32 fold_work, fold_long, fold_long_work; // fold-back screen: next piece, long-list size, next long piece
    u32 contam_list_n, contam_work;           // contaminant attribution: listed pieces, next listed piece
};

struct Slot {
    Stream stream;
    Stream stream2; // side stream: the end-window search runs next to the middle scan
    Event ev_fork, ev_join;
    Event ev_start, ev_k0, ev_k1, ev_end;
    Event ev_stage[TGSF_N_STAGES + 1];
    bool busy = false;
    // input
    DBuf in_bases, in_quals, in_offsets, in_packed, in_exc_pos, in_exc_val;
    DevBatch B{};
    u64 n_bases = 0;
    bool has_qual = false;
    // work arrays
    DBuf seg_start, seg_len, seg_sum, seg_flag, tile_cnt, tile_off, tiles;
    DBuf read_active, piece_cnt, piece_begin, chunk_cnt, chunk_off, chunks, chunk_min, chunk_hits, chunk_first;
    DBuf run_cnt, run_off, runs, run_perm, run_hist; // middle-scan work items: runs of consecutive chunks
    int chunk_shift = MID_CHUNK_SHIFT_MIN, run_shift = 0;
    DBuf best_mid, mid_n, mid_off, end_n, end_pos, pool, sortbuf, tmp, pieces, res, header;
    DBuf scan_tmp, kmer_long_list, mid_work, gz_blob, gz_spans;
    DBuf contam_cnt, contam_off, contam_chunks; // chunk lists of the contaminant and the DUST screen (only while on)
    DBuf contam_list;                            // contaminant attribution: pieces to attribute (labelled sets only)
    DBuf dust_masked;                            // DUST screen: masked bases per piece (only while on)
    DBuf fold_long_list, fold_ws;                // fold-back screen (only while enabled)
    Scratch scratch, scratch2; // traceback stores: main stream (k_mid_count) / side stream (k_ends)
    u32 pool_cap = 0, pieces_cap = 0, chunks_cap = 0, runs_cap = 0, tiles_cap = 0;
    // host results
    HBuf h_res, h_pieces, h_header;
    u32 h_pieces_copied = 0;
    float kernel_ms = 0, total_ms = 0;
};

// Contaminant k-mer set (tgsf_set_contaminants).
struct ContamSet {
    DBuf table, pf_bits; // pf_bits: prefilter bitmap, only for sets of <= CONTAM_PF_MAX_KEYS keys
    DBuf labels, tally;  // labelled sets only: u32 label per table slot; u64 reads[n_records + 1], bases[n_records + 1]
    u64 mask = 0;        // table capacity - 1
    u64 n_keys = 0;
    u64 ppm = 0;
    int k = 0;
    u32 n_records = 0;
    bool installed() const { return table.p != nullptr; }
    bool labelled() const { return labels.p != nullptr; }
};

}  // namespace

struct tgsf_ctx {
    int device = 0;
    int sm_count = TGSF_SM_COUNT_FALLBACK;
    DevParams P{};
    AdapterSet ads;
    ContamSet contam;
    bool foldback = false;
    int dust_level = 0; // DUST screen (tgsf_set_dust): 0 = off
    u64 dust_ppm = 0;
    DBuf fold_stats; // u64[4] (tgsf_foldback_stats), allocated when the screen is first enabled
    DBuf counters;
    std::vector<Slot> slots;
    u32 head = 0, tail = 0, outstanding = 0; // ring: submit at head, collect at tail
    u64 launches = 0;
    int kmer16_ctas_per_sm = 2;
    int attr_ctas_per_sm = 1; // k_contam_attr<false> CTAs per SM (occupancy): more probes in flight
    int mid_ctas_per_sm = 0; // TGSF_MID_CTAS=n: cap on resident k_mid_scan CTAs per SM (0 = as many as fit)
    int res_ctas_per_sm = 6; // grid of the resolve kernels (k_ends, k_mid_count, k_mid_emit) in CTAs per SM; TGSF_RES_CTAS
    bool fork_ends = true; // TGSF_FORK_ENDS=0: k_ends on the batch's main stream after the middle scan (A/B)
    u32 kmer16_list_cap = KMER16_LIST_CAP; // TGSF_KMER16_LIST_CAP=n: smaller pending list (tests of the retry path)
    u32 kmer_fill_cap = ~0u; // TGSF_KMER_FILL_CAP=n: at most n new keys per k_kmer pass (tests of the pass split)
    float last_kernel_ms = 0, last_total_ms = 0;
    float last_stage_ms[TGSF_N_STAGES] = {};
    int last_chunk_shift = 0; // middle-scan chunk shift of the last collected batch (tgsf_launch_shape)
    int last_run_shift = 0;   // and its run shift (tgsf_mid_run_shift)
    Event ev_epoch; // recorded at creation: origin of tgsf_last_span
    float last_span_start = 0, last_span_end = 0;
};

namespace {

// A context owned by the entry point that creates it, until it is handed out.
struct CtxDestroy { void operator()(tgsf_ctx *c) const { tgsf_destroy(c); } };
using CtxPtr = std::unique_ptr<tgsf_ctx, CtxDestroy>;

inline u32 cdiv(u64 a, u64 b) { return (u32)((a + b - 1) / b); }

// exclusive scan of in[0..n) -> out[0..n], out[n] = total.  tmp: scratch u32 array.
int exclusive_scan(tgsf_ctx *c, cudaStream_t st, const u32 *in, u32 *out, u32 n, u32 *tmp, size_t tmp_words) {
    if (n == 0) {
        CU(cudaMemsetAsync(out, 0, sizeof(u32), st));
        return TGSF_OK;
    }
    const u32 nb = cdiv(n, SCANB_TILE);
    if ((size_t)nb * 2 + 8 > tmp_words) { set_err("scan scratch too small"); return TGSF_ERR_INVALID; }
    u32 *sums = tmp;               // nb
    u32 *sums_sc = tmp + nb;       // nb + 1
    u32 *rest = tmp + 2 * (size_t)nb + 1;
    k_scan_block<<<nb, UTIL_THREADS, 0, st>>>(in, out, n, sums);
    c->launches++;
    if (nb == 1) { // single block: its total is the grand total
        CU(cudaMemcpyAsync(out + n, sums, sizeof(u32), cudaMemcpyDeviceToDevice, st));
        return TGSF_OK;
    }
    TRY(exclusive_scan(c, st, sums, sums_sc, nb, rest, tmp_words - (2 * (size_t)nb + 1)));
    k_scan_add<<<cdiv(n, UTIL_THREADS), UTIL_THREADS, 0, st>>>(out, n, sums_sc, sums_sc + nb);
    c->launches++;
    return TGSF_OK;
}

int slot_init(Slot &s) {
    TRY(create(s.stream));
    TRY(create(s.stream2));
    TRY(create(s.ev_fork, cudaEventDisableTiming));
    TRY(create(s.ev_join, cudaEventDisableTiming));
    for (Event *e : {&s.ev_start, &s.ev_k0, &s.ev_k1, &s.ev_end}) TRY(create(*e));
    for (auto &e : s.ev_stage) TRY(create(e));
    return TGSF_OK;
}

// Size every work array for a batch of n reads / n_bases bases.
int slot_reserve(tgsf_ctx *c, Slot &s, u32 n, u64 n_bases) {
    const int A = std::max(c->P.n_adapters, 1);
    if (s.pool_cap == 0) s.pool_cap = 65536;
    s.pieces_cap = n + s.pool_cap;
    // longer chunks amortise the halo; keep >= ~16 chunks per resident thread slot for balance
    s.chunk_shift = MID_CHUNK_SHIFT_MIN;
    while (s.chunk_shift < MID_CHUNK_SHIFT_MAX &&
           (n_bases >> (s.chunk_shift + 1)) >= (u64)c->sm_count * 2048ull * 4ull)
        s.chunk_shift++;
    s.chunks_cap = (u32)((n_bases >> s.chunk_shift) + 2ull * n + 16);
    // the middle scan restarts a halo per run of 2^run_shift chunks, not per chunk: runs of 4 096 columns (B200,
    // DESIGN.md §4: with 1 024-column chunks runs of 4 beat 1, 2 and 8; with 4 096-column chunks every longer run
    // was slower than none)
    s.run_shift = MID_RUN_BLOCK_SHIFT - s.chunk_shift;
    s.runs_cap = (u32)((n_bases >> (s.chunk_shift + s.run_shift)) + 2ull * n + 16);
    s.tiles_cap = (u32)(n_bases / SCAN_TILE + (u64)s.pieces_cap + 16);
    const size_t nseg = std::max<size_t>(n, s.pieces_cap) + 1;
    TRY(s.seg_start.ensure(nseg * sizeof(u64)));
    TRY(s.seg_len.ensure(nseg * sizeof(int)));
    TRY(s.seg_sum.ensure(nseg * sizeof(u64)));
    TRY(s.seg_flag.ensure(nseg * sizeof(int)));
    TRY(s.tile_cnt.ensure(nseg * sizeof(u32)));
    TRY(s.tile_off.ensure((nseg + 1) * sizeof(u32)));
    TRY(s.tiles.ensure((size_t)s.tiles_cap * sizeof(TileEntry)));
    TRY(s.read_active.ensure(((size_t)n + 1) * sizeof(int)));
    TRY(s.piece_cnt.ensure(((size_t)n + 1) * sizeof(u32)));
    TRY(s.piece_begin.ensure(((size_t)n + 2) * sizeof(u32)));
    TRY(s.chunk_cnt.ensure(((size_t)n + 1) * sizeof(u32)));
    TRY(s.chunk_off.ensure(((size_t)n + 2) * sizeof(u32)));
    TRY(s.chunks.ensure((size_t)s.chunks_cap * sizeof(ChunkEntry)));
    TRY(s.chunk_min.ensure((size_t)s.chunks_cap * (size_t)A));
    TRY(s.chunk_hits.ensure((size_t)s.chunks_cap * (size_t)A * sizeof(u32)));
    TRY(s.chunk_first.ensure((size_t)s.chunks_cap * (size_t)A * sizeof(u64)));
    TRY(s.run_cnt.ensure(((size_t)n + 1) * sizeof(u32)));
    TRY(s.run_off.ensure(((size_t)n + 2) * sizeof(u32)));
    TRY(s.runs.ensure((size_t)s.runs_cap * sizeof(ChunkEntry)));
    TRY(s.run_perm.ensure((size_t)s.runs_cap * sizeof(u32)));
    TRY(s.run_hist.ensure(CHUNK_BUCKETS * sizeof(u32)));
    TRY(s.best_mid.ensure(((size_t)n * A + 1) * sizeof(u32)));
    TRY(s.mid_n.ensure(((size_t)n * A + 1) * sizeof(u32)));
    TRY(s.mid_off.ensure(((size_t)n * A + 2) * sizeof(u32)));
    TRY(s.end_n.ensure(((size_t)n * A * 2 + 1) * sizeof(int)));
    TRY(s.end_pos.ensure(((size_t)n * A * 2 + 1) * sizeof(int)));
    TRY(s.pool.ensure((size_t)s.pool_cap * sizeof(Region)));
    TRY(s.sortbuf.ensure((size_t)s.pool_cap * 5 * sizeof(Region)));
    TRY(s.tmp.ensure((size_t)s.pieces_cap * sizeof(TmpPiece)));
    TRY(s.pieces.ensure((size_t)s.pieces_cap * sizeof(tgsf_piece)));
    TRY(s.res.ensure(((size_t)n + 1) * sizeof(tgsf_read_result)));
    TRY(s.header.ensure(sizeof(DevHeader)));
    TRY(s.mid_work.ensure((size_t)A * sizeof(u32))); // one work counter per k_mid_scan launch
    if (c->P.flags & TGSF_FLAG_GZ_BLOCKS) {
        // literal-only Huffman coding: <= 9/8 bytes per symbol on average, plus headers and padding per piece
        const u64 syms = n_bases * ((c->P.flags & TGSF_FLAG_GZ_FASTA) ? 1ull : 2ull);
        TRY(s.gz_blob.ensure((size_t)(syms + syms / 8 + (u64)s.pieces_cap * 512ull + 4096ull)));
        TRY(s.gz_spans.ensure((size_t)s.pieces_cap * sizeof(GzSpan)));
    }
    const size_t scan_words = 4 * (std::max<size_t>(nseg, (size_t)n * A) / SCANB_TILE) + 4096;
    TRY(s.scan_tmp.ensure(scan_words * sizeof(u32)));
    TRY(s.h_res.ensure(((size_t)n + 1) * sizeof(tgsf_read_result)));
    TRY(s.h_pieces.ensure(((size_t)n + 4096) * sizeof(tgsf_piece)));
    TRY(s.h_header.ensure(sizeof(DevHeader)));
    TRY(s.scratch.ensure(c->ads.host, c->sm_count * c->res_ctas_per_sm, RES_THREADS));
    if (c->fork_ends) TRY(s.scratch2.ensure(c->ads.host, c->sm_count * c->res_ctas_per_sm, RES_THREADS));
    return TGSF_OK;
}

// Myers word counts with an instantiation: the exact count up to 4 (adapters <= 256 bp, state in registers), then
// 8, 16 and 32 (<= 2048 bp; the state of those lives mostly in local memory, they are rare and only have to be right).
inline int round_nw(int nw) { return nw <= 4 ? nw : nw <= 8 ? 8 : nw <= 16 ? 16 : 32; }

template <typename F>
int for_nw(int nw, F f) {
    switch (nw) {
        case 1: return f(std::integral_constant<int, 1>());
        case 2: return f(std::integral_constant<int, 2>());
        case 3: return f(std::integral_constant<int, 3>());
        case 4: return f(std::integral_constant<int, 4>());
        case 8: return f(std::integral_constant<int, 8>());
        case 16: return f(std::integral_constant<int, 16>());
        case 32: return f(std::integral_constant<int, 32>());
        default: set_err("adapter longer than %d", TGSF_MAX_ADAPTER_LEN); return TGSF_ERR_INVALID;
    }
}

int check_launch(const char *what) {
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) {
        set_err("launch %s: %s", what, cudaGetErrorString(e));
        return TGSF_ERR_CUDA;
    }
    return TGSF_OK;
}

// K1 over a segment list (raw reads or kept pieces) + tile table construction.
int launch_scan_pass(tgsf_ctx *c, Slot &s, u32 n_seg, u64 *bin_cnt, u64 *bin_qual) {
    cudaStream_t st = s.stream.get();
    const size_t scan_words = s.scan_tmp.cap / sizeof(u32);
    TRY(exclusive_scan(c, st, s.tile_cnt.as<u32>(), s.tile_off.as<u32>(), n_seg, s.scan_tmp.as<u32>(), scan_words));
    if (n_seg) {
        k_fill_tiles<<<cdiv(n_seg, 256), 256, 0, st>>>(s.tile_off.as<u32>(), n_seg, s.seg_start.as<u64>(), s.seg_len.as<int>(), s.tiles.as<TileEntry>());
        c->launches++;
    }
    // the tile count lives on the device; the persistent grid reads it through tile_off[n_seg]
    const int grid = c->sm_count;
    u32 *status = &s.header.as<DevHeader>()->status;
    // n_tiles is passed by value through a tiny indirection kernel-free trick: tiles_cap bounds it,
    // and the kernel takes the device-side total.
    auto launch = [&](auto kern, size_t smem) {
        kern<<<grid, SCAN_THREADS, smem, st>>>(s.B.bases, s.B.quals, s.tiles.as<TileEntry>(), s.tile_off.as<u32>() + n_seg,
                                               s.seg_sum.as<u64>(), bin_cnt, bin_qual, c->P.qtype, c->P.L.max_bins, status);
    };
    if (!s.has_qual) launch(k_scan_tiles_dyn<false, false>, SCAN_SMEM_BYTES); // counts only
    else if (scan_needs_wide(s.tiles_cap, grid, c->P.qtype)) launch(k_scan_tiles_dyn<true, true>, SCAN_SMEM_BYTES_WIDE);
    else launch(k_scan_tiles_dyn<true, false>, SCAN_SMEM_BYTES);
    c->launches++;
    return check_launch("k_scan_tiles");
}

int launch_ends_qc(tgsf_ctx *c, Slot &s, u32 n_seg, const int *flag, bool clean) {
    if (c->P.bc_len <= 0 || n_seg == 0) return TGSF_OK;
    u64 *C = c->counters.as<u64>();
    const tgsf_counter_layout &L = c->P.L;
    u64 *cnt5 = C + (clean ? L.clean5p_cnt : L.raw5p_cnt), *q5 = C + (clean ? L.clean5p_qual : L.raw5p_qual);
    u64 *cnt3 = C + (clean ? L.clean3p_cnt : L.raw3p_cnt), *q3 = C + (clean ? L.clean3p_qual : L.raw3p_qual);
    const int grid = std::min<u32>((u32)c->sm_count * 4, cdiv(n_seg, ENDS_THREADS / 32));
    const size_t sm = c->P.bc_len <= ENDS_SMEM_ROWS ? (size_t)2 * c->P.bc_len * 10 * sizeof(u32) : 0;
    if (s.has_qual)
        k_ends_qc<true><<<grid, ENDS_THREADS, sm, s.stream.get()>>>(s.B.bases, s.B.quals, n_seg, s.seg_start.as<u64>(),
                                                                    s.seg_len.as<int>(), flag, c->P.bc_len, c->P.qtype,
                                                                    cnt5, q5, cnt3, q3);
    else
        k_ends_qc<false><<<grid, ENDS_THREADS, sm, s.stream.get()>>>(s.B.bases, s.B.quals, n_seg, s.seg_start.as<u64>(),
                                                                     s.seg_len.as<int>(), flag, c->P.bc_len, c->P.qtype,
                                                                     cnt5, q5, cnt3, q3);
    c->launches++;
    return check_launch("k_ends_qc");
}

// Everything up to (and including) the pool-size check: raw QC, quality band, K3 scans + counts.
int launch_head(tgsf_ctx *c, Slot &s) {
    cudaStream_t st = s.stream.get();
    const u32 n = s.B.n_reads;
    const int A = c->P.n_adapters;
    u64 *C = c->counters.as<u64>();
    const tgsf_counter_layout &L = c->P.L;
    DevParams P = c->P;
    P.has_qual = s.has_qual;
    CU(cudaMemsetAsync(s.header.p, 0, sizeof(DevHeader), st));
    u32 *status = &s.header.as<DevHeader>()->status;
    if (n == 0) {
        for (int i = 0; i <= 4; ++i) CU(cudaEventRecord(s.ev_stage[i].get(), st));
        return TGSF_OK;
    }

    CU(cudaEventRecord(s.ev_stage[0].get(), st));
    k_read_segments<<<cdiv(n, 256), 256, 0, st>>>(s.B, s.seg_start.as<u64>(), s.seg_len.as<int>(),
                                                  s.seg_sum.as<u64>(), s.tile_cnt.as<u32>(), L.max_bins, status);
    c->launches++;
    TRY(launch_scan_pass(c, s, n, C + L.raw_bin_cnt, C + L.raw_bin_qual));
    CU(cudaEventRecord(s.ev_stage[1].get(), st));
    if (s.has_qual)
        k_finalize_raw<true><<<cdiv(n, REG_THREADS), REG_THREADS, 0, st>>>(
            s.B, P, s.seg_sum.as<u64>(), s.res.as<tgsf_read_result>(), s.read_active.as<int>(),
            s.piece_cnt.as<u32>(), C);
    else
        k_finalize_raw<false><<<cdiv(n, REG_THREADS), REG_THREADS, 0, st>>>(
            s.B, P, s.seg_sum.as<u64>(), s.res.as<tgsf_read_result>(), s.read_active.as<int>(),
            s.piece_cnt.as<u32>(), C);
    c->launches++;
    TRY(launch_ends_qc(c, s, n, nullptr, false));
    CU(cudaEventRecord(s.ev_stage[2].get(), st));

    const bool filter = (P.flags & TGSF_FLAG_FILTER) != 0;
    if (filter && A > 0) {
        // End windows (k_ends): they only need read_active, so they are forked onto the slot's side stream and run
        // NEXT TO the middle scan: k_ends is a latency-bound serial chain per read end, k_mid_scan saturates the ALU
        // pipe with few warps, and together they fill the SM better than one after the other.  Adapters of one or two
        // words go two per thread (paired by word count).
        const AdapterCtx ACe = c->ads.ctx();
        const int res_grid_e = c->sm_count * c->res_ctas_per_sm;
        auto launch_ends = [&](cudaStream_t es, Scratch &sc) -> int {
            const AdapterCtx &AC = ACe;
            const int res_grid = res_grid_e;
        for (int nw : {1, 2, 3, 4, 8, 16, 32}) {
            std::vector<int> grp;
            for (int a = 0; a < A; ++a)
                if (c->ads.host[(size_t)a].nw == nw) grp.push_back(a);
            const size_t step = nw <= 2 ? 2 : 1;
            for (size_t i = 0; i < grp.size(); i += step) {
                const int a0 = grp[i], a1 = (step == 2 && i + 1 < grp.size()) ? grp[i + 1] : grp[i];
                const int qmax = std::max(c->ads.host[(size_t)a0].qlen, c->ads.host[(size_t)a1].qlen);
                const int grid_a = Scratch::grid_for(res_grid, RES_THREADS, 2 * qmax + 2, nw);
                const u64 stride_a = (u64)grid_a * RES_THREADS;
                TRY(for_nw(nw, [&](auto nwc) {
                    constexpr int NW = decltype(nwc)::value;
                    if constexpr (NW <= 2) {
                        if (a1 != a0)
                            k_ends<NW, 2><<<grid_a, RES_THREADS, 2 * 4 * 256 * NW * sizeof(u64), es>>>(
                                s.B, AC, a0, a1, P.end_len, A, s.read_active.as<int>(), s.end_n.as<int>(), s.end_pos.as<int>(),
                                sc.buf.as<u64>(), stride_a);
                        else
                            k_ends<NW, 1><<<grid_a, RES_THREADS, 4 * 256 * NW * sizeof(u64), es>>>(
                                s.B, AC, a0, a0, P.end_len, A, s.read_active.as<int>(), s.end_n.as<int>(), s.end_pos.as<int>(),
                                sc.buf.as<u64>(), stride_a);
                    } else {
                        k_ends<NW, 1><<<grid_a, RES_THREADS, NW <= 4 ? 4 * 256 * NW * sizeof(u64) : 0, es>>>(
                            s.B, AC, a0, a0, P.end_len, A, s.read_active.as<int>(), s.end_n.as<int>(), s.end_pos.as<int>(),
                            sc.buf.as<u64>(), stride_a);
                    }
                    c->launches++;
                    return check_launch("k_ends");
                }));
            }
        }
            return TGSF_OK;
        };
        if (c->fork_ends) {
            CU(cudaEventRecord(s.ev_fork.get(), st));
            CU(cudaStreamWaitEvent(s.stream2.get(), s.ev_fork.get(), 0));
            TRY(launch_ends(s.stream2.get(), s.scratch2));
            CU(cudaEventRecord(s.ev_join.get(), s.stream2.get()));
        }
        k_count_chunks<<<cdiv(n, 256), 256, 0, st>>>(s.B, s.read_active.as<int>(), P.end_len, s.chunk_shift, s.run_shift,
                                                     c->ads.min_q, s.chunk_cnt.as<u32>(), s.run_cnt.as<u32>(),
                                                     s.best_mid.as<u32>(), s.mid_n.as<u32>(), A);
        c->launches++;
        TRY(exclusive_scan(c, st, s.chunk_cnt.as<u32>(), s.chunk_off.as<u32>(), n, s.scan_tmp.as<u32>(),
                           s.scan_tmp.cap / sizeof(u32)));
        TRY(exclusive_scan(c, st, s.run_cnt.as<u32>(), s.run_off.as<u32>(), n, s.scan_tmp.as<u32>(),
                           s.scan_tmp.cap / sizeof(u32)));
        const int run_block = s.chunk_shift + s.run_shift;
        k_fill_chunks<<<cdiv(n, 256), 256, 0, st>>>(s.B, s.chunk_off.as<u32>(), P.end_len, s.chunk_shift, s.chunks.as<ChunkEntry>());
        k_fill_chunks<<<cdiv(n, 256), 256, 0, st>>>(s.B, s.run_off.as<u32>(), P.end_len, run_block, s.runs.as<ChunkEntry>());
        c->launches += 2;
        CU(cudaMemsetAsync(s.run_hist.p, 0, CHUNK_BUCKETS * sizeof(u32), st));
        k_chunk_hist<<<cdiv(n, UTIL_THREADS), UTIL_THREADS, 0, st>>>(s.B, s.run_off.as<u32>(), s.runs.as<ChunkEntry>(),
                                                                   P.end_len, run_block, s.run_hist.as<u32>());
        k_chunk_base<<<1, 32, 0, st>>>(s.run_hist.as<u32>());
        k_chunk_scatter<<<cdiv(n, UTIL_THREADS), UTIL_THREADS, 0, st>>>(s.B, s.run_off.as<u32>(), s.runs.as<ChunkEntry>(),
                                                                      P.end_len, run_block, s.run_hist.as<u32>(),
                                                                      s.run_perm.as<u32>());
        c->launches += 3;
        const AdapterCtx AC = c->ads.ctx();
        const u32 *n_runs_ptr = s.run_off.as<u32>() + n;
        const int res_grid = c->sm_count * c->res_ctas_per_sm;
        int mid_launch = 0;
        CU(cudaMemsetAsync(s.mid_work.p, 0, (size_t)A * sizeof(u32), st));
        // adapters with a live middle search, paired by word count: two per thread (long adapters: one)
        for (int nw : {1, 2, 3, 4, 8, 16, 32}) {
            std::vector<int> grp;
            for (int a = 0; a < A; ++a)
                if (c->ads.host[(size_t)a].nw == nw && c->ads.host[(size_t)a].k_mid > 0) grp.push_back(a);
            const size_t step = nw <= 4 ? 2 : 1;
            for (size_t i = 0; i < grp.size(); i += step) {
                const bool pair = step == 2 && i + 1 < grp.size();
                MidScanArgs M;
                M.a[0] = grp[i];
                M.a[1] = pair ? grp[i + 1] : grp[i];
                M.end_len = P.end_len;
                M.chunk_shift = s.chunk_shift;
                M.run_shift = s.run_shift;
                M.chunk_stride = s.chunks_cap;
                M.n_adapters = A;
                M.byte_mul[0] = 1u << 24;
                M.byte_mul[1] = 1u << 16;
                M.byte_mul[2] = 1u << 8;
                // a pair of adapters of at most 50 bp runs as one 96-bit filter vector (k_mid_scan_packed): dropping
                // their first <= 2 rows leaves the filter flagging well under 1 % of the chunks for an exact re-check
                const bool packed = pair && c->ads.host[(size_t)M.a[0]].qlen <= MID_PACKED_MAX_Q &&
                                    c->ads.host[(size_t)M.a[1]].qlen <= MID_PACKED_MAX_Q;
                TRY(for_nw(nw, [&](auto nwc) {
                    constexpr int NW = decltype(nwc)::value;
                    // row_bytes: the table row of a byte value, the stride mid_row_off scales by (AP * NW words in
                    // k_mid_scan_dyn, 16 bytes in k_mid_scan_packed)
                    auto launch = [&](auto kern, size_t smem, u32 row_bytes) {
                        M.byte_mul[3] = row_bytes;
                        int occ = 0; // persistent grid: exactly the resident CTA count
                        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, MID_THREADS, smem) != cudaSuccess || occ < 1) occ = 4;
                        if (c->mid_ctas_per_sm > 0) occ = std::min(occ, c->mid_ctas_per_sm);
                        kern<<<c->sm_count * occ, MID_THREADS, smem, st>>>(
                            s.B, AC, M, s.chunk_off.as<u32>(), s.runs.as<ChunkEntry>(), s.run_perm.as<u32>(), n_runs_ptr,
                            s.chunk_min.as<uint8_t>(), s.chunk_hits.as<u32>(), s.chunk_first.as<u64>(),
                            s.best_mid.as<u32>(), s.mid_work.as<u32>() + mid_launch);
                    };
                    if constexpr (NW <= 4) {
                        if (packed) launch(k_mid_scan_packed, 0, 16);
                        else if (pair) launch(k_mid_scan_dyn<NW, 2>, 256 * 2 * NW * sizeof(u64), 8 * 2 * NW);
                        else launch(k_mid_scan_dyn<NW, 1>, 256 * NW * sizeof(u64), 8 * NW);
                    } else {
                        launch(k_mid_scan_dyn<NW, 1>, 0, 8 * NW); // table read from global memory
                    }
                    c->launches++;
                    ++mid_launch;
                    return check_launch("k_mid_scan");
                }));
            }
        }
        CU(cudaEventRecord(s.ev_stage[3].get(), st));
        for (int a = 0; a < A; ++a) {
            const DevAdapter &Ah = c->ads.host[(size_t)a];
            if (Ah.k_mid <= 0) continue;
            const int grid_a = Scratch::grid_for(res_grid, RES_THREADS, 2 * Ah.qlen + 2, Ah.nw);
            TRY(for_nw(Ah.nw, [&](auto nwc) {
                constexpr int NW = decltype(nwc)::value;
                k_mid_count<NW><<<grid_a, RES_THREADS, 0, st>>>(
                    s.B, AC, a, P.end_len, A, s.best_mid.as<u32>(), s.chunk_off.as<u32>(), s.chunks_cap,
                    s.chunk_min.as<uint8_t>(), s.chunk_hits.as<u32>(), s.chunk_first.as<u64>(),
                    s.mid_n.as<u32>(), s.scratch.buf.as<u64>(), (u64)grid_a * RES_THREADS);
                c->launches++;
                return check_launch("k_mid_count");
            }));
        }
        if (c->fork_ends) CU(cudaStreamWaitEvent(st, s.ev_join.get(), 0)); // the end-window results (side stream)
        else TRY(launch_ends(st, s.scratch));
        TRY(exclusive_scan(c, st, s.mid_n.as<u32>(), s.mid_off.as<u32>(), n * (u32)A, s.scan_tmp.as<u32>(),
                           s.scan_tmp.cap / sizeof(u32)));
        k_check_pool<<<1, 1, 0, st>>>(s.mid_off.as<u32>() + (size_t)n * A, s.pool_cap, status);
        c->launches++;
    } else {
        CU(cudaEventRecord(s.ev_stage[3].get(), st));
    }
    CU(cudaEventRecord(s.ev_stage[4].get(), st));
    return check_launch("head");
}

// K4, the -p repeat check.  k <= 16: k_kmer_tag16 over all pieces, as many CTAs per SM as fit; it hands the pieces too
// long for its 16-bit positions to a long list, which k_kmer_smem (k <= 12) or the hash kernel k_kmer (k = 13 .. 16)
// works through next.  k > 16: k_kmer over all pieces.
int launch_kmer(tgsf_ctx *c, Slot &s, const DevParams &P) {
    cudaStream_t st = s.stream.get();
    DevHeader *H = s.header.as<DevHeader>();
    u64 *C = c->counters.as<u64>();
    tgsf_piece *pieces = s.pieces.as<tgsf_piece>();
    if (P.kmer > 16) {
        k_kmer<u64><<<c->sm_count, KMER_THREADS, KMER_SMEM_BYTES, st>>>(s.B, P, pieces, &H->tmp_cursor, C, &H->status, nullptr,
                                                                       c->kmer_fill_cap);
        c->launches++;
        return check_launch("k_kmer");
    }
    TRY(s.kmer_long_list.ensure((size_t)s.pieces_cap * sizeof(u32)));
    u32 *long_list = s.kmer_long_list.as<u32>();
    k_kmer_tag16<<<c->sm_count * c->kmer16_ctas_per_sm, KMER16_THREADS, KMER16_SMEM_BYTES, st>>>(
        s.B, P, pieces, &H->tmp_cursor, C, &H->status, &H->kmer_work, long_list, &H->kmer_long, c->kmer16_list_cap);
    if (P.kmer <= 12)
        k_kmer_smem<<<c->sm_count, KMER_SB_THREADS, KMER_SB_SMEM_BYTES, st>>>(s.B, P, pieces, &H->kmer_long, C, &H->status,
                                                                             long_list);
    else if (P.kmer <= 15)
        k_kmer<u32><<<c->sm_count, KMER_THREADS, KMER_SMEM_BYTES, st>>>(s.B, P, pieces, &H->kmer_long, C, &H->status, long_list,
                                                                       c->kmer_fill_cap);
    else
        k_kmer<u64><<<c->sm_count, KMER_THREADS, KMER_SMEM_BYTES, st>>>(s.B, P, pieces, &H->kmer_long, C, &H->status, long_list,
                                                                       c->kmer_fill_cap);
    c->launches += 2;
    return check_launch("k_kmer");
}

// Contaminant screen of set cs over the pieces still emitted after K4; writes piece fields only.  A labelled set also
// attributes the pieces: the contaminant ones into the set's tallies, or, with attr_out (tgsf_contam_classify), every
// piece with a hit into attr_out[piece].
int launch_contam(tgsf_ctx *c, Slot &s, const ContamSet &cs, int2 *attr_out) {
    cudaStream_t st = s.stream.get();
    DevHeader *H = s.header.as<DevHeader>();
    const u32 cap = s.pieces_cap;
    // pieces are disjoint parts of the reads: at most n_bases / CHUNK full chunks plus one partial chunk per piece
    const size_t chunks_cap = (size_t)(s.n_bases / CONTAM_CHUNK) + cap + 16;
    TRY(s.contam_cnt.ensure((size_t)cap * sizeof(u32)));
    TRY(s.contam_off.ensure(((size_t)cap + 1) * sizeof(u32)));
    TRY(s.contam_chunks.ensure(chunks_cap * sizeof(ContamChunk)));
    k_contam_count<<<cdiv(cap, 256), 256, 0, st>>>(s.pieces.as<tgsf_piece>(), &H->tmp_cursor, cap, cs.k,
                                                   CONTAM_CHUNK, s.contam_cnt.as<u32>(), &H->status);
    c->launches++;
    TRY(exclusive_scan(c, st, s.contam_cnt.as<u32>(), s.contam_off.as<u32>(), cap, s.scan_tmp.as<u32>(),
                       s.scan_tmp.cap / sizeof(u32)));
    k_contam_fill<<<cdiv(cap, 256), 256, 0, st>>>(s.B, s.pieces.as<tgsf_piece>(), s.contam_off.as<u32>(), cap, cs.k,
                                                  CONTAM_CHUNK, s.contam_chunks.as<ContamChunk>());
    c->launches++;
    if (cs.pf_bits.p)
        k_contam_screen<true><<<c->sm_count, CONTAM_THREADS, CONTAM_PF_SMEM_BYTES, st>>>(
            s.B.bases, s.contam_chunks.as<ContamChunk>(), s.contam_off.as<u32>() + cap, cs.k, cs.table.as<u64>(), cs.mask,
            cs.pf_bits.as<u32>(), s.pieces.as<tgsf_piece>(), &H->status);
    else
        k_contam_screen<false><<<c->sm_count * 4, CONTAM_THREADS, 0, st>>>(
            s.B.bases, s.contam_chunks.as<ContamChunk>(), s.contam_off.as<u32>() + cap, cs.k, cs.table.as<u64>(), cs.mask,
            nullptr, s.pieces.as<tgsf_piece>(), &H->status);
    c->launches++;
    if (!cs.labelled()) {
        k_contam_decide<false><<<cdiv(cap, 256), 256, 0, st>>>(s.pieces.as<tgsf_piece>(), &H->tmp_cursor, cap, cs.k,
                                                               cs.ppm, &H->status, nullptr, nullptr, false);
        c->launches++;
        return check_launch("contam");
    }
    TRY(s.contam_list.ensure((size_t)std::max<u32>(cap, 1) * sizeof(u32)));
    k_contam_decide<true><<<cdiv(cap, 256), 256, 0, st>>>(s.pieces.as<tgsf_piece>(), &H->tmp_cursor, cap, cs.k, cs.ppm,
                                                          &H->status, s.contam_list.as<u32>(), &H->contam_list_n,
                                                          attr_out != nullptr);
    unsigned long long *tally = attr_out ? nullptr : cs.tally.as<unsigned long long>();
    if (cs.pf_bits.p)
        k_contam_attr<true><<<c->sm_count, ATTR_THREADS, CONTAM_PF_SMEM_BYTES, st>>>(
            s.B, s.pieces.as<tgsf_piece>(), s.contam_list.as<u32>(), &H->contam_list_n, &H->contam_work, cs.k,
            cs.table.as<u64>(), cs.mask, cs.labels.as<u32>(), cs.pf_bits.as<u32>(), cs.n_records, tally, attr_out,
            &H->status);
    else
        k_contam_attr<false><<<c->sm_count * c->attr_ctas_per_sm, ATTR_THREADS, 0, st>>>(
            s.B, s.pieces.as<tgsf_piece>(), s.contam_list.as<u32>(), &H->contam_list_n, &H->contam_work, cs.k,
            cs.table.as<u64>(), cs.mask, cs.labels.as<u32>(), nullptr, cs.n_records, tally, attr_out, &H->status);
    c->launches += 2;
    return check_launch("contam");
}

// DUST screen over the pieces still emitted after K4 and the contaminant screen: the contaminant screen's chunk
// kernels with 64-base windows and DUST_CHUNK windows a chunk (the two screens run one after the other on the slot's
// stream and share the chunk-list buffers), the masked bases of every piece into s.dust_masked, then the threshold.
// ppm 0 skips the threshold (tgsf_dust_detect).  Writes piece status only.
int launch_dust(tgsf_ctx *c, Slot &s, int level, u64 ppm) {
    cudaStream_t st = s.stream.get();
    DevHeader *H = s.header.as<DevHeader>();
    const u32 cap = s.pieces_cap;
    const size_t chunks_cap = (size_t)(s.n_bases / DUST_CHUNK) + cap + 16;
    TRY(s.contam_cnt.ensure((size_t)cap * sizeof(u32)));
    TRY(s.contam_off.ensure(((size_t)cap + 1) * sizeof(u32)));
    TRY(s.contam_chunks.ensure(chunks_cap * sizeof(ContamChunk)));
    TRY(s.dust_masked.ensure((size_t)std::max<u32>(cap, 1) * sizeof(u32)));
    CU(cudaMemsetAsync(s.dust_masked.p, 0, (size_t)cap * sizeof(u32), st));
    k_contam_count<<<cdiv(cap, 256), 256, 0, st>>>(s.pieces.as<tgsf_piece>(), &H->tmp_cursor, cap, DUST_WINDOW,
                                                   DUST_CHUNK, s.contam_cnt.as<u32>(), &H->status);
    c->launches++;
    TRY(exclusive_scan(c, st, s.contam_cnt.as<u32>(), s.contam_off.as<u32>(), cap, s.scan_tmp.as<u32>(),
                       s.scan_tmp.cap / sizeof(u32)));
    k_contam_fill<<<cdiv(cap, 256), 256, 0, st>>>(s.B, s.pieces.as<tgsf_piece>(), s.contam_off.as<u32>(), cap,
                                                  DUST_WINDOW, DUST_CHUNK, s.contam_chunks.as<ContamChunk>());
    c->launches++;
    k_dust_screen<<<c->sm_count * (2048 / DUST_THREADS), DUST_THREADS, 0, st>>>(
        s.B.bases, s.contam_chunks.as<ContamChunk>(), s.contam_off.as<u32>() + cap, (u32)(61 * level),
        s.dust_masked.as<u32>(), &H->status);
    c->launches++;
    if (ppm) {
        k_dust_decide<<<cdiv(cap, 256), 256, 0, st>>>(s.pieces.as<tgsf_piece>(), &H->tmp_cursor, cap,
                                                      s.dust_masked.as<u32>(), ppm, &H->status);
        c->launches++;
    }
    return check_launch("dust");
}

// Fold-back screen over the pieces K5 emitted, before K4: the shared-memory path for every piece, then the global
// path for the pieces it handed over.  Writes piece fields and the context's fold statistics only.
int launch_fold(tgsf_ctx *c, Slot &s, tgsf_piece *pieces, const u32 *n_pieces, DevHeader *H, tgsf_fold_result *out,
                u32 max_len) {
    cudaStream_t st = s.stream.get();
    const u32 bins_cap = fold_bins(std::max<u32>(max_len, FOLD_K));
    const u32 grid = (u32)c->sm_count;
    TRY(s.fold_long_list.ensure((size_t)std::max<u32>(s.pieces_cap, 1) * sizeof(u32)));
    TRY(s.fold_ws.ensure((size_t)grid * fold_ws_bytes(bins_cap)));
    unsigned long long *stats = out ? nullptr : c->fold_stats.as<unsigned long long>();
    k_fold_smem<<<grid, FOLD_THREADS, FOLD_SMEM_BYTES, st>>>(s.B, pieces, n_pieces, &H->fold_work,
                                                             s.fold_long_list.as<u32>(), &H->fold_long, c->P.min_len,
                                                             stats, out, &H->status);
    k_fold_global<<<grid, FOLD_THREADS, 0, st>>>(s.B, pieces, s.fold_long_list.as<u32>(), &H->fold_long,
                                                 &H->fold_long_work, s.fold_ws.as<uint8_t>(), bins_cap, c->P.min_len,
                                                 stats, out, &H->status);
    c->launches += 2;
    return check_launch("fold");
}

// From the region pool onwards; re-runnable after a pool overflow (touches no counter before the
// overflow check has passed).
int launch_tail(tgsf_ctx *c, Slot &s) {
    cudaStream_t st = s.stream.get();
    const u32 n = s.B.n_reads;
    const int A = c->P.n_adapters;
    u64 *C = c->counters.as<u64>();
    const tgsf_counter_layout &L = c->P.L;
    DevParams P = c->P;
    P.has_qual = s.has_qual;
    DevHeader *H = s.header.as<DevHeader>();
    if (n == 0) {
        for (int i = 5; i <= TGSF_N_STAGES; ++i) CU(cudaEventRecord(s.ev_stage[i].get(), st));
        return TGSF_OK;
    }
    const bool filter = (P.flags & TGSF_FLAG_FILTER) != 0;
    const AdapterCtx AC = c->ads.ctx();
    const int res_grid = c->sm_count * c->res_ctas_per_sm;
    if (filter && A > 0) {
        for (int a = 0; a < A; ++a) {
            const DevAdapter &Ah = c->ads.host[(size_t)a];
            if (Ah.k_mid <= 0) continue;
            TRY(for_nw(Ah.nw, [&](auto nwc) {
                constexpr int NW = decltype(nwc)::value;
                k_mid_emit<NW><<<res_grid, RES_THREADS, 0, st>>>(
                    s.B, AC, a, P.end_len, s.chunk_shift, P.extra_len, A, s.best_mid.as<u32>(), s.chunk_off.as<u32>(),
                    s.chunks.as<ChunkEntry>(), s.chunks_cap, s.chunk_min.as<uint8_t>(), s.chunk_hits.as<u32>(),
                    s.chunk_first.as<u64>(), s.mid_n.as<u32>(), s.mid_off.as<u32>(), s.pool.as<Region>(), &H->status);
                c->launches++;
                return check_launch("k_mid_emit");
            }));
        }
    } else if (filter) {
        // no adapters: adapterMap still applies the fixed trims; no location arrays to read
        CU(cudaMemsetAsync(s.mid_n.p, 0, sizeof(u32), st));
    }
    // the host copies an optimistic prefix of the piece array before the count is known (enqueue_d2h): define it
    CU(cudaMemsetAsync(s.pieces.p, 0, (size_t)std::min<u32>(s.pieces_cap, n + 4096) * sizeof(tgsf_piece), st));
    k_regions<<<cdiv(n, REG_THREADS), REG_THREADS, 0, st>>>(
        s.B, P, s.read_active.as<int>(), s.end_n.as<int>(), s.end_pos.as<int>(), s.mid_n.as<u32>(),
        s.mid_off.as<u32>(), s.pool.as<Region>(), s.sortbuf.as<Region>(), s.pool_cap * 5, &H->sort_cursor,
        s.res.as<tgsf_read_result>(), s.piece_cnt.as<u32>(), s.tmp.as<TmpPiece>(), s.pieces_cap,
        &H->tmp_cursor, C, &H->status);
    c->launches++;
    TRY(exclusive_scan(c, st, s.piece_cnt.as<u32>(), s.piece_begin.as<u32>(), n, s.scan_tmp.as<u32>(),
                       s.scan_tmp.cap / sizeof(u32)));
    const u32 place_n = std::max(n, s.pieces_cap);
    k_place_pieces<<<cdiv(place_n, 256), 256, 0, st>>>(s.tmp.as<TmpPiece>(), &H->tmp_cursor,
                                                       s.piece_begin.as<u32>(), s.res.as<tgsf_read_result>(),
                                                       s.pieces.as<tgsf_piece>(), n,
                                                       (P.flags & TGSF_FLAG_ONLY_QC) ? 1 : 0, &H->status);
    c->launches++;
    CU(cudaEventRecord(s.ev_stage[5].get(), st));
    if (!(P.flags & TGSF_FLAG_ONLY_QC)) {
        if (c->foldback)
            TRY(launch_fold(c, s, s.pieces.as<tgsf_piece>(), &H->tmp_cursor, H, nullptr, P.L.max_bins * SCAN_BIN));
        if (P.min_repeat > 0) TRY(launch_kmer(c, s, P));
        if (c->contam.installed()) TRY(launch_contam(c, s, c->contam, nullptr));
        if (c->dust_level) TRY(launch_dust(c, s, c->dust_level, c->dust_ppm));
        CU(cudaEventRecord(s.ev_stage[6].get(), st));
        // clean pass over the kept pieces (T.cpp:1991-2009); piece count is device-side, the
        // kernels are launched over the capacity and bound themselves by the header.
        k_piece_segments_dyn<<<cdiv(s.pieces_cap, 256), 256, 0, st>>>(
            s.B, s.pieces.as<tgsf_piece>(), &H->tmp_cursor, s.pieces_cap, s.seg_start.as<u64>(),
            s.seg_len.as<int>(), s.seg_sum.as<u64>(), s.tile_cnt.as<u32>(), &H->status);
        c->launches++;
        TRY(launch_scan_pass(c, s, s.pieces_cap, C + L.clean_bin_cnt, C + L.clean_bin_qual));
        if (s.has_qual)
            k_finalize_clean_dyn<true><<<cdiv(s.pieces_cap, REG_THREADS), REG_THREADS, 0, st>>>(
                P, s.pieces.as<tgsf_piece>(), &H->tmp_cursor, s.pieces_cap, s.seg_sum.as<u64>(),
                s.seg_flag.as<int>(), C, &H->status);
        else
            k_finalize_clean_dyn<false><<<cdiv(s.pieces_cap, REG_THREADS), REG_THREADS, 0, st>>>(
                P, s.pieces.as<tgsf_piece>(), &H->tmp_cursor, s.pieces_cap, s.seg_sum.as<u64>(),
                s.seg_flag.as<int>(), C, &H->status);
        c->launches++;
        TRY(launch_ends_qc(c, s, s.pieces_cap, s.seg_flag.as<int>(), true));
    } else {
        CU(cudaEventRecord(s.ev_stage[6].get(), st));
    }
    if ((P.flags & TGSF_FLAG_GZ_BLOCKS) && !(P.flags & TGSF_FLAG_ONLY_QC)) {
        // deflate blocks of the emitted pieces (timed with the clean stage)
        const bool fasta = (P.flags & TGSF_FLAG_GZ_FASTA) || !s.has_qual;
        const u64 syms = s.n_bases * (fasta ? 1ull : 2ull);
        const u64 used_cap = std::min<u64>(s.gz_blob.cap, syms + syms / 8 + (u64)s.pieces_cap * 512ull + 4096ull) & ~3ull;
        CU(cudaMemsetAsync(s.gz_blob.p, 0, (size_t)used_cap, st));
        k_gz_encode<<<c->sm_count * 6, GZ_THREADS, 0, st>>>(s.B, s.pieces.as<tgsf_piece>(), &H->tmp_cursor, fasta ? 1 : 0,
                                                          s.gz_blob.as<u32>(), used_cap, &H->gz_cursor,
                                                          s.gz_spans.as<GzSpan>(), &H->gz_overflow, &H->status);
        c->launches++;
    }
    CU(cudaEventRecord(s.ev_stage[7].get(), st));
    return check_launch("tail");
}

int enqueue_d2h(tgsf_ctx *c, Slot &s) {
    (void)c;
    cudaStream_t st = s.stream.get();
    const u32 n = s.B.n_reads;
    CU(cudaMemcpyAsync(s.h_header.p, s.header.p, sizeof(DevHeader), cudaMemcpyDeviceToHost, st));
    if (n) CU(cudaMemcpyAsync(s.h_res.p, s.res.p, (size_t)n * sizeof(tgsf_read_result), cudaMemcpyDeviceToHost, st));
    // the piece count is only known on the device: copy an optimistic prefix without waiting for it (entries
    // beyond the count are never read; tgsf_collect fetches the rest if a batch produced more)
    s.h_pieces_copied = std::min<u32>(s.pieces_cap, n + 4096);
    if (s.h_pieces_copied)
        CU(cudaMemcpyAsync(s.h_pieces.p, s.pieces.p, (size_t)s.h_pieces_copied * sizeof(tgsf_piece),
                           cudaMemcpyDeviceToHost, st));
    return TGSF_OK;
}

int run_pipeline(tgsf_ctx *c, Slot &s) {
    TRY(launch_head(c, s));
    TRY(launch_tail(c, s));
    CU(cudaEventRecord(s.ev_k1.get(), s.stream.get()));
    TRY(enqueue_d2h(c, s));
    CU(cudaEventRecord(s.ev_end.get(), s.stream.get()));
    return TGSF_OK;
}

int validate_params(const tgsf_params *p) {
    if (!p) { set_err("params is NULL"); return TGSF_ERR_INVALID; }
    if (p->n_adapters < 0 || p->n_adapters > TGSF_MAX_ADAPTERS) { set_err("n_adapters out of range"); return TGSF_ERR_INVALID; }
    if (p->n_adapters > 0 && (!p->adapter_seq || !p->adapter_len)) { set_err("adapter arrays missing"); return TGSF_ERR_INVALID; }
    for (int a = 0; a < p->n_adapters; ++a)
        if (p->adapter_len[a] <= 0 || p->adapter_len[a] > TGSF_MAX_ADAPTER_LEN || !p->adapter_seq[a]) {
            set_err("adapter %d has invalid length %d", a, p->adapter_len[a]);
            return TGSF_ERR_INVALID;
        }
    if ((p->flags & TGSF_FLAG_FILTER) && p->n_adapters > 0 && !(p->end_sim > 0.0f && p->mid_sim > 0.0f)) {
        set_err("end_sim / mid_sim must be > 0 when filtering");
        return TGSF_ERR_INVALID;
    }
    if (p->min_repeat > 0 && (p->kmer < 1 || p->kmer > 31)) { set_err("kmer must be in [1,31]"); return TGSF_ERR_INVALID; }
    if (p->bc_len < 0 || p->end_len < 0 || p->extra_len < 0) { set_err("negative length parameter"); return TGSF_ERR_INVALID; }
    if (p->n_slots < 0 || p->n_slots > 4) { set_err("n_slots out of range"); return TGSF_ERR_INVALID; }
    return TGSF_OK;
}

// Integer stand-ins for the float tests of GetEditDistance, evaluated with the same C++ float
// expressions the reference uses.
void fill_thresholds(DevAdapter &A, const tgsf_params *p) {
    const int qLen = A.qlen;
    const float endSim = p->end_sim, midSim = p->mid_sim;
    auto min_mlen = [&](float sim, int match_len) {
        int m = 0;
        for (; m <= qLen; ++m) {
            float s = static_cast<float>(m) / qLen; // T.cpp:1250 / 1287
            if (s >= sim) break;
        }
        return std::max(m, match_len); // m == qLen + 1: can never pass
    };
    A.k_mid = std::min(qLen - p->mid_match_len + 1, qLen - 1); // T.cpp:1233
    A.k_end = std::min(qLen - p->end_match_len + 1, qLen - 1); // T.cpp:1271
    A.thr_mid = min_mlen(midSim, p->mid_match_len);
    A.thr_end = min_mlen(endSim, p->end_match_len);
    if (A.thr_mid > qLen) A.k_mid = 0;
    if (A.thr_end > qLen) A.k_end = 0;
    A.end_extra = endSim > 0.0f ? int(qLen / endSim) : 0; // T.cpp:1267
    A.halo_mid = A.k_mid > 0 ? ((qLen + A.k_mid - 1 + 15) / 16) * 16 : 0;
}

// The set-up of the screens' stand-alone entry points (tgsf_fold_detect, tgsf_dust_detect): n > 0 host records
// seq[offsets[i], offsets[i+1]) become whole TGSF_PIECE_EMIT pieces in the slot of a bare context (no adapters, one
// slot), so that the pipeline's kernels run on them unchanged.  The arguments are checked (offsets[0] == 0, ascending,
// each piece < 2^31 bases, seq present) before the device is touched; the copies are enqueued on the slot's stream.
struct RecordPieces {
    CtxPtr c;
    DBuf d_off;
    u64 longest = 0;

    int setup(const char *fn, int device, const uint8_t *seq, const uint64_t *offsets, uint32_t n) {
        if (offsets[0] != 0) { set_err("%s: offsets[0] must be 0", fn); return TGSF_ERR_INVALID; }
        for (uint32_t i = 0; i < n; ++i) {
            if (offsets[i + 1] < offsets[i]) { set_err("%s: offsets not ascending at %u", fn, i); return TGSF_ERR_INVALID; }
            longest = std::max<u64>(longest, offsets[i + 1] - offsets[i]);
        }
        if (longest >= (1ull << 31)) { set_err("%s: a piece of %llu bases", fn, (unsigned long long)longest); return TGSF_ERR_INVALID; }
        const u64 n_bytes = offsets[n];
        if (n_bytes && !seq) { set_err("%s: seq is NULL", fn); return TGSF_ERR_INVALID; }
        CU(cudaSetDevice(device));
        tgsf_params p;
        memset(&p, 0, sizeof(p));
        p.n_slots = 1;
        tgsf_ctx *raw = nullptr;
        TRY(tgsf_create(device, &p, &raw));
        c.reset(raw);
        Slot &s = slot();
        cudaStream_t st = s.stream.get();
        s.pieces_cap = n;
        s.n_bases = n_bytes;
        TRY(s.in_bases.ensure(std::max<u64>(n_bytes, 1)));
        TRY(d_off.ensure(((size_t)n + 1) * sizeof(u64)));
        TRY(s.pieces.ensure((size_t)n * sizeof(tgsf_piece)));
        TRY(s.header.ensure(sizeof(DevHeader)));
        TRY(s.scan_tmp.ensure((4 * ((size_t)n / SCANB_TILE) + 4096) * sizeof(u32)));
        pc.resize((size_t)n);
        for (uint32_t i = 0; i < n; ++i) {
            memset(&pc[i], 0, sizeof(tgsf_piece));
            pc[i].read = (int32_t)i;
            pc[i].len = (int32_t)(offsets[i + 1] - offsets[i]);
            pc[i].repeat_len = -1;
            pc[i].status = TGSF_PIECE_EMIT;
        }
        memset(&h, 0, sizeof(h));
        h.tmp_cursor = n;
        if (n_bytes) CU(cudaMemcpyAsync(s.in_bases.p, seq, n_bytes, cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(d_off.p, offsets, ((size_t)n + 1) * sizeof(u64), cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(s.pieces.p, pc.data(), (size_t)n * sizeof(tgsf_piece), cudaMemcpyHostToDevice, st));
        CU(cudaMemcpyAsync(s.header.p, &h, sizeof(h), cudaMemcpyHostToDevice, st));
        s.B.bases = s.in_bases.as<uint8_t>();
        s.B.quals = nullptr;
        s.B.offsets = d_off.as<u64>();
        s.B.n_reads = n;
        return TGSF_OK;
    }
    Slot &slot() { return c->slots[0]; }
    // Waits for the stream (the caller's result copies enqueued) and checks the device status.
    int finish(const char *fn) {
        Slot &s = slot();
        CU(cudaMemcpyAsync(&h, s.header.p, sizeof(h), cudaMemcpyDeviceToHost, s.stream.get()));
        CU(cudaStreamSynchronize(s.stream.get()));
        if (h.status == DEV_STATUS_HASH_OVERFLOW) { set_err("%s: %s", fn, HASH_OVERFLOW_MSG); return TGSF_ERR_CAPACITY; }
        if (h.status != DEV_STATUS_OK) { set_err("%s: device status %u", fn, h.status); return TGSF_ERR_CUDA; }
        return TGSF_OK;
    }

private:
    std::vector<tgsf_piece> pc; // host staging of the copies, alive until finish()
    DevHeader h;
};

}  // namespace

// ---------------------------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------------------------
extern "C" {

const char *tgsf_version(void) { return "libtgsf_cuda 0.1 (sm_100a; TGSFilter v1.11 per-read path)"; }
const char *tgsf_last_error(void) { return g_err; }

int tgsf_create(int device, const tgsf_params *params, tgsf_ctx **out) {
    if (!out) { set_err("out is NULL"); return TGSF_ERR_INVALID; }
    *out = nullptr;
    TRY(validate_params(params));
    CU(cudaSetDevice(device));
    CtxPtr c(new (std::nothrow) tgsf_ctx());
    if (!c) return TGSF_ERR_NOMEM;
    c->device = device;
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    c->sm_count = prop.multiProcessorCount;
    DevParams &P = c->P;
    P.min_len = params->min_len;
    P.max_len = params->max_len;
    P.min_q = (double)params->min_q;
    P.max_q = (double)params->max_q;
    P.bc_len = params->bc_len;
    P.head_trim = params->head_trim;
    P.tail_trim = params->tail_trim;
    P.end_len = params->end_len;
    P.extra_len = params->extra_len;
    P.kmer = params->kmer;
    P.min_repeat = params->min_repeat;
    P.qtype = params->qtype;
    P.flags = params->flags;
    P.n_adapters = params->n_adapters;
    P.has_qual = 1;
    tgsf_make_layout(params->bc_len, params->max_read_len, &P.L);

    TRY(c->ads.build((const uint8_t *const *)params->adapter_seq, params->adapter_len, params->n_adapters));
    for (auto &A : c->ads.host) fill_thresholds(A, params);
    TRY(c->ads.upload());
    TRY(c->counters.ensure((size_t)P.L.n_u64 * sizeof(u64)));
    CU(cudaMemset(c->counters.p, 0, (size_t)P.L.n_u64 * sizeof(u64)));
    c->slots.resize((size_t)(params->n_slots > 0 ? params->n_slots : 2));
    for (auto &s : c->slots) TRY(slot_init(s));
    TRY(create(c->ev_epoch));
    CU(cudaEventRecord(c->ev_epoch.get(), c->slots[0].stream.get()));
    CU(cudaEventSynchronize(c->ev_epoch.get()));
    // dynamic shared-memory limits only: no kernel asks for a carve-out (measured, DESIGN §8)
    auto smem = [](auto kern, int bytes) { return cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes); };
    CU(smem(k_scan_tiles_dyn<true, false>, SCAN_SMEM_BYTES));
    CU(smem(k_scan_tiles_dyn<false, false>, SCAN_SMEM_BYTES));
    CU(smem(k_scan_tiles_dyn<true, true>, SCAN_SMEM_BYTES_WIDE));
    CU(smem(k_kmer<u32>, KMER_SMEM_BYTES));
    CU(smem(k_kmer<u64>, KMER_SMEM_BYTES));
    CU(smem(k_kmer_smem, KMER_SB_SMEM_BYTES));
    CU(smem(k_kmer_tag16, KMER16_SMEM_BYTES));
    CU(smem(k_contam_screen<true>, CONTAM_PF_SMEM_BYTES));
    CU(smem(k_contam_attr<true>, CONTAM_PF_SMEM_BYTES));
    CU(smem(k_fold_smem, FOLD_SMEM_BYTES));
    int occ = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_kmer_tag16, KMER16_THREADS, KMER16_SMEM_BYTES) == cudaSuccess && occ >= 1)
        c->kmer16_ctas_per_sm = occ;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_contam_attr<false>, ATTR_THREADS, 0) == cudaSuccess && occ >= 1)
        c->attr_ctas_per_sm = occ;
    if (const char *e = getenv("TGSF_MID_CTAS")) c->mid_ctas_per_sm = atoi(e);
    if (const char *e = getenv("TGSF_FORK_ENDS")) c->fork_ends = atoi(e) != 0;
    if (const char *e = getenv("TGSF_RES_CTAS")) c->res_ctas_per_sm = std::max(1, std::min(16, atoi(e)));
    // TGSF_SM_COUNT=n: size every grid and the chunk-shift rule as if the device had n SMs (clamped to
    // [1, real count]), so that tests reach the launch shapes of multi-Gbase batches with small batches
    if (const char *e = getenv("TGSF_SM_COUNT")) c->sm_count = std::max(1, std::min(c->sm_count, atoi(e)));
    if (const char *e = getenv("TGSF_KMER16_LIST_CAP")) c->kmer16_list_cap = (u32)std::min<long>(std::max<long>(atol(e), 32), (long)KMER16_LIST_CAP);
    if (const char *e = getenv("TGSF_KMER_FILL_CAP")) c->kmer_fill_cap = (u32)std::min<long long>(std::max<long long>(atoll(e), 1), ~0u);
    *out = c.release();
    return TGSF_OK;
}

int tgsf_destroy(tgsf_ctx *c) {
    if (!c) return TGSF_OK;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    delete c;
    return TGSF_OK;
}

// tgsf_set_contaminants, and with record_kmers tgsf_set_contaminants_labelled: the labels, their key counts and zeroed
// tallies besides the table.
static int install_contaminants(const char *fn, tgsf_ctx *c, const uint8_t *seq, const uint64_t *offsets,
                                uint32_t n_seqs, int32_t k, float min_frac, uint64_t *n_kmers, uint64_t *record_kmers) {
    const bool labelled = record_kmers != nullptr;
    if (!c || !offsets || !n_kmers || n_seqs == 0) { set_err("%s: missing argument", fn); return TGSF_ERR_INVALID; }
    if (c->outstanding) { set_err("%s with %u batch(es) outstanding", fn, c->outstanding); return TGSF_ERR_STATE; }
    if (labelled && n_seqs > TGSF_CONTAM_MAX_RECORDS) { set_err("%s: more than %u records", fn, TGSF_CONTAM_MAX_RECORDS); return TGSF_ERR_INVALID; }
    if (k < CONTAM_K_MIN || k > CONTAM_K_MAX) { set_err("contaminant k must be in [%d,%d], got %d", CONTAM_K_MIN, CONTAM_K_MAX, k); return TGSF_ERR_INVALID; }
    const double fd = (double)min_frac;
    const long long ppm = fd == fd && fd >= 0.0 && fd <= 2.0 ? llround(fd * 1e6) : -1;
    if (ppm < 1 || ppm > 1000000) { set_err("contaminant min_frac must give ppm in [1,1000000], got %g", fd); return TGSF_ERR_INVALID; }
    if (offsets[0] != 0) { set_err("contaminant offsets[0] must be 0"); return TGSF_ERR_INVALID; }
    for (uint32_t i = 0; i < n_seqs; ++i)
        if (offsets[i + 1] < offsets[i]) { set_err("contaminant offsets not ascending at %u", i); return TGSF_ERR_INVALID; }
    const u64 n_bytes = offsets[n_seqs];
    if (n_bytes < (u64)k || !seq) { set_err("contaminant set has no valid %d-mer", k); return TGSF_ERR_INVALID; }
    if (n_bytes > (1ull << 36)) { set_err("contaminant set of %llu bytes is too large", (unsigned long long)n_bytes); return TGSF_ERR_NOMEM; }
    CU(cudaSetDevice(c->device));
    // distinct keys <= windows < n_bytes, so a capacity >= 2 x n_bytes keeps the load <= 0.5
    u64 cap = 1024;
    while (cap < 2 * n_bytes) cap <<= 1;
    cudaStream_t st = c->slots[0].stream.get();
    ContamSet next;
    DBuf d_seq, d_off, d_cnt;
    TRY(next.table.ensure(cap * sizeof(u64)));
    if (labelled) {
        TRY(next.labels.ensure(cap * sizeof(u32)));
        CU(cudaMemsetAsync(next.labels.p, 0xFF, cap * sizeof(u32), st));
    }
    TRY(d_seq.ensure(n_bytes));
    TRY(d_off.ensure(((size_t)n_seqs + 1) * sizeof(u64)));
    TRY(d_cnt.ensure(sizeof(unsigned long long)));
    CU(cudaMemsetAsync(next.table.p, 0xFF, cap * sizeof(u64), st));
    CU(cudaMemsetAsync(d_cnt.p, 0, sizeof(unsigned long long), st));
    CU(cudaMemcpyAsync(d_seq.p, seq, n_bytes, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(d_off.p, offsets, ((size_t)n_seqs + 1) * sizeof(u64), cudaMemcpyHostToDevice, st));
    const u64 threads = (n_bytes + CONTAM_BUILD_SEG - 1) / CONTAM_BUILD_SEG;
    const u32 grid = (u32)std::min<u64>((threads + 255) / 256, (u64)c->sm_count * 16);
    if (labelled)
        k_contam_build<true><<<grid, 256, 0, st>>>(d_seq.as<uint8_t>(), d_off.as<u64>(), n_seqs, k, next.table.as<u64>(),
                                                   cap - 1, d_cnt.as<unsigned long long>(), next.labels.as<u32>());
    else
        k_contam_build<false><<<grid, 256, 0, st>>>(d_seq.as<uint8_t>(), d_off.as<u64>(), n_seqs, k, next.table.as<u64>(),
                                                    cap - 1, d_cnt.as<unsigned long long>(), nullptr);
    c->launches++;
    TRY(check_launch("k_contam_build"));
    unsigned long long n = 0;
    CU(cudaMemcpyAsync(&n, d_cnt.p, sizeof(n), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    next.n_keys = n;
    if (n == 0) { set_err("contaminant set has no valid %d-mer", k); return TGSF_ERR_INVALID; }
    if (n <= CONTAM_PF_MAX_KEYS) {
        TRY(next.pf_bits.ensure(CONTAM_PF_SMEM_BYTES));
        CU(cudaMemsetAsync(next.pf_bits.p, 0, CONTAM_PF_SMEM_BYTES, st));
        k_contam_bitmap<<<(u32)std::min<u64>(cap / 256 + 1, (u64)c->sm_count * 8), 256, 0, st>>>(
            next.table.as<u64>(), cap, next.pf_bits.as<u32>());
        c->launches++;
        TRY(check_launch("k_contam_bitmap"));
        CU(cudaStreamSynchronize(st));
    }
    std::vector<u64> rk;
    if (labelled) {
        const size_t rows = (size_t)n_seqs + 1;
        DBuf d_rk;
        TRY(d_rk.ensure(rows * sizeof(u64)));
        TRY(next.tally.ensure(2 * rows * sizeof(u64)));
        CU(cudaMemsetAsync(d_rk.p, 0, rows * sizeof(u64), st));
        CU(cudaMemsetAsync(next.tally.p, 0, next.tally.cap, st));
        k_contam_label_count<<<(u32)std::min<u64>(cap / 256, (u64)c->sm_count * 8), 256, 0, st>>>(
            next.table.as<u64>(), next.labels.as<u32>(), cap, n_seqs, d_rk.as<unsigned long long>());
        c->launches++;
        TRY(check_launch("k_contam_label_count"));
        rk.resize(rows);
        CU(cudaMemcpyAsync(rk.data(), d_rk.p, rows * sizeof(u64), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        next.n_records = n_seqs;
    }
    next.mask = cap - 1;
    next.ppm = (u64)ppm;
    next.k = k;
    c->contam = std::move(next); // frees the set it replaces
    *n_kmers = c->contam.n_keys;
    if (labelled) memcpy(record_kmers, rk.data(), rk.size() * sizeof(u64));
    return TGSF_OK;
}

int tgsf_set_contaminants(tgsf_ctx *c, const uint8_t *seq, const uint64_t *offsets, uint32_t n_seqs, int32_t k,
                          float min_frac, uint64_t *n_kmers) {
    return install_contaminants("tgsf_set_contaminants", c, seq, offsets, n_seqs, k, min_frac, n_kmers, nullptr);
}

int tgsf_set_contaminants_labelled(tgsf_ctx *c, const uint8_t *seq, const uint64_t *offsets, uint32_t n_seqs,
                                   int32_t k, float min_frac, uint64_t *n_kmers, uint64_t *record_kmers) {
    if (!record_kmers) { set_err("tgsf_set_contaminants_labelled: missing argument"); return TGSF_ERR_INVALID; }
    return install_contaminants("tgsf_set_contaminants_labelled", c, seq, offsets, n_seqs, k, min_frac, n_kmers,
                                record_kmers);
}

int tgsf_contam_record_stats(tgsf_ctx *c, uint64_t *reads, uint64_t *bases, uint32_t n) {
    if (!c || !reads || !bases) { set_err("tgsf_contam_record_stats: NULL argument"); return TGSF_ERR_INVALID; }
    if (!c->contam.labelled()) { set_err("tgsf_contam_record_stats: the installed contaminant set has no labels"); return TGSF_ERR_INVALID; }
    if ((u64)n != (u64)c->contam.n_records + 1) {
        set_err("tgsf_contam_record_stats: n must be n_seqs + 1 = %llu, got %u", (unsigned long long)c->contam.n_records + 1, n);
        return TGSF_ERR_INVALID;
    }
    if (c->outstanding) { set_err("collect all batches first"); return TGSF_ERR_STATE; }
    CU(cudaSetDevice(c->device));
    const u64 *T = c->contam.tally.as<u64>();
    CU(cudaMemcpy(reads, T, (size_t)n * sizeof(u64), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(bases, T + n, (size_t)n * sizeof(u64), cudaMemcpyDeviceToHost));
    return TGSF_OK;
}

int tgsf_contam_classify(tgsf_ctx *c, const uint8_t *seq, const uint64_t *offsets, uint32_t n, tgsf_contam_class *out) {
    if (!c) { set_err("tgsf_contam_classify: ctx is NULL"); return TGSF_ERR_INVALID; }
    if (c->outstanding) { set_err("tgsf_contam_classify with %u batch(es) outstanding", c->outstanding); return TGSF_ERR_STATE; }
    if (!c->contam.labelled()) { set_err("tgsf_contam_classify: no labelled contaminant set installed"); return TGSF_ERR_STATE; }
    if (n == 0) return TGSF_OK;
    if (!offsets || !out) { set_err("tgsf_contam_classify: NULL argument"); return TGSF_ERR_INVALID; }
    RecordPieces R;
    TRY(R.setup("tgsf_contam_classify", c->device, seq, offsets, n));
    Slot &s = R.slot();
    DBuf d_out;
    TRY(d_out.ensure((size_t)n * sizeof(int2)));
    CU(cudaMemsetAsync(d_out.p, 0xFF, (size_t)n * sizeof(int2), s.stream.get())); // record -1: not attributed
    TRY(launch_contam(R.c.get(), s, c->contam, d_out.as<int2>()));
    std::vector<tgsf_piece> pc((size_t)n);
    std::vector<int2> attr((size_t)n);
    CU(cudaMemcpyAsync(pc.data(), s.pieces.p, (size_t)n * sizeof(tgsf_piece), cudaMemcpyDeviceToHost, s.stream.get()));
    CU(cudaMemcpyAsync(attr.data(), d_out.p, (size_t)n * sizeof(int2), cudaMemcpyDeviceToHost, s.stream.get()));
    TRY(R.finish("tgsf_contam_classify"));
    for (uint32_t i = 0; i < n; ++i) {
        out[i].hits = pc[i].contam_hits;
        out[i].record = attr[i].x;
        out[i].record_hits = attr[i].x < 0 ? 0 : attr[i].y;
        out[i].contam = pc[i].status == TGSF_PIECE_CONTAM ? 1 : 0;
    }
    return TGSF_OK;
}

int tgsf_set_foldback(tgsf_ctx *c, int32_t enable) {
    if (!c) { set_err("tgsf_set_foldback: ctx is NULL"); return TGSF_ERR_INVALID; }
    if (enable != 0 && enable != 1) { set_err("tgsf_set_foldback: enable must be 0 or 1, got %d", enable); return TGSF_ERR_INVALID; }
    if (c->outstanding) { set_err("tgsf_set_foldback with %u batch(es) outstanding", c->outstanding); return TGSF_ERR_STATE; }
    if (enable && !c->fold_stats.p) {
        CU(cudaSetDevice(c->device));
        TRY(c->fold_stats.ensure(4 * sizeof(u64)));
        CU(cudaMemset(c->fold_stats.p, 0, 4 * sizeof(u64)));
    }
    c->foldback = enable != 0;
    return TGSF_OK;
}

int tgsf_foldback_stats(tgsf_ctx *c, uint64_t out[4]) {
    if (!c || !out) { set_err("tgsf_foldback_stats: NULL argument"); return TGSF_ERR_INVALID; }
    if (c->outstanding) { set_err("collect all batches first"); return TGSF_ERR_STATE; }
    if (!c->fold_stats.p) {
        memset(out, 0, 4 * sizeof(uint64_t));
        return TGSF_OK;
    }
    CU(cudaSetDevice(c->device));
    CU(cudaMemcpy(out, c->fold_stats.p, 4 * sizeof(u64), cudaMemcpyDeviceToHost));
    return TGSF_OK;
}

int tgsf_fold_detect(int device, const uint8_t *seq, const uint64_t *offsets, uint32_t n, tgsf_fold_result *out) {
    if (n == 0) return TGSF_OK;
    if (!offsets || !out) { set_err("tgsf_fold_detect: NULL argument"); return TGSF_ERR_INVALID; }
    RecordPieces R;
    TRY(R.setup("tgsf_fold_detect", device, seq, offsets, n));
    Slot &s = R.slot();
    DBuf d_out;
    TRY(d_out.ensure((size_t)n * sizeof(tgsf_fold_result)));
    DevHeader *H = s.header.as<DevHeader>();
    TRY(launch_fold(R.c.get(), s, s.pieces.as<tgsf_piece>(), &H->tmp_cursor, H, d_out.as<tgsf_fold_result>(),
                    (u32)R.longest));
    CU(cudaMemcpyAsync(out, d_out.p, (size_t)n * sizeof(tgsf_fold_result), cudaMemcpyDeviceToHost, s.stream.get()));
    return R.finish("tgsf_fold_detect");
}

int tgsf_set_dust(tgsf_ctx *c, int32_t level, float min_frac) {
    if (!c) { set_err("tgsf_set_dust: ctx is NULL"); return TGSF_ERR_INVALID; }
    if (level != 0 && (level < DUST_LEVEL_MIN || level > DUST_LEVEL_MAX)) {
        set_err("tgsf_set_dust: level must be 0 or in [%d,%d], got %d", DUST_LEVEL_MIN, DUST_LEVEL_MAX, level);
        return TGSF_ERR_INVALID;
    }
    const double fd = (double)min_frac;
    const long long ppm = fd == fd && fd >= 0.0 && fd <= 2.0 ? llround(fd * 1e6) : -1;
    if (level != 0 && (ppm < 1 || ppm > 1000000)) {
        set_err("tgsf_set_dust: min_frac must give ppm in [1,1000000], got %g", fd);
        return TGSF_ERR_INVALID;
    }
    if (c->outstanding) { set_err("tgsf_set_dust with %u batch(es) outstanding", c->outstanding); return TGSF_ERR_STATE; }
    c->dust_level = level;
    c->dust_ppm = level ? (u64)ppm : 0;
    return TGSF_OK;
}

int tgsf_dust_detect(int device, const uint8_t *seq, const uint64_t *offsets, uint32_t n, int32_t level,
                     uint32_t *masked) {
    if (level < DUST_LEVEL_MIN || level > DUST_LEVEL_MAX) {
        set_err("tgsf_dust_detect: level must be in [%d,%d], got %d", DUST_LEVEL_MIN, DUST_LEVEL_MAX, level);
        return TGSF_ERR_INVALID;
    }
    if (n == 0) return TGSF_OK;
    if (!offsets || !masked) { set_err("tgsf_dust_detect: NULL argument"); return TGSF_ERR_INVALID; }
    RecordPieces R;
    TRY(R.setup("tgsf_dust_detect", device, seq, offsets, n));
    Slot &s = R.slot();
    TRY(launch_dust(R.c.get(), s, level, 0));
    CU(cudaMemcpyAsync(masked, s.dust_masked.p, (size_t)n * sizeof(u32), cudaMemcpyDeviceToHost, s.stream.get()));
    return R.finish("tgsf_dust_detect");
}

int tgsf_device_count(int *count) {
    if (!count) return TGSF_ERR_INVALID;
    *count = 0;
    CU(cudaGetDeviceCount(count));
    return TGSF_OK;
}

int tgsf_host_alloc(void **ptr, size_t bytes) {
    if (!ptr) return TGSF_ERR_INVALID;
    CU(cudaHostAlloc(ptr, bytes ? bytes : 1, cudaHostAllocDefault));
    return TGSF_OK;
}
int tgsf_host_free(void *ptr) {
    if (ptr) CU(cudaFreeHost(ptr));
    return TGSF_OK;
}

// The per-100 bp tables are sized by the longest read the context has seen so far (the reference sizes them by
// every read's own length, T.cpp:1445): a batch with a longer read first moves the counter block to a larger layout.
// Only the four bin tables at the end of the block depend on the length; everything in front keeps its offset.
static int grow_counters_to(tgsf_ctx *c, u32 new_bins) { // exactly new_bins bins per table
    if (new_bins <= c->P.L.max_bins) return TGSF_OK;
    for (auto &s : c->slots) // batches in flight were launched on the old block
        if (s.busy) CU(cudaStreamSynchronize(s.stream.get()));
    const tgsf_counter_layout OL = c->P.L;
    tgsf_counter_layout NL;
    tgsf_make_layout(OL.bc_len, (int32_t)((u64)(new_bins - 1) * SCAN_BIN), &NL);
    DBuf nb;
    TRY(nb.ensure((size_t)NL.n_u64 * sizeof(u64)));
    CU(cudaMemset(nb.p, 0, (size_t)NL.n_u64 * sizeof(u64)));
    const u64 *o = c->counters.as<u64>();
    u64 *n = nb.as<u64>();
    CU(cudaMemcpy(n, o, (size_t)OL.raw_bin_cnt * sizeof(u64), cudaMemcpyDeviceToDevice));
    const u32 osec[4] = {OL.raw_bin_cnt, OL.raw_bin_qual, OL.clean_bin_cnt, OL.clean_bin_qual};
    const u32 nsec[4] = {NL.raw_bin_cnt, NL.raw_bin_qual, NL.clean_bin_cnt, NL.clean_bin_qual};
    for (int i = 0; i < 4; ++i)
        CU(cudaMemcpy(n + nsec[i], o + osec[i], (size_t)OL.max_bins * 5 * sizeof(u64), cudaMemcpyDeviceToDevice));
    c->counters = std::move(nb);
    c->P.L = NL;
    return TGSF_OK;
}
static int grow_counters(tgsf_ctx *c, u64 longest) { // room for a read of `longest` bases (+ 25 % slack when growing)
    if (longest / SCAN_BIN + 1 <= (u64)c->P.L.max_bins) return TGSF_OK;
    if (longest > 0x7fffffffull) { set_err("a read of %llu bases is longer than 2^31 - 1", (unsigned long long)longest); return TGSF_ERR_INVALID; }
    return grow_counters_to(c, (u32)(std::min<u64>(longest + longest / 4 + 1024, 0x7fffffffull) / SCAN_BIN + 1));
}

struct PackedIn { // optional 2-bit input of tgsf_submit_packed
    const uint8_t *packed = nullptr;
    const u64 *exc_pos = nullptr;
    const uint8_t *exc_val = nullptr;
    u64 n_exc = 0;
};

static int submit_common(tgsf_ctx *c, const uint8_t *bases, const uint8_t *quals, const u64 *offsets,
                         u32 n_reads, u64 n_bases, bool on_device, const PackedIn *pk = nullptr) {
    if (!c) { set_err("ctx is NULL"); return TGSF_ERR_INVALID; }
    if (n_reads && ((!bases && !pk) || !offsets)) { set_err("bases/offsets NULL"); return TGSF_ERR_INVALID; }
    if (n_reads > (1u << 24)) { set_err("more than 2^24 reads in one batch"); return TGSF_ERR_INVALID; }
    if (c->outstanding == c->slots.size()) { set_err("all %zu slots busy: collect first", c->slots.size()); return TGSF_ERR_STATE; }
    CU(cudaSetDevice(c->device));
    if (!on_device && n_reads) { // host offsets: make room for the longest read of this batch before anything is launched
        u64 longest = 0;
        for (u32 i = 0; i < n_reads; ++i) longest = std::max<u64>(longest, offsets[i + 1] - offsets[i]);
        TRY(grow_counters(c, longest));
    }
    Slot &s = c->slots[c->head];
    s.has_qual = quals != nullptr;
    s.n_bases = n_bases;
    TRY(slot_reserve(c, s, n_reads, n_bases));
    CU(cudaEventRecord(s.ev_start.get(), s.stream.get()));
    if (on_device) {
        if (((uintptr_t)bases & 15) || ((uintptr_t)quals & 15)) { set_err("device streams must be 16-byte aligned"); return TGSF_ERR_INVALID; }
        s.B.bases = bases;
        s.B.quals = quals;
        s.B.offsets = offsets;
    } else {
        const size_t pad = 64;
        TRY(s.in_bases.ensure((size_t)n_bases + pad));
        TRY(s.in_offsets.ensure(((size_t)n_reads + 1) * sizeof(u64)));
        if (pk) {
            const u64 n_words = (n_bases + 15) / 16; // u32 words of packed input = 16 bases each
            TRY(s.in_bases.ensure((size_t)n_words * 16 + pad));
            TRY(s.in_packed.ensure((size_t)n_words * 4 + pad));
            if (n_bases) {
                // the unpack kernel reads whole 32-bit words: define the bytes of the last word beyond the copy
                CU(cudaMemsetAsync((uint8_t *)s.in_packed.p + (n_words - 1) * 4, 0, 4, s.stream.get()));
                CU(cudaMemcpyAsync(s.in_packed.p, pk->packed, (size_t)((n_bases + 3) / 4), cudaMemcpyHostToDevice, s.stream.get()));
                k_unpack_bases<<<c->sm_count * 8, 256, 0, s.stream.get()>>>(s.in_packed.as<u32>(), n_words, s.in_bases.as<uint4>());
                c->launches++;
            }
            if (pk->n_exc) {
                TRY(s.in_exc_pos.ensure((size_t)pk->n_exc * sizeof(u64)));
                TRY(s.in_exc_val.ensure((size_t)pk->n_exc));
                CU(cudaMemcpyAsync(s.in_exc_pos.p, pk->exc_pos, (size_t)pk->n_exc * sizeof(u64), cudaMemcpyHostToDevice, s.stream.get()));
                CU(cudaMemcpyAsync(s.in_exc_val.p, pk->exc_val, (size_t)pk->n_exc, cudaMemcpyHostToDevice, s.stream.get()));
                k_apply_exceptions<<<c->sm_count, 256, 0, s.stream.get()>>>(s.in_bases.as<uint8_t>(), s.in_exc_pos.as<u64>(),
                                                                           s.in_exc_val.as<uint8_t>(), pk->n_exc);
                c->launches++;
            }
        } else if (n_bases) {
            CU(cudaMemcpyAsync(s.in_bases.p, bases, (size_t)n_bases, cudaMemcpyHostToDevice, s.stream.get()));
        }
        if (quals) {
            TRY(s.in_quals.ensure((size_t)n_bases + pad));
            if (n_bases) CU(cudaMemcpyAsync(s.in_quals.p, quals, (size_t)n_bases, cudaMemcpyHostToDevice, s.stream.get()));
        }
        if (n_reads) CU(cudaMemcpyAsync(s.in_offsets.p, offsets, ((size_t)n_reads + 1) * sizeof(u64), cudaMemcpyHostToDevice, s.stream.get()));
        s.B.bases = s.in_bases.as<uint8_t>();
        s.B.quals = quals ? s.in_quals.as<uint8_t>() : nullptr;
        s.B.offsets = s.in_offsets.as<u64>();
    }
    s.B.n_reads = n_reads;
    CU(cudaEventRecord(s.ev_k0.get(), s.stream.get()));
    TRY(run_pipeline(c, s));
    s.busy = true;
    c->head = (c->head + 1) % (u32)c->slots.size();
    c->outstanding++;
    return TGSF_OK;
}

int tgsf_submit(tgsf_ctx *c, const uint8_t *bases, const uint8_t *quals, const uint64_t *offsets, uint32_t n_reads) {
    if (n_reads && !offsets) { set_err("offsets NULL"); return TGSF_ERR_INVALID; }
    const u64 n_bases = n_reads ? offsets[n_reads] : 0;
    return submit_common(c, bases, quals, (const u64 *)offsets, n_reads, n_bases, false);
}

int tgsf_submit_packed(tgsf_ctx *c, const uint8_t *packed_bases, const uint8_t *quals, const uint64_t *offsets,
                       uint32_t n_reads, const uint64_t *exc_pos, const uint8_t *exc_byte, uint64_t n_exc) {
    if (n_reads && (!offsets || !packed_bases)) { set_err("packed/offsets NULL"); return TGSF_ERR_INVALID; }
    if (n_exc && (!exc_pos || !exc_byte)) { set_err("exception arrays NULL"); return TGSF_ERR_INVALID; }
    const u64 n_bases = n_reads ? offsets[n_reads] : 0;
    for (u64 i = 0; i < n_exc; ++i)
        if (exc_pos[i] >= n_bases) { set_err("exception position out of range"); return TGSF_ERR_INVALID; }
    PackedIn pk;
    pk.packed = packed_bases;
    pk.exc_pos = (const u64 *)exc_pos;
    pk.exc_val = exc_byte;
    pk.n_exc = n_exc;
    return submit_common(c, nullptr, quals, (const u64 *)offsets, n_reads, n_bases, false, &pk);
}

extern "C" int tgsf_pack_has_avx2();
extern "C" uint64_t tgsf_pack_groups_avx2(const uint8_t *bases, uint8_t *packed, uint64_t g0, uint64_t n_groups);

int tgsf_pack_bases(const uint8_t *bases, uint64_t n, uint8_t *packed, uint64_t *exc_pos, uint8_t *exc_byte,
                    uint64_t exc_cap, uint64_t *n_exc) {
    if ((n && (!bases || !packed)) || !n_exc) { set_err("pack: NULL argument"); return TGSF_ERR_INVALID; }
    static const struct Lut { uint8_t code[256]; Lut() { memset(code, 4, 256); code['A'] = 0; code['C'] = 1; code['G'] = 2; code['T'] = 3; } } lut;
    u64 ne = 0;
    const u64 full = n / 4;
    static const bool avx2 = tgsf_pack_has_avx2() != 0;
    const u64 groups = avx2 ? n / 32 : 0; // 32 bases = 8 packed bytes per AVX2 step (pack_host.cpp)
    auto scalar_word = [&](u64 i) {
        const uint8_t c0 = lut.code[bases[4 * i]], c1 = lut.code[bases[4 * i + 1]], c2 = lut.code[bases[4 * i + 2]],
                      c3 = lut.code[bases[4 * i + 3]];
        if ((c0 | c1 | c2 | c3) & 4) { // rare: at least one byte is not upper-case ACGT
            uint8_t v = 0;
            for (int j = 0; j < 4; ++j) {
                const uint8_t cj = lut.code[bases[4 * i + j]];
                if (cj & 4) {
                    if (exc_pos && ne < exc_cap) { exc_pos[ne] = 4 * i + j; exc_byte[ne] = bases[4 * i + j]; }
                    ++ne;
                } else {
                    v |= (uint8_t)(cj << (2 * j));
                }
            }
            packed[i] = v;
        } else {
            packed[i] = (uint8_t)(c0 | (c1 << 2) | (c2 << 4) | (c3 << 6));
        }
    };
    u64 i = 0;
    while (i < full) {
        if ((i & 7) == 0 && (i >> 3) < groups) {
            const u64 g = tgsf_pack_groups_avx2(bases, packed, i >> 3, groups);
            i = g << 3;
            if (g < groups) { // group g holds an exception byte: its 8 words go through the scalar path
                for (int w = 0; w < 8; ++w) scalar_word(i + (u64)w);
                i += 8;
            }
            continue;
        }
        scalar_word(i++);
    }
    if (n & 3) {
        uint8_t v = 0;
        for (u64 j = 0; j < (n & 3); ++j) {
            const uint8_t cj = lut.code[bases[4 * full + j]];
            if (cj & 4) {
                if (exc_pos && ne < exc_cap) { exc_pos[ne] = 4 * full + j; exc_byte[ne] = bases[4 * full + j]; }
                ++ne;
            } else {
                v |= (uint8_t)(cj << (2 * j));
            }
        }
        packed[full] = v;
    }
    *n_exc = ne;
    if (ne > exc_cap) { set_err("pack: %llu exceptions, capacity %llu", (unsigned long long)ne, (unsigned long long)exc_cap); return TGSF_ERR_CAPACITY; }
    return TGSF_OK;
}

int tgsf_submit_device(tgsf_ctx *c, const uint8_t *d_bases, const uint8_t *d_quals, const uint64_t *d_offsets,
                       uint32_t n_reads, uint64_t n_bases) {
    return submit_common(c, d_bases, d_quals, (const u64 *)d_offsets, n_reads, n_bases, true);
}

int tgsf_collect_gz(tgsf_ctx *c, uint8_t *blob, uint64_t blob_cap, uint64_t *blob_bytes, tgsf_gz_span *spans,
                    uint32_t spans_cap, uint32_t *n_spans) {
    if (!c || !blob_bytes || !n_spans) { set_err("collect_gz: NULL argument"); return TGSF_ERR_INVALID; }
    if (!(c->P.flags & TGSF_FLAG_GZ_BLOCKS)) { set_err("context was created without TGSF_FLAG_GZ_BLOCKS"); return TGSF_ERR_STATE; }
    if (c->outstanding == 0) { set_err("nothing outstanding"); return TGSF_ERR_STATE; }
    CU(cudaSetDevice(c->device));
    Slot &s = c->slots[c->tail];
    CU(cudaEventSynchronize(s.ev_end.get()));
    const DevHeader *H = (const DevHeader *)s.h_header.p;
    if (H->status == DEV_STATUS_POOL_OVERFLOW) { // the tail has to be re-run first: tgsf_collect does that
        set_err("collect_gz: this batch overflowed the region pool; tgsf_collect re-runs it, compress its records on the host");
        return TGSF_ERR_STATE;
    }
    if (H->gz_overflow) { set_err("deflate blob overflow"); return TGSF_ERR_CUDA; }
    const u32 np = H->tmp_cursor;
    *blob_bytes = (uint64_t)H->gz_cursor;
    *n_spans = np;
    if (H->gz_cursor > blob_cap || np > spans_cap) { set_err("collect_gz: buffers too small"); return TGSF_ERR_CAPACITY; }
    if (H->gz_cursor) CU(cudaMemcpyAsync(blob, s.gz_blob.p, (size_t)H->gz_cursor, cudaMemcpyDeviceToHost, s.stream.get()));
    if (np) CU(cudaMemcpyAsync(spans, s.gz_spans.p, (size_t)np * sizeof(tgsf_gz_span), cudaMemcpyDeviceToHost, s.stream.get()));
    CU(cudaStreamSynchronize(s.stream.get()));
    return TGSF_OK;
}

int tgsf_collect(tgsf_ctx *c, tgsf_read_result *reads, uint32_t n_reads, tgsf_piece *pieces, uint32_t pieces_cap,
                 uint32_t *n_pieces) {
    if (!c) { set_err("ctx is NULL"); return TGSF_ERR_INVALID; }
    if (c->outstanding == 0) { set_err("nothing outstanding"); return TGSF_ERR_STATE; }
    CU(cudaSetDevice(c->device));
    Slot &s = c->slots[c->tail];
    CU(cudaEventSynchronize(s.ev_end.get()));
    DevHeader *H = (DevHeader *)s.h_header.p;
    float extra_ms = 0;
    int guard = 0;
    while (H->status == DEV_STATUS_POOL_OVERFLOW && guard++ < 8) {
        // grow the region pool to what k_mid_count asked for and re-run the tail
        u32 need = 0;
        CU(cudaMemcpy(&need, s.mid_off.as<u32>() + (size_t)s.B.n_reads * std::max(c->P.n_adapters, 1), sizeof(u32),
                      cudaMemcpyDeviceToHost));
        s.pool_cap = std::max(need + need / 4 + 1024, s.pool_cap * 2);
        TRY(slot_reserve(c, s, s.B.n_reads, s.n_bases));
        CU(cudaMemsetAsync(s.header.p, 0, sizeof(DevHeader), s.stream.get()));
        Event e0, e1;
        TRY(create(e0));
        TRY(create(e1));
        CU(cudaEventRecord(e0.get(), s.stream.get()));
        TRY(launch_tail(c, s));
        CU(cudaEventRecord(e1.get(), s.stream.get()));
        TRY(enqueue_d2h(c, s));
        CU(cudaStreamSynchronize(s.stream.get()));
        float ms = 0;
        cudaEventElapsedTime(&ms, e0.get(), e1.get());
        extra_ms += ms;
    }
    float k_ms = 0, t_ms = 0;
    cudaEventElapsedTime(&k_ms, s.ev_k0.get(), s.ev_k1.get());
    cudaEventElapsedTime(&t_ms, s.ev_start.get(), s.ev_end.get());
    c->last_kernel_ms = k_ms + extra_ms;
    c->last_total_ms = t_ms + extra_ms;
    cudaEventElapsedTime(&c->last_span_start, c->ev_epoch.get(), s.ev_k0.get());
    cudaEventElapsedTime(&c->last_span_end, c->ev_epoch.get(), s.ev_k1.get());
    c->last_span_end += extra_ms;
    for (int i = 0; i < TGSF_N_STAGES; ++i) {
        float ms = 0;
        cudaEventElapsedTime(&ms, s.ev_stage[i].get(), s.ev_stage[i + 1].get());
        c->last_stage_ms[i] = ms;
    }
    c->last_chunk_shift = s.chunk_shift;
    c->last_run_shift = s.run_shift;

    auto retire = [&]() {
        s.busy = false;
        c->tail = (c->tail + 1) % (u32)c->slots.size();
        c->outstanding--;
    };
    if (H->status == DEV_STATUS_BIN_OVERFLOW) {
        retire();
        set_err("a read is longer than max_read_len allows (per-100 bp bins)");
        return TGSF_ERR_CAPACITY;
    }
    if (H->status == DEV_STATUS_HASH_OVERFLOW) {
        retire();
        set_err("%s", HASH_OVERFLOW_MSG);
        return TGSF_ERR_CAPACITY;
    }
    if (H->status != DEV_STATUS_OK) {
        retire();
        set_err("device status %u", H->status);
        return TGSF_ERR_CUDA;
    }
    const u32 total = H->tmp_cursor;
    if (n_pieces) *n_pieces = total;
    if (reads) {
        if (n_reads < s.B.n_reads) { set_err("reads array too small"); return TGSF_ERR_CAPACITY; }
        memcpy(reads, s.h_res.p, (size_t)s.B.n_reads * sizeof(tgsf_read_result));
    }
    if (pieces) {
        if (pieces_cap < total) { set_err("pieces array too small: need %u", total); return TGSF_ERR_CAPACITY; }
        const u32 have = std::min(total, s.h_pieces_copied);
        memcpy(pieces, s.h_pieces.p, (size_t)have * sizeof(tgsf_piece));
        if (total > have)
            CU(cudaMemcpy(pieces + have, s.pieces.as<tgsf_piece>() + have, (size_t)(total - have) * sizeof(tgsf_piece),
                          cudaMemcpyDeviceToHost));
    }
    retire();
    return TGSF_OK;
}

int tgsf_last_timing(tgsf_ctx *c, float *kernel_ms, float *total_ms) {
    if (!c) return TGSF_ERR_INVALID;
    if (kernel_ms) *kernel_ms = c->last_kernel_ms;
    if (total_ms) *total_ms = c->last_total_ms;
    return TGSF_OK;
}

int tgsf_last_span(tgsf_ctx *c, float *start_ms, float *end_ms) {
    if (!c) return TGSF_ERR_INVALID;
    if (start_ms) *start_ms = c->last_span_start;
    if (end_ms) *end_ms = c->last_span_end;
    return TGSF_OK;
}

int tgsf_last_stage_ms(tgsf_ctx *c, float *out, int n) {
    if (!c || !out) return TGSF_ERR_INVALID;
    for (int i = 0; i < n && i < TGSF_N_STAGES; ++i) out[i] = c->last_stage_ms[i];
    return TGSF_OK;
}

int tgsf_counter_layout_get(const tgsf_ctx *c, tgsf_counter_layout *out) {
    if (!c || !out) return TGSF_ERR_INVALID;
    *out = c->P.L;
    return TGSF_OK;
}

int tgsf_counters(tgsf_ctx *c, uint64_t *out, uint32_t n_u64) {
    if (!c || !out) return TGSF_ERR_INVALID;
    if (c->outstanding) { set_err("collect all batches first"); return TGSF_ERR_STATE; }
    if (n_u64 < c->P.L.n_u64) { set_err("counter array too small"); return TGSF_ERR_CAPACITY; }
    CU(cudaSetDevice(c->device));
    CU(cudaMemcpy(out, c->counters.p, (size_t)c->P.L.n_u64 * sizeof(u64), cudaMemcpyDeviceToHost));
    return TGSF_OK;
}

int tgsf_counters_reset(tgsf_ctx *c) {
    if (!c) return TGSF_ERR_INVALID;
    if (c->outstanding) { set_err("collect all batches first"); return TGSF_ERR_STATE; }
    CU(cudaSetDevice(c->device));
    CU(cudaMemset(c->counters.p, 0, (size_t)c->P.L.n_u64 * sizeof(u64)));
    if (c->fold_stats.p) CU(cudaMemset(c->fold_stats.p, 0, 4 * sizeof(u64)));
    if (c->contam.labelled()) CU(cudaMemset(c->contam.tally.p, 0, c->contam.tally.cap));
    return TGSF_OK;
}

int tgsf_counters_device(tgsf_ctx *c, void **d_ptr, uint32_t *n_u64) {
    if (!c || !d_ptr) return TGSF_ERR_INVALID;
    *d_ptr = c->counters.p;
    if (n_u64) *n_u64 = c->P.L.n_u64;
    return TGSF_OK;
}

uint64_t tgsf_launch_count(const tgsf_ctx *c) { return c ? c->launches : 0; }

int tgsf_launch_shape(const tgsf_ctx *c, int32_t *sm_count, int32_t *last_chunk_shift) {
    if (!c) { set_err("ctx is NULL"); return TGSF_ERR_INVALID; }
    if (sm_count) *sm_count = c->sm_count;
    if (last_chunk_shift) *last_chunk_shift = c->last_chunk_shift;
    return TGSF_OK;
}

int tgsf_mid_run_shift(const tgsf_ctx *c, int32_t *last_run_shift) {
    if (!c) { set_err("ctx is NULL"); return TGSF_ERR_INVALID; }
    if (last_run_shift) *last_run_shift = c->last_run_shift;
    return TGSF_OK;
}


int tgsf_allreduce(tgsf_ctx **ctxs, int n) {
    if (!ctxs || n <= 0) { set_err("allreduce: no contexts"); return TGSF_ERR_INVALID; }
    for (int i = 0; i < n; ++i) {
        if (!ctxs[i]) { set_err("allreduce: NULL context"); return TGSF_ERR_INVALID; }
        if (ctxs[i]->outstanding) { set_err("allreduce: collect all batches first"); return TGSF_ERR_STATE; }
        if (ctxs[i]->P.L.bc_len != ctxs[0]->P.L.bc_len) { set_err("allreduce: counter layouts differ"); return TGSF_ERR_INVALID; }
    }
    u32 bins = 0; // contexts that met longer reads have grown their bin tables: bring all to the largest layout
    for (int i = 0; i < n; ++i) bins = std::max(bins, ctxs[i]->P.L.max_bins);
    for (int i = 0; i < n; ++i)
        if (ctxs[i]->P.L.max_bins < bins) {
            CU(cudaSetDevice(ctxs[i]->device));
            TRY(grow_counters_to(ctxs[i], bins));
        }
    if (n == 1) return TGSF_OK;
    tgsf_ctx *root = ctxs[0];
    const u32 words = root->P.L.n_u64;
    const size_t bytes = (size_t)words * sizeof(u64);
    CU(cudaSetDevice(root->device));
    for (int i = 1; i < n; ++i) { // direct NVLink path where the topology allows it
        int can = 0;
        if (cudaDeviceCanAccessPeer(&can, root->device, ctxs[i]->device) == cudaSuccess && can) {
            cudaError_t e = cudaDeviceEnablePeerAccess(ctxs[i]->device, 0);
            if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) { /* staged copy still works */ }
            cudaGetLastError();
        }
    }
    DBuf scratch;
    TRY(scratch.ensure(bytes));
    for (int i = 1; i < n; ++i) {
        CU(cudaMemcpyPeer(scratch.p, root->device, ctxs[i]->counters.p, ctxs[i]->device, bytes));
        k_add_u64<<<root->sm_count, 256>>>(root->counters.as<u64>(), scratch.as<u64>(), words);
        root->launches++;
        CU(cudaDeviceSynchronize());
    }
    for (int i = 1; i < n; ++i)
        CU(cudaMemcpyPeer(ctxs[i]->counters.p, ctxs[i]->device, root->counters.p, root->device, bytes));
    return TGSF_OK;
}

int tgsf_prepass(int device, const uint8_t *ends5p, const uint8_t *ends3p, uint32_t n, uint32_t row_len,
                 const uint8_t *const *lib_seq, const int32_t *lib_len, int32_t n_lib, float min_sim,
                 int32_t *bases_num5p, int32_t *bases_num3p, int64_t *map5p, int64_t *map3p) {
    if (!ends5p || !ends3p || !bases_num5p || !bases_num3p || row_len == 0) {
        set_err("prepass: bad arguments");
        return TGSF_ERR_INVALID;
    }
    if (lib_seq && (n_lib <= 0 || n_lib > 1024 || !lib_len || !map5p || !map3p)) { set_err("prepass: bad library"); return TGSF_ERR_INVALID; }
    for (int32_t a = 0; lib_seq && a < n_lib; ++a)
        if (!lib_seq[a] || lib_len[a] <= 0 || lib_len[a] > TGSF_MAX_ADAPTER_LEN) {
            set_err("prepass: library adapter %d: length %d outside [1, %d]", a, lib_len[a], TGSF_MAX_ADAPTER_LEN);
            return TGSF_ERR_INVALID;
        }
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    const int sms = prop.multiProcessorCount;
    DBuf d_rows, d_cnt;
    const size_t row_bytes = (size_t)n * row_len;
    TRY(d_rows.ensure(2 * row_bytes + 64));
    TRY(d_cnt.ensure((size_t)2 * row_len * 4 * sizeof(int)));
    uint8_t *r5 = d_rows.as<uint8_t>(), *r3 = r5 + row_bytes;
    if (row_bytes) {
        CU(cudaMemcpy(r5, ends5p, row_bytes, cudaMemcpyHostToDevice));
        CU(cudaMemcpy(r3, ends3p, row_bytes, cudaMemcpyHostToDevice));
    }
    CU(cudaMemset(d_cnt.p, 0, (size_t)2 * row_len * 4 * sizeof(int)));
    int *c5 = d_cnt.as<int>(), *c3 = c5 + (size_t)row_len * 4;
    if (n) {
        // column tiles on y; about 4 CTAs per SM in all, so the flush of the per-CTA tables does not grow with row_len
        const u32 tiles = cdiv(row_len, PRE_TILE_COLS);
        const dim3 grid(std::max<u32>(1, std::min<u32>(cdiv((u64)sms * 4, tiles), cdiv(n, PRE_THREADS / 32))), tiles);
        const size_t smem = (size_t)std::min<u32>(row_len, PRE_TILE_COLS) * 4 * sizeof(u32);
        k_base_content<<<grid, PRE_THREADS, smem>>>(r5, n, row_len, c5);
        k_base_content<<<grid, PRE_THREADS, smem>>>(r3, n, row_len, c3);
        TRY(check_launch("k_base_content"));
    }
    if (lib_seq) {
        AdapterSet ads;
        DBuf d_maps;
        Scratch scratch;
        TRY(ads.build(lib_seq, lib_len, n_lib));
        if (min_sim < 0.9) min_sim = 0.9; // T.cpp:1151-1154 (float compared against a double literal)
        for (auto &A : ads.host) {
            int minK = static_cast<int>((1 - min_sim) * A.qlen) + 1; // T.cpp:1161
            A.k_end = std::min(minK, A.qlen - 1);
        }
        TRY(ads.upload());
        TRY(d_maps.ensure((size_t)2 * n_lib * sizeof(long long)));
        TRY(scratch.ensure(ads.host, sms * 4, RES_THREADS));
        CU(cudaMemset(d_maps.p, 0, (size_t)2 * n_lib * sizeof(long long)));
        long long *m5 = d_maps.as<long long>(), *m3 = m5 + n_lib;
        const AdapterCtx AC = ads.ctx();
        for (int a = 0; a < n_lib && n; ++a) {
            const DevAdapter &Ah = ads.host[(size_t)a];
            const int grid_a = Scratch::grid_for(sms * 4, RES_THREADS, 2 * Ah.qlen + 2, Ah.nw);
            const u64 stride_a = (u64)grid_a * RES_THREADS;
            TRY(for_nw(Ah.nw, [&](auto nwc) {
                constexpr int NW = decltype(nwc)::value;
                k_lib_search<NW><<<grid_a, RES_THREADS>>>(r5, n, row_len, AC, a, m5 + a, scratch.buf.as<u64>(), stride_a);
                k_lib_search<NW><<<grid_a, RES_THREADS>>>(r3, n, row_len, AC, a, m3 + a, scratch.buf.as<u64>(), stride_a);
                return check_launch("k_lib_search");
            }));
        }
        CU(cudaMemcpy(map5p, m5, (size_t)n_lib * sizeof(long long), cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(map3p, m3, (size_t)n_lib * sizeof(long long), cudaMemcpyDeviceToHost));
    }
    CU(cudaMemcpy(bases_num5p, c5, (size_t)row_len * 4 * sizeof(int), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(bases_num3p, c3, (size_t)row_len * 4 * sizeof(int), cudaMemcpyDeviceToHost));
    return TGSF_OK;
}

int tgsf_end_kmer_counts(int device, const uint8_t *rows, uint32_t n, uint32_t row_len, int32_t k, uint32_t split,
                         uint32_t *outer, uint32_t *inner) {
    if (k < 1 || k > 13) { set_err("end_kmer_counts: k must be in [1,13], got %d", k); return TGSF_ERR_INVALID; }
    if (n > 0 && (!rows || !outer || !inner)) { set_err("end_kmer_counts: NULL argument"); return TGSF_ERR_INVALID; }
    const u64 windows = row_len >= (u32)k ? (u64)row_len - k + 1 : 0;
    if ((u64)n * windows >= (1ull << 32)) { set_err("end_kmer_counts: 2^32 windows or more"); return TGSF_ERR_INVALID; }
    const size_t table_bytes = ((size_t)1 << (2 * k)) * sizeof(u32);
    if (n == 0 || windows == 0) {
        if (outer) memset(outer, 0, table_bytes);
        if (inner) memset(inner, 0, table_bytes);
        return TGSF_OK;
    }
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    DBuf d_rows, d_table;
    const size_t row_bytes = (size_t)n * row_len;
    TRY(d_rows.ensure(row_bytes));
    TRY(d_table.ensure(table_bytes));
    CU(cudaMemcpy(d_rows.p, rows, row_bytes, cudaMemcpyHostToDevice));
    // one band per launch into one table: at k = 12 a band's table (64 MB) stays resident in the 126 MB L2, where the
    // two bands' tables together would not
    const u32 grid = std::max<u32>(1, std::min<u32>(cdiv(n, PRE_THREADS / 32), (u32)prop.multiProcessorCount * 8));
    const u32 cut = (u32)std::min<u64>(split, windows);
    const u32 bands[2][2] = {{0, cut}, {cut, (u32)windows}};
    uint32_t *out[2] = {outer, inner};
    for (int b = 0; b < 2; ++b) {
        CU(cudaMemset(d_table.p, 0, table_bytes));
        if (bands[b][1] > bands[b][0]) {
            k_end_kmers<<<grid, PRE_THREADS>>>(d_rows.as<uint8_t>(), n, row_len, k, bands[b][0], bands[b][1],
                                               d_table.as<u32>());
            TRY(check_launch("k_end_kmers"));
        }
        CU(cudaMemcpy(out[b], d_table.p, table_bytes, cudaMemcpyDeviceToHost));
    }
    return TGSF_OK;
}

int tgsf_align_hw(int device, const uint8_t *queries, const uint32_t *q_off, const uint8_t *targets,
                  const uint32_t *t_off, const int32_t *k, uint32_t n, tgsf_align_result *out) {
    if (!q_off || !t_off || !k || !out) { set_err("align: NULL argument"); return TGSF_ERR_INVALID; }
    if (n == 0) return TGSF_OK;
    if (n > (1u << 20)) { set_err("align: at most 2^20 pairs per call"); return TGSF_ERR_INVALID; }
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    const int sms = prop.multiProcessorCount;
    std::vector<const uint8_t *> seqs(n);
    std::vector<int32_t> lens(n);
    for (u32 i = 0; i < n; ++i) {
        seqs[i] = queries + q_off[i];
        lens[i] = (int32_t)(q_off[i + 1] - q_off[i]);
        if (lens[i] > TGSF_MAX_ADAPTER_LEN) { set_err("align: query %u longer than %d", i, TGSF_MAX_ADAPTER_LEN); return TGSF_ERR_INVALID; }
    }
    AdapterSet ads;
    DBuf d_t, d_toff, d_k, d_out;
    Scratch scratch;
    TRY(ads.build(seqs.data(), lens.data(), (int)n));
    for (u32 i = 0; i < n; ++i)
        if (lens[i] == 0 || t_off[i + 1] == t_off[i]) ads.host[i].nw = 0; // handled on the host below
    TRY(ads.upload());
    const size_t tbytes = t_off[n];
    TRY(d_t.ensure(tbytes + 64));
    TRY(d_toff.ensure(((size_t)n + 1) * sizeof(u32)));
    TRY(d_k.ensure((size_t)n * sizeof(int)));
    TRY(d_out.ensure((size_t)n * sizeof(tgsf_align_result)));
    TRY(scratch.ensure(ads.host, sms * 2, RES_THREADS));
    if (tbytes) CU(cudaMemcpy(d_t.p, targets, tbytes, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_toff.p, t_off, ((size_t)n + 1) * sizeof(u32), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_k.p, k, (size_t)n * sizeof(int), cudaMemcpyHostToDevice));
    CU(cudaMemset(d_out.p, 0, (size_t)n * sizeof(tgsf_align_result)));
    const AdapterCtx AC = ads.ctx();
    for (int nw : {1, 2, 3, 4, 8, 16, 32}) {
        int max_q = 0;
        for (u32 i = 0; i < n; ++i)
            if (ads.host[i].nw == nw) max_q = std::max(max_q, ads.host[i].qlen);
        if (max_q == 0) continue;
        const int grid_nw = Scratch::grid_for(sms * 2, RES_THREADS, 2 * max_q + 2, nw);
        TRY(for_nw(nw, [&](auto nwc) {
            constexpr int NW = decltype(nwc)::value;
            k_align_pairs<NW><<<grid_nw, RES_THREADS>>>(d_t.as<uint8_t>(), d_toff.as<u32>(), d_k.as<int>(), AC, n, NW,
                                                        d_out.as<tgsf_align_result>(), scratch.buf.as<u64>(),
                                                        (u64)grid_nw * RES_THREADS);
            return check_launch("k_align_pairs");
        }));
    }
    CU(cudaMemcpy(out, d_out.p, (size_t)n * sizeof(tgsf_align_result), cudaMemcpyDeviceToHost));
    for (u32 i = 0; i < n; ++i) {
        if (lens[i] == 0 || t_off[i + 1] == t_off[i]) { // E.cpp:161-179
            tgsf_align_result R;
            memset(&R, 0, sizeof(R));
            R.edit_distance = lens[i];
            R.n_locations = 1;
            R.first_end = R.last_end = -1;
            u32 h = 2166136261u;
            const u32 v[2] = {0u, (u32)-1};
            for (int w = 0; w < 2; ++w)
                for (int b = 0; b < 4; ++b) { h ^= (v[w] >> (8 * b)) & 0xffu; h *= 16777619u; }
            R.loc_hash = h;
            out[i] = R;
        }
    }
    return TGSF_OK;
}

}  // extern "C"
