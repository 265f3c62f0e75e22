/*
 * libtgsf_cuda — C-ABI of the B200-native per-read filter/trim hot path of TGSFilter.
 *
 * The reference (HuiyangYu/TGSFilter v1.11, src/TGSFilter.cpp = "T.cpp") has no FFI seam; the seam
 * this library replaces is "one worker iteration" of TGSFilterTask::filter_sequence
 * (T.cpp:1939-2061) plus the two pre-pass bodies GetFilterParameterTask::CheckBaseContent /
 * adapterSearch (T.cpp:1079-1209).  Every entry point cites what it replaces.
 *
 * Conventions: C linkage, int status return (TGSF_OK == 0), never throws, never writes to
 * stdout/stderr.  The caller owns all host buffers; the library owns all device memory.  One
 * context per GPU; a context is single-threaded; different contexts may be driven from different
 * host threads / processes.  The same structs are produced by the CPU oracle (oracle/tgsf_oracle.c,
 * test infrastructure only) so the parity tests compare them field by field.
 */
#ifndef TGSF_H_
#define TGSF_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TGSF_OK 0
#define TGSF_ERR_INVALID 1  /* bad argument / parameter combination */
#define TGSF_ERR_CUDA 2     /* a CUDA runtime call failed; see tgsf_last_error() */
#define TGSF_ERR_NOMEM 3
#define TGSF_ERR_STATE 4    /* submit with all slots busy, collect with nothing outstanding */
#define TGSF_ERR_CAPACITY 5 /* caller's output array too small; required size is reported */

#define TGSF_DROPINFO_N 17      /* DropInfo[17], T.cpp:1776, index meaning T.cpp:3216-3230 */
#define TGSF_QUAL_HIST_N 256    /* raw/cleanDiffQualReadsBases[256], T.cpp:1777-1778 */
#define TGSF_MAX_ADAPTERS 65536 /* size of the global `adapters` set (T.cpp:1324) we accept; the work arrays grow with it */
#define TGSF_MAX_ADAPTER_LEN 2048 /* 32 x 64-bit Myers words (1-4 words: exact count in registers; longer: 8, 16 or 32) */
#define TGSF_LIB_ADAPTERS 22    /* adapterLib, T.cpp:2969-2991 */

/* tgsf_params.flags */
#define TGSF_FLAG_FILTER 1u      /* Para_A24::Filter  (T.cpp:115, cleared by -F / --qc) */
#define TGSF_FLAG_ONLY_QC 2u     /* Para_A24::OnlyQC  (T.cpp:119) */
#define TGSF_FLAG_DISCARD_MID 4u /* Para_A24::discard (-D, T.cpp:108) */
#define TGSF_FLAG_GZ_BLOCKS 8u   /* also deflate-encode every emitted piece on the GPU (tgsf_collect_gz) */
#define TGSF_FLAG_GZ_FASTA 16u   /* ... as FASTA records (bases only), like -f / FASTA input */

/* All thresholds consumed by the per-read path: the subset of Para_A24 (T.cpp:82-172) that
 * filter_sequence/adapterMap/GetEditDistance read, after the pre-pass has resolved qType, MinQ,
 * HeadTrim/TailTrim and the adapter set (T.cpp:3058-3126). */
typedef struct tgsf_params {
    int32_t min_len;        /* -l MinLen */
    int32_t max_len;        /* -L MaxLen */
    float min_q;            /* -q MinQ  (float, compared against the fp64 mean, T.cpp:1947) */
    float max_q;            /* -Q MaxQ */
    int32_t bc_len;         /* -e BCLen: number of 5'/3' QC positions (T.cpp:1490) */
    int32_t head_trim;      /* resolved -5 HeadTrim (<=0: none, T.cpp:1334) */
    int32_t tail_trim;      /* resolved -3 TailTrim */
    int32_t end_len;        /* -E EndLen */
    int32_t end_match_len;  /* -m EndMatchLen (constructor default 4, T.cpp:148) */
    int32_t mid_match_len;  /* -M MidMatchLen */
    int32_t extra_len;      /* -T ExtraLen */
    float end_sim;          /* -s EndSim  (already defaulted per read type, T.cpp:449-457) */
    float mid_sim;          /* -S MidSim */
    int32_t kmer;           /* -k Kmer */
    int32_t min_repeat;     /* -p MinRepeat (0: k-mer stage off) */
    int32_t qtype;          /* 33 or 64: global qType (T.cpp:80), 0 when there are no qualities */
    uint32_t flags;         /* TGSF_FLAG_* */
    int32_t n_adapters;     /* size of the global adapter set (both strands already inserted) */
    const uint8_t *const *adapter_seq; /* n_adapters byte strings (compared byte-wise like edlib) */
    const int32_t *adapter_len;
    int32_t max_read_len;   /* INITIAL capacity of the per-100 bp QC bins (0 -> 4 Mi bases); tgsf_submit / tgsf_submit_packed
                             * grow the counter block when a batch brings a longer read (ask tgsf_counter_layout_get again
                             * before tgsf_counters); tgsf_submit_device cannot see the lengths: size it up front there */
    int32_t n_slots;        /* batches in flight (1..4); 0 -> 2 */
} tgsf_params;

/* One per input read, index-aligned with the submitted batch. */
typedef struct tgsf_read_result {
    uint64_t sum_q;      /* sum(qual - qType) over the read: numerator of CalcAvgQuality (T.cpp:1451-1478) */
    int32_t status;      /* TGSF_READ_* */
    int32_t n_mid;       /* adapterMap's numMid / num5p / num3p (T.cpp:1329-1352) */
    int32_t n_5p;
    int32_t n_3p;
    int32_t piece_begin; /* first entry of this read in the pieces array */
    int32_t n_pieces;    /* keepRegions.size() (T.cpp:1960-1965) */
} tgsf_read_result;

#define TGSF_READ_EVALUATED 0 /* went through adapterMap (or Filter off) */
#define TGSF_READ_LOWQ 1      /* mean quality outside [MinQ,MaxQ]: DropInfo[0]/[1] (T.cpp:1946-1952) */
#define TGSF_READ_EMPTY 2     /* zero-length read, skipped by `if (rawSeqLen > 0)` (T.cpp:1939) */

/* One per keepRegion (T.cpp:1976-2059), ordered by (read, start): exactly the order the reference
 * worker emits records for one read; the n-th emitted piece (status OK) of a read gets the
 * ":n" name suffix for n >= 2 (newSeqName, T.cpp:1680-1701, 2011-2017). */
typedef struct tgsf_piece {
    uint64_t sum_q;     /* numerator of the piece's CalcAvgQuality (0 if not evaluated) */
    int32_t read;       /* index of the read in the batch */
    int32_t start;      /* keepRegion {start,len} */
    int32_t len;
    int32_t repeat_len; /* GetKmerCount result (T.cpp:1703-1753), -1 when MinRepeat == 0 */
    int32_t status;     /* TGSF_PIECE_* */
    int32_t contam_hits; /* windows whose canonical k-mer is in the contaminant set (tgsf_set_contaminants);
                          * 0 without a set and for pieces that are not screened */
} tgsf_piece;

#define TGSF_PIECE_EMIT 0         /* becomes an output record */
#define TGSF_PIECE_SHORT_REPEAT 1 /* DropInfo[15]/[16] (T.cpp:1982-1989) */
#define TGSF_PIECE_LOWQ 2         /* DropInfo[13]/[14] (T.cpp:1995-2000) */
#define TGSF_PIECE_QC_ONLY 3      /* --qc: region kept but nothing emitted (T.cpp:1976) */
#define TGSF_PIECE_CONTAM 4       /* contaminant screen: hit share >= min_frac (tgsf_set_contaminants) */

/* Layout (in uint64 words) of the cumulative counter block.  Every member is a sum, so blocks of
 * different GPUs combine with one allreduce(sum, u64).  [x][5] = {A,T,G,C,all} as in T.cpp:1462-1476. */
typedef struct tgsf_counter_layout {
    uint32_t n_u64;        /* total words */
    uint32_t bc_len;       /* rows of the 5p/3p tables */
    uint32_t max_bins;     /* rows of the per-100 bp tables */
    uint32_t drop_info;    /* [17] */
    uint32_t raw_hist;     /* [256]  rawDiffQualReadsBases */
    uint32_t clean_hist;   /* [256]  cleanDiffQualReadsBases */
    uint32_t raw5p_cnt;    /* [bc_len][5] raw5pBaseCounts */
    uint32_t raw5p_qual;   /* [bc_len][5] raw5pBaseQual */
    uint32_t raw3p_cnt;
    uint32_t raw3p_qual;
    uint32_t clean5p_cnt;
    uint32_t clean5p_qual;
    uint32_t clean3p_cnt;
    uint32_t clean3p_qual;
    uint32_t raw_bin_cnt;  /* [max_bins][5] rawBaseCounts */
    uint32_t raw_bin_qual; /* [max_bins][5] rawBaseQual */
    uint32_t clean_bin_cnt;
    uint32_t clean_bin_qual;
} tgsf_counter_layout;

typedef struct tgsf_ctx tgsf_ctx;

/* Library / build identification; never fails.  "sm_100a" is part of the string. */
const char *tgsf_version(void);
/* Text of the last CUDA / argument error seen by this thread. */
const char *tgsf_last_error(void);

/* Replaces: construction of TGSFilterTask + the globals qType/adapters (T.cpp:80,1324,1757-1790).
 * Copies params and adapters; precomputes the Myers Peq tables and the integer thresholds that
 * stand in for the float comparisons of GetEditDistance (T.cpp:1250,1267,1287). */
int tgsf_create(int device, const tgsf_params *params, tgsf_ctx **out);
int tgsf_destroy(tgsf_ctx *ctx);

/* Number of CUDA devices this process can use (0 and TGSF_ERR_CUDA without a driver / device).  The
 * host uses it to validate --gpus and, in the tests, to place several contexts on one device. */
int tgsf_device_count(int *count);

/* Pinned host memory for batch buffers (the packer of T.cpp:1845-1916's replacement fills these). */
int tgsf_host_alloc(void **ptr, size_t bytes);
int tgsf_host_free(void *ptr);

/* Replaces: N iterations of the filter_sequence loop body (T.cpp:1939-2061) for a batch of reads.
 * bases/quals: concatenated bytes, read i = [offsets[i], offsets[i+1]); quals == NULL for FASTA /
 * quality-less input (T.cpp:1954-1958).  Host buffers; the H2D copy, all kernels and the D2H copy
 * of the results are enqueued on the slot's stream and the call returns without waiting. */
int tgsf_submit(tgsf_ctx *ctx, const uint8_t *bases, const uint8_t *quals, const uint64_t *offsets,
                uint32_t n_reads);
/* Same, with the bases 2-bit packed on the host (A0 C1 G2 T3; base i in bits 2*(i%4) of byte i/4,
 * packing runs over the concatenated stream) — 1.25 instead of 2 bytes per base over PCIe.  Every
 * byte that is not upper-case ACGT is listed in (exc_pos, exc_byte) and patched in on the device,
 * so the kernels see exactly the bytes the host parsed.  tgsf_pack_bases is the host-side packer
 * (CPU, allocation-free; returns TGSF_ERR_CAPACITY with *n_exc = required entries). */
int tgsf_submit_packed(tgsf_ctx *ctx, const uint8_t *packed_bases, const uint8_t *quals, const uint64_t *offsets,
                       uint32_t n_reads, const uint64_t *exc_pos, const uint8_t *exc_byte, uint64_t n_exc);
int tgsf_pack_bases(const uint8_t *bases, uint64_t n, uint8_t *packed, uint64_t *exc_pos, uint8_t *exc_byte,
                    uint64_t exc_cap, uint64_t *n_exc);
/* Same, with the three arrays already resident in this GPU's memory (device pointers). */
int tgsf_submit_device(tgsf_ctx *ctx, const uint8_t *d_bases, const uint8_t *d_quals,
                       const uint64_t *d_offsets, uint32_t n_reads, uint64_t n_bases);
/* Deflate blocks of the emitted pieces of the OLDEST outstanding batch (contexts created with
 * TGSF_FLAG_GZ_BLOCKS; replaces the compression half of DeflateCompress, T.cpp:786-812).  Must be called
 * before tgsf_collect for that batch.  spans[i] describes piece i of the batch (same order as tgsf_collect's
 * pieces; bytes == 0 for pieces that are not emitted): blob[offset, offset + bytes) holds, byte aligned,
 * the dynamic-Huffman blocks of bases + "\n+\n" + qualities + "\n" (FASTA: bases + "\n"), the last one
 * final.  A gzip member of the record is: 10-byte gzip header, a non-final stored block with the header
 * line ("@name\n"), these bytes, CRC-32 and ISIZE of the whole record.  blob_cap too small:
 * TGSF_ERR_CAPACITY with *blob_bytes = required size. */
typedef struct tgsf_gz_span {
    uint64_t offset;
    uint32_t bytes;
    uint32_t reserved;
} tgsf_gz_span;
int tgsf_collect_gz(tgsf_ctx *ctx, uint8_t *blob, uint64_t blob_cap, uint64_t *blob_bytes, tgsf_gz_span *spans,
                    uint32_t spans_cap, uint32_t *n_spans);
/* Waits for the oldest outstanding batch and copies its results out.  reads: n_reads entries;
 * pieces: up to pieces_cap entries, *n_pieces receives the number produced (TGSF_ERR_CAPACITY and
 * no copy if it exceeds pieces_cap; call again with a larger array).  reads/pieces may be NULL to
 * only retire the batch (counters are still updated). */
int tgsf_collect(tgsf_ctx *ctx, tgsf_read_result *reads, uint32_t n_reads, tgsf_piece *pieces,
                 uint32_t pieces_cap, uint32_t *n_pieces);
/* Contaminant screen (an extension; the reference has none).  Installs on this context's device the set of every
 * canonical k-mer (min of forward and reverse-complement code, A0 C1 G2 T3, 2 bits per base) of the records
 * seq[offsets[i], offsets[i+1]), i < n_seqs (host buffers, offsets[0] == 0).  Bases are case-insensitive; a window
 * with any other byte contributes nothing.  From the next batch on, every piece that is still TGSF_PIECE_EMIT after
 * the repeat check (not with TGSF_FLAG_ONLY_QC) is screened: windows = len - k + 1, contam_hits = valid windows
 * whose k-mer is in the set, and the piece becomes TGSF_PIECE_CONTAM iff windows >= 1 and
 * contam_hits * 1000000 >= ppm * windows (u64), ppm = llround((double)min_frac * 1e6).  Contaminant pieces touch no
 * counter; callers count them from the piece array.  k in [11, 31], ppm in [1, 1000000], otherwise TGSF_ERR_INVALID,
 * as for a set without a valid k-mer; TGSF_ERR_STATE while a batch is outstanding; TGSF_ERR_NOMEM when the table
 * (8 bytes x the next power of two >= 2 x set bytes) does not fit.  *n_kmers receives the number of distinct
 * canonical k-mers.  A second call replaces the set; on error the previous set stays installed.  The screen's
 * kernels are timed in TGSF_STAGE_KMER. */
int tgsf_set_contaminants(tgsf_ctx *ctx, const uint8_t *seq, const uint64_t *offsets, uint32_t n_seqs, int32_t k,
                          float min_frac, uint64_t *n_kmers);

/* Device time (ms, CUDA events on the slot's stream) of the batch retired by the last collect:
 * kernels only, and H2D+kernels+D2H. */
int tgsf_last_timing(tgsf_ctx *ctx, float *kernel_ms, float *total_ms);

/* Device time (ms) of each pipeline stage of the batch retired by the last collect, measured with
 * CUDA events on the slot's stream (bench.py's per-kernel roofline comes from here). */
#define TGSF_N_STAGES 7
#define TGSF_STAGE_RAW_SCAN 0    /* K1 over the reads (tile table + k_scan_tiles) */
#define TGSF_STAGE_RAW_FINAL 1   /* quality band, histogram, raw 5'/3' tables */
#define TGSF_STAGE_MID_SCAN 2    /* K3 k_mid_scan, all adapters (chunk table included) */
#define TGSF_STAGE_RESOLVE 3     /* K3 k_mid_count + k_ends (start search, traceback, thresholds) */
#define TGSF_STAGE_REGIONS 4     /* K3 k_mid_emit + K5 regions / piece compaction */
#define TGSF_STAGE_KMER 5        /* K4 + the contaminant screen */
#define TGSF_STAGE_CLEAN 6       /* K1 over the kept pieces + clean decisions + clean 5'/3' */
int tgsf_last_stage_ms(tgsf_ctx *ctx, float *out, int n);

/* Device-clock interval of the batch retired by the last tgsf_collect, in ms since the context was
 * created: [start_ms, end_ms] brackets its kernels (not the copies).  Batches in different slots run
 * on different streams and may overlap on the GPU, so the device time of a group of batches is
 * max(end) - min(start), not the sum of tgsf_last_timing (bench.py measures a step this way). */
int tgsf_last_span(tgsf_ctx *ctx, float *start_ms, float *end_ms);

/* Replaces: the per-thread accumulators of TGSFilterTask and their merge (T.cpp:1796-1806,
 * 3208-3213).  Cumulative since create / the last reset.  All batches must have been collected. */
int tgsf_counter_layout_get(const tgsf_ctx *ctx, tgsf_counter_layout *out);
int tgsf_counters(tgsf_ctx *ctx, uint64_t *out, uint32_t n_u64);
int tgsf_counters_reset(tgsf_ctx *ctx);
/* Device address of the counter block (n_u64 words) for an in-place NCCL allreduce(sum). */
int tgsf_counters_device(tgsf_ctx *ctx, void **d_ptr, uint32_t *n_u64);
/* Single-process multi-GPU: sums the counter blocks of n contexts (one per GPU) over peer copies
 * (NVLink where peer access is available) and leaves the total in every context.  Replaces the
 * per-thread merge loop T.cpp:3208-3213 across devices.  Multi-process jobs use an NCCL allreduce
 * on tgsf_counters_device instead (bench.py). */
int tgsf_allreduce(tgsf_ctx **ctxs, int n);
/* Number of kernels launched by this context since create (bench.py's gpu_launches). */
uint64_t tgsf_launch_count(const tgsf_ctx *ctx);
/* The SM count every grid of this context is sized by (the device's, or TGSF_SM_COUNT=n at create,
 * clamped to [1, device SM count]) and the middle-scan chunk shift (log2 of the chunk length in
 * bases, chosen per batch from its size and that SM count) of the last collected batch (0 before
 * the first).  Lets tests check which launch regime a batch ran in. */
int tgsf_launch_shape(const tgsf_ctx *ctx, int32_t *sm_count, int32_t *last_chunk_shift);
/* log2 of the number of chunks per middle-scan run (the scan restarts a halo once per run) of the last collected
 * batch, chosen per batch like the chunk shift (0 before the first). */
int tgsf_mid_run_shift(const tgsf_ctx *ctx, int32_t *last_run_shift);

/* Replaces: the compute of the pre-pass, CheckBaseContent's counting loop (T.cpp:1080-1095) and
 * adapterSearch's edlib loop (T.cpp:1156-1176), for both read ends.  ends5p / ends3p: n rows of
 * row_len bytes (seq[0:checkLen] and revcomp(seq[-checkLen:]), T.cpp:966-969).  Outputs:
 * bases_num5p/3p [row_len][4] int32 in A,T,G,C order; map5p/3p [n_lib] int64 = sum of
 * (alignmentLength - editDistance) over the rows where the library adapter aligned with
 * k = int((1-minSim)*qLen)+1.  lib == NULL skips the adapter search (AdapterFile given).  Any row_len >= 1;
 * 1 <= n_lib <= 1024 and library adapters of 1..TGSF_MAX_ADAPTER_LEN bases, otherwise TGSF_ERR_INVALID before
 * the device is touched. */
int tgsf_prepass(int device, const uint8_t *ends5p, const uint8_t *ends3p, uint32_t n,
                 uint32_t row_len, const uint8_t *const *lib_seq, const int32_t *lib_len,
                 int32_t n_lib, float min_sim, int32_t *bases_num5p, int32_t *bases_num3p,
                 int64_t *map5p, int64_t *map3p);

/* Extension (no counterpart in v1.11): k-mer counts of sampled read ends for the de novo adapter assembly
 * (--adapter-denovo).  rows: n rows of row_len bytes (ends5p or ends3p of tgsf_prepass).  Window j of a row is
 * row[j, j+k), never wrapped, and counts only when its k bytes are all upper-case A/C/G/T; its code is 2 bits per
 * base, A0 C1 G2 T3, first base most significant.  outer[x] / inner[x] ([4^k] u32 each) count the valid windows of
 * k-mer x with j < split / j >= split.  k in [1, 13]; NULL rows, outer or inner with n > 0, or n x max(0,
 * row_len - k + 1) >= 2^32, give TGSF_ERR_INVALID before the device is touched.  n = 0 (or no window) zeroes the
 * tables without touching the device. */
int tgsf_end_kmer_counts(int device, const uint8_t *rows, uint32_t n, uint32_t row_len, int32_t k, uint32_t split,
                         uint32_t *outer, uint32_t *inner);

/* Stand-alone adapter alignment with edlib semantics (EDLIB_MODE_HW + EDLIB_TASK_PATH,
 * include/edlib.cpp:141-296) for n independent (query, target) pairs: the unit the parity tests
 * pin against edlib's known answers.  Pair i: query = queries + q_off[i] .. q_off[i+1], likewise
 * targets.  Outputs per pair: edit_distance (-1: none <= k), n_locations, align_len
 * (alignmentLength of the first location), first_start/first_end/last_start/last_end, and
 * loc_hash = FNV-1a over all (start,end) pairs so that every location is pinned. */
typedef struct tgsf_align_result {
    int32_t edit_distance;
    int32_t n_locations;
    int32_t align_len;
    int32_t first_start, first_end, last_start, last_end;
    uint32_t loc_hash;
} tgsf_align_result;
int tgsf_align_hw(int device, const uint8_t *queries, const uint32_t *q_off, const uint8_t *targets,
                  const uint32_t *t_off, const int32_t *k, uint32_t n, tgsf_align_result *out);

#ifdef __cplusplus
}
#endif
#endif /* TGSF_H_ */
