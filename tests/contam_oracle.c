/*
 * contam_oracle.c — CPU restatement of the contaminant screen (tgsf_set_contaminants).  TEST INFRASTRUCTURE ONLY,
 * built by tests/contam_oracle.py into a temporary directory.
 *
 * The per-read path is the pinned oracle itself: this file includes oracle/tgsf_oracle.c unchanged and runs
 * tgsfo_run.  The screen sits between the repeat check and the clean-side step of the piece loop, so a piece it
 * marks as a contaminant must not have reached the clean step.  tgsfo_run_contam therefore screens every piece that
 * the repeat check kept (status EMIT or LOWQ after tgsfo_run) and, for each contaminant, replays that piece's clean
 * step (tgsf_oracle.c, the `if (!dropped)` branch of tgsfo_run) into a zeroed block and subtracts it: the result is
 * the counter block of a loop that dropped the piece before the clean step.
 *
 * Set semantics: every canonical k-mer (min of forward and reverse-complement code, A0 C1 G2 T3, 2 bits per base)
 * of every record; acgt counts as ACGT; a window with any other byte contributes nothing.  The set is a sorted
 * array searched with bsearch.
 */
#include <math.h>

#include "../oracle/tgsf_oracle.c"

static int contam_code(uint8_t b) {
    switch (b) {
        case 'A': case 'a': return 0;
        case 'C': case 'c': return 1;
        case 'G': case 'g': return 2;
        case 'T': case 't': return 3;
        default: return -1;
    }
}

/* Canonical k-mer of seq[0, k), or UINT64_MAX when a byte is not ACGT/acgt. */
static uint64_t contam_key(const uint8_t *seq, int k) {
    uint64_t fwd = 0, rev = 0;
    for (int i = 0; i < k; i++) {
        int c = contam_code(seq[i]);
        if (c < 0) return UINT64_MAX;
        fwd = (fwd << 2) | (uint64_t)c;
        rev |= (uint64_t)(3 - c) << (2 * i);
    }
    return fwd < rev ? fwd : rev;
}

/* Sorted distinct canonical k-mers of the records seq[offs[i], offs[i+1]) (malloc'ed). */
static uint64_t *contam_keys(const uint8_t *seq, const uint64_t *offs, uint32_t n_seqs, int k, uint64_t *n_out) {
    uint64_t n = 0;
    uint64_t *v = (uint64_t *)malloc(sizeof(uint64_t) * (size_t)(offs[n_seqs] + 1));
    for (uint32_t r = 0; r < n_seqs; r++)
        for (uint64_t i = offs[r]; i + (uint64_t)k <= offs[r + 1]; i++) {
            uint64_t key = contam_key(seq + i, k);
            if (key != UINT64_MAX) v[n++] = key;
        }
    qsort(v, (size_t)n, sizeof(uint64_t), compare_u64);
    uint64_t d = 0;
    for (uint64_t i = 0; i < n; i++)
        if (d == 0 || v[i] != v[d - 1]) v[d++] = v[i];
    *n_out = d;
    return v;
}

/* Distinct canonical k-mers of a contaminant set (tgsf_set_contaminants' *n_kmers). */
uint64_t tgsfo_contam_kmers(const uint8_t *seq, const uint64_t *offs, uint32_t n_seqs, int k) {
    uint64_t n = 0;
    free(contam_keys(seq, offs, n_seqs, k, &n));
    return n;
}

/* Windows of seq[0, len) whose canonical k-mer is in keys[0, n_keys). */
static int contam_hits(const uint8_t *seq, int len, int k, const uint64_t *keys, uint64_t n_keys) {
    int hits = 0;
    for (int i = 0; i + k <= len; i++) {
        uint64_t key = contam_key(seq + i, k);
        if (key != UINT64_MAX && bsearch(&key, keys, (size_t)n_keys, sizeof(uint64_t), compare_u64)) hits++;
    }
    return hits;
}

/* What the clean step of tgsfo_run added to the counters for one piece (same calls, into D). */
static void clean_step(const tgsf_params *p, const tgsf_counter_layout *L, const uint8_t *cs, const uint8_t *cq,
                       int len, uint64_t *D) {
    if (cq) {
        uint64_t sumQ = calc_sum_quality(cs, cq, len, p->qtype, D + L->clean_bin_qual, D + L->clean_bin_cnt);
        double cleanQuality = (double)sumQ / (double)(uint64_t)len;
        if ((p->flags & TGSF_FLAG_FILTER) && (cleanQuality < p->min_q || cleanQuality > p->max_q)) {
            D[L->drop_info + 13]++;
            D[L->drop_info + 14] += (uint64_t)len;
        } else {
            D[L->clean_hist + qual_hist_index(cleanQuality)] += (uint64_t)len;
            ends_base_qual(cs, cq, len, p->bc_len, p->qtype, D + L->clean5p_qual, D + L->clean5p_cnt,
                           D + L->clean3p_qual, D + L->clean3p_cnt);
        }
    } else {
        fasta_counts(cs, len, p->bc_len, D + L->clean_bin_cnt, D + L->clean5p_cnt, D + L->clean3p_cnt);
    }
}

/* tgsfo_run with the contaminant set seq[coffs[i], coffs[i+1]), i < n_cseqs, installed. */
int tgsfo_run_contam(const tgsf_params *p, const uint8_t *bases, const uint8_t *quals,
                     const uint64_t *offsets, uint32_t n_reads, tgsf_read_result *reads,
                     tgsf_piece *pieces, uint32_t pieces_cap, uint32_t *n_pieces_out, uint64_t *C,
                     const uint8_t *cseq, const uint64_t *coffs, uint32_t n_cseqs, int ck, float min_frac) {
    long long q = llround((double)min_frac * 1e6);
    if (n_cseqs == 0 || ck < 11 || ck > 31 || q < 1 || q > 1000000) return TGSF_ERR_INVALID;
    const uint64_t ppm = (uint64_t)q;
    tgsf_counter_layout L;
    tgsf_make_layout(p->bc_len, p->max_read_len, &L);
    uint32_t np = 0;
    int rc = tgsfo_run(p, bases, quals, offsets, n_reads, reads, pieces, pieces_cap, &np, C);
    if (n_pieces_out) *n_pieces_out = np;
    if (rc != TGSF_OK) return rc;
    uint64_t n_keys = 0;
    uint64_t *keys = contam_keys(cseq, coffs, n_cseqs, ck, &n_keys);
    if (n_keys == 0) { free(keys); return TGSF_ERR_INVALID; }
    uint64_t *D = (uint64_t *)malloc(sizeof(uint64_t) * L.n_u64);
    for (uint32_t i = 0; i < np; i++) {
        tgsf_piece *P = &pieces[i];
        if (P->status != TGSF_PIECE_EMIT && P->status != TGSF_PIECE_LOWQ) continue; /* kept by the repeat check */
        const uint8_t *cs = bases + offsets[P->read] + P->start;
        const uint8_t *cq = quals ? quals + offsets[P->read] + P->start : NULL;
        P->contam_hits = contam_hits(cs, P->len, ck, keys, n_keys);
        uint64_t windows = P->len >= ck ? (uint64_t)(P->len - ck + 1) : 0;
        if (windows >= 1 && (uint64_t)P->contam_hits * 1000000ull >= ppm * windows) {
            memset(D, 0, sizeof(uint64_t) * L.n_u64);
            clean_step(p, &L, cs, cq, P->len, D);
            for (uint32_t w = 0; w < L.n_u64; w++) C[w] -= D[w];
            P->status = TGSF_PIECE_CONTAM;
            P->sum_q = 0;
        }
    }
    free(D);
    free(keys);
    return TGSF_OK;
}
