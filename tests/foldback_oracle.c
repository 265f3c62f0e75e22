/*
 * foldback_oracle.c — CPU restatement of the fold-back screen (tgsf_set_foldback).  TEST INFRASTRUCTURE ONLY, built by
 * tests/foldback_oracle.py into a temporary directory.
 *
 * The per-read path is the pinned oracle (through contam_oracle.c, which includes oracle/tgsf_oracle.c unchanged):
 * tgsfo_run_foldback runs tgsfo_run, then for every piece that is not QC-only it detects a fold on the original
 * piece.  If there is one, it takes that piece's tail (the short-repeat counters, or the clean step) back out of the
 * counters, cuts the piece, and replays the tail on the kept arm: the repeat check, the optional contaminant screen,
 * then the clean step.  A piece without a fold only goes through the optional contaminant screen, as in
 * tgsfo_run_contam.
 *
 * Detection: every sampled window is listed as (key, o, position) and the list is sorted by key; a key is an anchor
 * when its group is exactly one o = 0 and one o = 1 entry.  The constants are restated here on purpose.
 */
#include "contam_oracle.c"

#define FO_K 15
#define FO_SAMPLE_MASK 7u
#define FO_BIN_SHIFT 7
#define FO_MIN_ANCHORS 8
#define FO_MAX_GAP 500
#define FO_DENSITY 400

typedef struct { int32_t fold, anchors, centre, min_gap; } fo_result;
typedef struct { uint32_t key, o, pos; } fo_sample;

static uint32_t fo_fmix32(uint32_t h) {
    h ^= h >> 16;
    h *= 0x85ebca6bu;
    h ^= h >> 13;
    h *= 0xc2b2ae35u;
    h ^= h >> 16;
    return h;
}

static int fo_cmp(const void *a, const void *b) {
    const fo_sample *x = (const fo_sample *)a, *y = (const fo_sample *)b;
    if (x->key != y->key) return x->key < y->key ? -1 : 1;
    if (x->o != y->o) return x->o < y->o ? -1 : 1;
    return x->pos < y->pos ? -1 : x->pos > y->pos;
}

void tgsfo_fold_detect(const uint8_t *s, int32_t L, fo_result *r) {
    r->fold = -1;
    r->anchors = 0;
    r->centre = -1;
    r->min_gap = -1;
    if (L < FO_K) return;
    fo_sample *v = (fo_sample *)malloc(sizeof(fo_sample) * (size_t)(L - FO_K + 1));
    size_t n = 0;
    for (int32_t i = 0; i + FO_K <= L; i++) {
        uint64_t f = 0, rc = 0;
        int ok = 1;
        for (int j = 0; j < FO_K && ok; j++) {
            int c = contam_code(s[i + j]);
            if (c < 0) { ok = 0; break; }
            f = (f << 2) | (uint64_t)c;
            rc |= (uint64_t)(3 - c) << (2 * j);
        }
        if (!ok) continue;
        uint32_t key = (uint32_t)(f < rc ? f : rc);
        if (fo_fmix32(key) & FO_SAMPLE_MASK) continue;
        v[n].key = key;
        v[n].o = f < rc ? 0u : 1u;
        v[n].pos = (uint32_t)i;
        n++;
    }
    qsort(v, n, sizeof(fo_sample), fo_cmp);
    const uint32_t nb = ((2u * (uint32_t)L - FO_K) >> FO_BIN_SHIFT) + 2u;
    uint32_t *cnt = (uint32_t *)calloc(nb, sizeof(uint32_t));
    uint64_t *sum = (uint64_t *)calloc(nb, sizeof(uint64_t));
    int32_t *ming = (int32_t *)malloc(sizeof(int32_t) * nb);
    for (uint32_t b = 0; b < nb; b++) ming[b] = INT32_MAX;
    for (size_t i = 0; i < n;) {
        size_t j = i;
        while (j < n && v[j].key == v[i].key) j++;
        if (j - i == 2 && v[i].o == 0 && v[i + 1].o == 1) {
            uint32_t p0 = v[i].pos, p1 = v[i + 1].pos;
            uint32_t d = p0 + p1 + FO_K;
            int32_t g = (int32_t)(p1 > p0 ? p1 - p0 : p0 - p1) - FO_K;
            uint32_t b = d >> FO_BIN_SHIFT;
            cnt[b]++;
            sum[b] += d;
            if (g < ming[b]) ming[b] = g;
        }
        i = j;
    }
    uint32_t best = 0, bb = 0;
    for (uint32_t b = 0; b + 1 < nb; b++)
        if (cnt[b] + cnt[b + 1] > best) { best = cnt[b] + cnt[b + 1]; bb = b; }
    if (best > 0) {
        uint64_t c = (sum[bb] + sum[bb + 1]) / (2ull * best);
        int32_t g = ming[bb] < ming[bb + 1] ? ming[bb] : ming[bb + 1];
        uint64_t shorter = c < (uint64_t)L - c ? c : (uint64_t)L - c;
        r->anchors = (int32_t)best;
        r->centre = (int32_t)c;
        r->min_gap = g;
        if (best >= FO_MIN_ANCHORS && g <= FO_MAX_GAP && (uint64_t)FO_DENSITY * best >= shorter && c > 0 && c < (uint64_t)L)
            r->fold = (int32_t)c;
    }
    free(v);
    free(cnt);
    free(sum);
    free(ming);
}

/* tgsfo_run with the fold-back screen on and, when n_cseqs > 0, the contaminant set seq[coffs[i], coffs[i+1])
 * installed.  stats: {pieces cut, bases removed, pieces dropped as TGSF_PIECE_FOLDBACK, their kept-arm bases}. */
int tgsfo_run_foldback(const tgsf_params *p, const uint8_t *bases, const uint8_t *quals, const uint64_t *offsets,
                       uint32_t n_reads, tgsf_read_result *reads, tgsf_piece *pieces, uint32_t pieces_cap,
                       uint32_t *n_pieces_out, uint64_t *C, uint64_t *stats, const uint8_t *cseq,
                       const uint64_t *coffs, uint32_t n_cseqs, int ck, float min_frac) {
    uint64_t *keys = NULL, n_keys = 0, ppm = 0;
    if (n_cseqs > 0) {
        long long q = llround((double)min_frac * 1e6);
        if (ck < 11 || ck > 31 || q < 1 || q > 1000000) return TGSF_ERR_INVALID;
        ppm = (uint64_t)q;
        keys = contam_keys(cseq, coffs, n_cseqs, ck, &n_keys);
        if (n_keys == 0) { free(keys); return TGSF_ERR_INVALID; }
    }
    tgsf_counter_layout L;
    tgsf_make_layout(p->bc_len, p->max_read_len, &L);
    uint64_t *DropInfo = C + L.drop_info;
    uint32_t np = 0;
    int rc = tgsfo_run(p, bases, quals, offsets, n_reads, reads, pieces, pieces_cap, &np, C);
    if (n_pieces_out) *n_pieces_out = np;
    if (rc != TGSF_OK) { free(keys); return rc; }
    memset(stats, 0, 4 * sizeof(uint64_t));
    uint64_t *D = (uint64_t *)malloc(sizeof(uint64_t) * L.n_u64);
    for (uint32_t i = 0; i < np; i++) {
        tgsf_piece *P = &pieces[i];
        if (P->status == TGSF_PIECE_QC_ONLY) continue;
        const uint8_t *seq = bases + offsets[P->read];
        const uint8_t *qual = quals ? quals + offsets[P->read] : NULL;
        fo_result fr;
        tgsfo_fold_detect(seq + P->start, P->len, &fr);
        int dropped = 0;
        if (fr.fold >= 0) {
            /* take the tail of the uncut piece back out */
            if (P->status == TGSF_PIECE_SHORT_REPEAT) {
                DropInfo[15]--;
                DropInfo[16] -= (uint64_t)P->len;
            } else {
                memset(D, 0, sizeof(uint64_t) * L.n_u64);
                clean_step(p, &L, seq + P->start, qual ? qual + P->start : NULL, P->len, D);
                for (uint32_t w = 0; w < L.n_u64; w++) C[w] -= D[w];
            }
            const int c = fr.fold, len = P->len;
            const int arm = c >= len - c ? c : len - c;
            if (arm != c) P->start += c;
            P->len = arm;
            P->sum_q = 0;
            P->repeat_len = -1;
            P->status = TGSF_PIECE_EMIT;
            stats[0]++;
            stats[1] += (uint64_t)(len - arm);
            if (arm < p->min_len) {
                P->status = TGSF_PIECE_FOLDBACK;
                stats[2]++;
                stats[3] += (uint64_t)arm;
                continue;
            }
            if (p->min_repeat > 0) { /* the repeat check on the arm */
                P->repeat_len = kmer_repeat_len(seq + P->start, P->len, p->kmer);
                if (P->repeat_len < p->min_repeat) {
                    DropInfo[15]++;
                    DropInfo[16] += (uint64_t)P->len;
                    P->status = TGSF_PIECE_SHORT_REPEAT;
                    dropped = 1;
                }
            }
        } else if (P->status == TGSF_PIECE_SHORT_REPEAT) {
            dropped = 1;
        }
        if (dropped) continue;
        const uint8_t *cs = seq + P->start;
        const uint8_t *cq = qual ? qual + P->start : NULL;
        if (keys) {
            P->contam_hits = contam_hits(cs, P->len, ck, keys, n_keys);
            uint64_t windows = P->len >= ck ? (uint64_t)(P->len - ck + 1) : 0;
            if (windows >= 1 && (uint64_t)P->contam_hits * 1000000ull >= ppm * windows) {
                if (fr.fold < 0) { /* the uncut piece went through the clean step in tgsfo_run */
                    memset(D, 0, sizeof(uint64_t) * L.n_u64);
                    clean_step(p, &L, cs, cq, P->len, D);
                    for (uint32_t w = 0; w < L.n_u64; w++) C[w] -= D[w];
                }
                P->status = TGSF_PIECE_CONTAM;
                P->sum_q = 0;
                continue;
            }
        }
        if (fr.fold < 0) continue; /* tgsfo_run's clean step stands */
        clean_step(p, &L, cs, cq, P->len, C);
        if (cq) { /* status and sum_q as the clean step of tgsfo_run sets them */
            memset(D, 0, sizeof(uint64_t) * L.n_u64);
            uint64_t sumQ = calc_sum_quality(cs, cq, P->len, p->qtype, D + L.clean_bin_qual, D + L.clean_bin_cnt);
            P->sum_q = sumQ;
            double q = (double)sumQ / (double)(uint64_t)P->len;
            if ((p->flags & TGSF_FLAG_FILTER) && (q < p->min_q || q > p->max_q)) P->status = TGSF_PIECE_LOWQ;
        }
    }
    free(D);
    free(keys);
    return TGSF_OK;
}
