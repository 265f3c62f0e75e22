/*
 * contam_label_oracle.c — CPU restatement of the contaminant screen's per-record attribution
 * (tgsf_set_contaminants_labelled, tgsf_contam_classify).  TEST INFRASTRUCTURE ONLY, built by
 * tests/contam_label_oracle.py into a temporary directory.
 *
 * Keys are the ones of tests/contam_oracle.c: canonical k-mers (min of forward and reverse-complement code, A0 C1 G2
 * T3, 2 bits per base), acgt counts as ACGT, a window with any other byte carries no key.  Every valid window of
 * record r contributes the pair (key, r); after sorting the pairs, a key whose pairs all name one record r gets
 * label r, any other key gets LABEL_SHARED.  A piece's hits are its valid windows whose key is in the set; v_r counts
 * those whose key has label r.  Its record is the r with the largest v_r >= 1 (smallest r on a tie) and record_hits
 * that v_r; else n_seqs (the shared row) with record_hits 0 when hits >= 1; else -1 with record_hits 0.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define LABEL_SHARED UINT32_MAX

typedef struct { uint64_t key; uint32_t rec; } pair_t;

static int code_of(uint8_t b) {
    switch (b) {
        case 'A': case 'a': return 0;
        case 'C': case 'c': return 1;
        case 'G': case 'g': return 2;
        case 'T': case 't': return 3;
        default: return -1;
    }
}

/* Canonical k-mer of seq[0, k), or UINT64_MAX when a byte is not ACGT/acgt. */
static uint64_t key_of(const uint8_t *seq, int k) {
    uint64_t fwd = 0, rev = 0;
    for (int i = 0; i < k; i++) {
        int c = code_of(seq[i]);
        if (c < 0) return UINT64_MAX;
        fwd = (fwd << 2) | (uint64_t)c;
        rev |= (uint64_t)(3 - c) << (2 * i);
    }
    return fwd < rev ? fwd : rev;
}

static int cmp_pair(const void *a, const void *b) {
    const pair_t *x = (const pair_t *)a, *y = (const pair_t *)b;
    if (x->key != y->key) return x->key < y->key ? -1 : 1;
    return x->rec < y->rec ? -1 : x->rec > y->rec ? 1 : 0;
}

static int cmp_u64(const void *a, const void *b) {
    uint64_t x = *(const uint64_t *)a, y = *(const uint64_t *)b;
    return x < y ? -1 : x > y ? 1 : 0;
}

/* Sorted distinct keys of the set and their labels (both malloc'ed); returns the number of keys. */
static uint64_t build(const uint8_t *seq, const uint64_t *offs, uint32_t n_seqs, int k, uint64_t **keys_out,
                      uint32_t **labels_out) {
    pair_t *v = (pair_t *)malloc(sizeof(pair_t) * (size_t)(offs[n_seqs] + 1));
    uint64_t n = 0;
    for (uint32_t r = 0; r < n_seqs; r++)
        for (uint64_t i = offs[r]; i + (uint64_t)k <= offs[r + 1]; i++) {
            uint64_t key = key_of(seq + i, k);
            if (key != UINT64_MAX) { v[n].key = key; v[n].rec = r; n++; }
        }
    qsort(v, (size_t)n, sizeof(pair_t), cmp_pair);
    uint64_t *keys = (uint64_t *)malloc(sizeof(uint64_t) * (size_t)(n + 1));
    uint32_t *labels = (uint32_t *)malloc(sizeof(uint32_t) * (size_t)(n + 1));
    uint64_t d = 0;
    for (uint64_t i = 0; i < n; i++) {
        if (d > 0 && keys[d - 1] == v[i].key) {
            if (labels[d - 1] != v[i].rec) labels[d - 1] = LABEL_SHARED;
        } else {
            keys[d] = v[i].key;
            labels[d] = v[i].rec;
            d++;
        }
    }
    free(v);
    *keys_out = keys;
    *labels_out = labels;
    return d;
}

/* n_kmers of the set; record_kmers[r] = keys labelled r, record_kmers[n_seqs] = shared keys. */
uint64_t tgsfo_contam_labels(const uint8_t *seq, const uint64_t *offs, uint32_t n_seqs, int k,
                             uint64_t *record_kmers) {
    uint64_t *keys;
    uint32_t *labels;
    uint64_t n = build(seq, offs, n_seqs, k, &keys, &labels);
    memset(record_kmers, 0, sizeof(uint64_t) * ((size_t)n_seqs + 1));
    for (uint64_t i = 0; i < n; i++) record_kmers[labels[i] == LABEL_SHARED ? n_seqs : labels[i]]++;
    free(keys);
    free(labels);
    return n;
}

/* out[3 i .. 3 i + 2] = (hits, record, record_hits) of piece seq[poffs[i], poffs[i+1]) against the set. */
void tgsfo_contam_attribute(const uint8_t *cseq, const uint64_t *coffs, uint32_t n_cseqs, int k, const uint8_t *seq,
                            const uint64_t *poffs, uint32_t n, int32_t *out) {
    uint64_t *keys;
    uint32_t *labels;
    uint64_t n_keys = build(cseq, coffs, n_cseqs, k, &keys, &labels);
    int32_t *votes = (int32_t *)calloc((size_t)n_cseqs, sizeof(int32_t));
    for (uint32_t p = 0; p < n; p++) {
        const uint8_t *s = seq + poffs[p];
        const int64_t len = (int64_t)(poffs[p + 1] - poffs[p]);
        int32_t hits = 0;
        memset(votes, 0, sizeof(int32_t) * (size_t)n_cseqs);
        for (int64_t i = 0; i + k <= len; i++) {
            uint64_t key = key_of(s + i, k);
            if (key == UINT64_MAX) continue;
            const uint64_t *f = (const uint64_t *)bsearch(&key, keys, (size_t)n_keys, sizeof(uint64_t), cmp_u64);
            if (!f) continue;
            hits++;
            uint32_t l = labels[f - keys];
            if (l != LABEL_SHARED) votes[l]++;
        }
        int32_t record = -1, best = 0;
        for (uint32_t r = 0; r < n_cseqs; r++)
            if (votes[r] > best) { best = votes[r]; record = (int32_t)r; }
        if (record < 0 && hits > 0) record = (int32_t)n_cseqs;
        out[3 * (size_t)p] = hits;
        out[3 * (size_t)p + 1] = record;
        out[3 * (size_t)p + 2] = best;
    }
    free(votes);
    free(keys);
    free(labels);
}
