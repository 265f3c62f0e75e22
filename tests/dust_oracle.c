/*
 * dust_oracle.c — CPU restatement of the low-complexity (DUST) screen (tgsf_set_dust).  TEST INFRASTRUCTURE ONLY,
 * built by tests/dust_oracle.py into a temporary directory.
 *
 * The per-read path is the pinned oracle (through foldback_oracle.c and contam_oracle.c, which include
 * oracle/tgsf_oracle.c unchanged).  tgsfo_run_dust runs tgsfo_run, tgsfo_run_contam or tgsfo_run_foldback, whichever
 * the case needs, then screens every piece whose status is EMIT or LOWQ: the GPU screens a piece before the clean
 * step, which is where LOWQ is decided.  For each piece it drops it replays that piece's clean step into a zeroed block
 * and subtracts it, as tgsfo_run_contam does.
 *
 * Detection scores every window from scratch (no rolling update) and shares no code with the kernel.  The constants
 * are restated here on purpose.
 */
#include "foldback_oracle.c"

#define DO_WINDOW 64
#define DO_TRIPLETS 62
#define DO_LEVEL_MIN 1
#define DO_LEVEL_MAX 30

/* S of window s[j, j+64), or -1 when a byte of it is not ACGT/acgt. */
int tgsfo_dust_score(const uint8_t *s, int32_t j) {
    int code[DO_WINDOW];
    for (int i = 0; i < DO_WINDOW; i++) {
        code[i] = contam_code(s[j + i]);
        if (code[i] < 0) return -1;
    }
    int cnt[64] = {0};
    for (int i = 0; i < DO_TRIPLETS; i++) cnt[16 * code[i] + 4 * code[i + 1] + code[i + 2]]++;
    int S = 0;
    for (int t = 0; t < 64; t++) S += cnt[t] * (cnt[t] - 1) / 2;
    return S;
}

/* M of piece s[0, L) at this level: the bases covered by the masked windows. */
uint32_t tgsfo_dust_masked(const uint8_t *s, int32_t L, int32_t level) {
    uint32_t M = 0;
    int64_t prev = -1;
    for (int32_t j = 0; j + DO_WINDOW <= L; j++) {
        if (tgsfo_dust_score(s, j) <= 61 * level) continue;
        M += prev < 0 || j - prev >= DO_WINDOW ? DO_WINDOW : (uint32_t)(j - prev);
        prev = j;
    }
    return M;
}

/* tgsfo_run with the DUST screen at (level, dust_frac), after the fold-back screen when fold_stats is not NULL
 * (fold_stats receives its statistics) and after the contaminant screen when n_cseqs > 0. */
int tgsfo_run_dust(const tgsf_params *p, const uint8_t *bases, const uint8_t *quals, const uint64_t *offsets,
                   uint32_t n_reads, tgsf_read_result *reads, tgsf_piece *pieces, uint32_t pieces_cap,
                   uint32_t *n_pieces_out, uint64_t *C, uint64_t *fold_stats, const uint8_t *cseq,
                   const uint64_t *coffs, uint32_t n_cseqs, int ck, float contam_frac, int32_t level,
                   float dust_frac) {
    long long q = llround((double)dust_frac * 1e6);
    if (level < DO_LEVEL_MIN || level > DO_LEVEL_MAX || q < 1 || q > 1000000) return TGSF_ERR_INVALID;
    const uint64_t ppm = (uint64_t)q;
    uint32_t np = 0;
    int rc;
    if (fold_stats)
        rc = tgsfo_run_foldback(p, bases, quals, offsets, n_reads, reads, pieces, pieces_cap, &np, C, fold_stats,
                                cseq, coffs, n_cseqs, ck, contam_frac);
    else if (n_cseqs > 0)
        rc = tgsfo_run_contam(p, bases, quals, offsets, n_reads, reads, pieces, pieces_cap, &np, C, cseq, coffs,
                              n_cseqs, ck, contam_frac);
    else
        rc = tgsfo_run(p, bases, quals, offsets, n_reads, reads, pieces, pieces_cap, &np, C);
    if (n_pieces_out) *n_pieces_out = np;
    if (rc != TGSF_OK) return rc;
    tgsf_counter_layout L;
    tgsf_make_layout(p->bc_len, p->max_read_len, &L);
    uint64_t *D = (uint64_t *)malloc(sizeof(uint64_t) * L.n_u64);
    for (uint32_t i = 0; i < np; i++) {
        tgsf_piece *P = &pieces[i];
        if (P->status != TGSF_PIECE_EMIT && P->status != TGSF_PIECE_LOWQ) continue;
        if (P->len < DO_WINDOW) continue;
        const uint8_t *cs = bases + offsets[P->read] + P->start;
        const uint8_t *cq = quals ? quals + offsets[P->read] + P->start : NULL;
        const uint64_t M = tgsfo_dust_masked(cs, P->len, level);
        if (M * 1000000ull < ppm * (uint64_t)P->len) continue;
        memset(D, 0, sizeof(uint64_t) * L.n_u64);
        clean_step(p, &L, cs, cq, P->len, D);
        for (uint32_t w = 0; w < L.n_u64; w++) C[w] -= D[w];
        P->status = TGSF_PIECE_LOWCOMPLEX;
        P->sum_q = 0;
    }
    free(D);
    return TGSF_OK;
}
