/*
 * tests/guided_oracle.c -- CPU restatement of psa_align_batch_guided over per-row bands.  TEST INFRASTRUCTURE ONLY.
 *
 * Built by tests/guided_oracle.py into a temporary directory.  It compiles tests/banded_oracle.c (and through it
 * oracle/gotoh_oracle.c) into the same library unchanged and adds fill, traceback and linear-space score over an
 * arbitrary monotone band given row by row.
 */
#include "banded_oracle.c"



/* ---- per-row bands (psa_align_batch_guided) ----------------------------------------------------------------------
 * Row i's cells are lo[i] <= j <= hi[i] (0 <= lo[i] <= hi[i] <= n, both non-decreasing, lo[0] = 0): the band of an anchor
 * chain (tests/guided_oracle.py: guide_rows).  Row 0's T2 border exists for j <= hi[0], column 0's T3 border where
 * lo[i] = 0; everything else as orc_fill_banded / orc_align_banded / orc_score_banded, which are these functions on the
 * diagonal band's rows. */
int orc_fill_rows(const char* a, const char* b, int64_t m, int64_t n, int g, int h, int mode, const int64_t* lo,
                  const int64_t* hi, int32_t* T1, int32_t* T2, int32_t* T3) {
    if (m < 1 || n < 1 || g < 0 || h < 0) return -1;
    const int64_t W = n + 1;
    const int32_t go = g + h;
    T1[0] = mode == 0 ? 0 : ORC_NEG; T2[0] = ORC_NEG; T3[0] = ORC_NEG;
    for (int64_t j = 1; j <= n; ++j) {
        T1[j] = ORC_NEG; T3[j] = ORC_NEG;
        T2[j] = (mode == 0 && j <= hi[0]) ? (int32_t)(-h - (int64_t)g * j) : ORC_NEG;
    }
    for (int64_t i = 1; i <= m; ++i) {
        int32_t *r1 = T1 + i * W, *r2 = T2 + i * W, *r3 = T3 + i * W;
        const int32_t *p1 = r1 - W, *p2 = r2 - W, *p3 = r3 - W;
        r1[0] = ORC_NEG; r2[0] = ORC_NEG;
        r3[0] = (mode == 0 && lo[i] == 0) ? (int32_t)(-h - (int64_t)g * i) : ORC_NEG;
        const char ai = a[i - 1];
        for (int64_t j = 1; j <= n; ++j) {
            if (j < lo[i] || j > hi[i]) { r1[j] = ORC_NEG; r2[j] = ORC_NEG; r3[j] = ORC_NEG; continue; }
            const int32_t f = (ai == b[j - 1]) ? 1 : 0;
            int32_t d = orc_max3(p1[j - 1], p2[j - 1], p3[j - 1]);
            if (mode == 1) d = orc_max(d, 0);
            r1[j] = orc_add(d, f);
            r3[j] = orc_max3(orc_add(p1[j], -go), orc_add(p2[j], -go), orc_add(p3[j], -g));
            r2[j] = orc_max3(orc_add(r1[j - 1], -go), orc_add(r2[j - 1], -g), orc_add(r3[j - 1], -go));
        }
    }
    return 0;
}

int orc_align_rows(const char* a, const char* b, int64_t m, int64_t n, int g, int h, int mode, const int64_t* lo,
                   const int64_t* hi, orc_result* res, uint8_t* ops, char* row_a, char* row_b) {
    if (m == 0 || n == 0) return orc_align_full(a, b, m, n, g, h, -1, -1, mode, res, ops, row_a, row_b, NULL);
    const size_t cells = (size_t)(m + 1) * (size_t)(n + 1);
    int32_t* T = (int32_t*)malloc(3 * cells * sizeof(int32_t));
    if (!T) return -3;
    int rc = orc_fill_rows(a, b, m, n, g, h, mode, lo, hi, T, T + cells, T + 2 * cells);
    if (rc == 0 && mode == 0 && orc_max3(T[cells - 1], T[2 * cells - 1], T[3 * cells - 1]) <= ORC_NEG) {
        orc_band_no_path(m, n, res);
    } else if (rc == 0) {
        rc = orc_traceback_full(a, b, m, n, g, h, -1, mode, T, T + cells, T + 2 * cells, res, ops);
        if (rc == 0 && row_a && row_b) orc_render_rows(a, b, ops, res->aln_len, res->start_i, res->start_j, row_a, row_b);
    }
    free(T);
    return rc;
}

/* Linear-space score and end cell over per-row bands: two rows of the widest row's width. */
int orc_score_rows(const char* a, const char* b, int64_t m, int64_t n, int g, int h, int mode, const int64_t* lo,
                   const int64_t* hi, orc_result* res) {
    if (g < 0 || h < 0) return -1;
    if (m == 0 || n == 0) return orc_score_linear(a, b, m, n, g, h, mode, res);
    const int32_t go = g + h;
    int64_t width = 1;
    for (int64_t i = 0; i <= m; ++i) width = hi[i] - lo[i] + 1 > width ? hi[i] - lo[i] + 1 : width;
    int32_t* buf = (int32_t*)malloc(6 * (size_t)width * sizeof(int32_t));
    if (!buf) return -3;
    int32_t *p1 = buf, *p2 = p1 + width, *p3 = p2 + width, *c1 = p3 + width, *c2 = c1 + width, *c3 = c2 + width;
    memset(res, 0, sizeof(*res));
    int64_t plo = 0, phi = hi[0];
    for (int64_t j = 0; j <= phi; ++j) {
        p1[j] = (j == 0 && mode == 0) ? 0 : ORC_NEG;
        p3[j] = ORC_NEG;
        p2[j] = (j > 0 && mode == 0) ? (int32_t)(-h - (int64_t)g * j) : ORC_NEG;
    }
    int32_t best = 0; int64_t bi = 0, bj = 0;
    for (int64_t i = 1; i <= m; ++i) {
        const int64_t rlo = lo[i], rhi = hi[i];
        const char ai = a[i - 1];
#define ORC_P(arr, j) (((j) >= plo && (j) <= phi) ? (arr)[(j) - plo] : ORC_NEG)
        for (int64_t j = rlo; j <= rhi; ++j) {
            const int64_t x = j - rlo;
            if (j == 0) {
                c1[x] = ORC_NEG; c2[x] = ORC_NEG;
                c3[x] = mode == 0 ? (int32_t)(-h - (int64_t)g * i) : ORC_NEG;
                continue;
            }
            const int32_t f = (ai == b[j - 1]) ? 1 : 0;
            int32_t d = orc_max3(ORC_P(p1, j - 1), ORC_P(p2, j - 1), ORC_P(p3, j - 1));
            if (mode == 1) d = orc_max(d, 0);
            c1[x] = orc_add(d, f);
            c3[x] = orc_max3(orc_add(ORC_P(p1, j), -go), orc_add(ORC_P(p2, j), -go), orc_add(ORC_P(p3, j), -g));
            const int32_t l1 = x > 0 ? c1[x - 1] : ORC_NEG, l2 = x > 0 ? c2[x - 1] : ORC_NEG, l3 = x > 0 ? c3[x - 1] : ORC_NEG;
            c2[x] = orc_max3(orc_add(l1, -go), orc_add(l2, -g), orc_add(l3, -go));
            if (mode == 1 && c1[x] > best) { best = c1[x]; bi = i; bj = j; }
        }
#undef ORC_P
        int32_t* t;
        t = p1; p1 = c1; c1 = t; t = p2; p2 = c2; c2 = t; t = p3; p3 = c3; c3 = t;
        plo = rlo; phi = rhi;
    }
    if (mode == 0) {
        const int64_t x = n - plo;        /* hi[m] = n */
        res->t1 = p1[x]; res->t2 = p2[x]; res->t3 = p3[x];
        res->score = orc_max3(res->t1, res->t2, res->t3);
        res->end_i = m; res->end_j = n;
        res->end_state = (res->t1 >= res->t2 && res->t1 >= res->t3) ? 1 : (res->t2 >= res->t1 && res->t2 >= res->t3) ? 2 : 3;
        if (res->score <= ORC_NEG) orc_band_no_path(m, n, res);
    } else {
        res->score = best; res->t1 = best; res->t2 = ORC_NEG; res->t3 = ORC_NEG;
        res->end_i = bi; res->end_j = bj; res->end_state = 1;
    }
    free(buf);
    return 0;
}
