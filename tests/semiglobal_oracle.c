/*
 * semiglobal_oracle.c -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
 *
 * Plain-C CPU statement of the semi-global mode (B2A_MODE_SEMIGLOBAL, include/b2align.h): the whole pattern
 * against the substring of the text that suits it best.  It is hw2's Needleman-Wunsch (hw2.cpp:118-190, the
 * oracle's orc_global) with two changes at the borders:
 *   - row 0 is free: H(0, j) = 0 for j = 0..n (leading text costs nothing); column 0 keeps H(i, 0) = i * gap;
 *   - the end cell is (m, j*), j* = the smallest j in 0..n with H(m, j) = max_j H(m, j) (trailing text is free).
 * Cells use hw2's recurrence and tie order d > l > u (hw2.cpp:140-153).  The traceback applies hw2's NW test order
 * from (m, j*) -- (i>0, j>0, 'd') -> 'M', (i>0, 'u') -> 'D', (j>0, 'l') -> 'I'; column 0 holds 'u' -- and STOPS when
 * it reaches row 0: no 'I' tail along the free row.  start = (0, column where the walk reached row 0).
 * overlap = overlapLongestExactMatch (hw2.cpp:267-278), as in global mode.
 *
 * Same result record and op letters as oracle/hw2_oracle.c, which tests/semiglobal_oracle.py loads beside it.
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

typedef struct {
    int32_t  score;
    uint32_t end_i, end_j, start_i, start_j;
    int32_t  overlap;
    uint32_t n_ops;
} orc_result;

/* full matrices + direction letters + traceback; ops (traceback order) must hold m + n bytes */
int orc_semiglobal(const uint8_t* p, uint32_t m, const uint8_t* t, uint32_t n,
                   int match, int mismatch, int gap, orc_result* res, uint8_t* ops)
{
    const size_t W = (size_t)n + 1;
    int32_t* dp = (int32_t*)malloc(sizeof(int32_t) * ((size_t)m + 1) * W);
    char*    tb = (char*)malloc(((size_t)m + 1) * W);
    if (!dp || !tb) { free(dp); free(tb); return -1; }
    memset(tb, ' ', ((size_t)m + 1) * W);
    for (uint32_t j = 0; j <= n; ++j) dp[j] = 0;                                   /* free leading text */
    for (uint32_t i = 1; i <= m; ++i) { dp[i * W] = (int32_t)((int64_t)i * gap); tb[i * W] = 'u'; }
    for (uint32_t i = 1; i <= m; ++i) {
        for (uint32_t j = 1; j <= n; ++j) {                                        /* hw2.cpp:140-153 */
            int up   = dp[(i - 1) * W + j] + gap;
            int left = dp[i * W + j - 1] + gap;
            int v    = dp[(i - 1) * W + j - 1] + (p[i - 1] == t[j - 1] ? match : mismatch);
            char d = 'd';
            if (left > v) { v = left; d = 'l'; }
            if (up > v)   { v = up;   d = 'u'; }
            dp[i * W + j] = v; tb[i * W + j] = d;
        }
    }
    uint32_t bj = 0;                                                               /* first maximum of row m */
    for (uint32_t j = 1; j <= n; ++j) if (dp[(size_t)m * W + j] > dp[(size_t)m * W + bj]) bj = j;
    uint32_t ti = m, tj = bj, k = 0;
    int cur = 0, best = 0;
    while (ti > 0) {
        char d = tb[ti * W + tj];
        if (tj > 0 && d == 'd') {
            ops[k++] = 'M';
            if (p[ti - 1] == t[tj - 1] && p[ti - 1] != '-') { if (++cur > best) best = cur; } else cur = 0;
            --ti; --tj;
        } else if (d == 'u') { ops[k++] = 'D'; cur = 0; --ti; }
        else if (tj > 0 && d == 'l') { ops[k++] = 'I'; cur = 0; --tj; }
        else { free(dp); free(tb); return -2; }
    }
    res->score = dp[(size_t)m * W + bj];
    res->end_i = m; res->end_j = bj; res->start_i = 0; res->start_j = tj;
    res->overlap = best; res->n_ops = k;
    free(dp); free(tb);
    return 0;
}

/* linear memory: score and end cell only (same values as orc_semiglobal), for pairs whose matrices do not fit */
int orc_semiglobal_score(const uint8_t* p, uint32_t m, const uint8_t* t, uint32_t n,
                         int match, int mismatch, int gap, orc_result* res)
{
    int32_t* row = (int32_t*)malloc(sizeof(int32_t) * ((size_t)n + 1) * 2);
    if (!row) return -1;
    int32_t* tmp = row + (size_t)n + 1;
    for (uint32_t j = 0; j <= n; ++j) row[j] = 0;
    for (uint32_t i = 1; i <= m; ++i) {
        const uint8_t pc = p[i - 1];
        for (uint32_t j = 1; j <= n; ++j) {                                        /* max(diag + s, up + gap): previous row only */
            const int d = row[j - 1] + (pc == t[j - 1] ? match : mismatch);
            const int u = row[j] + gap;
            tmp[j] = d > u ? d : u;
        }
        int32_t left = (int32_t)((int64_t)i * gap);
        row[0] = left;
        for (uint32_t j = 1; j <= n; ++j) { int v = tmp[j]; const int l = left + gap; if (l > v) v = l; row[j] = v; left = v; }
    }
    uint32_t bj = 0;
    for (uint32_t j = 1; j <= n; ++j) if (row[j] > row[bj]) bj = j;
    memset(res, 0, sizeof(*res));
    res->score = row[bj]; res->end_i = m; res->end_j = bj;
    free(row);
    return 0;
}
