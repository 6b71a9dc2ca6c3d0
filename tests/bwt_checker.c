/* bwt_checker.c -- sequential CPU checkers of the Burrows-Wheeler transform (include/sab200.h), for the tests and
 * the CPU baseline of tools/bwt_bench.py.  Test infrastructure: the product never loads it.
 *
 *   checker_bwt          the definition itself: L[j] = s[sa[j]-1] over the n+1 rows of a given suffix array, the row
 *                        with sa[j] = 0 is the primary index and is left out
 *   checker_inverse_bwt  the LF walk: from row 0 (the empty suffix) back through s[n-1], ..., s[0]; -1 unless the
 *                        walk reaches the primary row after exactly n steps, i.e. unless the cycle through it has
 *                        n+1 rows
 */
#include <stdint.h>
#include <stdlib.h>

int checker_bwt(const uint8_t *s, uint64_t n, const uint32_t *sa, uint8_t *u, uint64_t *primary) {
    uint64_t k = 0;
    *primary = 0;
    for (uint64_t j = 0; j <= n; ++j) {
        if (sa[j] > n) return -1;
        if (sa[j] == 0) *primary = j;
        else u[k++] = s[sa[j] - 1];
    }
    return k == n ? 0 : -1;
}

int checker_inverse_bwt(const uint8_t *u, uint64_t n, uint64_t p, uint8_t *s) {
    if (n == 0) return p == 0 ? 0 : -1;
    if (p < 1 || p > n) return -1;
    uint64_t first[257] = {0}; /* first row of each byte value in the first column; row 0 is '$' */
    for (uint64_t i = 0; i < n; ++i) first[u[i] + 1]++;
    first[0] = 1;
    for (int c = 1; c <= 256; ++c) first[c] += first[c - 1];
    uint32_t *lf = (uint32_t *)malloc((n + 1) * sizeof(uint32_t)); /* LF(row) */
    if (!lf) return -2;
    lf[p] = 0;
    for (uint64_t j = 0; j <= n; ++j) {
        if (j == p) continue;
        const uint8_t c = u[j < p ? j : j - 1];
        lf[j] = (uint32_t)first[c]++;
    }
    uint64_t j = 0;
    int rc = 0;
    for (uint64_t k = n; k-- > 0;) {
        if (j == p) { /* the cycle closes before the whole text is read */
            rc = -1;
            break;
        }
        s[k] = u[j < p ? j : j - 1];
        j = lf[j];
    }
    if (rc == 0 && j != p) rc = -1;
    free(lf);
    return rc;
}
