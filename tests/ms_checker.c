/* ms_checker.c -- sequential CPU checkers of the matching statistics (sab200_matching_statistics_batch,
 * include/sab200.h), for the tests and tools/ms_bench.py.  Test infrastructure: the product never loads it.
 *
 * Queries are qs[offs[q] .. offs[q+1]); the outputs are indexed by the absolute offset in qs.  For position i of a
 * query ending at e: len[i] = the longest prefix of qs[i .. e) that occurs in s, [lo[i], hi[i]) = the suffix-array
 * range of the suffixes (the empty one included) that start with it, [0, n+1) when len[i] = 0.
 *
 *   checker_ms_naive    the definition by brute force over every text position; the range counts the suffixes
 *                       smaller than the match and those that start with it.  No suffix array.  Small inputs.
 *   checker_ms_bisect   per position: lower bound of qs[i .. e) over a given suffix array, the longer common prefix
 *                       with the two neighbours of the insertion point, then two bisections for the range.
 */
#include <stdint.h>

/* common prefix of the suffix at p and w[0 .. m) */
static uint64_t lcp_with(const uint8_t *s, uint64_t n, uint64_t p, const uint8_t *w, uint64_t m) {
    uint64_t d = 0;
    while (d < m && p + d < n && s[p + d] == w[d]) ++d;
    return d;
}

/* < 0: the suffix at p is smaller than w[0 .. m) and does not start with it; 0: it starts with it; > 0: greater */
static int cmp_prefix(const uint8_t *s, uint64_t n, uint64_t p, const uint8_t *w, uint64_t m) {
    const uint64_t d = lcp_with(s, n, p, w, m);
    if (d == m) return 0;
    if (p + d == n) return -1;
    return s[p + d] < w[d] ? -1 : 1;
}

int checker_ms_naive(const uint8_t *s, uint64_t n, const uint8_t *qs, const uint64_t *offs, uint64_t nq, uint32_t *len,
                     uint32_t *lo, uint32_t *hi) {
    for (uint64_t q = 0; q < nq; ++q) {
        for (uint64_t i = offs[q]; i < offs[q + 1]; ++i) {
            const uint64_t m = offs[q + 1] - i;
            uint64_t best = 0;
            for (uint64_t p = 0; p < n; ++p) {
                const uint64_t d = lcp_with(s, n, p, qs + i, m);
                if (d > best) best = d;
            }
            uint64_t below = 0, occ = 0;
            if (best > 0)
                for (uint64_t p = 0; p <= n; ++p) {
                    const int c = cmp_prefix(s, n, p, qs + i, best);
                    below += c < 0;
                    occ += c == 0;
                }
            len[i] = (uint32_t)best;
            lo[i] = best ? (uint32_t)below : 0;
            hi[i] = best ? (uint32_t)(below + occ) : (uint32_t)(n + 1);
        }
    }
    return 0;
}

/* first j in [0, n] whose suffix compares >= 0 (strict = 0) or > 0 (strict = 1) with w[0 .. m) */
static uint64_t bound(const uint8_t *s, uint64_t n, const uint32_t *sa, const uint8_t *w, uint64_t m, int strict) {
    uint64_t a = 0, b = n + 1;
    while (a < b) {
        const uint64_t mid = a + (b - a) / 2;
        const int c = cmp_prefix(s, n, sa[mid], w, m);
        if (c < 0 || (strict && c == 0)) a = mid + 1;
        else b = mid;
    }
    return a;
}

int checker_ms_bisect(const uint8_t *s, uint64_t n, const uint32_t *sa, const uint8_t *qs, const uint64_t *offs, uint64_t nq,
                      uint32_t *len, uint32_t *lo, uint32_t *hi) {
    for (uint64_t j = 0; j <= n; ++j)
        if (sa[j] > n) return -1;
    for (uint64_t q = 0; q < nq; ++q) {
        for (uint64_t i = offs[q]; i < offs[q + 1]; ++i) {
            const uint8_t *w = qs + i;
            const uint64_t m = offs[q + 1] - i;
            const uint64_t x = bound(s, n, sa, w, m, 0);
            uint64_t best = 0;
            if (x > 0) best = lcp_with(s, n, sa[x - 1], w, m);
            if (x <= n) {
                const uint64_t d = lcp_with(s, n, sa[x], w, m);
                if (d > best) best = d;
            }
            len[i] = (uint32_t)best;
            lo[i] = best ? (uint32_t)bound(s, n, sa, w, best, 0) : 0;
            hi[i] = best ? (uint32_t)bound(s, n, sa, w, best, 1) : (uint32_t)(n + 1);
        }
    }
    return 0;
}
