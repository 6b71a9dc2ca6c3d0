/* lz77_checker.c -- sequential CPU checkers of the LZ77 factorization (include/sab200.h), for the tests and the CPU
 * baseline of tools/lz77_bench.py.  Test infrastructure: the product never loads it.
 *
 *   checker_lz77_brute   the greedy parse by brute force: at every factor start the longest earlier match over all
 *                        p < b (O(n^2) and more: small texts only).  Lengths and literals only: it picks no source.
 *   checker_lz77_sa      the definition over a given suffix array: inverse, Kasai's LCP, PSV / NSV with their running
 *                        LCP minima by pointer chasing (a stack in disguise, amortized linear), the tie rule, then the
 *                        sequential walk b -> b + max(1, LPF[b]).
 *   checker_lz77_verify  properties of any greedy parse: the factors tile the text, literals hold their byte, every copy
 *                        matches its source, which lies before its start, and is maximal (no earlier occurrence one byte
 *                        longer; brute force over the earlier positions).
 *   checker_lz77_decode  the sequential decoder; -1 on a parse that breaks a rule of sab200_lz77_decode.
 */
#include <stdint.h>
#include <stdlib.h>

static uint64_t match(const uint8_t *s, uint64_t n, uint64_t p, uint64_t b, uint64_t cap) {
    uint64_t l = 0;
    while (l < cap && b + l < n && s[p + l] == s[b + l]) ++l;
    return l;
}

int checker_lz77_brute(const uint8_t *s, uint64_t n, uint32_t *pos, uint32_t *len, uint64_t *z) {
    uint64_t t = 0;
    for (uint64_t b = 0; b < n; ++t) {
        uint64_t best = 0;
        for (uint64_t p = 0; p < b; ++p) {
            const uint64_t l = match(s, n, p, b, n);
            if (l > best) best = l;
        }
        len[t] = (uint32_t)best;
        pos[t] = best ? 0 : s[b];
        b += best ? best : 1;
    }
    *z = t;
    return 0;
}

int checker_lz77_sa(const uint8_t *s, uint64_t n, const uint32_t *sa, uint32_t *pos, uint32_t *len, uint64_t *z) {
    *z = 0;
    if (n == 0) return 0;
    const uint64_t N = n + 1;
    uint32_t *isa = malloc(N * 4), *lcp = malloc((N + 1) * 4), *psv = malloc(N * 4), *nsv = malloc(N * 4);
    uint32_t *lp = malloc(N * 4), *ln = malloc(N * 4);
    if (!isa || !lcp || !psv || !nsv || !lp || !ln) return -2;
    for (uint64_t j = 0; j < N; ++j) isa[sa[j]] = (uint32_t)j;
    lcp[0] = 0;
    lcp[N] = 0;
    for (uint64_t i = 0, h = 0; i < n; ++i) { /* Kasai */
        const uint64_t j = isa[i], p = sa[j - 1]; /* j >= 1: row 0 is the empty suffix */
        while (i + h < n && p + h < n && s[i + h] == s[p + h]) ++h;
        lcp[j] = (uint32_t)h;
        if (h) --h;
    }
    /* PSV: the nearest row k < j with sa[k] < sa[j] (0 = none: sa[0] = n is below nothing), lp[j] = min lcp over (k, j] */
    psv[0] = 0;
    lp[0] = 0;
    for (uint64_t j = 1; j < N; ++j) {
        uint64_t k = j - 1, m = lcp[j];
        while (k > 0 && sa[k] > sa[j]) {
            if (lp[k] < m) m = lp[k];
            k = psv[k];
        }
        psv[j] = (uint32_t)k;
        lp[j] = k ? (uint32_t)m : 0;
    }
    /* NSV: the nearest row k > j with sa[k] < sa[j] (N = none), ln[j] = min lcp over (j, k] */
    for (uint64_t j = N; j-- > 1;) {
        uint64_t k = j + 1, m = j + 1 < N ? lcp[j + 1] : 0;
        while (k < N && sa[k] > sa[j]) {
            if (ln[k] < m) m = ln[k];
            k = nsv[k];
        }
        nsv[j] = (uint32_t)k;
        ln[j] = k < N ? (uint32_t)m : 0;
    }
    uint64_t t = 0;
    for (uint64_t b = 0; b < n; ++t) {
        const uint64_t j = isa[b];
        const uint32_t a = lp[j], c = ln[j];
        const uint32_t l = a > c ? a : c;
        len[t] = l;
        pos[t] = l == 0 ? s[b] : (a >= c ? sa[psv[j]] : sa[nsv[j]]);
        b += l ? l : 1;
    }
    *z = t;
    free(isa), free(lcp), free(psv), free(nsv), free(lp), free(ln);
    return 0;
}

/* 0 when (pos, len) is a greedy parse of s; else 1 + the index of the first bad factor */
int64_t checker_lz77_verify(const uint8_t *s, uint64_t n, const uint32_t *pos, const uint32_t *len, uint64_t z) {
    uint64_t b = 0;
    for (uint64_t t = 0; t < z; ++t) {
        const uint64_t l = len[t], p = pos[t];
        if (b >= n) return (int64_t)t + 1;
        if (l == 0) {
            if (p != s[b]) return (int64_t)t + 1;
            for (uint64_t q = 0; q < b; ++q)
                if (s[q] == s[b]) return (int64_t)t + 1; /* the byte occurs before: not maximal */
            b += 1;
            continue;
        }
        if (p >= b || b + l > n || match(s, n, p, b, l) != l) return (int64_t)t + 1;
        if (b + l < n)
            for (uint64_t q = 0; q < b; ++q)
                if (match(s, n, q, b, l + 1) == l + 1) return (int64_t)t + 1;
        b += l;
    }
    return b == n ? 0 : (int64_t)z + 1;
}

int checker_lz77_decode(const uint32_t *pos, const uint32_t *len, uint64_t z, uint64_t n, uint8_t *s) {
    if (z > n) return -1;
    uint64_t b = 0;
    for (uint64_t t = 0; t < z; ++t) { /* the rules first: s stays unwritten on a bad parse */
        if (len[t] == 0 && pos[t] > 255) return -1;
        if (len[t] != 0 && pos[t] >= b) return -1;
        b += len[t] ? len[t] : 1;
    }
    if (b != n) return -1;
    b = 0;
    for (uint64_t t = 0; t < z; ++t) {
        if (len[t] == 0) {
            s[b++] = (uint8_t)pos[t];
        } else {
            for (uint64_t k = 0; k < len[t]; ++k) s[b + k] = s[pos[t] + k];
            b += len[t];
        }
    }
    return 0;
}
