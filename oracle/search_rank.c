/*
 * oracle/search_rank.c -- Diff.Search's answer at every scan position, in
 * linear time.
 *
 * TEST INFRASTRUCTURE ONLY (see oracle/README.md).
 *
 * oracle_search_all (bsdiff.c) replays Diff.cs:267-298 literally and costs a
 * match length per binary-search step, so it is quadratic inside long matches.
 * This file computes the same table from ranks, and tests pin the two together
 * (tests/test_search_reference.py) so that the GPU search can be checked at
 * every position of inputs of many megabytes.
 *
 * Why ranks suffice.  Let L be the number of old suffixes that sort strictly
 * below q = new[scan..] in SequenceCompareTo order (bytes first, a prefix
 * before the longer string), and I = SA(old) followed by I[n] = 0
 * (Diff.cs:78,90).  The binary search keeps I[start] < q <= I[end] and ends on
 * e = max(L, 1), s = e - 1.  With x = MatchLength(old[I[s]..], q) and
 * y = MatchLength(old[I[e]..], q) it answers (I[s], x) if x > y, else
 * (I[e], y).  So only L and two match lengths are needed per position.
 *
 * How L and the match lengths are found.  The generalized text
 *     T = old[0..n) + 2, 1, new[scan_begin..m) + 2, 0
 * over 258 symbols is sorted with the oracle's SA-IS.  The separator 1 puts an
 * old suffix equal to a new suffix after it and a proper prefix of either kind
 * before the longer string, as compare_bytes does; old suffixes keep their
 * order in SA(old).  L of a query is the number of old entries before it.
 * Kasai's LCP over T never crosses the unique separators, so the running
 * minimum of the LCP since the previous old entry (forward sweep) is the match
 * with the predecessor I[L-1], and the running minimum up to the next old
 * entry (backward sweep) is the match with the successor I[L].  Two leaves are
 * not rank-adjacent to the query:
 *   L == 0: e = 1 holds SA(old)[1]; its match is min(match with SA(old)[0],
 *           LCP_old[1]);
 *   L == n: e = n holds the quirk I[n] = 0, old suffix 0 at rank r0; its match
 *           is min(match with SA(old)[n-1], min LCP_old over (r0, n-1]).
 * n == 0 gives (0, 0) everywhere.
 *
 * Memory: four int32 arrays of n + (m - scan_begin) + 2 entries.
 */
#include <stdint.h>
#include <stdlib.h>

int oracle_sais_int(const int32_t *text, int32_t n, int32_t k, int32_t *sa);

static void lcp_kasai_int(const int32_t *T, int32_t N, const int32_t *SA, int32_t *rank, int32_t *LCP)
{
    for (int32_t r = 0; r < N; ++r)
        rank[SA[r]] = r;
    int32_t h = 0;
    for (int32_t i = 0; i < N; ++i) {
        int32_t r = rank[i];
        if (r == 0) {
            LCP[0] = 0;
            h = 0;
            continue;
        }
        int32_t j = SA[r - 1];
        while (i + h < N && j + h < N && T[i + h] == T[j + h])
            ++h;
        LCP[r] = h;
        if (h > 0)
            --h;
    }
}

static inline int32_t min32(int32_t a, int32_t b) { return a < b ? a : b; }

/*
 * Diff.Search(I, old, new[scan..], 0, n) for scan in [scan_begin, scan_begin + count), I = SA(old) + [0]:
 * the same (pos, len) as oracle_search_all.  Returns 0, -1 on bad arguments or a text over 2^31 - 1 symbols,
 * -2 on allocation failure.
 */
int oracle_search_table(const uint8_t *old, int32_t n, const uint8_t *nw, int32_t m,
                        int32_t scan_begin, int32_t count, int32_t *pos_out, int32_t *len_out)
{
    if (n < 0 || m < 0 || scan_begin < 0 || count < 0 || (int64_t)scan_begin + count > m)
        return -1;
    if (count == 0)
        return 0;
    if (n == 0) {
        for (int32_t j = 0; j < count; ++j)
            pos_out[j] = len_out[j] = 0;
        return 0;
    }
    int64_t N64 = (int64_t)n + (m - scan_begin) + 2;
    if (N64 > INT32_MAX)
        return -1;
    int32_t N = (int32_t)N64, q0 = n + 1;
    int32_t *T = malloc(sizeof(int32_t) * (size_t)N);
    int32_t *sa = malloc(sizeof(int32_t) * (size_t)N);
    int32_t *rank = malloc(sizeof(int32_t) * (size_t)N);
    int32_t *lcp = malloc(sizeof(int32_t) * (size_t)N);
    int rc = -2;
    if (!T || !sa || !rank || !lcp)
        goto out;
    for (int32_t i = 0; i < n; ++i)
        T[i] = old[i] + 2;
    T[n] = 1;
    for (int32_t i = scan_begin; i < m; ++i)
        T[q0 + i - scan_begin] = nw[i] + 2;
    T[N - 1] = 0;
    if (oracle_sais_int(T, N, 258, sa) != 0)
        goto out;
    lcp_kasai_int(T, N, sa, rank, lcp);

    /* T and rank are no longer needed: they hold SA(old) and LCP_old (n <= N entries each) */
    int32_t *sa_old = rank, *lcp_old = T;
    int32_t L = 0, r0 = 0, run = INT32_MAX;
    for (int32_t r = 0; r < N; ++r) {               /* forward: L and the match with the predecessor */
        int32_t i = sa[r];
        run = min32(run, lcp[r]);
        if (i < n) {
            lcp_old[L] = L ? run : 0;
            sa_old[L] = i;
            if (i == 0)
                r0 = L;
            ++L;
            run = INT32_MAX;
        } else if (i >= q0 && i - q0 < count) {
            pos_out[i - q0] = L;
            len_out[i - q0] = run;                  /* meaningless when L == 0; not read then */
        }
    }
    int32_t m0 = INT32_MAX;                          /* min LCP_old over (r0, n-1] */
    for (int32_t k = r0 + 1; k < n; ++k)
        m0 = min32(m0, lcp_old[k]);

    run = 0;                                         /* backward: the match with the successor, then the answer */
    for (int32_t r = N - 1; r >= 0; --r) {
        int32_t i = sa[r];
        if (i < n) {
            run = lcp[r];
            continue;
        }
        if (i >= q0 && i - q0 < count) {
            int32_t j = i - q0, Lq = pos_out[j], pm = len_out[j], sm = run;   /* sm is meaningless when Lq == n */
            int32_t e = Lq > 1 ? Lq : 1;
            int32_t ps = Lq ? sa_old[Lq - 1] : sa_old[0];
            int32_t x = Lq ? pm : sm;
            int32_t pe, y;
            if (e == n) {
                pe = 0;
                y = Lq == n ? min32(pm, m0) : sm;  /* Lq < n here only for n == 1, where old suffix 0 is the successor */
            } else if (e == Lq) {
                pe = sa_old[Lq];
                y = sm;
            } else {                                 /* Lq == 0, e == 1 < n */
                pe = sa_old[1];
                y = min32(sm, lcp_old[1]);
            }
            if (x > y) {
                pos_out[j] = ps;
                len_out[j] = x;
            } else {
                pos_out[j] = pe;
                len_out[j] = y;
            }
        }
        run = min32(run, lcp[r]);
    }
    rc = 0;
out:
    free(T);
    free(sa);
    free(rank);
    free(lcp);
    return rc;
}
