/*
 * oracle/sais.c -- CPU restatement of the reference's SA-IS suffix sorter.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under oracle/ is part of the product:
 * only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl
 * reference legs may load it, and only as the checker / the timed CPU arm.
 *
 * Follows (reference paths relative to /root/reference):
 *   src/DeltaQ.SuffixSorting.SAIS/SAIS.cs:25-42    SAIS.Sort (n<=1 short-circuit)
 *   src/DeltaQ.SuffixSorting.SAIS/SAIS.cs:52-71    GetCounts / GetBuckets
 *   src/DeltaQ.SuffixSorting.SAIS/SAIS.cs:75-133   LMS_sort
 *   src/DeltaQ.SuffixSorting.SAIS/SAIS.cs:135-217  LMS_post_proc
 *   src/DeltaQ.SuffixSorting.SAIS/SAIS.cs:219-274  InduceSA
 *   src/DeltaQ.SuffixSorting.SAIS/SAIS.cs:280-495  sais_main
 *   src/DeltaQ.SuffixSorting.SAIS/TextAccessor.cs:7-34 (byte text at level 0,
 *     int text in the recursion) -- here the `cs` (character size) argument.
 *
 * Parity pin: the reference holds no golden suffix array; its tests pin the
 * result by property (LibDivSufSortTests.cs:43-64, SAISChecker.cs:7-100) and
 * the suffix array of a byte string is unique, so this port is pinned by
 * oracle/sufcheck.c (the restated checkers) on the reference's 13 fixture
 * files and its random sizes (tests/test_oracle.py).
 */
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#define MIN_BUCKET_SIZE 256 /* SAIS.cs:49 */

typedef struct {
    const void *p;
    int cs; /* 1 = byte text, 4 = int text */
} text_t;

static inline int chr(text_t T, int i)
{
    return T.cs == 1 ? (int)((const uint8_t *)T.p)[i] : ((const int32_t *)T.p)[i];
}

/* SAIS.cs:52-60 */
static void get_counts(text_t T, int *c, int n, int k)
{
    memset(c, 0, (size_t)k * sizeof(int));
    for (int i = 0; i < n; ++i)
        c[chr(T, i)]++;
}

/* SAIS.cs:63-70 */
static void get_buckets(const int *c, int *b, int k, int end)
{
    int sum = 0;
    for (int i = 0; i < k; ++i) {
        int ci = c[i]; /* c and b may alias (flags & 8) */
        sum += ci;
        b[i] = end ? sum : sum - ci;
    }
}

/* SAIS.cs:75-133 */
static void lms_sort(text_t T, int *sa, int *c, int *b, int n, int k)
{
    int bb, i, j, c0, c1;

    if (c == b)
        get_counts(T, c, n, k);
    get_buckets(c, b, k, 0);

    j = n - 1;
    c1 = chr(T, j);
    bb = b[c1];
    --j;
    sa[bb++] = chr(T, j) < c1 ? ~j : j;
    for (i = 0; i < n; ++i) {
        j = sa[i];
        if (0 < j) {
            c0 = chr(T, j);
            if (c0 != c1) {
                b[c1] = bb;
                c1 = c0;
                bb = b[c1];
            }
            --j;
            sa[bb++] = chr(T, j) < c1 ? ~j : j;
            sa[i] = 0;
        } else if (j < 0) {
            sa[i] = ~j;
        }
    }

    if (c == b)
        get_counts(T, c, n, k);
    get_buckets(c, b, k, 1);

    c1 = 0;
    bb = b[c1];
    for (i = n - 1; 0 <= i; --i) {
        j = sa[i];
        if (0 < j) {
            c0 = chr(T, j);
            if (c0 != c1) {
                b[c1] = bb;
                c1 = c0;
                bb = b[c1];
            }
            --j;
            sa[--bb] = chr(T, j) > c1 ? ~(j + 1) : j;
            sa[i] = 0;
        }
    }
}

/* SAIS.cs:135-217 */
static int lms_post_proc(text_t T, int *sa, int n, int m)
{
    int i, j, p, q, qlen, name, c0, c1;

    for (i = 0; (p = sa[i]) < 0; ++i)
        sa[i] = ~p;
    if (i < m) {
        for (j = i, ++i;; ++i) {
            p = sa[i];
            if (p < 0) {
                sa[j++] = ~p;
                sa[i] = 0;
                if (j == m)
                    break;
            }
        }
    }

    /* lengths of the LMS substrings */
    i = n - 1;
    j = n - 1;
    c0 = chr(T, n - 1);
    do {
        c1 = c0;
    } while (0 <= --i && (c0 = chr(T, i)) >= c1);
    while (0 <= i) {
        do {
            c1 = c0;
        } while (0 <= --i && (c0 = chr(T, i)) <= c1);
        if (0 <= i) {
            sa[m + ((i + 1) >> 1)] = j - i;
            j = i + 1;
            do {
                c1 = c0;
            } while (0 <= --i && (c0 = chr(T, i)) >= c1);
        }
    }

    /* lexicographic names */
    for (i = 0, name = 0, q = n, qlen = 0; i < m; ++i) {
        p = sa[i];
        int plen = sa[m + (p >> 1)];
        int diff = 1;
        if (plen == qlen && q + plen < n) {
            for (j = 0; j < plen && chr(T, p + j) == chr(T, q + j); ++j) {
            }
            if (j == plen)
                diff = 0;
        }
        if (diff) {
            ++name;
            q = p;
            qlen = plen;
        }
        sa[m + (p >> 1)] = name;
    }
    return name;
}

/* SAIS.cs:219-274 */
static void induce_sa(text_t T, int *sa, int *c, int *b, int n, int k)
{
    int bb, i, j, c0, c1;

    if (c == b)
        get_counts(T, c, n, k);
    get_buckets(c, b, k, 0);

    j = n - 1;
    c1 = chr(T, j);
    bb = b[c1];
    sa[bb++] = (0 < j && chr(T, j - 1) < c1) ? ~j : j;
    for (i = 0; i < n; ++i) {
        j = sa[i];
        sa[i] = ~j;
        if (0 < j) {
            c0 = chr(T, --j);
            if (c0 != c1) {
                b[c1] = bb;
                c1 = c0;
                bb = b[c1];
            }
            sa[bb++] = (0 < j && chr(T, j - 1) < c1) ? ~j : j;
        }
    }

    if (c == b)
        get_counts(T, c, n, k);
    get_buckets(c, b, k, 1);

    c1 = 0;
    bb = b[c1];
    for (i = n - 1; 0 <= i; --i) {
        j = sa[i];
        if (0 < j) {
            c0 = chr(T, --j);
            if (c0 != c1) {
                b[c1] = bb;
                c1 = c0;
                bb = b[c1];
            }
            sa[--bb] = (j == 0 || chr(T, j - 1) > c1) ? ~j : j;
        } else {
            sa[i] = ~j;
        }
    }
}

/* SAIS.cs:280-495.  Returns 0, or -1 when a bucket allocation fails. */
static int sais_main(text_t T, int *sa, int fs, int n, int k)
{
    int *c, *b, *c_heap = NULL, *b_heap = NULL;
    int i, j, bb, m, name, c0, c1;
    unsigned flags;

    /* bucket-array placement, SAIS.cs:288-325 */
    if (k <= MIN_BUCKET_SIZE) {
        c = c_heap = (int *)malloc((size_t)k * sizeof(int));
        if (!c) return -1;
        if (k <= fs) {
            b = sa + (n + fs - k);
            flags = 1;
        } else {
            b = b_heap = (int *)malloc((size_t)k * sizeof(int));
            if (!b) { free(c_heap); return -1; }
            flags = 3;
        }
    } else if (k <= fs) {
        c = sa + (n + fs - k);
        if (k <= fs - k) {
            b = sa + (n + fs - k * 2);
            flags = 0;
        } else if (k <= MIN_BUCKET_SIZE * 4) {
            b = b_heap = (int *)malloc((size_t)k * sizeof(int));
            if (!b) return -1;
            flags = 2;
        } else {
            b = c;
            flags = 8;
        }
    } else {
        c = b = c_heap = (int *)malloc((size_t)k * sizeof(int));
        if (!c) return -1;
        flags = 4 | 8;
    }

    /* stage 1: sort all LMS substrings, SAIS.cs:327-382 */
    get_counts(T, c, n, k);
    get_buckets(c, b, k, 1);
    memset(sa, 0, (size_t)n * sizeof(int));

    bb = -1;
    i = n - 1;
    j = n;
    m = 0;
    c0 = chr(T, n - 1);
    do {
        c1 = c0;
    } while (0 <= --i && (c0 = chr(T, i)) >= c1);
    while (0 <= i) {
        do {
            c1 = c0;
        } while (0 <= --i && (c0 = chr(T, i)) <= c1);
        if (0 <= i) {
            if (0 <= bb)
                sa[bb] = j;
            bb = --b[c1];
            j = i;
            ++m;
            do {
                c1 = c0;
            } while (0 <= --i && (c0 = chr(T, i)) >= c1);
        }
    }
    if (1 < m) {
        lms_sort(T, sa, c, b, n, k);
        name = lms_post_proc(T, sa, n, m);
    } else if (m == 1) {
        sa[bb] = j + 1;
        name = 1;
    } else {
        name = 0;
    }

    /* stage 2: recurse when names are not unique, SAIS.cs:384-455 */
    if (name < m) {
        if (flags & 4) {
            free(c_heap);
            c_heap = NULL;
            c = b = NULL;
        }
        if (flags & 2) {
            free(b_heap);
            b_heap = NULL;
            b = NULL;
        }
        int newfs = n + fs - m * 2;
        if ((flags & (1 | 4 | 8)) == 0) {
            if (k + name <= newfs)
                newfs -= k;
            else
                flags |= 8;
        }
        for (i = m + (n >> 1) - 1, j = m * 2 + newfs - 1; m <= i; --i) {
            if (sa[i] != 0)
                sa[j--] = sa[i] - 1;
        }

        text_t R = { sa + m + newfs, 4 };
        if (sais_main(R, sa, newfs, m, name) != 0) {
            free(c_heap);
            free(b_heap);
            return -1;
        }

        i = n - 1;
        j = m * 2 - 1;
        c0 = chr(T, n - 1);
        do {
            c1 = c0;
        } while (0 <= --i && (c0 = chr(T, i)) >= c1);
        while (0 <= i) {
            do {
                c1 = c0;
            } while (0 <= --i && (c0 = chr(T, i)) <= c1);
            if (0 <= i) {
                sa[j--] = i + 1;
                do {
                    c1 = c0;
                } while (0 <= --i && (c0 = chr(T, i)) >= c1);
            }
        }
        for (i = 0; i < m; ++i)
            sa[i] = sa[m + sa[i]];
        if (flags & 4) {
            c = b = c_heap = (int *)malloc((size_t)k * sizeof(int));
            if (!c) return -1;
        }
        if (flags & 2) {
            b = b_heap = (int *)malloc((size_t)k * sizeof(int));
            if (!b) { free(c_heap); return -1; }
        }
    }

    /* stage 3: induce, SAIS.cs:457-494 */
    if (flags & 8)
        get_counts(T, c, n, k);
    if (1 < m) {
        get_buckets(c, b, k, 1);
        i = m - 1;
        j = n;
        int p = sa[m - 1];
        c1 = chr(T, p);
        do {
            c0 = c1;
            int q = b[c0];
            while (q < j)
                sa[--j] = 0;
            do {
                sa[--j] = p;
                if (--i < 0)
                    break;
                p = sa[i];
            } while ((c1 = chr(T, p)) == c0);
        } while (0 <= i);
        while (0 < j)
            sa[--j] = 0;
    }
    induce_sa(T, sa, c, b, n, k);

    free(c_heap);
    free(b_heap);
    return 0;
}

/*
 * ISuffixSort.Sort(text, suffixes) as SAIS.cs:25-42 implements it.
 * Returns 0 on success, -1 on allocation failure.  The length check of
 * SAIS.cs:27-30 is the caller's (one length is passed for both buffers).
 */
int oracle_sais(const uint8_t *text, int32_t n, int32_t *sa)
{
    if (n <= 1) {
        if (n == 1)
            sa[0] = 0;
        return 0;
    }
    text_t T = { text, 1 };
    return sais_main(T, sa, 0, n, 256);
}

/*
 * The same sorter on a text of int32 symbols in [0, k): the recursion's int
 * accessor at level 0.  oracle/search_rank.c sorts its generalized text
 * (old, separator, new, terminator) over 258 symbols with it.
 */
int oracle_sais_int(const int32_t *text, int32_t n, int32_t k, int32_t *sa)
{
    if (n <= 1) {
        if (n == 1)
            sa[0] = 0;
        return 0;
    }
    text_t T = { text, 4 };
    return sais_main(T, sa, 0, n, k);
}
