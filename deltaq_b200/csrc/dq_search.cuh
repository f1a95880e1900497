// dq_search.cuh -- the bsdiff match search: Diff.Search for EVERY scan position of `new`, bit-exact.
//
// Reference: /root/reference/src/DeltaQ.BsDiff/Diff.cs:267-298 (Search), :245-246 (CompareBytes =
// Span.SequenceCompareTo), :249-265 (MatchLength), call site :106 with start = 0, end = n, I[n] == 0.
//
// The reference's result is a pure function of L = #{old suffixes < query} (SURVEY.md section 0): the leaf it
// reaches is (start, end) = (max(L,1)-1, max(L,1)), and it returns the longer of the two matches there
// (ties -> end).  A literal per-position replay costs O(match length) per probe, i.e. quadratic work inside
// unchanged regions that the reference's greedy loop hops over (scan += len, Diff.cs:104).  These kernels
// compute the same L -- and the same two match lengths -- for all positions with amortised O(1) probes:
//
//   * if the query at j matched old suffix p for l bytes, the query at j+s matches suffix p+s for exactly
//     l-s bytes and lies on the same side of it, so rank ISA[p+s] is an exact anchor for j+s;
//   * from an anchor, L is found by walking the suffix array with the LCP array of `old`
//     (LCP[r] = lcp(SA[r-1], SA[r])): a neighbour that shares less than the anchor does with the query is
//     decided without touching the text, one that shares more is skipped (64- and 4096-rank block minima
//     skip whole blocks), and only an exact tie extends the byte comparison from where it stopped;
//   * chains of `kChunk` consecutive positions are walked by one thread; their heads are produced by a
//     stride-kChunk chain, and only every kChunk^2-th position is searched from scratch (binary search with
//     Manber-Myers lcp skipping).  The LCP array itself is built by the same two-level chaining (Kasai's
//     PLCP[i+1] >= PLCP[i]-1 along the text).
#pragma once
#include "dq_common.cuh"
#include "dq_suffix.cuh"

namespace dq {
namespace search {

#ifndef DQ_SEARCH_CHUNK
#define DQ_SEARCH_CHUNK 32
#endif
constexpr int kChunk = DQ_SEARCH_CHUNK; // positions per chain
#ifndef DQ_SEARCH_HEADS
#define DQ_SEARCH_HEADS 64
#endif
constexpr int kHeads = DQ_SEARCH_HEADS;  // chain heads walked by one warp of the head kernels
constexpr int kSuper = kChunk * kHeads; // positions per from-scratch search
constexpr int kThreads = 128;
constexpr uint32_t kNone = 0xffffffffu;

#ifdef DQ_EMU
struct DebugCounters { unsigned long long scratch, probes, cmp_bytes, walk, walk_max, anchors, thr_max[4], thr_hist[4][24]; };
inline DebugCounters g_dbg;
#define DQ_DBG(x) x
#else
#define DQ_DBG(x)
#endif

#ifdef DQ_PROF
// debug build only (scripts/prof_chains.py): clocks / bytes a warp spends inside common_prefix_warp (reset by the level-A
// launch of search_heads_kernel, so they describe that launch)
__device__ unsigned long long g_prof_cmp_clk[1u << 16];
__device__ unsigned long long g_prof_cmp_bytes[1u << 16];
__device__ unsigned int g_prof_cmp_calls[1u << 16];
#endif

// 8 bytes at an arbitrary address; the buffers are padded so that reading up to 16 bytes past p is safe
__device__ __forceinline__ uint64_t load64u(const uint8_t *p)
{
    const uintptr_t a = reinterpret_cast<uintptr_t>(p);
    const uint64_t *w = reinterpret_cast<const uint64_t *>(a & ~(uintptr_t)7);
    const unsigned sh = (unsigned)(a & 7u) * 8u;
    // no branch on the alignment: both words are always read, so the loads of several calls can all be in flight
    // before the first result is needed (the warp-cooperative comparison issues up to 64 of them per lane)
    const uint64_t lo = __ldg(w);
    const uint64_t hi = __ldg(w + 1);
    return (lo >> sh) | (sh ? (hi << ((64u - sh) & 63u)) : 0ull);
}

// number of equal leading bytes of a[0..la) and b[0..lb).  Both buffers are readable (zero padded) for 64
// bytes past their ends.  Short matches leave after one unaligned 8-byte step; long ones run a loop that
// consumes 32 bytes per iteration with `a` word-aligned and `b` realigned through a carried word.
__device__ __forceinline__ uint32_t common_prefix(const uint8_t *a, uint32_t la, const uint8_t *b, uint32_t lb)
{
    const uint32_t lim = min(la, lb);
    if (lim == 0) return 0;
    DQ_DBG(g_dbg.cmp_bytes += 8;)
    {
        const uint64_t x = load64u(a) ^ load64u(b);
        if (x) return min((uint32_t)(__ffsll((long long)x) - 1) >> 3, lim);
        if (lim <= 8) return lim;
    }
    // the first 8 bytes agree: restart at the first 8-aligned byte of a (1..8 bytes in)
    uint32_t k = 8u - (uint32_t)(reinterpret_cast<uintptr_t>(a) & 7u);
    const uint64_t *pa = reinterpret_cast<const uint64_t *>(a + k);
    const uintptr_t ab = reinterpret_cast<uintptr_t>(b + k);
    const uint64_t *pb = reinterpret_cast<const uint64_t *>(ab & ~(uintptr_t)7);
    const unsigned sh = (unsigned)(ab & 7u) * 8u;
    if (sh == 0) {
        while (k < lim) {
            DQ_DBG(g_dbg.cmp_bytes += 32;)
            const uint64_t x0 = __ldg(pa) ^ __ldg(pb), x1 = __ldg(pa + 1) ^ __ldg(pb + 1);
            const uint64_t x2 = __ldg(pa + 2) ^ __ldg(pb + 2), x3 = __ldg(pa + 3) ^ __ldg(pb + 3);
            if (x0 | x1 | x2 | x3) {
                uint32_t off;
                uint64_t x;
                if (x0) { off = 0; x = x0; } else if (x1) { off = 8; x = x1; } else if (x2) { off = 16; x = x2; } else { off = 24; x = x3; }
                return min(k + off + ((uint32_t)(__ffsll((long long)x) - 1) >> 3), lim);
            }
            k += 32;
            pa += 4;
            pb += 4;
        }
    } else {
        uint64_t carry = __ldg(pb);
        const unsigned rs = 64u - sh;
        while (k < lim) {
            DQ_DBG(g_dbg.cmp_bytes += 32;)
            const uint64_t w1 = __ldg(pb + 1), w2 = __ldg(pb + 2), w3 = __ldg(pb + 3), w4 = __ldg(pb + 4);
            const uint64_t x0 = __ldg(pa) ^ ((carry >> sh) | (w1 << rs));
            const uint64_t x1 = __ldg(pa + 1) ^ ((w1 >> sh) | (w2 << rs));
            const uint64_t x2 = __ldg(pa + 2) ^ ((w2 >> sh) | (w3 << rs));
            const uint64_t x3 = __ldg(pa + 3) ^ ((w3 >> sh) | (w4 << rs));
            if (x0 | x1 | x2 | x3) {
                uint32_t off;
                uint64_t x;
                if (x0) { off = 0; x = x0; } else if (x1) { off = 8; x = x1; } else if (x2) { off = 16; x = x2; } else { off = 24; x = x3; }
                return min(k + off + ((uint32_t)(__ffsll((long long)x) - 1) >> 3), lim);
            }
            carry = w4;
            k += 32;
            pa += 4;
            pb += 4;
        }
    }
    return lim;
}

// warp-cooperative version: all 32 lanes call it with the same arguments and get the same result.  The first
// step compares 256 bytes (lane l takes the 8 bytes at 8l) so that short matches cost one round trip; the next one
// 1 KiB; long matches then continue 4 KiB per step (sixteen independent 8-byte words per lane per stream in flight:
// a warp inside a repeat of R bytes is bound by round trips, R / 4 KiB of them).
template <int kWords>
__device__ __forceinline__ bool common_prefix_warp_step(const uint8_t *a, const uint8_t *b, uint32_t k, uint32_t lim,
                                                        uint32_t *result)
{
    // word w of lane l covers bytes k + 256w + 8l: each of the loads of a warp is one coalesced 256 B row
    const uint32_t lane = lane_id();
    // Every load is issued unconditionally (offsets past the end are clamped to lim: the buffers are readable there)
    // and masked afterwards.  A conditional load puts each word into its own divergence region, the compiler waits
    // for it before entering the next one, and the warp moves 256 bytes per round trip instead of 256 * kWords
    // (measured: 0.64 GB/s per warp, profiles/r01_search_chain_timing.md).
    uint64_t x[kWords];
#pragma unroll
    for (int w = 0; w < kWords; ++w) {
        const uint32_t off = k + 256u * w + lane * 8u;
        const uint32_t at = min(off, lim);
        x[w] = load64u(a + at) ^ load64u(b + at);
    }
#pragma unroll
    for (int w = 0; w < kWords; ++w)
        if (k + 256u * w + lane * 8u >= lim) x[w] = 0ull;
    DQ_DBG(g_dbg.cmp_bytes += 8 * kWords;)
#pragma unroll
    for (int w = 0; w < kWords; ++w) {
        const unsigned m = __ballot_sync(kFullMask, x[w] != 0);
        if (m) {
            const int first = __ffs((int)m) - 1;
            const uint64_t xx = __shfl_sync(kFullMask, x[w], first);
            *result = min(k + 256u * w + (uint32_t)first * 8u + ((uint32_t)(__ffsll((long long)xx) - 1) >> 3), lim);
            return true;
        }
    }
    return false;
}

__device__ __forceinline__ uint32_t common_prefix_warp(const uint8_t *a, uint32_t la, const uint8_t *b, uint32_t lb)
{
    const uint32_t lim = min(la, lb);
    if (lim == 0) return 0;
#ifdef DQ_PROF
    const long long pt0 = clock64();
    struct PF { long long t0; uint32_t *res; __device__ ~PF() { const uint32_t w = (uint32_t)((((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5) & 0xffffu); if (lane_id() == 0) { g_prof_cmp_clk[w] += (unsigned long long)(clock64() - t0); g_prof_cmp_bytes[w] += *res; g_prof_cmp_calls[w] += 1; } } };
    uint32_t r = lim;
    PF pf{pt0, &r};
#else
    uint32_t r;
#endif
    if (common_prefix_warp_step<1>(a, b, 0, lim, &r)) return r;
    if (lim <= 256) return r = lim;
    if (common_prefix_warp_step<4>(a, b, 256, lim, &r)) return r;
    for (uint32_t k = 1280; k < lim; k += 4096)
        if (common_prefix_warp_step<16>(a, b, k, lim, &r)) return r;
    return r = lim;
}

template <bool WARP>
__device__ __forceinline__ uint32_t common_prefix_t(const uint8_t *a, uint32_t la, const uint8_t *b, uint32_t lb)
{
    if (WARP) return common_prefix_warp(a, la, b, lb);
    return common_prefix(a, la, b, lb);
}

struct Texts {
    const uint8_t *old_;
    const uint8_t *new_;
    uint32_t n, m;
    // run_end arrays of both texts (dq_suffix.cuh), or nullptr: lets a comparison jump over an equal-byte run that
    // both sides are inside of (zero padding) instead of reading it
    const uint32_t *run_old = nullptr;
    const uint32_t *run_new = nullptr;
};

// lcp of old suffix p with the query at j, given that the first `known` bytes agree; *less = (suffix < query)
// under Span.SequenceCompareTo: first differing byte, else the shorter one is smaller.
template <bool WARP = false>
__device__ __forceinline__ uint32_t match_from(const Texts &t, uint32_t p, uint32_t j, uint32_t known, bool *less)
{
    const uint32_t la = t.n - p, lq = t.m - j;
    if (t.run_old && la - known >= 8 && lq - known >= 8) {
        const uint64_t wa = load64u(t.old_ + p + known), wb = load64u(t.new_ + j + known);
        if (wa == wb && wa == (wa & 0xffull) * 0x0101010101010101ull) {
            const uint32_t a0 = p + known, b0 = j + known;
            known += min(t.run_old[a0] - a0, t.run_new[b0] - b0);  // >= 8: both runs cover the word just read
        }
    }
    const uint32_t c = known + common_prefix_t<WARP>(t.old_ + p + known, la - known, t.new_ + j + known, lq - known);
    if (c == la)
        *less = c < lq;
    else if (c == lq)
        *less = false;
    else
        *less = t.old_[p + c] < t.new_[j + c];
    return c;
}

constexpr int kMaxLevels = 6;  // 64^5 > 2^30: enough block-minimum levels for any int32-sized input

struct Index {
    const int32_t *SA;    // n
    const uint32_t *ISA;  // n
    // lv[0] = LCP (n entries, LCP[0] = 0); lv[k] = minima of lv[k-1] over blocks of 64 (size[k] entries)
    const uint32_t *lv[kMaxLevels];
    uint32_t size[kMaxLevels];
    int top;              // highest level in use
    // 2-byte prefix buckets: ranks [bkt_lo[k], bkt_hi[k]) hold exactly the suffixes (>= 2 bytes long) that
    // start with the byte pair k
    const uint32_t *bkt_lo, *bkt_hi;
    // 3-byte prefix table (prefix3_* kernels below), or nullptr: pre3[k] = number of suffixes whose first three bytes
    // (zero padded for the two suffixes shorter than that), read as a big-endian number, are < k (k in [0, 2^24]) --
    // also their ranks, because a shorter suffix sorts in front of everything its padded value could tie with.
    // pre3[2^24 + 1] and [2^24 + 2] hold the padded values of the 1-byte and the 2-byte suffix (kNone if n is too short
    // to have them).  Ranks [lo, hi) = [pre3[k] + a, pre3[k+1]), a = how many of those two values are == k, hold exactly
    // the suffixes (>= 3 bytes long) that start with k.
    const uint32_t *pre3;
};

constexpr uint32_t kPrefix3Bins = 1u << 24;

#ifdef DQ_PROF
// debug build only (scripts/prof_chains.py): elapsed clocks / 64 of every chain of the last search_chain_kernel and
// of every warp of the last search_heads_kernel launch
__device__ uint32_t g_prof_chain[1u << 21];
__device__ uint32_t g_prof_heads[1u << 16];
__device__ uint32_t g_prof_seeds[1u << 16];
#endif

// rank interval of the suffixes that start with the three bytes at q (see Index::pre3)
__device__ __forceinline__ void prefix3_bounds(const Index &ix, const uint8_t *q, uint32_t *lo, uint32_t *hi)
{
    const uint32_t k = ((uint32_t)q[0] << 16) | ((uint32_t)q[1] << 8) | q[2];
    const uint32_t a = (uint32_t)(ix.pre3[kPrefix3Bins + 1] == k) + (uint32_t)(ix.pre3[kPrefix3Bins + 2] == k);
    *lo = ix.pre3[k] + a;
    *hi = ix.pre3[k + 1];
}

struct Bracket {
    uint32_t L;  // #{old suffixes < query}
    uint32_t x;  // lcp(query, suffix SA[L-1])   (valid when L > 0)
    uint32_t y;  // lcp(query, suffix SA[L])     (valid when L < n)
    // SA[L-1] / SA[L] when the search already knows them (kNone otherwise): the common anchored step then needs
    // no read of SA at all (ISA and LCP only) -- the chain kernel is bound by random 32-byte sectors
    uint32_t sx = kNone, sy = kNone;
};

// binary search from scratch, with Manber-Myers skipping of the bytes both ends are known to share.  The
// first two query bytes select a bucket of the suffix array, so ~16 of the ~log2(n) probes are a table read.
// BKT = false: the index has no bucket or prefix tables (a batch chunk's pairs), the search spans all n ranks.
template <bool WARP = false, bool BKT = true>
__device__ __forceinline__ Bracket locate_scratch(const Texts &t, const Index &ix, uint32_t j)
{
    DQ_DBG(g_dbg.scratch++;)
    const uint32_t n = t.n;
    int64_t lo = -1, hi = n;
    uint32_t llo = 0, lhi = 0;
    bool lo_virtual = true, hi_virtual = true;  // bounds not yet compared with the query
    if (BKT && ix.pre3 && t.m - j >= 3) {
        uint32_t b_lo, b_hi;
        prefix3_bounds(ix, t.new_ + j, &b_lo, &b_hi);
        lo = (int64_t)b_lo - 1;
        hi = b_hi;
        llo = lhi = 3;  // every suffix strictly inside shares the three bytes
    } else if (BKT && t.m - j >= 2) {
        const uint32_t k = ((uint32_t)t.new_[j] << 8) | t.new_[j + 1];
        lo = (int64_t)ix.bkt_lo[k] - 1;
        hi = ix.bkt_hi[k];
        llo = lhi = 2;  // every suffix strictly inside shares the byte pair
    } else {
        lo_virtual = hi_virtual = false;
    }
    while (hi - lo > 1) {
        DQ_DBG(g_dbg.probes++;)
        const uint32_t mid = (uint32_t)((lo + hi) >> 1);
        bool less;
        const uint32_t c = match_from<WARP>(t, (uint32_t)ix.SA[mid], j, min(llo, lhi), &less);
        if (less) {
            lo = mid;
            llo = c;
            lo_virtual = false;
        } else {
            hi = mid;
            lhi = c;
            hi_virtual = false;
        }
    }
    // bucket bounds were never compared: their true lcp with the query is 0 or 1 byte
    bool dummy;
    if (lo_virtual) llo = lo >= 0 ? match_from<WARP>(t, (uint32_t)ix.SA[lo], j, 0, &dummy) : 0u;
    if (hi_virtual) lhi = hi < (int64_t)n ? match_from<WARP>(t, (uint32_t)ix.SA[hi], j, 0, &dummy) : 0u;
    return Bracket{(uint32_t)hi, llo, lhi};
}

// One probe of a from-scratch search whose 8 bytes of `old` past the known prefix (wa) are already in a register: the
// common case in unrelated data -- a mismatch inside those 8 bytes, or one side ending there -- is decided at once;
// anything longer goes through match_from.  Same result as match_from(t, p, j, known, less).
__device__ __forceinline__ uint32_t match_quick(const Texts &t, uint32_t p, uint64_t wa, uint32_t j, uint32_t known, bool *less)
{
    const uint32_t la = t.n - p, lq = t.m - j;
    const uint32_t rem = min(la, lq) - known;
    const uint64_t wb = load64u(t.new_ + j + known);
    const uint64_t x = wa ^ wb;
    const uint32_t nb = x ? ((uint32_t)(__ffsll((long long)x) - 1) >> 3) : 8u;
    if (nb < 8 && nb < rem) {
        *less = (uint32_t)((wa >> (8 * nb)) & 0xffu) < (uint32_t)((wb >> (8 * nb)) & 0xffu);
        return known + nb;
    }
    if (rem <= 8) {  // all rem bytes agree and one side ends there
        const uint32_t c = known + rem;
        *less = c == la ? c < lq : false;
        return c;
    }
    return match_from(t, p, j, known + 8, less);
}

// kB independent from-scratch searches (queries j0 .. j0+kB-1) with their probes interleaved: the kB reads of SA and
// then the kB reads of `old` of one round are in flight together, so a round costs two round trips for all of them
// instead of two each.  out[i] is what locate_scratch(t, ix, j0 + i) returns, plus the neighbours' suffixes when seen.
template <int kB, bool BKT = true>
__device__ __forceinline__ void locate_scratch_batch(const Texts &t, const Index &ix, uint32_t j0, Bracket *out)
{
    const uint32_t n = t.n;
    int32_t lo[kB], hi[kB];
    uint32_t llo[kB], lhi[kB], plo[kB], phi[kB];
    uint32_t lo_virtual = 0, hi_virtual = 0;  // bit i: bound of search i not yet compared with its query
#pragma unroll
    for (int i = 0; i < kB; ++i) {
        const uint32_t j = j0 + i;
        lo[i] = -1;
        hi[i] = (int32_t)n;
        llo[i] = lhi[i] = 0;
        plo[i] = phi[i] = kNone;
        if (BKT && ix.pre3 && t.m - j >= 3) {
            uint32_t b_lo, b_hi;
            prefix3_bounds(ix, t.new_ + j, &b_lo, &b_hi);
            lo[i] = (int32_t)b_lo - 1;
            hi[i] = (int32_t)b_hi;
            llo[i] = lhi[i] = 3;
            lo_virtual |= 1u << i;
            hi_virtual |= 1u << i;
        } else if (BKT && t.m - j >= 2) {
            const uint32_t k = ((uint32_t)t.new_[j] << 8) | t.new_[j + 1];
            lo[i] = (int32_t)ix.bkt_lo[k] - 1;
            hi[i] = (int32_t)ix.bkt_hi[k];
            llo[i] = lhi[i] = 2;
            lo_virtual |= 1u << i;
            hi_virtual |= 1u << i;
        }
    }
    for (;;) {
        uint32_t active = 0, p[kB];
        uint64_t wa[kB];
#pragma unroll
        for (int i = 0; i < kB; ++i) {
            p[i] = 0;
            if (hi[i] - lo[i] > 1) {
                active |= 1u << i;
                p[i] = (uint32_t)ix.SA[lo[i] + ((hi[i] - lo[i]) >> 1)];
            }
        }
        if (!active) break;
#pragma unroll
        for (int i = 0; i < kB; ++i) wa[i] = load64u(t.old_ + p[i] + min(llo[i], lhi[i]));
#pragma unroll
        for (int i = 0; i < kB; ++i) {
            if (!(active >> i & 1u)) continue;
            DQ_DBG(g_dbg.probes++;)
            bool less;
            const uint32_t c = match_quick(t, p[i], wa[i], j0 + i, min(llo[i], lhi[i]), &less);
            const int32_t mid = lo[i] + ((hi[i] - lo[i]) >> 1);
            if (less) {
                lo[i] = mid;
                llo[i] = c;
                plo[i] = p[i];
                lo_virtual &= ~(1u << i);
            } else {
                hi[i] = mid;
                lhi[i] = c;
                phi[i] = p[i];
                hi_virtual &= ~(1u << i);
            }
        }
    }
    // bucket bounds that were never compared: their true lcp with the query is at most the bucket's prefix minus one
    uint64_t wl[kB], wh[kB];
#pragma unroll
    for (int i = 0; i < kB; ++i) {
        if ((lo_virtual >> i & 1u) && lo[i] >= 0) plo[i] = (uint32_t)ix.SA[lo[i]];
        if ((hi_virtual >> i & 1u) && hi[i] < (int32_t)n) phi[i] = (uint32_t)ix.SA[hi[i]];
    }
#pragma unroll
    for (int i = 0; i < kB; ++i) {
        wl[i] = ((lo_virtual >> i & 1u) && lo[i] >= 0) ? load64u(t.old_ + plo[i]) : 0ull;
        wh[i] = ((hi_virtual >> i & 1u) && hi[i] < (int32_t)n) ? load64u(t.old_ + phi[i]) : 0ull;
    }
#pragma unroll
    for (int i = 0; i < kB; ++i) {
        bool dummy;
        if (lo_virtual >> i & 1u) llo[i] = lo[i] >= 0 ? match_quick(t, plo[i], wl[i], j0 + i, 0, &dummy) : 0u;
        if (hi_virtual >> i & 1u) lhi[i] = hi[i] < (int32_t)n ? match_quick(t, phi[i], wh[i], j0 + i, 0, &dummy) : 0u;
        out[i] = Bracket{(uint32_t)hi[i], llo[i], lhi[i], lo[i] >= 0 ? plo[i] : kNone, hi[i] < (int32_t)n ? phi[i] : kNone};
    }
}

// locate_scratch that gives up (*aborted) as soon as one probe shares `cap` more bytes than known with the query:
// the cheap, fully parallel first pass of the head kernel -- queries inside long matches abort after a few
// probes and are left to the inheriting pass, queries in unrelated data (short matches) finish here.
template <bool BKT = true>
__device__ __forceinline__ Bracket locate_scratch_capped(const Texts &t, const Index &ix, uint32_t j, uint32_t cap,
                                                         bool *aborted)
{
    const uint32_t n = t.n;
    int64_t lo = -1, hi = n;
    uint32_t llo = 0, lhi = 0;
    bool lo_virtual = true, hi_virtual = true;
    *aborted = false;
    if (BKT && ix.pre3 && t.m - j >= 3) {
        uint32_t b_lo, b_hi;
        prefix3_bounds(ix, t.new_ + j, &b_lo, &b_hi);
        lo = (int64_t)b_lo - 1;
        hi = b_hi;
        llo = lhi = 3;
    } else if (BKT && t.m - j >= 2) {
        const uint32_t k = ((uint32_t)t.new_[j] << 8) | t.new_[j + 1];
        lo = (int64_t)ix.bkt_lo[k] - 1;
        hi = ix.bkt_hi[k];
        llo = lhi = 2;
    } else {
        lo_virtual = hi_virtual = false;
    }
    const uint32_t lq = t.m - j;
    auto probe = [&](uint32_t p, uint32_t known, bool *less) -> uint32_t {
        const uint32_t la = n - p;
        const uint32_t ra = la - known, rq = lq - known;
        const uint32_t c = known + common_prefix(t.old_ + p + known, min(ra, cap), t.new_ + j + known, min(rq, cap));
        if (c - known >= cap && ra > cap && rq > cap) {
            *aborted = true;
            return c;
        }
        if (c == la)
            *less = c < lq;
        else if (c == lq)
            *less = false;
        else
            *less = t.old_[p + c] < t.new_[j + c];
        return c;
    };
    while (hi - lo > 1) {
        const uint32_t mid = (uint32_t)((lo + hi) >> 1);
        bool less = false;
        const uint32_t c = probe((uint32_t)ix.SA[mid], min(llo, lhi), &less);
        if (*aborted) return Bracket{0, 0, 0};
        if (less) {
            lo = mid;
            llo = c;
            lo_virtual = false;
        } else {
            hi = mid;
            lhi = c;
            hi_virtual = false;
        }
    }
    bool dummy = false;
    if (lo_virtual) llo = lo >= 0 ? probe((uint32_t)ix.SA[lo], 0, &dummy) : 0u;
    if (hi_virtual) lhi = hi < (int64_t)n ? probe((uint32_t)ix.SA[hi], 0, &dummy) : 0u;
    if (*aborted) return Bracket{0, 0, 0};
    return Bracket{(uint32_t)hi, llo, lhi};
}

// first u >= u0 with LCP[u] < c, or n: climbs the block-minimum hierarchy, at most 63 steps per level
__device__ __forceinline__ uint32_t next_smaller(const Index &ix, uint32_t u0, uint32_t c)
{
    int l = 0;
    uint32_t idx = u0;
    for (;;) {
        DQ_DBG(g_dbg.walk++;)
        if (idx >= ix.size[l]) return ix.size[0];
        if ((idx & 63u) == 0 && l < ix.top) {  // block aligned: the block starting here, one level up
            idx >>= 6;
            ++l;
            continue;
        }
        if (ix.lv[l][idx] < c) break;
        ++idx;
    }
    while (l > 0) {
        --l;
        idx <<= 6;
        const uint32_t *A = ix.lv[l];
        while (A[idx] >= c) {
            DQ_DBG(g_dbg.walk++;)
            ++idx;
        }
    }
    return idx;
}

// last u <= u0 with LCP[u] < c (c > 0, so u = 0 always qualifies)
__device__ __forceinline__ uint32_t prev_smaller(const Index &ix, uint32_t u0, uint32_t c)
{
    int l = 0;
    uint32_t idx = u0;
    for (;;) {
        const uint32_t *A = ix.lv[l];
        bool found = false;
        for (;;) {
            DQ_DBG(g_dbg.walk++;)
            if (A[idx] < c) {
                found = true;
                break;
            }
            if ((idx & 63u) == 0 && l < ix.top) break;
            --idx;  // cannot underflow: entry 0 of every level is 0 < c
        }
        if (found) break;
        idx = (idx >> 6) - 1;  // the block before this one, one level up
        ++l;
    }
    while (l > 0) {
        --l;
        idx = min(idx * 64u + 63u, ix.size[l] - 1u);
        const uint32_t *A = ix.lv[l];
        while (A[idx] >= c) {
            DQ_DBG(g_dbg.walk++;)
            --idx;
        }
    }
    return idx;
}

constexpr uint32_t kMinAnchor = 3;  // anchors sharing fewer bytes name intervals so wide that scratch is cheaper

// anchor: rank r whose suffix shares exactly c bytes with the query and is (less ? < : >=) the query.
// All suffixes sharing >= c bytes with suffix r form one contiguous rank interval (delimited by LCP < c);
// the query sorts inside it, so L is found by a binary search over that interval only, every probe
// starting at byte c.
template <bool WARP = false, bool BKT = true>
__device__ __forceinline__ Bracket locate_anchor(const Texts &t, const Index &ix, uint32_t j, uint32_t r, uint32_t c,
                                                 bool less, uint32_t anchor_suffix = kNone)
{
    const uint32_t n = t.n;
    const uint32_t *LCP = ix.lv[0];
    DQ_DBG(g_dbg.anchors++;)
    if (c < kMinAnchor) return locate_scratch<WARP, BKT>(t, ix, j);
    if (less) {
        if (r + 1 >= n) return Bracket{n, c, 0};
        const uint32_t g = LCP[r + 1];
        if (g < c) return Bracket{r + 1, c, g, anchor_suffix, kNone};
        const uint32_t e = next_smaller(ix, r + 1, c);  // interval is [.., e)
        uint32_t lo = r, hi = e, llo = c, lhi = c;
        bool boundary = true;
        while (hi - lo > 1) {
            DQ_DBG(g_dbg.probes++;)
            const uint32_t mid = lo + ((hi - lo) >> 1);
            bool ls;
            const uint32_t cc = match_from<WARP>(t, (uint32_t)ix.SA[mid], j, min(llo, lhi), &ls);
            if (ls) {
                lo = mid;
                llo = cc;
            } else {
                hi = mid;
                lhi = cc;
                boundary = false;
            }
        }
        return Bracket{hi, llo, boundary ? (e < n ? LCP[e] : 0u) : lhi};
    } else {
        if (r == 0) return Bracket{0, 0, c};
        const uint32_t g = LCP[r];
        if (g < c) return Bracket{r, g, c, kNone, anchor_suffix};
        const uint32_t s = prev_smaller(ix, r, c);  // interval is [s, ..]; suffix s-1 (if any) is < query
        int64_t lo = (int64_t)s - 1, hi = r;
        uint32_t llo = c, lhi = c;
        bool boundary = true;
        while (hi - lo > 1) {
            DQ_DBG(g_dbg.probes++;)
            const uint32_t mid = (uint32_t)(lo + ((hi - lo) >> 1));
            bool ls;
            const uint32_t cc = match_from<WARP>(t, (uint32_t)ix.SA[mid], j, min(llo, lhi), &ls);
            if (ls) {
                lo = mid;
                llo = cc;
                boundary = false;
            } else {
                hi = mid;
                lhi = cc;
            }
        }
        return Bracket{(uint32_t)hi, boundary ? LCP[s] : llo, lhi};
    }
}

// chain state carried from one position to the next: matched old suffix, match length, side
struct Carry {
    uint32_t p, l;
    bool less;
};

template <bool WARP = false, bool BKT = true>
__device__ __forceinline__ Bracket locate_step(const Texts &t, const Index &ix, uint32_t j, const Carry &cy,
                                               uint32_t stride, bool have)
{
    if (have && cy.l > stride)
        return locate_anchor<WARP, BKT>(t, ix, j, ix.ISA[cy.p + stride], cy.l - stride, cy.less, cy.p + stride);
    return locate_scratch<WARP, BKT>(t, ix, j);
}

__device__ __forceinline__ uint32_t sa_at(const Index &ix, uint32_t rank, uint32_t known)
{
    return known != kNone ? known : (uint32_t)ix.SA[rank];
}

// the neighbour to inherit from: the one sharing more with the query (ties: the lower one -- measured 2x faster
// chains on the exe-like workload than inheriting from the upper one)
__device__ __forceinline__ Carry carry_of(const Texts &t, const Index &ix, const Bracket &b)
{
    const bool hx = b.L > 0, hy = b.L < t.n;
    if (hx && (!hy || b.x >= b.y)) return Carry{sa_at(ix, b.L - 1, b.sx), b.x, true};
    if (hy) return Carry{sa_at(ix, b.L, b.sy), b.y, false};
    return Carry{0, 0, false};  // n == 0
}

// what Diff.Search returns for this bracket (Diff.cs:271-286), including the I[n] == 0 leaf; also hands back the
// carry for the next position (same neighbour as the result in the common case, so SA is read at most once)
__device__ __forceinline__ Carry reference_result(const Texts &t, const Index &ix, uint32_t j, const Bracket &b,
                                                  int32_t *pos, int32_t *len)
{
    const uint32_t n = t.n;
    if (n == 0) {
        *pos = 0;
        *len = 0;
        return Carry{0, 0, false};
    }
    if (b.L > 0 && b.L < n) {  // leaf (L-1, L)
        if (b.x > b.y) {
            const uint32_t ps = sa_at(ix, b.L - 1, b.sx);
            *pos = (int32_t)ps;
            *len = (int32_t)b.x;
            return Carry{ps, b.x, true};
        }
        const uint32_t pe = sa_at(ix, b.L, b.sy);
        *pos = (int32_t)pe;
        *len = (int32_t)b.y;
        if (b.x == b.y) return Carry{sa_at(ix, b.L - 1, b.sx), b.x, true};  // tie: result = upper, carry = lower
        return Carry{pe, b.y, false};
    }
    uint32_t ps, pe, x, y;
    if (b.L == 0) {  // leaf (0, 1)
        ps = sa_at(ix, 0, b.sy);
        x = b.y;
        if (n == 1) {
            pe = 0;  // I[1] == I[n] == 0, the same suffix again
            y = x;
        } else {
            pe = (uint32_t)ix.SA[1];
            const uint32_t g = ix.lv[0][1];
            if (g < x)
                y = g;
            else if (g > x)
                y = x;
            else {
                bool ls;
                y = match_from(t, pe, j, x, &ls);
            }
        }
    } else {  // leaf (n-1, n): I[n] == 0 -> the whole of `old`
        ps = sa_at(ix, n - 1, b.sx);
        x = b.x;
        pe = 0;
        bool ls;
        y = match_from(t, 0, j, 0, &ls);
    }
    if (x > y) {
        *pos = (int32_t)ps;
        *len = (int32_t)x;
    } else {
        *pos = (int32_t)pe;
        *len = (int32_t)y;
    }
    return carry_of(t, ix, b);
}

// ---- kernels ---------------------------------------------------------------------------------------------

// ISA[SA[r]] = r for a suffix array that came from the caller (any ISuffixSort provider, Diff.cs:90): nothing about
// it is trusted.  ISA starts as all kUnset; entries outside [0, n) are counted in *bad instead of being followed, and
// check_inverse_kernel counts the positions no entry named -- n values in n slots, so a duplicate leaves a gap.
constexpr uint32_t kUnset = 0xffffffffu;

__global__ void __launch_bounds__(256) invert_sa_kernel(const int32_t *__restrict__ SA, uint32_t n,
                                                         uint32_t *__restrict__ ISA, uint32_t *__restrict__ bad)
{
    uint32_t wrong = 0;
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t p = (uint32_t)SA[r];
        if (p < n)
            ISA[p] = (uint32_t)r;
        else
            ++wrong;
    }
    if (wrong) atomicAdd(bad, wrong);
}

__global__ void __launch_bounds__(256) check_inverse_kernel(const uint32_t *__restrict__ ISA, uint32_t n,
                                                             uint32_t *__restrict__ bad)
{
    uint32_t wrong = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x)
        wrong += ISA[i] == kUnset ? 1u : 0u;
    if (wrong) atomicAdd(bad, wrong);
}

// 2-byte bucket bounds of the suffix array.  Suffix p has the 17-bit key 2*pair+1 (pair = T[p]<<8 | T[p+1]),
// the one-byte suffix n-1 has 2*(T[n-1]<<8), which puts it in front of its bucket and outside [lo, hi).
// One thread per pair k: lo[k] = #{key < 2k+1}, hi[k] = #{key < 2k+2}, by binary search over SA.
__global__ void __launch_bounds__(256) bucket_bounds_kernel(const uint8_t *__restrict__ T, uint32_t n,
                                                             const int32_t *__restrict__ SA,
                                                             uint32_t *__restrict__ bkt_lo, uint32_t *__restrict__ bkt_hi)
{
    const uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= 65536u) return;
#pragma unroll
    for (int which = 0; which < 2; ++which) {
        const uint32_t target = 2u * k + 1u + (uint32_t)which;
        uint32_t lo = 0, hi = n;  // first rank whose key >= target
        while (lo < hi) {
            const uint32_t mid = lo + ((hi - lo) >> 1);
            const uint32_t p = (uint32_t)SA[mid];
            const uint32_t key = (p + 1 < n) ? 2u * (((uint32_t)T[p] << 8) | T[p + 1]) + 1u : 2u * ((uint32_t)T[p] << 8);
            if (key < target)
                lo = mid + 1;
            else
                hi = mid;
        }
        (which ? bkt_hi : bkt_lo)[k] = lo;
    }
}

// ---- 3-byte prefix table (Index::pre3) -----------------------------------------------------------------------
// Two ways to build it.  From the text alone: a histogram of the 3-byte prefixes of all suffixes (equal keys inside a
// warp are added with one atomic: zero padding would otherwise send a million increments to one address), then an
// exclusive scan over the 2^24 bins in three small kernels (~0.35 ms at 16 MiB, the atomics).  Or, when this library's
// own sort produced the suffix array, from the keys of its round 0 while they are still in sorted order: the first
// index of every 3-byte value is marked (one coalesced read of the keys) and the empty bins are filled from the right
// (~0.06 ms) -- prefix3_mark_kernel + prefix3_fill_* below.
__global__ void __launch_bounds__(256) prefix3_hist_kernel(const uint8_t *__restrict__ T, uint32_t n,
                                                            uint32_t *__restrict__ hist, uint64_t p_begin = 0,
                                                            uint64_t p_end = ~0ull)
{
    // suffixes [p_begin, min(p_end, n)); the text is zero padded, which is the padding the short ones need
    const uint64_t total = p_end < n ? p_end : n;
    const uint64_t span = p_begin + ((total - min(total, p_begin) + 31) & ~(uint64_t)31);  // whole warps: the match below is warp-wide
    for (uint64_t p = p_begin + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; p < span; p += (uint64_t)gridDim.x * blockDim.x) {
        const bool valid = p < total;
        const uint32_t key = valid ? (((uint32_t)T[p] << 16) | ((uint32_t)T[p + 1] << 8) | T[p + 2]) : (0xff000000u + lane_id());
        const unsigned same = __match_any_sync(kFullMask, key);
        if (valid && (unsigned)(__ffs((int)same) - 1) == lane_id()) atomicAdd(hist + key, (uint32_t)__popc(same));
    }
}

// ---- a device group builds the index by text range (dq_group.inl, group_build_index) -----------------------------
// Every shard has filled, in its own zero-initialised copy of an array, the entries its text range produced; shard s
// then combines elements [begin, end) of all copies (max for LCP values, sum for counts) and writes the result into
// every copy.  Reads and writes of peer copies are plain coalesced loads and stores over NVLink.
struct PeerArrays {
    uint32_t *p[16];
    int count;
};
template <bool SUM>
__global__ void __launch_bounds__(256) merge_copies_kernel(const PeerArrays arr, uint64_t begin, uint64_t end)
{
    for (uint64_t i = begin + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < end; i += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t v = 0;
#pragma unroll
        for (int k = 0; k < 16; ++k)
            if (k < arr.count) {
                const uint32_t x = arr.p[k][i];
                v = SUM ? v + x : max(v, x);
            }
#pragma unroll
        for (int k = 0; k < 16; ++k)
            if (k < arr.count) arr.p[k][i] = v;
    }
}

constexpr uint32_t kPrefix3Tile = 4096;  // bins per block of the scan kernels (256 threads x 16)
constexpr uint32_t kPrefix3Tiles = kPrefix3Bins / kPrefix3Tile;

__global__ void __launch_bounds__(256) prefix3_tile_sum_kernel(const uint32_t *__restrict__ hist,
                                                                uint32_t *__restrict__ tile_sum)
{
    __shared__ uint32_t warp_sum[8];
    const uint4 *src = reinterpret_cast<const uint4 *>(hist + (size_t)blockIdx.x * kPrefix3Tile) + threadIdx.x * 4;
    uint32_t s = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const uint4 v = src[q];
        s += v.x + v.y + v.z + v.w;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(kFullMask, s, o);
    if (lane_id() == 0) warp_sum[warp_id()] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t tot = 0;
        for (int w = 0; w < 8; ++w) tot += warp_sum[w];
        tile_sum[blockIdx.x] = tot;
    }
}

// one block: exclusive scan of the kPrefix3Tiles tile sums in place; also the tail of the table (total, and the padded
// values of the two short suffixes)
__global__ void __launch_bounds__(1024) prefix3_tile_scan_kernel(uint32_t *__restrict__ tile_sum, const uint8_t *__restrict__ T,
                                                                  uint32_t n, uint32_t *__restrict__ table)
{
    static_assert(kPrefix3Tiles == 4096, "four tile sums per thread");
    __shared__ uint32_t warp_sum[32];
    uint32_t v[4], s = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        v[q] = tile_sum[threadIdx.x * 4 + q];
        s += v[q];
    }
    uint32_t incl = s;
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t u = __shfl_up_sync(kFullMask, incl, d);
        if ((int)lane_id() >= d) incl += u;
    }
    if (lane_id() == 31) warp_sum[warp_id()] = incl;
    __syncthreads();
    if (warp_id() == 0) {
        const uint32_t w = warp_sum[lane_id()];
        uint32_t wi = w;
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t u = __shfl_up_sync(kFullMask, wi, d);
            if ((int)lane_id() >= d) wi += u;
        }
        warp_sum[lane_id()] = wi - w;
    }
    __syncthreads();
    uint32_t run = warp_sum[warp_id()] + incl - s;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        tile_sum[threadIdx.x * 4 + q] = run;
        run += v[q];
    }
    if (threadIdx.x == 0) {
        table[kPrefix3Bins] = n;
        table[kPrefix3Bins + 1] = n >= 1 ? ((uint32_t)T[n - 1] << 16) : kNone;
        table[kPrefix3Bins + 2] = n >= 2 ? (((uint32_t)T[n - 2] << 16) | ((uint32_t)T[n - 1] << 8)) : kNone;
    }
}

__global__ void __launch_bounds__(256) prefix3_apply_kernel(uint32_t *__restrict__ table, const uint32_t *__restrict__ tile_off)
{
    __shared__ uint32_t warp_sum[8];
    uint4 *dst = reinterpret_cast<uint4 *>(table + (size_t)blockIdx.x * kPrefix3Tile) + threadIdx.x * 4;
    uint4 v[4];
    uint32_t s = 0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        v[q] = dst[q];
        s += v[q].x + v[q].y + v[q].z + v[q].w;
    }
    uint32_t incl = s;
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t u = __shfl_up_sync(kFullMask, incl, d);
        if ((int)lane_id() >= d) incl += u;
    }
    if (lane_id() == 31) warp_sum[warp_id()] = incl;
    __syncthreads();
    uint32_t run = tile_off[blockIdx.x] + incl - s;
    for (int w = 0; w < (int)warp_id(); ++w) run += warp_sum[w];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        uint4 o;
        o.x = run;
        run += v[q].x;
        o.y = run;
        run += v[q].y;
        o.z = run;
        run += v[q].z;
        o.w = run;
        run += v[q].w;
        dst[q] = o;
    }
}

// pre3 from the sorted round-0 keys (big-endian packed 8 bytes, zero padded): table[k] = first index whose key starts
// with k, for the values that occur; the table must hold kNone everywhere before
__global__ void __launch_bounds__(256) prefix3_mark_kernel(const uint64_t *__restrict__ sorted_keys, uint32_t n,
                                                            uint32_t *__restrict__ table)
{
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t k = (uint32_t)(sorted_keys[i] >> 40);
        if (i == 0 || (uint32_t)(sorted_keys[i - 1] >> 40) != k) table[k] = (uint32_t)i;
    }
}

// empty bins take the value of the next marked bin to their right (n if there is none): a suffix-minimum scan, in the
// same three steps as the sum scan above
__global__ void __launch_bounds__(256) prefix3_fill_tile_min_kernel(const uint32_t *__restrict__ table,
                                                                     uint32_t *__restrict__ tile_min)
{
    __shared__ uint32_t warp_min[8];
    const uint4 *src = reinterpret_cast<const uint4 *>(table + (size_t)blockIdx.x * kPrefix3Tile) + threadIdx.x * 4;
    uint32_t m = kNone;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const uint4 v = src[q];
        m = min(m, min(min(v.x, v.y), min(v.z, v.w)));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = min(m, __shfl_xor_sync(kFullMask, m, o));
    if (lane_id() == 0) warp_min[warp_id()] = m;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t t = kNone;
        for (int w = 0; w < 8; ++w) t = min(t, warp_min[w]);
        tile_min[blockIdx.x] = t;
    }
}

// one block: tile_min[t] <- min over the tiles to the right of t (n if none); also the tail of the table
__global__ void __launch_bounds__(1024) prefix3_fill_tile_scan_kernel(uint32_t *__restrict__ tile_min, const uint8_t *__restrict__ T,
                                                                       uint32_t n, uint32_t *__restrict__ table)
{
    __shared__ uint32_t sm[kPrefix3Tiles];
    for (uint32_t t = threadIdx.x; t < kPrefix3Tiles; t += blockDim.x) sm[t] = tile_min[t];
    __syncthreads();
    // 4096 values: thread x owns tiles [4x, 4x+4); suffix minima inside, then across threads through shared memory
    __shared__ uint32_t part[1024];
    uint32_t v[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) v[q] = sm[threadIdx.x * 4 + q];
    part[threadIdx.x] = min(min(v[0], v[1]), min(v[2], v[3]));
    __syncthreads();
    for (int d = 1; d < 1024; d <<= 1) {
        const uint32_t other = threadIdx.x + d < 1024 ? part[threadIdx.x + d] : kNone;
        __syncthreads();
        part[threadIdx.x] = min(part[threadIdx.x], other);
        __syncthreads();
    }
    uint32_t run = min(threadIdx.x + 1 < 1024 ? part[threadIdx.x + 1] : kNone, n);  // everything right of this thread's tiles
#pragma unroll
    for (int q = 3; q >= 0; --q) {
        tile_min[threadIdx.x * 4 + q] = run;
        run = min(run, v[q]);
    }
    if (threadIdx.x == 0) {
        table[kPrefix3Bins] = n;
        table[kPrefix3Bins + 1] = n >= 1 ? ((uint32_t)T[n - 1] << 16) : kNone;
        table[kPrefix3Bins + 2] = n >= 2 ? (((uint32_t)T[n - 2] << 16) | ((uint32_t)T[n - 1] << 8)) : kNone;
    }
}

__global__ void __launch_bounds__(256) prefix3_fill_apply_kernel(uint32_t *__restrict__ table, const uint32_t *__restrict__ tile_right)
{
    __shared__ uint32_t warp_min[8];
    uint4 *dst = reinterpret_cast<uint4 *>(table + (size_t)blockIdx.x * kPrefix3Tile) + threadIdx.x * 4;
    uint32_t v[16];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const uint4 u = dst[q];
        v[4 * q] = u.x, v[4 * q + 1] = u.y, v[4 * q + 2] = u.z, v[4 * q + 3] = u.w;
    }
    uint32_t mine = kNone;
#pragma unroll
    for (int e = 0; e < 16; ++e) mine = min(mine, v[e]);
    // minimum over the threads to the right inside the warp, then over the warps to the right
    uint32_t incl = mine;
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t u = __shfl_down_sync(kFullMask, incl, d);
        if ((int)lane_id() + d < 32) incl = min(incl, u);
    }
    if (lane_id() == 0) warp_min[warp_id()] = incl;
    __syncthreads();
    uint32_t right = tile_right[blockIdx.x];
    for (int w = (int)warp_id() + 1; w < 8; ++w) right = min(right, warp_min[w]);
    const uint32_t next_lane = __shfl_down_sync(kFullMask, incl, 1);
    if (lane_id() < 31) right = min(right, next_lane);
    uint32_t run = right;
#pragma unroll
    for (int e = 15; e >= 0; --e) {
        run = min(run, v[e]);
        v[e] = run;
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) dst[q] = make_uint4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
}

// LCP array, levels S and A.  One WARP walks `per_warp` text positions `stride` apart; the byte comparisons are
// warp-cooperative (a position inside a long repeat costs length/256 steps, not length/8), and each position
// starts from what the one before it leaves: PLCP[i + stride] >= PLCP[i] - stride.  out_l[i / stride] = PLCP[i].
//   level S (seeds):  stride = kSuper, per_warp = a few supers, seed_l = nullptr -- the first position of a warp is
//                     compared from byte 0, which inside a repeat of length R costs R bytes: this level keeps the
//                     number of such cold starts to a few thousand however long the text is;
//   level A (heads):  stride = kChunk, per_warp = kHeads; the first head of super s is position s*kSuper, whose
//                     value level S has already written to seed_l[s].
// PHI[i] = the suffix that precedes suffix i in rank order (kNone for the smallest one), for i in [p_begin, p_end).
// The LCP kernels below walk the text and need, at every position, "my rank predecessor": two dependent random reads
// (ISA, then SA) in the middle of a latency-bound walk.  Done here instead, as one streaming pass -- coalesced ISA
// reads, independent random SA reads, coalesced writes -- the walks then read PHI in text order.
__global__ void __launch_bounds__(256) phi_kernel(const int32_t *__restrict__ SA, const uint32_t *__restrict__ ISA,
                                                  uint32_t *__restrict__ PHI, uint64_t p_begin, uint64_t p_end)
{
    for (uint64_t i = p_begin + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < p_end; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t r = ISA[i];
        PHI[i] = r ? (uint32_t)__ldg(SA + r - 1) : kNone;
    }
}

// PHI of a batch chunk (dq_suffix.cuh, "batches"), from its text-major suffix array of per-text indices: rank slot r
// belongs to the text t that holds compact position r, and PHI[offs[t] + SA[r]] = offs[t] + SA[r-1], kNone for the
// first rank of every text.  Rank order instead of phi_kernel's text order: the chunk's ISA is padded.  grid-stride.
__global__ void __launch_bounds__(256) batch_phi_kernel(const int32_t *__restrict__ SA, const uint32_t *__restrict__ offs,
                                                        uint32_t count, uint32_t *__restrict__ PHI, uint32_t n)
{
    for (uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; s < n; s += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t r = (uint32_t)s;
        const uint32_t base = __ldg(offs + suffix::batch_owner(offs, count, r));
        PHI[base + (uint32_t)SA[r]] = r > base ? base + (uint32_t)__ldg(SA + r - 1) : kNone;
    }
}

// Where the comparisons of the LCP walks stop: at the end of the text that holds the position (a suffix and its rank
// predecessor always belong to the same text).  `n` is the length of the whole buffer.  A walk moves forward and calls
// enter(i) before it reads end() or begin() for position i.
// One text: everything ends at n.
struct OneText {
    static constexpr bool kRunEnds = true;  // lcp_heads_kernel may be given the sort's run ends
    uint32_t n;
    __device__ __forceinline__ void enter(uint32_t) {}
    __device__ __forceinline__ uint32_t begin() const { return 0; }
    __device__ __forceinline__ uint32_t end() const { return n; }
    // most bytes lcp_chain_kernel may compare backwards from the head ih and its predecessor qh
    __device__ __forceinline__ uint32_t back_cap(uint32_t, uint32_t qh) const { return min((uint32_t)kChunk - 1, qh); }
};

// The texts of a batch chunk, back to back with no separator byte: text t is [offs[t], offs[t+1]).  Without the bound
// a comparison runs on into the next text, and clamping afterwards would be too late: Kasai's PLCP[i+1] >= PLCP[i] - 1
// and the reducible positions of lcp_chain_kernel need the values inside the text.  The owner is looked up where a walk
// starts and again only where it crosses an offset.
struct ChunkTexts {
    static constexpr bool kRunEnds = false;  // a chunk's sort has none; without the branch the head walk needs no spill
    uint32_t n;
    const uint32_t *offs;
    uint32_t count;
    uint32_t lo = 0, hi = 0;  // the text entered last
    __device__ __forceinline__ void enter(uint32_t i)
    {
        if (i >= hi) {
            const uint32_t t = suffix::batch_owner(offs, count, i);
            lo = __ldg(offs + t);
            hi = __ldg(offs + t + 1);
        }
    }
    __device__ __forceinline__ uint32_t begin() const { return lo; }
    __device__ __forceinline__ uint32_t end() const { return hi; }
    // the backward step must not reach across the start of the text of ih (which holds qh as well)
    __device__ __forceinline__ uint32_t back_cap(uint32_t ih, uint32_t qh) const
    {
        ChunkTexts h = *this;
        h.enter(ih);
        return min((uint32_t)kChunk - 1, min(ih, qh) - h.lo);
    }
};

// LCP[ISA[i]] = PLCP[i] for i in [p_begin, p_end) (a device group: every shard scatters its own text range), or
// LCP[r] = PLCP[SA[r]] for every rank r (one GPU: coalesced writes, random reads)
__global__ void __launch_bounds__(256) lcp_scatter_kernel(const uint32_t *__restrict__ ISA, const uint32_t *__restrict__ PLCP,
                                                          uint32_t *__restrict__ LCP, uint64_t p_begin, uint64_t p_end)
{
    for (uint64_t i = p_begin + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < p_end; i += (uint64_t)gridDim.x * blockDim.x)
        LCP[ISA[i]] = PLCP[i];
}
// (ChunkTexts: SA holds per-text indices, and rank slot r belongs to the text that holds position r)
template <class Texts>
__global__ void __launch_bounds__(256) lcp_gather_kernel(const int32_t *__restrict__ SA, const uint32_t *__restrict__ PLCP,
                                                         uint32_t *__restrict__ LCP, Texts tx)
{
    for (uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; r < tx.n; r += (uint64_t)gridDim.x * blockDim.x) {
        tx.enter((uint32_t)r);
        LCP[r] = __ldg(PLCP + tx.begin() + SA[r]);
    }
}

template <class Texts>
__global__ void __launch_bounds__(kThreads)
lcp_heads_kernel(const uint8_t *__restrict__ T, Texts tx, const uint32_t *__restrict__ PHI,
                 uint32_t *__restrict__ out_l,
                 const uint32_t *__restrict__ run_end, uint32_t stride, uint32_t per_warp,
                 const uint32_t *__restrict__ seed_l, uint64_t w_begin = 0, uint64_t w_end = ~0ull)
{
    const uint32_t n = tx.n;
    // [w_begin, w_end): the warps of this launch (a device group builds the array by text range, dq_group.inl)
    const uint64_t w = w_begin + (((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const uint64_t i0 = w * stride * per_warp;
    if (w >= w_end || i0 >= n) return;
    uint32_t l = 0;
    for (uint32_t k = 0; k < per_warp; ++k) {
        const uint64_t i64 = i0 + (uint64_t)k * stride;
        if (i64 >= n) break;
        const uint32_t i = (uint32_t)i64;
        if (k == 0 && seed_l) {
            l = seed_l[w];
        } else {
            const uint32_t q = PHI[i];
            if (q == kNone) {
                l = 0;
            } else {
                uint32_t known = l > stride ? l - stride : 0;
                // both suffixes inside runs of the same byte: the shorter run is common prefix, no need to read it
                // (zero padding: without this one warp walks up to a megabyte here and the kernel waits for it)
                if (Texts::kRunEnds && run_end && known == 0 && T[i] == T[q]) {
                    const uint32_t ri = run_end[i] - i, rq = run_end[q] - q;
                    const uint32_t skip = min(ri, rq);
                    if (skip >= 64) known = skip;
                }
                tx.enter(i);
                const uint32_t e = tx.end();
                l = known + common_prefix_warp(T + i + known, e - i - known, T + q + known, e - q - known);
            }
        }
        if (lane_id() == 0) out_l[i / stride] = l;
    }
}

// number of equal bytes walking backwards from a[-1], b[-1], at most cap
__device__ __forceinline__ uint32_t common_suffix(const uint8_t *a, const uint8_t *b, uint32_t cap, bool room32 = false)
{
    // room32: the 32 bytes in front of both pointers are readable.  Then the usual case (cap = kChunk - 1 = 31) is four
    // independent 8-byte reads per side instead of up to 31 dependent byte reads.
    if (room32 && cap == 31u) {
        uint64_t x[4];
#pragma unroll
        for (int w = 0; w < 4; ++w) x[w] = load64u(a - 8 * (w + 1)) ^ load64u(b - 8 * (w + 1));
        uint32_t e = 0;
#pragma unroll
        for (int w = 0; w < 4; ++w) {
            if (e == 8u * w) e += x[w] ? ((uint32_t)__clzll((long long)x[w]) >> 3) : 8u;  // a[-1] is the top byte of x[0]
        }
        return min(e, 31u);
    }
    uint32_t e = 0;
    while (e < cap && a[-(int)e - 1] == b[-(int)e - 1]) ++e;
    return e;
}

constexpr uint32_t kBackMin = 32;  // look at the next head only when it sits inside a repeat at least this long

// LCP array, level B: one thread per chunk, stride 1.  Writes PLCP[i] (the LCP entry of suffix i, in text order).
template <class Texts>
__global__ void __launch_bounds__(kThreads)
lcp_chain_kernel(const uint8_t *__restrict__ T, Texts tx, const uint32_t *__restrict__ PHI,
                 const uint32_t *__restrict__ head_l, uint32_t *__restrict__ PLCP,
                 uint64_t c_begin = 0, uint64_t c_end = ~0ull)
{
    const uint32_t n = tx.n;
    const uint64_t c = c_begin + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;  // [c_begin, c_end): this launch's chunks
    const uint64_t i0 = c * kChunk;
    if (c >= c_end || i0 >= n) return;
    tx.enter((uint32_t)i0);
    DQ_DBG(unsigned long long b0 = g_dbg.cmp_bytes;)
    DQ_DBG(struct Fin { unsigned long long b0; ~Fin() { unsigned long long d = g_dbg.cmp_bytes - b0; g_dbg.thr_max[0] = max(g_dbg.thr_max[0], d); int k = 0; while ((d >> k) > 1 && k < 23) ++k; g_dbg.thr_hist[0][k]++; } } fin{b0};)
    uint32_t l = head_l[c];
    PLCP[i0] = l;
    // The next head ih shares nl bytes with its rank predecessor qh.  If the `back` bytes before ih and qh
    // agree too, then for d <= back suffix ih-d shares d+nl bytes with the smaller suffix qh-d, and its own
    // rank predecessor shares at least as much: a second lower bound, so a repeat that starts inside this
    // chunk and reaches the next head is not re-compared byte by byte.
    uint32_t nl = 0, back = 0;
    const uint64_t ih = i0 + kChunk;
    if (ih < n) {
        nl = head_l[c + 1];
        if (nl >= kBackMin) {
            const uint32_t qh = PHI[ih];  // nl > 0 => the head has a predecessor
            back = common_suffix(T + ih, T + qh, tx.back_cap((uint32_t)ih, qh), kChunk == 32 && qh >= 32);
        }
    }
    uint32_t q_prev = PHI[i0];  // rank predecessor of the position just done (kNone: it has none)
    for (int k = 1; k < kChunk; ++k) {
        // Reducible positions: if the rank predecessor of i+s is the rank predecessor of i moved s bytes on, the two
        // pairs of suffixes are the same strings minus their first s bytes, so PLCP[i+s] = PLCP[i] - s exactly (for
        // s < PLCP[i]) and nothing has to be compared.  kBatch positions are tested with independent reads.
        while (q_prev != kNone && k < kChunk) {
            constexpr int kBatch = 8;
            const uint64_t base = i0 + k - 1;  // the position just done
            const int room = (int)min((uint64_t)min(kBatch, kChunk - k), n - 1 - base);
            if (room <= 0 || l <= (uint32_t)room) break;
            uint32_t qq[kBatch];
#pragma unroll
            for (int s = 1; s <= kBatch; ++s) qq[s - 1] = s <= room ? PHI[base + s] : kNone;
            int run = 0;
#pragma unroll
            for (int s = 1; s <= kBatch; ++s)
                if (run == s - 1 && s <= room && qq[s - 1] == q_prev + (uint32_t)s) run = s;
#pragma unroll
            for (int s = 1; s <= kBatch; ++s)
                if (s <= run) PLCP[base + s] = l - (uint32_t)s;
            k += run;
            l -= (uint32_t)run;
            q_prev += (uint32_t)run;
            if (run < room) break;
        }
        if (k >= kChunk) break;
        const uint64_t i64 = i0 + k;
        if (i64 >= n) break;
        const uint32_t i = (uint32_t)i64;
        const uint32_t q = PHI[i];
        if (q == kNone) {
            l = 0;
            q_prev = kNone;
        } else {
            uint32_t known = l > 0 ? l - 1 : 0;
            const uint32_t d = (uint32_t)(kChunk - k);
            if (d <= back) known = max(known, d + nl);
            tx.enter(i);
            const uint32_t e = tx.end();
            l = known + common_prefix(T + i + known, e - i - known, T + q + known, e - q - known);
            q_prev = q;
        }
        PLCP[i] = l;
    }
}

// block minima: out[b] = min(in[b*W .. b*W+W)) ; one warp per block of W entries
__global__ void __launch_bounds__(256) block_min_kernel(const uint32_t *__restrict__ in, uint32_t count, uint32_t W,
                                                         uint32_t *__restrict__ out, uint32_t nblocks)
{
    const uint32_t warps_per_cta = blockDim.x / 32;
    for (uint64_t b = (uint64_t)blockIdx.x * warps_per_cta + warp_id(); b < nblocks;
         b += (uint64_t)gridDim.x * warps_per_cta) {
        uint32_t mn = 0xffffffffu;
        const uint64_t lo = b * W;
        for (uint64_t k = lo + lane_id(); k < lo + W && k < count; k += 32) mn = min(mn, in[k]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mn = min(mn, __shfl_xor_sync(kFullMask, mn, o));
        if (lane_id() == 0) out[b] = mn;
    }
}

// search, levels S and A: the carry (neighbour of the query with the longer match) of positions `stride` apart,
// `per_warp` (<= 64) of them per WARP (uniform control flow, warp-cooperative byte comparisons).
// out_p / out_l [k / stride] hold the carry of table position k (bit 31 of out_l = less).
//   level S (seeds):  stride = kSuper, seed_* = nullptr;  level A (heads): stride = kChunk, per_warp = kHeads, the
//   first head of a super comes from level S.  Same reason as in lcp_heads_kernel: a from-scratch search inside a
//   long match compares the whole match, so only a few thousand warps are ever allowed to start cold.
// search_heads is the work of warp w; search_heads_kernel and batch_search_heads_kernel (one pair of a chunk) run it.
template <bool BKT>
__device__ __forceinline__ void search_heads(const Texts &t, const Index &ix, uint32_t scan_begin, uint32_t count,
                                             uint32_t *__restrict__ out_p, uint32_t *__restrict__ out_l, uint32_t stride,
                                             uint32_t per_warp, const uint32_t *__restrict__ seed_p,
                                             const uint32_t *__restrict__ seed_l, uint64_t w)
{
    const uint64_t k0 = w * stride * per_warp;
    if (k0 >= count || t.n == 0) return;
#ifdef DQ_PROF
    if (seed_l != nullptr && lane_id() == 0 && w < (1u << 16)) g_prof_cmp_clk[w] = 0, g_prof_cmp_bytes[w] = 0, g_prof_cmp_calls[w] = 0;
    const long long prof_t0 = clock64();
    struct ProfFin { long long t0; uint64_t w; bool seeds; __device__ ~ProfFin() { if (w < (1u << 16) && lane_id() == 0) (seeds ? g_prof_seeds : g_prof_heads)[w] = (uint32_t)((clock64() - t0) >> 6); } } prof_fin{prof_t0, w, seed_l == nullptr && stride == (uint32_t)kSuper};
#endif
    // pass 1, lanes in parallel: every position tries a capped from-scratch search on its own.  Positions in
    // unrelated data (short matches, no inheritance possible anyway) finish here; those inside long matches give up
    // after a few probes.  Without this pass a warp over a mutated region runs its binary searches back to back.
    constexpr int kPerLane = 2;
    static_assert(kHeads <= 32 * kPerLane, "a warp's positions must fit its lanes in pass 1");
    constexpr uint32_t kAbort = 0xffffffffu;
    uint32_t rp[kPerLane], rl[kPerLane];
#pragma unroll
    for (int q = 0; q < kPerLane; ++q) {
        const uint32_t h = lane_id() * kPerLane + q;
        const uint64_t kk = k0 + (uint64_t)h * stride;
        rp[q] = 0;
        rl[q] = kAbort;
        if (h < per_warp && kk < count && !(h == 0 && seed_l)) {
            bool aborted;
            const Bracket b = locate_scratch_capped<BKT>(t, ix, scan_begin + (uint32_t)kk, 128u, &aborted);
            if (!aborted) {
                const Carry c1 = carry_of(t, ix, b);
                rp[q] = c1.p;
                rl[q] = c1.l | (c1.less ? 0x80000000u : 0u);
            }
        }
    }
    if (seed_l && lane_id() == 0) {
        rp[0] = seed_p[w];
        rl[0] = seed_l[w];
    }
    __syncwarp();
    // pass 2, the warp together: the positions pass 1 left open inherit from their predecessor (or search from
    // scratch with warp-cooperative comparisons)
    Carry cy{0, 0, false};
    bool have = false;
    Bracket lastb{0, 0, 0};  // bracket of the position just handled, when pass 2 computed it itself
    bool lastb_ok = false;
    for (uint32_t k = 0; k < per_warp; ++k) {
        const uint64_t kk = k0 + (uint64_t)k * stride;
        if (kk >= count) break;
        const uint32_t j = scan_begin + (uint32_t)kk;
        uint32_t p1 = 0, l1 = kAbort;
#pragma unroll
        for (int q = 0; q < kPerLane; ++q) {
            const uint32_t pp = __shfl_sync(kFullMask, rp[q], k / kPerLane);
            const uint32_t ll = __shfl_sync(kFullMask, rl[q], k / kPerLane);
            if ((int)(k % kPerLane) == q) {
                p1 = pp;
                l1 = ll;
            }
        }
        if (l1 != kAbort) {
            cy = Carry{p1, l1 & 0x7fffffffu, (l1 >> 31) != 0};
            lastb_ok = false;
        } else {
            lastb = locate_step<true, BKT>(t, ix, j, cy, stride, have);
            lastb_ok = true;
            cy = carry_of(t, ix, lastb);
        }
        have = true;
        if (lane_id() == 0) {
            out_p[kk / stride] = cy.p;
            out_l[kk / stride] = cy.l | (cy.less ? 0x80000000u : 0u);
        }
        // The positions after a resolved one are often predictable; both checks below let lane s test position k+s with
        // independent reads, and the run of positions that check out is written at once.  Repeated until neither
        // makes progress.
        for (;;) {
            const uint64_t at = k0 + (uint64_t)k * stride;  // table position of the last resolved one
            const uint32_t s1 = lane_id();
            const uint64_t step = (uint64_t)s1 * stride;
            const bool in_range = s1 >= 1 && k + s1 < per_warp && at + step < count;
            uint32_t run = 0;
            // (a) two-sided inheritance (see search_chain_kernel): the two neighbours of the bracket, moved s positions
            // on, are still adjacent in rank
            if (lastb_ok && lastb.L > 0 && lastb.L < t.n) {
                const uint32_t A = sa_at(ix, lastb.L - 1, lastb.sx), B = sa_at(ix, lastb.L, lastb.sy);
                bool ok = false;
                uint32_t r2 = 0;
                if (in_range && (uint64_t)min(lastb.x, lastb.y) > step) {
                    r2 = ix.ISA[B + (uint32_t)step];
                    ok = r2 == ix.ISA[A + (uint32_t)step] + 1u;
                }
                const unsigned m = __ballot_sync(kFullMask, ok) >> 1;
                run = (uint32_t)__ffs((int)~m) - 1u;  // consecutive lanes 1..run checked out (<= 31)
                if (run) {
                    const bool lower = lastb.x >= lastb.y;  // carry_of: the neighbour sharing more, ties -> the lower one
                    if (s1 >= 1 && s1 <= run) {
                        out_p[at / stride + s1] = (lower ? A : B) + (uint32_t)step;
                        out_l[at / stride + s1] = ((lower ? lastb.x : lastb.y) - (uint32_t)step) | (lower ? 0x80000000u : 0u);
                    }
                    const uint32_t adv = run * stride;
                    lastb = Bracket{__shfl_sync(kFullMask, r2, (int)run), lastb.x - adv, lastb.y - adv, A + adv, B + adv};
                    cy = carry_of(t, ix, lastb);
                    k += run;
                    continue;
                }
            }
            // (b) inside a unique long match: anchor (p + s*stride, l - s*stride, same side) whose neighbour on the
            // query's side shares less -- the anchor is the answer, with no byte compared
            {
                const uint32_t *LCP = ix.lv[0];
                bool ok = false;
                uint32_t ps = 0, cs = 0;
                if (in_range && cy.l >= s1 * stride + kMinAnchor) {
                    ps = cy.p + s1 * stride;
                    cs = cy.l - s1 * stride;
                    const uint32_t r = ix.ISA[ps];
                    const bool edge = cy.less ? (r + 1 >= t.n) : (r == 0);
                    ok = !edge && LCP[cy.less ? r + 1 : r] < cs;
                }
                const unsigned m = __ballot_sync(kFullMask, ok) >> 1;
                run = (uint32_t)__ffs((int)~m) - 1u;
                if (run == 0) break;
                if (s1 >= 1 && s1 <= run) {
                    out_p[at / stride + s1] = ps;
                    out_l[at / stride + s1] = cs | (cy.less ? 0x80000000u : 0u);
                }
                k += run;
                cy.p += run * stride;
                cy.l -= run * stride;
                lastb_ok = false;  // lastb describes an earlier position now
            }
        }
    }
}

__global__ void __launch_bounds__(kThreads)
search_heads_kernel(Texts t, Index ix, uint32_t scan_begin, uint32_t count, uint32_t *__restrict__ out_p,
                    uint32_t *__restrict__ out_l, uint32_t stride, uint32_t per_warp,
                    const uint32_t *__restrict__ seed_p, const uint32_t *__restrict__ seed_l)
{
    search_heads<true>(t, ix, scan_begin, count, out_p, out_l, stride, per_warp, seed_p, seed_l,
                       ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
}

// search, level B: one thread per chunk; writes the reference's (pos, len) for every position.  search_chain is the work
// of chunk c (heads_ready: heads [0, heads_ready) have been computed -- a slice's last chain cannot look at the next
// head); search_chain_kernel and batch_search_chain_kernel run it.
template <bool BKT>
__device__ __forceinline__ void search_chain(const Texts &t, const Index &ix, uint32_t scan_begin, uint32_t count,
                                             const uint32_t *__restrict__ head_p, const uint32_t *__restrict__ head_l,
                                             int32_t *__restrict__ pos_out, int32_t *__restrict__ len_out, uint64_t c,
                                             uint32_t heads_ready)
{
    const uint64_t k0 = c * kChunk;
    if (k0 >= count) return;
#ifdef DQ_PROF
    const long long prof_t0 = clock64();
    struct ProfFin { long long t0; uint64_t c; __device__ ~ProfFin() { if (c < (1u << 21)) g_prof_chain[c] = (uint32_t)((clock64() - t0) >> 6); } } prof_fin{prof_t0, c};
#endif
    DQ_DBG(unsigned long long b0 = g_dbg.cmp_bytes + 64 * g_dbg.probes;)
    DQ_DBG(struct Fin { unsigned long long b0; ~Fin() { unsigned long long d = g_dbg.cmp_bytes + 64 * g_dbg.probes - b0; g_dbg.thr_max[1] = max(g_dbg.thr_max[1], d); int k = 0; while ((d >> k) > 1 && k < 23) ++k; g_dbg.thr_hist[1][k]++; } } fin{b0};)
    if (t.n == 0) {
        for (int k = 0; k < kChunk && k0 + k < count; ++k) {
            pos_out[k0 + k] = 0;
            len_out[k0 + k] = 0;
        }
        return;
    }
    // the head's carry describes the head itself: re-derive its bracket from it (stride 0)
    const uint32_t hl = head_l[c];
    Carry cy{head_p[c], hl & 0x7fffffffu, (hl >> 31) != 0};
    // The next head matched old suffix np for nl bytes.  If the `back` bytes before the head and before np
    // agree, the query d <= back positions earlier matches suffix np-d for exactly d+nl bytes on the same
    // side: a second exact anchor, so a long match that begins inside this chunk and reaches the next head
    // is never re-compared byte by byte.
    uint32_t np = 0, nl = 0, back = 0;
    bool nless = false;
    if (k0 + kChunk < count && c + 1 < heads_ready) {
        const uint32_t v = head_l[c + 1];
        nl = v & 0x7fffffffu;
        nless = (v >> 31) != 0;
        np = head_p[c + 1];
        if (nl >= kBackMin)
            back = common_suffix(t.new_ + scan_begin + k0 + kChunk, t.old_ + np, min((uint32_t)kChunk - 1, np), kChunk == 32 && np >= 32);
    }
    const uint32_t *LCP = ix.lv[0];
    const uint32_t n = t.n;
    for (int k = 0; k < kChunk; ++k) {
        const uint64_t kk = k0 + k;
        if (kk >= count) break;
        const uint32_t j = scan_begin + (uint32_t)kk;
        Bracket b;
        const uint32_t d = (uint32_t)(kChunk - k);
        if (k == 0)
            b = locate_anchor<false, BKT>(t, ix, j, ix.ISA[cy.p], cy.l, cy.less, cy.p);
        else if (d <= back && d + nl + 1 > cy.l)
            b = locate_anchor<false, BKT>(t, ix, j, ix.ISA[np - d], d + nl, nless, np - d);
        else
            b = locate_step<false, BKT>(t, ix, j, cy, 1, true);
        int32_t pos, len;
        cy = reference_result(t, ix, j, b, &pos, &len);
        pos_out[kk] = pos;
        len_out[kk] = len;
        // Inside a long match the next positions are predictable: position k+s inherits the anchor (p+s, l-s, same
        // side), and when that suffix's neighbour on the query's side shares fewer than l-s bytes with it, the anchor
        // IS the answer: pos = p+s, len = l-s (locate_anchor's first exit and reference_result's strict case, with no
        // byte compared).  The kBatch ranks and their kBatch LCP entries are independent reads, so they are issued
        // together instead of as 2*kBatch dependent round trips; the run of positions that check out is written at
        // once and the loop resumes at the first one that does not.
        // Two-sided inheritance, for matches that are long but NOT unique (zero runs, periodic records: the anchor's LCP
        // interval is wide and the general path would binary-search it at every position).  If the query sits between
        // suffixes A < query <= B, adjacent in rank, sharing x and y >= s+1 bytes with it, then dropping the first s bytes
        // of all three keeps their order; when A+s and B+s are still adjacent in rank nothing sorts between them, so the
        // bracket of position k+s is exactly (rank of B+s; x-s, y-s) -- two independent ISA reads per position, no
        // LCP walk, no probe.
        while (k + 1 < kChunk && b.L > 0 && b.L < n) {
            constexpr int kBatch = 8;
            const int room = min(kBatch, kChunk - 1 - k);
            if (min(b.x, b.y) <= (uint32_t)room || k0 + k + room >= count) break;
            const uint32_t A = sa_at(ix, b.L - 1, b.sx), B = sa_at(ix, b.L, b.sy);
            uint32_t r1[kBatch], r2[kBatch];
#pragma unroll
            for (int s = 1; s <= kBatch; ++s) {
                r1[s - 1] = s <= room ? ix.ISA[A + s] : 0u;
                r2[s - 1] = s <= room ? ix.ISA[B + s] : 0u;
            }
            int run = 0;
#pragma unroll
            for (int s = 1; s <= kBatch; ++s)
                if (run == s - 1 && s <= room && r2[s - 1] == r1[s - 1] + 1u) run = s;
            if (run == 0) break;
            const bool lower = b.x > b.y;  // Diff.cs:281-286: the longer match, ties -> the upper neighbour
            for (int s = 1; s <= run; ++s) {
                pos_out[k0 + k + s] = (int32_t)((lower ? A : B) + s);
                len_out[k0 + k + s] = (int32_t)((lower ? b.x : b.y) - s);
            }
            uint32_t rank_b = 0;
#pragma unroll
            for (int s = 1; s <= kBatch; ++s)
                if (s == run) rank_b = r2[s - 1];
            b = Bracket{rank_b, b.x - (uint32_t)run, b.y - (uint32_t)run, A + (uint32_t)run, B + (uint32_t)run};
            cy = carry_of(t, ix, b);
            k += run;
            if (run < room) break;
        }
        while (k + 1 < kChunk) {
            constexpr int kBatch = 8;
            const int room = min(kBatch, kChunk - 1 - k);
            if (cy.l < (uint32_t)room + kMinAnchor || k0 + k + room >= count) break;
            uint32_t rr[kBatch], gg[kBatch];
#pragma unroll
            for (int s = 1; s <= kBatch; ++s) rr[s - 1] = s <= room ? ix.ISA[cy.p + s] : 0u;
#pragma unroll
            for (int s = 1; s <= kBatch; ++s) {
                const uint32_t r = rr[s - 1];
                // the entry between the anchor and its neighbour on the query's side; edge ranks go the general way
                const bool edge = cy.less ? (r + 1 >= n) : (r == 0);
                gg[s - 1] = (s <= room && !edge) ? LCP[cy.less ? r + 1 : r] : 0xffffffffu;
            }
            int run = 0;
#pragma unroll
            for (int s = 1; s <= kBatch; ++s)
                if (run == s - 1 && s <= room && gg[s - 1] < cy.l - (uint32_t)s) run = s;
            for (int s = 1; s <= run; ++s) {
                pos_out[k0 + k + s] = (int32_t)(cy.p + s);
                len_out[k0 + k + s] = (int32_t)(cy.l - s);
            }
            k += run;
            cy.p += (uint32_t)run;
            cy.l -= (uint32_t)run;
            if (run < room) break;
        }
        // In unrelated data (the match just found is too short to inherit from) the next positions are searched from
        // scratch whatever they turn out to be, and those searches do not depend on each other: kScratchBatch of them
        // run with their probes interleaved.  (A from-scratch search is always exact; inheriting is only cheaper.)
#ifndef DQ_SCRATCH_BATCH
#define DQ_SCRATCH_BATCH 2
#endif
        constexpr int kScratchBatch = DQ_SCRATCH_BATCH;
        while (kScratchBatch > 1 && cy.l <= kMinAnchor && k + kScratchBatch < kChunk - (int)back &&
               k0 + k + kScratchBatch < count) {
            Bracket bb[kScratchBatch > 1 ? kScratchBatch : 1];
            locate_scratch_batch<(kScratchBatch > 1 ? kScratchBatch : 1), BKT>(t, ix, scan_begin + (uint32_t)(k0 + k) + 1u, bb);
#pragma unroll
            for (int s = 0; s < kScratchBatch; ++s) {
                int32_t pos2, len2;
                cy = reference_result(t, ix, scan_begin + (uint32_t)(k0 + k) + 1u + s, bb[s], &pos2, &len2);
                pos_out[k0 + k + 1 + s] = pos2;
                len_out[k0 + k + 1 + s] = len2;
            }
            k += kScratchBatch;
        }
    }
}

__global__ void __launch_bounds__(kThreads)
search_chain_kernel(Texts t, Index ix, uint32_t scan_begin, uint32_t count, const uint32_t *__restrict__ head_p,
                    const uint32_t *__restrict__ head_l, int32_t *__restrict__ pos_out, int32_t *__restrict__ len_out,
                    uint32_t chain_begin, uint32_t chain_end, uint32_t heads_ready)
{
    // chains [chain_begin, chain_end) of the search: lets the host pipeline the table in slices
    const uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x + chain_begin;
    if (c >= chain_end) return;
    search_chain<true>(t, ix, scan_begin, count, head_p, head_l, pos_out, len_out, c, heads_ready);
}

// ---- batches: every pair of a chunk searched in its own coordinates (dq_cuda_bsdiff_search_batch) ---------------------
// A chunk's olds were sorted together (dq_suffix.cuh, "batches"), and its news lie back to back in one buffer.  Pair i
// is searched exactly as the single-pair kernels search (old_i, new_i): its Texts and Index are views into the chunk's
// arrays at the pair's offsets, with its own lengths.  Behind every view lie the next pair's bytes and entries, so the
// lengths are what stops a comparison or a walk there.  The index has no bucket or prefix tables (BKT = false): a
// from-scratch search spans the pair's n_i ranks.  Work units (warps of the head level, chains) never cross a pair.
enum BatchTable { kTabOld, kTabNew, kTabSuper, kTabChunk, kTabLevel };  // kTabLevel + l - 1: level l >= 1
constexpr int kBatchTables = kTabLevel + kMaxLevels - 1;

struct BatchPairs {
    const uint8_t *olds, *news;  // the chunk's olds (zero padded) and news (zero padded)
    const int32_t *SA;           // suffix array of the chunk, text-major, values local to their text
    const uint32_t *ISA;         // local ranks: ISA[ob_i + p] = rank of suffix p of old_i among the suffixes of old_i
    const uint32_t *lv[kMaxLevels];  // lv[0]: LCP arrays in rank order (pair i at ob_i); lv[l]: pair i's level l at
                                     // lv[l] + tab[kTabLevel + l - 1][i]
    const uint32_t *tab;         // kBatchTables prefix tables of count + 1 entries each, tab[k * (count + 1) + i]:
                                 // offsets of olds and news, and prefix sums of supers, chunks and level sizes
    uint32_t count;

    __device__ __forceinline__ const uint32_t *table(int k) const { return tab + (size_t)k * (count + 1); }

    // the Texts and Index of pair i, what the single-pair path builds for (old_i, new_i) without buckets
    __device__ __forceinline__ void pair(uint32_t i, Texts &t, Index &ix) const
    {
        const uint32_t ob = table(kTabOld)[i], n = table(kTabOld)[i + 1] - ob;
        const uint32_t nb = table(kTabNew)[i], m = table(kTabNew)[i + 1] - nb;
        t = Texts{olds + ob, news + nb, n, m};
        ix = Index{};
        ix.SA = SA + ob;
        ix.ISA = ISA + ob;
        ix.lv[0] = lv[0] + ob;
        ix.size[0] = n;
        ix.top = 0;
        // lcp_levels (dq_search_host.inl) over n
        while (ix.size[ix.top] > 64 && ix.top + 1 < kMaxLevels) {
            const int l = ix.top + 1;
            ix.size[l] = (uint32_t)div_up(ix.size[l - 1], 64);
            ix.lv[l] = lv[l] + table(kTabLevel + l - 1)[i];
            ix.top = l;
        }
    }
};

// local ranks from the chunk's localized suffix array: rank slot r belongs to the text t that holds compact position r,
// and its suffix SA[r] of text t has local rank r - offs[t].  grid-stride.
__global__ void __launch_bounds__(256) batch_local_isa_kernel(const int32_t *__restrict__ SA, const uint32_t *__restrict__ offs,
                                                              uint32_t count, uint32_t *__restrict__ ISA, uint32_t n)
{
    for (uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; s < n; s += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t r = (uint32_t)s;
        const uint32_t base = __ldg(offs + suffix::batch_owner(offs, count, r));
        ISA[base + (uint32_t)SA[r]] = r - base;
    }
}

// block minima of every pair at once: output entry b belongs to the pair i with out_off[i] <= b < out_off[i+1], and is
// the minimum of that pair's input entries [64 (b - out_off[i]), + 64), which end at in_off[i+1].  One warp per entry;
// block_min_kernel over the whole chunk would make blocks that straddle two pairs.
__global__ void __launch_bounds__(256) batch_block_min_kernel(const uint32_t *__restrict__ in, const uint32_t *__restrict__ in_off,
                                                              uint32_t *__restrict__ out, const uint32_t *__restrict__ out_off,
                                                              uint32_t count, uint32_t total)
{
    const uint32_t warps_per_cta = blockDim.x / 32;
    for (uint64_t b = (uint64_t)blockIdx.x * warps_per_cta + warp_id(); b < total; b += (uint64_t)gridDim.x * warps_per_cta) {
        const uint32_t i = suffix::batch_owner(out_off, count, (uint32_t)b);
        const uint64_t lo = (uint64_t)__ldg(in_off + i) + ((uint64_t)b - __ldg(out_off + i)) * 64u;
        const uint64_t hi = min(lo + 64u, (uint64_t)__ldg(in_off + i + 1));
        uint32_t mn = 0xffffffffu;
        for (uint64_t k = lo + lane_id(); k < hi; k += 32) mn = min(mn, in[k]);
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) mn = min(mn, __shfl_xor_sync(kFullMask, mn, o));
        if (lane_id() == 0) out[b] = mn;
    }
}

// level A of the search for every pair: warp w is super w - sup[i] of the pair i with sup[i] <= w < sup[i+1], its heads
// go to the pair's chunk range of head_p / head_l.  No seed level: the first head of every super starts cold.
__global__ void __launch_bounds__(kThreads)
batch_search_heads_kernel(const BatchPairs bp, uint32_t *__restrict__ head_p, uint32_t *__restrict__ head_l, uint32_t supers)
{
    const uint64_t w = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    if (w >= supers) return;
    const uint32_t *sup = bp.table(kTabSuper);
    const uint32_t i = suffix::batch_owner(sup, bp.count, (uint32_t)w);
    Texts t;
    Index ix;
    bp.pair(i, t, ix);
    const uint32_t c0 = bp.table(kTabChunk)[i];
    search_heads<false>(t, ix, 0, t.m, head_p + c0, head_l + c0, (uint32_t)kChunk, (uint32_t)kHeads, nullptr, nullptr,
                        w - sup[i]);
}

// level B for every pair: thread c is chain c - chk[i] of the pair i with chk[i] <= c < chk[i+1]; it reads only that
// pair's heads and writes only its (pos, len) entries
__global__ void __launch_bounds__(kThreads)
batch_search_chain_kernel(const BatchPairs bp, const uint32_t *__restrict__ head_p, const uint32_t *__restrict__ head_l,
                          int32_t *__restrict__ pos_out, int32_t *__restrict__ len_out, uint32_t chunks)
{
    const uint64_t c = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= chunks) return;
    const uint32_t *chk = bp.table(kTabChunk);
    const uint32_t i = suffix::batch_owner(chk, bp.count, (uint32_t)c);
    Texts t;
    Index ix;
    bp.pair(i, t, ix);
    const uint32_t c0 = chk[i], nb = bp.table(kTabNew)[i];
    search_chain<false>(t, ix, 0, t.m, head_p + c0, head_l + c0, pos_out + nb, len_out + nb, c - c0, chk[i + 1] - c0);
}


// ---- compact form of the (pos, len) table for the host loop of dq_cuda_bsdiff_streams -------------------------------
// The loop of Diff.cs:100-223 reads len at every position it visits but uses pos only where the scan stops, and a
// stop needs len > oldscore + 8 >= 9 (Diff.cs:116) -- except the very last one, served by a single device read.
// So the table crosses PCIe as one byte per position, min(len, kLongLen), plus the list of "match heads": the
// positions with len >= kLongLen whose (pos, len) is not (pos+1, len-1) of the position before.  Every other
// long position continues the head before it (if y is long and continues y-1 then len[y-1] = len[y]+1 is long
// too, so walking back ends at a head with no other head in between): len = head.len - (y - head.at),
// pos = head.pos + (y - head.at).  Heads are written tile by tile, in position order inside a tile, at a base the
// tile reserves with one atomic; tile_tab[tile] = (base, count) lets the host walk them in order.
constexpr int kLongLen = 9;
constexpr int kCodeTile = 1024;

struct MatchHead {
    int32_t at, pos, len;
};

__global__ void __launch_bounds__(256)
    encode_table_kernel(const int32_t *__restrict__ pos, const int32_t *__restrict__ len, uint32_t count,
                        uint32_t tile_begin, uint8_t *__restrict__ code, MatchHead *__restrict__ heads,
                        uint32_t heads_cap, uint32_t *__restrict__ head_count, uint2 *__restrict__ tile_tab)
{
    __shared__ uint32_t warp_total[8];
    __shared__ uint32_t tile_base;
    const uint32_t tile = tile_begin + blockIdx.x;
    const uint64_t x0 = (uint64_t)tile * kCodeTile + (uint64_t)threadIdx.x * 4;
    int32_t p[5], l[5];  // [0]: the position before this thread's four
    p[0] = 0;
    l[0] = 0;
    if (x0 > 0 && x0 <= count) {
        p[0] = pos[x0 - 1];
        l[0] = len[x0 - 1];
    }
    if (x0 + 4 <= count) {
        const int4 pv = *reinterpret_cast<const int4 *>(pos + x0), lv = *reinterpret_cast<const int4 *>(len + x0);
        p[1] = pv.x, p[2] = pv.y, p[3] = pv.z, p[4] = pv.w;
        l[1] = lv.x, l[2] = lv.y, l[3] = lv.z, l[4] = lv.w;
    } else {
        for (int k = 0; k < 4; ++k) {
            const bool in = x0 + k < count;
            p[k + 1] = in ? pos[x0 + k] : 0;
            l[k + 1] = in ? len[x0 + k] : 0;
        }
    }
    uint32_t packed = 0, is_head = 0, mine = 0;
    for (int k = 0; k < 4; ++k) {
        const int32_t lk = l[k + 1];
        packed |= (uint32_t)(lk < kLongLen ? lk : kLongLen) << (8 * k);
        const bool continues = (x0 + k > 0) && p[k + 1] == p[k] + 1 && lk == l[k] - 1;
        if (lk >= kLongLen && !continues) {
            is_head |= 1u << k;
            ++mine;
        }
    }
    if (x0 + 4 <= count) {
        *reinterpret_cast<uint32_t *>(code + x0) = packed;
    } else {
        for (int k = 0; k < 4; ++k)
            if (x0 + k < count) code[x0 + k] = (uint8_t)(packed >> (8 * k));
    }
    // ordered compaction of the heads of this tile
    uint32_t incl = mine;
    for (int d = 1; d < 32; d <<= 1) {
        const uint32_t v = __shfl_up_sync(kFullMask, incl, d);
        if ((int)lane_id() >= d) incl += v;
    }
    if (lane_id() == 31) warp_total[warp_id()] = incl;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t run = 0;
        for (int w = 0; w < 8; ++w) {
            const uint32_t c = warp_total[w];
            warp_total[w] = run;
            run += c;
        }
        const uint32_t base = run ? atomicAdd(head_count, run) : 0u;
        tile_base = base;
        tile_tab[tile] = make_uint2(base, run);
    }
    __syncthreads();
    uint32_t at = tile_base + warp_total[warp_id()] + incl - mine;
    for (int k = 0; k < 4; ++k)
        if (is_head >> k & 1u) {
            if (at < heads_cap) heads[at] = MatchHead{(int32_t)(x0 + k), p[k + 1], l[k + 1]};
            ++at;
        }
}

}  // namespace search
}  // namespace dq
