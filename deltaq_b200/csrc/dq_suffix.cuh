// dq_suffix.cuh -- kernels of the prefix-doubling suffix sorter (everything except the radix passes).
//
// Data model (all device resident, n = text length, a = number of still-unresolved suffixes):
//   T[n(+pad)]      text, zero padded by >= 16 bytes
//   ISA[n]          rank of every suffix = SA slot of the head of its group (final once the group is a singleton)
//   SA[n]           output; slot s is written exactly once, when the suffix occupying it becomes a singleton
//   active set      three parallel arrays of length a, in SA order with resolved slots squeezed out:
//                     sa[k]    suffix start,  rank[k] current group rank (== ISA[sa[k]]),
//                     slot[k]  the SA slot that position k of the active set stands for
//   A group is a maximal run of equal ranks; its members are contiguous in the active set and own the
//   contiguous SA slots [rank, rank + size).  Sorting the active set by (rank, ISA[sa+h]+1) therefore only
//   permutes suffixes inside groups and `slot` stays put.
//
// Round 0 sorts all n suffixes by their first 8 bytes (big-endian packed, zero padded).  The elements enter
// the stable sort in DESCENDING suffix order, so inside a run of equal keys the (at most 7) suffixes shorter
// than 8 bytes -- which can only tie with longer ones through zero padding -- come first, shortest first,
// which is exactly their final order ("a proper prefix sorts first": Span.SequenceCompareTo,
// /root/reference/test/DeltaQ.SuffixSorting.LibDivSufSort.Tests/LibDivSufSortTests.cs:46-59).  The rank
// kernel makes each of them a singleton.  From then on every non-singleton group agrees on its first h
// bytes and all members are at least h long, so at most one member has sa + h == n and key half 0 is free
// for it.
//
// Replaces (by result) DivSufSort.sort_typeBstar / construct_SA
// (/root/reference/src/DeltaQ.SuffixSorting.LibDivSufSort/DivSufSort.cs:186-511, :44-153) and
// SAIS.sais_main (/root/reference/src/DeltaQ.SuffixSorting.SAIS/SAIS.cs:280-495).
#pragma once
#include "dq_common.cuh"
#include "dq_radix.cuh"

namespace dq {
namespace suffix {

constexpr int kPackThreads = 256;
constexpr int kPackItems = 8;

// big-endian value of T[i..i+8), reading three aligned little-endian words (T is zero padded)
__device__ __forceinline__ uint64_t load_key8(const uint8_t *__restrict__ T, uint32_t i)
{
    const uint32_t *w = reinterpret_cast<const uint32_t *>(T) + (i >> 2);
    const uint32_t w0 = __ldg(w), w1 = __ldg(w + 1), w2 = __ldg(w + 2);
    const unsigned sh = (i & 3u) * 8u;
    const uint32_t a = __funnelshift_r(w0, w1, sh);  // T[i..i+4) little-endian
    const uint32_t b = __funnelshift_r(w1, w2, sh);  // T[i+4..i+8)
    return ((uint64_t)__byte_perm(a, 0, 0x0123) << 32) | (uint64_t)__byte_perm(b, 0, 0x0123);
}

// ---- small alphabets: more than 8 characters per 64-bit key ------------------------------------------------------
// Round 0 sorts by as many leading characters as fit one key.  A text with at most 16 distinct byte values (DNA, binary
// data) is first rewritten with order-preserving codes of b = 1, 2 or 4 bits per character, packed most significant
// bit first; the key of suffix i is then the 64-bit window at bit i*b of that stream: 64, 32 or 16 characters instead of
// 8, so round 0 alone resolves what plain keys need two or three more doubling rounds for (BASELINE config #4: iid
// {A,C,G,T} -- everything outside the tandem repeats is unique after 32 characters).  Past the end the stream is zero,
// which is also the code of the smallest character: the same tie, and the same resolution, as the zero padding of
// plain keys (header comment; the rank kernel's "shorter than the key" rule takes the key length in characters).
struct AlphabetCode {
    uint8_t code[256];  // order-preserving code of every byte value that occurs
    int bits;           // bits per character: 1, 2 or 4 (8 = no recoding, keys come from the text itself)
};

// 256-bin histogram of the text (which byte values occur).  grid-stride, 256 threads
__global__ void __launch_bounds__(256) byte_hist_kernel(const uint8_t *__restrict__ T, uint32_t n,
                                                        uint32_t *__restrict__ hist)
{
    __shared__ uint32_t sh[256];
    sh[threadIdx.x] = 0;
    __syncthreads();
    const uint32_t words = n >> 2;
    const uint32_t *W = reinterpret_cast<const uint32_t *>(T);
    for (uint64_t w = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; w < words; w += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t v = __ldg(W + w);
        atomicAdd(&sh[v & 255u], 1u);
        atomicAdd(&sh[(v >> 8) & 255u], 1u);
        atomicAdd(&sh[(v >> 16) & 255u], 1u);
        atomicAdd(&sh[v >> 24], 1u);
    }
    if (blockIdx.x == 0 && threadIdx.x < (n & 3u)) atomicAdd(&sh[T[(words << 2) + threadIdx.x]], 1u);
    __syncthreads();
    if (sh[threadIdx.x]) atomicAdd(&hist[threadIdx.x], sh[threadIdx.x]);
}

// P[j] = the codes of characters [j * 8/b, (j+1) * 8/b), first character in the most significant bits; characters at
// or past n (and everything up to out_bytes) are zero.  T must be readable up to n.
__global__ void __launch_bounds__(256) encode_text_kernel(const uint8_t *__restrict__ T, uint32_t n,
                                                          const AlphabetCode ac, uint8_t *__restrict__ P,
                                                          uint64_t out_bytes)
{
    __shared__ uint8_t lut[256];
    lut[threadIdx.x] = ac.code[threadIdx.x];
    __syncthreads();
    const uint32_t per = 8u / (uint32_t)ac.bits;
    for (uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; j < out_bytes; j += (uint64_t)gridDim.x * blockDim.x) {
        uint32_t v = 0;
        const uint64_t c0 = j * per;
        for (uint32_t k = 0; k < per; ++k) {
            const uint64_t c = c0 + k;
            v = (v << ac.bits) | (c < n ? (uint32_t)lut[T[c]] : 0u);
        }
        P[j] = (uint8_t)v;
    }
}

// 64-bit window of the packed stream at bit offset i * bits (bits in {1, 2, 4}); P is zero padded by >= 16 bytes
__device__ __forceinline__ uint64_t load_window(const uint8_t *__restrict__ P, uint32_t i, int bits)
{
    const uint64_t bit = (uint64_t)i * (uint64_t)bits;
    const uint32_t j = (uint32_t)(bit >> 3);
    const unsigned s = (unsigned)(bit & 7u);
    const uint64_t k0 = load_key8(P, j);
    return s ? (k0 << s) | ((uint64_t)P[j + 8] >> (8u - s)) : k0;
}

// first characters of suffix i as one key: from the text (bits == 8) or from its packed recoding
__device__ __forceinline__ uint64_t load_key(const uint8_t *__restrict__ T, const uint8_t *__restrict__ P, uint32_t i,
                                            int bits)
{
    return bits == 8 ? load_key8(T, i) : load_window(P, i, bits);
}

// K0: element k stands for suffix i = n-1-k.  keys[k] = first 8 bytes, vals[k] = i; digit histograms of all
// 8 passes are accumulated on the way.  grid-stride; dynamic smem = npass*256*4.
__global__ void __launch_bounds__(kPackThreads)
pack_keys_kernel(const uint8_t *__restrict__ T, uint32_t n, uint64_t *__restrict__ keys,
                 uint32_t *__restrict__ vals, radix::PassPlan plan, uint32_t *__restrict__ ghist,
                 uint32_t *__restrict__ uniform_count, const uint8_t *__restrict__ P = nullptr, int bits = 8)
{
    DQ_DYN_SMEM(smem);
    uint32_t *sh = reinterpret_cast<uint32_t *>(smem);
    for (int i = threadIdx.x; i < plan.npass * radix::kRadix; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    const uint32_t chunk = kPackThreads * kPackItems;
    uint32_t uniform = 0;  // suffixes whose 8-byte key is one repeated byte: they sit inside equal-byte runs
    for (uint64_t base = (uint64_t)blockIdx.x * chunk; base < n; base += (uint64_t)gridDim.x * chunk) {
#pragma unroll
        for (int j = 0; j < kPackItems; ++j) {
            uint64_t k = base + (uint64_t)j * kPackThreads + threadIdx.x;
            if (k < n) {
                const uint32_t i = n - 1u - (uint32_t)k;
                const uint64_t key = load_key(T, P, i, bits);
                keys[k] = key;
                vals[k] = i;
                radix::hist_accumulate(sh, plan, key);
                uniform += key == (key & 0xffull) * 0x0101010101010101ull;
            }
        }
    }
    __syncthreads();
    radix::hist_flush(sh, plan.npass, ghist);
    uniform = __reduce_add_sync(kFullMask, uniform);
    if (lane_id() == 0 && uniform) atomicAdd(uniform_count, uniform);
}

// K6: key[k] = rank[k] << 32 | (sa[k]+d < n ? ISA[sa[k]+d] + 1 : 0), plus the digit histograms.  d = depth[k],
// the number of leading bytes the group of position k is known to share (per active-set position: sorting only
// permutes inside groups, so the array stays put); depth == nullptr means the uniform depth h.
__global__ void __launch_bounds__(kPackThreads)
build_keys_kernel(const uint32_t *__restrict__ sa, const uint32_t *__restrict__ rank,
                  const uint32_t *__restrict__ ISA, uint32_t n, uint32_t a, uint64_t h,
                  const uint32_t *__restrict__ depth, uint64_t *__restrict__ keys, radix::PassPlan plan,
                  uint32_t *__restrict__ ghist)
{
    DQ_DYN_SMEM(smem);
    uint32_t *sh = reinterpret_cast<uint32_t *>(smem);
    for (int i = threadIdx.x; i < plan.npass * radix::kRadix; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    const uint32_t chunk = kPackThreads * kPackItems;
    for (uint64_t base = (uint64_t)blockIdx.x * chunk; base < a; base += (uint64_t)gridDim.x * chunk) {
        uint32_t s[kPackItems], r[kPackItems], r2[kPackItems];
#pragma unroll
        for (int j = 0; j < kPackItems; ++j) {
            uint64_t k = base + (uint64_t)j * kPackThreads + threadIdx.x;
            s[j] = k < a ? sa[k] : 0u;
            r[j] = k < a ? rank[k] : 0u;
        }
#pragma unroll
        for (int j = 0; j < kPackItems; ++j) {
            uint64_t k = base + (uint64_t)j * kPackThreads + threadIdx.x;
            uint64_t p = (uint64_t)s[j] + (depth && k < a ? (uint64_t)depth[k] : h);
            r2[j] = (k < a && p < n) ? __ldg(ISA + p) + 1u : 0u;
        }
#pragma unroll
        for (int j = 0; j < kPackItems; ++j) {
            uint64_t k = base + (uint64_t)j * kPackThreads + threadIdx.x;
            if (k < a) {
                const uint64_t key = ((uint64_t)r[j] << 32) | r2[j];
                keys[k] = key;
                radix::hist_accumulate(sh, plan, key);
            }
        }
    }
    __syncthreads();
    radix::hist_flush(sh, plan.npass, ghist);
}

// K0 for a slice of text positions [pos_begin, pos_begin + count): element k stands for suffix
// pos_begin + count - 1 - k (descending, as in pack_keys_kernel).  T points at the slice (T[0] is text position
// pos_begin), zero padded.  uniform_count (may be null) is incremented by the number of one-repeated-byte keys.
__global__ void __launch_bounds__(kPackThreads)
pack_slice_kernel(const uint8_t *__restrict__ T, uint32_t pos_begin, uint32_t count, uint64_t *__restrict__ keys,
                  uint32_t *__restrict__ vals, uint32_t *__restrict__ uniform_count,
                  const uint8_t *__restrict__ P = nullptr, int bits = 8)
{
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    const uint64_t rounds = (count + stride - 1) / stride;
    uint32_t uniform = 0;  // suffixes whose 8-byte key is one repeated byte (see pack_keys_kernel)
    for (uint64_t r = 0; r < rounds; ++r) {
        const uint64_t k = r * stride + (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (k < count) {
            const uint32_t off = count - 1u - (uint32_t)k;
            const uint64_t key = load_key(T, P, off, bits);
            keys[k] = key;
            vals[k] = pos_begin + off;
            uniform += key == (key & 0xffull) * 0x0101010101010101ull;
        }
    }
    if (uniform_count) {
        uniform = __reduce_add_sync(kFullMask, uniform);
        if (lane_id() == 0 && uniform) atomicAdd(uniform_count, uniform);
    }
}

// ---- batches: many texts in one prefix-doubling sort (dq_cuda_suffix_sort_batch) ------------------------------
// A chunk holds `count` texts back to back in T (compact positions; text t is [offs[t], offs[t+1])).  Suffix positions
// are PADDED positions, compact + t: one sentinel position follows every text, and its ISA entry stays 0xffffffff, so
// build_keys_kernel's ISA[p] + 1 reads 0 exactly at the end of the suffix's own text.  The round-0 key
//     t << 48 | (5 bytes of the suffix, big-endian, bytes at or past the end of text t zeroed) << 8 | min(L, 5)
// sorts the chunk text-major (text t owns the SA slots [offs[t], offs[t+1])), keeps equal suffixes of different texts
// apart, and settles the end-of-text rule inside the key: a suffix shorter than 5 bytes is alone in its group (no other
// suffix of its text has its length), so the rank kernel runs with hmin = 0.  Every unresolved group then shares 5
// bytes and its members are at least 5 long, which is the invariant of the header comment at h = 5.
constexpr int kBatchKeyBytes = 5;
constexpr int kBatchTextShift = 48;

// the text of a chunk that holds compact position k: the largest t with offs[t] <= k (empty texts hold nothing)
__device__ __forceinline__ uint32_t batch_owner(const uint32_t *__restrict__ offs, uint32_t count, uint32_t k)
{
    uint32_t lo = 0, hi = count;  // offs[lo] <= k < offs[hi]
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (__ldg(offs + mid) <= k) lo = mid;
        else hi = mid;
    }
    return lo;
}

// K0 of a chunk: element k stands for the suffix at compact position k; keys[k] = the key above, vals[k] = its padded
// position, and the digit histograms of all passes are accumulated on the way.  T is zero padded by >= 16 bytes.
// grid-stride; dynamic smem = npass*256*4.
__global__ void __launch_bounds__(kPackThreads)
pack_keys_batch_kernel(const uint8_t *__restrict__ T, const uint32_t *__restrict__ offs, uint32_t count, uint32_t n,
                       uint64_t *__restrict__ keys, uint32_t *__restrict__ vals, radix::PassPlan plan,
                       uint32_t *__restrict__ ghist)
{
    DQ_DYN_SMEM(smem);
    uint32_t *sh = reinterpret_cast<uint32_t *>(smem);
    for (int i = threadIdx.x; i < plan.npass * radix::kRadix; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n; k += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t i = (uint32_t)k;
        const uint32_t t = batch_owner(offs, count, i);
        const uint32_t len = min(__ldg(offs + t + 1) - i, (uint32_t)kBatchKeyBytes);
        uint64_t b5 = load_key8(T, i) >> (8 * (8 - kBatchKeyBytes));
        b5 &= ~((1ull << (8 * (kBatchKeyBytes - len))) - 1ull);  // the bytes past the end belong to the next text
        const uint64_t key = ((uint64_t)t << kBatchTextShift) | (b5 << 8) | len;
        keys[k] = key;
        vals[k] = i + t;
        radix::hist_accumulate(sh, plan, key);
    }
    __syncthreads();
    radix::hist_flush(sh, plan.npass, ghist);
}

// SA[s] (a padded position) -> the suffix's index inside its own text, in place; slot s belongs to the text that
// holds compact position s (the chunk is sorted text-major).  grid-stride.
__global__ void __launch_bounds__(256) batch_localize_kernel(int32_t *__restrict__ SA, const uint32_t *__restrict__ offs,
                                                             uint32_t count, uint32_t n)
{
    for (uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; s < n; s += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t t = batch_owner(offs, count, (uint32_t)s);
        SA[s] = (int32_t)((uint32_t)SA[s] - __ldg(offs + t) - t);
    }
}

// ---- equal-byte runs ----------------------------------------------------------------------------------------
// Plain doubling needs log2(L) rounds for the suffixes inside a run of L equal bytes (zero padding in
// executables: the 16 MiB exe-like workload kept 3.5 M suffixes unresolved for 15 rounds).  A suffix inside a run
// of byte b with R bytes of the run left is b^R followed by the suffix at the run's end, which starts with a byte
// c != b (or is empty).  Among suffixes with the same b:
//     c < b (or text end):  shorter run first   (it differs from a longer run at offset R with c < b)
//     c > b             :  longer run first, and the whole "c < b" class sorts before the "c > b" class.
// So after round 0 the groups whose 8-byte key is b^8 are refined in ONE round by the 32-bit key
// (class << 31 | R or 2^31-1-R), and the resulting subgroups share exactly their R run bytes: their depth is R,
// and the next round compares the suffixes at the run ends.
constexpr uint32_t kRunTile = 4096;        // positions per block of the run_end kernels
constexpr uint32_t kDepthFromKey = 0xffffffffu;  // depth[] marker: "this group was refined by run length"

// first run boundary (position j >= 1 with T[j] != T[j-1]) of every tile, or 0xffffffff
__global__ void __launch_bounds__(256) run_tile_first_kernel(const uint8_t *__restrict__ T, uint32_t n,
                                                              uint32_t *__restrict__ tile_first)
{
    __shared__ uint32_t s_min[8];
    const uint64_t base = (uint64_t)blockIdx.x * kRunTile;
    uint32_t mn = 0xffffffffu;
    for (uint32_t o = threadIdx.x; o < kRunTile; o += 256) {
        const uint64_t j = base + o;
        if (j >= 1 && j < n && T[j] != T[j - 1]) mn = min(mn, (uint32_t)j);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mn = min(mn, __shfl_xor_sync(kFullMask, mn, o));
    if (lane_id() == 0) s_min[warp_id()] = mn;
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < 8; ++w) mn = min(mn, s_min[w]);
        tile_first[blockIdx.x] = mn;
    }
}

// next_after[t] = first run boundary in any tile after t, or n.  One block; reverse exclusive min-scan.
__global__ void __launch_bounds__(1024) run_tile_scan_kernel(const uint32_t *__restrict__ tile_first, uint32_t ntiles,
                                                              uint32_t n, uint32_t *__restrict__ next_after)
{
    __shared__ uint32_t s_part[1024];
    const uint32_t per = (ntiles + 1023u) / 1024u;
    const uint32_t lo = threadIdx.x * per, hi = min(ntiles, lo + per);
    uint32_t mn = n;
    for (uint32_t t = lo; t < hi; ++t) mn = min(mn, tile_first[t]);
    s_part[threadIdx.x] = mn;
    __syncthreads();
    uint32_t run = n;  // min over the chunks of higher threads
    for (uint32_t w = threadIdx.x + 1; w < 1024; ++w) run = min(run, s_part[w]);
    for (uint32_t t = hi; t-- > lo;) {
        next_after[t] = run;
        run = min(run, tile_first[t]);
    }
}

// run_end[i] = first position j > i with T[j] != T[i], or n
__global__ void __launch_bounds__(256) run_end_kernel(const uint8_t *__restrict__ T, uint32_t n,
                                                       const uint32_t *__restrict__ next_after,
                                                       uint32_t *__restrict__ run_end)
{
    __shared__ uint32_t s_first[256];
    constexpr uint32_t kPer = kRunTile / 256;  // 16 consecutive positions per thread
    const uint64_t base = (uint64_t)blockIdx.x * kRunTile + (uint64_t)threadIdx.x * kPer;
    uint8_t b[kPer + 1];
#pragma unroll
    for (uint32_t o = 0; o <= kPer; ++o) b[o] = base + o < n ? T[base + o] : 0;
    // first boundary strictly after each of my positions that I can see (up to base + kPer)
    uint32_t nxt[kPer];
    uint32_t cur = 0xffffffffu;
#pragma unroll
    for (int o = (int)kPer - 1; o >= 0; --o) {
        const uint64_t j = base + o + 1;  // boundary candidate between o and o+1
        if (j < n && b[o + 1] != b[o]) cur = (uint32_t)j;
        nxt[o] = cur;
    }
    // first boundary inside my 16 positions (j in (base, base+kPer], plus j = base itself seen from the left)
    uint32_t mine = cur;  // = first boundary in (base, base + kPer]
    s_first[threadIdx.x] = mine;
    __syncthreads();
    uint32_t after = next_after[blockIdx.x];  // first boundary in later tiles
    // boundaries owned by later threads of this tile.  Thread t+1's window (base', base'+kPer] starts where mine ends.
    for (uint32_t w = threadIdx.x + 1; w < 256; ++w) {
        const uint32_t f = s_first[w];
        if (f != 0xffffffffu) {
            after = f;
            break;
        }
    }
#pragma unroll
    for (uint32_t o = 0; o < kPer; ++o)
        if (base + o < n) run_end[base + o] = min(min(nxt[o], after), n);
}

// K6 of round 1: groups whose 8-byte key is one repeated byte are refined by run length (see above) and marked
// kDepthFromKey; every other group by ISA[sa+8]+1 with depth 8 (its new depth is then 16, like plain doubling).
__global__ void __launch_bounds__(kPackThreads)
build_keys_round1_kernel(const uint32_t *__restrict__ sa, const uint32_t *__restrict__ rank,
                         const uint32_t *__restrict__ ISA, const uint8_t *__restrict__ T,
                         const uint32_t *__restrict__ run_end, uint32_t n, uint32_t a, uint64_t *__restrict__ keys,
                         uint32_t *__restrict__ depth, radix::PassPlan plan, uint32_t *__restrict__ ghist)
{
    DQ_DYN_SMEM(smem);
    uint32_t *sh = reinterpret_cast<uint32_t *>(smem);
    for (int i = threadIdx.x; i < plan.npass * radix::kRadix; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < a; k += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t s = sa[k];
        const uint64_t k8 = load_key8(T, s);
        uint32_t r2, d;
        if ((uint64_t)s + 8 <= n && k8 == (k8 & 0xffull) * 0x0101010101010101ull) {
            const uint32_t e = run_end[s];
            const uint32_t R = e - s;
            const uint32_t bb = (uint32_t)(k8 & 0xffu);
            const bool below = e >= n || T[e] < bb;
            r2 = below ? R : (0x80000000u | (0x7fffffffu - R));
            d = kDepthFromKey;
        } else {
            const uint64_t p = (uint64_t)s + 8;
            r2 = p < n ? __ldg(ISA + p) + 1u : 0u;
            d = 8;
        }
        const uint64_t key = ((uint64_t)rank[k] << 32) | r2;
        keys[k] = key;
        depth[k] = d;
        radix::hist_accumulate(sh, plan, key);
    }
    __syncthreads();
    radix::hist_flush(sh, plan.npass, ghist);
}

// digit histograms of an existing key array (used by dq_cuda_radix_sort_pairs only; the suffix sorter's
// producers accumulate their histograms while they write the keys)
__global__ void __launch_bounds__(kPackThreads)
hist_only_kernel(const uint64_t *__restrict__ keys, uint32_t count, radix::PassPlan plan, uint32_t *__restrict__ ghist)
{
    DQ_DYN_SMEM(smem);
    uint32_t *sh = reinterpret_cast<uint32_t *>(smem);
    for (int i = threadIdx.x; i < plan.npass * radix::kRadix; i += blockDim.x) sh[i] = 0;
    __syncthreads();
    for (uint64_t k = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; k < count; k += (uint64_t)gridDim.x * blockDim.x)
        radix::hist_accumulate(sh, plan, keys[k]);
    __syncthreads();
    radix::hist_flush(sh, plan.npass, ghist);
}

// ISA slices of a device group, as the rank kernel needs them in a small round (dq_dist.cuh, IsaParts): shard o owns
// ISA[o << kb, (o + 1) << kb); p[0] == nullptr: not used
struct PeerIsa {
    uint32_t *p[16];
    int kb;
};

// ---- K4+K5: group heads, new ranks, singleton retirement, compaction -- one pass, decoupled look-back ----
constexpr int kRankThreads = 512;
constexpr int kRankItems = 8;
constexpr int kRankTile = kRankThreads * kRankItems;
constexpr int kRankWarps = kRankThreads / 32;

// descriptor: status(2) | last head's slot (31) | survivors (31)
constexpr uint64_t kField31 = 0x7fffffffull;
__host__ __device__ __forceinline__ uint64_t rk_pack(uint32_t mx, uint32_t sm) { return ((uint64_t)mx << 31) | sm; }
__host__ __device__ __forceinline__ uint32_t rk_max(uint64_t v) { return (uint32_t)((v >> 31) & kField31); }
__host__ __device__ __forceinline__ uint32_t rk_sum(uint64_t v) { return (uint32_t)(v & kField31); }

// keys/sa: the sorted active set (a entries).  slot_in == nullptr in round 0 (slot[k] = k).
// hmin: in round 0 the number of characters a key holds (8 for plain keys); later the depth all ranks are consistent to.
// Outputs: ISA, SA, the compacted next active set (sa_out, rank_out, slot_out) and *count_out = its size.
//
// Warp-striped: warp w of the tile owns 32*kRankItems consecutive positions, row j of lane l is position
// base + j*32 + l, so every load and the compacted stores are coalesced.  Head flags and survivor flags live
// as one ballot per row (uniform registers), which turns both scans into bit arithmetic:
//   "slot of the last head at or before me" = shfl from the highest head bit at or below my lane,
//   "survivors before me"                   = popc of the survivor ballot below my lane.
//
// DIST (multi-GPU, dq_dist.cuh / dq_group.inl): this GPU sorts one key bucket that owns the SA slots
// [slot_base, slot_base + bucket size); ISA is partitioned by text position across the GPUs, so instead of
// writing ISA the kernel emits one update (rank << 32 | position) per element (upd, dense, in sorted order) for
// the exchange pass to route to the owners, SA is the bucket-local array (index slot - slot_base), and the next
// active set is written packed the same way (act_out) instead of as sa_out / rank_out.
template <bool ROUND0, bool DIST = false>
__global__ void __launch_bounds__(kRankThreads)
rank_compact_kernel(const uint64_t *__restrict__ keys, const uint32_t *__restrict__ sa,
                    const uint32_t *__restrict__ slot_in, uint32_t a, uint32_t n, uint32_t *__restrict__ ISA,
                    int32_t *__restrict__ SA, uint32_t *__restrict__ sa_out, uint32_t *__restrict__ rank_out,
                    uint32_t *__restrict__ slot_out, uint64_t *__restrict__ lb, uint32_t *__restrict__ tile_ticket,
                    uint32_t *__restrict__ count_out, uint32_t slot_base = 0, uint64_t *__restrict__ upd = nullptr,
                    uint64_t *__restrict__ act_out = nullptr, const uint32_t *__restrict__ depth_in = nullptr,
                    uint32_t *__restrict__ depth_out = nullptr, uint32_t hmin = 0,
                    uint32_t *__restrict__ min_depth_inv = nullptr, const PeerIsa peer_isa = PeerIsa{},
                    uint64_t *__restrict__ late = nullptr, uint32_t *__restrict__ late_count = nullptr)
{
    __shared__ uint32_t s_tile;
    __shared__ uint32_t s_wmax[kRankWarps], s_wsum[kRankWarps];
    __shared__ uint64_t s_excl;

    const unsigned tid = threadIdx.x, lane = lane_id(), warp = warp_id();
    if (tid == 0) s_tile = atomicAdd(tile_ticket, 1u);
    __syncthreads();
    const uint32_t tile = s_tile;
    const uint32_t wbase = tile * (uint32_t)kRankTile + warp * (32u * kRankItems);

    uint64_t key[kRankItems];
    uint32_t s[kRankItems], sl[kRankItems];
    unsigned hb[kRankItems + 1];  // hb[j] = ballot of "a group starts here" over row j; positions >= a count as heads
    unsigned vb[kRankItems];      // ballot of k < a
#pragma unroll
    for (int j = 0; j < kRankItems; ++j) {
        const uint32_t k = wbase + j * 32 + lane;
        const bool valid = k < a;
        key[j] = valid ? keys[k] : 0ull;
        s[j] = valid ? sa[k] : 0u;
        sl[j] = ROUND0 ? slot_base + k : (valid ? slot_in[k] : 0u);
    }
#pragma unroll
    for (int j = 0; j < kRankItems; ++j) {
        const uint32_t k = wbase + j * 32 + lane;
        const bool valid = k < a;
        // previous element: the lane to the left, or (lane 0) a reload of the element before the row
        uint64_t pk = __shfl_up_sync(kFullMask, key[j], 1);
        uint32_t ps = __shfl_up_sync(kFullMask, s[j], 1);
        bool hd = true;
        if (valid && k > 0) {
            if (lane == 0) {
                pk = keys[k - 1];
                if (ROUND0) ps = sa[k - 1];
            }
            hd = key[j] != pk;
            if (ROUND0) hd = hd || (n - ps < hmin);  // the previous suffix is shorter than the key: it stands alone
        }
        hb[j] = __ballot_sync(kFullMask, hd);
        vb[j] = __ballot_sync(kFullMask, valid);
    }
    {   // does a group start right after this warp's last position?
        const uint32_t k = wbase + 32u * kRankItems;
        bool hd = true;
        if (lane == 31 && k < a) {
            hd = keys[k] != key[kRankItems - 1];
            if (ROUND0) hd = hd || (n - s[kRankItems - 1] < hmin);
        }
        hb[kRankItems] = __shfl_sync(kFullMask, hd ? 1u : 0u, 31);
    }

    // survivor ballots and the warp's aggregates
    unsigned sb[kRankItems];
    uint32_t wsum = 0, wmax = 0;
#pragma unroll
    for (int j = 0; j < kRankItems; ++j) {
        const unsigned next = (hb[j] >> 1) | ((hb[j + 1] & 1u) << 31);  // head flag of the element after each lane
        sb[j] = vb[j] & ~(hb[j] & next);
        wsum += __popc(sb[j]);
        const unsigned hm = hb[j] & vb[j];
        const uint32_t last = __shfl_sync(kFullMask, sl[j], hm ? 31 - __clz((int)hm) : 0);
        if (hm) wmax = last;  // slots increase with position: the last head of the last row with one wins
    }
    if (lane == 0) {
        s_wmax[warp] = wmax;
        s_wsum[warp] = wsum;
    }
    __syncthreads();
    uint32_t emax = 0, esum = 0, bmax = 0, bsum = 0;
#pragma unroll
    for (int w = 0; w < kRankWarps; ++w) {
        if ((unsigned)w < warp) {
            emax = max(emax, s_wmax[w]);
            esum += s_wsum[w];
        }
        bmax = max(bmax, s_wmax[w]);
        bsum += s_wsum[w];
    }

    // tile prefix by decoupled look-back: warp 0 inspects 32 predecessors per round trip
    if (warp == 0) {
        const uint64_t agg = rk_pack(bmax, bsum);
        uint32_t xm = 0, xs = 0;
        if (tile > 0) {
            if (lane == 0) st_desc(lb + tile, ((uint64_t)radix::kStatusAggregate << 62) | agg);
            int64_t base = (int64_t)tile - 1;
            for (;;) {
                const int64_t t = base - lane;
                // before tile 0 there is nothing: a virtual inclusive descriptor of zero ends the walk
                const uint64_t v = t >= 0 ? ld_desc(lb + t) : ((uint64_t)radix::kStatusInclusive << 62);
                const unsigned st = (unsigned)(v >> 62);
                const unsigned ready = __ballot_sync(kFullMask, st != 0);
                const unsigned incl = __ballot_sync(kFullMask, st == radix::kStatusInclusive);
                // lanes up to (and including) the nearest inclusive predecessor must all be published
                const unsigned need = incl ? (0xffffffffu >> (31 - (__ffs((int)incl) - 1))) : 0xffffffffu;
                if ((ready & need) != need) {
                    DQ_SPIN_HINT();
                    continue;
                }
                const bool mine = (need >> lane) & 1u;
                xm = max(xm, __reduce_max_sync(kFullMask, mine ? rk_max(v) : 0u));
                xs += __reduce_add_sync(kFullMask, mine ? rk_sum(v) : 0u);
                if (incl) break;
                base -= 32;
            }
        }
        if (lane == 0) {
            const uint64_t excl = rk_pack(xm, xs);
            const uint64_t inc = rk_pack(max(xm, bmax), xs + bsum);
            st_desc(lb + tile, ((uint64_t)radix::kStatusInclusive << 62) | inc);
            s_excl = excl;
            if ((uint64_t)(tile + 1) * kRankTile >= a) *count_out = rk_sum(inc);
        }
    }
    __syncthreads();
    uint32_t carry = max(emax, rk_max(s_excl));  // slot of the last head before this warp's chunk
    uint32_t out = esum + rk_sum(s_excl);        // survivors before this warp's chunk
    uint32_t inv_min = 0;                        // max over my survivors of ~depth (0 = none)

#pragma unroll
    for (int j = 0; j < kRankItems; ++j) {
        const unsigned hm = hb[j] & vb[j];
        const unsigned le = hm & (0xffffffffu >> (31 - lane));  // heads at or below my lane
        const uint32_t mine = __shfl_sync(kFullMask, sl[j], le ? 31 - __clz((int)le) : 0);
        const uint32_t nr = le ? mine : carry;
        const bool valid = (vb[j] >> lane) & 1u;
        if (valid) {
            if (DIST) {
                if (upd) {
                    upd[wbase + j * 32 + lane] = ((uint64_t)nr << 32) | s[j];
                } else if (ROUND0 || nr != (uint32_t)(key[j] >> 32)) {
                    // small round of a device group: the changed rank goes straight to the owner's slice
                    peer_isa.p[s[j] >> peer_isa.kb][s[j] & ((1u << peer_isa.kb) - 1u)] = nr;
                }
            }
            if ((sb[j] >> lane) & 1u) {
                const uint32_t o = out + __popc(sb[j] & lanemask_lt());
                if (!DIST && (ROUND0 || nr != (uint32_t)(key[j] >> 32))) ISA[s[j]] = nr;
                if (DIST) {
                    act_out[o] = ((uint64_t)nr << 32) | s[j];
                } else {
                    sa_out[o] = s[j];
                    rank_out[o] = nr;
                }
                slot_out[o] = sl[j];
                if (depth_out) {
                    // bytes the (sub)group now shares: a run-length refined group shares exactly its run, any
                    // other group gained at least hmin bytes (every rank is consistent to depth hmin)
                    const uint32_t din = depth_in[wbase + j * 32 + lane];
                    uint32_t dn;
                    if (din == kDepthFromKey) {
                        const uint32_t r2 = (uint32_t)key[j];
                        dn = (r2 & 0x80000000u) ? 0x7fffffffu - (r2 & 0x7fffffffu) : r2;
                    } else {
                        dn = din + hmin;
                    }
                    depth_out[o] = dn;
                    inv_min = max(inv_min, ~dn);
                }
            } else {
                SA[sl[j] - slot_base] = (int32_t)s[j];
                if (!DIST) ISA[s[j]] = nr;
            }
        }
        if (!ROUND0 && late) {
            // the suffix array is already on its way to the host (see sort_resident, "early copy"): slots resolved from
            // now on are listed as (slot << 32 | suffix) and patched into the host array once that copy has landed
            const unsigned rb = vb[j] & ~sb[j];
            if (rb) {
                uint32_t base = 0;
                if (lane == 0) base = atomicAdd(late_count, (uint32_t)__popc(rb));
                base = __shfl_sync(kFullMask, base, 0);
                if ((rb >> lane) & 1u) late[base + __popc(rb & lanemask_lt())] = ((uint64_t)sl[j] << 32) | s[j];
            }
        }
        out += __popc(sb[j]);
        if (hm) carry = __shfl_sync(kFullMask, sl[j], 31 - __clz((int)hm));
    }
    if (min_depth_inv) {
        // smallest depth among the unresolved groups = the depth every rank is consistent to next round
        inv_min = __reduce_max_sync(kFullMask, inv_min);
        if (lane == 0 && inv_min) atomicMax(min_depth_inv, inv_min);
    }
}

// host_sa[slot] = suffix for every listed pair: host_sa is pinned host memory mapped into the device's address space
__global__ void __launch_bounds__(256) patch_host_sa_kernel(const uint64_t *__restrict__ late,
                                                            const uint32_t *__restrict__ late_count,
                                                            int32_t *__restrict__ host_sa)
{
    const uint32_t cnt = *late_count;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < cnt; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t v = late[i];
        host_sa[(uint32_t)(v >> 32)] = (int32_t)(uint32_t)v;
    }
}

// ---- small inputs: the whole sort in one CTA ----------------------------------------------------------------
// The multi-kernel path costs ~17 stream operations (~130 us) whatever n is; the reference's own benchmark
// (bench/DeltaQ.Benchmarks/SuffixSortingBenchmarks.cs:27-53) is mostly sizes <= 32 KiB.  For n <= kSmallN one
// CTA keeps text, keys, suffix indices and ISA in shared memory and runs the same prefix doubling with a bitonic
// sort: one launch.  Round 0 orders equal 8-byte keys by descending suffix index (the end-of-text rule above).
constexpr int kSmallN = 4096;
constexpr int kSmallThreads = 1024;
constexpr size_t small_sort_smem_bytes() { return (size_t)kSmallN * (8 + 4 + 4) + kSmallN + 64 + 256; }

constexpr uint32_t kSmallPad = 0xffffffffu;  // index of the padding elements of the bitonic sort

// (key ascending, suffix index descending), padding behind every real element
__device__ __forceinline__ bool small_less(uint64_t ka, uint32_t ia, uint64_t kb, uint32_t ib)
{
    return ka < kb || (ka == kb && ia != kSmallPad && (ib == kSmallPad || ia > ib));
}

__global__ void __launch_bounds__(kSmallThreads)
small_sort_kernel(const uint8_t *__restrict__ T, uint32_t n, int32_t *__restrict__ SA, uint32_t *__restrict__ ISA)
{
    DQ_DYN_SMEM(smem);
    uint64_t *key = reinterpret_cast<uint64_t *>(smem);
    uint32_t *idx = reinterpret_cast<uint32_t *>(smem + (size_t)kSmallN * 8);
    uint32_t *isa = idx + kSmallN;
    uint8_t *txt = reinterpret_cast<uint8_t *>(isa + kSmallN);
    uint32_t *misc = reinterpret_cast<uint32_t *>(txt + kSmallN + 64);  // [0] = number of groups, [1..33] warp maxima
    const unsigned tid = threadIdx.x;
    uint32_t N = 1;
    while (N < n) N <<= 1;  // bitonic size

    for (uint32_t i = tid; i < (uint32_t)kSmallN + 64; i += kSmallThreads) txt[i] = i < n ? T[i] : 0;
    __syncthreads();
    for (uint32_t i = tid; i < N; i += kSmallThreads) {
        uint64_t k8 = ~0ull;
        if (i < n) {
            k8 = 0;
#pragma unroll
            for (int b = 0; b < 8; ++b) k8 = (k8 << 8) | txt[i + b];
        }
        key[i] = k8;
        idx[i] = i < n ? i : kSmallPad;  // padding: largest key, and behind any real suffix that has that key too
    }
    __syncthreads();

    for (uint64_t h = 8;; h *= 2) {
        // bitonic sort of (key, idx) ascending by small_less
        for (uint32_t size = 2; size <= N; size <<= 1) {
            for (uint32_t stride = size >> 1; stride > 0; stride >>= 1) {
                for (uint32_t t = tid; t < (N >> 1); t += kSmallThreads) {
                    const uint32_t lo = 2 * t - (t & (stride - 1));
                    const uint32_t hi = lo + stride;
                    const bool up = (lo & size) == 0;
                    const uint64_t ka = key[lo], kb = key[hi];
                    const uint32_t ia = idx[lo], ib = idx[hi];
                    const bool swap = up ? small_less(kb, ib, ka, ia) : small_less(ka, ia, kb, ib);
                    if (swap) {
                        key[lo] = kb;
                        key[hi] = ka;
                        idx[lo] = ib;
                        idx[hi] = ia;
                    }
                }
                __syncthreads();
            }
        }
        // group heads and ranks (rank = position of the group head); positions >= n are padding
        if (tid == 0) misc[0] = 0;
        __syncthreads();
        constexpr uint32_t kPer = kSmallN / kSmallThreads;  // 4 consecutive positions per thread
        uint32_t head_pos[kPer];
        uint32_t last = 0, heads = 0;
#pragma unroll
        for (uint32_t o = 0; o < kPer; ++o) {
            const uint32_t k = tid * kPer + o;
            bool hd = false;
            if (k < n) {
                hd = k == 0 || key[k] != key[k - 1];
                if (h == 8 && k > 0 && n - idx[k - 1] < 8u) hd = true;  // the previous suffix is shorter than the key
            }
            if (hd) {
                last = k;
                heads++;
            }
            head_pos[o] = last;  // last head at or before k within this thread (0 if none yet)
        }
        // block max-scan of `last` (heads positions increase with k)
        uint32_t incl = last;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(kFullMask, incl, o);
            if (lane_id() >= (unsigned)o) incl = max(incl, v);
        }
        if (lane_id() == 31) misc[1 + warp_id()] = incl;
        heads = __reduce_add_sync(kFullMask, heads);
        if (lane_id() == 0 && heads) atomicAdd(&misc[0], heads);
        __syncthreads();
        uint32_t before = __shfl_up_sync(kFullMask, incl, 1);
        if (lane_id() == 0) before = 0;
        for (unsigned w = 0; w < warp_id(); ++w) before = max(before, misc[1 + w]);
        // new keys need the ranks of the PREVIOUS round in isa[]: first ranks into registers, then all keys, then isa
        uint32_t rk[kPer];
#pragma unroll
        for (uint32_t o = 0; o < kPer; ++o) rk[o] = max(head_pos[o], before);
        const bool done = misc[0] == n;
        __syncthreads();
#pragma unroll
        for (uint32_t o = 0; o < kPer; ++o) {
            const uint32_t k = tid * kPer + o;
            if (k < n) isa[idx[k]] = rk[o];
        }
        __syncthreads();
        if (done) break;
        const uint64_t hn = h;  // this round sorted to depth h; the next key looks h bytes ahead
#pragma unroll
        for (uint32_t o = 0; o < kPer; ++o) {
            const uint32_t k = tid * kPer + o;
            if (k < n) {
                const uint64_t p = (uint64_t)idx[k] + hn;
                key[k] = ((uint64_t)rk[o] << 32) | (p < n ? isa[p] + 1u : 0u);
            }
        }
        __syncthreads();
    }
    for (uint32_t k = tid; k < n; k += kSmallThreads) {
        SA[k] = (int32_t)idx[k];
        ISA[k] = isa[k];
    }
}

}  // namespace suffix
}  // namespace dq
