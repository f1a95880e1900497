// dq_radix.cuh -- onesweep-style least-significant-digit radix sort of (uint64 key, uint32 value) pairs.
//
// One kernel launch per digit.  Digit histograms for ALL passes are accumulated up front by the kernel
// that produces the keys (pack_keys / build_keys in dq_suffix.cuh), so a pass reads each pair once and
// writes it once: 24 algorithmic bytes per pair per pass.  Tile digit offsets come from a decoupled
// look-back over per-tile digit counts (one descriptor per tile per digit), tile order comes from an
// atomic ticket so that a tile only ever waits on tiles that already started.
//
// Replaces (by result, not by method) the comparison sorts of the reference's suffix sorters:
//   /root/reference/src/DeltaQ.SuffixSorting.LibDivSufSort/SsSort.cs:23 (sssort),
//   /root/reference/src/DeltaQ.SuffixSorting.LibDivSufSort/TrSort.cs:19 (trsort).
#pragma once
#include "dq_common.cuh"

namespace dq {
namespace radix {

constexpr int kRadixBits = 8;
constexpr int kRadix = 1 << kRadixBits;
constexpr int kMaxPasses = 8;

#ifndef DQ_PASS_ITEMS
#define DQ_PASS_ITEMS 16
#endif
#ifndef DQ_PASS_MIN_BLOCKS
#define DQ_PASS_MIN_BLOCKS 3
#endif
constexpr int kThreads = 256;  // == kRadix: thread d owns digit d in the look-back
constexpr int kItems = DQ_PASS_ITEMS;
constexpr int kWarps = kThreads / 32;
constexpr int kTile = kThreads * kItems;

struct PassPlan {
    int npass;
    int shift[kMaxPasses];
    int bits[kMaxPasses];
};

// cover key bits [lo, lo+nbits) with digits of <= 8 bits, as evenly as possible
inline void plan_add_field(PassPlan &p, int lo, int nbits)
{
    if (nbits <= 0) return;
    int nd = (nbits + kRadixBits - 1) / kRadixBits;
    int base = nbits / nd, extra = nbits % nd;
    for (int i = 0; i < nd; ++i) {
        int b = base + (i < extra ? 1 : 0);
        p.shift[p.npass] = lo;
        p.bits[p.npass] = b;
        p.npass++;
        lo += b;
    }
}

// ---- digit histograms, accumulated by the key producers ------------------------------------------------
// sh: shared [npass][kRadix] counters, zeroed by the caller block
__device__ __forceinline__ void hist_accumulate(uint32_t *sh, const PassPlan &plan, uint64_t key)
{
#pragma unroll
    for (int p = 0; p < kMaxPasses; ++p) {
        if (p < plan.npass) {
            uint32_t d = (uint32_t)(key >> plan.shift[p]) & ((1u << plan.bits[p]) - 1u);
            atomicAdd(&sh[p * kRadix + d], 1u);
        }
    }
}

__device__ __forceinline__ void hist_flush(const uint32_t *sh, int npass, uint32_t *ghist)
{
    for (int i = threadIdx.x; i < npass * kRadix; i += blockDim.x) {
        uint32_t c = sh[i];
        if (c) atomicAdd(&ghist[i], c);
    }
}

// exclusive scan of each pass's 256 counters: ghist[p][d] -> gbase[p][d].  grid = npass, block = 256.
// Also decides how the pass ranks its items (see match_digit): use_match[p] = 1 when a warp row of 32 items is
// expected to hold at most kMatchMaxDistinct distinct digits.  force_mask bit p: the caller knows pass p's digits
// are locally ordered (rank digits of the doubling rounds), skip the estimate there.
constexpr float kMatchMaxDistinct = 16.0f;

__global__ void __launch_bounds__(kRadix) scan_hist_kernel(const uint32_t *__restrict__ ghist,
                                                          uint32_t *__restrict__ gbase,
                                                          uint32_t *__restrict__ use_match, uint32_t total,
                                                          uint32_t force_mask)
{
    __shared__ uint32_t warp_tot[kRadix / 32];
    __shared__ float warp_exp[kRadix / 32];
    const unsigned d = threadIdx.x;
    const uint32_t c = ghist[blockIdx.x * kRadix + d];
    uint32_t incl = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        uint32_t t = __shfl_up_sync(kFullMask, incl, o);
        if (lane_id() >= (unsigned)o) incl += t;
    }
    // expected number of distinct digits among 32 independent draws: sum_d 1 - (1 - p_d)^32
    float e = 0.f;
    if (c) {
        float q = 1.f - (float)c / (float)total;
        q *= q; q *= q; q *= q; q *= q; q *= q;  // ^32
        e = 1.f - q;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) e += __shfl_xor_sync(kFullMask, e, o);
    if (lane_id() == 31) warp_tot[warp_id()] = incl;
    if (lane_id() == 0) warp_exp[warp_id()] = e;
    __syncthreads();
    uint32_t woff = 0;
    for (unsigned w = 0; w < warp_id(); ++w) woff += warp_tot[w];
    gbase[blockIdx.x * kRadix + d] = woff + incl - c;
    if (d == 0) {
        float tot = 0.f;
        for (int w = 0; w < kRadix / 32; ++w) tot += warp_exp[w];
        use_match[blockIdx.x] = (((force_mask >> blockIdx.x) & 1u) || tot <= kMatchMaxDistinct) ? 1u : 0u;
    }
}

// lanes of the warp whose digit equals this lane's.  MATCH.ANY costs time proportional to the number of
// DISTINCT digits in the warp row (measured on B200: uniform digits 2.1 TB/s with MATCH vs 2.8 TB/s with
// ballots; locally ordered digits 3.0-3.4 TB/s with MATCH vs 2.5-2.7 with ballots); one ballot per digit bit
// costs the same whatever the data.  The choice is made once per pass by scan_hist_kernel.
template <bool USE_MATCH>
__device__ __forceinline__ unsigned match_digit(uint32_t d, int nbits)
{
    if (USE_MATCH) return __match_any_sync(kFullMask, d);
    unsigned peers = kFullMask;
#pragma unroll
    for (int b = 0; b < kRadixBits; ++b) {
        if (b < nbits) {
            const bool bit = (d >> b) & 1u;
            const unsigned bal = __ballot_sync(kFullMask, bit);
            peers &= bit ? bal : ~bal;
        }
    }
    return peers;
}

// ---- look-back descriptors -----------------------------------------------------------------------------
template <typename DescT> struct Desc;
template <> struct Desc<uint32_t> {
    static constexpr int kValBits = 30;
};
template <> struct Desc<uint64_t> {
    static constexpr int kValBits = 62;
};
constexpr unsigned kStatusAggregate = 1, kStatusInclusive = 2;

// One LSD pass.  grid = #tiles, block = kThreads, dynamic smem = pass_smem_bytes().
//   lb          [#tiles][kRadix] descriptors, zero before the launch
//   tile_ticket one counter, zero before the launch
//   gbase       [kRadix] exclusive digit offsets of this pass over the whole input
//
// Order of work inside a tile (what the ncu captures in profiles/ asked for):
//   1. load keys; count digits per warp with shared-memory atomics ("early counts");
//   2. thread d publishes digit d's tile count at once, so successors never wait on this tile's ranking;
//   3. look-back immediately, kLookWindow predecessors per round trip (independent loads), publish inclusive;
//   4. stable ranking (match_any within the warp, running per-warp counters that already include the tile
//      and warp offsets) writes every key straight to its slot of the shared staging area;
//   5. values (requested before the look-back) are staged through the same slots; coalesced write-out.
#ifndef DQ_LOOK_WINDOW
#define DQ_LOOK_WINDOW 8
#endif
constexpr int kLookWindow = DQ_LOOK_WINDOW;

constexpr size_t pass_smem_bytes()
{
    return (size_t)kTile * 8 + (size_t)kTile * 4 + (size_t)kWarps * kRadix * 4 + kRadix * 4 + 128;
}


// ---- what a pass sorts by and where it puts the result ------------------------------------------------------
// A policy names the digit of a key and stores one ranked pair.  `dst` is the pair's index inside the output
// sequence of its digit, counted from gbase[digit] (for the plain pass: the global output index).
// digit of a pair under a policy: from the key alone, or -- kDigitFromVal -- from key and value
template <typename Policy>
__device__ __forceinline__ uint32_t digit_of(const Policy &pol, uint64_t key, uint32_t val)
{
    if constexpr (Policy::kDigitFromVal)
        return pol.digit(key, val);
    else
        return pol.digit(key);
}

struct PlainPolicy {
    static constexpr bool kHasVal = true;
    static constexpr bool kDigitFromVal = false;
    int shift;
    uint32_t mask;
    uint64_t *__restrict__ kout;
    uint32_t *__restrict__ vout;
    __device__ __forceinline__ uint32_t digit(uint64_t key) const { return (uint32_t)(key >> shift) & mask; }
    __device__ __forceinline__ int nbits() const { return __popc(mask); }
    __device__ __forceinline__ void store(uint32_t, uint32_t dst, uint64_t key, uint32_t val) const
    {
        kout[dst] = key;
        vout[dst] = val;
    }
};

// stable rank of every item of the warp among the tile's items with the same digit; wh[] = the warp's
// running counters, pre-loaded with (slot of the digit in the tile) + (items of earlier warps)
template <bool FULL, bool USE_MATCH, typename Policy>
__device__ __forceinline__ void rank_and_stage(const uint64_t (&key)[kItems], const uint32_t (&val)[kItems],
                                               uint32_t (&rk)[kItems / 2], uint32_t *wh, uint64_t *skeys, uint32_t wbase,
                                               uint32_t tile_count, const Policy &pol, int nbits)
{
    const unsigned lane = lane_id();
#pragma unroll
    for (int j = 0; j < kItems; ++j) {
        const uint32_t dj = digit_of(pol, key[j], val[j]);
        unsigned peers = match_digit<USE_MATCH>(dj, nbits);
        bool valid = true;
        if (!FULL) {
            valid = wbase + j * 32 < tile_count;
            peers &= __ballot_sync(kFullMask, valid);
        }
        const int leader = valid ? (__ffs(peers) - 1) : (int)lane;
        uint32_t before = 0;
        if (valid && (int)lane == leader) {
            before = wh[dj];
            wh[dj] = before + __popc(peers);
        }
        before = __shfl_sync(kFullMask, before, leader);
        const uint32_t r = before + __popc(peers & lanemask_lt());
        if (valid) skeys[r] = key[j];
        if (j & 1)
            rk[j >> 1] |= r << 16;
        else
            rk[j >> 1] = r;
        __syncwarp();
    }
}

template <typename DescT, bool FULL, typename Policy>
__device__ __forceinline__ void onesweep_tile(const uint64_t *__restrict__ kin, const uint32_t *__restrict__ vin,
                                              const Policy &pol, uint32_t tile, uint32_t tile_count,
                                              const uint32_t *__restrict__ gbase, DescT *__restrict__ lb,
                                              uint64_t *skeys, uint32_t *svals, uint32_t *whist, uint32_t *sout,
                                              uint32_t *smisc, bool few_distinct)
{
    const unsigned tid = threadIdx.x, lane = lane_id(), warp = warp_id();
    const uint32_t tile_base = tile * (uint32_t)kTile;

    // ---- 1. keys, warp-striped: item j of lane l in warp w is tile_base + w*32*kItems + j*32 + l
    uint64_t key[kItems];
    const uint32_t wbase = warp * (32 * kItems) + lane;
#pragma unroll
    for (int j = 0; j < kItems; ++j) {
        const uint32_t li = wbase + j * 32;
        key[j] = (FULL || li < tile_count) ? ld_stream(kin + tile_base + li) : ~0ull;
    }
    // values: requested after the early counts, so that they land during the look-back and the ranking -- unless the
    // digit depends on them
    uint32_t val[kItems];
    if (Policy::kDigitFromVal) {
#pragma unroll
        for (int j = 0; j < kItems; ++j) {
            const uint32_t li = wbase + j * 32;
            val[j] = (FULL || li < tile_count) ? ld_stream(vin + tile_base + li) : 0u;
        }
    }
    uint32_t *wh = whist + warp * kRadix;
#pragma unroll
    for (int j = 0; j < kItems; ++j)
        if (FULL || wbase + j * 32 < tile_count) atomicAdd(&wh[digit_of(pol, key[j], val[j])], 1u);
    __syncthreads();

    // ---- 2. thread d: tile count of digit d, published immediately
    constexpr int VB = Desc<DescT>::kValBits;
    constexpr DescT kValMask = ((DescT)1 << VB) - 1;
    const unsigned d = tid;
    uint32_t cw[kWarps];
    uint32_t sum = 0;
#pragma unroll
    for (int w = 0; w < kWarps; ++w) {
        cw[w] = whist[w * kRadix + d];
        sum += cw[w];
    }
    DescT *my = lb + (size_t)tile * kRadix + d;
    if (tile > 0) st_desc(my, ((DescT)kStatusAggregate << VB) | (DescT)sum);
    const int nbits = pol.nbits();

    // values are requested now and land during the look-back and the ranking
    if (!Policy::kDigitFromVal) {
#pragma unroll
        for (int j = 0; j < kItems; ++j) {
            const uint32_t li = wbase + j * 32;
            val[j] = (Policy::kHasVal && (FULL || li < tile_count)) ? ld_stream(vin + tile_base + li) : 0u;
        }
    }

    // exclusive scan of the 256 digit counts -> first slot of each digit inside the tile
    uint32_t incl = sum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(kFullMask, incl, o);
        if (lane >= (unsigned)o) incl += t;
    }
    if (lane == 31) smisc[1 + warp] = incl;
    __syncthreads();
    uint32_t first = incl - sum;
    for (unsigned w = 0; w < warp; ++w) first += smisc[1 + w];
    {   // running counters of the ranking start at (slot of the digit in the tile) + (items of earlier warps)
        uint32_t run = first;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) {
            whist[w * kRadix + d] = run;
            run += cw[w];
        }
    }

    // ---- 3. look-back: kLookWindow predecessors per round trip
    DescT excl = 0;
    if (tile > 0) {
        int64_t t = (int64_t)tile - 1;
        bool done = false;
        while (!done) {
            DescT v[kLookWindow];
#pragma unroll
            for (int i = 0; i < kLookWindow; ++i)
                v[i] = (t - i >= 0) ? ld_desc(lb + (size_t)(t - i) * kRadix + d) : ((DescT)kStatusInclusive << VB);
            int used = 0;
#pragma unroll
            for (int i = 0; i < kLookWindow; ++i) {
                if (!done && used == i) {
                    const unsigned st = (unsigned)(v[i] >> VB);
                    if (st != 0) {
                        excl += v[i] & kValMask;
                        used = i + 1;
                        if (st == kStatusInclusive) done = true;
                    }
                }
            }
            t -= used;
            if (!done && used == 0) DQ_SPIN_HINT();
        }
    }
    st_desc(my, ((DescT)kStatusInclusive << VB) | (excl + (DescT)sum));
    sout[d] = gbase[d] + (uint32_t)excl - first;
    __syncthreads();

    // ---- 4. stable ranking; keys go straight to their slot
    uint32_t rk[kItems / 2];  // two 16-bit slots per register (slots are < kTile <= 65536)
    if (few_distinct)
        rank_and_stage<FULL, true>(key, val, rk, wh, skeys, wbase, tile_count, pol, nbits);
    else
        rank_and_stage<FULL, false>(key, val, rk, wh, skeys, wbase, tile_count, pol, nbits);
    // ---- 5. values through the same slots, then stream the tile out
    if (Policy::kHasVal) {
#pragma unroll
        for (int j = 0; j < kItems; ++j)
            if (FULL || wbase + j * 32 < tile_count) svals[(rk[j >> 1] >> (16 * (j & 1))) & 0xffffu] = val[j];
    }
    __syncthreads();
#pragma unroll
    for (int j = 0; j < kItems; ++j) {
        const uint32_t i = tid + j * kThreads;
        if (FULL || i < tile_count) {
            const uint64_t k = skeys[i];
            const uint32_t v = Policy::kHasVal ? svals[i] : 0u;
            const uint32_t dg = digit_of(pol, k, v);
            pol.store(dg, sout[dg] + i, k, v);
        }
    }
}

template <typename DescT, typename Policy>
__device__ __forceinline__ void onesweep_pass_body(const uint64_t *__restrict__ kin, const uint32_t *__restrict__ vin,
                                                   const Policy &pol, uint32_t count,
                                                   const uint32_t *__restrict__ gbase, DescT *__restrict__ lb,
                                                   uint32_t *__restrict__ tile_ticket,
                                                   const uint32_t *__restrict__ use_match)
{
    DQ_DYN_SMEM(smem);
    uint64_t *skeys = reinterpret_cast<uint64_t *>(smem);
    uint32_t *svals = reinterpret_cast<uint32_t *>(smem + (size_t)kTile * 8);
    uint32_t *whist = svals + kTile;            // [kWarps][kRadix]
    uint32_t *sout = whist + kWarps * kRadix;   // [kRadix] global slot of staged item i with digit d = sout[d] + i
    uint32_t *smisc = sout + kRadix;

    const unsigned tid = threadIdx.x;
    const uint32_t ntiles = (count + (uint32_t)kTile - 1u) / (uint32_t)kTile;
    if (tid == 0) {
        smisc[0] = atomicAdd(tile_ticket, 1u);
        smisc[16] = *use_match;
    }
    for (int i = tid; i < kWarps * kRadix; i += kThreads) whist[i] = 0;
    __syncthreads();
    const uint32_t tile = smisc[0];
    const bool few = smisc[16] != 0;
    if (tile >= ntiles) return;
    const uint32_t tile_base = tile * (uint32_t)kTile;
    const uint32_t tile_count = min((uint32_t)kTile, count - tile_base);
    if (tile_count == (uint32_t)kTile)
        onesweep_tile<DescT, true>(kin, vin, pol, tile, tile_count, gbase, lb, skeys, svals, whist, sout, smisc, few);
    else
        onesweep_tile<DescT, false>(kin, vin, pol, tile, tile_count, gbase, lb, skeys, svals, whist, sout, smisc, few);
}

template <typename DescT>
__global__ void __launch_bounds__(kThreads, DQ_PASS_MIN_BLOCKS)
onesweep_pass_kernel(const uint64_t *__restrict__ kin, const uint32_t *__restrict__ vin,
                     uint64_t *__restrict__ kout, uint32_t *__restrict__ vout, uint32_t count, int shift,
                     uint32_t mask, const uint32_t *__restrict__ gbase, DescT *__restrict__ lb,
                     uint32_t *__restrict__ tile_ticket, const uint32_t *__restrict__ use_match)
{
    const PlainPolicy pol{shift, mask, kout, vout};
    onesweep_pass_body<DescT>(kin, vin, pol, count, gbase, lb, tile_ticket, use_match);
}

// The same pass with a caller-defined digit and destination (dq_dist.cuh: partition + peer-memory exchange in one
// kernel).  Counts are < 2^30 on this path (one shard's share of an int32-sized text).
template <typename Policy>
__global__ void __launch_bounds__(kThreads, DQ_PASS_MIN_BLOCKS)
onesweep_policy_kernel(const uint64_t *__restrict__ kin, const uint32_t *__restrict__ vin, const Policy pol,
                       uint32_t count, const uint32_t *__restrict__ gbase, uint32_t *__restrict__ lb,
                       uint32_t *__restrict__ tile_ticket, const uint32_t *__restrict__ use_match)
{
    onesweep_pass_body<uint32_t>(kin, vin, pol, count, gbase, lb, tile_ticket, use_match);
}

}  // namespace radix
}  // namespace dq
