// deltaq_cuda.cu -- context, host orchestration and the C ABI of libdeltaq_cuda (include/deltaq_cuda.h).
//
// There is no CPU fallback in this library: without a CUDA device dq_cuda_create fails with
// DQ_ERR_NO_DEVICE.  (The g++ -DDQ_EMU build of this file is the test-side logic emulator, see
// tests/emu/cuda_emu.h; it is never shipped or loaded by the product package.)
#include "../../include/deltaq_cuda.h"

#if defined(__linux__)
#include <sys/mman.h>
#include <sys/syscall.h>
#include <unistd.h>
#endif

#include <algorithm>
#include <chrono>
#include <functional>
#include <memory>
#include <thread>
#include <utility>
#include <cstdlib>
#include <mutex>
#include <new>
#include <stdexcept>
#include <string>
#include <vector>

#include "dq_common.cuh"
#include "dq_radix.cuh"
#include "dq_suffix.cuh"
#include "dq_search.cuh"
#include "dq_dist.cuh"
#include "dq_diff_host.h"
#include "dq_patch_host.h"
#include "dq_bz2_host.h"

namespace {

std::string g_create_error;

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
    template <typename T> T *as() const { return static_cast<T *>(p); }
};

struct EventPair {
    cudaEvent_t a, b;
    uint64_t pairs;
    int shift;
    float ms;
};

struct PinBuf {
    void *p = nullptr;
    size_t cap = 0;
};

// one doubling round of the last sort (timing on): event at its start, what entered it, how many radix passes
struct RoundRec {
    cudaEvent_t begin;
    uint64_t active;
    int passes;
    float ms;
};

struct Group;  // dq_group.inl: the shards of a context created with ndev > 1

// what a context's text / sa / isa hold and what is built from them (include/deltaq_cuda.h, "the resident index")
struct Resident {
    int32_t n = -1;       // length of the text they hold; -1: nothing
    int32_t rounds = -1;  // doubling rounds of the sort that produced sa; -1: the caller's SA
    bool runs = false;    // runend[] holds the run ends of this text (run-aware sort)
    bool lcp = false;     // lcp + block-minimum levels + bucket bounds are built
    bool pre3 = false;    // the 3-byte prefix table is built
};

}  // namespace

struct dq_ctx {
    Group *group = nullptr;
    int device = 0;
    int sm_count = 148;
    cudaStream_t stream = nullptr;
    std::mutex mu;
    std::string err;
    dq_stats stats{};
    bool timing = false;

    // suffix-sort state (device)
    DevBuf text, keyA, keyB, valA, valB, isa, sa, slotA, slotB, lb, hist, auxK, auxV, partK, partV, runend, depthA, depthB,
        runtile, runend_new, runtile_new, seedp, seedl, pre3, pre3tile, packed, late, boffs;
    uint32_t *h_count = nullptr;  // pinned
    Resident res;
    cudaEvent_t ev_copy = nullptr;  // early copy of the suffix array: started / landed
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_index = nullptr;  // ev_index: the search's index of `old` is built
    std::vector<EventPair> pass_events;
    size_t pass_events_used = 0;
    std::vector<RoundRec> round_recs;
    size_t rounds_used = 0;

    // search state (device)
    DevBuf newtext, s_pos, s_len, lcp, headp, headl, bkt, phi, plcp;
    DevBuf bisa, blevels, btab;   // dq_cuda_bsdiff_search_batch: a chunk's local ranks, block minima, per-pair tables
    int32_t runend_new_m = -1;    // runend_new[] describes ctx->newtext of this length
    bool search_seen = false; // this context has run a match search: sorts prepare the 3-byte prefix table on the way

    // pipelined D2H of the (pos, len) table for dq_cuda_bsdiff_streams
    cudaStream_t copy_stream = nullptr;
    cudaStream_t slice_stream[8] = {};  // one per table slice, so the tail of one slice's chains overlaps the next
    cudaEvent_t heads_done = nullptr;  // search_heads_kernel (and all before it) finished
    cudaEvent_t slice_ready[8] = {}, slice_done[8] = {};  // slice's chains finished / slice's code bytes on the host
    int32_t slice_end[8] = {};
    int slices_used = 0;

    // diff streams (host)
    dq::diffhost::Streams streams;
    dq::bz2host::RawBuf patch;  // dq_cuda_bsdiff_patch: the BSDIFF40 file
    PinBuf h_pos, h_len;             // full table: fallback only
    PinBuf h_code, h_heads, h_tiles; // coded table (encode_table_kernel)
    DevBuf d_code, d_headcount;
    uint32_t heads_cap = 0, heads_cap_override = 0;  // override: DQ_HEADS_CAP, to exercise the fallback in tests
};

namespace {

using dq::div_up;
namespace rx = dq::radix;
namespace sx = dq::suffix;

#define DQ_CK(ctx, call)                                                                          \
    do {                                                                                          \
        cudaError_t e_ = (call);                                                                  \
        if (e_ != cudaSuccess) {                                                                  \
            (ctx)->err = std::string(#call) + ": " + cudaGetErrorString(e_);                      \
            return e_ == cudaErrorMemoryAllocation ? DQ_ERR_OUT_OF_MEMORY : DQ_ERR_CUDA;          \
        }                                                                                         \
    } while (0)

#define DQ_TRY(expr)             \
    do {                         \
        int rc_ = (expr);        \
        if (rc_ != DQ_OK) return rc_; \
    } while (0)

int ensure(dq_ctx *ctx, DevBuf &b, size_t bytes)
{
    if (b.cap >= bytes && b.p) return DQ_OK;
    if (b.p) {
        DQ_CK(ctx, cudaFree(b.p));
        b.p = nullptr;
        b.cap = 0;
    }
    size_t want = std::max<size_t>(bytes, 256);
    want = (want + 255) & ~(size_t)255;
    DQ_CK(ctx, cudaMalloc(&b.p, want));
    b.cap = want;
    return DQ_OK;
}

int bit_length(uint64_t v)
{
    int b = 0;
    while (v) {
        ++b;
        v >>= 1;
    }
    return b;
}

struct SortBufs {
    uint64_t *kin, *kout;
    uint32_t *vin, *vout;
};

// Sorts `count` pairs in (s.kin, s.vin) by the digits of `plan`; histograms for all passes are already
// in ctx->hist ([npass][256] counters at offset 0).  On return the sorted pairs are in (s.kin, s.vin).
int run_passes(dq_ctx *ctx, SortBufs &s, uint32_t count, const rx::PassPlan &plan, bool locally_ordered)
{
    if (count == 0 || plan.npass == 0) return DQ_OK;
    uint32_t *ghist = ctx->hist.as<uint32_t>();
    uint32_t *gbase = ghist + rx::kMaxPasses * rx::kRadix;
    uint32_t *use_match = gbase + rx::kMaxPasses * rx::kRadix;
    auto scan = rx::scan_hist_kernel;
    // every pass of a doubling round ranks with MATCH; other sorts decide each pass from its histogram
    const uint32_t force_mask = locally_ordered ? (1u << plan.npass) - 1u : 0u;
    DQ_LAUNCH(scan, plan.npass, rx::kRadix, 0, ctx->stream, ghist, gbase, use_match, count, force_mask);
    ctx->stats.kernel_launches++;

    const uint32_t tiles = (uint32_t)div_up(count, rx::kTile);
    const bool wide = count >= (1u << 30);
    const size_t desc_bytes = wide ? 8 : 4;
    const size_t per_pass = (size_t)tiles * rx::kRadix * desc_bytes;
    const size_t ticket_bytes = 256;  // [kMaxPasses] tickets, padded
    const bool one_memset = per_pass * plan.npass <= ((size_t)256 << 20);
    const size_t lb_bytes = ticket_bytes + (one_memset ? per_pass * plan.npass : per_pass);
    DQ_TRY(ensure(ctx, ctx->lb, lb_bytes));
    uint8_t *lbp = ctx->lb.as<uint8_t>();
    uint32_t *tickets = reinterpret_cast<uint32_t *>(lbp);
    if (one_memset) DQ_CK(ctx, cudaMemsetAsync(lbp, 0, lb_bytes, ctx->stream));

    for (int p = 0; p < plan.npass; ++p) {
        uint8_t *region = lbp + ticket_bytes + (one_memset ? per_pass * p : 0);
        if (!one_memset) {
            DQ_CK(ctx, cudaMemsetAsync(region, 0, per_pass, ctx->stream));
            if (p == 0) DQ_CK(ctx, cudaMemsetAsync(lbp, 0, ticket_bytes, ctx->stream));
        }
        const uint32_t mask = (1u << plan.bits[p]) - 1u;
        EventPair *ep = nullptr;
        if (ctx->timing) {
            if (ctx->pass_events_used == ctx->pass_events.size()) {
                EventPair e{};
                DQ_CK(ctx, cudaEventCreate(&e.a));
                DQ_CK(ctx, cudaEventCreate(&e.b));
                ctx->pass_events.push_back(e);
            }
            ep = &ctx->pass_events[ctx->pass_events_used++];
            ep->pairs = count;
            ep->shift = plan.shift[p];
            DQ_CK(ctx, cudaEventRecord(ep->a, ctx->stream));
        }
        if (wide) {
            auto k = rx::onesweep_pass_kernel<uint64_t>;
            DQ_LAUNCH(k, tiles, rx::kThreads, rx::pass_smem_bytes(), ctx->stream, s.kin, s.vin, s.kout, s.vout,
                      count, plan.shift[p], mask, gbase + p * rx::kRadix, reinterpret_cast<uint64_t *>(region),
                      tickets + p, use_match + p);
        } else {
            auto k = rx::onesweep_pass_kernel<uint32_t>;
            DQ_LAUNCH(k, tiles, rx::kThreads, rx::pass_smem_bytes(), ctx->stream, s.kin, s.vin, s.kout, s.vout,
                      count, plan.shift[p], mask, gbase + p * rx::kRadix, reinterpret_cast<uint32_t *>(region),
                      tickets + p, use_match + p);
        }
        if (ep) DQ_CK(ctx, cudaEventRecord(ep->b, ctx->stream));
        ctx->stats.kernel_launches++;
        ctx->stats.radix_passes++;
        std::swap(s.kin, s.kout);
        std::swap(s.vin, s.vout);
    }
    DQ_CK(ctx, cudaGetLastError());
    return DQ_OK;
}

// timing on: the round that starts now (active suffixes entering it, radix passes it will run)
int mark_round(dq_ctx *ctx, uint64_t active, int passes)
{
    if (!ctx->timing) return DQ_OK;
    if (ctx->rounds_used == ctx->round_recs.size()) {
        RoundRec r{};
        DQ_CK(ctx, cudaEventCreate(&r.begin));
        ctx->round_recs.push_back(r);
    }
    RoundRec &r = ctx->round_recs[ctx->rounds_used++];
    r.active = active;
    r.passes = passes;
    r.ms = 0.f;
    DQ_CK(ctx, cudaEventRecord(r.begin, ctx->stream));
    return DQ_OK;
}

// timing on, after a sort has synchronised (its last event is ctx->ev1): per-launch pass times, their sum, and per-round times
int read_timing(dq_ctx *ctx)
{
    if (!ctx->timing) return DQ_OK;
    dq_stats &st = ctx->stats;
    float tot = 0.f;
    uint64_t pairs = 0;
    for (size_t i = 0; i < ctx->pass_events_used; ++i) {
        float ms = 0.f;
        DQ_CK(ctx, cudaEventElapsedTime(&ms, ctx->pass_events[i].a, ctx->pass_events[i].b));
        ctx->pass_events[i].ms = ms;
        tot += ms;
        pairs += ctx->pass_events[i].pairs;
    }
    st.pass_ms = tot;
    st.pass_pairs = (int64_t)pairs;
    for (size_t i = 0; i < ctx->rounds_used; ++i)
        DQ_CK(ctx, cudaEventElapsedTime(&ctx->round_recs[i].ms, ctx->round_recs[i].begin,
                                        i + 1 < ctx->rounds_used ? ctx->round_recs[i + 1].begin : ctx->ev1));
    return DQ_OK;
}

int zero_hist(dq_ctx *ctx)
{
    DQ_TRY(ensure(ctx, ctx->hist, (size_t)2 * rx::kMaxPasses * rx::kRadix * 4 + 256));
    DQ_CK(ctx, cudaMemsetAsync(ctx->hist.p, 0, (size_t)rx::kMaxPasses * rx::kRadix * 4, ctx->stream));
    return DQ_OK;
}

// Small alphabets (dq_suffix.cuh): the order-preserving code for a text with the byte histogram `hist`, or bits == 8
// when more than 16 byte values occur.  compact_min: shortest text that is recoded (DQ_COMPACT_MIN; the histogram costs
// a host round trip, which only long texts amortise).
uint32_t compact_min()
{
    const char *e = getenv("DQ_COMPACT_MIN");  // read per call: tests lower it
    return e ? (uint32_t)strtoul(e, nullptr, 10) : (4u << 20);
}

sx::AlphabetCode choose_code(const uint64_t hist[256])
{
    sx::AlphabetCode ac{};
    int sigma = 0;
    for (int b = 0; b < 256; ++b) {
        ac.code[b] = (uint8_t)(sigma & 255);
        if (hist[b]) ++sigma;
    }
    ac.bits = sigma <= 2 ? 1 : sigma <= 4 ? 2 : sigma <= 16 ? 4 : 8;
    return ac;
}

// recodes ctx-resident text T (n bytes) into P; returns the code (bits == 8: nothing done)
int encode_text(dq_ctx *ctx, const uint8_t *T, uint32_t n, const sx::AlphabetCode &ac, DevBuf &P)
{
    const uint64_t out_bytes = (((uint64_t)n * ac.bits + 7) >> 3) + 64;  // zero tail: windows and aligned reads past the end
    DQ_TRY(ensure(ctx, P, out_bytes + 16));
    auto k = sx::encode_text_kernel;
    const uint32_t g = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(div_up(out_bytes, 256), (uint64_t)ctx->sm_count * 16));
    DQ_LAUNCH(k, g, 256, 0, ctx->stream, T, n, ac, P.as<uint8_t>(), out_bytes + 16);
    ctx->stats.kernel_launches++;
    DQ_CK(ctx, cudaGetLastError());
    return DQ_OK;
}

// byte histogram of T (n bytes) into hist[256] on the host (one stream synchronisation)
int byte_histogram(dq_ctx *ctx, const uint8_t *T, uint32_t n, uint64_t hist[256])
{
    DQ_TRY(ensure(ctx, ctx->hist, (size_t)2 * rx::kMaxPasses * rx::kRadix * 4 + 256));
    uint32_t *d = ctx->hist.as<uint32_t>();
    DQ_CK(ctx, cudaMemsetAsync(d, 0, 256 * 4, ctx->stream));
    auto k = sx::byte_hist_kernel;
    const uint32_t g = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(div_up(n, 256 * 16), (uint64_t)ctx->sm_count * 8));
    DQ_LAUNCH(k, g, 256, 0, ctx->stream, T, n, d);
    ctx->stats.kernel_launches++;
    uint32_t h32[256];
    DQ_CK(ctx, cudaMemcpyAsync(h32, d, sizeof h32, cudaMemcpyDeviceToHost, ctx->stream));
    DQ_CK(ctx, cudaStreamSynchronize(ctx->stream));
    for (int b = 0; b < 256; ++b) hist[b] = h32[b];
    return DQ_OK;
}

uint32_t producer_grid(const dq_ctx *ctx, uint64_t items)
{
    uint64_t blocks = div_up(items, (uint64_t)sx::kPackThreads * sx::kPackItems);
    return (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(blocks, (uint64_t)ctx->sm_count * 8));
}

// rank_compact over the sorted active set.  enqueue_rank launches it and the copy of its counters; finish_rank waits
// and reads them (the group paths enqueue on every shard before they wait on any).
template <bool ROUND0, bool DIST = false>
int enqueue_rank(dq_ctx *ctx, const uint64_t *keys, const uint32_t *sa, const uint32_t *slot_in, uint32_t a,
                 uint32_t n, uint32_t *sa_out, uint32_t *rank_out, uint32_t *slot_out, int32_t *sa_array = nullptr,
                 uint32_t slot_base = 0, uint64_t *upd = nullptr, uint64_t *act_out = nullptr,
                 const uint32_t *depth_in = nullptr, uint32_t *depth_out = nullptr, uint32_t hmin = 0,
                 const sx::PeerIsa &peer_isa = sx::PeerIsa{}, uint64_t *late = nullptr, uint32_t *late_count = nullptr)
{
    const uint32_t tiles = (uint32_t)div_up(a, sx::kRankTile);
    const size_t bytes = 256 + (size_t)tiles * 8;
    DQ_TRY(ensure(ctx, ctx->lb, bytes));
    uint8_t *lbp = ctx->lb.as<uint8_t>();
    DQ_CK(ctx, cudaMemsetAsync(lbp, 0, bytes, ctx->stream));
    uint32_t *ticket = reinterpret_cast<uint32_t *>(lbp);
    uint32_t *count = ticket + 1;
    uint64_t *desc = reinterpret_cast<uint64_t *>(lbp + 256);
    auto k = sx::rank_compact_kernel<ROUND0, DIST>;
    DQ_LAUNCH(k, tiles, sx::kRankThreads, 0, ctx->stream, keys, sa, slot_in, a, n, ctx->isa.as<uint32_t>(),
              sa_array ? sa_array : ctx->sa.as<int32_t>(), sa_out, rank_out, slot_out, desc, ticket, count, slot_base,
              upd, act_out, depth_in, depth_out, hmin, depth_out ? count + 1 : nullptr, peer_isa, late, late_count);
    ctx->stats.kernel_launches++;
    DQ_CK(ctx, cudaGetLastError());
    DQ_CK(ctx, cudaMemcpyAsync(ctx->h_count, count, 8, cudaMemcpyDeviceToHost, ctx->stream));
    return DQ_OK;
}

int finish_rank(dq_ctx *ctx, uint32_t *next_a, uint32_t *min_depth)
{
    DQ_CK(ctx, cudaSetDevice(ctx->device));
    DQ_CK(ctx, cudaStreamSynchronize(ctx->stream));
    *next_a = ctx->h_count[0];
    if (min_depth) *min_depth = ~ctx->h_count[1];  // the kernel keeps max(~depth) in a word that starts at 0
    return DQ_OK;
}

template <bool ROUND0>
int run_rank(dq_ctx *ctx, const uint64_t *keys, const uint32_t *sa, const uint32_t *slot_in, uint32_t a,
             uint32_t n, uint32_t *sa_out, uint32_t *rank_out, uint32_t *slot_out, uint32_t *next_a,
             const uint32_t *depth_in = nullptr, uint32_t *depth_out = nullptr, uint32_t hmin = 0,
             uint32_t *min_depth = nullptr, uint64_t *late = nullptr, uint32_t *late_count = nullptr)
{
    DQ_TRY((enqueue_rank<ROUND0, false>(ctx, keys, sa, slot_in, a, n, sa_out, rank_out, slot_out, nullptr, 0, nullptr,
                                        nullptr, depth_in, depth_out, hmin, sx::PeerIsa{}, late, late_count)));
    return finish_rank(ctx, next_a, min_depth);
}

// Early copy of the suffix array (sort_resident / group_sort): once few suffixes are unresolved, the array as it stands
// starts towards the host on the copy stream while the remaining rounds run; those rounds list the slots they
// resolve, and the list is patched into the host array when the copy has landed.  Needs a host array the device can
// write (pinned memory: dq_cuda_host_alloc, or anything cudaHostRegister'ed as mapped).
struct EarlyCopy {
    int32_t *host_sa = nullptr;  // device-visible address of the caller's array, or null: not available
    bool started = false;
    uint64_t *late = nullptr;
    uint32_t *late_count = nullptr;
};

int32_t *device_visible_host(const void *p)
{
    if (!p) return nullptr;
    cudaPointerAttributes at{};
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
        (void)cudaGetLastError();
        return nullptr;
    }
    return at.type == cudaMemoryTypeHost ? static_cast<int32_t *>(at.devicePointer) : nullptr;
}

// `a` suffixes of `total` are still unresolved: start the copy of src[0..count) -> dst if it has not started and the
// rest is small.  The late list can take `a` entries.
int early_copy_maybe_start(dq_ctx *ctx, EarlyCopy &ec, const int32_t *src, int32_t *dst, uint32_t count, uint32_t a,
                           uint32_t total)
{
    const char *e = getenv("DQ_EARLY_COPY_MIN");  // tests lower it; 0 = never
    const uint32_t min_total = e ? (uint32_t)strtoul(e, nullptr, 10) : (1u << 20);
    if (ec.started || !ec.host_sa || a == 0 || (uint64_t)a * 8 > total || total < min_total || min_total == 0) return DQ_OK;
    DQ_TRY(ensure(ctx, ctx->late, (size_t)a * 8 + 256));
    ec.late_count = ctx->late.as<uint32_t>();
    ec.late = reinterpret_cast<uint64_t *>(ctx->late.as<uint8_t>() + 256);
    DQ_CK(ctx, cudaMemsetAsync(ec.late_count, 0, 4, ctx->stream));
    DQ_CK(ctx, cudaEventRecord(ctx->ev_copy, ctx->stream));
    DQ_CK(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_copy, 0));
    if (count) DQ_CK(ctx, cudaMemcpyAsync(dst, src, (size_t)count * 4, cudaMemcpyDeviceToHost, ctx->copy_stream));
    ec.started = true;
    return DQ_OK;
}

// after the last round: wait for the copy, then patch the late slots into the host array
int early_copy_finish(dq_ctx *ctx, EarlyCopy &ec)
{
    if (!ec.started) return DQ_OK;
    DQ_CK(ctx, cudaEventRecord(ctx->ev_copy, ctx->copy_stream));
    DQ_CK(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_copy, 0));
    auto k = sx::patch_host_sa_kernel;
    DQ_LAUNCH(k, (uint32_t)ctx->sm_count * 4, 256, 0, ctx->stream, ec.late, ec.late_count, ec.host_sa);
    ctx->stats.kernel_launches++;
    DQ_CK(ctx, cudaGetLastError());
    return DQ_OK;
}

// ctx->text holds n bytes followed by >= 16 zero bytes.  Produces ctx->sa (the suffix array) and ctx->isa.
// 3-byte prefix table of the text being sorted, from the round-0 keys while they are in sorted order (dq_search.cuh)
int build_prefix3_sorted(dq_ctx *ctx, const uint64_t *sorted_keys, uint32_t n)
{
    namespace sr = dq::search;
    DQ_TRY(ensure(ctx, ctx->pre3, ((size_t)sr::kPrefix3Bins + 4) * 4));
    DQ_TRY(ensure(ctx, ctx->pre3tile, (size_t)sr::kPrefix3Tiles * 4));
    uint32_t *table = ctx->pre3.as<uint32_t>(), *tiles = ctx->pre3tile.as<uint32_t>();
    DQ_CK(ctx, cudaMemsetAsync(table, 0xff, (size_t)sr::kPrefix3Bins * 4, ctx->stream));
    const uint32_t g = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(div_up(n, 256), (uint64_t)ctx->sm_count * 16));
    auto k1 = sr::prefix3_mark_kernel;
    DQ_LAUNCH(k1, g, 256, 0, ctx->stream, sorted_keys, n, table);
    auto k2 = sr::prefix3_fill_tile_min_kernel;
    DQ_LAUNCH(k2, sr::kPrefix3Tiles, 256, 0, ctx->stream, table, tiles);
    auto k3 = sr::prefix3_fill_tile_scan_kernel;
    DQ_LAUNCH(k3, 1, 1024, 0, ctx->stream, tiles, ctx->text.as<uint8_t>(), n, table);
    auto k4 = sr::prefix3_fill_apply_kernel;
    DQ_LAUNCH(k4, sr::kPrefix3Tiles, 256, 0, ctx->stream, table, tiles);
    ctx->stats.kernel_launches += 4;
    ctx->res.pre3 = true;
    return DQ_OK;
}

// host_sa_out: when not null, the caller's host array (it must be device-visible, see EarlyCopy) receives the suffix
// array here -- overlapped with the last rounds when they are small -- and *delivered says so
// mid: when not null, called once round 0's kernels are enqueued and before the host first waits for them (not on
// the paths that return before that: n == 0, the one-CTA sort) -- work of the caller's that should sit behind round 0 in
// the queues, or that blocks the host while the GPU is busy with round 0 (dq_cuda_bsdiff_streams: the upload of `new`)
int sort_resident(dq_ctx *ctx, uint32_t n, int32_t *host_sa_out = nullptr, bool *delivered = nullptr,
                  const std::function<int()> *mid = nullptr)
{
    if (delivered) *delivered = false;
    EarlyCopy ec{};
    ec.host_sa = device_visible_host(host_sa_out);
    dq_stats &st = ctx->stats;
    st = dq_stats{};
    st.n = (int32_t)n;
    ctx->pass_events_used = 0;
    ctx->rounds_used = 0;
    if (n == 0) return DQ_OK;

    if (n <= (uint32_t)sx::kSmallN) {
        // one CTA, one launch (dq_suffix.cuh, "small inputs")
        DQ_TRY(ensure(ctx, ctx->isa, (size_t)n * 4));
        DQ_TRY(ensure(ctx, ctx->sa, (size_t)n * 4));
        DQ_CK(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
        auto k = sx::small_sort_kernel;
        DQ_LAUNCH(k, 1, sx::kSmallThreads, sx::small_sort_smem_bytes(), ctx->stream, ctx->text.as<uint8_t>(), n,
                  ctx->sa.as<int32_t>(), ctx->isa.as<uint32_t>());
        DQ_CK(ctx, cudaGetLastError());
        DQ_CK(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
        DQ_CK(ctx, cudaStreamSynchronize(ctx->stream));
        DQ_CK(ctx, cudaEventElapsedTime(&st.device_ms, ctx->ev0, ctx->ev1));
        st.rounds = 1;
        st.kernel_launches = 1;
        st.active_sum = n;
        st.algorithmic_bytes = (int64_t)n * 5;
        return DQ_OK;
    }
    const size_t n8 = (size_t)n * 8, n4 = (size_t)n * 4;
    DQ_TRY(ensure(ctx, ctx->keyA, n8));
    DQ_TRY(ensure(ctx, ctx->keyB, n8));
    DQ_TRY(ensure(ctx, ctx->valA, n4));
    DQ_TRY(ensure(ctx, ctx->valB, n4));
    DQ_TRY(ensure(ctx, ctx->isa, n4));
    DQ_TRY(ensure(ctx, ctx->sa, n4));
    DQ_TRY(ensure(ctx, ctx->slotA, n4));
    DQ_TRY(ensure(ctx, ctx->slotB, n4));

    DQ_CK(ctx, cudaEventRecord(ctx->ev0, ctx->stream));

    // ---- round 0: all suffixes by their first 8 bytes -- or, for a long text over at most 16 byte values, by their
    // first 16 / 32 / 64 characters (dq_suffix.cuh, "small alphabets")
    rx::PassPlan plan{};
    rx::plan_add_field(plan, 0, 64);
    DQ_TRY(mark_round(ctx, n, plan.npass));
    sx::AlphabetCode ac{};
    ac.bits = 8;
    if (n >= compact_min()) {
        uint64_t bh[256];
        DQ_TRY(byte_histogram(ctx, ctx->text.as<uint8_t>(), n, bh));
        ac = choose_code(bh);
        if (ac.bits < 8) DQ_TRY(encode_text(ctx, ctx->text.as<uint8_t>(), n, ac, ctx->packed));
    }
    const uint32_t key_chars = 64u / (uint32_t)ac.bits;
    DQ_TRY(zero_hist(ctx));
    // counter of suffixes inside equal-byte runs, kept behind the histogram tables
    uint32_t *uniform_count = ctx->hist.as<uint32_t>() + 2 * rx::kMaxPasses * rx::kRadix + 32;
    DQ_CK(ctx, cudaMemsetAsync(uniform_count, 0, 4, ctx->stream));
    {
        auto k = sx::pack_keys_kernel;
        DQ_LAUNCH(k, producer_grid(ctx, n), sx::kPackThreads, plan.npass * rx::kRadix * 4, ctx->stream,
                  ctx->text.as<uint8_t>(), n, ctx->keyA.as<uint64_t>(), ctx->valA.as<uint32_t>(), plan,
                  ctx->hist.as<uint32_t>(), uniform_count, ac.bits < 8 ? ctx->packed.as<uint8_t>() : (const uint8_t *)nullptr,
                  ac.bits);
        st.kernel_launches++;
    }
    DQ_CK(ctx, cudaMemcpyAsync(ctx->h_count + 4, uniform_count, 4, cudaMemcpyDeviceToHost, ctx->stream));
    SortBufs s{ctx->keyA.as<uint64_t>(), ctx->keyB.as<uint64_t>(), ctx->valA.as<uint32_t>(), ctx->valB.as<uint32_t>()};
    DQ_TRY(run_passes(ctx, s, n, plan, false));
    // a context that searches gets its 3-byte prefix table here, from the keys while they are in sorted order
    {
        const char *min_env = getenv("DQ_PREFIX3_SORTED_MIN");  // tests: lets small inputs take this path
        const uint32_t min_n = min_env ? (uint32_t)atoi(min_env) : (1u << 20);
        if (ctx->search_seen && n >= min_n && ac.bits == 8 && !getenv("DQ_PREFIX3")) DQ_TRY(build_prefix3_sorted(ctx, s.kin, n));
    }
    st.rounds = 1;
    st.active_sum = n;
    st.algorithmic_bytes = (int64_t)n * (41 + 24 * plan.npass);

    if (mid) DQ_TRY((*mid)());

    uint32_t *slot_cur = ctx->slotA.as<uint32_t>(), *slot_nxt = ctx->slotB.as<uint32_t>();
    uint32_t a = 0;
    // sorted pairs are in (s.kin, s.vin); (s.kout, s.vout) are free
    DQ_TRY(run_rank<true>(ctx, s.kin, s.vin, nullptr, n, n, s.vout, reinterpret_cast<uint32_t *>(s.kout), slot_cur, &a,
                          nullptr, nullptr, key_chars));

    // ---- doubling rounds over the unresolved suffixes.  Every group carries its own depth (bytes its members
    // share); h is the depth every rank in ISA is consistent to.  Round 1 refines equal-byte-run groups by run
    // length in one step (dq_suffix.cuh), so zero padding does not cost log2(run length) rounds.
    const int bits_r2 = bit_length(n);                      // ISA[.]+1 in [0, n]
    const int bits_rank = bit_length(n > 1 ? n - 1 : 1);    // rank in [0, n-1]
    uint64_t h = key_chars;
    uint32_t *depth_cur = nullptr, *depth_nxt = nullptr;
    // Run-length refinement pays when a visible share of the text sits in equal-byte runs (zero padding); without
    // such runs plain doubling (uniform depth, no depth arrays) is the shorter path.
    const bool run_aware = a > 0 && ac.bits == 8 && (uint64_t)ctx->h_count[4] * 64 >= n;
    if (run_aware) {
        DQ_TRY(ensure(ctx, ctx->depthA, n4));
        DQ_TRY(ensure(ctx, ctx->depthB, n4));
        DQ_TRY(ensure(ctx, ctx->runend, n4));
        const uint32_t ntiles = (uint32_t)div_up(n, sx::kRunTile);
        DQ_TRY(ensure(ctx, ctx->runtile, (size_t)ntiles * 8));
        uint32_t *tile_first = ctx->runtile.as<uint32_t>(), *next_after = tile_first + ntiles;
        auto k1 = sx::run_tile_first_kernel;
        DQ_LAUNCH(k1, ntiles, 256, 0, ctx->stream, ctx->text.as<uint8_t>(), n, tile_first);
        auto k2 = sx::run_tile_scan_kernel;
        DQ_LAUNCH(k2, 1, 1024, 0, ctx->stream, tile_first, ntiles, n, next_after);
        auto k3 = sx::run_end_kernel;
        DQ_LAUNCH(k3, ntiles, 256, 0, ctx->stream, ctx->text.as<uint8_t>(), n, next_after, ctx->runend.as<uint32_t>());
        st.kernel_launches += 3;
        ctx->res.runs = true;
        depth_cur = ctx->depthA.as<uint32_t>();
        depth_nxt = ctx->depthB.as<uint32_t>();
    }
    bool first = true;
    while (a > 0) {
        DQ_TRY(early_copy_maybe_start(ctx, ec, ctx->sa.as<int32_t>(), host_sa_out, n, a, n));
        // active set: sa = s.vout, rank = (uint32*)s.kout, slot = slot_cur, depth = depth_cur.  Keys go to s.kin.
        rx::PassPlan rp{};
        rx::plan_add_field(rp, 0, (first && run_aware) ? 32 : bits_r2);
        rx::plan_add_field(rp, 32, bits_rank);
        DQ_TRY(mark_round(ctx, a, rp.npass));
        DQ_TRY(zero_hist(ctx));
        if (first && run_aware) {
            auto k = sx::build_keys_round1_kernel;
            DQ_LAUNCH(k, producer_grid(ctx, a), sx::kPackThreads, rp.npass * rx::kRadix * 4, ctx->stream, s.vout,
                      reinterpret_cast<uint32_t *>(s.kout), ctx->isa.as<uint32_t>(), ctx->text.as<uint8_t>(),
                      ctx->runend.as<uint32_t>(), n, a, s.kin, depth_cur, rp, ctx->hist.as<uint32_t>());
        } else {
            auto k = sx::build_keys_kernel;
            DQ_LAUNCH(k, producer_grid(ctx, a), sx::kPackThreads, rp.npass * rx::kRadix * 4, ctx->stream, s.vout,
                      reinterpret_cast<uint32_t *>(s.kout), ctx->isa.as<uint32_t>(), n, a, h, depth_cur, s.kin, rp,
                      ctx->hist.as<uint32_t>());
        }
        st.kernel_launches++;
        // sort (s.kin, s.vout) using (s.kout, s.vin) as the alternate
        std::swap(s.vin, s.vout);
        DQ_TRY(run_passes(ctx, s, a, rp, true));
        st.rounds++;
        st.active_sum += a;
        st.algorithmic_bytes += (int64_t)a * (52 + 24 * rp.npass);

        uint32_t next_a = 0, min_depth = 0;
        DQ_TRY(run_rank<false>(ctx, s.kin, s.vin, slot_cur, a, n, s.vout, reinterpret_cast<uint32_t *>(s.kout), slot_nxt,
                               &next_a, depth_cur, depth_nxt, (uint32_t)h, &min_depth, ec.late, ec.late_count));
        std::swap(slot_cur, slot_nxt);
        std::swap(depth_cur, depth_nxt);
        if (next_a > a) {
            ctx->err = "internal: active set grew";
            return DQ_ERR_INTERNAL;
        }
        a = next_a;
        first = false;
        // every rank is now consistent to the smallest depth of an unresolved group (2h for plain doubling; a run
        // refined group may share fewer bytes than that)
        if (!run_aware) {
            h *= 2;
            if (h > ((uint64_t)1 << 31)) h = (uint64_t)1 << 31;
        } else if (a > 0) {
            if (min_depth <= h && st.rounds > 2) {
                ctx->err = "internal: group depth did not grow";
                return DQ_ERR_INTERNAL;
            }
            h = min_depth;
        }
        if (st.rounds > 200) {
            ctx->err = "internal: doubling did not converge";
            return DQ_ERR_INTERNAL;
        }
    }
    st.algorithmic_bytes += (int64_t)n * 4;
    DQ_CK(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    if (ec.started) {
        DQ_TRY(early_copy_finish(ctx, ec));
        if (delivered) *delivered = true;
    }
    DQ_CK(ctx, cudaStreamSynchronize(ctx->stream));
    DQ_CK(ctx, cudaEventElapsedTime(&st.device_ms, ctx->ev0, ctx->ev1));
    return read_timing(ctx);
}

int upload_text(dq_ctx *ctx, DevBuf &buf, const uint8_t *src, uint32_t n, cudaMemcpyKind kind)
{
    DQ_TRY(ensure(ctx, buf, (size_t)n + 64));
    if (n) DQ_CK(ctx, cudaMemcpyAsync(buf.p, src, n, kind, ctx->stream));
    DQ_CK(ctx, cudaMemsetAsync(buf.as<uint8_t>() + n, 0, 64, ctx->stream));
    return DQ_OK;
}

int check_args(dq_ctx *ctx, bool ok, const char *what)
{
    if (!ok) {
        ctx->err = what;
        return DQ_ERR_INVALID_ARGUMENT;
    }
    return DQ_OK;
}

// A call that writes text, sa or isa forgets the Resident record (on a group context the group's too: dq_group.inl)
// before its first write, and holds its text once all three are complete.
void forget_resident(dq_ctx *ctx);

// runs, lcp and pre3 stay as they are: a sort sets runs and pre3 on the way, and the search that follows needs them
void hold_resident(dq_ctx *ctx, int32_t n, int32_t rounds) { ctx->res.n = n; ctx->res.rounds = rounds; }

// a call with I == NULL: the resident text must have n bytes
int require_resident(dq_ctx *ctx, int32_t n, const char *what)
{
    if (ctx->res.n == n) return DQ_OK;
    ctx->err = std::string(what) + ": I is NULL but no suffix array of this length is resident on the device";
    return DQ_ERR_INVALID_ARGUMENT;
}

#include "dq_search_host.inl"

int dist_reserve(dq_ctx *ctx, uint32_t count)
{
    const size_t c8 = (size_t)std::max<uint32_t>(count, 1) * 8, c4 = (size_t)std::max<uint32_t>(count, 1) * 4;
    DQ_TRY(ensure(ctx, ctx->keyA, c8));
    DQ_TRY(ensure(ctx, ctx->keyB, c8));
    DQ_TRY(ensure(ctx, ctx->valA, c4));
    DQ_TRY(ensure(ctx, ctx->valB, c4));
    DQ_TRY(ensure(ctx, ctx->slotA, c4));
    DQ_TRY(ensure(ctx, ctx->slotB, c4));
    return DQ_OK;
}

int create_single(dq_ctx **out, int dev);
int destroy_single(dq_ctx *ctx);

#include "dq_group.inl"

void forget_resident(dq_ctx *ctx)
{
    ctx->res = Resident{};
    if (ctx->group) ctx->group->res = GroupResident{};
}

// body of dq_cuda_lcp (the caller holds ctx->mu): with I == NULL on a group that holds the text, the group's index
int lcp_host(dq_ctx *ctx, const uint8_t *text, int32_t n, const int32_t *I_or_null, int32_t *lcp_out)
{
    if (!I_or_null && lcp_out && group_holds(ctx, n)) return group_lcp(ctx, n, lcp_out);
    return lcp_common(ctx, text, n, I_or_null, lcp_out, false);
}

// body of dq_cuda_suffix_sort (the caller holds ctx->mu and has selected the device): one text of host memory, sorted
// by the group when it is large enough, else on this context's device; sa_out receives n entries (none when it is null)
int suffix_sort_host(dq_ctx *ctx, const uint8_t *text, uint32_t n, int32_t *sa_out)
{
    forget_resident(ctx);
    if (ctx->group && n >= ctx->group->shard_min) return group_sort(ctx, text, n, sa_out);
    DQ_TRY(upload_text(ctx, ctx->text, text, n, cudaMemcpyHostToDevice));
    bool delivered = false;
    DQ_TRY(sort_resident(ctx, n, sa_out, &delivered));
    if (n && !delivered && sa_out) DQ_CK(ctx, cudaMemcpyAsync(sa_out, ctx->sa.p, (size_t)n * 4, cudaMemcpyDeviceToHost, ctx->stream));
    DQ_CK(ctx, cudaStreamSynchronize(ctx->stream));
    hold_resident(ctx, (int32_t)n, ctx->stats.rounds);
    return DQ_OK;
}

// ---- batches (dq_cuda_suffix_sort_batch) ------------------------------------------------------------------------------
// Texts of at least batch_single_min() bytes are sorted one by one, as dq_cuda_suffix_sort sorts them; the others are
// packed into chunks of at most batch_chunk_bytes() bytes and kBatchMaxTexts texts, and every chunk is sorted by one
// prefix doubling over all its texts (dq_suffix.cuh, "batches").  Neither threshold changes a result.
constexpr uint32_t kBatchMaxTexts = 1u << (64 - sx::kBatchTextShift);

// From 2 MiB up a text with zero runs sorts faster alone, where round 1 refines its runs by length, than in a chunk's
// plain doubling (exe-like texts: 1.22x from the chunks at 1 MiB, 0.85x at 2 MiB); random texts gain from the chunks
// at every size (profiles/r03_batch_sort.md, W4)
uint32_t batch_single_min()
{
    const char *e = getenv("DQ_BATCH_SINGLE_MIN");  // read per call: tests lower it
    return e ? (uint32_t)strtoul(e, nullptr, 10) : (2u << 20);
}

uint64_t batch_chunk_bytes()
{
    const char *e = getenv("DQ_BATCH_CHUNK");
    return e ? (uint64_t)strtoull(e, nullptr, 10) : ((uint64_t)256 << 20);
}

// adds the figures of one sort to those of the whole batch call
void batch_add_stats(dq_stats &acc, const dq_stats &st)
{
    acc.rounds = std::max(acc.rounds, st.rounds);
    acc.radix_passes += st.radix_passes;
    acc.kernel_launches += st.kernel_launches;
    acc.active_sum += st.active_sum;
    acc.algorithmic_bytes += st.algorithmic_bytes;
    acc.device_ms += st.device_ms;
    acc.pass_ms += st.pass_ms;
    acc.pass_pairs += st.pass_pairs;
}

// LCP arrays of a sorted chunk of n compact positions (ctx->sa: per-text indices, text-major) into ctx->lcp in rank
// order: PHI from rank order, PLCP along the chunk's text with every comparison stopped at the end of its own text
// (sr::ChunkTexts), gathered back to rank order.  Only level 0: the block minima and tables are search index.
int lcp_batch_chunk(dq_ctx *ctx, const uint32_t *d_offs, uint32_t count, uint32_t n, int32_t rounds)
{
    const uint64_t chunks = div_up(n, sr::kChunk), supers = div_up(n, sr::kSuper);
    DQ_TRY(ensure(ctx, ctx->phi, ((size_t)n + 64) * 4));
    DQ_TRY(ensure(ctx, ctx->plcp, ((size_t)n + 64) * 4));
    DQ_TRY(ensure(ctx, ctx->headl, ((size_t)chunks + 1) * 4));
    DQ_TRY(ensure(ctx, ctx->seedl, ((size_t)supers + 1) * 4));
    DQ_TRY(ensure(ctx, ctx->lcp, (size_t)n * 4));
    const int32_t *SA = ctx->sa.as<int32_t>();
    uint32_t *PHI = ctx->phi.as<uint32_t>(), *PLCP = ctx->plcp.as<uint32_t>();
    const sr::ChunkTexts tx{n, d_offs, count};
    const uint32_t g = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(div_up(n, 256 * 4), (uint64_t)ctx->sm_count * 16));
    {
        auto k = sr::batch_phi_kernel;
        DQ_LAUNCH(k, g, 256, 0, ctx->stream, SA, d_offs, count, PHI, n);
        ctx->stats.kernel_launches++;
    }
    DQ_TRY(plcp_walks(ctx, ctx->text.as<uint8_t>(), tx, PHI, PLCP, nullptr,
                      seeds_per_warp(rounds, n, (uint32_t)supers), 0, supers, 0, chunks));
    {
        auto k = sr::lcp_gather_kernel<sr::ChunkTexts>;
        DQ_LAUNCH(k, g, 256, 0, ctx->stream, SA, PLCP, ctx->lcp.as<uint32_t>(), tx);
        ctx->stats.kernel_launches++;
    }
    // PHI: SA twice + PHI; the walks: PHI + PLCP (the text bytes they compare depend on the texts); gather: SA, PLCP, LCP
    ctx->stats.algorithmic_bytes += (int64_t)n * 32;
    DQ_CK(ctx, cudaGetLastError());
    return DQ_OK;
}

// Sorts texts [t0, t1) of a batch, which lie back to back at `texts` + offsets[t0] (host memory), and leaves the chunk on
// the device: ctx->text (zero padded), ctx->boffs (its text offsets), ctx->sa (local suffix arrays, text-major) and,
// with lcp, ctx->lcp (their LCP arrays).  ev0 / ev1 bracket the device work; nothing is waited for.
// Plain doubling at uniform depth (sort_resident with run_aware off); the run-length refinement, the small-alphabet
// recoding, the early copy and the 3-byte prefix table assume one text.
int sort_batch_chunk_device(dq_ctx *ctx, const uint8_t *texts, const int32_t *offsets, int32_t t0, int32_t t1, bool lcp)
{
    const uint32_t base = (uint32_t)offsets[t0];
    const uint32_t n = (uint32_t)offsets[t1] - base;   // compact positions
    const uint32_t count = (uint32_t)(t1 - t0);
    const uint64_t np = (uint64_t)n + count;           // padded positions: one sentinel after every text
    dq_stats &st = ctx->stats;
    st = dq_stats{};
    ctx->pass_events_used = 0;
    ctx->rounds_used = 0;
    if (n == 0) return DQ_OK;

    std::vector<uint32_t> offs(count + 1);
    for (uint32_t i = 0; i <= count; ++i) offs[i] = (uint32_t)offsets[t0 + i] - base;
    DQ_TRY(ensure(ctx, ctx->boffs, offs.size() * 4));
    DQ_TRY(upload_text(ctx, ctx->text, texts + base, n, cudaMemcpyHostToDevice));
    DQ_CK(ctx, cudaMemcpyAsync(ctx->boffs.p, offs.data(), offs.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    const uint32_t *d_offs = ctx->boffs.as<uint32_t>();

    const size_t n8 = (size_t)n * 8, n4 = (size_t)n * 4;
    DQ_TRY(ensure(ctx, ctx->keyA, n8));
    DQ_TRY(ensure(ctx, ctx->keyB, n8));
    DQ_TRY(ensure(ctx, ctx->valA, n4));
    DQ_TRY(ensure(ctx, ctx->valB, n4));
    DQ_TRY(ensure(ctx, ctx->isa, (size_t)np * 4));
    DQ_TRY(ensure(ctx, ctx->sa, n4));
    DQ_TRY(ensure(ctx, ctx->slotA, n4));
    DQ_TRY(ensure(ctx, ctx->slotB, n4));
    DQ_CK(ctx, cudaMemsetAsync(ctx->isa.p, 0xff, (size_t)np * 4, ctx->stream));  // the sentinels

    DQ_CK(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    // ---- round 0: (text, first 5 bytes, length code)
    rx::PassPlan plan{};
    rx::plan_add_field(plan, 0, sx::kBatchTextShift + bit_length(count - 1));
    DQ_TRY(mark_round(ctx, n, plan.npass));
    DQ_TRY(zero_hist(ctx));
    {
        auto k = sx::pack_keys_batch_kernel;
        DQ_LAUNCH(k, producer_grid(ctx, n), sx::kPackThreads, plan.npass * rx::kRadix * 4, ctx->stream,
                  ctx->text.as<uint8_t>(), d_offs, count, n, ctx->keyA.as<uint64_t>(), ctx->valA.as<uint32_t>(), plan,
                  ctx->hist.as<uint32_t>());
        st.kernel_launches++;
    }
    SortBufs s{ctx->keyA.as<uint64_t>(), ctx->keyB.as<uint64_t>(), ctx->valA.as<uint32_t>(), ctx->valB.as<uint32_t>()};
    DQ_TRY(run_passes(ctx, s, n, plan, false));
    st.rounds = 1;
    st.active_sum = n;
    st.algorithmic_bytes = (int64_t)n * (41 + 24 * plan.npass);
    uint32_t *slot_cur = ctx->slotA.as<uint32_t>(), *slot_nxt = ctx->slotB.as<uint32_t>();
    uint32_t a = 0;
    // hmin = 0: the key's length code has already set every suffix shorter than the key apart
    DQ_TRY(run_rank<true>(ctx, s.kin, s.vin, nullptr, n, n, s.vout, reinterpret_cast<uint32_t *>(s.kout), slot_cur, &a));

    // ---- doubling rounds at uniform depth h = 5, 10, 20, ...; positions, ISA indices and n are padded
    const int bits_r2 = bit_length(n);                    // ISA[.]+1 in [0, n]: ranks are compact SA slots
    const int bits_rank = bit_length(n > 1 ? n - 1 : 1);  // rank in [0, n-1]
    uint64_t h = sx::kBatchKeyBytes;
    while (a > 0) {
        rx::PassPlan rp{};
        rx::plan_add_field(rp, 0, bits_r2);
        rx::plan_add_field(rp, 32, bits_rank);
        DQ_TRY(mark_round(ctx, a, rp.npass));
        DQ_TRY(zero_hist(ctx));
        {
            auto k = sx::build_keys_kernel;
            DQ_LAUNCH(k, producer_grid(ctx, a), sx::kPackThreads, rp.npass * rx::kRadix * 4, ctx->stream, s.vout,
                      reinterpret_cast<uint32_t *>(s.kout), ctx->isa.as<uint32_t>(), (uint32_t)np, a, h,
                      (const uint32_t *)nullptr, s.kin, rp, ctx->hist.as<uint32_t>());
            st.kernel_launches++;
        }
        std::swap(s.vin, s.vout);
        DQ_TRY(run_passes(ctx, s, a, rp, true));
        st.rounds++;
        st.active_sum += a;
        st.algorithmic_bytes += (int64_t)a * (52 + 24 * rp.npass);
        uint32_t next_a = 0;
        DQ_TRY(run_rank<false>(ctx, s.kin, s.vin, slot_cur, a, (uint32_t)np, s.vout, reinterpret_cast<uint32_t *>(s.kout),
                               slot_nxt, &next_a, nullptr, nullptr, (uint32_t)h));
        std::swap(slot_cur, slot_nxt);
        if (next_a > a) {
            ctx->err = "internal: active set grew";
            return DQ_ERR_INTERNAL;
        }
        a = next_a;
        h = std::min<uint64_t>(h * 2, (uint64_t)1 << 31);
        if (st.rounds > 200) {
            ctx->err = "internal: doubling did not converge";
            return DQ_ERR_INTERNAL;
        }
    }
    {
        auto k = sx::batch_localize_kernel;
        const uint32_t g = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(div_up(n, 256), (uint64_t)ctx->sm_count * 16));
        DQ_LAUNCH(k, g, 256, 0, ctx->stream, ctx->sa.as<int32_t>(), d_offs, count, n);
        st.kernel_launches++;
        DQ_CK(ctx, cudaGetLastError());
    }
    st.algorithmic_bytes += (int64_t)n * 4;
    if (lcp) DQ_TRY(lcp_batch_chunk(ctx, d_offs, count, n, st.rounds));
    DQ_CK(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    return DQ_OK;
}

// sort_batch_chunk_device, then the local suffix arrays to sa_out + offsets[t0], and the LCP arrays to
// lcp_out + offsets[t0] unless lcp_out is null
int sort_batch_chunk(dq_ctx *ctx, const uint8_t *texts, const int32_t *offsets, int32_t t0, int32_t t1, int32_t *sa_out,
                     int32_t *lcp_out)
{
    DQ_TRY(sort_batch_chunk_device(ctx, texts, offsets, t0, t1, lcp_out != nullptr));
    const uint32_t base = (uint32_t)offsets[t0];
    const size_t n4 = (size_t)((uint32_t)offsets[t1] - base) * 4;
    if (n4 == 0) return DQ_OK;
    DQ_CK(ctx, cudaMemcpyAsync(sa_out + base, ctx->sa.p, n4, cudaMemcpyDeviceToHost, ctx->stream));
    if (lcp_out) DQ_CK(ctx, cudaMemcpyAsync(lcp_out + base, ctx->lcp.p, n4, cudaMemcpyDeviceToHost, ctx->stream));
    DQ_CK(ctx, cudaStreamSynchronize(ctx->stream));
    DQ_CK(ctx, cudaEventElapsedTime(&ctx->stats.device_ms, ctx->ev0, ctx->ev1));
    return read_timing(ctx);
}

// body of dq_cuda_suffix_sort_batch and dq_cuda_suffix_sort_lcp_batch (lcp_out != null); the arguments are checked
int suffix_sort_batch(dq_ctx *ctx, const uint8_t *texts, const int32_t *offsets, int32_t count, int32_t *sa_out,
                      int32_t *lcp_out)
{
    const uint32_t single_min = batch_single_min();
    const uint64_t chunk_max = batch_chunk_bytes();
    dq_stats acc{};
    int32_t begin = 0;  // first text of the chunk being gathered
    auto flush = [&](int32_t end) -> int {
        if (end == begin) return DQ_OK;
        DQ_TRY(sort_batch_chunk(ctx, texts, offsets, begin, end, sa_out, lcp_out));
        batch_add_stats(acc, ctx->stats);
        begin = end;
        return DQ_OK;
    };
    for (int32_t t = 0; t < count; ++t) {
        const uint32_t len = (uint32_t)(offsets[t + 1] - offsets[t]);
        if (len >= single_min && len > 0) {
            DQ_TRY(flush(t));
            DQ_TRY(suffix_sort_host(ctx, texts + offsets[t], len, sa_out + offsets[t]));
            // level 0 of the index of the text it left resident, as dq_cuda_lcp with I == NULL builds it
            if (lcp_out) DQ_TRY(lcp_host(ctx, texts + offsets[t], (int32_t)len, nullptr, lcp_out + offsets[t]));
            batch_add_stats(acc, ctx->stats);
            begin = t + 1;
            continue;
        }
        // a chunk holds at least one text
        if ((uint32_t)(t - begin) == kBatchMaxTexts || (t > begin && (uint64_t)(offsets[t + 1] - offsets[begin]) > chunk_max))
            DQ_TRY(flush(t));
    }
    DQ_TRY(flush(count));
    acc.n = count ? offsets[count] : 0;
    ctx->stats = acc;
    return DQ_OK;
}

// the two batch entry points: the same checks (with_lcp: lcp_out is one more output buffer), then the batch
int batch_entry(dq_ctx *ctx, const char *fn, const uint8_t *texts, const int32_t *offsets, int32_t count, int32_t *sa_out,
                int32_t *lcp_out, bool with_lcp)
{
    if (!ctx) return DQ_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    auto check = [&](bool ok, const char *what) { return check_args(ctx, ok, (std::string(fn) + ": " + what).c_str()); };
    DQ_TRY(check(count >= 0, "negative count"));
    DQ_TRY(check(offsets || count == 0, "offsets is null"));
    if (offsets) {
        DQ_TRY(check(offsets[0] == 0, "offsets[0] must be 0"));
        for (int32_t i = 0; i < count; ++i) DQ_TRY(check(offsets[i + 1] >= offsets[i], "offsets decrease"));
        DQ_TRY(check(offsets[count] == 0 || (texts && sa_out && (lcp_out || !with_lcp)), "null buffer"));
    }
    DQ_CK(ctx, cudaSetDevice(ctx->device));
    const int rc = suffix_sort_batch(ctx, texts, offsets, count, sa_out, with_lcp ? lcp_out : nullptr);
    // after the batch, not before: its chunks overwrite text / SA / ISA, and a text it sorts alone holds itself
    forget_resident(ctx);
    return rc;
}

// ---- batched match search (dq_cuda_bsdiff_search_batch) --------------------------------------------------------------
// Pairs [p0, p1) of a batch in one chunk: their olds are sorted together with their LCP arrays (sort_batch_chunk_device),
// the local ranks and every pair's block minima are built, and every pair is searched in its own coordinates
// (dq_search.cuh, "batches").  The (pos, len) table of pair i lands at pos_out / len_out + new_offsets[i].
int search_batch_chunk(dq_ctx *ctx, const uint8_t *olds, const int32_t *old_offsets, const uint8_t *news,
                       const int32_t *new_offsets, int32_t p0, int32_t p1, int32_t *pos_out, int32_t *len_out)
{
    const uint32_t count = (uint32_t)(p1 - p0);
    const uint32_t obase = (uint32_t)old_offsets[p0], n = (uint32_t)old_offsets[p1] - obase;
    const uint32_t nbase = (uint32_t)new_offsets[p0], m = (uint32_t)new_offsets[p1] - nbase;
    ctx->stats = dq_stats{};
    if (m == 0) return DQ_OK;  // no position to answer
    forget_resident(ctx);
    DQ_TRY(sort_batch_chunk_device(ctx, olds, old_offsets, p0, p1, true));
    dq_stats &st = ctx->stats;
    if (n) {
        DQ_CK(ctx, cudaStreamSynchronize(ctx->stream));
        DQ_CK(ctx, cudaEventElapsedTime(&st.device_ms, ctx->ev0, ctx->ev1));
        DQ_TRY(read_timing(ctx));
    }

    // the per-pair prefix tables (sr::BatchTable) and where each block-minimum level starts in ctx->blevels
    const size_t stride = (size_t)count + 1;
    std::vector<uint32_t> tab((size_t)sr::kBatchTables * stride, 0u);
    auto table = [&](int k) { return tab.data() + (size_t)k * stride; };
    for (uint32_t i = 0; i <= count; ++i) {
        table(sr::kTabOld)[i] = (uint32_t)old_offsets[p0 + i] - obase;
        table(sr::kTabNew)[i] = (uint32_t)new_offsets[p0 + i] - nbase;
    }
    for (uint32_t i = 0; i < count; ++i) {
        const uint32_t ni = table(sr::kTabOld)[i + 1] - table(sr::kTabOld)[i];
        const uint32_t mi = table(sr::kTabNew)[i + 1] - table(sr::kTabNew)[i];
        table(sr::kTabSuper)[i + 1] = table(sr::kTabSuper)[i] + (uint32_t)div_up(mi, sr::kSuper);
        table(sr::kTabChunk)[i + 1] = table(sr::kTabChunk)[i] + (uint32_t)div_up(mi, sr::kChunk);
        uint32_t size[sr::kMaxLevels];
        lcp_levels(ni, size);
        for (int l = 1; l < sr::kMaxLevels; ++l)
            table(sr::kTabLevel + l - 1)[i + 1] = table(sr::kTabLevel + l - 1)[i] + size[l];
    }
    size_t level_at[sr::kMaxLevels] = {}, levels_total = 0;
    for (int l = 1; l < sr::kMaxLevels; ++l) {
        level_at[l] = levels_total;
        levels_total += ((size_t)table(sr::kTabLevel + l - 1)[count] + 63) & ~(size_t)63;
    }
    const uint32_t supers = table(sr::kTabSuper)[count], chunks = table(sr::kTabChunk)[count];

    DQ_TRY(ensure(ctx, ctx->btab, tab.size() * 4));
    DQ_TRY(ensure(ctx, ctx->bisa, (size_t)n * 4));
    DQ_TRY(ensure(ctx, ctx->blevels, levels_total * 4));
    DQ_TRY(ensure(ctx, ctx->headp, (size_t)chunks * 4));
    DQ_TRY(ensure(ctx, ctx->headl, (size_t)chunks * 4));
    DQ_TRY(ensure(ctx, ctx->s_pos, (size_t)m * 4));
    DQ_TRY(ensure(ctx, ctx->s_len, (size_t)m * 4));
    DQ_CK(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    DQ_CK(ctx, cudaMemcpyAsync(ctx->btab.p, tab.data(), tab.size() * 4, cudaMemcpyHostToDevice, ctx->stream));
    DQ_TRY(upload_text(ctx, ctx->newtext, news + nbase, m, cudaMemcpyHostToDevice));
    ctx->runend_new_m = -1;
    const uint32_t *d_tab = ctx->btab.as<uint32_t>();
    sr::BatchPairs bp{};
    bp.olds = ctx->text.as<uint8_t>();
    bp.news = ctx->newtext.as<uint8_t>();
    bp.SA = ctx->sa.as<int32_t>();
    bp.ISA = ctx->bisa.as<uint32_t>();
    bp.lv[0] = ctx->lcp.as<uint32_t>();
    for (int l = 1; l < sr::kMaxLevels; ++l) bp.lv[l] = ctx->blevels.as<uint32_t>() + level_at[l];
    bp.tab = d_tab;
    bp.count = count;
    if (n) {
        const uint32_t g = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(div_up(n, 256 * 4), (uint64_t)ctx->sm_count * 16));
        auto k = sr::batch_local_isa_kernel;
        DQ_LAUNCH(k, g, 256, 0, ctx->stream, bp.SA, d_tab + sr::kTabOld * stride, count, ctx->bisa.as<uint32_t>(), n);
        st.kernel_launches++;
        st.algorithmic_bytes += (int64_t)n * 12;  // SA read, offsets probed (cached), ISA written
    }
    for (int l = 1; l < sr::kMaxLevels; ++l) {
        const uint32_t total = table(sr::kTabLevel + l - 1)[count];
        if (total == 0) break;
        const uint32_t *in = l == 1 ? bp.lv[0] : bp.lv[l - 1];
        const uint32_t *in_off = d_tab + (l == 1 ? (size_t)sr::kTabOld : (size_t)(sr::kTabLevel + l - 2)) * stride;
        const uint32_t in_total = l == 1 ? n : table(sr::kTabLevel + l - 2)[count];
        auto k = sr::batch_block_min_kernel;
        const uint32_t g = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(div_up(total, 8), (uint64_t)ctx->sm_count * 16));
        DQ_LAUNCH(k, g, 256, 0, ctx->stream, in, in_off, const_cast<uint32_t *>(bp.lv[l]),
                  d_tab + (size_t)(sr::kTabLevel + l - 1) * stride, count, total);
        st.kernel_launches++;
        st.algorithmic_bytes += (int64_t)(in_total + total) * 4;
    }
    if (supers) {
        auto k = sr::batch_search_heads_kernel;
        DQ_LAUNCH(k, (uint32_t)div_up((uint64_t)supers * 32, sr::kThreads), sr::kThreads, 0, ctx->stream, bp,
                  ctx->headp.as<uint32_t>(), ctx->headl.as<uint32_t>(), supers);
        auto kc = sr::batch_search_chain_kernel;
        DQ_LAUNCH(kc, (uint32_t)div_up(chunks, sr::kThreads), sr::kThreads, 0, ctx->stream, bp, ctx->headp.as<uint32_t>(),
                  ctx->headl.as<uint32_t>(), ctx->s_pos.as<int32_t>(), ctx->s_len.as<int32_t>(), chunks);
        st.kernel_launches += 2;
    }
    DQ_CK(ctx, cudaGetLastError());
    DQ_CK(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    DQ_CK(ctx, cudaMemcpyAsync(pos_out + nbase, ctx->s_pos.p, (size_t)m * 4, cudaMemcpyDeviceToHost, ctx->stream));
    DQ_CK(ctx, cudaMemcpyAsync(len_out + nbase, ctx->s_len.p, (size_t)m * 4, cudaMemcpyDeviceToHost, ctx->stream));
    DQ_CK(ctx, cudaStreamSynchronize(ctx->stream));
    DQ_CK(ctx, cudaEventElapsedTime(&st.search_ms, ctx->ev0, ctx->ev1));
    return DQ_OK;
}

// body of dq_cuda_bsdiff_search_batch; the arguments are checked.  Routing as suffix_sort_batch's: a pair whose old has
// at least batch_single_min() bytes, or whose new alone exceeds batch_chunk_bytes(), is sorted and searched on its own
// (dq_cuda_suffix_sort + dq_cuda_bsdiff_search with I == NULL, group paths included); the others go in chunks of at most
// batch_chunk_bytes() of olds, as many of news, and kBatchMaxTexts pairs.
int search_batch(dq_ctx *ctx, const uint8_t *olds, const int32_t *old_offsets, const uint8_t *news,
                 const int32_t *new_offsets, int32_t count, int32_t *pos_out, int32_t *len_out)
{
    const uint32_t single_min = batch_single_min();
    const uint64_t chunk_max = batch_chunk_bytes();
    dq_stats acc{};
    auto add = [&]() {
        batch_add_stats(acc, ctx->stats);
        acc.search_ms += ctx->stats.search_ms;
    };
    int32_t begin = 0;  // first pair of the chunk being gathered
    auto flush = [&](int32_t end) -> int {
        if (end == begin) return DQ_OK;
        DQ_TRY(search_batch_chunk(ctx, olds, old_offsets, news, new_offsets, begin, end, pos_out, len_out));
        add();
        begin = end;
        return DQ_OK;
    };
    for (int32_t i = 0; i < count; ++i) {
        const uint32_t n = (uint32_t)(old_offsets[i + 1] - old_offsets[i]), m = (uint32_t)(new_offsets[i + 1] - new_offsets[i]);
        if ((n >= single_min && n > 0) || m > chunk_max) {
            DQ_TRY(flush(i));
            const uint8_t *o = olds + old_offsets[i], *w = news + new_offsets[i];
            int32_t *po = pos_out + new_offsets[i], *lo = len_out + new_offsets[i];
            DQ_TRY(suffix_sort_host(ctx, o, n, nullptr));
            if (group_wants_search(ctx, (int32_t)n, nullptr, (int32_t)m))
                DQ_TRY(group_search_common(ctx, o, (int32_t)n, nullptr, w, (int32_t)m, 0, (int32_t)m, po, lo));
            else
                DQ_TRY(search_common(ctx, o, (int32_t)n, nullptr, w, (int32_t)m, 0, (int32_t)m, po, lo, false));
            DQ_CK(ctx, cudaSetDevice(ctx->device));
            add();
            begin = i + 1;
            continue;
        }
        // a chunk holds at least one pair
        if ((uint32_t)(i - begin) == kBatchMaxTexts ||
            (i > begin && ((uint64_t)(old_offsets[i + 1] - old_offsets[begin]) > chunk_max ||
                           (uint64_t)(new_offsets[i + 1] - new_offsets[begin]) > chunk_max)))
            DQ_TRY(flush(i));
    }
    DQ_TRY(flush(count));
    acc.n = count ? old_offsets[count] : 0;
    acc.search_queries = count ? new_offsets[count] : 0;
    ctx->stats = acc;
    return DQ_OK;
}

void export_streams(dq_ctx *ctx, dq_diff_streams *out);

#if defined(__linux__) && !defined(DQ_EMU)
// ---- pinned host memory interleaved over the NUMA nodes (dq_cuda_host_alloc) ---------------------------------------
std::mutex g_interleaved_mu;
std::vector<std::pair<void *, size_t>> g_interleaved;  // mappings made by interleaved_alloc

int numa_node_count()
{
    int nodes = 0;
    for (int i = 0; i < 64; ++i) {
        char path[64];
        snprintf(path, sizeof path, "/sys/devices/system/node/node%d", i);
        if (access(path, F_OK) != 0) break;
        ++nodes;
    }
    return nodes;
}

bool interleave_wanted()
{
    const char *e = getenv("DQ_HOST_INTERLEAVE");
    if (e && atoi(e) == 0) return false;
    return numa_node_count() > 1;
}

void *interleaved_alloc(size_t bytes)
{
    const size_t len = (bytes + 4095) & ~(size_t)4095;
    void *p = mmap(nullptr, len, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0);
    if (p == MAP_FAILED) return nullptr;
    const int nodes = numa_node_count();
    unsigned long mask = nodes >= 64 ? ~0ul : ((1ul << nodes) - 1ul);
    // mbind(addr, len, MPOL_INTERLEAVE = 3, nodemask, maxnode, 0): pages go round-robin over the nodes as they are touched
    if (syscall(SYS_mbind, p, len, 3, &mask, (unsigned long)(sizeof mask * 8), 0u) != 0) {
        munmap(p, len);
        return nullptr;
    }
    // touch every page (that places it), with a few threads: first touch of gigabytes is slow on one
    {
        const int nt = 8;
        std::vector<std::thread> th;
        for (int t = 0; t < nt; ++t)
            th.emplace_back([=]() {
                const size_t lo = len / nt * t, hi = t == nt - 1 ? len : len / nt * (t + 1);
                for (size_t o = lo & ~(size_t)4095; o < hi; o += 4096) static_cast<volatile char *>(p)[o] = 0;
            });
        for (auto &t : th) t.join();
    }
    if (cudaHostRegister(p, len, cudaHostRegisterPortable | cudaHostRegisterMapped) != cudaSuccess) {
        (void)cudaGetLastError();
        munmap(p, len);
        return nullptr;
    }
    std::lock_guard<std::mutex> lock(g_interleaved_mu);
    g_interleaved.emplace_back(p, len);
    return p;
}

bool interleaved_free(void *p)
{
    size_t len = 0;
    {
        std::lock_guard<std::mutex> lock(g_interleaved_mu);
        for (size_t i = 0; i < g_interleaved.size(); ++i)
            if (g_interleaved[i].first == p) {
                len = g_interleaved[i].second;
                g_interleaved.erase(g_interleaved.begin() + (long)i);
                break;
            }
    }
    if (!len) return false;
    cudaHostUnregister(p);
    munmap(p, len);
    return true;
}
#endif

int destroy_single(dq_ctx *ctx)
{
    if (!ctx) return DQ_OK;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    DevBuf *bufs[] = {&ctx->text, &ctx->keyA, &ctx->keyB, &ctx->valA, &ctx->valB, &ctx->isa, &ctx->sa,
                      &ctx->slotA, &ctx->slotB, &ctx->lb, &ctx->hist, &ctx->auxK, &ctx->auxV, &ctx->partK, &ctx->partV, &ctx->runend, &ctx->depthA, &ctx->depthB,
                      &ctx->runtile, &ctx->runend_new, &ctx->runtile_new, &ctx->seedp, &ctx->seedl, &ctx->pre3, &ctx->pre3tile, &ctx->packed, &ctx->late, &ctx->boffs, &ctx->newtext, &ctx->s_pos,
                      &ctx->s_len, &ctx->lcp, &ctx->headp, &ctx->headl, &ctx->bkt, &ctx->phi, &ctx->plcp, &ctx->d_code, &ctx->d_headcount};
    for (DevBuf *b : bufs)
        if (b->p) cudaFree(b->p);
    for (auto &e : ctx->pass_events) {
        cudaEventDestroy(e.a);
        cudaEventDestroy(e.b);
    }
    for (auto &r : ctx->round_recs) cudaEventDestroy(r.begin);
    if (ctx->h_count) cudaFreeHost(ctx->h_count);
    if (ctx->h_pos.p) cudaFreeHost(ctx->h_pos.p);
    if (ctx->h_len.p) cudaFreeHost(ctx->h_len.p);
    if (ctx->h_code.p) cudaFreeHost(ctx->h_code.p);
    if (ctx->h_heads.p) cudaFreeHost(ctx->h_heads.p);
    if (ctx->h_tiles.p) cudaFreeHost(ctx->h_tiles.p);
    if (ctx->ev0) cudaEventDestroy(ctx->ev0);
    if (ctx->ev1) cudaEventDestroy(ctx->ev1);
    if (ctx->ev_index) cudaEventDestroy(ctx->ev_index);
    if (ctx->ev_copy) cudaEventDestroy(ctx->ev_copy);
    for (int i = 0; i < 8; ++i) {
        if (ctx->slice_ready[i]) cudaEventDestroy(ctx->slice_ready[i]);
        if (ctx->slice_done[i]) cudaEventDestroy(ctx->slice_done[i]);
        if (ctx->slice_stream[i]) cudaStreamDestroy(ctx->slice_stream[i]);
    }
    if (ctx->heads_done) cudaEventDestroy(ctx->heads_done);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return DQ_OK;
}

int create_single(dq_ctx **out, int dev)
{
    cudaError_t e = cudaSuccess;
    dq_ctx *ctx = new (std::nothrow) dq_ctx();
    if (!ctx) return DQ_ERR_OUT_OF_MEMORY;
    ctx->device = dev;
    if (const char *hc = getenv("DQ_HEADS_CAP")) ctx->heads_cap_override = (uint32_t)atoi(hc);
    auto fail = [&](const char *what, cudaError_t err) {
        g_create_error = std::string(what) + ": " + cudaGetErrorString(err);
        destroy_single(ctx);
        return DQ_ERR_CUDA;
    };
    if ((e = cudaSetDevice(dev)) != cudaSuccess) return fail("cudaSetDevice", e);
    if ((e = cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, dev)) != cudaSuccess)
        return fail("cudaDeviceGetAttribute", e);
    if ((e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess)
        return fail("cudaStreamCreate", e);
    if ((e = cudaStreamCreateWithFlags(&ctx->copy_stream, cudaStreamNonBlocking)) != cudaSuccess)
        return fail("cudaStreamCreate", e);
    if ((e = cudaEventCreate(&ctx->heads_done)) != cudaSuccess)
        return fail("cudaEventCreate", e);
    for (int i = 0; i < 8; ++i) {
        if ((e = cudaStreamCreateWithFlags(&ctx->slice_stream[i], cudaStreamNonBlocking)) != cudaSuccess)
            return fail("cudaStreamCreate", e);
        if ((e = cudaEventCreate(&ctx->slice_ready[i])) != cudaSuccess)
            return fail("cudaEventCreate", e);
        if ((e = cudaEventCreate(&ctx->slice_done[i])) != cudaSuccess)
            return fail("cudaEventCreate", e);
    }
    if ((e = cudaEventCreate(&ctx->ev0)) != cudaSuccess) return fail("cudaEventCreate", e);
    if ((e = cudaEventCreate(&ctx->ev1)) != cudaSuccess) return fail("cudaEventCreate", e);
    if ((e = cudaEventCreate(&ctx->ev_index)) != cudaSuccess) return fail("cudaEventCreate", e);
    if ((e = cudaEventCreateWithFlags(&ctx->ev_copy, cudaEventDisableTiming)) != cudaSuccess) return fail("cudaEventCreate", e);
    if ((e = cudaHostAlloc((void **)&ctx->h_count, 64, cudaHostAllocDefault)) != cudaSuccess)
        return fail("cudaHostAlloc", e);
    if ((e = cudaFuncSetAttribute(rx::onesweep_pass_kernel<uint32_t>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)rx::pass_smem_bytes())) != cudaSuccess)
        return fail("cudaFuncSetAttribute", e);
    if ((e = cudaFuncSetAttribute(rx::onesweep_pass_kernel<uint64_t>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)rx::pass_smem_bytes())) != cudaSuccess)
        return fail("cudaFuncSetAttribute", e);
    if ((e = cudaFuncSetAttribute(sx::small_sort_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)sx::small_sort_smem_bytes())) != cudaSuccess)
        return fail("cudaFuncSetAttribute", e);
    if ((e = cudaFuncSetAttribute(rx::onesweep_policy_kernel<ds::BucketPolicy>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)rx::pass_smem_bytes())) != cudaSuccess)
        return fail("cudaFuncSetAttribute", e);
    if ((e = cudaFuncSetAttribute(rx::onesweep_policy_kernel<ds::RunBucketPolicy>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)rx::pass_smem_bytes())) != cudaSuccess)
        return fail("cudaFuncSetAttribute", e);
    if ((e = cudaFuncSetAttribute(rx::onesweep_policy_kernel<ds::RequestPolicy>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)rx::pass_smem_bytes())) != cudaSuccess)
        return fail("cudaFuncSetAttribute", e);
    if ((e = cudaFuncSetAttribute(rx::onesweep_policy_kernel<ds::UpdatePolicy>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)rx::pass_smem_bytes())) != cudaSuccess)
        return fail("cudaFuncSetAttribute", e);
    *out = ctx;
    return DQ_OK;
}


}  // namespace

// ======================================================================================================
extern "C" {

int dq_cuda_create(dq_ctx **out, const int *devices, int ndev)
{
    if (!out) return DQ_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    if (ndev < 0 || ndev > ds::kMaxShards || (ndev > 0 && !devices)) {
        g_create_error = "dq_cuda_create: ndev must be 0.." + std::to_string(ds::kMaxShards) + " with a device list";
        return DQ_ERR_INVALID_ARGUMENT;
    }
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        g_create_error = std::string("no CUDA device (") + cudaGetErrorString(e) + "); libdeltaq_cuda has no CPU fallback";
        return DQ_ERR_NO_DEVICE;
    }
    int dev = 0;
    if (ndev >= 1)
        dev = devices[0];
    else
        cudaGetDevice(&dev);
    dq_ctx *ctx = nullptr;
    int rc = create_single(&ctx, dev);
    if (rc != DQ_OK) return rc;
    if (ndev > 1) {
        rc = create_group(ctx, devices, ndev);
        if (rc != DQ_OK) {
            g_create_error = ctx->err;
            destroy_group(ctx);
            destroy_single(ctx);
            return rc;
        }
    }
    *out = ctx;
    return DQ_OK;
}

int dq_cuda_destroy(dq_ctx *ctx)
{
    if (!ctx) return DQ_OK;
    destroy_group(ctx);
    destroy_single(ctx);
    return DQ_OK;
}

const char *dq_cuda_last_error(dq_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }

int dq_cuda_get_stats(dq_ctx *ctx, dq_stats *out)
{
    if (!ctx || !out) return DQ_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    *out = ctx->stats;
    return DQ_OK;
}

int dq_cuda_set_timing(dq_ctx *ctx, int on)
{
    if (!ctx) return DQ_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    ctx->timing = on != 0;
    return DQ_OK;
}

int dq_cuda_get_pass_times(dq_ctx *ctx, float *ms, int64_t *pairs, int32_t *shift, int cap)
{
    if (!ctx || cap < 0) return DQ_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    const int n = (int)ctx->pass_events_used;
    for (int i = 0; i < n && i < cap; ++i) {
        if (ms) ms[i] = ctx->pass_events[i].ms;
        if (pairs) pairs[i] = (int64_t)ctx->pass_events[i].pairs;
        if (shift) shift[i] = ctx->pass_events[i].shift;
    }
    return n;
}

int dq_cuda_get_round_times(dq_ctx *ctx, float *ms, int64_t *active, int32_t *passes, int cap)
{
    if (!ctx || cap < 0) return DQ_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    const int n = (int)ctx->rounds_used;
    for (int i = 0; i < n && i < cap; ++i) {
        if (ms) ms[i] = ctx->round_recs[i].ms;
        if (active) active[i] = (int64_t)ctx->round_recs[i].active;
        if (passes) passes[i] = ctx->round_recs[i].passes;
    }
    return n;
}

int dq_cuda_host_alloc(void **out, size_t bytes)
{
    if (!out) return DQ_ERR_INVALID_ARGUMENT;
    *out = nullptr;
#if defined(__linux__) && !defined(DQ_EMU)
    // Large buffers on a multi-socket host: pages interleaved over the NUMA nodes, then pinned.  Eight GPUs copying
    // their parts of one suffix array into memory of ONE node are limited by that node (measured: 93 GB/s in all for
    // 8 x 256 MiB), and a single GPU loses nothing.  DQ_HOST_INTERLEAVE=0 turns it off.
    if (bytes >= ((size_t)64 << 20) && interleave_wanted()) {
        void *p = interleaved_alloc(bytes);
        if (p) {
            *out = p;
            return DQ_OK;
        }
    }
#endif
    cudaError_t e = cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault);
    if (e != cudaSuccess) {
        g_create_error = std::string("cudaHostAlloc: ") + cudaGetErrorString(e);
        return DQ_ERR_OUT_OF_MEMORY;
    }
    return DQ_OK;
}

int dq_cuda_host_free(void *p)
{
    if (!p) return DQ_OK;
#if defined(__linux__) && !defined(DQ_EMU)
    if (interleaved_free(p)) return DQ_OK;
#endif
    cudaFreeHost(p);
    return DQ_OK;
}

int dq_cuda_suffix_sort(dq_ctx *ctx, const uint8_t *text, int32_t n, int32_t *sa_out)
{
    if (!ctx) return DQ_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    DQ_TRY(check_args(ctx, n >= 0 && (n == 0 || (text && sa_out)), "dq_cuda_suffix_sort: null buffer or negative length"));
    DQ_CK(ctx, cudaSetDevice(ctx->device));
    return suffix_sort_host(ctx, text, (uint32_t)n, sa_out);
}

int dq_cuda_suffix_sort_batch(dq_ctx *ctx, const uint8_t *texts, const int32_t *offsets, int32_t count, int32_t *sa_out)
{
    return batch_entry(ctx, "dq_cuda_suffix_sort_batch", texts, offsets, count, sa_out, nullptr, false);
}

int dq_cuda_suffix_sort_lcp_batch(dq_ctx *ctx, const uint8_t *texts, const int32_t *offsets, int32_t count,
                                  int32_t *sa_out, int32_t *lcp_out)
{
    return batch_entry(ctx, "dq_cuda_suffix_sort_lcp_batch", texts, offsets, count, sa_out, lcp_out, true);
}

int dq_cuda_suffix_sort_device(dq_ctx *ctx, const uint8_t *d_text, int32_t n, int32_t *d_sa_out)
{
    if (!ctx) return DQ_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    DQ_TRY(check_args(ctx, n >= 0 && (n == 0 || (d_text && d_sa_out)), "dq_cuda_suffix_sort_device: null buffer or negative length"));
    DQ_CK(ctx, cudaSetDevice(ctx->device));
    forget_resident(ctx);
    if (ctx->group && (uint32_t)n >= ctx->group->shard_min) return group_sort(ctx, d_text, (uint32_t)n, d_sa_out);
    DQ_TRY(upload_text(ctx, ctx->text, d_text, (uint32_t)n, cudaMemcpyDeviceToDevice));
    DQ_TRY(sort_resident(ctx, (uint32_t)n));
    if (n) DQ_CK(ctx, cudaMemcpyAsync(d_sa_out, ctx->sa.p, (size_t)n * 4, cudaMemcpyDeviceToDevice, ctx->stream));
    DQ_CK(ctx, cudaStreamSynchronize(ctx->stream));
    hold_resident(ctx, n, ctx->stats.rounds);
    return DQ_OK;
}

int dq_cuda_radix_sort_pairs(dq_ctx *ctx, uint64_t *keys, uint32_t *vals, int32_t count, int32_t key_bits)
{
    if (!ctx) return DQ_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    DQ_TRY(check_args(ctx, count >= 0 && key_bits >= 0 && key_bits <= 64 && (count == 0 || (keys && vals)),
                      "dq_cuda_radix_sort_pairs: bad arguments"));
    if (count == 0 || key_bits == 0) return DQ_OK;
    DQ_CK(ctx, cudaSetDevice(ctx->device));
    ctx->stats = dq_stats{};
    ctx->pass_events_used = 0;
    const size_t c8 = (size_t)count * 8, c4 = (size_t)count * 4;
    DQ_TRY(ensure(ctx, ctx->keyA, c8));
    DQ_TRY(ensure(ctx, ctx->keyB, c8));
    DQ_TRY(ensure(ctx, ctx->valA, c4));
    DQ_TRY(ensure(ctx, ctx->valB, c4));
    DQ_CK(ctx, cudaMemcpyAsync(ctx->keyA.p, keys, c8, cudaMemcpyHostToDevice, ctx->stream));
    DQ_CK(ctx, cudaMemcpyAsync(ctx->valA.p, vals, c4, cudaMemcpyHostToDevice, ctx->stream));
    rx::PassPlan plan{};
    rx::plan_add_field(plan, 0, key_bits);
    DQ_TRY(zero_hist(ctx));
    {
        auto k = sx::hist_only_kernel;
        DQ_LAUNCH(k, producer_grid(ctx, (uint64_t)count), sx::kPackThreads, plan.npass * rx::kRadix * 4, ctx->stream,
                  ctx->keyA.as<uint64_t>(), (uint32_t)count, plan, ctx->hist.as<uint32_t>());
    }
    SortBufs s{ctx->keyA.as<uint64_t>(), ctx->keyB.as<uint64_t>(), ctx->valA.as<uint32_t>(), ctx->valB.as<uint32_t>()};
    DQ_TRY(run_passes(ctx, s, (uint32_t)count, plan, false));
    DQ_CK(ctx, cudaMemcpyAsync(keys, s.kin, c8, cudaMemcpyDeviceToHost, ctx->stream));
    DQ_CK(ctx, cudaMemcpyAsync(vals, s.vin, c4, cudaMemcpyDeviceToHost, ctx->stream));
    DQ_CK(ctx, cudaStreamSynchronize(ctx->stream));
    return DQ_OK;
}

}  // extern "C"

extern "C" {

int dq_cuda_bsdiff_search(dq_ctx *ctx, const uint8_t *old_, int32_t n, const int32_t *I_or_null, const uint8_t *new_,
                          int32_t m, int32_t scan_begin, int32_t count, int32_t *pos_out, int32_t *len_out)
{
    if (!ctx) return DQ_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (group_wants_search(ctx, n, I_or_null, count))
        return group_search_common(ctx, old_, n, I_or_null, new_, m, scan_begin, count, pos_out, len_out);
    return search_common(ctx, old_, n, I_or_null, new_, m, scan_begin, count, pos_out, len_out, false);
}

int dq_cuda_bsdiff_search_device(dq_ctx *ctx, const uint8_t *d_old, int32_t n, const int32_t *d_I_or_null,
                                 const uint8_t *d_new, int32_t m, int32_t scan_begin, int32_t count,
                                 int32_t *d_pos_out, int32_t *d_len_out)
{
    if (!ctx) return DQ_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (group_wants_search(ctx, n, d_I_or_null, count))
        return group_search_common(ctx, d_old, n, d_I_or_null, d_new, m, scan_begin, count, d_pos_out, d_len_out);
    return search_common(ctx, d_old, n, d_I_or_null, d_new, m, scan_begin, count, d_pos_out, d_len_out, true);
}

int dq_cuda_bsdiff_search_batch(dq_ctx *ctx, const uint8_t *olds, const int32_t *old_offsets, const uint8_t *news,
                                const int32_t *new_offsets, int32_t count, int32_t *pos_out, int32_t *len_out)
{
    if (!ctx) return DQ_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    auto check = [&](bool ok, const char *what) {
        return check_args(ctx, ok, (std::string("dq_cuda_bsdiff_search_batch: ") + what).c_str());
    };
    DQ_TRY(check(count >= 0, "negative count"));
    DQ_TRY(check((old_offsets && new_offsets) || count == 0, "offsets is null"));
    if (count == 0) return DQ_OK;
    for (const int32_t *offsets : {old_offsets, new_offsets}) {
        DQ_TRY(check(offsets[0] == 0, "offsets[0] must be 0"));
        for (int32_t i = 0; i < count; ++i) DQ_TRY(check(offsets[i + 1] >= offsets[i], "offsets decrease"));
    }
    DQ_TRY(check((old_offsets[count] == 0 || olds) && (new_offsets[count] == 0 || (news && pos_out && len_out)),
                 "null buffer"));
    DQ_CK(ctx, cudaSetDevice(ctx->device));
    ctx->search_seen = true;
    const int rc = search_batch(ctx, olds, old_offsets, news, new_offsets, count, pos_out, len_out);
    // after the batch: its chunks overwrite text / SA / ISA, and a pair it searches alone holds its old
    forget_resident(ctx);
    return rc;
}

int dq_cuda_lcp(dq_ctx *ctx, const uint8_t *text, int32_t n, const int32_t *I_or_null, int32_t *lcp_out)
{
    if (!ctx) return DQ_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    return lcp_host(ctx, text, n, I_or_null, lcp_out);
}

int dq_cuda_lcp_device(dq_ctx *ctx, const uint8_t *d_text, int32_t n, const int32_t *d_I_or_null, int32_t *d_lcp_out)
{
    if (!ctx) return DQ_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    if (!d_I_or_null && d_lcp_out && group_holds(ctx, n)) return group_lcp(ctx, n, d_lcp_out);
    return lcp_common(ctx, d_text, n, d_I_or_null, d_lcp_out, true);
}

// Diff.cs:90 and :106 for dq_cuda_bsdiff_streams: makes `old` resident and enqueues the (pos, len) table of every scan
// position, whose coded slices reach the host as slice_done[0 .. slices_used) fire; sets *group_search_ms on a group
static int sort_and_search(dq_ctx *ctx, const uint8_t *old_, int32_t n, const uint8_t *new_, int32_t m, bool trace,
                           const std::function<double()> &since, float *group_search_ms)
{
    // Diff.cs:90 -- suffixSort.Sort(oldData, I[..^1]); the suffix array stays on the device
    forget_resident(ctx);
    ctx->search_seen = true;
    if (ctx->group && m > 0 && (uint32_t)n >= ctx->group->shard_min) {
        // a device group and a large pair (BASELINE config #5): `old` is sorted by all GPUs, every GPU answers its share
        // of the scan positions into this context's table (peer copies), which is then coded and consumed by the caller
        DQ_TRY(ensure(ctx, ctx->s_pos, (size_t)m * 4));
        DQ_TRY(ensure(ctx, ctx->s_len, (size_t)m * 4));
        DQ_TRY(group_sort(ctx, old_, (uint32_t)n, nullptr));
        const int32_t sort_rounds = ctx->stats.rounds;
        const float sort_ms = ctx->stats.device_ms;
        if (trace) fprintf(stderr, "[dq trace] sorted by the group %.3f ms\n", since());
        DQ_TRY(group_search_common(ctx, old_, n, nullptr, new_, m, 0, m, ctx->s_pos.as<int32_t>(), ctx->s_len.as<int32_t>()));
        *group_search_ms = ctx->stats.search_ms;
        if (trace) fprintf(stderr, "[dq trace] searched by the group %.3f ms\n", since());
        DQ_CK(ctx, cudaSetDevice(ctx->device));
        DQ_TRY(search_resident(ctx, (uint32_t)n, (uint32_t)m, 0, (uint32_t)m, true, true));
        ctx->stats.rounds = sort_rounds;
        ctx->stats.device_ms = sort_ms;
        return DQ_OK;
    }
    // `old` goes up first and alone -- the sort waits for it, nothing waits for `new` before the search -- and `new`
    // follows on the copy stream once round 0 of the sort is enqueued: the two uploads do not share the PCIe link, and
    // where the caller's buffer is pageable (a managed caller's `fixed` span: the copy call then holds the host until
    // the bytes are staged) the host is held while the GPU has round 0 to work on, not in front of the sort.
    DQ_TRY(ensure(ctx, ctx->newtext, (size_t)m + 64));
    ctx->runend_new_m = -1;
    DQ_TRY(upload_text(ctx, ctx->text, old_, (uint32_t)n, cudaMemcpyHostToDevice));
    DQ_CK(ctx, cudaEventRecord(ctx->ev_copy, ctx->stream));   // (no early copy of the suffix array on this path)
    bool new_sent = false;
    const std::function<int()> send_new = [&]() -> int {
        if (new_sent) return DQ_OK;
        new_sent = true;
        DQ_CK(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_copy, 0));
        if (m) DQ_CK(ctx, cudaMemcpyAsync(ctx->newtext.p, new_, (size_t)m, cudaMemcpyHostToDevice, ctx->copy_stream));
        DQ_CK(ctx, cudaMemsetAsync(ctx->newtext.as<uint8_t>() + m, 0, 64, ctx->copy_stream));
        // run ends of `new` (used by the search when the sort finds `old` full of equal-byte runs): computed
        // beside the sort, rather than in front of the search
        if (m >= (1 << 20)) DQ_TRY(run_ends_of_new(ctx, (uint32_t)m, ctx->copy_stream));
        DQ_CK(ctx, cudaEventRecord(ctx->slice_done[0], ctx->copy_stream));
        return DQ_OK;
    };
    DQ_TRY(sort_resident(ctx, (uint32_t)n, nullptr, nullptr, &send_new));
    DQ_TRY(send_new());   // the sorts that return before round 0 (n == 0, one CTA)
    hold_resident(ctx, n, ctx->stats.rounds);
    if (ctx->runend_new_m == m) ctx->stats.kernel_launches += 3;  // run_ends_of_new above (the sort resets the stats)
    if (trace) fprintf(stderr, "[dq trace] sorted %.3f ms\n", since());
    DQ_CK(ctx, cudaStreamWaitEvent(ctx->stream, ctx->slice_done[0], 0));
    // Diff.cs:106 for every scan position, in slices; each slice crosses PCIe in its coded form (dq_search.cuh,
    // encode_table_kernel) while later slices are still being searched and the host loop runs
    return search_resident(ctx, (uint32_t)n, (uint32_t)m, 0, (uint32_t)m, true);
}

// body of dq_cuda_bsdiff_streams; the caller holds ctx->mu
static int bsdiff_streams_locked(dq_ctx *ctx, const uint8_t *old_, int32_t n, const uint8_t *new_, int32_t m,
                                 dq_diff_streams *out)
{
    DQ_TRY(check_args(ctx, n >= 0 && m >= 0 && (n == 0 || old_) && (m == 0 || new_), "bsdiff_streams: bad arguments"));
    // the host loop looks up to 64 positions ahead in 32-bit arithmetic
    DQ_TRY(check_args(ctx, m <= INT32_MAX - 64, "bsdiff_streams: newData longer than INT32_MAX - 64 bytes"));
    DQ_CK(ctx, cudaSetDevice(ctx->device));
    const bool trace = getenv("DQ_TRACE") != nullptr;
    const auto t_begin = std::chrono::steady_clock::now();
    auto since = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_begin).count(); };
    float group_search_ms = -1.f;  // >= 0: the search ran on a device group and this is its time
    DQ_TRY(sort_and_search(ctx, old_, n, new_, m, trace, since, &group_search_ms));
    // Diff.cs:100-223 on the host, consuming the table as its slices land
    int next = 0;
    int32_t ready_end = 0;
    cudaError_t werr = cudaSuccess;
    auto ready = [&](int32_t upto) {
        if (upto > m) upto = m;
        while (ready_end < upto && next < ctx->slices_used) {
            cudaError_t e_ = cudaEventSynchronize(ctx->slice_done[next]);
            if (e_ != cudaSuccess) {
                werr = e_;
                throw std::runtime_error("table slice did not arrive");  // never walk a table that was not filled
            }
            ready_end = ctx->slice_end[next++];
            if (trace) fprintf(stderr, "[dq trace] slice %d landed %.3f ms\n", next - 1, since());
        }
    };
    // pos of a short match: only the last stop of the scan can ask (see dq_search.cuh), by then every slice is done
    auto fetch_pos = [&](int32_t scan) -> int32_t {
        int32_t v = 0;
        cudaError_t e_ = cudaMemcpyAsync(&v, ctx->s_pos.as<int32_t>() + scan, 4, cudaMemcpyDeviceToHost, ctx->copy_stream);
        if (e_ == cudaSuccess) e_ = cudaStreamSynchronize(ctx->copy_stream);
        if (e_ != cudaSuccess) {
            werr = e_;
            throw std::runtime_error("could not fetch a table entry");
        }
        return v;
    };
    if (trace) fprintf(stderr, "[dq trace] search enqueued %.3f ms\n", since());
    bool overflow = false;
    // nothing thrown by the host loop (allocation failures, thread creation, a table slice that never arrived) may cross
    // the C ABI: it becomes a status
    try {
    if (m) {
        static_assert(sizeof(dq::diffhost::MatchHead) == sizeof(dq::search::MatchHead) && sizeof(dq::diffhost::TileEntry) == sizeof(uint2),
                      "host and device views of the coded table must agree");
        dq::diffhost::CodedTable<decltype(fetch_pos)> tab{static_cast<const uint8_t *>(ctx->h_code.p),
                                                          static_cast<const dq::diffhost::TileEntry *>(ctx->h_tiles.p),
                                                          static_cast<const dq::diffhost::MatchHead *>(ctx->h_heads.p),
                                                          ctx->heads_cap, fetch_pos};
        try {
            dq::diffhost::greedy_emit_pipelined(old_, n, new_, m, tab, ctx->streams, ready);
        } catch (const dq::diffhost::CodedOverflow &) {
            overflow = true;
        }
    } else {
        dq::diffhost::reset_streams(ctx->streams, 0);
        dq::diffhost::FullTable none{nullptr, nullptr};
        dq::diffhost::greedy_emit_pipelined(old_, n, new_, m, none, ctx->streams, ready);
    }
    if (overflow) {
        // more match heads than the pinned list holds (every few positions starts a new long match): take the
        // whole table across and run the same loop over the plain arrays
        DQ_CK(ctx, cudaStreamSynchronize(ctx->copy_stream));
        DQ_CK(ctx, cudaStreamSynchronize(ctx->stream));
        DQ_TRY(ensure_pinned(ctx, ctx->h_pos, (size_t)m * 4 + 4));
        DQ_TRY(ensure_pinned(ctx, ctx->h_len, (size_t)m * 4 + 4));
        int32_t *h_pos = static_cast<int32_t *>(ctx->h_pos.p), *h_len = static_cast<int32_t *>(ctx->h_len.p);
        DQ_CK(ctx, cudaMemcpyAsync(h_pos, ctx->s_pos.p, (size_t)m * 4, cudaMemcpyDeviceToHost, ctx->stream));
        DQ_CK(ctx, cudaMemcpyAsync(h_len, ctx->s_len.p, (size_t)m * 4, cudaMemcpyDeviceToHost, ctx->stream));
        DQ_CK(ctx, cudaStreamSynchronize(ctx->stream));
        dq::diffhost::FullTable full{h_pos, h_len};
        dq::diffhost::greedy_emit_pipelined(old_, n, new_, m, full, ctx->streams, [](int32_t) {});
        ctx->stats.table_fallbacks++;
    }
    } catch (const std::bad_alloc &) {
        cudaStreamSynchronize(ctx->copy_stream);
        cudaStreamSynchronize(ctx->stream);
        ctx->err = "bsdiff_streams: out of host memory";
        return DQ_ERR_OUT_OF_MEMORY;
    } catch (const std::exception &ex) {
        cudaStreamSynchronize(ctx->copy_stream);
        cudaStreamSynchronize(ctx->stream);
        ctx->err = std::string("bsdiff_streams: ") + ex.what() +
                   (werr != cudaSuccess ? std::string(" (") + cudaGetErrorString(werr) + ")" : std::string());
        return werr != cudaSuccess ? DQ_ERR_CUDA : DQ_ERR_INTERNAL;
    }
    if (trace) fprintf(stderr, "[dq trace] host loop done %.3f ms (scan side %.3f ms, extender done %.3f ms / busy %.3f ms), %zu stops, %lld bytes certified equal%s\n", since(), ctx->streams.scan_done_ms, ctx->streams.extender_done_ms, ctx->streams.extender_busy_ms, ctx->streams.ctrl.size() / 24, (long long)ctx->streams.cert_bytes, overflow ? " [full-table fallback]" : "");
    DQ_CK(ctx, cudaStreamSynchronize(ctx->copy_stream));
    DQ_CK(ctx, cudaStreamSynchronize(ctx->stream));
    DQ_CK(ctx, werr);
    if (m) DQ_CK(ctx, cudaEventElapsedTime(&ctx->stats.search_ms, ctx->ev0, ctx->ev1));
    if (m) DQ_CK(ctx, cudaEventElapsedTime(&ctx->stats.search_index_ms, ctx->ev0, ctx->ev_index));
    if (group_search_ms >= 0.f) ctx->stats.search_ms += group_search_ms;  // the coding above + the group's search
    if (m) {
        uint32_t heads = 0;
        DQ_CK(ctx, cudaMemcpy(&heads, ctx->d_headcount.p, 4, cudaMemcpyDeviceToHost));
        ctx->stats.table_heads = (int32_t)heads;
    }
    if (trace && m) {
        float a = 0, b = 0;
        cudaEventElapsedTime(&a, ctx->ev0, ctx->heads_done);
        fprintf(stderr, "[dq trace] device: search start -> heads done %.3f ms, -> all done %.3f ms\n", a, ctx->stats.search_ms);
        for (int sl = 0; sl < ctx->slices_used; ++sl) {
            cudaEventElapsedTime(&a, ctx->ev0, ctx->slice_ready[sl]);
            cudaEventElapsedTime(&b, ctx->ev0, ctx->slice_done[sl]);
            fprintf(stderr, "[dq trace] device: slice %d chains done %.3f ms, code on host %.3f ms\n", sl, a, b);
        }
    }
    export_streams(ctx, out);
    return DQ_OK;
}

int dq_cuda_bsdiff_streams(dq_ctx *ctx, const uint8_t *old_, int32_t n, const uint8_t *new_, int32_t m,
                           dq_diff_streams *out)
{
    if (!ctx || !out) return DQ_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    return bsdiff_streams_locked(ctx, old_, n, new_, m, out);
}

int64_t dq_cuda_bz2_bound(int64_t n) { return n < 0 ? -1 : dq::bz2host::bound(n); }

int dq_cuda_bz2_compress(const uint8_t *const *src, const int64_t *len, int count, int level, int threads,
                         uint8_t *const *out, const int64_t *cap, int64_t *out_len, int32_t *info)
{
    if (count < 0 || count > 64 || level < 0 || level > 9 || threads < 0) return DQ_ERR_INVALID_ARGUMENT;
    if (count && (!src || !len || !out || !cap || !out_len)) return DQ_ERR_INVALID_ARGUMENT;
    dq::bz2host::StreamJob jobs[64];
    for (int s = 0; s < count; ++s) {
        if (len[s] < 0 || (len[s] && !src[s]) || !out[s] || cap[s] < dq::bz2host::bound(len[s])) return DQ_ERR_INVALID_ARGUMENT;
        jobs[s].src = src[s];
        jobs[s].len = len[s];
        jobs[s].out = out[s];
        jobs[s].cap = cap[s];
    }
    int rc;
    try {
        rc = dq::bz2host::compress_streams(jobs, count, level, threads);
    } catch (const std::bad_alloc &) {
        return DQ_ERR_OUT_OF_MEMORY;
    } catch (...) {
        return DQ_ERR_INTERNAL;
    }
    if (rc != 0) return DQ_ERR_INTERNAL;  // libbz2 missing or failing; the buffers were checked above
    for (int s = 0; s < count; ++s) {
        out_len[s] = jobs[s].out_len;
        if (info) {
            info[3 * s] = jobs[s].level;
            info[3 * s + 1] = jobs[s].pieces;
            info[3 * s + 2] = jobs[s].fell_back ? 1 : 0;
        }
    }
    return DQ_OK;
}

int dq_cuda_bz2_decompress(const uint8_t *src, int64_t len, int threads, uint8_t *out, int64_t cap, int64_t *out_len,
                           int32_t *info)
{
    if (len < 0 || (len && !src) || threads < 0 || cap < 0 || (cap && !out) || !out_len) return DQ_ERR_INVALID_ARGUMENT;
    dq::bz2host::DecodeJob job;
    job.src = src;
    job.len = len;
    int rc;
    try {
        rc = dq::bz2host::decompress_streams(&job, 1, threads);
    } catch (const std::bad_alloc &) {
        return DQ_ERR_OUT_OF_MEMORY;
    } catch (...) {
        return DQ_ERR_INTERNAL;
    }
    if (rc == -3) return DQ_ERR_INTERNAL;
    if (rc != 0) return DQ_ERR_CORRUPT_PATCH;
    *out_len = (int64_t)job.out.size();
    if (info) {
        info[0] = job.blocks;
        info[1] = job.fell_back ? 1 : 0;
    }
    if ((int64_t)job.out.size() > cap) return DQ_ERR_INVALID_ARGUMENT;  // *out_len says how much room is needed
    if (!job.out.empty()) memcpy(out, job.out.data(), job.out.size());
    return DQ_OK;
}

int dq_cuda_bspatch(const uint8_t *old_, int64_t n, const uint8_t *patch, int64_t patch_len, int threads, uint8_t *out,
                    int64_t out_cap, int64_t *new_size)
{
    if (n < 0 || (n && !old_) || patch_len < 0 || (patch_len && !patch) || threads < 0 || out_cap < 0 || !new_size)
        return DQ_ERR_INVALID_ARGUMENT;
    namespace bz = dq::bz2host;
    // Patch.cs:52-93: signature, the two section lengths and the size of the new file, all packed longs
    if (patch_len < 32 || memcmp(patch, "BSDIFF40", 8) != 0) return DQ_ERR_CORRUPT_PATCH;
    const int64_t ctrl_len = dq::patchhost::read_packed_long(patch + 8);
    const int64_t diff_len = dq::patchhost::read_packed_long(patch + 16);
    const int64_t size = dq::patchhost::read_packed_long(patch + 24);
    if (ctrl_len < 0 || diff_len < 0 || size < 0) return DQ_ERR_CORRUPT_PATCH;
    if (ctrl_len > patch_len - 32 || diff_len > patch_len - 32 - ctrl_len) return DQ_ERR_CORRUPT_PATCH;
    *new_size = size;
    if (out_cap < size || (size && !out)) return DQ_ERR_INVALID_ARGUMENT;  // *new_size says how much room is needed
    try {
        bz::DecodeJob jobs[3];
        jobs[0].src = patch + 32;
        jobs[0].len = ctrl_len;
        jobs[1].src = patch + 32 + ctrl_len;
        jobs[1].len = diff_len;
        jobs[2].src = patch + 32 + ctrl_len + diff_len;
        jobs[2].len = patch_len - 32 - ctrl_len - diff_len;
        // what a patch for `size` bytes can use: at most size diff bytes, size extra bytes and one triple per output byte
        // (+ one); a section that decodes to more than that (plus slack) is damaged or hostile, and is not unpacked further
        const int64_t slack = 1 << 20;
        jobs[0].limit = size > (INT64_MAX - slack) / 24 - 1 ? INT64_MAX : 24 * (size + 1) + slack;
        jobs[1].limit = jobs[2].limit = size + slack;
        const int rc = bz::decompress_streams(jobs, 3, threads);
        if (rc == -3) return DQ_ERR_INTERNAL;
        if (rc != 0) return DQ_ERR_CORRUPT_PATCH;
        return dq::patchhost::apply_streams(old_, n, jobs[0].out.data(), (int64_t)jobs[0].out.size(), jobs[1].out.data(),
                                            (int64_t)jobs[1].out.size(), jobs[2].out.data(), (int64_t)jobs[2].out.size(),
                                            out, size) == 0
                   ? DQ_OK
                   : DQ_ERR_CORRUPT_PATCH;
    } catch (const std::bad_alloc &) {
        return DQ_ERR_OUT_OF_MEMORY;
    } catch (...) {
        return DQ_ERR_INTERNAL;
    }
}

int dq_cuda_bsdiff_patch(dq_ctx *ctx, const uint8_t *old_, int32_t n, const uint8_t *new_, int32_t m, int level,
                         const uint8_t **patch, int64_t *patch_len)
{
    if (!ctx || !patch || !patch_len || level < 0 || level > 9) return DQ_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    dq_diff_streams st;
    DQ_TRY(bsdiff_streams_locked(ctx, old_, n, new_, m, &st));
    // Diff.cs:54-70, :226-241: header (signature, compressed sizes of ctrl and diff, size of newData), then the sections
    namespace bz = dq::bz2host;
    try {
        bz::StreamJob jobs[3];
        const uint8_t *srcs[3] = {st.ctrl, st.diff, st.extra};
        const int64_t lens[3] = {st.ctrl_len, st.diff_len, st.extra_len};
        for (int s = 0; s < 3; ++s) {
            jobs[s].src = srcs[s];
            jobs[s].len = lens[s];
            jobs[s].out = nullptr;
            jobs[s].cap = 0;
        }
        bz::SectionCompressor sections;
        const int rc = sections.run(jobs, 3, level, 0);
        if (rc != 0) {
            ctx->err = rc == -3 ? "bsdiff_patch: libbz2 not found" : "bsdiff_patch: libbz2 failed";
            return DQ_ERR_INTERNAL;
        }
        // the sizes are known before a byte is stitched: the sections go straight to their places behind the header
        const int64_t size[3] = {sections.size(0), sections.size(1), sections.size(2)};
        ctx->patch.len = 0;
        ctx->patch.reserve((size_t)(32 + size[0] + size[1] + size[2]));
        uint8_t *p = ctx->patch.p;
        auto packed = [](uint8_t *b, int64_t y) {  // SpanExtensions.WritePackedLong (SpanExtensions.cs:7-18), y >= 0 here
            for (int i = 0; i < 8; ++i) b[i] = (uint8_t)((uint64_t)y >> (8 * i));
        };
        memcpy(p, "BSDIFF40", 8);
        packed(p + 8, size[0]);
        packed(p + 16, size[1]);
        packed(p + 24, (int64_t)m);
        int64_t at = 32;
        for (int s = 0; s < 3; ++s) {
            if (!sections.write(s, p + at, size[s]) || jobs[s].out_len != size[s]) {
                ctx->err = "bsdiff_patch: section size mismatch";
                return DQ_ERR_INTERNAL;
            }
            at += size[s];
        }
        ctx->patch.len = (size_t)at;
    } catch (const std::bad_alloc &) {
        ctx->err = "bsdiff_patch: out of host memory";
        return DQ_ERR_OUT_OF_MEMORY;
    }
    *patch = ctx->patch.p;
    *patch_len = (int64_t)ctx->patch.len;
    return DQ_OK;
}

int dq_cuda_patch_apply(const uint8_t *old_, int64_t n, const uint8_t *ctrl, int64_t ctrl_len, const uint8_t *diff,
                        int64_t diff_len, const uint8_t *extra, int64_t extra_len, uint8_t *out, int64_t new_size)
{
    if (n < 0 || ctrl_len < 0 || diff_len < 0 || extra_len < 0 || new_size < 0) return DQ_ERR_INVALID_ARGUMENT;
    if ((n && !old_) || (ctrl_len && !ctrl) || (diff_len && !diff) || (extra_len && !extra) || (new_size && !out))
        return DQ_ERR_INVALID_ARGUMENT;
    return dq::patchhost::apply_streams(old_, n, ctrl, ctrl_len, diff, diff_len, extra, extra_len, out, new_size) == 0
               ? DQ_OK
               : DQ_ERR_CORRUPT_PATCH;
}

int dq_cuda_greedy_emit(dq_ctx *ctx, const uint8_t *old_, int32_t n, const uint8_t *new_, int32_t m,
                        const int32_t *pos_tab, const int32_t *len_tab, dq_diff_streams *out)
{
    if (!ctx || !out) return DQ_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    DQ_TRY(check_args(ctx, n >= 0 && m >= 0 && m <= INT32_MAX - 64 && (n == 0 || old_) && (m == 0 || (new_ && pos_tab && len_tab)),
                      "greedy_emit: bad arguments"));
    // same threads as dq_cuda_bsdiff_streams uses (scan / extender + crew / writers), over the caller's arrays
    dq::diffhost::FullTable tab{pos_tab, len_tab};
    try {
        dq::diffhost::greedy_emit_pipelined(old_, n, new_, m, tab, ctx->streams, [](int32_t) {});
    } catch (const std::bad_alloc &) {
        ctx->err = "greedy_emit: out of host memory";
        return DQ_ERR_OUT_OF_MEMORY;
    } catch (const std::exception &ex) {
        ctx->err = std::string("greedy_emit: ") + ex.what();
        return DQ_ERR_INTERNAL;
    }
    export_streams(ctx, out);
    return DQ_OK;
}

}  // extern "C"

namespace {
void export_streams(dq_ctx *ctx, dq_diff_streams *out)
{
    out->ctrl = ctx->streams.ctrl.data();
    out->ctrl_len = (int64_t)ctx->streams.ctrl.size();
    out->diff = ctx->streams.diff.data();
    out->diff_len = (int64_t)ctx->streams.diff.size();
    out->extra = ctx->streams.extra.data();
    out->extra_len = (int64_t)ctx->streams.extra.size();
    out->search_visits = ctx->streams.visits;
}
}  // namespace

#ifdef DQ_PROF
extern "C" int dq_debug_read_prof_cmp(unsigned long long *clk, unsigned long long *bytes, unsigned int *calls)
{
    if (cudaMemcpyFromSymbol(clk, dq::search::g_prof_cmp_clk, 8u << 16) != cudaSuccess) return -1;
    if (cudaMemcpyFromSymbol(bytes, dq::search::g_prof_cmp_bytes, 8u << 16) != cudaSuccess) return -1;
    return cudaMemcpyFromSymbol(calls, dq::search::g_prof_cmp_calls, 4u << 16) == cudaSuccess ? 0 : -1;
}
extern "C" int dq_debug_read_prof_seeds(uint32_t *seeds)
{
    return cudaMemcpyFromSymbol(seeds, dq::search::g_prof_seeds, sizeof(uint32_t) << 16) == cudaSuccess ? 0 : -1;
}
extern "C" int dq_debug_read_prof(uint32_t *chains, uint32_t *heads)
{
    if (cudaMemcpyFromSymbol(chains, dq::search::g_prof_chain, sizeof(uint32_t) << 21) != cudaSuccess) return -1;
    if (cudaMemcpyFromSymbol(heads, dq::search::g_prof_heads, sizeof(uint32_t) << 16) != cudaSuccess) return -1;
    return 0;
}
#endif

#ifdef DQ_EMU
extern "C" void dq_emu_debug_counters(unsigned long long *out, int reset)
{
    auto &d = dq::search::g_dbg;
    out[0] = d.scratch; out[1] = d.probes; out[2] = d.cmp_bytes; out[3] = d.walk; out[4] = d.walk_max; out[5] = d.anchors;
    out[6] = d.thr_max[0]; out[7] = d.thr_max[1];
    for (int k = 0; k < 24; ++k) { out[8 + k] = d.thr_hist[0][k]; out[32 + k] = d.thr_hist[1][k]; }
    if (reset) d = dq::search::DebugCounters{};
}
#endif

// ======================================================================================================
// building blocks exported for tests and reuse
extern "C" {

// sorts in place, optionally returns the first digit's counts
static int radix_sort_device_locked(dq_ctx *ctx, uint64_t *d_keys, uint32_t *d_vals, int32_t count, int32_t bit_lo,
                                    int32_t nbits, int64_t *hist_out_host)
{
    if (hist_out_host) std::fill(hist_out_host, hist_out_host + 256, (int64_t)0);
    if (count == 0 || nbits == 0) return DQ_OK;
    const size_t c8 = (size_t)count * 8, c4 = (size_t)count * 4;
    // own scratch: keyA/keyB/valA/valB may hold a multi-GPU session's unresolved set
    DQ_TRY(ensure(ctx, ctx->auxK, c8));
    DQ_TRY(ensure(ctx, ctx->auxV, c4));
    rx::PassPlan plan{};
    rx::plan_add_field(plan, bit_lo, nbits);
    DQ_TRY(zero_hist(ctx));
    {
        auto k = sx::hist_only_kernel;
        DQ_LAUNCH(k, producer_grid(ctx, (uint64_t)count), sx::kPackThreads, plan.npass * rx::kRadix * 4, ctx->stream, d_keys,
                  (uint32_t)count, plan, ctx->hist.as<uint32_t>());
    }
    if (hist_out_host) {
        // The sort's first pass covers fewer than 8 bits whenever nbits > 8 is not a multiple of 8 (plan_add_field
        // splits the field evenly), so the promised first digit, bits [bit_lo, bit_lo + min(nbits, 8)), is counted
        // on its own.  Its counters go to the gbase table, which run_passes' scan rewrites before any pass reads it.
        rx::PassPlan first{};
        rx::plan_add_field(first, bit_lo, std::min(nbits, rx::kRadixBits));
        uint32_t *first_hist = ctx->hist.as<uint32_t>() + rx::kMaxPasses * rx::kRadix;
        DQ_CK(ctx, cudaMemsetAsync(first_hist, 0, rx::kRadix * 4, ctx->stream));
        auto k = sx::hist_only_kernel;
        DQ_LAUNCH(k, producer_grid(ctx, (uint64_t)count), sx::kPackThreads, first.npass * rx::kRadix * 4, ctx->stream,
                  d_keys, (uint32_t)count, first, first_hist);
        uint32_t h32[256];
        DQ_CK(ctx, cudaMemcpyAsync(h32, first_hist, sizeof h32, cudaMemcpyDeviceToHost, ctx->stream));
        DQ_CK(ctx, cudaStreamSynchronize(ctx->stream));
        for (int i = 0; i < 256; ++i) hist_out_host[i] = h32[i];
    }
    SortBufs s{d_keys, ctx->auxK.as<uint64_t>(), d_vals, ctx->auxV.as<uint32_t>()};
    DQ_TRY(run_passes(ctx, s, (uint32_t)count, plan, false));
    if (s.kin != d_keys) {
        DQ_CK(ctx, cudaMemcpyAsync(d_keys, s.kin, c8, cudaMemcpyDeviceToDevice, ctx->stream));
        DQ_CK(ctx, cudaMemcpyAsync(d_vals, s.vin, c4, cudaMemcpyDeviceToDevice, ctx->stream));
    }
    DQ_CK(ctx, cudaStreamSynchronize(ctx->stream));
    return DQ_OK;
}

int dq_cuda_radix_sort_pairs_device(dq_ctx *ctx, uint64_t *d_keys, uint32_t *d_vals, int32_t count, int32_t bit_lo,
                                    int32_t nbits, int64_t *hist_out_host)
{
    if (!ctx) return DQ_ERR_INVALID_ARGUMENT;
    std::lock_guard<std::mutex> lock(ctx->mu);
    DQ_TRY(check_args(ctx, count >= 0 && bit_lo >= 0 && nbits >= 0 && bit_lo + nbits <= 64 && (count == 0 || (d_keys && d_vals)),
                      "radix_sort_pairs_device: bad arguments"));
    DQ_CK(ctx, cudaSetDevice(ctx->device));
    return radix_sort_device_locked(ctx, d_keys, d_vals, count, bit_lo, nbits, hist_out_host);
}

}  // extern "C"
