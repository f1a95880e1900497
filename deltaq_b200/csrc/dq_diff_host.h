// dq_diff_host.h -- host consumer of the bulk (pos, len) table: the reference's greedy scan / extend / emit
// loop, /root/reference/src/DeltaQ.BsDiff/Diff.cs:92-223, kept statement for statement except that the call
//     len = Search(I, oldData, newData[scan..], 0, oldData.Length, out pos);          (Diff.cs:106)
// is the array read  len = len_tab[scan]; pos = pos_tab[scan];  -- the hook SURVEY.md section 8(b) describes.
// Emits the three UNCOMPRESSED streams (ctrl triples as packed longs, SpanExtensions.cs:7-30).
//
// Same results, faster stepping: the byte-at-a-time loops of the reference are advanced many bytes at a time wherever
// a whole stretch behaves uniformly (all bytes equal, a running maximum that cannot be beaten, a test whose outcome
// is already decided), which leaves every variable the loop looks at again exactly as the reference's loop would
// (the argument is written at each site); anything else falls back to the reference's own single-byte step.
// The loop runs on a few host threads (greedy_emit_pipelined): scan -> extender (+ crew) -> writers.
#pragma once
#include <cstdint>
#include <chrono>
#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <memory>
#include <stdexcept>
#include <thread>
#include <vector>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif
#if defined(__linux__)
#include <sched.h>
#endif

namespace dq {
namespace diffhost {

// grow-only byte sink whose new bytes are NOT value-initialised (the diff stream is as long as `new`)
struct ByteBuf {
    std::unique_ptr<uint8_t[]> p;
    size_t len = 0, cap = 0;
    void reserve(size_t c)
    {
        if (c <= cap) return;
        std::unique_ptr<uint8_t[]> q(new uint8_t[c]);
        if (len) std::memcpy(q.get(), p.get(), len);
        p = std::move(q);
        cap = c;
    }
    uint8_t *grow(size_t k)
    {
        if (len + k > cap) reserve(std::max(len + k, cap * 2 + 4096));
        uint8_t *at = p.get() + len;
        len += k;
        return at;
    }
    void clear() { len = 0; }
    const uint8_t *data() const { return p.get(); }
    size_t size() const { return len; }
};

struct Streams {
    std::vector<uint8_t> ctrl;
    ByteBuf diff, extra;
    int64_t visits = 0;
    // DQ_TRACE: when the scan side finished (relative to the start of the loop), and how long the other threads
    // spent working rather than waiting
    double scan_done_ms = 0, extender_busy_ms = 0, writer_busy_ms = 0, extender_done_ms = 0;
    int64_t cert_errors = 0, cert_bytes = 0;  // DQ_CHECK_CERTS: certified stretches that were not equal; bytes certified
};

// bit k of the result is set iff a[k] == b[k], k in [0, 32)
inline uint32_t eq_mask32(const uint8_t *a, const uint8_t *b)
{
#if defined(__SSE2__)
    const __m128i a0 = _mm_loadu_si128(reinterpret_cast<const __m128i *>(a));
    const __m128i b0 = _mm_loadu_si128(reinterpret_cast<const __m128i *>(b));
    const __m128i a1 = _mm_loadu_si128(reinterpret_cast<const __m128i *>(a + 16));
    const __m128i b1 = _mm_loadu_si128(reinterpret_cast<const __m128i *>(b + 16));
    return (uint32_t)_mm_movemask_epi8(_mm_cmpeq_epi8(a0, b0)) |
           ((uint32_t)_mm_movemask_epi8(_mm_cmpeq_epi8(a1, b1)) << 16);
#else
    uint32_t m = 0;
    for (int k = 0; k < 32; ++k) m |= (uint32_t)(a[k] == b[k]) << k;
    return m;
#endif
}

// any of v[0..16) > 8 ?
inline bool any_greater_than_8(const int32_t *v)
{
#if defined(__SSE2__)
    const __m128i eight = _mm_set1_epi32(8);
    __m128i g = _mm_cmpgt_epi32(_mm_loadu_si128(reinterpret_cast<const __m128i *>(v)), eight);
    g = _mm_or_si128(g, _mm_cmpgt_epi32(_mm_loadu_si128(reinterpret_cast<const __m128i *>(v + 4)), eight));
    g = _mm_or_si128(g, _mm_cmpgt_epi32(_mm_loadu_si128(reinterpret_cast<const __m128i *>(v + 8)), eight));
    g = _mm_or_si128(g, _mm_cmpgt_epi32(_mm_loadu_si128(reinterpret_cast<const __m128i *>(v + 12)), eight));
    return _mm_movemask_epi8(g) != 0;
#else
    for (int k = 0; k < 16; ++k)
        if (v[k] > 8) return true;
    return false;
#endif
}

inline int32_t count_equal(const uint8_t *a, const uint8_t *b, int32_t len)
{
    int32_t cnt = 0, k = 0;
    for (; k + 32 <= len; k += 32) cnt += __builtin_popcount(eq_mask32(a + k, b + k));
    for (; k < len; ++k) cnt += (a[k] == b[k]);
    return cnt;
}

// index of the last k in [0, len) with a[k] != b[k], or -1
inline int32_t last_mismatch(const uint8_t *a, const uint8_t *b, int32_t len)
{
    int32_t k = len;
    while (k > 0 && (k & 31)) {
        --k;
        if (a[k] != b[k]) return k;
    }
    while (k >= 32) {
        const uint32_t ne = ~eq_mask32(a + k - 32, b + k - 32);
        if (ne) return k - 32 + (31 - __builtin_clz(ne));
        k -= 32;
    }
    return -1;
}

inline void put_packed_long(std::vector<uint8_t> &out, int64_t y)
{
    uint64_t u = y < 0 ? (uint64_t)0 - (uint64_t)y : (uint64_t)y;
    uint8_t b[8];
    for (int i = 0; i < 8; ++i) b[i] = (uint8_t)(u >> (8 * i));
    if (y < 0) b[7] |= 0x80;
    out.insert(out.end(), b, b + 8);
}

// ---- what the scan reads of the (pos, len) table ------------------------------------------------------------
constexpr int32_t kPosUnknown = INT32_MIN;

// the table as two plain arrays (dq_cuda_greedy_emit, and the fallback of dq_cuda_bsdiff_streams)
struct FullTable {
    static constexpr bool kExactMatches = false;  // the caller's arrays are taken as they are
    const int32_t *pos_tab, *len_tab;
    int32_t short_len(int32_t scan) const { return len_tab[scan]; }
    bool any_long16(int32_t scan) const { return any_greater_than_8(len_tab + scan); }
    // max(e, scan + i + len[scan + i]) over i in [0, 16); only called when any_long16(scan) is false
    int32_t max_end16(int32_t scan, int32_t e) const
    {
        for (int32_t i = 0; i < 16; ++i) {
            const int32_t t = scan + i + len_tab[scan + i];
            e = t > e ? t : e;
        }
        return e;
    }
    void get(int32_t scan, int32_t &len, int32_t &pos)
    {
        len = len_tab[scan];
        pos = pos_tab[scan];
    }
    int32_t fetch_pos(int32_t scan) { return pos_tab[scan]; }
};

// the table as the device encodes it for the trip over PCIe (encode_table_kernel, dq_search.cuh): one byte
// min(len, 9) per position, and (at, pos, len) for the head of every chain of long matches.  The scan only moves
// forwards, so the head that governs a long position is found by a cursor that only moves forwards too.
struct MatchHead {
    int32_t at, pos, len;
};
struct TileEntry {
    uint32_t base, count;
};
struct CodedOverflow {};  // thrown by the scan when the head list did not fit: the caller falls back to FullTable

template <typename FetchPos> struct CodedTable {
    static constexpr bool kExactMatches = true;  // written by this library's own search: len is the longest match
    static constexpr int kTileShift = 10;
    static constexpr int32_t kLong = 9;
    const uint8_t *code;
    const TileEntry *tiles;
    const MatchHead *heads;
    uint32_t heads_cap;
    FetchPos fetch;
    uint32_t next_tile = 0, next_k = 0;
    MatchHead cur{-1, 0, 0};

    // masks over positions scan + i, i in [0, 16): len > 8 / len != 0 / len == 1
    void classify16(int32_t scan, uint32_t &is_long, uint32_t &nonzero, uint32_t &one) const
    {
#if defined(__SSE2__)
        const __m128i c = _mm_loadu_si128(reinterpret_cast<const __m128i *>(code + scan));
        is_long = (uint32_t)_mm_movemask_epi8(_mm_cmpgt_epi8(c, _mm_set1_epi8(8)));
        nonzero = ~(uint32_t)_mm_movemask_epi8(_mm_cmpeq_epi8(c, _mm_setzero_si128())) & 0xffffu;
        one = (uint32_t)_mm_movemask_epi8(_mm_cmpeq_epi8(c, _mm_set1_epi8(1)));
#else
        is_long = nonzero = one = 0;
        for (int k = 0; k < 16; ++k) {
            is_long |= (uint32_t)(code[scan + k] > 8) << k;
            nonzero |= (uint32_t)(code[scan + k] != 0) << k;
            one |= (uint32_t)(code[scan + k] == 1) << k;
        }
#endif
    }
    int32_t short_len(int32_t scan) const { return code[scan]; }
    void advance(int32_t scan)
    {
        const uint32_t last_tile = (uint32_t)scan >> kTileShift;
        for (;;) {
            while (next_tile <= last_tile && next_k >= tiles[next_tile].count) {
                ++next_tile;
                next_k = 0;
            }
            if (next_tile > last_tile) return;
            const uint32_t at = tiles[next_tile].base + next_k;
            if (at >= heads_cap) throw CodedOverflow{};
            const MatchHead h = heads[at];
            if (h.at > scan) return;
            cur = h;
            ++next_k;
        }
    }
    void get(int32_t scan, int32_t &len, int32_t &pos)
    {
        const int32_t c = code[scan];
        if (c < kLong) {
            len = c;
            pos = kPosUnknown;
            return;
        }
        advance(scan);
        len = cur.len - (scan - cur.at);
        pos = cur.pos + (scan - cur.at);
    }
    int32_t fetch_pos(int32_t scan) { return fetch(scan); }
    // get(scan) just returned a long match: the last position whose long match still continues it (its len keeps
    // scan + len where it is).  Looks at heads up to that position: the caller makes sure they have arrived.
    int32_t chain_reach(int32_t scan) const { return cur.at + cur.len - kLong > scan ? cur.at + cur.len - kLong : scan; }
    int32_t chain_last(int32_t reach) const
    {
        uint32_t t = next_tile, k = next_k;
        const uint32_t last_tile = (uint32_t)reach >> kTileShift;
        while (t <= last_tile && k >= tiles[t].count) {
            ++t;
            k = 0;
        }
        if (t > last_tile) return reach;
        const uint32_t at = tiles[t].base + k;
        if (at >= heads_cap) throw CodedOverflow{};
        const int32_t next_head = heads[at].at;
        return next_head - 1 < reach ? next_head - 1 : reach;
    }
};

// ---- Diff.cs:132-145 / :152-164: the best extension ---------------------------------------------------------
// Both loops walk i = 1..span counting matches s and keep the FIRST i at which 2*s - i exceeds everything before
// it (and 0).  Restated over 8 steps at a time: for the 8 equal/unequal outcomes of a group, the table gives the
// group's total, its best running value and the first step reaching that -- the one update the byte loop would
// be left with.  Two more shortcuts, both exact: an all-equal block of 32 rises by one per step, so its last step
// is the update; and once even a perfect remainder cannot beat the best so far, the loop has nothing left to do.
struct StepLut {
    int8_t total[256], best[256], first[256];     // steps taken from bit 0 upwards
    int8_t rtotal[256], rbest[256], rfirst[256];  // steps taken from bit 7 downwards
    StepLut()
    {
        for (int m = 0; m < 256; ++m) {
            int run = 0, b = -100, at = 0;
            for (int k = 0; k < 8; ++k) {
                run += ((m >> k) & 1) ? 1 : -1;
                if (run > b) b = run, at = k + 1;
            }
            total[m] = (int8_t)run, best[m] = (int8_t)b, first[m] = (int8_t)at;
            run = 0, b = -100, at = 0;
            for (int k = 0; k < 8; ++k) {
                run += ((m >> (7 - k)) & 1) ? 1 : -1;
                if (run > b) b = run, at = k + 1;
            }
            rtotal[m] = (int8_t)run, rbest[m] = (int8_t)b, rfirst[m] = (int8_t)at;
        }
    }
};
inline const StepLut &step_lut()
{
    static const StepLut lut;
    return lut;
}

// What a stretch of steps does to the walk: its total, the best running value inside it and the first step
// (1-based) reaching that.  Stretches combine left to right exactly like single steps do.
struct Run {
    int32_t total, best, first;
};
constexpr int32_t kNoBest = INT32_MIN / 2;

// step i (1-based) compares a[i-1] with b[i-1].  kWhole: walk all of span with no best to beat (a Run for
// combining); otherwise start from (0, 0) and leave as soon as the rest cannot matter.
template <bool kWhole> inline Run walk_forward(const uint8_t *a, const uint8_t *b, int32_t span)
{
    const StepLut &lut = step_lut();
    int32_t cur = 0, best = kWhole ? kNoBest : 0, at = 0, done = 0;
    while (done + 32 <= span) {
        if (!kWhole && cur + (span - done) <= best) return Run{cur, best, at};
        const uint32_t eq = eq_mask32(a + done, b + done);
        if (eq == 0xffffffffu) {
            cur += 32;
            done += 32;
            if (cur > best) best = cur, at = done;
            continue;
        }
        const int32_t p = __builtin_popcount(eq);
        if (cur + p > best) {
            int32_t c = cur;
            for (int q = 0; q < 4; ++q) {
                const uint32_t m = (eq >> (8 * q)) & 255u;
                if (c + lut.best[m] > best) best = c + lut.best[m], at = done + 8 * q + lut.first[m];
                c += lut.total[m];
            }
        }
        cur += 2 * p - 32;
        done += 32;
    }
    for (; done < span;) {
        cur += (a[done] == b[done]) ? 1 : -1;
        ++done;
        if (cur > best) best = cur, at = done;
    }
    return Run{cur, best, at};
}

// step i (1-based) compares a_end[-i] with b_end[-i]
template <bool kWhole> inline Run walk_backward(const uint8_t *a_end, const uint8_t *b_end, int32_t span)
{
    const StepLut &lut = step_lut();
    int32_t cur = 0, best = kWhole ? kNoBest : 0, at = 0, done = 0;
    while (done + 32 <= span) {
        if (!kWhole && cur + (span - done) <= best) return Run{cur, best, at};
        // bit k <-> step done + 32 - k (the block is read forwards, the loop walks backwards)
        const uint32_t eq = eq_mask32(a_end - done - 32, b_end - done - 32);
        if (eq == 0xffffffffu) {
            cur += 32;
            done += 32;
            if (cur > best) best = cur, at = done;
            continue;
        }
        const int32_t p = __builtin_popcount(eq);
        if (cur + p > best) {
            int32_t c = cur;
            for (int q = 3; q >= 0; --q) {
                const uint32_t m = (eq >> (8 * q)) & 255u;
                if (c + lut.rbest[m] > best) best = c + lut.rbest[m], at = done + 8 * (3 - q) + lut.rfirst[m];
                c += lut.rtotal[m];
            }
        }
        cur += 2 * p - 32;
        done += 32;
    }
    for (; done < span;) {
        ++done;
        cur += (a_end[-done] == b_end[-done]) ? 1 : -1;
        if (cur > best) best = cur, at = done;
    }
    return Run{cur, best, at};
}

// One step of waiting for another thread of the pipeline: pause for the first `pauses` steps (the hand-offs of a busy
// pipeline are microseconds apart), then yield, and after a few milliseconds of yields sleep, so that a stage with nothing to
// do (a crew waiting for the next long extension, the stages of other processes sharing the cores when one process per
// GPU runs this loop) leaves its core to the threads that have work.
inline void wait_step(int &spins, int pauses)
{
    ++spins;
    if (spins < pauses) {
#if defined(__SSE2__)
        _mm_pause();
#endif
    } else if (spins < pauses + 20000) {  // a few milliseconds of yields: longer than any gap inside one call
        std::this_thread::yield();
    } else {
        std::this_thread::sleep_for(std::chrono::microseconds(50));
    }
}

// ---- helper threads for the long stretches --------------------------------------------------------------------
// fork-join over a fixed crew: run(f) calls f(part) for part in [0, parts()), part 0 on the calling thread
class Crew {
    std::vector<std::thread> th_;
    std::atomic<uint64_t> epoch_{0};
    std::atomic<int> pending_{0};
    std::atomic<bool> quit_{false};
    std::function<void(int)> job_;
    static void idle(int &spins) { wait_step(spins, 2048); }

public:
    explicit Crew(int helpers)
    {
        for (int h = 0; h < helpers; ++h)
            th_.emplace_back([this, h]() {
                uint64_t seen = 0;
                for (;;) {
                    int spins = 0;
                    while (epoch_.load(std::memory_order_acquire) == seen && !quit_.load(std::memory_order_acquire)) idle(spins);
                    if (quit_.load(std::memory_order_acquire)) return;
                    ++seen;
                    job_(h + 1);
                    pending_.fetch_sub(1, std::memory_order_acq_rel);
                }
            });
    }
    ~Crew()
    {
        quit_.store(true, std::memory_order_release);
        for (auto &t : th_) t.join();
    }
    int parts() const { return (int)th_.size() + 1; }
    template <typename F> void run(F &&f)
    {
        if (th_.empty()) {
            f(0);
            return;
        }
        job_ = f;
        pending_.store((int)th_.size(), std::memory_order_release);
        epoch_.fetch_add(1, std::memory_order_acq_rel);
        f(0);
        int spins = 0;
        while (pending_.load(std::memory_order_acquire) > 0) idle(spins);
    }
};

// bytes one crew member walks per wave / stretches shorter than this stay on the calling thread
// (DQ_HOST_THREADS="helpers,writers,part_kib,min_kib" overrides both)
inline int32_t &crew_part() { static int32_t v = 64 << 10; return v; }
inline int32_t &crew_min() { static int32_t v = 128 << 10; return v; }

// The first step at which the walk's running value exceeds everything before it (and 0), or 0 if none does --
// what all three loops of Diff.cs:132-188 compute.  walk(lo, len, whole) returns the Run of steps [lo, lo+len);
// no step raises the value by more than one.  Long stretches go to the crew in waves: each member walks one part
// into a Run, the Runs are combined in order (the same updates the byte loop would make), and the early exit is
// tested between waves.
template <typename Walk> inline int32_t first_best_step(Crew *crew, int32_t span, Walk &&walk)
{
    if (!crew || crew->parts() == 1 || span < crew_min()) return walk(0, span, false).first;
    const int P = crew->parts();
    int32_t cur = 0, best = 0, at = 0, done = 0;
    Run r[16];
    while (done < span) {
        if (cur + (span - done) <= best) break;
        const int32_t wave = (int32_t)std::min<int64_t>(span - done, (int64_t)P * crew_part());
        const int32_t per = (int32_t)((((int64_t)wave + P - 1) / P + 31) & ~(int64_t)31);
        crew->run([&](int part) {
            const int32_t lo = (int32_t)std::min<int64_t>(wave, (int64_t)part * per);
            const int32_t hi = (int32_t)std::min<int64_t>(wave, (int64_t)(part + 1) * per);
            r[part] = lo < hi ? walk(done + lo, hi - lo, true) : Run{0, kNoBest, 0};
        });
        for (int part = 0; part < P; ++part) {
            if (r[part].best != kNoBest && cur + r[part].best > best) {
                best = cur + r[part].best;
                at = done + (int32_t)std::min<int64_t>(wave, (int64_t)part * per) + r[part].first;
            }
            cur += r[part].total;
        }
        done += wave;
    }
    return at;
}

// A stretch of new the scan has PROVED equal to old at the alignment of the piece it lies in: new[start .. start+len) ==
// old[start+lastoffset .. +len).  The scan gets this for free -- it leaves its inner loop either at a match whose len bytes
// all agree at the current alignment (Diff.cs:117, len == oldscore: no stop, the same piece goes on) or at a stop, whose
// exact match (pos, len) starts the next piece at the alignment pos - scan -- and most of an edited file is made of such
// stretches.  The forward extension (Diff.cs:132-145) walks them without reading them (every step is +1, so the last one
// is the update), and their diff bytes are zeros.
struct Cert {
    int32_t start, len;
};
constexpr int32_t kCertMin = 256;      // shorter stretches are not worth a queue slot
constexpr int32_t kZeroJobMin = 4096;  // shorter ones are not worth a writer job of their own

// first_best_step for the forward walk of a piece that starts at new offset `base`, with the certified stretches of that
// piece (ascending, disjoint).  Real steps run in whole-mode Runs (chunks on this thread, waves on the crew) and combine
// exactly as single steps do; the early exit is tested between them.
template <typename Walk>
inline int32_t first_best_step_certified(Crew *crew, int32_t span, int32_t base, const Cert *certs, size_t ncerts, Walk &&walk)
{
    const int P = crew ? crew->parts() : 1;
    constexpr int32_t kChunk = 8 << 10;
    int32_t cur = 0, best = 0, at = 0, done = 0;
    size_t c = 0;
    Run r[16];
    auto take = [&](const Run &x, int32_t lo) {
        if (x.best != kNoBest && cur + x.best > best) {
            best = cur + x.best;
            at = lo + x.first;
        }
        cur += x.total;
    };
    while (done < span) {
        if (cur + (span - done) <= best) break;
        while (c < ncerts && (int64_t)certs[c].start + certs[c].len - base <= done) ++c;
        int32_t cs = span, ce = span;  // the next certified stretch in steps, clipped to what is left
        if (c < ncerts) {
            cs = (int32_t)std::min<int64_t>(span, std::max<int64_t>(done, (int64_t)certs[c].start - base));
            ce = (int32_t)std::min<int64_t>(span, std::max<int64_t>(cs, (int64_t)certs[c].start + certs[c].len - base));
        }
        if (cs == done) {
            if (ce > done) {  // inside it: the value rises by one per step
                cur += ce - done;
                done = ce;
                if (cur > best) best = cur, at = done;
            }
            continue;
        }
        const int32_t gap = cs - done;
        if (P == 1 || gap < crew_min()) {
            const int32_t len = std::min(gap, kChunk);
            take(walk(done, len, true), done);
            done += len;
            continue;
        }
        const int32_t wave = (int32_t)std::min<int64_t>(gap, (int64_t)P * crew_part());
        const int32_t per = (int32_t)((((int64_t)wave + P - 1) / P + 31) & ~(int64_t)31);
        crew->run([&](int part) {
            const int32_t lo = (int32_t)std::min<int64_t>(wave, (int64_t)part * per);
            const int32_t hi = (int32_t)std::min<int64_t>(wave, (int64_t)(part + 1) * per);
            r[part] = lo < hi ? walk(done + lo, hi - lo, true) : Run{0, kNoBest, 0};
        });
        for (int part = 0; part < P; ++part) take(r[part], done + (int32_t)std::min<int64_t>(wave, (int64_t)part * per));
        done += wave;
    }
    return at;
}

// Diff.cs:172-188: step i (1-based) adds (n1[i-1] == o1[i-1]) - (n2[i-1] == o2[i-1])
template <bool kWhole>
inline Run walk_overlap(const uint8_t *n1, const uint8_t *o1, const uint8_t *n2, const uint8_t *o2, int32_t span)
{
    int32_t cur = 0, best = kWhole ? kNoBest : 0, at = 0, i = 0;
    while (i < span) {
        if (!kWhole && cur + (span - i) <= best) break;
        if (i + 32 <= span) {
            const uint32_t ma = eq_mask32(n1 + i, o1 + i), mb = eq_mask32(n2 + i, o2 + i);
            // the value can rise only where the first comparison alone matches
            if (cur + __builtin_popcount(ma & ~mb) <= best) {
                cur += __builtin_popcount(ma) - __builtin_popcount(mb);
                i += 32;
                continue;
            }
            for (int k = 0; k < 32; ++k, ++i) {
                cur += (int32_t)((ma >> k) & 1u) - (int32_t)((mb >> k) & 1u);
                if (cur > best) best = cur, at = i + 1;
            }
            continue;
        }
        cur += (int32_t)(n1[i] == o1[i]) - (int32_t)(n2[i] == o2[i]);
        ++i;
        if (cur > best) best = cur, at = i;
    }
    return Run{cur, best, at};
}

// One stop of the scan, in two steps.  extend_stop: forward/backward extension and overlap split (Diff.cs:127-194),
// which chain lastscan/lastpos from one stop to the next.  write_piece: the emission (Diff.cs:196-217), which feeds
// nothing back.
struct EmitState {
    int32_t lastscan = 0, lastpos = 0;
};
struct Piece {
    int32_t lastscan, lastpos, lenf, extra;
    int64_t seek;
};

inline Piece extend_stop(const uint8_t *oldData, int32_t oldLen, const uint8_t *newData, int32_t newLen, int32_t scan,
                         int32_t pos, EmitState &st, Crew *crew = nullptr, const Cert *certs = nullptr, size_t ncerts = 0)
{
    int32_t &lastscan = st.lastscan, &lastpos = st.lastpos;
    // Diff.cs:132-145
    const int32_t fspan = (scan - lastscan) < (oldLen - lastpos) ? (scan - lastscan) : (oldLen - lastpos);
    const uint8_t *fo = oldData + lastpos, *fn = newData + lastscan;
    auto fwalk = [&](int32_t lo, int32_t len, bool whole) {
        return whole ? walk_forward<true>(fo + lo, fn + lo, len) : walk_forward<false>(fo + lo, fn + lo, len);
    };
    int32_t lenf = ncerts ? first_best_step_certified(crew, fspan, lastscan, certs, ncerts, fwalk)
                          : first_best_step(crew, fspan, fwalk);

    // Diff.cs:147-165
    int32_t lenb = 0;
    if (scan < newLen) {
        const int32_t bspan = (scan - lastscan) < pos ? (scan - lastscan) : pos;
        const uint8_t *bo = oldData + pos, *bn = newData + scan;
        lenb = first_best_step(crew, bspan, [&](int32_t lo, int32_t len, bool whole) {
            return whole ? walk_backward<true>(bo - lo, bn - lo, len) : walk_backward<false>(bo - lo, bn - lo, len);
        });
    }

    // Diff.cs:167-194
    if (lastscan + lenf > scan - lenb) {
        const int32_t overlap = (lastscan + lenf) - (scan - lenb);
        const uint8_t *n1 = newData + lastscan + lenf - overlap, *o1 = oldData + lastpos + lenf - overlap;
        const uint8_t *n2 = newData + scan - lenb, *o2 = oldData + pos - lenb;
        // n1 == n2 (both name the overlapping range of new); when the two matches also share their offset into
        // old, every step adds and takes away the same comparison and the value never leaves 0: lens = 0
        const int32_t lens = o1 == o2 ? 0 : first_best_step(crew, overlap, [&](int32_t lo, int32_t len, bool whole) {
            return whole ? walk_overlap<true>(n1 + lo, o1 + lo, n2 + lo, o2 + lo, len)
                         : walk_overlap<false>(n1 + lo, o1 + lo, n2 + lo, o2 + lo, len);
        });
        lenf += lens - overlap;
        lenb -= lens;
    }

    const Piece pc{lastscan, lastpos, lenf, (scan - lenb) - (lastscan + lenf), (int64_t)((pos - lenb) - (lastpos + lenf))};
    lastscan = scan - lenb;
    lastpos = pos - lenb;
    return pc;
}

inline void write_piece(const uint8_t *oldData, const uint8_t *newData, const Piece &pc, Streams &out)
{
    const int32_t lenf = pc.lenf;
    {
        // Diff.cs:197-200
        uint8_t *dst = out.diff.grow((size_t)(lenf > 0 ? lenf : 0));
        const uint8_t *pn = newData + pc.lastscan, *po = oldData + pc.lastpos;
        int32_t i = 0;
#if defined(__SSE2__)
        for (; i + 16 <= lenf; i += 16)
            _mm_storeu_si128(reinterpret_cast<__m128i *>(dst + i),
                             _mm_sub_epi8(_mm_loadu_si128(reinterpret_cast<const __m128i *>(pn + i)),
                                          _mm_loadu_si128(reinterpret_cast<const __m128i *>(po + i))));
#endif
        for (; i < lenf; i++) dst[i] = (uint8_t)(pn[i] - po[i]);
    }
    if (pc.extra > 0) std::memcpy(out.extra.grow((size_t)pc.extra), newData + pc.lastscan + lenf, (size_t)pc.extra);
    put_packed_long(out.ctrl, lenf);
    put_packed_long(out.ctrl, pc.extra);
    put_packed_long(out.ctrl, pc.seek);
}

// ready(upto): returns once table entries [0, min(upto, newLen)) are valid (the table may still be arriving from
// the device in slices while the loop runs)
struct NoCerts {
    void operator()(int32_t, int32_t) const {}
};
// certified(start, len): see Cert; called only for tables whose entries are exact longest matches
template <typename Table, typename Ready, typename Sink, typename CertSink = NoCerts>
inline void greedy_scan(const uint8_t *oldData, int32_t oldLen, const uint8_t *newData, int32_t newLen,
                        Table &tab, Streams &out, Ready &&ready, Sink &&sink, CertSink &&certified = CertSink{})
{
    int32_t scan = 0, pos = 0, len = 0;
    int32_t lastoffset = 0;
    int32_t last_read = -1;  // the position pos was read at (a coded table hands out short-match pos on demand)

    while (scan < newLen) {
        int32_t oldscore = 0;

        for (int32_t scsc = scan += len; scan < newLen; scan++) {
            ready(scan + 64);
            if constexpr (Table::kExactMatches) {
                // Sixteen positions at a time while all of them hold short matches (len <= 8).  With len the
                // longest match at each position, scan + len never decreases along the scan, so when position x is
                // tested scsc == x + len[x] and oldscore counts exactly the bytes of new[x .. x+len[x]) equal to
                // their partners at the current offset (whatever was added for earlier positions has been taken
                // away again by Diff.cs:123-125).  A short position therefore stops the scan iff len != 0 and all
                // of its len bytes agree (len == oldscore; len > oldscore + 8 cannot hold), which is read off
                // one 32-byte comparison mask.  Leaving the block with scsc = scan and oldscore = 0 is the same
                // state as the reference's as far as every later test can tell.
                bool stopped = false;
                while (scan + 48 <= newLen && (int64_t)scan + lastoffset + 32 <= (int64_t)oldLen) {
                    uint32_t is_long, nonzero, one;
                    tab.classify16(scan, is_long, nonzero, one);
                    if (is_long) break;
                    const uint32_t eq = eq_mask32(oldData + scan + lastoffset, newData + scan);
                    // a stop needs its first byte equal, and its second too unless len == 1
                    uint32_t cand = eq & nonzero & ((eq >> 1) | one);
                    while (cand) {
                        const int32_t i = __builtin_ctz(cand);
                        cand &= cand - 1;
                        const int32_t c = tab.short_len(scan + i);
                        const uint32_t run = (1u << c) - 1u;
                        if (((eq >> i) & run) == run) {
                            scan += i;
                            len = c;
                            pos = kPosUnknown;
                            last_read = scan;
                            oldscore = c;
                            out.visits += i + 1;
                            stopped = true;
                            break;
                        }
                    }
                    if (stopped) break;
                    scan += 16;
                    out.visits += 16;
                    scsc = scan;
                    oldscore = 0;
                    ready(scan + 64);
                }
                if (stopped) break;
            } else {
            // Block step over positions that cannot end the scan.  While oldscore == 0 and no byte of
            // new[scan .. scan+kBlk+8) equals its partner at the current offset, nothing can be added to or
            // taken from oldscore by the next kBlk positions (their matches are <= 8 long, so scsc stays inside
            // that window): each of them evaluates "(len == 0 && len != 0) || len > 8" = false.  The reference
            // would visit them one by one with the same outcome; scsc ends at the same running maximum.
                constexpr int32_t kBlk = 16;
                while (oldscore == 0 && scan + 32 + kBlk <= newLen && scsc <= scan + kBlk + 8 &&
                       (int64_t)scan + lastoffset + 32 <= (int64_t)oldLen) {
                    if (eq_mask32(oldData + scan + lastoffset, newData + scan) & 0x00ffffffu) break;
                    if (tab.any_long16(scan)) break;
                    scsc = tab.max_end16(scan, scsc);
                    scan += kBlk;
                    out.visits += kBlk;
                    ready(scan + 64);
                }
            }
            tab.get(scan, len, pos);
            last_read = scan;
            out.visits++;

            bool far_off = false;  // more than 8 bytes of the match disagree at the current offset
            {
                // Diff.cs:108-114.  scsc + lastoffset >= lastpos >= 0, so only the upper bound can fire: count
                // equal bytes over the part of [scsc, scan+len) that stays inside oldData.
                const int64_t lim = (int64_t)oldLen - lastoffset;  // scsc < lim  <=>  scsc + lastoffset < oldLen
                const int32_t stop = scan + len;
                const int32_t inb = (int32_t)(lim < stop ? (lim > scsc ? lim : scsc) : stop);
                if (Table::kExactMatches && pos != kPosUnknown && pos - scan == lastoffset && scsc <= stop) {
                    // the match found IS the current alignment: every byte of [scan, stop) equals its partner, and
                    // whatever oldscore held for [scan, scsc) is part of that, so the count comes out at len
                    oldscore = len;
                } else if (len > 8 && scsc >= scan && inb > scsc) {
                    // Same count, but it may stop early: the test below only asks whether the bytes of
                    // [scan, stop) that disagree number 0, 1..8 or more, and once they pass 8 the scan stops here
                    // and oldscore is not looked at again (it is reset at Diff.cs:102).
                    int32_t miss = (scsc - scan) - oldscore + (stop - inb);  // seen so far + bytes past the end of old
                    const uint8_t *a = oldData + lastoffset + scsc, *b = newData + scsc;
                    const int32_t total = inb - scsc;
                    int32_t k = 0;
                    for (; miss <= 8 && k + 32 <= total; k += 32) {
                        const int32_t e = __builtin_popcount(eq_mask32(a + k, b + k));
                        oldscore += e;
                        miss += 32 - e;
                    }
                    if (miss <= 8) {
                        const int32_t e = count_equal(a + k, b + k, total - k);
                        oldscore += e;
                        miss += (total - k) - e;
                    }
                    far_off = miss > 8;
                } else if (inb > scsc) {
                    oldscore += count_equal(oldData + lastoffset + scsc, newData + scsc, inb - scsc);
                }
                if (scsc < stop) scsc = stop;
            }

            if (far_off || (len == oldscore && len != 0) || (len > oldscore + 8)) break;

            if constexpr (Table::kExactMatches) {
                // A long match that is neither the current alignment nor far from it: 1..8 of its bytes disagree
                // at the current offset.  The positions after this one continue the same match (len one less each,
                // scan + len fixed) for as long as the table says so, and for them the test only changes when the
                // LAST disagreeing byte has dropped out of [scan, scan + len): nothing stops the scan before that
                // position, so go there directly (the reference visits every position in between; count them).
                if (len > 8 && scsc == scan + len) {
                    const int32_t stop = scan + len;
                    const int32_t reach = tab.chain_reach(scan);
                    if (reach > scan + 1) {
                        ready(reach + 64);
                        const int32_t chain_last = tab.chain_last(reach);
                        const int64_t lim = (int64_t)oldLen - lastoffset;
                        const int32_t inb = (int32_t)(lim < stop ? (lim > scan ? lim : scan) : stop);
                        const int32_t lastmiss =
                            inb < stop ? stop - 1 : scan + last_mismatch(oldData + lastoffset + scan, newData + scan, stop - scan);
                        const int32_t target = lastmiss < chain_last ? lastmiss + 1 : chain_last + 1;
                        if (target > scan + 1) {
                            oldscore = lastmiss < target ? stop - target
                                                         : (inb > target ? count_equal(oldData + lastoffset + target, newData + target, inb - target) : 0);
                            out.visits += target - scan - 1;
                            scan = target - 1;
                            continue;
                        }
                    }
                }
            }

            if ((scan + lastoffset < oldLen) && (oldData[scan + lastoffset] == newData[scan])) oldscore--;
        }

        if (len != oldscore || scan == newLen) {
            // Diff.cs:127-222 for this stop of the scan.  lastoffset (all the scan needs) does not depend on the
            // extension results, so the emission may run on the consumer side (see greedy_emit_pipelined).
            if (pos == kPosUnknown) pos = tab.fetch_pos(last_read);
            sink(scan, pos);
            lastoffset = pos - scan;
            // the match that ended the scan opens the next piece: new[scan .. scan+len) == old[pos .. pos+len)
            if constexpr (Table::kExactMatches)
                if (scan < newLen && len >= kCertMin) certified(scan, len);
        } else if constexpr (Table::kExactMatches) {
            // no stop: all len bytes of this match agree at the current alignment, the piece goes on behind it
            if (len >= kCertMin) certified(scan, len);
        }
    }
}

inline void reset_streams(Streams &out, int32_t newLen)
{
    out.ctrl.clear();
    out.diff.clear();
    out.extra.clear();
    out.visits = 0;
    out.diff.reserve((size_t)newLen);  // sum of lenf <= newLen: the diffed ranges of `new` are disjoint
}

// single-producer single-consumer hand-off between the stages of greedy_emit_pipelined
template <typename T, int kSlots = 1024> class Handoff {
    T slot_[kSlots];
    std::atomic<uint32_t> head_{0}, tail_{0};
    std::atomic<bool> closed_{false};
    static void idle(int &spins) { wait_step(spins, 64); }

public:
    void push(const T &v)
    {
        const uint32_t t = tail_.load(std::memory_order_relaxed);
        int spins = 0;
        while (t - head_.load(std::memory_order_acquire) >= (uint32_t)kSlots) idle(spins);
        slot_[t % kSlots] = v;
        tail_.store(t + 1, std::memory_order_release);
    }
    void close() { closed_.store(true, std::memory_order_release); }
    // false once the queue is closed and drained
    bool pop(T &v)
    {
        const uint32_t h = head_.load(std::memory_order_relaxed);
        int spins = 0;
        for (;;) {
            if (tail_.load(std::memory_order_acquire) != h) break;
            if (closed_.load(std::memory_order_acquire)) {
                if (tail_.load(std::memory_order_acquire) != h) break;
                return false;
            }
            idle(spins);
        }
        v = slot_[h % kSlots];
        head_.store(h + 1, std::memory_order_release);
        return true;
    }
};

// how many host threads greedy_emit_pipelined may use besides the caller's
struct PipelineShape {
    int crew_helpers;  // extra walkers for long extensions
    int writers;       // threads producing diff/extra bytes
    // DQ_HOST_THREADS="helpers,writers" overrides the choice (tests run every shape on whatever cores there are)
    static PipelineShape for_this_machine()
    {
        if (const char *e = std::getenv("DQ_HOST_THREADS")) {
            int h = 0, w = 1, part = 0, mn = 0;
            const int got = std::sscanf(e, "%d,%d,%d,%d", &h, &w, &part, &mn);
            if (got >= 4 && part > 0 && mn > 0) {
                crew_part() = std::min(part, 1 << 20) << 10;   // KiB values: clamped so the shifts cannot overflow
                crew_min() = std::min(mn, 1 << 20) << 10;
            }
            if (got >= 1) return PipelineShape{std::max(0, std::min(h, 64)), std::max(1, std::min(w, 64))};
        }
        unsigned hw = std::thread::hardware_concurrency();
#if defined(__linux__)
        {   // the CPUs this process may actually run on (containers, taskset), not the machine's
            cpu_set_t set;
            if (sched_getaffinity(0, sizeof set, &set) == 0) {
                const unsigned allowed = (unsigned)CPU_COUNT(&set);
                if (allowed && allowed < hw) hw = allowed;
            }
        }
#endif
        // Few cores (one process per GPU sharing a host: 4 cores per rank on an 8-GPU box with 32) get no helpers: with
        // {2,1} on 4 cores the end-to-end step of eight concurrent ranks went from 13.7 to 24.1 ms (oversubscription
        // while the scan still polls the device); measured, bench.py under torchrun, N=8
        if (hw >= 12) return PipelineShape{3, 2};
        if (hw >= 6) return PipelineShape{1, 2};
        return PipelineShape{0, 1};
    }
};

// One job of a writer thread: dst[i] = n[i] - o[i] (o != nullptr, Diff.cs:197-200), dst[i] = n[i] (extra bytes,
// Diff.cs:202-207), or dst[i] = 0 (n == nullptr: a certified stretch of the piece).  dst ranges of different jobs are
// disjoint.
struct WriteJob {
    const uint8_t *n, *o;
    uint8_t *dst;
    int32_t len;
};
inline void run_write_job(const WriteJob &j)
{
    if (!j.n) {  // a certified stretch: new == old there, the diff bytes are zeros
        std::memset(j.dst, 0, (size_t)j.len);
        return;
    }
    if (!j.o) {
        std::memcpy(j.dst, j.n, (size_t)j.len);
        return;
    }
    int32_t i = 0;
#if defined(__SSE2__)
    for (; i + 16 <= j.len; i += 16)
        _mm_storeu_si128(reinterpret_cast<__m128i *>(j.dst + i),
                         _mm_sub_epi8(_mm_loadu_si128(reinterpret_cast<const __m128i *>(j.n + i)),
                                      _mm_loadu_si128(reinterpret_cast<const __m128i *>(j.o + i))));
#endif
    for (; i < j.len; i++) j.dst[i] = (uint8_t)(j.n[i] - j.o[i]);
}

// The loop on several host threads.  The caller runs the scan (it may block on table slices still in flight from
// the device); every stop goes to an extender thread, which does the extensions -- the only part that chains from
// stop to stop -- with a crew of helpers for the long ones, appends the control triple, and hands the byte ranges
// to writer threads at output offsets it has already fixed.  The scan needs only lastoffset = pos - scan from a
// stop, never the extension results, and the writers feed nothing back, so all sides compute exactly what the
// single-threaded loop computes and every output byte lands where that loop would put it.
template <typename Table, typename Ready>
inline void greedy_emit_pipelined(const uint8_t *oldData, int32_t oldLen, const uint8_t *newData, int32_t newLen,
                                  Table &tab, Streams &out, Ready &&ready,
                                  PipelineShape shape = PipelineShape::for_this_machine())
{
    reset_streams(out, newLen);
    out.extra.reserve((size_t)newLen);  // like diff: disjoint ranges of new; no reallocation under the writers
    struct Stop {  // certified == false: a stop (scan, pos); true: a certified stretch (start, len) of the piece being scanned
        int32_t scan, pos;
        bool certified;
    };
    constexpr int32_t kJobBytes = 256 << 10;
    const bool check_certs = std::getenv("DQ_CHECK_CERTS") != nullptr;  // tests: compare every certified stretch
    const int W = std::max(1, std::min(shape.writers, 4));
    const auto t_loop = std::chrono::steady_clock::now();
    out.extender_busy_ms = out.writer_busy_ms = 0;
    out.cert_errors = out.cert_bytes = 0;
    auto stops = std::make_unique<Handoff<Stop>>();
    std::vector<std::unique_ptr<Handoff<WriteJob>>> jobs;
    for (int w = 0; w < W; ++w) jobs.push_back(std::make_unique<Handoff<WriteJob>>());
    std::vector<std::thread> writers;
    for (int w = 0; w < W; ++w)
        writers.emplace_back([&, w]() {
            WriteJob j;
            while (jobs[w]->pop(j)) run_write_job(j);
        });
    std::thread extender([&]() {
        Crew crew(std::max(0, std::min(shape.crew_helpers, 15)));
        EmitState st;
        Stop sp;
        size_t diff_at = 0, extra_at = 0;
        int next_writer = 0;
        auto hand_out = [&](const uint8_t *n, const uint8_t *o, uint8_t *dst, int32_t len) {
            for (int32_t k = 0; k < len; k += kJobBytes) {
                jobs[next_writer]->push(WriteJob{n ? n + k : nullptr, o ? o + k : nullptr, dst + k, std::min(kJobBytes, len - k)});
                next_writer = (next_writer + 1) % W;
            }
        };
        std::vector<Cert> certs;  // of the piece that the next stop ends
        while (stops->pop(sp)) {
            if (sp.certified) {
                if (check_certs) {
                    const int64_t o = (int64_t)sp.scan - st.lastscan + st.lastpos;
                    if (o < 0 || o + sp.pos > oldLen || (int64_t)sp.scan + sp.pos > newLen ||
                        std::memcmp(newData + sp.scan, oldData + o, (size_t)sp.pos) != 0)
                        out.cert_errors++;
                }
                out.cert_bytes += sp.pos;
                certs.push_back(Cert{sp.scan, sp.pos});
                continue;
            }
            const auto t_a = std::chrono::steady_clock::now();
            const Piece pc = extend_stop(oldData, oldLen, newData, newLen, sp.scan, sp.pos, st, &crew, certs.data(), certs.size());
            out.extender_busy_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_a).count();
            if (pc.lenf > 0) {
                // diff bytes of [lastscan, lastscan + lenf): zeros over the certified stretches, new - old between them
                uint8_t *dst = out.diff.p.get() + diff_at;
                int32_t at = 0;  // offset into the piece
                for (const Cert &c : certs) {
                    const int32_t cb = (int32_t)std::min<int64_t>(pc.lenf, std::max<int64_t>(at, (int64_t)c.start - pc.lastscan));
                    const int32_t ce = (int32_t)std::min<int64_t>(pc.lenf, std::max<int64_t>(cb, (int64_t)c.start + c.len - pc.lastscan));
                    if (ce - cb < kZeroJobMin) continue;  // short ones stay inside the subtraction around them
                    if (cb > at) hand_out(newData + pc.lastscan + at, oldData + pc.lastpos + at, dst + at, cb - at);
                    hand_out(nullptr, nullptr, dst + cb, ce - cb);
                    at = ce;
                }
                if (pc.lenf > at) hand_out(newData + pc.lastscan + at, oldData + pc.lastpos + at, dst + at, pc.lenf - at);
                diff_at += (size_t)pc.lenf;
            }
            certs.clear();
            if (pc.extra > 0) {
                hand_out(newData + pc.lastscan + pc.lenf, nullptr, out.extra.p.get() + extra_at, pc.extra);
                extra_at += (size_t)pc.extra;
            }
            put_packed_long(out.ctrl, pc.lenf);
            put_packed_long(out.ctrl, pc.extra);
            put_packed_long(out.ctrl, pc.seek);
        }
        out.diff.len = diff_at;
        out.extra.len = extra_at;
        out.extender_done_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_loop).count();
        for (auto &q : jobs) q->close();
    });
    Streams scan_side;  // the scan only counts visits; keep its counter off the other threads' Streams
    auto finish = [&]() {
        stops->close();
        extender.join();
        for (auto &t : writers) t.join();
    };
    try {
        greedy_scan(oldData, oldLen, newData, newLen, tab, scan_side, ready,
                    [&](int32_t scan, int32_t pos) { stops->push(Stop{scan, pos, false}); },
                    [&](int32_t start, int32_t len) { stops->push(Stop{start, len, true}); });
    } catch (...) {
        finish();
        throw;
    }
    const double scan_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_loop).count();
    finish();
    out.visits = scan_side.visits;
    out.scan_done_ms = scan_ms;
    if (out.cert_errors) throw std::runtime_error("greedy loop: a certified stretch of new differs from old");
}

}  // namespace diffhost
}  // namespace dq
