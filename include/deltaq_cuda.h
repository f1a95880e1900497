/*
 * deltaq_cuda.h -- C ABI of libdeltaq_cuda, the B200 (sm_100a) suffix sorter and bsdiff match engine.
 *
 * The reference (jzebedee/deltaq, /root/reference) is 100 % managed C# and has NO native interface: the
 * plug-in point for this path is the managed interface
 *     DeltaQ.SuffixSorting.ISuffixSort        src/DeltaQ.SuffixSorting.Abstractions/ISuffixSort.cs:9-28
 * and the match search is the private method
 *     DeltaQ.BsDiff.Diff.Search               src/DeltaQ.BsDiff/Diff.cs:267-298
 * A new provider `DeltaQ.SuffixSorting.Cuda.CudaSuffixSort : ISuffixSort` (csharp/, INTEGRATION.md) binds
 * the entry points below through LibraryImport/P-Invoke; the same ABI is driven from Python ctypes
 * (deltaq_b200/_native.py) for every test and benchmark in this repository.
 *
 * Conventions: plain pointers and sizes; every function returns a status (0 = DQ_OK, negative = error
 * class) and never throws; the text of the last error of a context is dq_cuda_last_error(ctx).  A context
 * owns one device (or a device group, see dq_cuda_create), its streams and scratch memory; it serves one call at a time (calls on one context
 * are serialised by an internal lock); contexts are independent.
 */
#ifndef DELTAQ_CUDA_H
#define DELTAQ_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dq_ctx dq_ctx;

enum {
    DQ_OK = 0,
    DQ_ERR_INVALID_ARGUMENT = -1, /* maps to ArgumentException / ArgumentNullException */
    DQ_ERR_OUT_OF_MEMORY = -2,    /* maps to OutOfMemoryException */
    DQ_ERR_CUDA = -3,             /* maps to InvalidOperationException(dq_cuda_last_error) */
    DQ_ERR_NO_DEVICE = -4,        /* no CUDA device: there is NO CPU fallback */
    DQ_ERR_INTERNAL = -5,
    DQ_ERR_CORRUPT_PATCH = -6     /* maps to InvalidOperationException("Corrupt patch"), Patch.cs:68-70,128,151 */
};

/* Per-call statistics of the most recent dq_cuda_suffix_sort* / dq_cuda_bsdiff_search* on the context. */
typedef struct dq_stats {
    int32_t n;                 /* input length of the last sort */
    int32_t rounds;            /* doubling rounds run, round 0 included */
    int32_t radix_passes;      /* onesweep pass launches */
    int32_t kernel_launches;   /* all kernel launches of the call */
    int64_t active_sum;        /* sum over rounds of suffixes entering the round */
    int64_t algorithmic_bytes; /* SURVEY.md section 8(d) formula, summed over rounds (+4n output) */
    float   device_ms;         /* CUDA-event time of the device work of the last call (no host copies) */
    float   pass_ms;           /* CUDA-event time spent inside onesweep pass launches (0 unless timing on) */
    int64_t pass_pairs;        /* pairs moved by those launches (sum of per-launch counts) */
    int32_t search_queries;    /* positions answered by the last search */
    float   search_ms;         /* CUDA-event time of the last search's device work (LCP build included when it ran) */
    int32_t table_fallbacks;   /* dq_cuda_bsdiff_streams: 1 if the coded (pos,len) table overflowed and the full one was used */
    int32_t table_heads;       /* dq_cuda_bsdiff_streams: match heads in the coded table (12 B each over PCIe, + 1 B/position) */
    float   search_index_ms;   /* part of search_ms spent building the index of `old` (LCP array, block minima, bucket and
                                  prefix tables) before the first query kernel; 0 when the index was already resident */
} dq_stats;

/* Environment variables read by the library (tests and tuning only; none changes a result):
 *   DQ_TRACE=1            dq_cuda_bsdiff_streams prints its host/device timeline to stderr
 *   DQ_HOST_THREADS=h,w[,part_kib,min_kib]  helper walkers / writer threads of the host greedy loop
 *   DQ_HEADS_CAP=k        capacity of the match-head list of the coded (pos,len) table (forces the full-table fallback)
 *   DQ_SEEDS_PER=k        super-chunks per warp of the seed level of the search's head kernels (0 = off)
 *   DQ_PREFIX3=0|1        3-byte prefix table of the search: never / always built from the text (default: from 32 MiB up,
 *                         or from 1 MiB up out of the sort's round-0 keys once the context has searched;
 *                         DQ_PREFIX3_SORTED_MIN=n lowers that 1 MiB)
 *   DQ_SHARD_MIN=bytes    device groups (dq_cuda_create with ndev > 1): smallest input that is sharded (default 128 MiB)
 *   DQ_BATCH_SINGLE_MIN=bytes  dq_cuda_suffix_sort_batch, dq_cuda_bsdiff_search_batch: smallest text (old) sorted on its
 *                         own (default 2 MiB)
 *   DQ_BATCH_CHUNK=bytes  the same two: most bytes of texts (olds; news) that go together in one chunk (default 256 MiB)
 *   DQ_CHECK_CERTS=1      host greedy loop: compare every certified stretch byte for byte, fail the call on a false one
 *                         (set by the test suite)
 *   others (DQ_DIRECT_MAX, DQ_SUB_MIN_LOG, DQ_COMPACT_MIN, DQ_EARLY_COPY_MIN, DQ_GROUP_THREADS, DQ_HOST_INTERLEAVE):
 *   thresholds of the sort / device-group paths, DESIGN.md sections 4 and 6
 */

/* ---- context ------------------------------------------------------------------------------------ */

/* devices/ndev: CUDA ordinals to use; NULL/0 = current device.
 * ndev > 1 (at most 16) makes a device GROUP: this one context, in this one process, drives all listed GPUs
 * (peer access between them is required and enabled here).  Every entry point keeps its meaning; inputs of at
 * least DQ_SHARD_MIN bytes (default 128 MiB) are worked on by all GPUs of the group (DESIGN.md section 6):
 *   dq_cuda_suffix_sort*     one text sorted by all GPUs -- distributed prefix doubling; every exchange between GPUs
 *                            is a partition kernel that scatters straight into peer memory over NVLink;
 *   dq_cuda_bsdiff_search*   scan positions sharded by new-data range over the index replicated by peer copies;
 *   dq_cuda_bsdiff_streams   both of the above, then the host loop.
 * Smaller inputs run on devices[0] alone.  The same ordinal may be listed more than once (logical shards on one
 * GPU: how a single-GPU box exercises the group paths). */
int dq_cuda_create(dq_ctx **out, const int *devices, int ndev);
int dq_cuda_destroy(dq_ctx *ctx);
const char *dq_cuda_last_error(dq_ctx *ctx); /* ctx may be NULL: last error of a failed dq_cuda_create */
int dq_cuda_get_stats(dq_ctx *ctx, dq_stats *out);
/* when on, onesweep launches are bracketed by CUDA events (serialises nothing, costs two records/launch) */
int dq_cuda_set_timing(dq_ctx *ctx, int on);

/* Per-launch CUDA-event times of the onesweep passes of the last sort (timing must be on): fills up to `cap`
 * entries of ms[] / pairs[] / shift[] in launch order and returns the number of launches (or a negative status). */
int dq_cuda_get_pass_times(dq_ctx *ctx, float *ms, int64_t *pairs, int32_t *shift, int cap);

/* Per-round CUDA-event times of the last single-device sort (timing must be on), round 0 first: ms[] from the start
 * of the round to the start of the next (or the end of the sort), active[] = suffixes entering the round, passes[] =
 * radix passes it ran.  SURVEY.md section 8(d) algorithmic bytes of a round: active * (41 + 24 * passes) for round 0,
 * active * (52 + 24 * passes) after.  Returns the number of rounds (or a negative status). */
int dq_cuda_get_round_times(dq_ctx *ctx, float *ms, int64_t *active, int32_t *passes, int cap);

/* Pinned host buffers (the provider's IMemoryOwner<int> can sit on these: no staging copy on D2H). */
int dq_cuda_host_alloc(void **out, size_t bytes);
int dq_cuda_host_free(void *p);

/* ---- the resident index --------------------------------------------------------------------------------
 * A context keeps one text on the device between calls: its bytes, suffix array and inverse, and the search index
 * built from them (LCP levels, prefix tables), on a device group on every GPU.  dq_cuda_bsdiff_search*, dq_cuda_lcp*
 * with I_or_null == NULL use that text, and check only its LENGTH: n must equal the resident text's length, else the
 * call fails with DQ_ERR_INVALID_ARGUMENT ("no suffix array of this length is resident"); the bytes passed are not
 * compared with it.  Which text is resident:
 *   - dq_cuda_suffix_sort, dq_cuda_suffix_sort_device, dq_cuda_bsdiff_streams and dq_cuda_bsdiff_patch leave the
 *     text they sorted;
 *   - dq_cuda_bsdiff_search* and dq_cuda_lcp* with a caller's I leave that text under that I;
 *   - dq_cuda_suffix_sort_batch, dq_cuda_suffix_sort_lcp_batch and dq_cuda_bsdiff_search_batch leave none;
 *   - one of these that fails before its suffix array is complete leaves none;
 *   - the radix sorts, dq_cuda_greedy_emit, and the bzip2 and patch-apply calls leave the index untouched. */

/* ---- ISuffixSort.Sort ------------------------------------------------------------------------------
 * Replaces ISuffixSort.Sort(ReadOnlySpan<byte> text, Span<int> suffixes) (ISuffixSort.cs:27; reference
 * implementations LibDivSufSort.cs:21-31, SAIS.cs:25-42).  text and sa_out are HOST pointers; writes
 * exactly sa_out[0..n) (Diff.Create relies on I[n] staying 0: Diff.cs:78,90); n == 0 is a no-op; sa_out
 * need not be zeroed.  The "lengths must match" ArgumentException of LibDivSufSort.cs:23-31 is raised by
 * the managed/Python wrapper, which owns both lengths.  Leaves `text` resident (see "the resident index"). */
int dq_cuda_suffix_sort(dq_ctx *ctx, const uint8_t *text, int32_t n, int32_t *sa_out);

/* Same, with DEVICE pointers; runs on the context's stream and returns after the stream is idle. */
int dq_cuda_suffix_sort_device(dq_ctx *ctx, const uint8_t *d_text, int32_t n, int32_t *d_sa_out);

/* Sorts `count` texts in one call.  Text i is texts[offsets[i] .. offsets[i+1]); its suffix array (values in
 * [0, offsets[i+1]-offsets[i]), i.e. local to text i) is written to sa_out[offsets[i] .. offsets[i+1]).  Host pointers.
 * offsets has count+1 entries, offsets[0] == 0, non-decreasing.  Exactly sa_out[0 .. offsets[count]) is written.
 * Every per-text array equals what dq_cuda_suffix_sort returns for that text alone; empty texts write nothing and
 * count == 0 is a no-op (offsets may then be NULL).  DQ_ERR_INVALID_ARGUMENT, before any text byte is read, for
 * count < 0, offsets[0] != 0, decreasing offsets, or null pointers with a non-zero total.
 * Texts of at least DQ_BATCH_SINGLE_MIN bytes are sorted one by one as dq_cuda_suffix_sort sorts them (on a device group
 * that includes the group sort from DQ_SHARD_MIN up); all others go, in chunks of at most DQ_BATCH_CHUNK bytes and
 * 65,536 texts, through one prefix-doubling sort per chunk on the context's own device (devices[0]).  The call leaves
 * nothing resident (see "the resident index").  dq_stats describe the whole
 * call: n = offsets[count], kernel_launches, device_ms and pass_ms summed, rounds = the most any chunk or text needed;
 * with timing on, dq_cuda_get_pass_times / dq_cuda_get_round_times describe the batch's last chunk or single text. */
int dq_cuda_suffix_sort_batch(dq_ctx *ctx, const uint8_t *texts, const int32_t *offsets, int32_t count,
                              int32_t *sa_out);

/* dq_cuda_suffix_sort_batch, and the LCP array of every text as well: lcp_out[offsets[i] + r] is the length of the
 * longest common prefix of suffixes SA_i[r-1] and SA_i[r] of text i alone (0 for r == 0), so every per-text array equals
 * what dq_cuda_lcp returns for that text.  Exactly lcp_out[0 .. offsets[count]) is written (host pointer).  Arguments,
 * errors, sa_out, routing and dq_stats are those of dq_cuda_suffix_sort_batch; lcp_out is one more buffer that must not
 * be NULL with a non-zero total.  A chunk builds its LCP arrays before it is overwritten, with every comparison stopped
 * at the end of its text; a text sorted on its own gets level 0 of the index, as dq_cuda_lcp with I_or_null == NULL
 * builds it.  Like dq_cuda_suffix_sort_batch, the call leaves nothing resident (see "the resident index"). */
int dq_cuda_suffix_sort_lcp_batch(dq_ctx *ctx, const uint8_t *texts, const int32_t *offsets, int32_t count,
                                  int32_t *sa_out, int32_t *lcp_out);

/* ---- Diff.Search -----------------------------------------------------------------------------------
 * Replaces the per-position calls  len = Search(I, oldData, newData[scan..], 0, oldData.Length, out pos)
 * of Diff.Create (Diff.cs:106, Search at :267-298) for scan in [scan_begin, scan_begin+count):
 * pos_out[k], len_out[k] are bit-identical to what the reference computes at scan = scan_begin + k,
 * including the I[n] == 0 leaf quirk.  I_or_null: the (n+1)-entry buffer of Diff.cs:78 (entry n is
 * ignored and treated as 0; validated to be a permutation of [0, n)), which then becomes the resident index, or NULL
 * to use the resident index (see "the resident index").  All pointers are HOST pointers. */
int dq_cuda_bsdiff_search(dq_ctx *ctx, const uint8_t *old_, int32_t n, const int32_t *I_or_null,
                          const uint8_t *new_, int32_t m, int32_t scan_begin, int32_t count,
                          int32_t *pos_out, int32_t *len_out);

/* Same with DEVICE pointers (d_I_or_null: n entries are read). */
int dq_cuda_bsdiff_search_device(dq_ctx *ctx, const uint8_t *d_old, int32_t n, const int32_t *d_I_or_null,
                                 const uint8_t *d_new, int32_t m, int32_t scan_begin, int32_t count,
                                 int32_t *d_pos_out, int32_t *d_len_out);

/* The (pos, len) table of many pairs in one call: Diff.Create's sort and search for a tree of files.  Pair i is
 * old_i = olds[old_offsets[i] .. old_offsets[i+1]) and new_i = news[new_offsets[i] .. new_offsets[i+1]); both offset
 * arrays have count+1 entries, start at 0 and never decrease.  Host pointers.  pos_out[new_offsets[i] + k] and
 * len_out[...] for k in [0, m_i) equal what dq_cuda_suffix_sort(old_i) followed by dq_cuda_bsdiff_search(old_i, NULL,
 * new_i, 0, m_i) return for that pair alone (n_i == 0 and the I[n] == 0 leaf included).  Exactly
 * [0, new_offsets[count]) of both outputs is written; count == 0 is a no-op (the offsets may then be NULL).
 * DQ_ERR_INVALID_ARGUMENT, before any byte is read, for the argument errors of dq_cuda_suffix_sort_batch on either offset
 * array, or null buffers with a non-zero total (olds for the olds' total; news, pos_out, len_out for the news').
 * Routing is dq_cuda_suffix_sort_batch's: a pair whose old has at least DQ_BATCH_SINGLE_MIN bytes, or whose new alone
 * exceeds DQ_BATCH_CHUNK, is sorted and searched on its own (on a device group with the group paths from DQ_SHARD_MIN
 * up); the others go, in chunks of at most DQ_BATCH_CHUNK bytes of olds, as many of news and 65,536 pairs, through one
 * sort of the chunk's olds and one search of all its pairs on devices[0].  The call leaves nothing resident (see "the
 * resident index").  dq_stats describe the whole call: n = total old bytes, search_queries = total new positions,
 * kernel_launches, device_ms and search_ms summed, rounds = the most any chunk or single pair needed. */
int dq_cuda_bsdiff_search_batch(dq_ctx *ctx, const uint8_t *olds, const int32_t *old_offsets, const uint8_t *news,
                                const int32_t *new_offsets, int32_t count, int32_t *pos_out, int32_t *len_out);

/* ---- Diff.Create, hot path + consumer ---------------------------------------------------------------
 * Mirror of Diff.Create (Diff.cs:27-242) up to the compression boundary: suffix sort and match search on
 * the device, then the reference's greedy scan/extend/emit loop (Diff.cs:100-223, textually unchanged
 * except that Search() is an array read) on the host.  Returns the three UNCOMPRESSED streams the
 * reference feeds to its bzip2 encoders.  Buffers are owned by the context and valid until the next call
 * on it. */
typedef struct dq_diff_streams {
    const uint8_t *ctrl;  int64_t ctrl_len;   /* packed-long triples, SpanExtensions.cs:7-30 */
    const uint8_t *diff;  int64_t diff_len;
    const uint8_t *extra; int64_t extra_len;
    int64_t search_visits;                    /* scan positions the greedy loop evaluated */
} dq_diff_streams;
int dq_cuda_bsdiff_streams(dq_ctx *ctx, const uint8_t *old_, int32_t n, const uint8_t *new_, int32_t m,
                           dq_diff_streams *out);

/* The host consumer alone: Diff.cs:100-223 over a caller-supplied (pos, len) table (m entries each, e.g. from
 * dq_cuda_bsdiff_search).  Pure host code (a few threads: scan, extensions, stream writers); no device work. */
int dq_cuda_greedy_emit(dq_ctx *ctx, const uint8_t *old_, int32_t n, const uint8_t *new_, int32_t m,
                        const int32_t *pos_tab, const int32_t *len_tab, dq_diff_streams *out);

/* ---- LCP array (SURVEY.md 8(f) rank 4: "on-device LCP array as an ISuffixSort extension") ------------------
 * lcp_out[r] = length of the longest common prefix of the suffixes SA[r-1] and SA[r] of `text`, lcp_out[0] = 0; n
 * entries.  This is level 0 of the index every bulk search is anchored on (built along the text, Phi/PLCP order, then
 * permuted to rank order), so a following dq_cuda_bsdiff_search with I == NULL reuses it.  I_or_null as for
 * dq_cuda_bsdiff_search: NULL = the resident index (see "the resident index"), else n (or n+1) caller-supplied
 * entries, validated to be a permutation.  The reference has no LCP array (its
 * Search is a binary search over I, Diff.cs:267-298); checked against Kasai's algorithm in tests/. */
int dq_cuda_lcp(dq_ctx *ctx, const uint8_t *text, int32_t n, const int32_t *I_or_null, int32_t *lcp_out);
int dq_cuda_lcp_device(dq_ctx *ctx, const uint8_t *d_text, int32_t n, const int32_t *d_I_or_null, int32_t *d_lcp_out);

/* ---- the patch file: Diff.Create as a whole ------------------------------------------------------------
 * Replaces the three BZip2OutputStream sections of Diff.Create (Diff.cs:14-19, :85-87, :197-207, :226-241).
 * bzip2 blocks are independent, so every section is cut where a serial libbz2 would start its blocks, the pieces
 * are compressed on a crew of host threads by the system's libbz2 (dlopen'ed) and stitched bit by bit into ONE
 * ordinary stream: the bytes are identical to what serial libbz2 writes at that level, so any bzip2 reader
 * (Patch.cs:52-93) decodes them.  level 1..9 = bzip2's block size (9 = what `bzip2 -9` and Python's bz2 write);
 * 0 = per section, the largest level that still leaves about two blocks per thread (C2's diff section: level 1,
 * +0.5 % bytes, 10 pieces).  threads 0 = the CPUs the process may run on.  Pure host code, no context. */
int64_t dq_cuda_bz2_bound(int64_t n);  /* capacity a caller must offer for n input bytes */
/* `count` (<= 64) sections by one crew.  cap[s] >= dq_cuda_bz2_bound(len[s]).  info (may be NULL): 3 ints per section
 * = level used, blocks, 1 if the section had to be compressed serially (never observed; counted for the tests). */
int dq_cuda_bz2_compress(const uint8_t *const *src, const int64_t *len, int count, int level, int threads,
                         uint8_t *const *out, const int64_t *cap, int64_t *out_len, int32_t *info);
/* dq_cuda_bsdiff_streams + the header and the three sections: *patch is a complete BSDIFF40 file (Diff.cs:54-70:
 * "BSDIFF40", packed lengths of the ctrl and diff sections, packed size of newData; then ctrl, diff, extra), owned by
 * the context and valid until the next call on it. */
int dq_cuda_bsdiff_patch(dq_ctx *ctx, const uint8_t *old_, int32_t n, const uint8_t *new_, int32_t m, int level,
                         const uint8_t **patch, int64_t *patch_len);

/* ---- Patch.Apply on the patch FILE ---------------------------------------------------------------------
 * Patch.Apply (Patch.cs:25-50) = CreatePatchStreams (:52-93: header checks, three bzip2 sections) + ApplyInternal
 * (:95-168).  The sections are decoded block-parallel: the 48-bit block magic is located at every bit alignment,
 * each block is decoded by the system's libbz2 on a crew of host threads as a one-block stream of its own, the
 * combined CRC is checked against the stream's; anything unexpected falls back to the serial decoder.  Works on any
 * BSDIFF40 file (the reference's, bsdiff 4.x's, this library's).  *new_size is set from the header as soon as the
 * header is valid; out_cap < *new_size returns DQ_ERR_INVALID_ARGUMENT (call with out_cap 0 to ask for the size).
 * DQ_ERR_CORRUPT_PATCH where the reference throws "Corrupt patch", for damaged sections, and for a section that decodes
 * to more than a patch for *new_size bytes can use (diff, extra: new_size; ctrl: 24 per output byte; + 1 MiB each) --
 * the reference streams its sections and would never notice; here nothing is unpacked past that point.  Pure host code. */
int dq_cuda_bspatch(const uint8_t *old_, int64_t n, const uint8_t *patch, int64_t patch_len, int threads, uint8_t *out,
                    int64_t out_cap, int64_t *new_size);
/* One bzip2 stream, blocks decoded in parallel.  *out_len = decoded size (also when cap is too small, which returns
 * DQ_ERR_INVALID_ARGUMENT).  info (may be NULL): blocks found, 1 if the serial decoder had to take the stream. */
int dq_cuda_bz2_decompress(const uint8_t *src, int64_t len, int threads, uint8_t *out, int64_t cap, int64_t *out_len,
                           int32_t *info);

/* ---- Patch.Apply ------------------------------------------------------------------------------------
 * Patch.ApplyInternal (Patch.cs:95-168) on the three UNCOMPRESSED streams (the caller has un-bzip2'ed them, as
 * Patch.CreatePatchStreams :52-93 does): writes exactly new_size bytes to out.  Pure host code (the add loop of
 * Patch.cs:143-144, 16 bytes per step); needs no context.  Returns DQ_ERR_CORRUPT_PATCH where the reference throws
 * "Corrupt patch", and also for negative sizes, a short control stream, or reads past the end of old/diff/extra. */
int dq_cuda_patch_apply(const uint8_t *old_, int64_t n, const uint8_t *ctrl, int64_t ctrl_len, const uint8_t *diff,
                        int64_t diff_len, const uint8_t *extra, int64_t extra_len, uint8_t *out, int64_t new_size);

/* ---- building blocks, exported for tests and reuse -------------------------------------------------- */
/* Stable LSD radix sort of device-resident (uint64 key, uint32 value) pairs on key bits [bit_lo, bit_lo+nbits),
 * in place.  hist_out_host (may be NULL): 256 counters of the FIRST digit (bits [bit_lo, bit_lo+min(nbits,8))). */
int dq_cuda_radix_sort_pairs_device(dq_ctx *ctx, uint64_t *d_keys, uint32_t *d_vals, int32_t count, int32_t bit_lo,
                                    int32_t nbits, int64_t *hist_out_host);

/* Stable LSD radix sort of (uint64 key, uint32 value) pairs on key bits [0, key_bits), host pointers. */
int dq_cuda_radix_sort_pairs(dq_ctx *ctx, uint64_t *keys, uint32_t *vals, int32_t count, int32_t key_bits);

#ifdef __cplusplus
}
#endif
#endif /* DELTAQ_CUDA_H */
