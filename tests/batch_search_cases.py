"""Batches of (old, new) pairs for dq_cuda_bsdiff_search_batch (bsdiff.search_many, Diff.create_many), shared by the
emulator and GPU tests.  Every pair's (pos, len) table must equal oracle.search_table for that pair alone -- linear time,
no algorithm in common with the library -- and what dq_cuda_suffix_sort + dq_cuda_bsdiff_search (I = NULL) return for it.

A chunk holds its olds and its news back to back, so behind every pair lie the next pair's bytes, suffix array, ranks
and LCP entries.  Most batches here are built so that a comparison, walk or inheritance that is not stopped at the end
of its own pair finds more equal bytes there and gives a wrong answer: olds that repeat or continue the old before
them, news that hold the next pair's old, zero tails before zero heads, and matches that run to the last byte."""
import ctypes
import io

import numpy as np
import pytest

import oracle
from batch_cases import exe_like_slices
from batch_lcp_cases import boundary_batches, repeat_batch

GUARD = 3          # sentinel entries on both sides of every output buffer
SENTINEL = -7


def _flat(arrays):
    offsets = np.zeros(len(arrays) + 1, np.int32)
    np.cumsum([a.size for a in arrays], out=offsets[1:])
    flat = np.concatenate(arrays) if arrays else np.zeros(0, np.uint8)
    return np.ascontiguousarray(flat, dtype=np.uint8), offsets


def search_batch(ctx, pairs):
    """One dq_cuda_bsdiff_search_batch over `pairs` through Context.bsdiff_search_batch; the guards checked, the
    per-pair (pos, len) returned as copies."""
    olds, old_offsets = _flat([o for o, _ in pairs])
    news, new_offsets = _flat([w for _, w in pairs])
    total = int(new_offsets[-1])
    pos = np.full(total + 2 * GUARD, SENTINEL, np.int32)
    ln = np.full(total + 2 * GUARD, SENTINEL, np.int32)
    ctx.bsdiff_search_batch(olds, old_offsets, news, new_offsets, pos[GUARD:GUARD + total], ln[GUARD:GUARD + total])
    for a in (pos, ln):
        assert np.all(a[:GUARD] == SENTINEL) and np.all(a[GUARD + total:] == SENTINEL), "written outside the table"
    return [(pos[GUARD + b:GUARD + e].copy(), ln[GUARD + b:GUARD + e].copy())
            for b, e in zip(new_offsets[:-1], new_offsets[1:])]


def single_search(ctx, old, new):
    """The loop the batch replaces, for one pair: dq_cuda_suffix_sort, then dq_cuda_bsdiff_search with I = NULL."""
    ctx.suffix_sort(old, np.empty(old.size, np.int32))
    pos, ln = np.full(new.size, SENTINEL, np.int32), np.full(new.size, SENTINEL, np.int32)
    ctx.bsdiff_search(old, None, new, 0, new.size, pos, ln)
    return pos, ln


def check_pairs(ctx, pairs, singles=True):
    """The batch against the oracle at every position of every pair, then (singles) against the single-pair calls."""
    got = search_batch(ctx, pairs)
    bad = []
    for i, (o, w) in enumerate(pairs):
        ref = oracle.search_table(o, w)
        if not (np.array_equal(got[i][0], ref[0]) and np.array_equal(got[i][1], ref[1])):
            k = int(np.flatnonzero((got[i][0] != ref[0]) | (got[i][1] != ref[1]))[0])
            bad.append((i, o.size, w.size, k, (int(got[i][0][k]), int(got[i][1][k])), (int(ref[0][k]), int(ref[1][k]))))
    assert bad == [], f"{len(bad)} of {len(pairs)} pairs differ from the oracle; first (pair, n, m, scan, got, want): " \
                      f"{bad[0]}"
    if singles:
        for i, (o, w) in enumerate(pairs):
            pos, ln = single_search(ctx, o, w)
            assert np.array_equal(pos, got[i][0]) and np.array_equal(ln, got[i][1]), f"pair {i} differs from its single call"
    return got


# ---- batches ------------------------------------------------------------------------------------------------------
def _rng(seed):
    return np.random.default_rng(seed)


def leaf_pairs():
    """olds of 0, 1, 2 and 9 bytes against news of 0 to 20,000 bytes made of their own bytes, their neighbours' and
    zeros (the leaves L == 0, L == n and the I[n] == 0 quirk at every position), all-equal texts, empty news."""
    rng = _rng(41)
    olds = [np.zeros(0, np.uint8), np.array([7], np.uint8), np.array([7, 0], np.uint8),
            rng.integers(0, 3, 9, dtype=np.uint8)]
    pairs = []
    for o in olds:
        for m in (0, 1, 2, 3, 9, 33, 2049, 20_000):
            src = np.concatenate([o, np.array([0, 7, 1], np.uint8), o[::-1]]) if o.size else np.array([0, 7], np.uint8)
            pairs.append((o, src[rng.integers(0, src.size, m)].astype(np.uint8)))
    pairs.append((np.zeros(500, np.uint8), np.zeros(700, np.uint8)))
    pairs.append((np.full(300, 5, np.uint8), np.full(40, 5, np.uint8)))
    pairs.append((rng.integers(0, 256, 100, dtype=np.uint8), np.zeros(0, np.uint8)))
    pairs.append((np.zeros(64, np.uint8), np.zeros(64, np.uint8)))
    return pairs


def leak_pairs():
    """Pairs whose neighbours in the chunk continue their matches."""
    rng = _rng(43)
    t = rng.integers(0, 256, 3000, dtype=np.uint8)
    low = rng.integers(0, 2, 2000, dtype=np.uint8)
    pairs = []
    # old_{i+1} equals old_i, or continues it; new_i holds old_{i+1}'s bytes, so its best match lies in the wrong old
    olds = [t[:700], t[:700], t[700:1500], low[:300], low[300:900], low[:300]]
    for i, o in enumerate(olds):
        nxt = olds[(i + 1) % len(olds)]
        pairs.append((o, np.concatenate([o[100:200], nxt, o[-50:], nxt[:33]])))
    # zero tails before zero heads (the olds of batch_lcp_cases), news of zeros and of the next old
    zt = boundary_batches()["zero_tails_then_zero_heads"]
    for i, o in enumerate(zt):
        pairs.append((o, np.concatenate([np.zeros(40, np.uint8), zt[(i + 1) % len(zt)], o])))
    # news whose matches run to their own last byte, before a new that continues them
    for k in (1, 7, 8, 31, 64, 300):
        pairs.append((t[:1000], np.ascontiguousarray(t[1000 - k:1000])))
        pairs.append((t[:1000], np.ascontiguousarray(t[1000:1000 + k])))
        pairs.append((low[:500], np.ascontiguousarray(low[500 - k:500])))
    return pairs


def inheritance_pairs():
    """Identical pairs, news shifted by odd amounts, long repeats across the 32-position chains and 2048-position
    supers at odd offsets (repeat_batch), and news of 1, 31, 32, 33, 2047, 2048 and 2049 bytes."""
    rng = _rng(47)
    t = rng.integers(0, 256, 6000, dtype=np.uint8)
    pairs = [(t[:2500], t[:2500].copy()), (t[:33], t[:33].copy())]
    for s in (1, 3, 31, 33, 2047, 2049):
        pairs.append((t[:5000], np.concatenate([rng.integers(0, 256, s, dtype=np.uint8), t[:5000 - s]])))
    rep = repeat_batch(512, 12)
    for i, o in enumerate(rep):
        pairs.append((o, np.ascontiguousarray(rep[(i + 2) % len(rep)][::-1][:3000]) if i % 2 else o[5:].copy()))
    for m in (1, 31, 32, 33, 2047, 2048, 2049):
        pairs.append((t[1000:4000], np.ascontiguousarray(t[1500:1500 + m])))
    return pairs


def tree_pairs(count, max_len, seed=53):
    """A file tree: exe-like slices of 16 B .. max_len bytes, each against a mutated copy (sizes change a little)."""
    from deltaq_b200 import workloads
    rng = _rng(seed)
    olds = exe_like_slices(count, max_len, seed=seed)
    return [(o, workloads._mutate(o, rng, max(1, o.size + int(rng.integers(-8, 9))), regions=max(1, o.size // 512)))
            for o in olds]


def routing_pairs():
    return leaf_pairs()[::3] + leak_pairs()[::2] + inheritance_pairs()[:6]


# ---- whole files --------------------------------------------------------------------------------------------------
def check_create_many(sorter, pairs, patch_apply=True):
    """Diff.create_many: per pair the bytes of Diff.create, sections that Python's bz2 decodes to the oracle's
    uncompressed streams, and streams that the native add loop (and, with patch_apply, Patch.apply on the whole file)
    turn back into `new`."""
    import bz2
    from deltaq_b200.bsdiff import HEADER_SIZE, Diff, Patch, apply_streams, read_packed_long
    files = Diff.create_many(pairs, sorter)
    assert len(files) == len(pairs)
    for i, ((o, w), f) in enumerate(zip(pairs, files)):
        out = io.BytesIO()
        Diff.create(o, w, out, sorter)
        assert f == out.getvalue(), f"pair {i}: bytes differ from Diff.create"
        ctrl_len, diff_len = read_packed_long(f[8:16]), read_packed_long(f[16:24])
        sections = (f[HEADER_SIZE:HEADER_SIZE + ctrl_len], f[HEADER_SIZE + ctrl_len:HEADER_SIZE + ctrl_len + diff_len],
                    f[HEADER_SIZE + ctrl_len + diff_len:])
        ref = oracle.bsdiff_streams(o, w)
        streams = [bz2.decompress(sec) for sec in sections]
        assert streams == [ref["ctrl"], ref["diff"], ref["extra"]], f"pair {i}: streams differ from the oracle"
        assert apply_streams(o, *streams, w.size, lib=sorter.context.lib) == w.tobytes(), f"pair {i}: round trip"
        if patch_apply:
            back = io.BytesIO()
            Patch.apply(o, f, back)
            assert back.getvalue() == w.tobytes(), f"pair {i}: round trip of the file"


# ---- other behaviour ----------------------------------------------------------------------------------------------
def raw_search_batch(ctx, olds, old_offsets, news, new_offsets, count, pos, ln):
    ptr = lambda a: None if a is None else ctypes.c_void_p(a.ctypes.data)  # noqa: E731
    return ctx.lib.L.dq_cuda_bsdiff_search_batch(ctx._h, ptr(olds), ptr(old_offsets), ptr(news), ptr(new_offsets), count,
                                                 ptr(pos), ptr(ln))


def check_argument_errors(ctx):
    """The batch sort's argument errors on either offset array, and null buffers with a non-zero total: all
    DQ_ERR_INVALID_ARGUMENT with nothing written; count == 0 is a no-op."""
    from deltaq_b200 import _native
    d = _rng(3).integers(0, 256, 10, dtype=np.uint8)
    pos, ln = np.full(11, SENTINEL, np.int32), np.full(11, SENTINEL, np.int32)
    good = np.array([0, 4, 10], np.int32)
    bad_cases = [
        (d, good, d, good, -1, pos, ln),                                # count < 0
        (d, np.array([1, 4, 10], np.int32), d, good, 2, pos, ln),       # old offsets[0] != 0
        (d, good, d, np.array([1, 4, 10], np.int32), 2, pos, ln),       # new offsets[0] != 0
        (d, np.array([0, 6, 4], np.int32), d, good, 2, pos, ln),        # decreasing old offsets
        (d, good, d, np.array([0, 6, 4], np.int32), 2, pos, ln),        # decreasing new offsets
        (d, None, d, good, 2, pos, ln),                                 # null old offsets
        (d, good, d, None, 2, pos, ln),                                 # null new offsets
        (None, good, d, good, 2, pos, ln),                              # null olds
        (d, good, None, good, 2, pos, ln),                              # null news
        (d, good, d, good, 2, None, ln),                                # null pos_out
        (d, good, d, good, 2, pos, None),                               # null len_out
    ]
    for k, case in enumerate(bad_cases):
        assert raw_search_batch(ctx, *case) == _native.DQ_ERR_INVALID_ARGUMENT, k
        assert ctx.lib.L.dq_cuda_last_error(ctx._h).startswith(b"dq_cuda_bsdiff_search_batch: "), k
    zero = np.zeros(3, np.int32)
    assert raw_search_batch(ctx, None, None, None, None, 0, None, None) == _native.DQ_OK              # count == 0
    assert raw_search_batch(ctx, None, zero, None, zero, 2, None, None) == _native.DQ_OK              # zero totals
    assert raw_search_batch(ctx, None, zero, d, good, 2, pos, ln) == _native.DQ_OK                    # empty olds
    assert np.all(pos[10:] == SENTINEL) and np.array_equal(pos[:10], np.zeros(10, np.int32))
    assert np.array_equal(ln[:10], np.zeros(10, np.int32))


def check_leaves_nothing_resident(ctx, single_min, monkeypatch):
    """After a batch (a pair searched alone when single_min is set) a search and an LCP array with I = NULL fail."""
    import resident_cases
    from deltaq_b200._native import NativeError
    old1, old2, new = resident_cases.texts()
    ctx.suffix_sort(old1, np.empty(old1.size, np.int32))
    if single_min is not None:
        monkeypatch.setenv("DQ_BATCH_SINGLE_MIN", str(single_min))
    check_pairs(ctx, [(old2[:100], new[:300]), (old2, new)], singles=False)
    for old in (old1, old2):
        with pytest.raises(NativeError, match="no suffix array of this length is resident"):
            resident_cases.search(ctx, old, None, new, new.size)
        with pytest.raises(NativeError, match="no suffix array of this length is resident"):
            ctx.lcp(old)


def check_stats(ctx, monkeypatch):
    """n and search_queries are the totals; launches and times summed over the chunks and the pairs searched alone;
    rounds the largest count."""
    rng = _rng(5)
    big = np.zeros(5000, np.uint8)
    pairs = [(rng.integers(0, 256, 300, dtype=np.uint8), rng.integers(0, 256, 200, dtype=np.uint8)), (big, big[:700]),
             (rng.integers(0, 256, 200, dtype=np.uint8), rng.integers(0, 256, 900, dtype=np.uint8))]
    monkeypatch.setenv("DQ_BATCH_SINGLE_MIN", "4000")
    single_search(ctx, big, big[:700])
    alone = ctx.stats()
    check_pairs(ctx, pairs, singles=False)
    st = ctx.stats()
    assert st["n"] == 5500 and st["search_queries"] == 1800
    assert st["rounds"] >= alone["rounds"] and st["kernel_launches"] > alone["kernel_launches"]
    assert st["search_ms"] >= 0 and st["device_ms"] >= 0
