"""Which text a context keeps resident after each kind of call (include/deltaq_cuda.h, "the resident index"), shared by
the emulator and the GPU tests.

Every case starts on a fresh context that has made `old1` resident (a sort, or a whole diff), makes one call with a
second text `old2` of the same length, and then searches and builds the LCP array with I = NULL.  Both answers must be
the oracle's for the text the header says the call left resident, and both must fail with "no suffix array of this
length is resident" where it says the call leaves none.  On a device group whose shard threshold is below n, the
calls that overwrite `old1` on the group's own device alone must drop the group's sharded index of it as well."""
import numpy as np
import pytest

import oracle

N, M = 20_000, 21_000
SHARD_MIN = "2000"   # DQ_SHARD_MIN of the group cases: below N, above the short searches' count
SHORT = 100          # scan positions of a search that stays on the group's own device


def texts():
    """old1, old2 (executable-like, equal lengths, different bytes) and a `new` made from old2."""
    from deltaq_b200 import workloads as w
    old2, new = w.c2_exe_pair(N, M, seed_old=3, seed_new=4)
    old1, _ = w.c2_exe_pair(N, M, seed_old=5, seed_new=6)
    return old1, old2, new


def search(ctx, old, I, new, count):
    pos, ln = np.empty(count, np.int32), np.empty(count, np.int32)
    ctx.bsdiff_search(old, I, new, 0, count, pos, ln)
    return pos, ln


# ---- how old1 becomes resident -----------------------------------------------------------------------------------
SETUPS = {
    "suffix_sort": lambda ctx, old1, new: ctx.suffix_sort(old1, np.empty(old1.size, np.int32)),
    "bsdiff_streams": lambda ctx, old1, new: ctx.bsdiff_streams(old1, new),
}


# ---- the calls: each gets (ctx, mem, old2, its suffix array, new, monkeypatch) and checks its own result ------------
def _suffix_sort(ctx, mem, t, sa, new, mp):
    out = np.empty(t.size, np.int32)
    ctx.suffix_sort(t, out)
    assert np.array_equal(out, sa)


def _suffix_sort_device(ctx, mem, t, sa, new, mp):
    d_t, d_sa = mem.put(t), mem.put(np.zeros(t.size, np.int32))
    ctx.suffix_sort_device(mem.ptr(d_t), t.size, mem.ptr(d_sa))
    assert np.array_equal(mem.get(d_sa), sa)


def _batch(single_min):
    def call(ctx, mem, t, sa, new, mp):
        if single_min is not None:
            mp.setenv("DQ_BATCH_SINGLE_MIN", str(single_min))
        data = np.concatenate([t[:100], t])
        offsets = np.array([0, 100, data.size], np.int32)
        out = np.empty(data.size, np.int32)
        ctx.suffix_sort_batch(data, offsets, out)
        assert np.array_equal(out[100:], sa) and np.array_equal(out[:100], oracle.sais(t[:100]))
    return call


def _bsdiff_streams(m):
    def call(ctx, mem, t, sa, new, mp):
        got = ctx.bsdiff_streams(t, new[:m])
        ref = oracle.bsdiff_streams(t, new[:m], oracle.make_I(sa))
        assert all(got[k] == ref[k] for k in ("ctrl", "diff", "extra"))
    return call


def _bsdiff_search(count):
    def call(ctx, mem, t, sa, new, mp):
        I = oracle.make_I(sa)
        pos, ln = search(ctx, t, I, new, count)
        rp, rl = oracle.search_all(I, t, new, 0, count)
        assert np.array_equal(pos, rp) and np.array_equal(ln, rl)
    return call


def _lcp(ctx, mem, t, sa, new, mp):
    assert np.array_equal(ctx.lcp(t, sa), oracle.lcp_array(t, sa))


RADIX_COUNT = 3 * 4096 + 7


def _radix_keys():
    return np.random.default_rng(9).integers(0, 2**63, RADIX_COUNT, dtype=np.uint64)


def _radix_sort_pairs(ctx, mem, t, sa, new, mp):
    keys, vals = _radix_keys(), np.arange(RADIX_COUNT, dtype=np.uint32)
    ctx.radix_sort_pairs(keys, vals)
    assert np.array_equal(keys, np.sort(_radix_keys()))


def _radix_sort_pairs_device(ctx, mem, t, sa, new, mp):
    kbuf, vbuf = mem.put(_radix_keys()), mem.put(np.arange(RADIX_COUNT, dtype=np.uint32))
    ctx.radix_sort_pairs_device(mem.ptr(kbuf), mem.ptr(vbuf), RADIX_COUNT, 0, 64)
    assert np.array_equal(mem.get(kbuf), np.sort(_radix_keys()))


# name -> (call, the text it leaves resident: "old2", "old1" (untouched) or None)
CALLS = {
    "suffix_sort": (_suffix_sort, "old2"),
    "suffix_sort_device": (_suffix_sort_device, "old2"),
    "suffix_sort_batch": (_batch(None), None),
    "suffix_sort_batch_text_alone": (_batch(1000), None),   # old2 sorted on its own (by the group, on a group)
    "bsdiff_streams": (_bsdiff_streams(M), "old2"),
    "bsdiff_streams_empty_new": (_bsdiff_streams(0), "old2"),
    "bsdiff_search_caller_I_short": (_bsdiff_search(SHORT), "old2"),
    "bsdiff_search_caller_I_all": (_bsdiff_search(M), "old2"),
    "lcp_caller_I": (_lcp, "old2"),
    "radix_sort_pairs": (_radix_sort_pairs, "old1"),
    "radix_sort_pairs_device": (_radix_sort_pairs_device, "old1"),
}


def check_call(ctx, mem, setup, name, monkeypatch):
    """`setup` makes old1 resident, call `name` runs with old2, then the search and LCP array with I = NULL."""
    from deltaq_b200._native import NativeError
    old1, old2, new = texts()
    SETUPS[setup](ctx, old1, new)
    call, leaves = CALLS[name]
    sa2 = oracle.sais(old2)
    call(ctx, mem, old2, sa2, new, monkeypatch)
    if leaves is None:
        with pytest.raises(NativeError, match="no suffix array of this length is resident"):
            search(ctx, old2, None, new, new.size)
        with pytest.raises(NativeError, match="no suffix array of this length is resident"):
            ctx.lcp(old2)
        return
    text, sa = (old2, sa2) if leaves == "old2" else (old1, oracle.sais(old1))
    pos, ln = search(ctx, text, None, new, new.size)
    rp, rl = oracle.search_all(oracle.make_I(sa), text, new)
    bad = np.flatnonzero((pos != rp) | (ln != rl))
    assert bad.size == 0, f"{bad.size} positions differ from the oracle's for {leaves}, first at scan {bad[:1]}"
    assert np.array_equal(ctx.lcp(text), oracle.lcp_array(text, sa))
