"""Checks of the match search against oracle.search_table at every scan position, shared by the emulator and the GPU
tests.  They drive a deltaq_b200._native.Context through its host entry points."""
import numpy as np


def assert_table(pos, ln, ref, what, b=0):
    rp, rl = ref[0][b:b + pos.size], ref[1][b:b + pos.size]
    bad = np.flatnonzero((pos != rp) | (ln != rl))
    assert bad.size == 0, (what, f"{bad.size} of {pos.size} positions differ; first at scan {b + int(bad[0])}: "
                                 f"({pos[bad[0]]}, {ln[bad[0]]}) vs ({rp[bad[0]]}, {rl[bad[0]]})")


def host_search(ctx, old, I, new, b=0, c=None):
    c = new.size - b if c is None else c
    pos, ln = np.full(c, -7, np.int32), np.full(c, -7, np.int32)
    ctx.bsdiff_search(old, I, new, b, c, pos, ln)
    assert ctx.stats()["search_queries"] == c
    return pos, ln


def launches(ctx):
    return ctx.stats()["kernel_launches"]


def one_repeated_byte_keys(t):
    """Suffixes whose first 8 bytes are one byte: the sort goes run-aware when they are at least n / 64."""
    v = np.lib.stride_tricks.sliding_window_view(t, 8)
    return int((v == v[:, :1]).all(axis=1).sum())


def sorted_and_searched(ctx, old, new, ref, sa_ref, lcp_ref, what, ranges=()):
    """Library sort, index build (through dq_cuda_lcp), whole search and sub-ranges with I = NULL, each checked.
    Returns (rounds, launches of the index build, launches of the whole search)."""
    sa = np.empty(old.size, np.int32)
    ctx.suffix_sort(old, sa)
    assert np.array_equal(sa, sa_ref), what
    rounds, l0 = ctx.stats()["rounds"], launches(ctx)
    lcp = ctx.lcp(old)
    l1 = launches(ctx)
    assert np.array_equal(lcp, lcp_ref), (what, "lcp before the search")
    pos, ln = host_search(ctx, old, None, new)
    l2 = launches(ctx)
    assert_table(pos, ln, ref, what)
    for b, c in ranges:
        pos, ln = host_search(ctx, old, None, new, b, c)
        assert_table(pos, ln, ref, (what, b, c), b)
    assert np.array_equal(ctx.lcp(old), lcp_ref), (what, "lcp after the search")
    return rounds, l1 - l0, l2 - l1
