"""Batches for CudaSuffixSort.sort_many(texts, lcp=...) (dq_cuda_suffix_sort_lcp_batch), shared by the emulator and GPU
tests.  Every text's suffix array must equal the oracle's (or the golden one), and its LCP array must equal Kasai's
(oracle.lcp_array) for that text alone.

A chunk holds its texts back to back with no separator byte, so a comparison that is not stopped at the end of its own
text runs on into the next one.  Most batches here are built so that it would then find more equal bytes: duplicates,
prefixes and suffixes of one another, zero tails before zero heads, and long repeats that continue across a text
boundary."""
import numpy as np
import pytest

import oracle
import resident_cases
from batch_cases import edge_batches


def boundary_batches():
    """edge_batches(), and batches whose texts continue matching into the text that follows them."""
    rng = np.random.default_rng(23)
    t = rng.integers(0, 256, 500, dtype=np.uint8)
    low = rng.integers(0, 2, 300, dtype=np.uint8)
    out = dict(edge_batches())
    out["text_then_same_text"] = [t, t]
    out["low_text_repeated"] = [low, low, low[:77], low, low[5:]]
    zeros_around = []
    for k in (1, 2, 7, 8, 31, 33, 64, 100):
        zeros_around.append(np.concatenate([t[:k], np.zeros(k + 3, np.uint8)]))   # ends in zeros ...
        zeros_around.append(np.concatenate([np.zeros(k, np.uint8), low[:k]]))    # ... starts with zeros
    out["zero_tails_then_zero_heads"] = zeros_around
    return out


def repeat_batch(block, reps, seed=29):
    """Long repeats inside chunk texts, which take the seed and head inheritance of the LCP walks: `block` random bytes
    repeated `reps` times (just below reps * block bytes), beside short texts.  The two copies of the repeat are laid
    out so that it continues across a text boundary and across the 32-position chunks of the walks at odd offsets."""
    rng = np.random.default_rng(seed)
    b = rng.integers(0, 256, block, dtype=np.uint8)
    rep = np.tile(b, reps)[:-13]
    shorts = [rng.integers(0, 256, int(n), dtype=np.uint8) for n in (5, 37, 300, 1000)]
    return [shorts[0], np.concatenate([shorts[1], rep]), np.concatenate([rep, shorts[2]]), shorts[3],
            rep[:block * 3 + 17], rep[1:], shorts[1]]


def sort_many_lcp(sorter, texts):
    """sort_many(texts, lcp=True) as per-text copies of the suffix and LCP arrays; the owner's layout checked."""
    with sorter.sort_many(texts, lcp=True) as owner:
        total = int(owner.offsets[-1])
        assert owner.memory.size == owner.lcp_memory.size == total
        assert len(owner.arrays) == len(owner.lcp_arrays) == len(texts)
        return [a.copy() for a in owner.arrays], [a.copy() for a in owner.lcp_arrays]


def check_against_oracle(sorter, texts, expected=None):
    """Both overloads against the oracle (or the given suffix arrays) and Kasai, with a guard entry after both flat
    outputs; returns the per-text (suffix arrays, LCP arrays)."""
    sas, lcps = sort_many_lcp(sorter, texts)
    expected = expected if expected is not None else [oracle.sais(t) for t in texts]
    kasai = [oracle.lcp_array(t, e) for t, e in zip(texts, expected)]
    for i, t in enumerate(texts):
        assert np.array_equal(sas[i], expected[i]), f"suffix array of text {i} (length {t.size})"
        assert np.array_equal(lcps[i], kasai[i]), f"LCP array of text {i} (length {t.size})"
    total = sum(t.size for t in texts)
    sa_flat = np.full(total + 1, -7, dtype=np.int32)
    lcp_flat = np.full(total + 1, -7, dtype=np.int32)
    sorter.sort_many(texts, sa_flat[:total], lcp_flat[:total])
    assert sa_flat[total] == -7 and lcp_flat[total] == -7
    if texts:
        assert np.array_equal(sa_flat[:total], np.concatenate(expected))
        assert np.array_equal(lcp_flat[:total], np.concatenate(kasai))
    return sas, lcps


def check_against_single_calls(sorter, texts, got_sa, got_lcp):
    """Each text alone through dq_cuda_suffix_sort, then dq_cuda_lcp with I = NULL: the loop the batch replaces."""
    bad = []
    for i, t in enumerate(texts):
        sa = np.empty(t.size, np.int32)
        sorter.sort(t, sa)
        lcp = sorter.lcp_array(t) if t.size else np.zeros(0, np.int32)
        if not (np.array_equal(got_sa[i], sa) and np.array_equal(got_lcp[i], lcp)):
            bad.append(i)
    assert bad == []


def raw_lcp_batch(ctx, data, offsets, count, sa_out, lcp_out):
    import ctypes
    ptr = lambda a: None if a is None else ctypes.c_void_p(a.ctypes.data)  # noqa: E731
    return ctx.lib.L.dq_cuda_suffix_sort_lcp_batch(ctx._h, ptr(data), ptr(offsets), count, ptr(sa_out), ptr(lcp_out))


def raw_batch(ctx, data, offsets, count, sa_out):
    import ctypes
    ptr = lambda a: None if a is None else ctypes.c_void_p(a.ctypes.data)  # noqa: E731
    return ctx.lib.L.dq_cuda_suffix_sort_batch(ctx._h, ptr(data), ptr(offsets), count, ptr(sa_out))


def check_argument_errors(ctx):
    """Every argument error of dq_cuda_suffix_sort_batch gives the same status here, and a null lcp_out with a non-zero
    total is one more; nothing is written."""
    from deltaq_b200 import _native
    data = np.random.default_rng(3).integers(0, 256, 10, dtype=np.uint8)
    sa = np.full(11, -7, np.int32)
    lcp = np.full(11, -7, np.int32)
    cases = [
        (data, np.array([0, 10], np.int32), -1, sa),                # count < 0
        (data, np.array([1, 10], np.int32), 1, sa),                 # offsets[0] != 0
        (data, np.array([0, 6, 4, 10], np.int32), 3, sa),           # decreasing offsets
        (None, np.array([0, 10], np.int32), 1, sa),                 # null texts
        (data, np.array([0, 10], np.int32), 1, None),               # null sa_out
        (data, None, 1, sa),                                        # null offsets
        (None, np.array([0, 0, 0], np.int32), 2, None),             # zero total
        (None, None, 0, None),                                      # count == 0
    ]
    for d, o, c, s in cases:
        want = raw_batch(ctx, d, o, c, s)
        assert raw_lcp_batch(ctx, d, o, c, s, lcp if s is not None else None) == want, (c, o)
    assert raw_lcp_batch(ctx, data, np.array([0, 10], np.int32), 1, sa, None) == _native.DQ_ERR_INVALID_ARGUMENT
    assert ctx.lib.L.dq_cuda_last_error(ctx._h).startswith(b"dq_cuda_suffix_sort_lcp_batch: null buffer")
    assert raw_lcp_batch(ctx, None, np.array([0, 0], np.int32), 1, None, None) == _native.DQ_OK
    assert np.all(sa == -7) and np.all(lcp == -7)


def check_python_overloads(sorter):
    """sort_many's lcp argument: True only without suffixes, an int32 array of the total length with them."""
    from deltaq_b200.suffix_sort import LENGTH_MISMATCH
    data = np.random.default_rng(4).integers(0, 256, 10, dtype=np.uint8)
    with sorter.sort_many([data, data]) as owner:
        assert owner.lcp_arrays is None and owner.lcp_memory is None
    with sorter.sort_many([], lcp=True) as owner:
        assert owner.arrays == [] and owner.lcp_arrays == [] and owner.lcp_memory.size == 0
    sa = np.zeros(20, np.int32)
    with pytest.raises(ValueError, match=LENGTH_MISMATCH):
        sorter.sort_many([data, data], sa, np.zeros(19, np.int32))
    with pytest.raises(TypeError):
        sorter.sort_many([data, data], sa, True)
    with pytest.raises(TypeError):
        sorter.sort_many([data, data], sa, np.zeros(20, np.int64))
    with pytest.raises(TypeError):
        sorter.sort_many([data, data], lcp=np.zeros(20, np.int32))
    lcp = np.full(20, -7, np.int32)
    assert sorter.sort_many([data, data], sa, lcp) is None
    assert np.array_equal(lcp[10:], oracle.lcp_array(data, oracle.sais(data)))


# ---- the resident rule (include/deltaq_cuda.h, "the resident index"), in the style of resident_cases.py ---------------
def check_leaves_nothing_resident(ctx, setup, single_min, monkeypatch):
    """`setup` makes old1 resident; one LCP batch of old2[:100] and old2 (old2 sorted on its own when single_min is
    set: on a group with DQ_SHARD_MIN below its length, by the group) must give the oracle's arrays and leave nothing
    resident, so a search and an LCP array of old2 with I = NULL both fail afterwards."""
    from deltaq_b200._native import NativeError
    old1, old2, new = resident_cases.texts()
    resident_cases.SETUPS[setup](ctx, old1, new)
    if single_min is not None:
        monkeypatch.setenv("DQ_BATCH_SINGLE_MIN", str(single_min))
    data = np.concatenate([old2[:100], old2])
    offsets = np.array([0, 100, data.size], np.int32)
    sa, lcp = np.empty(data.size, np.int32), np.empty(data.size, np.int32)
    ctx.suffix_sort_lcp_batch(data, offsets, sa, lcp)
    for t, lo, hi in ((old2[:100], 0, 100), (old2, 100, data.size)):
        ref = oracle.sais(t)
        assert np.array_equal(sa[lo:hi], ref) and np.array_equal(lcp[lo:hi], oracle.lcp_array(t, ref))
    with pytest.raises(NativeError, match="no suffix array of this length is resident"):
        resident_cases.search(ctx, old2, None, new, new.size)
    with pytest.raises(NativeError, match="no suffix array of this length is resident"):
        ctx.lcp(old2)
