"""sort_many / dq_cuda_suffix_sort_batch on the CPU logic emulator (tests/emu; NOT the product, NOT a fallback -- see
tests/emu/cuda_emu.h): many texts sorted together by one prefix doubling, every per-text array against the oracle."""
import ctypes

import numpy as np
import pytest

import oracle
from batch_cases import check_against_oracle, edge_batches, exe_like_slices, fixture_batch, mixed_batch, sort_many
from conftest import random_bytes


@pytest.fixture(scope="module")
def sorter():
    from deltaq_b200 import CudaSuffixSort
    import emu
    s = CudaSuffixSort(_lib=emu.library())
    yield s
    s.dispose()


def test_mixed_batch(sorter):
    texts = mixed_batch()
    check_against_oracle(sorter, texts)
    st = sorter.stats()
    assert st["n"] == sum(t.size for t in texts)
    assert st["rounds"] >= 2 and st["kernel_launches"] > 0


def test_all_fixtures_in_one_batch(sorter):
    texts, golden = fixture_batch()
    assert len(texts) == 13
    check_against_oracle(sorter, texts, golden)


@pytest.mark.parametrize("name", sorted(edge_batches()))
def test_edge_batches(sorter, name):
    check_against_oracle(sorter, edge_batches()[name])


def test_exe_like_slices(sorter):
    check_against_oracle(sorter, exe_like_slices(12, 3000))


def test_empty_batches_and_one_text(sorter):
    with sorter.sort_many([]) as owner:
        assert owner.memory.size == 0 and owner.arrays == [] and list(owner.offsets) == [0]
    assert sorter.sort_many([], np.zeros(0, np.int32)) is None
    assert sorter.stats()["n"] == 0
    got = sort_many(sorter, [b"", b"", np.zeros(0, np.uint8)])
    assert [a.size for a in got] == [0, 0, 0]
    t = random_bytes(777, seed=4)
    with sorter.sort(t) as one:
        assert np.array_equal(sort_many(sorter, [t])[0], one.memory)


@pytest.mark.parametrize("chunk,single_min", [("1", None), ("700", None), ("5000", None), (None, "1"), (None, "100"),
                                               ("300", "2000")])
def test_chunking_and_single_text_routing(sorter, monkeypatch, chunk, single_min):
    """DQ_BATCH_CHUNK small: many chunks (one text each at "1"); DQ_BATCH_SINGLE_MIN small: texts go one by one through
    the single-text path, interleaved with chunks of the shorter ones.  Neither changes a result."""
    if chunk is not None:
        monkeypatch.setenv("DQ_BATCH_CHUNK", chunk)
    if single_min is not None:
        monkeypatch.setenv("DQ_BATCH_SINGLE_MIN", single_min)
    texts = mixed_batch()[:14] + edge_batches()["duplicates_between_others"] + edge_batches()["empties_between"]
    check_against_oracle(sorter, texts)


def test_stats_describe_the_whole_call(sorter, monkeypatch):
    monkeypatch.setenv("DQ_BATCH_SINGLE_MIN", "4000")   # the all-zero text goes alone and needs the most rounds
    texts = [random_bytes(300, seed=1), np.zeros(5000, np.uint8), random_bytes(200, seed=2)]
    sort_many(sorter, texts)
    st = sorter.stats()
    sa = np.empty(5000, np.int32)
    sorter.sort(texts[1], sa)
    alone = sorter.stats()
    assert st["n"] == 5500
    assert st["rounds"] == max(alone["rounds"], 1) and st["kernel_launches"] > alone["kernel_launches"]


def _raw_batch(ctx, data, offsets, count, sa_out):
    ptr = lambda a: None if a is None else ctypes.c_void_p(a.ctypes.data)  # noqa: E731
    return ctx.lib.L.dq_cuda_suffix_sort_batch(ctx._h, ptr(data), ptr(offsets), count, ptr(sa_out))


def test_argument_errors(sorter):
    from deltaq_b200 import _native
    from deltaq_b200.suffix_sort import LENGTH_MISMATCH
    ctx = sorter.context
    data = random_bytes(10)
    sa = np.full(11, -7, np.int32)
    bad = _native.DQ_ERR_INVALID_ARGUMENT
    assert _raw_batch(ctx, data, np.array([0, 10], np.int32), -1, sa) == bad                # count < 0
    assert _raw_batch(ctx, data, np.array([1, 10], np.int32), 1, sa) == bad                 # offsets[0] != 0
    assert _raw_batch(ctx, data, np.array([0, 6, 4, 10], np.int32), 3, sa) == bad           # decreasing offsets
    assert _raw_batch(ctx, None, np.array([0, 10], np.int32), 1, sa) == bad                 # null texts
    assert _raw_batch(ctx, data, np.array([0, 10], np.int32), 1, None) == bad               # null sa_out
    assert _raw_batch(ctx, data, None, 1, sa) == bad                                        # null offsets
    assert np.all(sa == -7)
    assert _raw_batch(ctx, None, np.array([0, 0, 0], np.int32), 2, None) == _native.DQ_OK   # zero total
    assert _raw_batch(ctx, None, None, 0, None) == _native.DQ_OK                            # count == 0
    with pytest.raises(_native.NativeError):
        ctx.suffix_sort_batch(data, np.array([0, 6, 4, 10], np.int32), sa)
    with pytest.raises(ValueError, match=LENGTH_MISMATCH):
        sorter.sort_many([data, data], np.zeros(19, np.int32))
    with pytest.raises(TypeError):
        sorter.sort_many([data, None])
    with pytest.raises(TypeError):
        sorter.sort_many(None)
    assert np.all(sa == -7)


def test_nothing_stays_resident(sorter):
    """A batch overwrites the context's text, SA and ISA: a search or an LCP array with I = None fails after it, and a
    following sort makes the text resident again."""
    from deltaq_b200 import _native
    ctx = sorter.context
    old = random_bytes(3000, seed=8)
    new = old.copy()
    new[100:140] = 7
    pos, ln = np.empty(new.size, np.int32), np.empty(new.size, np.int32)
    sa = np.empty(old.size, np.int32)
    sorter.sort(old, sa)
    sort_many(sorter, [old, old[:100]])
    with pytest.raises(_native.NativeError, match="no suffix array of this length is resident"):
        ctx.bsdiff_search(old, None, new, 0, new.size, pos, ln)
    with pytest.raises(_native.NativeError, match="no suffix array of this length is resident"):
        ctx.lcp(old)
    sorter.sort(old, sa)
    ctx.bsdiff_search(old, None, new, 0, new.size, pos, ln)
    rp, rl = oracle.search_all(oracle.make_I(oracle.sais(old)), old, new)
    assert np.array_equal(pos, rp) and np.array_equal(ln, rl)
    assert np.array_equal(ctx.lcp(old), oracle.lcp_array(old, sa))


@pytest.mark.parametrize("shard_min", [None, "2000"])
def test_group_context(monkeypatch, shard_min):
    """A device group of logical shards sorts the batch on its own device; with DQ_SHARD_MIN and DQ_BATCH_SINGLE_MIN
    lowered a text goes through the group sort.  The same arrays either way, and nothing stays resident."""
    import emu
    from deltaq_b200 import CudaSuffixSort, _native
    if shard_min is not None:
        monkeypatch.setenv("DQ_SHARD_MIN", shard_min)
        monkeypatch.setenv("DQ_BATCH_SINGLE_MIN", shard_min)
    texts = mixed_batch()
    with CudaSuffixSort(device=[0, 0, 0], _lib=emu.library()) as grp:
        check_against_oracle(grp, texts)
        big = texts[10]   # 0x8000 random bytes
        grp.sort(big, np.empty(big.size, np.int32))
        sort_many(grp, [big])
        with pytest.raises(_native.NativeError):
            grp.lcp_array(big)


def test_timing_of_a_batch(sorter):
    """With timing on, the batch sums its pass figures into the stats, and the per-launch / per-round lists describe its
    last chunk."""
    ctx = sorter.context
    texts = [random_bytes(3000, seed=5), np.zeros(2000, np.uint8), random_bytes(10, seed=6)]
    ctx.set_timing(True)
    try:
        sort_many(sorter, texts)
        st = sorter.stats()
        rounds = ctx.round_times()
        passes = ctx.pass_times()
    finally:
        ctx.set_timing(False)
    assert len(rounds) == st["rounds"] and rounds[0][1] == sum(t.size for t in texts)
    assert len(passes) == st["radix_passes"] == sum(r[2] for r in rounds)
    assert st["pass_pairs"] == sum(p[1] for p in passes)
