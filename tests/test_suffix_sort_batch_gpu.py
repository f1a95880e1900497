"""sort_many / dq_cuda_suffix_sort_batch on the GPU: the emulator's cases at full speed, then batches of the sizes a
caller that sorts a tree of files hands over, every per-text array against dq_cuda_suffix_sort or the oracle."""
import numpy as np
import pytest

import oracle
from batch_cases import check_against_oracle, edge_batches, exe_like_slices, fixture_batch, mixed_batch, sort_many
from conftest import random_bytes

pytestmark = pytest.mark.gpu

MIB = 1 << 20


@pytest.fixture(scope="module")
def sorter():
    from deltaq_b200 import CudaSuffixSort
    s = CudaSuffixSort()
    yield s
    s.dispose()


def _looped(sorter, texts):
    out = []
    for t in texts:
        sa = np.empty(t.size, np.int32)
        sorter.sort(t, sa)
        out.append(sa)
    return out


def _mixed_sizes(count, max_len, seed):
    rng = np.random.default_rng(seed)
    sizes = np.exp(rng.uniform(np.log(16), np.log(max_len), count)).astype(np.int64)
    return [rng.integers(0, 256, int(n), dtype=np.uint8) if i % 2 else rng.integers(0, 4, int(n), dtype=np.uint8)
            for i, n in enumerate(sizes)]


def test_mixed_batch(sorter):
    texts = mixed_batch()
    check_against_oracle(sorter, texts)
    assert sorter.stats()["n"] == sum(t.size for t in texts)


def test_all_fixtures_in_one_batch(sorter):
    texts, golden = fixture_batch()
    check_against_oracle(sorter, texts, golden)


@pytest.mark.parametrize("name", sorted(edge_batches()))
def test_edge_batches(sorter, name):
    check_against_oracle(sorter, edge_batches()[name])


def test_empty_batches_and_one_text(sorter):
    with sorter.sort_many([]) as owner:
        assert owner.memory.size == 0 and owner.arrays == []
    assert [a.size for a in sort_many(sorter, [b"", np.zeros(0, np.uint8)])] == [0, 0]
    t = random_bytes(100_000, seed=4)
    with sorter.sort(t) as one:
        assert np.array_equal(sort_many(sorter, [t])[0], one.memory)


@pytest.mark.parametrize("chunk,single_min", [("700", None), (None, "100"), ("300", "2000")])
def test_chunking_and_single_text_routing(sorter, monkeypatch, chunk, single_min):
    if chunk is not None:
        monkeypatch.setenv("DQ_BATCH_CHUNK", chunk)
    if single_min is not None:
        monkeypatch.setenv("DQ_BATCH_SINGLE_MIN", single_min)
    check_against_oracle(sorter, mixed_batch()[:14] + edge_batches()["duplicates_between_others"])


def test_two_thousand_mixed_texts_up_to_1_mib(sorter):
    """2,000 texts of 16 B .. 1 MiB (log-uniform, half over four byte values), one call, against dq_cuda_suffix_sort
    text by text; every 50th text also against the oracle."""
    texts = _mixed_sizes(2000, MIB, seed=31)
    got = sort_many(sorter, texts)
    ref = _looped(sorter, texts)
    bad = [i for i, (g, r) in enumerate(zip(got, ref)) if not np.array_equal(g, r)]
    assert bad == []
    for i in range(0, len(texts), 50):
        assert np.array_equal(got[i], oracle.sais(texts[i])), i


def test_more_texts_than_one_chunk_holds(sorter):
    """70,000 tiny texts: more than the 65,536 texts a chunk holds (the text id takes 16 bits of the round-0 key)."""
    rng = np.random.default_rng(41)
    sizes = rng.integers(0, 12, 70_000)
    data = rng.integers(0, 3, int(sizes.sum()), dtype=np.uint8)
    offsets = np.zeros(sizes.size + 1, np.int64)
    np.cumsum(sizes, out=offsets[1:])
    texts = [data[offsets[i]:offsets[i + 1]] for i in range(sizes.size)]
    got = sort_many(sorter, texts)
    for i, t in enumerate(texts):
        # suffixes of a tiny text: sort by bytes, a proper prefix first
        ref = sorted(range(t.size), key=lambda j: t[j:].tobytes())
        assert np.array_equal(got[i], ref), i


def test_exe_like_slices(sorter):
    """Slices of an executable-like text: zero runs, where plain doubling needs extra rounds."""
    texts = exe_like_slices(300, MIB)
    got = sort_many(sorter, texts)
    ref = _looped(sorter, texts)
    assert all(np.array_equal(g, r) for g, r in zip(got, ref))
    for i in range(0, len(texts), 30):
        assert np.array_equal(got[i], oracle.sais(texts[i])), i


def test_pinned_and_pageable_output(sorter):
    texts = _mixed_sizes(200, 256 * 1024, seed=7)
    total = sum(t.size for t in texts)
    ref = np.concatenate(_looped(sorter, texts))
    pageable = np.full(total + 1, -7, np.int32)
    sorter.sort_many(texts, pageable[:total])
    assert pageable[total] == -7 and np.array_equal(pageable[:total], ref)
    pinned = sorter.context.pinned(total + 1, np.int32)
    try:
        pinned.array[:] = -7
        sorter.sort_many(texts, pinned.array[:total])
        assert pinned.array[total] == -7 and np.array_equal(pinned.array[:total], ref)
    finally:
        pinned.free()


def test_nothing_stays_resident(sorter):
    from deltaq_b200 import _native
    ctx = sorter.context
    old = random_bytes(50_000, seed=8)
    new = old.copy()
    new[1000:1400] = 7
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


def test_group_context_with_a_text_for_the_group_sort(monkeypatch):
    """A device group (logical shards of the first GPU); DQ_SHARD_MIN and DQ_BATCH_SINGLE_MIN lowered so the 1 MiB text
    is sorted by all shards while the others go through a chunk on the group's own device."""
    from deltaq_b200 import CudaSuffixSort, _native
    monkeypatch.setenv("DQ_SHARD_MIN", str(512 * 1024))
    monkeypatch.setenv("DQ_BATCH_SINGLE_MIN", str(512 * 1024))
    texts = mixed_batch() + [random_bytes(MIB, seed=12)] + exe_like_slices(20, 64 * 1024)
    with CudaSuffixSort(device=[0, 0, 0]) as grp:
        got = sort_many(grp, texts)
        with pytest.raises(_native.NativeError):
            grp.lcp_array(texts[-21])
    for i, t in enumerate(texts):
        assert np.array_equal(got[i], oracle.sais(t)), i
