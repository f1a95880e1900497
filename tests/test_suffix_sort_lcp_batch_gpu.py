"""sort_many(texts, lcp=...) / dq_cuda_suffix_sort_lcp_batch on the GPU: the emulator's cases at full size, then batches
of the sizes a caller that indexes a tree of files hands over.  Every per-text LCP array against Kasai, or against the
loop the batch replaces: dq_cuda_suffix_sort, then dq_cuda_lcp with I = NULL, text by text."""
import numpy as np
import pytest

import oracle
from batch_cases import exe_like_slices, fixture_batch, mixed_batch
from batch_lcp_cases import (boundary_batches, check_against_oracle, check_against_single_calls, check_argument_errors,
                             check_leaves_nothing_resident, check_python_overloads, repeat_batch, sort_many_lcp)
from conftest import random_bytes
from resident_cases import SETUPS, SHARD_MIN

pytestmark = pytest.mark.gpu

MIB = 1 << 20


@pytest.fixture(scope="module")
def sorter():
    from deltaq_b200 import CudaSuffixSort
    s = CudaSuffixSort()
    yield s
    s.dispose()


def _mixed_sizes(count, max_len, seed):
    rng = np.random.default_rng(seed)
    sizes = np.exp(rng.uniform(np.log(16), np.log(max_len), count)).astype(np.int64)
    return [rng.integers(0, 256, int(n), dtype=np.uint8) if i % 2 else rng.integers(0, 4, int(n), dtype=np.uint8)
            for i, n in enumerate(sizes)]


def test_mixed_batch(sorter):
    check_against_oracle(sorter, mixed_batch())


def test_all_fixtures_in_one_batch(sorter):
    texts, golden = fixture_batch()
    check_against_oracle(sorter, texts, golden)


@pytest.mark.parametrize("name", sorted(boundary_batches()))
def test_texts_that_match_across_their_boundaries(sorter, name):
    check_against_oracle(sorter, boundary_batches()[name])


def test_long_repeats_in_chunk_texts(sorter):
    """64 KiB blocks repeated to just below 2 MiB, in one chunk beside short texts: about 20 doubling rounds, so the
    seed level of the LCP walks runs, and the repeat continues across a text boundary at odd offsets."""
    texts = repeat_batch(64 * 1024, 31)
    assert max(t.size for t in texts) < 2 * MIB
    check_against_oracle(sorter, texts)
    assert sorter.stats()["rounds"] >= 14


@pytest.mark.parametrize("chunk,single_min", [("700", None), (None, "100"), ("300", "2000")])
def test_chunking_and_single_text_routing(sorter, monkeypatch, chunk, single_min):
    if chunk is not None:
        monkeypatch.setenv("DQ_BATCH_CHUNK", chunk)
    if single_min is not None:
        monkeypatch.setenv("DQ_BATCH_SINGLE_MIN", single_min)
    check_against_oracle(sorter, mixed_batch()[:14] + boundary_batches()["duplicates_between_others"])


def test_two_thousand_mixed_texts_up_to_1_mib(sorter):
    """2,000 texts of 16 B .. 1 MiB (log-uniform, half over four byte values), one call, against the single calls; every
    50th text also against the oracle and Kasai."""
    texts = _mixed_sizes(2000, MIB, seed=31)
    sas, lcps = sort_many_lcp(sorter, texts)
    check_against_single_calls(sorter, texts, sas, lcps)
    for i in range(0, len(texts), 50):
        ref = oracle.sais(texts[i])
        assert np.array_equal(sas[i], ref) and np.array_equal(lcps[i], oracle.lcp_array(texts[i], ref)), i


def test_more_texts_than_one_chunk_holds(sorter):
    """70,000 tiny texts: more than the 65,536 texts a chunk holds."""
    rng = np.random.default_rng(41)
    sizes = rng.integers(0, 12, 70_000)
    data = rng.integers(0, 3, int(sizes.sum()), dtype=np.uint8)
    offsets = np.zeros(sizes.size + 1, np.int64)
    np.cumsum(sizes, out=offsets[1:])
    texts = [data[offsets[i]:offsets[i + 1]] for i in range(sizes.size)]
    sas, lcps = sort_many_lcp(sorter, texts)
    for i, t in enumerate(texts):
        ref = np.array(sorted(range(t.size), key=lambda j: t[j:].tobytes()), np.int32)
        assert np.array_equal(sas[i], ref) and np.array_equal(lcps[i], oracle.lcp_array(t, ref)), i


def test_exe_like_slices(sorter):
    """Slices of an executable-like text: zero runs, which end and start many texts."""
    texts = exe_like_slices(300, MIB)
    sas, lcps = sort_many_lcp(sorter, texts)
    check_against_single_calls(sorter, texts, sas, lcps)
    for i in range(0, len(texts), 30):
        ref = oracle.sais(texts[i])
        assert np.array_equal(lcps[i], oracle.lcp_array(texts[i], ref)), i


def test_pinned_and_pageable_output(sorter):
    texts = _mixed_sizes(200, 256 * 1024, seed=7)
    total = sum(t.size for t in texts)
    sas, lcps = sort_many_lcp(sorter, texts)
    pinned = sorter.context.pinned(2 * total + 2, np.int32)
    try:
        pinned.array[:] = -7
        sorter.sort_many(texts, pinned.array[:total], pinned.array[total + 1:2 * total + 1])
        assert pinned.array[total] == -7 and pinned.array[2 * total + 1] == -7
        assert np.array_equal(pinned.array[:total], np.concatenate(sas))
        assert np.array_equal(pinned.array[total + 1:2 * total + 1], np.concatenate(lcps))
    finally:
        pinned.free()


def test_empty_batches_and_one_text(sorter):
    assert [a.size for a in sort_many_lcp(sorter, [b"", np.zeros(0, np.uint8)])[1]] == [0, 0]
    t = random_bytes(100_000, seed=4)
    _, lcps = sort_many_lcp(sorter, [t])
    sorter.sort(t, np.empty(t.size, np.int32))
    assert np.array_equal(lcps[0], sorter.lcp_array(t))


def test_argument_errors(sorter):
    check_argument_errors(sorter.context)


def test_python_overloads(sorter):
    check_python_overloads(sorter)


@pytest.mark.parametrize("single_min", [None, 1000], ids=["chunk", "alone"])
@pytest.mark.parametrize("setup", sorted(SETUPS))
@pytest.mark.parametrize("group", [False, True], ids=["single", "group"])
def test_leaves_nothing_resident(group, setup, single_min, monkeypatch):
    from deltaq_b200._native import Context
    if group:
        monkeypatch.setenv("DQ_SHARD_MIN", SHARD_MIN)
    with Context(device=[0, 0, 0] if group else 0) as ctx:
        check_leaves_nothing_resident(ctx, setup, single_min, monkeypatch)


def test_group_context_with_a_text_for_the_group_sort(monkeypatch):
    """A device group of logical shards of the first GPU; the 1 MiB text is sorted by all shards and its LCP array built
    from the group's index, while the others go through a chunk on the group's own device."""
    from deltaq_b200 import CudaSuffixSort
    monkeypatch.setenv("DQ_SHARD_MIN", str(512 * 1024))
    monkeypatch.setenv("DQ_BATCH_SINGLE_MIN", str(512 * 1024))
    texts = mixed_batch() + [random_bytes(MIB, seed=12)] + exe_like_slices(20, 64 * 1024)
    with CudaSuffixSort(device=[0, 0, 0]) as grp:
        check_against_oracle(grp, texts)
