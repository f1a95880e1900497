"""sort_many(texts, lcp=...) / dq_cuda_suffix_sort_lcp_batch on the CPU logic emulator (tests/emu; NOT the product, NOT
a fallback -- see tests/emu/cuda_emu.h): suffix and LCP arrays of many texts in one call, every per-text LCP array
against Kasai on the oracle's suffix array.  The same cases run on the B200 in test_suffix_sort_lcp_batch_gpu.py."""
import numpy as np
import pytest

from batch_cases import exe_like_slices, fixture_batch, mixed_batch
from batch_lcp_cases import (boundary_batches, check_against_oracle, check_argument_errors, check_leaves_nothing_resident,
                             check_python_overloads, repeat_batch, sort_many_lcp)
from conftest import random_bytes
from resident_cases import SETUPS, SHARD_MIN


@pytest.fixture(scope="module")
def sorter():
    from deltaq_b200 import CudaSuffixSort
    import emu
    s = CudaSuffixSort(_lib=emu.library())
    yield s
    s.dispose()


def test_mixed_batch(sorter):
    check_against_oracle(sorter, mixed_batch())


def test_all_fixtures_in_one_batch(sorter):
    texts, golden = fixture_batch()
    check_against_oracle(sorter, texts, golden)


@pytest.mark.parametrize("name", sorted(boundary_batches()))
def test_texts_that_match_across_their_boundaries(sorter, name):
    check_against_oracle(sorter, boundary_batches()[name])


def test_exe_like_slices(sorter):
    check_against_oracle(sorter, exe_like_slices(12, 3000))


@pytest.mark.parametrize("seeds", [None, "1", "8"])
def test_long_repeats_in_chunk_texts(sorter, monkeypatch, seeds):
    """4 KiB blocks repeated to about 60 KB beside short texts: the head walks inherit inside the repeats, and with
    DQ_SEEDS_PER set the seed level runs as well (by default it runs from 14 doubling rounds up, as on the GPU case)."""
    if seeds is not None:
        monkeypatch.setenv("DQ_SEEDS_PER", seeds)
    check_against_oracle(sorter, repeat_batch(4096, 15))


@pytest.mark.parametrize("chunk,single_min", [("1", None), ("700", None), ("5000", None), (None, "1"), (None, "100"),
                                               ("300", "2000")])
def test_chunking_and_single_text_routing(sorter, monkeypatch, chunk, single_min):
    """Small DQ_BATCH_CHUNK: many chunks; small DQ_BATCH_SINGLE_MIN: texts sorted on their own, whose LCP arrays are
    level 0 of dq_cuda_lcp's index.  Neither changes a result."""
    if chunk is not None:
        monkeypatch.setenv("DQ_BATCH_CHUNK", chunk)
    if single_min is not None:
        monkeypatch.setenv("DQ_BATCH_SINGLE_MIN", single_min)
    texts = mixed_batch()[:14] + boundary_batches()["duplicates_between_others"] + boundary_batches()["empties_between"]
    check_against_oracle(sorter, texts)


def test_empty_batches_and_one_text(sorter):
    assert [a.size for a in sort_many_lcp(sorter, [b"", np.zeros(0, np.uint8)])[1]] == [0, 0]
    t = random_bytes(777, seed=4)
    sas, lcps = sort_many_lcp(sorter, [t])
    sorter.sort(t, np.empty(t.size, np.int32))
    assert np.array_equal(lcps[0], sorter.lcp_array(t))


def test_stats_describe_the_whole_call(sorter, monkeypatch):
    """Launches summed over the chunks and the texts sorted alone, the LCP steps included; rounds the largest count."""
    monkeypatch.setenv("DQ_BATCH_SINGLE_MIN", "4000")
    texts = [random_bytes(300, seed=1), np.zeros(5000, np.uint8), random_bytes(200, seed=2)]
    sorter.sort_many(texts, np.empty(5500, np.int32))
    plain = sorter.stats()
    sort_many_lcp(sorter, texts)
    st = sorter.stats()
    assert st["n"] == 5500 and st["rounds"] == plain["rounds"]
    assert st["kernel_launches"] > plain["kernel_launches"]


def test_argument_errors(sorter):
    check_argument_errors(sorter.context)


def test_python_overloads(sorter):
    check_python_overloads(sorter)


@pytest.mark.parametrize("single_min", [None, 1000], ids=["chunk", "alone"])
@pytest.mark.parametrize("setup", sorted(SETUPS))
@pytest.mark.parametrize("group", [False, True], ids=["single", "group"])
def test_leaves_nothing_resident(group, setup, single_min, monkeypatch):
    import emu
    from deltaq_b200._native import Context
    if group:
        monkeypatch.setenv("DQ_SHARD_MIN", SHARD_MIN)
    with Context(device=[0, 0, 0] if group else None, lib=emu.library()) as ctx:
        check_leaves_nothing_resident(ctx, setup, single_min, monkeypatch)


@pytest.mark.parametrize("shard_min", [None, "2000"])
def test_group_context(monkeypatch, shard_min):
    """A device group of logical shards: chunks on its own device; with DQ_SHARD_MIN and DQ_BATCH_SINGLE_MIN lowered a
    text goes through the group sort and its LCP array comes from the group's index."""
    import emu
    from deltaq_b200 import CudaSuffixSort
    if shard_min is not None:
        monkeypatch.setenv("DQ_SHARD_MIN", shard_min)
        monkeypatch.setenv("DQ_BATCH_SINGLE_MIN", shard_min)
    with CudaSuffixSort(device=[0, 0, 0], _lib=emu.library()) as grp:
        check_against_oracle(grp, mixed_batch())
