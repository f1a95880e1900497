"""bsdiff.search_many / dq_cuda_bsdiff_search_batch on the CPU logic emulator (tests/emu; NOT the product, NOT a fallback
-- see tests/emu/cuda_emu.h): the (pos, len) tables of many pairs in one call, every pair against oracle.search_table
and against its own sort + search.  The same cases run on the B200 in test_bsdiff_search_batch_gpu.py."""
import numpy as np
import pytest

import batch_search_cases as bsc
from resident_cases import SHARD_MIN


@pytest.fixture(scope="module")
def sorter():
    from deltaq_b200 import CudaSuffixSort
    import emu
    s = CudaSuffixSort(_lib=emu.library())
    yield s
    s.dispose()


@pytest.mark.parametrize("name", ["leaf", "leak", "inheritance"])
def test_pairs_against_oracle_and_single_calls(sorter, name):
    pairs = {"leaf": bsc.leaf_pairs, "leak": bsc.leak_pairs, "inheritance": bsc.inheritance_pairs}[name]()
    bsc.check_pairs(sorter.context, pairs)


def test_file_tree(sorter):
    bsc.check_pairs(sorter.context, bsc.tree_pairs(60, 3000))


def test_empty_batch(sorter):
    assert bsc.search_batch(sorter.context, []) == []
    from deltaq_b200.bsdiff import search_many
    assert search_many([], sorter) == []


@pytest.mark.parametrize("chunk,single_min", [("1", None), ("3000", None), (None, "1"), ("4000", "500")],
                         ids=["chunk_per_pair", "many_chunks", "all_alone", "mixed"])
def test_routing(sorter, monkeypatch, chunk, single_min):
    """Small DQ_BATCH_CHUNK: many chunks, and news larger than a chunk searched alone; small DQ_BATCH_SINGLE_MIN: pairs
    sorted and searched on their own.  Neither changes a result."""
    if chunk is not None:
        monkeypatch.setenv("DQ_BATCH_CHUNK", chunk)
    if single_min is not None:
        monkeypatch.setenv("DQ_BATCH_SINGLE_MIN", single_min)
    bsc.check_pairs(sorter.context, bsc.routing_pairs(), singles=False)


def test_device_group(monkeypatch):
    """Three logical shards with a small DQ_SHARD_MIN: pairs searched alone take the group sort and search, chunks run
    on devices[0]."""
    import emu
    from deltaq_b200._native import Context
    monkeypatch.setenv("DQ_SHARD_MIN", SHARD_MIN)
    monkeypatch.setenv("DQ_BATCH_SINGLE_MIN", SHARD_MIN)
    with Context(device=[0, 0, 0], lib=emu.library()) as ctx:
        pairs = bsc.tree_pairs(12, 6000, seed=59) + bsc.leak_pairs()[:4]
        assert any(o.size >= int(SHARD_MIN) and w.size >= int(SHARD_MIN) for o, w in pairs)
        bsc.check_pairs(ctx, pairs)


def test_argument_errors(sorter):
    bsc.check_argument_errors(sorter.context)


@pytest.mark.parametrize("single_min", [None, 1000], ids=["chunk", "alone"])
def test_leaves_nothing_resident(single_min, monkeypatch):
    import emu
    with emu.context() as ctx:
        bsc.check_leaves_nothing_resident(ctx, single_min, monkeypatch)


def test_stats_describe_the_whole_call(sorter, monkeypatch):
    bsc.check_stats(sorter.context, monkeypatch)


def test_create_many(sorter):
    pairs = bsc.tree_pairs(6, 4000, seed=61) + [(np.zeros(0, np.uint8), np.arange(50, dtype=np.uint8)),
                                                (np.arange(50, dtype=np.uint8), np.zeros(0, np.uint8))]
    bsc.check_create_many(sorter, pairs, patch_apply=False)  # Patch.apply loads the product library


def test_search_many_views(sorter):
    """search_many returns per-pair views of one flat buffer, equal to search_all for each pair."""
    from deltaq_b200.bsdiff import search_all, search_many
    pairs = bsc.tree_pairs(5, 2000, seed=67)
    got = search_many(pairs, sorter)
    base = got[0][0].base
    assert base is not None and all(p.base is base and ln.base is got[0][1].base for p, ln in got)
    for (o, w), (p, ln) in zip(pairs, got):
        rp, rl = search_all(o, w, sorter)
        assert np.array_equal(p, rp) and np.array_equal(ln, rl)
    with pytest.raises(TypeError):
        search_many(pairs, object())
