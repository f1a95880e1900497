"""bsdiff.search_many / dq_cuda_bsdiff_search_batch on the B200: the cases of test_emu_bsdiff_search_batch.py, every
pair against oracle.search_table and against its own sort + search, plus a batch of more than 65,536 pairs (two
chunks by count) and whole BSDIFF40 files through Diff.create_many."""
import numpy as np
import pytest

import batch_search_cases as bsc
from resident_cases import SHARD_MIN

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sorter():
    from deltaq_b200 import CudaSuffixSort
    s = CudaSuffixSort(device=0)
    yield s
    s.dispose()


@pytest.mark.parametrize("name", ["leaf", "leak", "inheritance"])
def test_pairs_against_oracle_and_single_calls(sorter, name):
    pairs = {"leaf": bsc.leaf_pairs, "leak": bsc.leak_pairs, "inheritance": bsc.inheritance_pairs}[name]()
    bsc.check_pairs(sorter.context, pairs)


def test_file_tree(sorter):
    bsc.check_pairs(sorter.context, bsc.tree_pairs(400, 16_000))


@pytest.mark.parametrize("chunk,single_min", [("1", None), ("3000", None), (None, "1"), ("4000", "500")],
                         ids=["chunk_per_pair", "many_chunks", "all_alone", "mixed"])
def test_routing(sorter, monkeypatch, chunk, single_min):
    if chunk is not None:
        monkeypatch.setenv("DQ_BATCH_CHUNK", chunk)
    if single_min is not None:
        monkeypatch.setenv("DQ_BATCH_SINGLE_MIN", single_min)
    bsc.check_pairs(sorter.context, bsc.routing_pairs(), singles=False)


def test_more_than_65536_pairs(sorter):
    """70,000 small pairs: two chunks by count, the second starting mid-batch."""
    rng = np.random.default_rng(71)
    base = rng.integers(0, 4, 4000, dtype=np.uint8)
    pairs = []
    for _ in range(70_000):
        a, n, m = int(rng.integers(0, 3000)), int(rng.integers(0, 12)), int(rng.integers(0, 12))
        pairs.append((base[a:a + n], base[a + int(rng.integers(0, 4)):][:m].copy()))
    bsc.check_pairs(sorter.context, pairs, singles=False)


def test_device_group(monkeypatch):
    from deltaq_b200._native import Context
    monkeypatch.setenv("DQ_SHARD_MIN", SHARD_MIN)
    monkeypatch.setenv("DQ_BATCH_SINGLE_MIN", SHARD_MIN)
    with Context(device=[0, 0, 0]) as ctx:
        pairs = bsc.tree_pairs(12, 6000, seed=59) + bsc.leak_pairs()[:4]
        assert any(o.size >= int(SHARD_MIN) and w.size >= int(SHARD_MIN) for o, w in pairs)
        bsc.check_pairs(ctx, pairs)


def test_argument_errors(sorter):
    bsc.check_argument_errors(sorter.context)


@pytest.mark.parametrize("single_min", [None, 1000], ids=["chunk", "alone"])
def test_leaves_nothing_resident(single_min, monkeypatch):
    from deltaq_b200._native import Context
    with Context(device=0) as ctx:
        bsc.check_leaves_nothing_resident(ctx, single_min, monkeypatch)


def test_stats_describe_the_whole_call(sorter, monkeypatch):
    bsc.check_stats(sorter.context, monkeypatch)


def test_create_many(sorter):
    pairs = bsc.tree_pairs(30, 20_000, seed=61) + [(np.zeros(0, np.uint8), np.arange(50, dtype=np.uint8)),
                                                   (np.arange(50, dtype=np.uint8), np.zeros(0, np.uint8))]
    bsc.check_create_many(sorter, pairs)
