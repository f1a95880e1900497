"""The suffix array's delivery into pinned memory (early copy and late patches) on one device and on device groups of
logical shards, and the per-round counts of round_times() against the oracle's LCP array -- on the CPU logic emulator
(tests/emu; NOT the product), at small sizes.  The same checks run on the B200 at bench.py's sizes in
test_sort_delivery_gpu.py; see sort_delivery_cases.py for what they prove.

On the emulator every host address is device-visible and every copy lands at once: the early copy starts for any
output buffer (the plain run turns it off with DQ_EARLY_COPY_MIN = 0), and whatever the late rounds resolve reaches the
host array only through the patch."""
import functools

import numpy as np
import pytest

import oracle
from conftest import random_bytes, small_alphabet_texts
from search_table_cases import one_repeated_byte_keys
from sort_delivery_cases import (Delivery, check_batch_rounds, check_early_copy, check_group_delivery,
                                 check_index_left_behind, check_plain_rounds, check_run_aware_rounds,
                                 check_sort_many_pinned, plain_rounds, tandem_repeats, zero_heavy)

DELIVERY = Delivery(copy_env={"DQ_EARLY_COPY_MIN": "1"}, plain_env={"DQ_EARLY_COPY_MIN": "0"})


@functools.lru_cache(maxsize=None)
def case(name):
    """-> (old, new or None, suffix array of old)."""
    from deltaq_b200 import workloads as w
    new = None
    if name == "c2_runs":            # an exe-like text whose zero section makes the sort run-aware
        old, new = w.c2_exe_pair(100_000, 104_000, seed_old=4)
    elif name == "c5":               # the C5 recipe, 8 pieces
        old, new = w.c5_pair(120_000, seed=11)
    elif name == "c3":
        old = w.c3_repetitive(100_000)    # the last round starts below n/8
    elif name == "c4":
        old = w.c4_genome(64_000)
    elif name == "tandem5":
        old = tandem_repeats(64_000, 0.05)
    elif name == "zero_heavy":
        old = zero_heavy(96_000, 2048)
    else:
        raise KeyError(name)
    return old, new, oracle.sais(old)


def group(shards):
    import emu
    from deltaq_b200._native import Context
    return Context(device=[0] * shards, lib=emu.library())


@pytest.fixture(scope="module")
def ctx():
    import emu
    from deltaq_b200._native import Context
    c = Context(lib=emu.library())
    yield c
    c.close()


# ---- A. early copy on one device ------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["c2_runs", "c3", "c4", "tandem5"])
def test_early_copy_one_device(ctx, name, monkeypatch):
    monkeypatch.setenv("DQ_COMPACT_MIN", "1")     # c4: recoded keys, as at bench.py's size
    old, _, sa = case(name)
    check_early_copy(ctx, DELIVERY, old, sa, name)


# ---- B. the group sort into pinned and pageable output --------------------------------------------------------------
@pytest.mark.parametrize("shards", [2, 3, 4, 8])
def test_group_run_aware(shards, monkeypatch):
    monkeypatch.setenv("DQ_SHARD_MIN", "4096")
    old, new, sa = case("c2_runs")
    assert one_repeated_byte_keys(old) * 64 >= old.size
    with group(shards) as g:
        check_group_delivery(g, DELIVERY, old, sa, ("c2_runs", shards))
        if shards == 3:
            check_index_left_behind(g, old, new, oracle.lcp_array(old, sa), oracle.search_table(old, new), "c2_runs")


@pytest.mark.parametrize("shards", [3, 8])
@pytest.mark.parametrize("direct_max", ["0", None])
def test_group_zero_heavy(shards, direct_max, monkeypatch):
    """The key of eight zero bytes holds more than 1/G of the suffixes: RunBucketPolicy spreads it over several
    buckets.  DQ_DIRECT_MAX = 0: round 0's ranks go to their owners through group_route_updates."""
    monkeypatch.setenv("DQ_SHARD_MIN", "4096")
    if direct_max is not None:
        monkeypatch.setenv("DQ_DIRECT_MAX", direct_max)
    old, _, sa = case("zero_heavy")
    assert np.count_nonzero(old == 0) >= 0.6 * old.size
    with group(shards) as g:
        check_group_delivery(g, DELIVERY, old, sa, ("zero_heavy", shards, direct_max))


def test_group_exchange_then_direct_rounds(monkeypatch):
    """4 shards: rounds above DQ_DIRECT_MAX go by request / reply exchanges, smaller ones by peer pointers; both kinds
    run after the copy started (the text's repeats keep a few per cent of it unresolved for many rounds), so both write
    late lists."""
    old, _, sa = case("tandem5")
    after = [a for a, _ in plain_rounds(old, sa, 8)[1:] if a <= old.size // 8]
    direct_max = after[len(after) // 2]
    assert any(a > direct_max for a in after) and len(after) >= 4, after
    monkeypatch.setenv("DQ_SHARD_MIN", "4096")
    monkeypatch.setenv("DQ_DIRECT_MAX", str(direct_max))
    with group(4) as g:
        check_group_delivery(g, DELIVERY, old, sa, "tandem5")


def test_group_c5_recipe(monkeypatch):
    monkeypatch.setenv("DQ_SHARD_MIN", "4096")
    old, new, sa = case("c5")
    with group(8) as g:
        check_group_delivery(g, DELIVERY, old, sa, "c5")
        check_index_left_behind(g, old, new, oracle.lcp_array(old, sa), oracle.search_table(old, new), "c5")


def test_sort_many_on_a_group(monkeypatch):
    """A batch whose exe-like text goes through the group sort, into the provider's pinned owner."""
    import emu
    from deltaq_b200 import CudaSuffixSort
    from deltaq_b200 import workloads as w
    monkeypatch.setenv("DQ_SHARD_MIN", "30000")
    monkeypatch.setenv("DQ_BATCH_SINGLE_MIN", "30000")
    big = case("c2_runs")[0]
    texts = [random_bytes(4097, seed=1), np.zeros(1000, np.uint8), random_bytes(4, seed=2), big, random_bytes(9000),
             np.zeros(0, np.uint8), small_alphabet_texts()["acgt_tandem"]]
    with CudaSuffixSort(device=[0, 0, 0], _lib=emu.library()) as sorter:
        check_sort_many_pinned(sorter, DELIVERY, texts, 3)


# ---- C. per-round counts against the oracle -------------------------------------------------------------------------
def _plain_cases():
    from deltaq_b200 import workloads as w
    rng = np.random.default_rng(8)
    sat = small_alphabet_texts()
    return {"c1": (w.c1_uniform(30_000), 8), "random_65537": (random_bytes(65537, seed=3), 8),
            "c3": (case("c3")[0], 8), "tandem5": (case("tandem5")[0], 8),
            "c4": (case("c4")[0], 32), "acgt_random": (np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, 50_000)], 32),
            "bin_70000": (sat["bin_70000"], 64), "hex16_30000": (sat["hex16_30000"], 16),
            "acgt_tandem": (sat["acgt_tandem"], 32)}


@pytest.mark.parametrize("name", sorted(_plain_cases()))
def test_round_counts_plain_doubling(ctx, name, monkeypatch):
    monkeypatch.setenv("DQ_COMPACT_MIN", "1")
    t, key_chars = _plain_cases()[name]
    check_plain_rounds(ctx, t, oracle.sais(t), key_chars, name)


def test_round_counts_run_aware(ctx):
    old, _, sa = case("c2_runs")
    check_run_aware_rounds(ctx, old, sa, "c2_runs")


def test_round_counts_of_a_batch_chunk():
    import emu
    from batch_cases import exe_like_slices
    from deltaq_b200 import CudaSuffixSort
    texts = exe_like_slices(40, 12_000) + [random_bytes(3000, seed=4), np.zeros(700, np.uint8), random_bytes(1, seed=5)]
    with CudaSuffixSort(_lib=emu.library()) as sorter:
        check_batch_rounds(sorter, texts, "exe-like slices")
