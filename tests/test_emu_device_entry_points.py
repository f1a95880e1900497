"""The device-pointer entry points (dq_cuda_suffix_sort_device, dq_cuda_bsdiff_search_device, dq_cuda_lcp_device,
dq_cuda_radix_sort_pairs_device) on the CPU logic emulator (tests/emu; NOT the product), against the oracle.  The
emulator's device pointers are host addresses, so numpy arrays stand in for device memory.  The same checks run on
the B200 in test_device_entry_points_gpu.py."""
import numpy as np
import pytest

from conftest import adversarial_texts, asset_names, load_asset, load_golden_sa, random_bytes, small_alphabet_texts
from device_entry_cases import (RADIX_DISTRIBUTIONS, RADIX_FIELDS, HostMem, check_group, check_lcp, check_radix,
                                check_radix_keeps_resident_index, check_radix_noop, check_search, check_suffix_sort)
from search_cases import small_random_pairs, structured_pairs

MEM = HostMem()


@pytest.fixture(scope="module")
def ctx():
    import emu
    from deltaq_b200._native import Context
    c = Context(lib=emu.library())
    yield c
    c.close()


@pytest.mark.parametrize("name", asset_names())
def test_sort_fixture_file(ctx, name):
    check_suffix_sort(ctx, MEM, load_asset(name), (0, 3), ref=load_golden_sa(name))


@pytest.mark.parametrize("name", sorted(adversarial_texts()))
def test_sort_adversarial(ctx, name):
    check_suffix_sort(ctx, MEM, adversarial_texts()[name], (0, 5))


@pytest.mark.parametrize("name", sorted(small_alphabet_texts()))
def test_sort_small_alphabet(ctx, name, monkeypatch):
    monkeypatch.setenv("DQ_COMPACT_MIN", "1")
    check_suffix_sort(ctx, MEM, small_alphabet_texts()[name], (0, 7))


# 4096 is both the one-CTA sort's limit (sx::kSmallN) and one radix tile (rx::kTile)
@pytest.mark.parametrize("size", [1, 2, 4095, 4096, 4097, 65537])
def test_sort_random(ctx, size):
    check_suffix_sort(ctx, MEM, random_bytes(size, seed=size), range(8) if size <= 4097 else (0, 1))


@pytest.mark.parametrize("name", sorted(structured_pairs()))
def test_search_structured(ctx, name):
    old, new = structured_pairs()[name]
    check_search(ctx, MEM, old, new)


def test_search_small_random_pairs(ctx):
    for k, (old, new) in enumerate(small_random_pairs(count=50)):
        check_search(ctx, MEM, old, new, old_offset=k % 8)


@pytest.mark.parametrize("name", ["point_edits", "zero_runs_with_islands", "periodic_records", "single_old"])
def test_lcp(ctx, name):
    old, new = structured_pairs()[name]
    check_lcp(ctx, MEM, old, new)


@pytest.mark.parametrize("bit_lo,nbits", RADIX_FIELDS)
def test_radix_sort_pairs_device(ctx, bit_lo, nbits):
    for count in (1, 4095, 4096, 4097, 3 * 4096 + 7):
        for k, dist in enumerate(RADIX_DISTRIBUTIONS):
            check_radix(ctx, MEM, count, bit_lo, nbits, dist, seed=count + 17 * k)


def test_radix_sort_pairs_device_nothing_to_sort(ctx):
    check_radix_noop(ctx, MEM)


def test_radix_sort_keeps_the_resident_index(ctx):
    old, new = structured_pairs()["point_edits"]
    check_radix_keeps_resident_index(ctx, MEM, old, new)


def test_group_of_logical_shards(monkeypatch):
    import emu
    from deltaq_b200 import workloads as w
    from deltaq_b200._native import Context
    monkeypatch.setenv("DQ_SHARD_MIN", "2000")
    old, new = w.c2_exe_pair(20_000, 21_000)
    with Context(device=[0, 0, 0], lib=emu.library()) as grp:
        check_group(grp, MEM, old, new)
