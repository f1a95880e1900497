"""Parity of the CUDA suffix sorter with the oracle, through the C ABI (ctypes) and the provider mirror.

Reads like the reference's own tests: LibDivSufSortTests.cs (CheckShruggy, CheckFile, CheckRandomBuffer),
SAISTester.cs -- same fixtures, same sizes, same Verify (+ exact equality with the oracle's SA)."""
import numpy as np
import pytest

import oracle
from conftest import (REF_RANDOM_SIZES, SHRUGGY, adversarial_texts, asset_names, load_asset, load_golden_sa,
                      random_bytes)

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sorter():
    from deltaq_b200 import CudaSuffixSort
    s = CudaSuffixSort()
    yield s
    s.dispose()


def _sort(sorter, t):
    with sorter.sort(t) as owner:
        assert owner.memory.size == t.size
        return owner.memory.copy()


def test_native_library_is_loaded(sorter):
    import os
    from deltaq_b200 import _native
    assert os.path.basename(sorter.context.lib.path) == "libdeltaq_cuda.so"
    assert any("libdeltaq_cuda.so" in line for line in open("/proc/self/maps"))
    assert _native.default_library() is sorter.context.lib


def test_shruggy(sorter):
    t = np.frombuffer(SHRUGGY, dtype=np.uint8)
    sa = _sort(sorter, t)
    oracle.verify(t, sa)
    assert np.array_equal(sa, oracle.sais(t))


@pytest.mark.parametrize("name", asset_names())
def test_fixture_file(sorter, name):
    t = load_asset(name)
    sa = _sort(sorter, t)
    oracle.verify(t, sa)
    assert np.array_equal(sa, load_golden_sa(name))


@pytest.mark.parametrize("size", REF_RANDOM_SIZES + [64, 128, 256, 512, 1024, 2048, 8192, 16384, 65536, 1 << 20])
def test_random_buffer(sorter, size):
    # sizes of LibDivSufSortTests.cs:126-137 plus the benchmark's (SuffixSortingBenchmarks.cs:27-53)
    t = random_bytes(size)
    sa = np.full(size + 1, -7, dtype=np.int32)       # caller buffer NOT zeroed, one guard slot
    sorter.sort(t, sa[:size])
    assert sa[size] == -7                            # only suffixes[0..n) may be written (Diff.cs:78,90)
    oracle.verify(t, sa[:size])
    assert np.array_equal(sa[:size], oracle.sais(t))


@pytest.mark.parametrize("name", sorted(adversarial_texts()))
def test_adversarial(sorter, name):
    t = adversarial_texts()[name]
    sa = _sort(sorter, t)
    oracle.verify(t, sa)
    assert np.array_equal(sa, oracle.sais(t))


def test_length_mismatch_raises(sorter):
    # LibDivSufSort.cs:23-31: ArgumentException("Text and suffix buffers should have the same length")
    with pytest.raises(ValueError, match="same length"):
        sorter.sort(random_bytes(10), np.zeros(9, dtype=np.int32))


def test_empty_and_single(sorter):
    assert _sort(sorter, np.zeros(0, np.uint8)).size == 0
    assert _sort(sorter, np.array([7], np.uint8)).tolist() == [0]
    assert _sort(sorter, np.array([2, 1], np.uint8)).tolist() == [1, 0]
    assert _sort(sorter, np.array([1, 1], np.uint8)).tolist() == [1, 0]


@pytest.mark.parametrize("sigma,n", [(2, 300_000), (4, 1_000_000), (256, 3_000_000)])
def test_medium_sizes_against_oracle(sorter, sigma, n):
    t = np.random.default_rng(n).integers(0, sigma, n, dtype=np.uint8)
    sa = _sort(sorter, t)
    assert np.array_equal(sa, oracle.sais(t))


def test_workload_shapes_small(sorter):
    from conftest import small_alphabet_texts
    from deltaq_b200 import workloads as w
    old, _ = w.c2_exe_pair(1 << 20, (1 << 20) + (1 << 16))
    texts = [old, w.c3_repetitive(1 << 20), w.c3_fibonacci(200_000), w.c4_genome(1 << 20)]
    # small alphabets with 8-bit keys (no DQ_COMPACT_MIN) and a mostly-unique text with tandem repeats
    texts += [small_alphabet_texts()[name] for name in ("acgt_tandem", "bin_70000", "acgt_a_tail")]
    texts.append(_texts_with_repeats()["rep10pct_60k"])
    for t in texts:
        sa = _sort(sorter, t)
        assert np.array_equal(sa, oracle.sais(t))


def test_full_size_properties(sorter):
    """BASELINE configs at full size: size-independent checks (sufcheck is O(n); plus the permutation
    property) -- C1 exactly against the oracle, C2-old and C3 by sufcheck + Verify."""
    from deltaq_b200 import workloads as w
    t = w.c1_uniform()
    assert np.array_equal(_sort(sorter, t), oracle.sais(t))
    old, _ = w.c2_exe_pair()
    sa = _sort(sorter, old)
    assert oracle.sufcheck(old, sa) == 0
    oracle.verify(old, sa)
    t = w.c3_repetitive()
    sa = _sort(sorter, t)
    assert oracle.sufcheck(t, sa) == 0


def test_radix_sort_pairs_is_stable(sorter):
    rng = np.random.default_rng(3)
    for count, bits in [(1, 64), (4095, 64), (4096, 64), (4097, 13), (100_000, 64), (1_000_003, 40), (50_000, 3)]:
        keys = rng.integers(0, 2 ** 63, count, dtype=np.uint64)
        if bits < 64:
            keys &= np.uint64((1 << bits) - 1)
        vals = np.arange(count, dtype=np.uint32)
        k2, v2 = keys.copy(), vals.copy()
        sorter.context.radix_sort_pairs(k2, v2, bits)
        order = np.argsort(keys, kind="stable")
        assert np.array_equal(k2, keys[order]) and np.array_equal(v2, vals[order])


def test_stats_and_reuse(sorter):
    t = random_bytes(100_000)
    a = _sort(sorter, t)
    st = sorter.stats()
    assert st["n"] == t.size and st["rounds"] >= 1 and st["radix_passes"] >= 8 and st["device_ms"] > 0
    z = np.zeros(50_000, np.uint8)
    assert np.array_equal(_sort(sorter, z), np.arange(49_999, -1, -1, dtype=np.int32))
    assert np.array_equal(_sort(sorter, t), a)


@pytest.mark.parametrize("name", sorted(__import__("conftest").small_alphabet_texts()))
def test_small_alphabets(sorter, name, monkeypatch):
    """Recoded keys (16 / 32 / 64 characters each) on small texts: DQ_COMPACT_MIN lowers the 4 MiB
    from which the product recodes."""
    from conftest import small_alphabet_texts
    monkeypatch.setenv("DQ_COMPACT_MIN", "1")
    t = small_alphabet_texts()[name]
    sa = np.full(t.size + 1, -7, dtype=np.int32)
    sorter.sort(t, sa[:t.size])
    assert sa[t.size] == -7
    assert np.array_equal(sa[:t.size], oracle.sais(t))


def _texts_with_repeats():
    """Mostly-unique texts with a few per cent inside tandem repeats: round 0 resolves most suffixes, a few rounds
    finish the rest -- the shape that takes the early copy of the suffix array (deltaq_cuda.cu, EarlyCopy)."""
    rng = np.random.default_rng(9)

    def make(n, frac, alphabet):
        t = rng.integers(0, alphabet, n, dtype=np.uint8)
        budget = int(n * frac)
        while budget > 0:
            unit = int(rng.integers(2, 40))
            total = int(min(budget, rng.integers(200, 3000)))
            p = int(rng.integers(0, n - total - unit))
            t[p:p + total] = np.tile(t[p:p + unit], total // unit + 1)[:total]
            budget -= total
        return t
    return {"rep5pct_100k": make(100_000, 0.05, 256), "rep10pct_60k": make(60_000, 0.10, 256),
            "rep1pct_acgt_80k": make(80_000, 0.01, 4), "rep30pct_50k": make(50_000, 0.30, 256)}


@pytest.mark.parametrize("name", sorted(_texts_with_repeats()))
def test_early_copy_of_the_suffix_array(sorter, name, monkeypatch):
    monkeypatch.setenv("DQ_EARLY_COPY_MIN", "1")
    monkeypatch.setenv("DQ_COMPACT_MIN", "1")
    t = _texts_with_repeats()[name]
    with sorter.sort(t) as owner:                      # pinned host memory: the device can patch it
        assert np.array_equal(owner.memory, oracle.sais(t))
    sa = np.full(t.size + 1, -7, dtype=np.int32)       # pageable memory: the plain copy at the end
    sorter.sort(t, sa[:t.size])
    assert sa[t.size] == -7 and np.array_equal(sa[:t.size], oracle.sais(t))
