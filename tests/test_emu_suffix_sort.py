"""Host logic + kernel indexing of the suffix sorter on the CPU logic emulator (tests/emu; NOT the product,
NOT a fallback -- see tests/emu/cuda_emu.h).  The same C ABI, the same Python wrappers."""
import numpy as np
import pytest

import oracle
from conftest import (REF_RANDOM_SIZES, SHRUGGY, adversarial_texts, asset_names, load_asset, load_golden_sa,
                      random_bytes)


@pytest.fixture(scope="module")
def sorter():
    from deltaq_b200 import CudaSuffixSort
    import emu
    s = CudaSuffixSort(_lib=emu.library())
    yield s
    s.dispose()


def _sort(sorter, t):
    with sorter.sort(t) as owner:
        return owner.memory.copy()


@pytest.mark.parametrize("name", asset_names())
def test_fixture_file(sorter, name):
    t = load_asset(name)
    assert np.array_equal(_sort(sorter, t), load_golden_sa(name))


@pytest.mark.parametrize("size", REF_RANDOM_SIZES)
def test_random_buffer(sorter, size):
    t = random_bytes(size)
    sa = np.full(size + 1, -7, dtype=np.int32)
    sorter.sort(t, sa[:size])
    assert sa[size] == -7
    assert np.array_equal(sa[:size], oracle.sais(t))


@pytest.mark.parametrize("name", sorted(adversarial_texts()))
def test_adversarial(sorter, name):
    t = adversarial_texts()[name]
    assert np.array_equal(_sort(sorter, t), oracle.sais(t))


def test_shruggy_and_errors(sorter):
    t = np.frombuffer(SHRUGGY, dtype=np.uint8)
    assert np.array_equal(_sort(sorter, t), oracle.sais(t))
    with pytest.raises(ValueError, match="same length"):
        sorter.sort(random_bytes(10), np.zeros(9, dtype=np.int32))
    with pytest.raises(TypeError):
        sorter.sort(None)


def test_multi_tile_low_entropy(sorter):
    # several radix tiles and rank tiles, many doubling rounds, partial last tiles
    from conftest import small_alphabet_texts
    rng = np.random.default_rng(11)
    texts = [rng.integers(0, sigma, n, dtype=np.uint8) for n, sigma in [(20_000, 2), (9_000, 3), (4097, 2), (8193, 256)]]
    # small alphabets with 8-bit keys (no DQ_COMPACT_MIN) and a mostly-unique text with tandem repeats
    texts += [small_alphabet_texts()[name] for name in ("acgt_tandem", "bin_70000", "acgt_a_tail")]
    texts.append(_texts_with_repeats()["rep10pct_60k"])
    for t in texts:
        assert np.array_equal(_sort(sorter, t), oracle.sais(t))


def test_radix_sort_pairs(sorter):
    rng = np.random.default_rng(3)
    for count, bits in [(1, 64), (4095, 64), (4097, 13), (30_000, 64), (10_000, 3)]:
        keys = rng.integers(0, 2 ** 63, count, dtype=np.uint64)
        if bits < 64:
            keys &= np.uint64((1 << bits) - 1)
        vals = np.arange(count, dtype=np.uint32)
        k2, v2 = keys.copy(), vals.copy()
        sorter.context.radix_sort_pairs(k2, v2, bits)
        order = np.argsort(keys, kind="stable")
        assert np.array_equal(k2, keys[order]) and np.array_equal(v2, vals[order])


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


def test_owners_are_rented_from_a_pool():
    """Sort(text) -> IMemoryOwner<int>: the reference rents from ArrayPool (LibDivSufSort.cs:14), so Sort(asset).Dispose()
    in a loop reuses one array; the provider keeps a disposed owner's pinned buffer for the next Sort.  A reused buffer is
    dirty (the sorter must not need zeroed output: SURVEY 8(b)), owners of different sizes coexist, and an owner that
    outlives its provider is still released."""
    import emu
    from deltaq_b200 import CudaSuffixSort
    rng = np.random.default_rng(3)
    with CudaSuffixSort(_lib=emu.library()) as s:
        t1 = rng.integers(0, 4, 3000, dtype=np.uint8)
        o1 = s.sort(t1)
        addr = o1.memory.ctypes.data
        assert o1.memory.size == t1.size and np.array_equal(o1.memory, oracle.sais(t1))
        o1.dispose()
        o1.dispose()                                       # idempotent
        t2 = rng.integers(0, 256, 2500, dtype=np.uint8)    # fits the kept buffer (capacity 4096)
        with s.sort(t2) as o2:
            assert o2.memory.ctypes.data == addr and o2.memory.size == t2.size
            assert np.array_equal(o2.memory, oracle.sais(t2))
            t3 = rng.integers(0, 2, 70000, dtype=np.uint8)  # while o2 is out: another buffer
            with s.sort(t3) as o3:
                assert o3.memory.ctypes.data != addr and np.array_equal(o3.memory, oracle.sais(t3))
        with s.sort(np.zeros(0, np.uint8)) as o0:
            assert o0.memory.size == 0
        assert 1 <= len(s._pool) <= s._POOL_KEEP
        late = s.sort(t1)
    assert s._pool == []
    assert np.array_equal(late.memory, oracle.sais(t1))    # still readable after the provider is gone
    late.dispose()                                          # freed, not pooled
