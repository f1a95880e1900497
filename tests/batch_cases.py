"""Batches of texts for CudaSuffixSort.sort_many (dq_cuda_suffix_sort_batch), shared by the emulator and GPU tests."""
import numpy as np

import oracle
from conftest import (REF_RANDOM_SIZES, SHRUGGY, adversarial_texts, asset_names, load_asset, load_golden_sa,
                      random_bytes, small_alphabet_texts)


def mixed_batch():
    """One text of every reference random size, SHRUGGY, every adversarial text and a few small-alphabet texts."""
    texts = [random_bytes(size) for size in REF_RANDOM_SIZES]
    texts.append(np.frombuffer(SHRUGGY, dtype=np.uint8))
    texts += [adversarial_texts()[name] for name in sorted(adversarial_texts())]
    texts += [small_alphabet_texts()[name] for name in ("acgt_tandem", "bin_4163", "one_value_5000", "bin_zero_tail")]
    return texts


def fixture_batch():
    """All fixture files in one batch, with their golden suffix arrays."""
    names = asset_names()
    return [load_asset(n) for n in names], [load_golden_sa(n) for n in names]


def edge_batches():
    """Batches whose texts share suffixes and prefixes: the text id in the round-0 key must keep them apart."""
    rng = np.random.default_rng(21)
    t = rng.integers(0, 256, 300, dtype=np.uint8)
    low = rng.integers(0, 3, 200, dtype=np.uint8)
    out = {}
    out["duplicates"] = [t] * 5
    out["prefixes"] = [low] + [low[:k] for k in range(low.size)]
    out["all_zero_0_to_20"] = [np.zeros(k, np.uint8) for k in range(21)]
    out["suffixes_of_one_another"] = [low[k:] for k in range(0, low.size + 1, 7)] + [low]
    out["duplicates_between_others"] = [t, low, t, np.zeros(9, np.uint8), t, low[:5], t[:5], t]
    out["empties_between"] = [np.zeros(0, np.uint8), t, np.zeros(0, np.uint8), np.zeros(0, np.uint8), low,
                              np.zeros(0, np.uint8)]
    return out


def exe_like_slices(count, max_len, seed=5):
    """Slices of the exe-like old text of the C2 workload: zero runs and other equal-byte runs (plain doubling needs
    extra rounds for them)."""
    from deltaq_b200 import workloads
    old, _ = workloads.c2_exe_pair(4 << 20, 4 << 20)
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(count):
        n = int(np.exp(rng.uniform(np.log(16), np.log(max_len))))
        p = int(rng.integers(0, old.size - n))
        out.append(np.ascontiguousarray(old[p:p + n]))
    return out


def sort_many(sorter, texts):
    """sort_many(texts) as a list of per-text arrays (copies), the owner's offsets checked on the way."""
    with sorter.sort_many(texts) as owner:
        assert owner.offsets.size == len(texts) + 1 and owner.offsets[0] == 0
        assert np.array_equal(np.diff(owner.offsets), [len(t) for t in texts])
        assert owner.memory.size == owner.offsets[-1]
        return [a.copy() for a in owner.arrays]


def check_against_oracle(sorter, texts, expected=None):
    """Both sort_many overloads against oracle.sais (or the given arrays), with a guard entry after the flat output."""
    got = sort_many(sorter, texts)
    expected = expected if expected is not None else [oracle.sais(t) for t in texts]
    for i, (g, e) in enumerate(zip(got, expected)):
        assert np.array_equal(g, e), f"text {i} (length {texts[i].size})"
    total = sum(t.size for t in texts)
    flat = np.full(total + 1, -7, dtype=np.int32)
    sorter.sort_many(texts, flat[:total])
    assert flat[total] == -7
    assert np.array_equal(flat[:total], np.concatenate(expected) if expected else flat[:0])
    return got
