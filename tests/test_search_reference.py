"""oracle.search_table -- Diff.Search at every scan position from the ranks of a generalized suffix array
(oracle/search_rank.c) -- pinned to the literal replay oracle.search_all wherever the replay is cheap.  The GPU tests
compare the match search with search_table at every position of inputs of many megabytes, so a wrong tie rule, a
missing I[n] = 0 quirk or a wrong leaf at L = 0 / L = n here would hide a wrong kernel there."""
import os

import numpy as np
import pytest

import oracle
from conftest import GOLDEN, adversarial_texts, random_bytes
from search_cases import small_random_pairs, structured_pairs, tiny_old_pairs


def replay(old, new, scan_begin=0, count=None):
    return oracle.search_all(oracle.make_I(oracle.sais(old)), old, new, scan_begin, count)


def assert_same(old, new, what, scan_begin=0, count=None):
    rp, rl = replay(old, new, scan_begin, count)
    p, ln = oracle.search_table(old, new, scan_begin, count)
    assert p.shape == rp.shape and ln.shape == rl.shape, what
    bad = np.flatnonzero((p != rp) | (ln != rl))
    assert bad.size == 0, (what, f"{bad.size} positions differ, first at scan {scan_begin + int(bad[0])}: "
                                 f"({p[bad[0]]}, {ln[bad[0]]}) vs the replay's ({rp[bad[0]]}, {rl[bad[0]]})")


@pytest.mark.parametrize("seed", [1, 2, 123, 777])
def test_small_random_pairs(seed):
    # n in {0, 1, 2}, alphabets of 1..4 values: L == 0, L == n, the I[n] == 0 leaf and ties x == y everywhere
    for k, (old, new) in enumerate(small_random_pairs(count=400, seed=seed)):
        assert_same(old, new, (seed, k))


@pytest.mark.parametrize("name", sorted(structured_pairs()))
def test_structured(name):
    old, new = structured_pairs()[name]
    assert_same(old, new, name)


def test_golden_bsdiff_cases():
    g = np.load(os.path.join(GOLDEN, "bsdiff_cases.npz"))
    for k in range(int(g["count"])):
        assert_same(g[f"c{k}_old"], g[f"c{k}_new"], k)


def test_tiny_old_against_a_large_new():
    for name, old, new in tiny_old_pairs(20_000):
        assert_same(old, new, name)


@pytest.mark.parametrize("name", sorted(adversarial_texts()))
def test_adversarial_old_against_its_rotation(name):
    old = adversarial_texts()[name]
    rng = np.random.default_rng(old.size)
    new = np.roll(old, int(rng.integers(0, old.size)) if old.size else 0).copy()
    if new.size:
        k = max(1, new.size // 500)
        new[rng.integers(0, new.size, k)] = rng.integers(0, 256, k, dtype=np.uint8)
    assert_same(old, new, name)


@pytest.mark.parametrize("n,m", [(1, 3000), (2, 3000), (4095, 4097), (65_537, 65_536), (1 << 20, (1 << 20) + 333)])
def test_random_pairs(n, m):
    # uniform bytes: matches are a few bytes long, so the replay stays cheap at a megabyte
    assert_same(random_bytes(n, seed=n), random_bytes(m, seed=m + 1), (n, m))


def test_exe_like_pair_1mib():
    """Long matches: the replay is quadratic there, so it is run at the positions the greedy loop visits and in
    windows of 300 positions."""
    from deltaq_b200 import workloads as w
    old, new = w.c2_exe_pair(1 << 20, (1 << 20) + (1 << 16))
    I = oracle.make_I(oracle.sais(old))
    pos, ln = oracle.search_table(old, new)
    ref = oracle.bsdiff_streams(old, new, I, trace=True)
    visited = ref["trace_len"] >= 0
    assert visited.sum() > 1000
    assert np.array_equal(pos[visited], ref["trace_pos"][visited])
    assert np.array_equal(ln[visited], ref["trace_len"][visited])
    rng = np.random.default_rng(0)
    for b in list(rng.integers(0, new.size - 300, 40)) + [0, new.size - 300]:
        rp, rl = oracle.search_all(I, old, new, int(b), 300)
        assert np.array_equal(pos[b:b + 300], rp) and np.array_equal(ln[b:b + 300], rl), int(b)


def test_sub_ranges():
    """search_table(scan_begin, count) sorts only new[scan_begin:]; its answers equal the whole table's."""
    pairs = [structured_pairs()[k] for k in ("periodic_records", "zero_runs_with_islands", "single_old", "fibonacci")]
    pairs += small_random_pairs(count=40, seed=9)
    for k, (old, new) in enumerate(pairs):
        m = new.size
        for b, c in [(0, m), (1, m - 1), (m // 3, m // 2), (m - 1, 1), (0, 1), (m // 2, 1), (m, 0), (m // 2, 0)]:
            if b >= 0 and c >= 0 and b + c <= m:
                assert_same(old, new, (k, b, c), b, c)


def test_bad_arguments():
    old, new = random_bytes(100), random_bytes(50, seed=3)
    for b, c in [(-1, 1), (0, 51), (50, 1), (10, -1)]:
        with pytest.raises(ValueError):
            oracle.search_table(old, new, b, c)
