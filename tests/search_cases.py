"""(old, new) pairs shared by the emulator and GPU search tests."""
import numpy as np


def small_random_pairs(count=120, seed=123):
    """Tiny alphabets and lengths: every leaf quirk of Diff.Search (L == 0, L == n, I[n] == 0, n in {0,1,2})."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(count):
        n = int(rng.integers(0, 40))
        m = int(rng.integers(0, 60))
        sigma = int(rng.integers(1, 5))
        hi = int(rng.integers(0, 2)) * 250
        old = (rng.integers(0, sigma, n) + hi).astype(np.uint8)
        new = (rng.integers(0, sigma, m) + int(rng.integers(0, 2)) * 250).astype(np.uint8) if rng.integers(0, 3) == 0 \
            else (rng.integers(0, sigma, m) + hi).astype(np.uint8)
        out.append((old, new))
    return out


def structured_pairs():
    rng = np.random.default_rng(5)
    out = {}
    z = np.zeros(5000, np.uint8)
    out["zeros_vs_zeros_then_one"] = (z, np.concatenate([np.zeros(3000, np.uint8), [1], np.zeros(500, np.uint8)]).astype(np.uint8))
    out["zeros_vs_longer_zeros"] = (np.zeros(700, np.uint8), np.zeros(1500, np.uint8))
    old = rng.integers(0, 256, 30000, dtype=np.uint8)
    out["identical"] = (old, old.copy())
    out["new_is_old_plus_tail"] = (old, np.concatenate([old, rng.integers(0, 256, 777, dtype=np.uint8)]))
    out["new_is_suffix_of_old"] = (old, old[12345:].copy())
    out["new_all_ff"] = (old, np.full(300, 255, np.uint8))
    out["new_all_00"] = (old, np.zeros(300, np.uint8))
    new = old.copy()
    new[rng.integers(0, new.size, 40)] ^= 0x55
    out["point_edits"] = (old, new)
    out["shifted"] = (old, np.concatenate([rng.integers(0, 256, 100, dtype=np.uint8), old[:-50]]))
    rec = np.tile(rng.integers(0, 256, 24, dtype=np.uint8), 600)
    rec2 = rec.copy()
    rec2[rng.integers(0, rec2.size, 25)] = 7
    out["periodic_records"] = (rec, np.concatenate([rec2[1000:], rec2[:1000]]))
    runs = np.zeros(20000, np.uint8)
    for p in rng.integers(0, 20000, 12):
        runs[p:p + int(rng.integers(1, 30))] = rng.integers(1, 256)
    runs2 = np.concatenate([runs[:7000], rng.integers(0, 256, 300, dtype=np.uint8), runs[6500:]])
    out["zero_runs_with_islands"] = (runs, runs2)
    bin_old = rng.integers(0, 2, 15000, dtype=np.uint8)
    bin_new = bin_old.copy()
    bin_new[5000:5050] = 1 - bin_new[5000:5050]
    out["binary_alphabet"] = (bin_old, np.concatenate([bin_new[:9000], bin_new[9100:]]))
    fa, fb = b"a", b"ab"
    while len(fb) < 6000:
        fa, fb = fb, fb + fa
    fib = np.frombuffer(fb, dtype=np.uint8).copy()
    out["fibonacci"] = (fib, fib[377:5000].copy())
    out["empty_old"] = (np.zeros(0, np.uint8), rng.integers(0, 256, 100, dtype=np.uint8))
    out["empty_new"] = (old[:100].copy(), np.zeros(0, np.uint8))
    out["single_old"] = (np.array([5], np.uint8), np.array([5, 5, 4, 6, 5], np.uint8))
    return out


def tiny_old_pairs(m, seed=3):
    """`old` of 0..9 bytes against a `new` of m bytes: the coded (pos, len) table of dq_cuda_bsdiff_streams at scale with
    almost nothing to search in, incl. a pair (9 zero bytes against m zero bytes) in which nearly every position is a
    match head, so the head list overflows and the full table crosses instead.  Yields (name, old, new)."""
    rng = np.random.default_rng(seed)
    for n_old in (0, 1, 2, 9):
        uni = rng.integers(0, 256, m, dtype=np.uint8)
        yield f"uniform_{n_old}", rng.integers(0, 256, n_old, dtype=np.uint8), uni
        zeros = np.zeros(m, np.uint8)
        yield f"zeros_{n_old}", zeros[:n_old].copy(), zeros
        mixed = rng.integers(0, 3, m, dtype=np.uint8)
        mixed[m // 40:m // 2] = 0
        yield f"mixed_{n_old}", mixed[:n_old].copy(), mixed


def block_repeat_pair(block, blocks, seed=11, pool=12):
    """`old` is `blocks` blocks of `block` bytes drawn from a pool of `pool` random blocks, with a few point edits, so
    its repeats are at least a block long (the sort then needs many doubling rounds); `new` moves, edits, drops and
    inserts blocks and ends inside one.  Yields repeats long enough for the search's seed level."""
    rng = np.random.default_rng(seed)
    bank = rng.integers(0, 256, (pool, block), dtype=np.uint8)
    old = bank[rng.integers(0, pool, blocks)].reshape(-1).copy()
    old[rng.integers(0, old.size, blocks // 4 + 1)] = rng.integers(0, 256, blocks // 4 + 1, dtype=np.uint8)
    parts = []
    for _ in range(blocks + blocks // 8):
        op = int(rng.integers(0, 10))
        if op < 6:                                   # a block of old, moved
            b = int(rng.integers(0, blocks))
            parts.append(old[b * block:(b + 1) * block].copy())
        elif op < 8:                                 # a stretch of old across a block boundary, with point edits
            p = int(rng.integers(0, old.size - block))
            s = old[p:p + int(rng.integers(1, block))].copy()
            s[rng.integers(0, s.size, 3)] ^= 0x21
            parts.append(s)
        elif op < 9:                                 # a pool block
            parts.append(bank[int(rng.integers(0, pool))].copy())
        else:                                        # fresh bytes
            parts.append(rng.integers(0, 256, int(rng.integers(1, block)), dtype=np.uint8))
    new = np.concatenate(parts)
    return old, new[:new.size - int(rng.integers(1, block))].copy()


def runs_pair(n, seed=12):
    """Exe-like-ish bytes with about 1/8 of the text in equal-byte runs of 8 to 4,000 bytes (zeros mostly): the sort's
    run-aware refinement (one-repeated-byte keys >= n / 64) and the search's run-end comparisons.  `new` changes run
    lengths, edits bytes and moves stretches."""
    rng = np.random.default_rng(seed)
    old = rng.integers(0, 256, n, dtype=np.uint8)
    old[rng.random(n) < 0.3] = 0
    covered = 0
    while covered < n // 8:
        L = int(rng.integers(8, 4000))
        p = int(rng.integers(0, n - L))
        old[p:p + L] = 0 if rng.integers(0, 4) else int(rng.integers(1, 256))
        covered += L
    old[n - int(rng.integers(1, 100)):] = 0          # ends inside a run
    parts = []
    pos = 0
    while pos < n:
        L = int(rng.integers(1000, 200_000))
        s = old[pos:pos + L].copy()
        op = int(rng.integers(0, 4))
        if op == 0:                                  # a run grows or shrinks
            z = np.flatnonzero(s == 0)
            if z.size:
                q = int(z[int(rng.integers(0, z.size))])
                s = np.concatenate([s[:q], np.zeros(int(rng.integers(1, 300)), np.uint8), s[q:]]) if rng.integers(0, 2) \
                    else np.concatenate([s[:q], s[q + int(rng.integers(1, 300)):]])
        elif op == 1:
            s[rng.integers(0, s.size, 5)] = rng.integers(0, 256, 5, dtype=np.uint8)
        elif op == 2:                                # a stretch from elsewhere in old
            p = int(rng.integers(0, n - 5000))
            s = np.concatenate([s, old[p:p + int(rng.integers(1, 5000))]])
        parts.append(s)
        pos += L
    return old, np.concatenate(parts)


def sub_ranges(m, per=8):
    """(scan_begin, count) pairs whose bounds sit at and +-1 around multiples of the search's chunk (32 positions),
    super-chunk (2,048) and seed-level warp (per super-chunks), plus the last position and all but the first."""
    out = [(1, m - 1), (m - 1, 1)]
    for unit in (32, 2048, per * 2048):
        out += [(unit - 1, unit + 1), (unit + 1, 2 * unit - 1), (2 * unit, 3 * unit + 1), (3 * unit - 1, 2 * unit),
                (m - unit - 1, unit + 1), (m - unit + 1, unit - 1)]
    return [(b, c) for b, c in out if b >= 0 and c >= 0 and b + c <= m]
