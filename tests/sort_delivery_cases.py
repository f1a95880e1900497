"""Checks of how the suffix sort delivers its array and of the per-round counts it reports, shared by the emulator
(test_emu_sort_delivery.py) and the GPU (test_sort_delivery_gpu.py) tests.

Early copy (deltaq_cuda.cu, EarlyCopy): when the caller's output is device-visible host memory, the sort starts copying
the suffix array there once at most n/8 suffixes (on a device group: of a bucket's) are unresolved; the rounds after
that list the slots they resolve, and patch_host_sa_kernel writes them into the host array once the copy has landed.
A dropped or misplaced patch leaves whatever the device array held in those slots.  So every pinned run here follows
the sort of a different text of the same length on the same context (the unresolved slots then hold wrong values, not
the right ones of an earlier sort of the same text), into a sentinel-filled buffer with guard entries on both sides.

Per-round counts: a suffix is unresolved after depth h exactly when it shares h characters with a neighbour in sorted
order, max(LCP[k], LCP[k+1]) >= h (Kasai's LCP, LCP[n] = 0).  Plain doubling enters round r >= 1 at depth
key_chars * 2^(r-1) (8 characters for byte keys, 16 / 32 / 64 for recoded small alphabets; a batch chunk starts at 5,
and there LCP is taken within each text), so the active count of every round follows from the oracle alone.

`Delivery` says how a test environment tells the two runs apart: on the GPU the plain run writes to pageable memory,
which the device cannot address; on the emulator every host address is device-visible, so the plain run switches the
early copy off (DQ_EARLY_COPY_MIN = 0) instead."""
import contextlib
import os

import numpy as np

import oracle

SENTINEL = -7
FRONT, BACK = 3, 5   # guard entries before and after the output; FRONT also puts it at a non-zero int32 offset


@contextlib.contextmanager
def env(values):
    """os.environ with `values` set for the duration (None removes a variable); the old values come back after."""
    old = {k: os.environ.get(k) for k in values}
    try:
        for k, v in values.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


class Delivery:
    """copy_env: environment of the run into pinned memory, whose early copy must start; plain_env: that of the run
    whose array arrives by the plain copy after the last round."""

    def __init__(self, copy_env=None, plain_env=None):
        self.copy_env = dict(copy_env or {})
        self.plain_env = dict(plain_env or {})


def assert_sa(got, ref, what):
    bad = np.flatnonzero(got != ref)
    assert bad.size == 0, (what, f"{bad.size} of {ref.size} slots differ; first at slot {int(bad[0])}: "
                                 f"{int(got[bad[0]])} instead of {int(ref[bad[0]])}; last at slot {int(bad[-1])}")


def tandem_repeats(n, frac, seed=9):
    """Uniform bytes with `frac` of them inside tandem repeats (units of 2-39 bytes, 200-3000 bytes each): round 0
    resolves most suffixes and a few rounds finish the rest -- the shape that takes the early copy."""
    rng = np.random.default_rng(seed)
    t = rng.integers(0, 256, n, dtype=np.uint8)
    budget = int(n * frac)
    while budget > 0:
        unit = int(rng.integers(2, 40))
        total = int(min(budget, rng.integers(200, 3000)))
        p = int(rng.integers(0, n - total - unit))
        t[p:p + total] = np.tile(t[p:p + unit], total // unit + 1)[:total]
        budget -= total
    return t


def zero_heavy(n, every, seed=12):
    """Zeros with a random island of every/8 to every/2 bytes in every stretch of `every`: about 70 % zeros, so the key
    of eight zero bytes holds more than a third of all suffixes."""
    rng = np.random.default_rng(seed)
    t = np.zeros(n, np.uint8)
    for s in range(0, n, every):
        k = int(rng.integers(every // 8, every // 2))
        p = s + int(rng.integers(0, every - k))
        t[p:min(n, p + k)] = rng.integers(0, 256, min(n, p + k) - p, dtype=np.uint8)
    return t


def decoy_of(t, seed=0):
    """A different text of the same length: `t` with its first and second halves swapped and a few bytes changed."""
    h = t.size // 2
    d = np.concatenate([t[h:], t[:h]])
    rng = np.random.default_rng(seed)
    idx = rng.integers(0, t.size, max(1, t.size // 4096))
    d[idx] ^= rng.integers(1, 256, idx.size, dtype=np.uint8)
    assert not np.array_equal(d, t)
    return d


# ---- early copy -----------------------------------------------------------------------------------------------------
def sort_plain(ctx, delivery, t):
    """dq_cuda_suffix_sort of `t` into pageable memory with a guard after it -> (suffix array, dq_stats)."""
    out = np.full(t.size + 1, SENTINEL, np.int32)
    with env(delivery.plain_env):
        ctx.suffix_sort(t, out[:t.size])
    assert out[t.size] == SENTINEL, "wrote past the output"
    return out[:t.size], ctx.stats()


def sort_pinned(ctx, delivery, t, decoy):
    """Sort `decoy` (same length) on ctx, then `t` into pinned memory from Context.pinned, filled with SENTINEL, at
    int32 offset FRONT and with BACK guard entries after it -> (suffix array, dq_stats, round_times)."""
    n = t.size
    assert decoy.size == n
    ctx.suffix_sort(decoy, np.empty(n, np.int32))
    buf = ctx.pinned(FRONT + n + BACK, np.int32)
    try:
        buf.array[:] = SENTINEL
        with env(delivery.copy_env):
            ctx.suffix_sort(t, buf.array[FRONT:FRONT + n])
        st, rounds = ctx.stats(), ctx.round_times()
        a = buf.array.copy()
    finally:
        buf.free()
    assert np.all(a[:FRONT] == SENTINEL) and np.all(a[FRONT + n:] == SENTINEL), "wrote outside the output"
    return a[FRONT:FRONT + n], st, rounds


def check_early_copy(ctx, delivery, t, sa_ref, what):
    """One device: the pinned run equals SA-IS, adds exactly one launch (patch_host_sa_kernel) to the plain run, and
    at least one round ran after the copy had started (a round entered with 0 < active <= n/8), so its slots came
    through the late list.  Returns the pinned run's round_times."""
    plain, plain_st = sort_plain(ctx, delivery, t)
    assert_sa(plain, sa_ref, (what, "plain copy"))
    ctx.set_timing(True)
    try:
        sa, st, rounds = sort_pinned(ctx, delivery, t, decoy_of(t))
    finally:
        ctx.set_timing(False)
    assert_sa(sa, sa_ref, (what, "early copy"))
    assert st["kernel_launches"] == plain_st["kernel_launches"] + 1, (what, st["kernel_launches"],
                                                                      plain_st["kernel_launches"])
    assert len(rounds) == st["rounds"], (what, rounds, st["rounds"])
    late = [a for _, a, _ in rounds[1:] if a * 8 <= t.size]
    assert late, (what, "no round ran after the copy started", [a for _, a, _ in rounds])
    return rounds


def check_group_delivery(ctx, delivery, t, sa_ref, what):
    """A device group: pinned and plain runs equal SA-IS, and every bucket whose copy started added one
    patch_host_sa_kernel to the launches (the shards' counters are folded into the group's stats).  Returns the number
    of such buckets."""
    plain, plain_st = sort_plain(ctx, delivery, t)
    assert_sa(plain, sa_ref, (what, "plain copy"))
    sa, st, _ = sort_pinned(ctx, delivery, t, decoy_of(t))
    assert_sa(sa, sa_ref, (what, "early copy"))
    assert st["n"] == t.size and st["rounds"] == plain_st["rounds"], (what, st, plain_st)
    patches = st["kernel_launches"] - plain_st["kernel_launches"]
    assert patches >= 1, (what, "no bucket started its early copy", st["kernel_launches"], plain_st["kernel_launches"])
    return patches


def check_index_left_behind(ctx, old, new, lcp_ref, table_ref, what):
    """After the last sort of `old`: dq_cuda_lcp and the whole search with I = NULL against the oracle."""
    from search_table_cases import assert_table, host_search
    assert np.array_equal(ctx.lcp(old), lcp_ref), (what, "lcp")
    pos, ln = host_search(ctx, old, None, new)
    assert_table(pos, ln, table_ref, (what, "search, I = NULL"))


def check_sort_many_pinned(sorter, delivery, texts, group_text):
    """sort_many into the provider's pinned owner, on a pooled buffer that a batch of decoys (same lengths) left filled
    with SENTINEL, then into pageable memory.  texts[group_text] is routed to the group sort and sits at an odd int32
    offset of the owner (4-byte aligned only).  Every array equals SA-IS, the owner's entries past the batch still
    hold SENTINEL, and the pinned call launches at least one kernel more (the group's patches)."""
    refs = [oracle.sais(t) for t in texts]
    offsets = np.concatenate([[0], np.cumsum([t.size for t in texts])])
    assert offsets[group_text] % 2 == 1, offsets[group_text]
    with env(delivery.copy_env):
        decoys = sorter.sort_many([decoy_of(t, seed=i) if t.size else t for i, t in enumerate(texts)])
        addr = decoys.memory.ctypes.data
        decoys._pinned.array[:] = SENTINEL
        decoys.dispose()
        with sorter.sort_many(texts) as owner:
            assert owner.memory.ctypes.data == addr, "the pooled buffer was not reused"
            st = sorter.stats()
            got = [a.copy() for a in owner.arrays]
            tail = owner._pinned.array[offsets[-1]:].copy()
    assert np.all(tail == SENTINEL), "wrote past the batch"
    for i, (g, r) in enumerate(zip(got, refs)):
        assert_sa(g, r, ("pinned owner, text", i, texts[i].size))
    flat = np.full(offsets[-1] + 1, SENTINEL, np.int32)
    with env(delivery.plain_env):
        sorter.sort_many(texts, flat[:offsets[-1]])
    plain_st = sorter.stats()
    assert flat[-1] == SENTINEL
    for i, r in enumerate(refs):
        assert_sa(flat[offsets[i]:offsets[i + 1]], r, ("pageable, text", i, texts[i].size))
    assert st["kernel_launches"] - plain_st["kernel_launches"] >= 1, (st["kernel_launches"], plain_st["kernel_launches"])
    return got


# ---- per-round counts -----------------------------------------------------------------------------------------------
def shared_depths(t, sa):
    """max(LCP[k], LCP[k+1]) for every rank k (LCP[n] = 0): a suffix is unresolved after depth h exactly when its entry
    is >= h."""
    lcp = oracle.lcp_array(t, sa).astype(np.int64)
    return np.maximum(lcp, np.append(lcp[1:], 0))


def active_counts(depths, start):
    """Suffixes entering rounds 1, 2, ... of plain doubling from depth `start`: #{depth >= start * 2^(r-1)}, up to the
    first round nobody enters."""
    d = np.sort(np.asarray(depths).reshape(-1))
    out = []
    h = start
    while True:
        c = int(d.size - np.searchsorted(d, h, side="left"))
        if c == 0:
            return out
        out.append(c)
        h *= 2


def field_passes(nbits):
    """Radix passes of one key field of nbits bits (rx::plan_add_field: digits of at most 8 bits)."""
    return -(-nbits // 8)


def doubling_passes(n):
    """Passes of a doubling round: ISA[.] + 1 in [0, n] and the rank in [0, n - 1]."""
    return field_passes(n.bit_length()) + field_passes(max(n - 1, 1).bit_length())


def plain_rounds(t, sa, key_chars):
    """(active, passes) of every round of a one-text sort by plain doubling."""
    n = t.size
    return [(n, 8)] + [(a, doubling_passes(n)) for a in active_counts(shared_depths(t, sa), key_chars)]


def batch_rounds(texts, sas, key_bytes=5, text_shift=48):
    """(active, passes) of every round of one batch chunk: round 0 sorts (text, first 5 bytes, length code), LCP is
    taken within each text."""
    n = sum(t.size for t in texts)
    depths = [shared_depths(t, sa) for t, sa in zip(texts, sas) if t.size]
    r0 = field_passes(text_shift + (len(texts) - 1).bit_length())
    return [(n, r0)] + [(a, doubling_passes(n)) for a in active_counts(np.concatenate(depths), key_bytes)]


def timed(ctx, fn):
    """fn() with timing on -> (what it returns, dq_stats, [(active, passes)] of round_times)."""
    ctx.set_timing(True)
    try:
        out = fn()
        st = ctx.stats()
        rounds = [(a, p) for _, a, p in ctx.round_times()]
    finally:
        ctx.set_timing(False)
    return out, st, rounds


def _round_readouts(st, rounds, what):
    assert len(rounds) == st["rounds"], (what, len(rounds), st["rounds"])
    assert sum(a for a, _ in rounds) == st["active_sum"], (what, rounds, st["active_sum"])
    assert sum(p for _, p in rounds) == st["radix_passes"], (what, rounds, st["radix_passes"])


def check_plain_rounds(ctx, t, sa_ref, key_chars, what):
    """round_times() of a plain-doubling sort of `t` against plain_rounds: every round's active count and passes, and
    the number of rounds."""
    sa = np.empty(t.size, np.int32)
    _, st, rounds = timed(ctx, lambda: ctx.suffix_sort(t, sa))
    assert_sa(sa, sa_ref, what)
    _round_readouts(st, rounds, what)
    expected = plain_rounds(t, sa_ref, key_chars)
    assert rounds == expected, (what, "(active, passes) per round", rounds, "expected", expected)
    return rounds


def check_run_aware_rounds(ctx, t, sa_ref, what):
    """A text with many equal-byte runs (run-aware rounds): round 0 and the set entering round 1 are exact, round 1
    sorts 32-bit run-length keys, and later active counts do not increase."""
    from search_table_cases import one_repeated_byte_keys
    n = t.size
    assert one_repeated_byte_keys(t) * 64 >= n, what     # the run-aware rule (deltaq_cuda.cu, run_aware)
    sa = np.empty(n, np.int32)
    _, st, rounds = timed(ctx, lambda: ctx.suffix_sort(t, sa))
    assert_sa(sa, sa_ref, what)
    _round_readouts(st, rounds, what)
    assert len(rounds) >= 2, (what, rounds)
    assert rounds[0] == (n, 8), (what, rounds[0])
    assert rounds[1] == (active_counts(shared_depths(t, sa_ref), 8)[0], 4 + field_passes((n - 1).bit_length())), \
        (what, "round 1", rounds[1])
    active = [a for a, _ in rounds]
    assert all(b <= a for a, b in zip(active[1:], active[2:])), (what, "active set grew", active)
    assert all(p == doubling_passes(n) for _, p in rounds[2:]), (what, rounds)
    return rounds


def check_batch_rounds(sorter, texts, what):
    """sort_many of one chunk (every text below DQ_BATCH_SINGLE_MIN, the total below DQ_BATCH_CHUNK) into pageable
    memory: arrays against SA-IS, round_times() against batch_rounds."""
    refs = [oracle.sais(t) for t in texts]
    total = sum(t.size for t in texts)
    flat = np.empty(total, np.int32)
    _, st, rounds = timed(sorter.context, lambda: sorter.sort_many(texts, flat))
    offsets = np.concatenate([[0], np.cumsum([t.size for t in texts])])
    for i, r in enumerate(refs):
        assert_sa(flat[offsets[i]:offsets[i + 1]], r, (what, "text", i))
    _round_readouts(st, rounds, what)
    expected = batch_rounds(texts, refs)
    assert rounds == expected, (what, "(active, passes) per round", rounds, "expected", expected)
    return rounds
