"""The device-pointer entry points on the B200, against the oracle: dq_cuda_suffix_sort_device,
dq_cuda_bsdiff_search_device, dq_cuda_lcp_device and dq_cuda_radix_sort_pairs_device, with buffers allocated as torch
CUDA tensors and passed by data_ptr() -- and bench.py's device step (sort, then search with I = NULL) three times on
one context at full size, with the timing readouts its roofline is built from."""
import numpy as np
import pytest

import oracle
from conftest import adversarial_texts, asset_names, load_asset, load_golden_sa, random_bytes, small_alphabet_texts
from device_entry_cases import (RADIX_DISTRIBUTIONS, RADIX_FIELDS, CudaMem, check_group, check_lcp, check_radix,
                                check_radix_keeps_resident_index, check_radix_noop, check_search, check_suffix_sort)
from search_cases import small_random_pairs, structured_pairs

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def mem():
    return CudaMem()


@pytest.fixture(scope="module")
def ctx():
    from deltaq_b200._native import Context
    c = Context(device=0)
    yield c
    c.close()


# ---- suffix_sort_device ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", asset_names())
def test_sort_fixture_file(ctx, mem, name):
    check_suffix_sort(ctx, mem, load_asset(name), range(8), ref=load_golden_sa(name))


@pytest.mark.parametrize("name", sorted(adversarial_texts()))
def test_sort_adversarial(ctx, mem, name):
    check_suffix_sort(ctx, mem, adversarial_texts()[name], range(8))


@pytest.mark.parametrize("name", sorted(small_alphabet_texts()))
def test_sort_small_alphabet(ctx, mem, name, monkeypatch):
    monkeypatch.setenv("DQ_COMPACT_MIN", "1")
    check_suffix_sort(ctx, mem, small_alphabet_texts()[name], range(8))


# 4096 is both the one-CTA sort's limit (sx::kSmallN) and one radix tile (rx::kTile)
@pytest.mark.parametrize("size", [1, 2, 4095, 4096, 4097, 65_537, 3_000_000])
def test_sort_random(ctx, mem, size):
    check_suffix_sort(ctx, mem, random_bytes(size, seed=size), range(8))


# ---- bsdiff_search_device, lcp_device ----------------------------------------------------------------------------
@pytest.mark.parametrize("name", sorted(structured_pairs()))
def test_search_structured(ctx, mem, name):
    old, new = structured_pairs()[name]
    check_search(ctx, mem, old, new)


def test_search_small_random_pairs(ctx, mem):
    for k, (old, new) in enumerate(small_random_pairs(count=50)):
        check_search(ctx, mem, old, new, old_offset=k % 8)


@pytest.mark.parametrize("name", ["point_edits", "zero_runs_with_islands", "periodic_records", "single_old"])
def test_lcp(ctx, mem, name):
    old, new = structured_pairs()[name]
    check_lcp(ctx, mem, old, new)


# ---- radix_sort_pairs_device -------------------------------------------------------------------------------------
@pytest.mark.parametrize("bit_lo,nbits", RADIX_FIELDS)
def test_radix_sort_pairs_device(ctx, mem, bit_lo, nbits):
    for count in (1, 4095, 4096, 4097, 3 * 4096 + 7, 262_145, 1_000_003):
        for k, dist in enumerate(RADIX_DISTRIBUTIONS):
            check_radix(ctx, mem, count, bit_lo, nbits, dist, seed=count + 17 * k)


def test_radix_sort_pairs_device_nothing_to_sort(ctx, mem):
    check_radix_noop(ctx, mem)


def test_radix_sort_keeps_the_resident_index(ctx, mem):
    old, new = structured_pairs()["point_edits"]
    check_radix_keeps_resident_index(ctx, mem, old, new)


def test_group_of_logical_shards(mem, monkeypatch):
    from deltaq_b200 import workloads as w
    from deltaq_b200._native import Context
    monkeypatch.setenv("DQ_SHARD_MIN", "2000")
    old, new = w.c2_exe_pair(50_000, 52_000)
    with Context(device=[0, 0, 0]) as grp:
        check_group(grp, mem, old, new)


# ---- bench.py's device step, three times on one context ------------------------------------------------------------
def run_bench_steps(ctx, mem, old, new, steps=3):
    """What bench.py's step_device does with timing on: sort, read the timing, search with I = NULL -- on the same
    buffers every step.  Returns per step the suffix array, the (pos, len) table and the readouts taken after the sort."""
    n, m = old.size, new.size
    d_old, d_new = mem.put(old), mem.put(new)
    d_sa, d_pos, d_len = (mem.put(np.zeros(k, np.int32)) for k in (n, m, m))
    out = []
    ctx.set_timing(True)
    try:
        for _ in range(steps):
            ctx.suffix_sort_device(mem.ptr(d_old), n, mem.ptr(d_sa))
            rec = {"stats": ctx.stats(), "pass_times": ctx.pass_times(), "round_times": ctx.round_times()}
            ctx.bsdiff_search_device(mem.ptr(d_old), n, None, mem.ptr(d_new), m, 0, m, mem.ptr(d_pos), mem.ptr(d_len))
            rec["search_queries"] = ctx.stats()["search_queries"]
            rec["sa"], rec["pos"], rec["len"] = mem.get(d_sa), mem.get(d_pos), mem.get(d_len)
            out.append(rec)
    finally:
        ctx.set_timing(False)
    return out


@pytest.fixture(scope="module")
def bench_run():
    """bench.py's rank-0 pair on a fresh context: step 1 sorts before the context has ever searched, steps 2 and 3 sort
    with the 3-byte prefix table built from the round-0 keys, which the search then starts from."""
    from deltaq_b200 import workloads as w
    from deltaq_b200._native import Context
    old, new = w.c2_exe_pair(seed_old=1, seed_new=2)
    with Context(device=0) as c:
        steps = run_bench_steps(c, CudaMem(), old, new)
        sa = oracle.sais(old)
        I = oracle.make_I(sa)
        # the host entry point adopts I: no prefix table from sorted keys
        host_pos, host_len = np.empty(new.size, np.int32), np.empty(new.size, np.int32)
        c.bsdiff_search(old, I, new, 0, new.size, host_pos, host_len)
        emitted = c.greedy_emit(old, new, steps[-1]["pos"], steps[-1]["len"])
    return {"old": old, "new": new, "sa": sa, "I": I, "steps": steps, "host_pos": host_pos, "host_len": host_len,
            "emitted": emitted}


def test_bench_steps_against_the_oracle(bench_run):
    old, new, steps = bench_run["old"], bench_run["new"], bench_run["steps"]
    first = steps[0]
    for k, st in enumerate(steps):
        assert np.array_equal(st["sa"], bench_run["sa"]), f"suffix array of step {k + 1}"
        assert st["search_queries"] == new.size
        # step 1 searched without the prefix table, steps 2 and 3 with it: one table
        assert st["pos"].tobytes() == first["pos"].tobytes() and st["len"].tobytes() == first["len"].tobytes(), k + 1
    pos, ln = first["pos"], first["len"]
    assert np.array_equal(pos, bench_run["host_pos"]) and np.array_equal(ln, bench_run["host_len"])
    ref = oracle.bsdiff_streams(old, new, bench_run["I"], trace=True)
    visited = ref["trace_len"] >= 0
    assert np.array_equal(pos[visited], ref["trace_pos"][visited])
    assert np.array_equal(ln[visited], ref["trace_len"][visited])
    rp, rl = oracle.search_table(old, new)
    bad = np.flatnonzero((pos != rp) | (ln != rl))
    assert bad.size == 0, f"{bad.size} positions differ from oracle.search_table, first at scan {bad[:1]}"
    for k in ("ctrl", "diff", "extra"):
        assert bench_run["emitted"][k] == ref[k], k


def test_bench_steps_timing_readouts(bench_run):
    """The per-launch and per-round lists read after each sort agree with the sort's stats, and algorithmic_bytes is
    the header's formula: active * (41 + 24 passes) for round 0, active * (52 + 24 passes) after, plus 4n."""
    n = bench_run["old"].size
    for k, step in enumerate(bench_run["steps"]):
        st, passes, rounds = step["stats"], step["pass_times"], step["round_times"]
        assert len(passes) == st["radix_passes"], k + 1
        assert sum(p[1] for p in passes) == st["pass_pairs"], k + 1
        assert len(rounds) == st["rounds"], k + 1
        active = [r[1] for r in rounds]
        assert active[0] == n and all(b <= a for a, b in zip(active, active[1:])), k + 1
        assert sum(r[2] for r in rounds) == st["radix_passes"], k + 1
        assert sum(active) == st["active_sum"], k + 1
        alg = sum(a * ((41 if r == 0 else 52) + 24 * p) for r, (_, a, p) in enumerate(rounds)) + 4 * n
        assert st["algorithmic_bytes"] == alg, k + 1
