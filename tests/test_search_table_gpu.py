"""The match search on the B200 at EVERY scan position of multi-megabyte pairs, against oracle.search_table (Diff.Search
from the ranks of a generalized suffix array, pinned to the literal replay by tests/test_search_reference.py).

The cases take the paths the search switches on by size, and assert from dq_stats that they took them:
  (a) bench.py's device step on the full C2 pair (16 -> 17 MiB), twice on one context: the second search starts from
      the 3-byte prefix table built from the sort's keys; then the host entry point with a caller-supplied I.
  (b) long repeats (~24 MiB of repeated 64 KiB blocks): the sort needs >= 14 rounds, so the index build and the
      search run their seed level with I = NULL; with DQ_PREFIX3 = 0 and 1.
  (c) the C5 recipe at 48 MiB with a caller-supplied I: seed level and a prefix table from the text by size alone;
      then again after the library's own sort.
  (d) ~8 MiB with an eighth of the text in equal-byte runs: the run-aware comparisons.
  (e) sub-ranges whose bounds sit around multiples of kChunk, kSuper and the seed warp, on (b) and (c).
  (f) a device group of three logical shards: group sort, sharded search and group LCP.
After each search the LCP array (dq_cuda_lcp) is compared with oracle.lcp_array.  Every pair and its reference table
is built once per module; (a) to (c) need several GB of host memory."""
import time

import numpy as np
import pytest

import oracle
from search_cases import block_repeat_pair, runs_pair, sub_ranges
from search_table_cases import assert_table, host_search, launches, one_repeated_byte_keys, sorted_and_searched

pytestmark = pytest.mark.gpu

MIB = 1 << 20
REPORT = {}


def report(key, value):
    REPORT[key] = value
    print(f"[search_table] {key}: {value}", flush=True)


def reference(name, old, new):
    t0 = time.perf_counter()
    pos, ln = oracle.search_table(old, new)
    report(f"{name} reference CPU s", round(time.perf_counter() - t0, 1))
    return pos, ln


# ---- (a) bench.py's step on the full C2 pair -------------------------------------------------------------------------
def test_c2_bench_sequence():
    from deltaq_b200 import workloads as w
    from deltaq_b200._native import Context
    from device_entry_cases import CudaMem
    old, new = w.c2_exe_pair()
    n, m = old.size, new.size
    ref = reference("(a) C2 16->17 MiB", old, new)
    sa_ref = oracle.sais(old)
    mem = CudaMem()
    d_old, d_new = mem.put(old), mem.put(new)
    d_sa, d_pos, d_len = (mem.put(np.zeros(k, np.int32)) for k in (n, m, m))
    sort_launches = []
    with Context(device=0) as ctx:
        for step in (1, 2):
            ctx.suffix_sort_device(mem.ptr(d_old), n, mem.ptr(d_sa))
            sort_launches.append(launches(ctx))
            ctx.bsdiff_search_device(mem.ptr(d_old), n, None, mem.ptr(d_new), m, 0, m, mem.ptr(d_pos), mem.ptr(d_len))
            assert ctx.stats()["search_queries"] == m
            assert np.array_equal(mem.get(d_sa), sa_ref), step
            assert_table(mem.get(d_pos), mem.get(d_len), ref, ("device step", step))
        # the second sort ran on a context that had searched: it built the prefix table from its round-0 keys
        assert sort_launches[1] > sort_launches[0], sort_launches
        report("(a) paths", f"sort launches {sort_launches}: step 2 adds the prefix table from sorted keys")
        lcp_ref = oracle.lcp_array(old, sa_ref)
        assert np.array_equal(ctx.lcp(old), lcp_ref), "lcp, resident index"
        I = oracle.make_I(sa_ref)
        pos, ln = host_search(ctx, old, I, new)
        assert_table(pos, ln, ref, "host entry point, caller I")
        assert np.array_equal(ctx.lcp(old, sa_ref), lcp_ref), "lcp, caller I"


# ---- (b) long repeats: seed level with I = NULL ----------------------------------------------------------------------
@pytest.fixture(scope="module")
def repeats():
    old, new = block_repeat_pair(64 * 1024, 384)
    sa = oracle.sais(old)
    return {"old": old, "new": new, "ref": reference("(b) repeats 24 MiB", old, new), "sa": sa,
            "lcp": oracle.lcp_array(old, sa)}


def test_long_repeats_seed_level(repeats, monkeypatch):
    from deltaq_b200._native import Context
    old, new = repeats["old"], repeats["new"]
    got = {}
    for p3, seeds in (("0", None), ("1", None), ("0", "0")):
        monkeypatch.setenv("DQ_PREFIX3", p3)
        if seeds is None:
            monkeypatch.delenv("DQ_SEEDS_PER", raising=False)
        else:
            monkeypatch.setenv("DQ_SEEDS_PER", seeds)
        ranges = sub_ranges(new.size) if seeds is None and p3 == "0" else ()
        with Context(device=0) as ctx:
            got[p3, seeds] = sorted_and_searched(ctx, old, new, repeats["ref"], repeats["sa"], repeats["lcp"],
                                                 ("DQ_PREFIX3", p3, "DQ_SEEDS_PER", seeds), ranges)
    rounds, index0, search0 = got["0", None]
    assert rounds >= 14, rounds                          # the rule that turns the seed level on for a resident SA
    _, index_p3, search_p3 = got["1", None]
    _, index_off, search_off = got["0", "0"]
    assert index0 > index_off and search0 > search_off, got   # seed level of the index build and of the search
    assert index_p3 > index0 and search_p3 == search0, got    # prefix table from the text, built with the index
    report("(b) paths", f"rounds {rounds}; (index, search) launches {got}")


# ---- (c) the C5 recipe at 48 MiB with a caller-supplied I -----------------------------------------------------------
@pytest.fixture(scope="module")
def c5():
    from deltaq_b200 import workloads as w
    old, new = w.c5_pair(48 * MIB)
    sa = oracle.sais(old)
    return {"old": old, "new": new, "ref": reference("(c) C5 recipe 48 MiB", old, new), "sa": sa,
            "lcp": oracle.lcp_array(old, sa)}


def test_c5_caller_index_then_library_sort(c5, monkeypatch):
    from deltaq_b200._native import Context
    old, new, ref, sa = c5["old"], c5["new"], c5["ref"], c5["sa"]
    assert old.size >= 32 * MIB          # a caller's I: the seed level and the prefix table are chosen by size
    monkeypatch.delenv("DQ_PREFIX3", raising=False)
    monkeypatch.delenv("DQ_SEEDS_PER", raising=False)
    with Context(device=0) as ctx:
        pos, ln = host_search(ctx, old, sa, new)
        full = launches(ctx)
        assert_table(pos, ln, ref, "caller I")
        for b, c in sub_ranges(new.size):
            pos, ln = host_search(ctx, old, None, new, b, c)
            assert_table(pos, ln, ref, ("caller I, resident after it", b, c), b)
        assert np.array_equal(ctx.lcp(old), c5["lcp"]), "lcp, resident caller index"
        assert np.array_equal(ctx.lcp(old, sa), c5["lcp"]), "lcp, caller I"
        off = {}
        for env in ("DQ_SEEDS_PER", "DQ_PREFIX3"):
            monkeypatch.setenv(env, "0")
            pos, ln = host_search(ctx, old, sa, new)
            off[env] = launches(ctx)
            assert_table(pos, ln, ref, (env, "0"))
            monkeypatch.delenv(env)
        assert full > off["DQ_SEEDS_PER"] and full > off["DQ_PREFIX3"], (full, off)
        report("(c) paths", f"caller I launches {full}, seed level off {off['DQ_SEEDS_PER']}, "
                            f"prefix table off {off['DQ_PREFIX3']}")
        # the library's own sort, on a context that has searched: prefix table from the sorted keys
        rounds, _, _ = sorted_and_searched(ctx, old, new, ref, sa, c5["lcp"], "library sort", sub_ranges(new.size)[:4])
        report("(c) library sort rounds", rounds)


# ---- (d) equal-byte runs ---------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def runs():
    old, new = runs_pair(8 * MIB)
    sa = oracle.sais(old)
    return {"old": old, "new": new, "ref": reference("(d) runs 8 MiB", old, new), "sa": sa,
            "lcp": oracle.lcp_array(old, sa)}


def test_equal_byte_runs(runs):
    from deltaq_b200._native import Context
    old, new = runs["old"], runs["new"]
    share = one_repeated_byte_keys(old) / old.size
    assert share >= 1 / 64, share                        # the sort's run-aware rule (deltaq_cuda.cu, run_aware)
    with Context(device=0) as ctx:
        sorted_and_searched(ctx, old, new, runs["ref"], runs["sa"], runs["lcp"], "runs, I = NULL")
        pos, ln = host_search(ctx, old, runs["sa"], new)
        assert_table(pos, ln, runs["ref"], "runs, caller I")
    report("(d) paths", f"one-repeated-byte keys {share:.3f} of n")


# ---- (f) a device group of three logical shards ----------------------------------------------------------------------
def test_device_group(repeats, monkeypatch):
    from deltaq_b200 import workloads as w
    from deltaq_b200._native import Context
    monkeypatch.setenv("DQ_SHARD_MIN", str(MIB))
    old, new = w.c2_exe_pair(8 * MIB, 8 * MIB + 1001)
    assert new.size % 3 != 0
    sa = oracle.sais(old)
    cases = [("c2 8 MiB", old, new, reference("(f) c2 8 MiB", old, new), sa, oracle.lcp_array(old, sa)),
             ("repeats", repeats["old"], repeats["new"], repeats["ref"], repeats["sa"], repeats["lcp"])]
    with Context(device=[0, 0, 0]) as grp:
        for name, o, nw, ref, s, lcp in cases:
            rounds, _, _ = sorted_and_searched(grp, o, nw, ref, s, lcp, ("group", name), sub_ranges(nw.size)[:6])
            report(f"(f) group {name} rounds", rounds)
