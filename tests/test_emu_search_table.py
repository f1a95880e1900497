"""The match search on the CPU logic emulator (tests/emu; NOT the product) at every scan position of pairs of about
100 to 150 KB with long repeats and equal-byte runs, against oracle.search_table, with the size-switched paths forced
on: the seed level (DQ_SEEDS_PER 1, 8 and 64 super-chunks per warp), the 3-byte prefix table from the text
(DQ_PREFIX3) and from the sort's round-0 keys (DQ_PREFIX3_SORTED_MIN), a resident index and a caller-supplied one, and
sub-ranges whose bounds sit around multiples of kChunk, kSuper and the seed warp.  The emulator runs a warp's lanes one
after another, so it shows wrong indexing and wrong bounds, not memory-ordering errors; tests/test_search_table_gpu.py
runs the same paths on the B200.  About 40 s on one 8-core x86 host."""
import numpy as np
import pytest

import oracle
from search_cases import block_repeat_pair, runs_pair, sub_ranges
from search_table_cases import assert_table, host_search, sorted_and_searched

PAIRS = {
    "repeats": lambda: block_repeat_pair(4096, 24, seed=21, pool=5),
    "runs": lambda: runs_pair(150_000, seed=22),
}


@pytest.fixture(scope="module")
def cases():
    out = {}
    for name, make in PAIRS.items():
        old, new = make()
        sa = oracle.sais(old)
        out[name] = {"old": old, "new": new, "ref": oracle.search_table(old, new), "sa": sa,
                     "lcp": oracle.lcp_array(old, sa)}
    return out


@pytest.fixture
def ctx():
    import emu
    c = emu.context()
    yield c
    c.close()


@pytest.mark.parametrize("per", ["1", "8", "64"])
@pytest.mark.parametrize("name", sorted(PAIRS))
def test_seed_level(cases, ctx, name, per, monkeypatch):
    monkeypatch.setenv("DQ_SEEDS_PER", per)
    c = cases[name]
    old, new = c["old"], c["new"]
    pos, ln = host_search(ctx, old, c["sa"], new)                    # caller-supplied I
    assert_table(pos, ln, c["ref"], ("caller I", per))
    with_seeds = ctx.stats()["kernel_launches"]
    monkeypatch.setenv("DQ_SEEDS_PER", "0")
    host_search(ctx, old, c["sa"], new)
    # the seed level is one more launch of the index build's head kernel and one of the search's
    assert with_seeds - ctx.stats()["kernel_launches"] == 2
    monkeypatch.setenv("DQ_SEEDS_PER", per)
    assert np.array_equal(ctx.lcp(old, c["sa"]), c["lcp"]), ("lcp, caller I", per)
    sorted_and_searched(ctx, old, new, c["ref"], c["sa"], c["lcp"], ("resident", per), sub_ranges(new.size, int(per)))


@pytest.mark.parametrize("p3", ["0", "1"])
@pytest.mark.parametrize("name", sorted(PAIRS))
def test_prefix3_from_the_text(cases, ctx, name, p3, monkeypatch):
    monkeypatch.setenv("DQ_PREFIX3", p3)
    c = cases[name]
    old, new = c["old"], c["new"]
    pos, ln = host_search(ctx, old, c["sa"], new)
    assert_table(pos, ln, c["ref"], ("caller I", p3))
    for b, cnt in sub_ranges(new.size)[:6]:
        pos, ln = host_search(ctx, old, None, new, b, cnt)
        assert_table(pos, ln, c["ref"], ("caller I, resident after it", p3, b, cnt), b)
    sorted_and_searched(ctx, old, new, c["ref"], c["sa"], c["lcp"], ("resident", p3))


@pytest.mark.parametrize("name", sorted(PAIRS))
def test_prefix3_from_the_sorted_keys(cases, ctx, name, monkeypatch):
    # the context searches with a caller's I first, so its sort then builds the table from the round-0 keys
    monkeypatch.delenv("DQ_PREFIX3", raising=False)
    monkeypatch.setenv("DQ_PREFIX3_SORTED_MIN", "1")
    c = cases[name]
    old, new = c["old"], c["new"]
    pos, ln = host_search(ctx, old, c["sa"], new)
    assert_table(pos, ln, c["ref"], "caller I")
    sa = np.empty(old.size, np.int32)
    ctx.suffix_sort(old, sa)
    plain = ctx.stats()["kernel_launches"]
    monkeypatch.setenv("DQ_PREFIX3_SORTED_MIN", str(old.size + 1))
    ctx.suffix_sort(old, sa)
    assert plain > ctx.stats()["kernel_launches"], "the sort did not build the prefix table"
    monkeypatch.setenv("DQ_PREFIX3_SORTED_MIN", "1")
    sorted_and_searched(ctx, old, new, c["ref"], c["sa"], c["lcp"], "resident, prefix table from sorted keys",
                        sub_ranges(new.size)[:6])
