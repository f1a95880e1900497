"""The suffix array's delivery into pinned memory, and the per-round counts bench.py's roofline divides by, on the B200
at bench.py's sizes, against the oracle (sort_delivery_cases.py says what each check proves; test_emu_sort_delivery.py
runs the same checks on the emulator).

  A. Early copy on one GPU with the default DQ_EARLY_COPY_MIN: C2's old text (16 MiB, run-aware), C3 at 32 MiB (many
     plain rounds after the copy starts), the 64 MiB C4 slice (recoded keys), 8 MiB with 5 % tandem repeats.
  B. The group sort into pinned and pageable output, on logical shards of one GPU or real peers: C2's old text on 2, 3,
     4 and 8 shards; a zero-heavy 32 MiB text whose 00^8 key holds more than 1/G of the suffixes, on 3 and 8 shards,
     with and without DQ_DIRECT_MAX = 0; C3 at 32 MiB on 4 shards through exchange and direct rounds after the copy
     started; the C5 recipe at 128 MiB on 8 shards with every default.  C2 and C5 then check dq_cuda_lcp and the whole
     search with I = NULL on the index the pinned run left.  Then sort_many on a group of three, with a 4 MiB text
     routed to the group sort at an odd int32 offset of the provider's pinned owner.
  C. round_times() against the oracle's LCP array: C1, C3 at 16 MiB, the 64 MiB C4 slice, 4-symbol random text at
     8 MiB, C2's old text (run-aware) and a batch chunk.
Most of the wall time is SA-IS and the search reference on the host, computed once per text."""
import functools
import time

import numpy as np
import pytest

import oracle
from sort_delivery_cases import (Delivery, check_batch_rounds, check_early_copy, check_group_delivery,
                                 check_index_left_behind, check_plain_rounds, check_run_aware_rounds,
                                 check_sort_many_pinned, plain_rounds, tandem_repeats, zero_heavy)

pytestmark = pytest.mark.gpu

MIB = 1 << 20
DELIVERY = Delivery()     # pinned memory from Context.pinned against pageable numpy arrays, every threshold default


def report(key, value):
    print(f"[sort_delivery] {key}: {value}", flush=True)


def c5_new(old):
    """Stretches of `old` with point edits and a few inserted bytes between them: matches deep inside the 128 MiB
    index, at a size whose search reference stays cheap."""
    rng = np.random.default_rng(55)
    parts = []
    for p in (5 * MIB, 61 * MIB + 7, 127 * MIB):
        s = old[p:p + 3 * MIB].copy()
        k = rng.integers(0, s.size, 300)
        s[k] = rng.integers(0, 256, k.size, dtype=np.uint8)
        parts += [s, rng.integers(0, 256, int(rng.integers(1, 500)), dtype=np.uint8)]
    return np.concatenate(parts)


@functools.lru_cache(maxsize=None)
def case(name):
    """-> dict(old, new, sa) and, for the texts that are searched, lcp and table.  Built once per module."""
    from deltaq_b200 import workloads as w
    t0 = time.perf_counter()
    new = None
    if name == "c2":
        old, new = w.c2_exe_pair()
    elif name == "c5":
        old = w.c5_old(128 * MIB, workers=8)
        new = c5_new(old)
    elif name == "c3_32":
        old = w.c3_repetitive(32 * MIB)
    elif name == "c3_16":
        old = w.c3_repetitive(16 * MIB)
    elif name == "c4":
        old = w.c4_genome(64 * MIB)
    elif name == "tandem5":
        old = tandem_repeats(8 * MIB, 0.05)
    elif name == "zero_heavy":
        old = zero_heavy(32 * MIB, 64 * 1024)
    else:
        raise KeyError(name)
    out = {"old": old, "new": new, "sa": oracle.sais(old)}
    if new is not None:
        out["lcp"] = oracle.lcp_array(old, out["sa"])
        out["table"] = oracle.search_table(old, new)
    report(f"{name} reference CPU s", round(time.perf_counter() - t0, 1))
    return out


def _devices(shards):
    import torch
    k = torch.cuda.device_count()
    return [i % k for i in range(shards)]


def group(shards):
    from deltaq_b200._native import Context
    return Context(device=_devices(shards))


@pytest.fixture(scope="module")
def ctx():
    from deltaq_b200._native import Context
    c = Context(device=0)
    yield c
    c.close()


@pytest.fixture()
def defaults(monkeypatch):
    for v in ("DQ_EARLY_COPY_MIN", "DQ_SHARD_MIN", "DQ_DIRECT_MAX", "DQ_COMPACT_MIN", "DQ_BATCH_SINGLE_MIN",
              "DQ_BATCH_CHUNK", "DQ_SUB_MIN_LOG"):
        monkeypatch.delenv(v, raising=False)
    return monkeypatch


# ---- A. early copy on one GPU ---------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["c2", "c3_32", "c4", "tandem5"])
def test_early_copy_one_gpu(ctx, defaults, name):
    c = case(name)
    rounds = check_early_copy(ctx, DELIVERY, c["old"], c["sa"], name)
    report(f"A {name} active per round", [a for _, a, _ in rounds])


# ---- B. the group sort into pinned and pageable output --------------------------------------------------------------
@pytest.mark.parametrize("shards", [2, 3, 4, 8])
def test_group_c2(defaults, shards):
    defaults.setenv("DQ_SHARD_MIN", str(MIB))
    c = case("c2")
    with group(shards) as g:
        patches = check_group_delivery(g, DELIVERY, c["old"], c["sa"], ("c2", shards))
        check_index_left_behind(g, c["old"], c["new"], c["lcp"], c["table"], ("c2", shards))
    report(f"B c2 on {shards} shards: buckets patched", patches)


@pytest.mark.parametrize("shards", [3, 8])
@pytest.mark.parametrize("direct_max", ["0", None])
def test_group_zero_heavy(defaults, shards, direct_max):
    defaults.setenv("DQ_SHARD_MIN", str(MIB))
    if direct_max is not None:
        defaults.setenv("DQ_DIRECT_MAX", direct_max)
    c = case("zero_heavy")
    old = c["old"]
    assert np.count_nonzero(old == 0) >= 0.6 * old.size
    with group(shards) as g:
        patches = check_group_delivery(g, DELIVERY, old, c["sa"], ("zero_heavy", shards, direct_max))
    report(f"B zero_heavy on {shards} shards, DQ_DIRECT_MAX {direct_max}: buckets patched", patches)


def test_group_c3_exchange_then_direct_rounds(defaults):
    """Rounds above DQ_DIRECT_MAX go by request / reply exchanges, smaller ones by peer pointers.  With 256 Ki both
    kinds run after the total active count fell below n/8, so some bucket's copy had started before each of them."""
    direct_max = 1 << 18
    defaults.setenv("DQ_SHARD_MIN", str(MIB))
    defaults.setenv("DQ_DIRECT_MAX", str(direct_max))
    c = case("c3_32")
    old = c["old"]
    active = [a for a, _ in plain_rounds(old, c["sa"], 8)[1:]]
    assert any(a > 8 * MIB for a in active), active
    assert any(direct_max < a <= old.size // 8 for a in active) and any(a <= direct_max for a in active), active
    with group(4) as g:
        patches = check_group_delivery(g, DELIVERY, old, c["sa"], "c3_32")
    report("B c3 32 MiB on 4 shards: buckets patched", patches)


def test_group_c5_defaults(defaults):
    c = case("c5")
    assert c["old"].size >= 128 * MIB           # DQ_SHARD_MIN's default: the group sorts it
    with group(8) as g:
        patches = check_group_delivery(g, DELIVERY, c["old"], c["sa"], "c5")
        check_index_left_behind(g, c["old"], c["new"], c["lcp"], c["table"], "c5")
    report("B c5 128 MiB on 8 shards: buckets patched", patches)


def test_sort_many_on_a_group(defaults):
    from conftest import random_bytes, small_alphabet_texts
    from deltaq_b200 import CudaSuffixSort
    from deltaq_b200 import workloads as w
    defaults.setenv("DQ_SHARD_MIN", str(MIB))
    defaults.setenv("DQ_BATCH_SINGLE_MIN", str(MIB))
    big = w.c2_exe_pair(4 * MIB, 4 * MIB)[0]
    texts = [random_bytes(4097, seed=1), np.zeros(1000, np.uint8), random_bytes(4, seed=2), big, random_bytes(90_000),
             np.zeros(0, np.uint8), small_alphabet_texts()["acgt_tandem"], random_bytes(300_001, seed=7)]
    with CudaSuffixSort(device=_devices(3)) as sorter:
        check_sort_many_pinned(sorter, DELIVERY, texts, 3)


# ---- C. per-round counts against the oracle -------------------------------------------------------------------------
def test_round_counts_plain_doubling(ctx, defaults):
    from deltaq_b200 import workloads as w
    rng = np.random.default_rng(8)
    c1 = w.c1_uniform()
    check_plain_rounds(ctx, c1, oracle.sais(c1), 8, "c1")
    for name in ("c3_16", "c4"):
        c = case(name)
        rounds = check_plain_rounds(ctx, c["old"], c["sa"], 32 if name == "c4" else 8, name)
        report(f"C {name} rounds", rounds)
    defaults.setenv("DQ_COMPACT_MIN", "1")
    acgt = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, 8 * MIB)]
    rounds = check_plain_rounds(ctx, acgt, oracle.sais(acgt), 32, "acgt 8 MiB")
    report("C acgt 8 MiB rounds", rounds)


def test_round_counts_run_aware(ctx, defaults):
    c = case("c2")
    rounds = check_run_aware_rounds(ctx, c["old"], c["sa"], "c2")
    report("C c2 rounds", rounds)


def test_round_counts_of_a_batch_chunk(defaults):
    from batch_cases import exe_like_slices
    from conftest import random_bytes
    from deltaq_b200 import CudaSuffixSort
    texts = exe_like_slices(300, 1 * MIB) + [random_bytes(1_500_000, seed=4), np.zeros(7000, np.uint8)]
    with CudaSuffixSort(device=0) as sorter:
        rounds = check_batch_rounds(sorter, texts, "exe-like slices")
    report("C batch rounds", rounds)
