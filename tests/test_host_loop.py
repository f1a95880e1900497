"""The host side of dq_cuda_bsdiff_streams (scan / extender + crew / writers, dq_diff_host.h) at sizes where the
helper threads take part, against the oracle's restatement of Diff.cs:92-223 (oracle/bsdiff.c).

Runs on the CPU: dq_cuda_greedy_emit is pure host code, reached here through the emulator build's library (the
same source as the product's).  The (pos, len) table is the oracle's own trace of Diff.Search -- filled only at the
positions the reference loop visits, which is all the loop may read."""
import numpy as np
import pytest

import oracle
from deltaq_b200 import workloads as w


@pytest.fixture(scope="module")
def pair():
    # a few long unchanged stretches (so single extensions run to hundreds of KiB), a shifted copy of a periodic
    # section (two alignments that both match: a long overlap split) and some point damage
    rng = np.random.default_rng(2024)
    old = w._exe_like(3 << 20, np.random.default_rng(7))
    period = np.tile(rng.integers(0, 256, 48, dtype=np.uint8), 6000)           # 288 KB of 48-byte records
    old = np.concatenate([old[:1 << 20], period, old[1 << 20:]])
    new = np.concatenate([old[:700_000], rng.integers(0, 256, 5000, dtype=np.uint8), old[703_000:(1 << 20) + 100_000],
                          period[24:200_000], old[(1 << 20) + 288_000 + 50_000:2_600_000], old[2_900_000:]]).copy()
    hits = rng.integers(0, new.size, 40)
    new[hits] ^= 0x55
    ref = oracle.bsdiff_streams(old, new, trace=True)
    return old, new, ref


@pytest.mark.parametrize("shape", ["0,1", "1,2", "3,2", "7,4"])
def test_greedy_emit_threads_match_reference(pair, shape, monkeypatch):
    import emu
    old, new, ref = pair
    monkeypatch.setenv("DQ_HOST_THREADS", shape)
    with emu.context() as ctx:
        got = ctx.greedy_emit(old, new, ref["trace_pos"], ref["trace_len"])
    for k in ("ctrl", "diff", "extra"):
        assert got[k] == ref[k], (shape, k)
    assert got["search_visits"] == ref["search_calls"]


def test_pair_has_stretches_long_enough_for_the_crew(pair):
    # the crew only walks stretches of 128 KiB and more (crew_min(), dq_diff_host.h): make sure this input has them
    _, _, ref = pair
    ctrl = np.frombuffer(ref["ctrl"], dtype="<i8").reshape(-1, 3)
    assert (ctrl[:, 0] >= (128 << 10)).sum() >= 3


@pytest.mark.parametrize("shape,cut", [("3,2", None), ("0,1", 900_000)])
def test_streams_end_to_end_on_emulator_at_crew_sizes(pair, monkeypatch, shape, cut):
    # the same pair through the whole of dq_cuda_bsdiff_streams on the logic emulator: sort, search,
    # encode_table_kernel, coded-table scan (block steps, chain walks, certified stretches), crew and writers; the
    # shape without helpers on the head of the pair only (the emulated sort and search are what takes the time)
    import emu
    from deltaq_b200 import CudaSuffixSort, bsdiff
    old, new, ref = pair
    if cut:
        old, new = old[:cut], new[:cut]
        ref = oracle.bsdiff_streams(old, new)
    monkeypatch.setenv("DQ_HOST_THREADS", shape)
    monkeypatch.setenv("DQ_CHECK_CERTS", "1")
    s = CudaSuffixSort(_lib=emu.library())
    try:
        got = bsdiff.create_streams(old, new, s)
        assert s._ctx.stats()["table_fallbacks"] == 0
    finally:
        s.dispose()
    for k in ("ctrl", "diff", "extra"):
        assert got[k] == ref[k], k
    assert got["search_visits"] == ref["search_calls"]


# ---- Patch.Apply (native add loop, dq_cuda_patch_apply) --------------------------------------------------------

def _patch_lib():
    import emu
    return emu.library()


def test_patch_apply_round_trip_and_corrupt_streams():
    """Patch.cs:95-168 on the oracle's streams; corrupt inputs raise "Corrupt patch" (Patch.cs:128,151) instead of
    reading out of bounds."""
    import numpy as np
    import oracle
    import pytest
    from deltaq_b200 import _native
    from search_cases import structured_pairs
    lib = _patch_lib()
    for name in ("point_edits", "shifted", "zero_runs_with_islands", "empty_old"):
        old, new = structured_pairs()[name]
        r = oracle.bsdiff_streams(old, new)
        out = _native.patch_apply(old, r["ctrl"], r["diff"], r["extra"], new.size, lib=lib)
        assert out.tobytes() == new.tobytes(), name
    old, new = structured_pairs()["point_edits"]
    r = oracle.bsdiff_streams(old, new)
    ctrl = bytearray(r["ctrl"])
    bad_cases = {
        "short_ctrl": (bytes(ctrl[:-5]), r["diff"], r["extra"], new.size),
        "short_diff": (bytes(ctrl), r["diff"][:-1], r["extra"], new.size),
        "short_extra": (bytes(ctrl), r["diff"], r["extra"][:max(0, len(r["extra"]) - 1)] if r["extra"] else b"", new.size + 1),
        "negative_add": (bytes(ctrl[:7]) + bytes([ctrl[7] | 0x80]) + bytes(ctrl[8:]), r["diff"], r["extra"], new.size),
        "too_long": (bytes(ctrl), r["diff"], r["extra"], new.size + 10),
    }
    for name, (c, d, e, sz) in bad_cases.items():
        with pytest.raises(RuntimeError, match="Corrupt patch"):
            _native.patch_apply(old, c, d, e, sz, lib=lib)
    # a seek that drives the old position below zero
    import struct
    bad = struct.pack("<q", 4) + struct.pack("<q", 0) + bytes([100, 0, 0, 0, 0, 0, 0, 0x80]) + struct.pack("<q", 4) + bytes(16)
    with pytest.raises(RuntimeError, match="Corrupt patch"):
        _native.patch_apply(np.zeros(50, np.uint8), bad, bytes(8), b"", 8, lib=lib)


@pytest.mark.parametrize("seed", [11, 12, 13])
def test_certified_stretches_on_exe_like_pairs(seed, monkeypatch):
    """Mutated copies of exe-like files (unchanged stretches of every length between overwrites, insertions and
    deletions; zero runs and periodic records where two alignments both match): dq_cuda_bsdiff_streams on the emulator with
    the certified stretches (every one compared byte for byte) gives the oracle's streams in every thread shape."""
    import emu
    from deltaq_b200 import CudaSuffixSort, bsdiff
    old, new = w.c2_exe_pair(260_000 + 7_000 * seed, 275_000 + 5_000 * seed, seed_old=seed, seed_new=100 + seed)
    ref = oracle.bsdiff_streams(old, new)
    monkeypatch.setenv("DQ_CHECK_CERTS", "1")
    for shape in ("0,1", "2,2", "1,1"):
        monkeypatch.setenv("DQ_HOST_THREADS", shape + ",16,32")   # crew parts of 16 KiB from 32 KiB up: the crew takes part
        s = CudaSuffixSort(_lib=emu.library())
        try:
            got = bsdiff.create_streams(old, new, s)
        finally:
            s.dispose()
        for k in ("ctrl", "diff", "extra"):
            assert got[k] == ref[k], (seed, shape, k)
        assert got["search_visits"] == ref["search_calls"]


def test_certified_stretches_with_many_small_edits(monkeypatch):
    """Dozens of stops: point overwrites, short insertions and deletions every few KiB, so the unchanged stretches between
    them come in every length around the 256-byte threshold of a certified stretch, and many pieces hold several."""
    import emu
    from deltaq_b200 import CudaSuffixSort, bsdiff
    rng = np.random.default_rng(99)
    old = w._exe_like(400_000, np.random.default_rng(5))
    parts, at = [], 0
    while at < old.size:
        keep = int(rng.choice([40, 200, 255, 256, 257, 300, 1000, 5000, 20000]))
        parts.append(old[at:at + keep])
        at += keep
        kind = rng.integers(0, 3)
        if kind == 0:                                       # overwrite a few bytes
            k = int(rng.integers(1, 12))
            parts.append(rng.integers(0, 256, k, dtype=np.uint8))
            at += k
        elif kind == 1:                                     # insert
            parts.append(rng.integers(0, 256, int(rng.integers(1, 600)), dtype=np.uint8))
        else:                                               # delete
            at += int(rng.integers(1, 600))
    new = np.concatenate(parts)
    ref = oracle.bsdiff_streams(old, new)
    assert len(ref["ctrl"]) // 24 > 50
    monkeypatch.setenv("DQ_CHECK_CERTS", "1")
    for shape in ("0,1", "3,2,16,32"):
        monkeypatch.setenv("DQ_HOST_THREADS", shape)
        s = CudaSuffixSort(_lib=emu.library())
        try:
            got = bsdiff.create_streams(old, new, s)
        finally:
            s.dispose()
        for k in ("ctrl", "diff", "extra"):
            assert got[k] == ref[k], (shape, k)
        assert got["search_visits"] == ref["search_calls"]
