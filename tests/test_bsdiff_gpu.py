"""Parity of the CUDA bsdiff match search (and the Diff.Create mirror built on it) with the oracle,
through the C ABI.  Oracle = literal replay of Diff.Search / Diff.Create's loop (oracle/bsdiff.c)."""
import io
import os

import numpy as np
import pytest

import oracle
from conftest import GOLDEN, random_bytes
from search_cases import small_random_pairs, structured_pairs

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def sorter():
    from deltaq_b200 import CudaSuffixSort
    s = CudaSuffixSort()
    yield s
    s.dispose()


def check_pair(sorter, old, new):
    from deltaq_b200 import bsdiff
    I = oracle.make_I(oracle.sais(old))
    rp, rl = oracle.search_all(I, old, new)
    pos, ln = bsdiff.search_all(old, new, sorter, I=I)
    assert np.array_equal(ln, rl) and np.array_equal(pos, rp)
    pos, ln = bsdiff.search_all(old, new, sorter)
    assert np.array_equal(ln, rl) and np.array_equal(pos, rp)
    if new.size > 10:
        b, c = new.size // 3, new.size // 2
        pos, ln = bsdiff.search_all(old, new, sorter, I=I, scan_begin=b, count=c)
        assert np.array_equal(ln, rl[b:b + c]) and np.array_equal(pos, rp[b:b + c])
    got = bsdiff.create_streams(old, new, sorter)
    ref = oracle.bsdiff_streams(old, new, I)
    for k in ("ctrl", "diff", "extra"):
        assert got[k] == ref[k], k
    assert got["search_visits"] == ref["search_calls"]


def test_small_random_pairs(sorter):
    for old, new in small_random_pairs(count=200):
        check_pair(sorter, old, new)


@pytest.mark.parametrize("name", sorted(structured_pairs()))
def test_structured(sorter, name):
    old, new = structured_pairs()[name]
    check_pair(sorter, old, new)


def test_golden_bsdiff_cases(sorter):
    from deltaq_b200 import bsdiff
    g = np.load(os.path.join(GOLDEN, "bsdiff_cases.npz"))
    for k in range(int(g["count"])):
        old, new = g[f"c{k}_old"], g[f"c{k}_new"]
        got = bsdiff.create_streams(old, new, sorter)
        for s in ("ctrl", "diff", "extra"):
            assert got[s] == g[f"c{k}_{s}"].tobytes(), (k, s)
        pos, ln = bsdiff.search_all(old, new, sorter)
        visited = g[f"c{k}_trace_len"] >= 0
        assert np.array_equal(pos[visited], g[f"c{k}_trace_pos"][visited])
        assert np.array_equal(ln[visited], g[f"c{k}_trace_len"][visited])


def test_exe_like_pair_1mib_all_positions(sorter):
    """Every scan position of a 1 MiB exe-like pair against oracle.search_table (the literal replay is quadratic
    inside long matches; tests/test_search_reference.py pins the two together), with a caller's I and resident."""
    from deltaq_b200 import bsdiff, workloads as w
    old, new = w.c2_exe_pair(1 << 20, (1 << 20) + (1 << 16))
    I = oracle.make_I(oracle.sais(old))
    rp, rl = oracle.search_table(old, new)
    pos, ln = bsdiff.search_all(old, new, sorter, I=I)
    assert np.array_equal(pos, rp) and np.array_equal(ln, rl)
    pos, ln = bsdiff.search_all(old, new, sorter)
    assert np.array_equal(pos, rp) and np.array_equal(ln, rl)
    ref = oracle.bsdiff_streams(old, new, I)
    got = bsdiff.create_streams(old, new, sorter)
    for k in ("ctrl", "diff", "extra"):
        assert got[k] == ref[k], k


def test_c2_full_size_streams_identical(sorter):
    """BASELINE config #2 at full size: 16 MiB -> 17 MiB exe-like pair; the uncompressed ctrl/diff/extra
    streams equal the oracle's, and applying them reproduces `new` (round trip, BsDiffTests.cs:30-78)."""
    from deltaq_b200 import bsdiff, workloads as w
    old, new = w.c2_exe_pair()
    got = bsdiff.create_streams(old, new, sorter)
    ref = oracle.bsdiff_streams(old, new)
    for k in ("ctrl", "diff", "extra"):
        assert got[k] == ref[k], k
    assert got["search_visits"] == ref["search_calls"]
    rebuilt = bsdiff.apply_streams(old, got["ctrl"], got["diff"], got["extra"], new.size)
    assert rebuilt == new.tobytes()


@pytest.mark.parametrize("size", [0, 1, 512, 999, 1024, 4096, 0x10000])
def test_diff_create_roundtrip(sorter, size):
    # BsDiffTests.cs:30-78 and BsPatchTests.cs:18-38
    from deltaq_b200.bsdiff import Diff, Patch
    old = random_bytes(size)
    for new in (old.copy(), random_bytes(size + 3, seed=9)):
        out = io.BytesIO()
        Diff.create(old, new, out, sorter)
        patch = out.getvalue()
        assert patch[:8] == b"BSDIFF40"
        rebuilt = io.BytesIO()
        Patch.apply(old, patch, rebuilt)
        assert rebuilt.getvalue() == new.tobytes()


def test_diff_create_argument_validation(sorter):
    # BsDiffTests.cs:80-100
    from deltaq_b200.bsdiff import Diff
    with pytest.raises(TypeError):
        Diff.create(b"", b"", None, sorter)
    with pytest.raises(TypeError):
        Diff.create(b"", b"", io.BytesIO(), None)

    class NotSeekable(io.BytesIO):
        def seekable(self):
            return False

    with pytest.raises(ValueError):
        Diff.create(b"", b"", NotSeekable(), sorter)


def test_search_without_resident_index_is_an_error(sorter):
    from deltaq_b200 import _native
    old, new = random_bytes(100), random_bytes(50, seed=2)
    sorter.sort(random_bytes(7), np.zeros(7, np.int32))     # resident index has another length
    pos = np.zeros(50, np.int32)
    with pytest.raises(_native.NativeError) as ei:
        sorter.context.bsdiff_search(old, None, new, 0, 50, pos, pos.copy())
    assert ei.value.status == _native.DQ_ERR_INVALID_ARGUMENT


def test_diff_create_accepts_any_isuffixsort(sorter):
    """Diff.Create takes any ISuffixSort (Diff.cs:27): a foreign provider sorts, the GPU searches."""
    from deltaq_b200 import bsdiff

    class OracleSort:                       # stands in for the reference's SAIS / LibDivSufSort providers
        def sort(self, text, suffixes):
            if suffixes.size != text.size:
                raise ValueError("Text and suffix buffers should have the same length")
            suffixes[:] = oracle.sais(text)

    old, new = structured_pairs()["point_edits"]
    got = bsdiff.create_streams(old, new, OracleSort())
    ref = oracle.bsdiff_streams(old, new)
    for k in ("ctrl", "diff", "extra"):
        assert got[k] == ref[k], k
    out = io.BytesIO()
    bsdiff.Diff.create(old, new, out, OracleSort())
    rebuilt = io.BytesIO()
    bsdiff.Patch.apply(old, out.getvalue(), rebuilt)
    assert rebuilt.getvalue() == new.tobytes()


def test_coded_table_overflow_falls_back_to_full_table(monkeypatch):
    # dq_cuda_bsdiff_streams ships the table as code bytes + match heads; a head list that does not fit must give
    # the same streams through the full-table path (DQ_HEADS_CAP shrinks the list for this test)
    from deltaq_b200 import CudaSuffixSort, bsdiff
    rng = np.random.default_rng(77)
    old = rng.integers(0, 4, 6000, dtype=np.uint8)
    new = np.concatenate([old[3000:4000], rng.integers(0, 4, 500, dtype=np.uint8), old[:2500], old[5000:]])
    ref = oracle.bsdiff_streams(old, new, oracle.make_I(oracle.sais(old)))
    for cap, fallbacks in (("1", 1), ("100000", 0)):
        monkeypatch.setenv("DQ_HEADS_CAP", cap)
        s = CudaSuffixSort()
        try:
            got = bsdiff.create_streams(old, new, s)
            assert s._ctx.stats()["table_fallbacks"] == fallbacks
        finally:
            s.dispose()
        for k in ("ctrl", "diff", "extra"):
            assert got[k] == ref[k], (cap, k)


@pytest.mark.parametrize("shape", ["0,1", "1,1", "7,3"])
def test_streams_identical_for_every_host_thread_shape(shape, monkeypatch):
    # the host loop of dq_cuda_bsdiff_streams (scan / extender + crew / writers) on the real library, with no helpers,
    # one helper, and more helpers than the default; same pair, same bytes
    from deltaq_b200 import CudaSuffixSort, bsdiff, workloads as w
    monkeypatch.setenv("DQ_HOST_THREADS", shape)
    old, new = w.c2_exe_pair(n_old=2 << 20, n_new=(2 << 20) + (1 << 17))
    ref = oracle.bsdiff_streams(old, new)
    with CudaSuffixSort() as s:
        got = bsdiff.create_streams(old, new, s)
    for k in ("ctrl", "diff", "extra"):
        assert got[k] == ref[k], (shape, k)
    assert got["search_visits"] == ref["search_calls"]


def _broken_suffix_arrays(n):
    """Suffix arrays a faulty ISuffixSort provider might hand to Diff.Create (ADVICE r1): in range but not a
    permutation, an entry == n, a negative entry."""
    good = np.arange(n, dtype=np.int32)
    zeros = np.zeros(n + 1, np.int32)
    too_big = np.concatenate([good, [0]]).astype(np.int32)
    too_big[n // 2] = n
    negative = np.concatenate([good, [0]]).astype(np.int32)
    negative[3] = -5
    dup = np.concatenate([good, [0]]).astype(np.int32)
    dup[7] = dup[8]
    return {"all_zero": zeros, "entry_eq_n": too_big, "negative": negative, "duplicate": dup}


@pytest.mark.parametrize("kind", ["all_zero", "entry_eq_n", "negative", "duplicate"])
def test_broken_provider_is_rejected(sorter, kind):
    """The search validates a caller-supplied suffix array on the device before following its entries."""
    from deltaq_b200 import _native
    n = 5000
    old, new = random_bytes(n), random_bytes(300, seed=3)
    I = _broken_suffix_arrays(n)[kind]
    pos = np.zeros(new.size, np.int32)
    with pytest.raises(_native.NativeError) as ei:
        sorter.context.bsdiff_search(old, I, new, 0, new.size, pos, pos.copy())
    assert ei.value.status == _native.DQ_ERR_INVALID_ARGUMENT
    assert "permutation" in str(ei.value)
    # the context is still usable
    sa = np.empty(n, np.int32)
    sorter.sort(old, sa)
    assert np.array_equal(sa, oracle.sais(old))


def test_native_patch_file(sorter):
    """dq_cuda_bsdiff_patch: header (Diff.cs:54-70) + three sections, each ONE ordinary bzip2 stream holding exactly the
    bytes of dq_cuda_bsdiff_streams; Patch.apply rebuilds `new`; every level gives the same streams."""
    import bz2
    from deltaq_b200 import bsdiff
    from search_cases import structured_pairs
    pairs = list(structured_pairs().values())[:4] + [(random_bytes(70000), random_bytes(70003, seed=9))]
    for old, new in pairs:
        ref = bsdiff.create_streams(old, new, sorter)
        for level in (0, 1, 9):
            patch = sorter.context.bsdiff_patch(old, new, level=level)
            assert patch[:8] == b"BSDIFF40"
            cl, dl, size = (bsdiff.read_packed_long(patch[8 + 8 * i:16 + 8 * i]) for i in range(3))
            assert size == new.size
            assert bz2.decompress(patch[32:32 + cl]) == ref["ctrl"]
            assert bz2.decompress(patch[32 + cl:32 + cl + dl]) == ref["diff"]
            assert bz2.decompress(patch[32 + cl + dl:]) == ref["extra"]
            rebuilt = io.BytesIO()
            bsdiff.Patch.apply(old, patch, rebuilt)
            assert rebuilt.getvalue() == new.tobytes()
        out = io.BytesIO()
        out.write(b"xx")                      # Diff.Create writes at the stream's current position (Diff.cs:56)
        bsdiff.Diff.create(old, new, out, sorter)
        assert out.getvalue()[2:] == sorter.context.bsdiff_patch(old, new) and out.tell() == len(out.getvalue())


def _lcp_texts():
    from conftest import adversarial_texts, small_alphabet_texts
    out = dict(adversarial_texts())
    out.update({k: v for k, v in small_alphabet_texts().items() if k in ("acgt_tandem", "bin_zero_tail", "one_value_5000")})
    out["random_300k"] = random_bytes(300_000)
    out["fuzz3"] = np.fromfile(os.path.join(GOLDEN, "assets", "fuzz3"), dtype=np.uint8)
    out["single"] = np.array([9], np.uint8)
    out["empty"] = np.zeros(0, np.uint8)
    return out


def test_lcp_array_export(sorter):
    """dq_cuda_lcp (SURVEY 8(f) rank 4): the LCP array under the resident suffix array and under a caller-supplied one,
    against the definition (oracle.lcp_array); a following search reuses the index; a broken array is rejected."""
    from deltaq_b200 import _native, bsdiff
    for name, t in _lcp_texts().items():
        sa = np.empty(t.size, np.int32)
        sorter.sort(t, sa)
        ref = oracle.lcp_array(t, sa)
        assert np.array_equal(sorter.lcp_array(t), ref), name            # resident
        assert np.array_equal(sorter.lcp_array(t, sa), ref), name        # adopted
        if t.size > 100:
            new = np.concatenate([t[50:], t[:60]])
            pos, ln = bsdiff.search_all(t, new, sorter, I=oracle.make_I(sa))
            lcp_again = sorter.lcp_array(t)                                # index still resident after the search
            assert np.array_equal(lcp_again, ref), name
            rp, rl = oracle.search_all(oracle.make_I(sa), t, new)
            assert np.array_equal(pos, rp) and np.array_equal(ln, rl), name
    t = random_bytes(5000)
    with pytest.raises(_native.NativeError):
        sorter.lcp_array(t, np.zeros(t.size, np.int32))                   # not a permutation
    with pytest.raises(_native.NativeError):
        sorter.sort(random_bytes(100), np.empty(100, np.int32))
        sorter.lcp_array(t)                                               # resident array has another length


def test_tiny_old_against_a_large_new(sorter):
    """VERDICT r1: `old` empty or a few bytes while the coded table is active at scale; the all-zero pair overflows the
    head list (full-table path at 2 MiB, not only at the 6 KB of the DQ_HEADS_CAP test)."""
    from deltaq_b200 import bsdiff
    from search_cases import tiny_old_pairs
    fallbacks = 0
    for name, old, new in tiny_old_pairs(2 << 20):
        got = bsdiff.create_streams(old, new, sorter)
        ref = oracle.bsdiff_streams(old, new)
        for k in ("ctrl", "diff", "extra"):
            assert got[k] == ref[k], (name, k)
        assert got["search_visits"] == ref["search_calls"], name
        fallbacks += sorter.stats()["table_fallbacks"]
    assert fallbacks >= 1


def test_patch_and_output_are_flushed_through_buffering_streams(sorter):
    """BsPatchTests.cs:18-38 (BsPatchFlushesOutput): Create and Apply write through buffering wrappers, and the test reads
    the wrapped streams directly afterwards -- so both must have pushed their bytes down."""
    import io
    from conftest import random_bytes
    from deltaq_b200.bsdiff import Diff, Patch
    old, new = random_bytes(0x123, seed=21), random_bytes(0x4567, seed=22)
    patch_ms = io.BytesIO()
    wrapped_patch = io.BufferedRandom(patch_ms, buffer_size=1 << 20)      # (kept alive: closing it closes patch_ms)
    Diff.create(old, new, wrapped_patch, sorter)
    patch = patch_ms.getvalue()
    assert patch[:8] == b"BSDIFF40"
    rebuilt_ms = io.BytesIO()
    wrapped_rebuilt = io.BufferedRandom(rebuilt_ms, buffer_size=1 << 20)
    Patch.apply(old, patch, wrapped_rebuilt)
    assert rebuilt_ms.getvalue() == new.tobytes()


@pytest.mark.parametrize("size", [0, 1, 512, 999, 1024, 4096])
def test_roundtrip_from_streams(sorter, size):
    """BsDiffTests.cs:57-78 (BsDiffRoundtripFromStreams): Create writes into a fixed 0x2000-byte memory stream; Apply takes
    the old data as a stream and the patch through an open-stream callback (offset, length; length 0 = the rest -- so
    the last section is followed by the unused tail of the buffer, which the reader must leave alone)."""
    import io
    from conftest import random_bytes
    from deltaq_b200.bsdiff import Diff, Patch
    old, new = random_bytes(size), random_bytes(size, seed=77)
    memory = io.BytesIO(bytes(0x2000))
    Diff.create(old, new, memory, sorter)
    buf = memory.getvalue()
    assert len(buf) == 0x2000

    def open_patch_stream(start, length):
        return io.BytesIO(buf[start:start + length] if length > 0 else buf[start:])

    out = io.BytesIO()
    Patch.apply(io.BytesIO(old.tobytes()), open_patch_stream, out)
    assert out.getvalue() == new.tobytes()


def test_apply_stream_argument_checks(sorter):
    """Patch.cs:60-63, :97-102: unreadable / unseekable patch or input streams and an unwritable output are argument
    errors; a bad signature or negative header fields are a corrupt patch (:68-78)."""
    import io
    from conftest import random_bytes
    from deltaq_b200.bsdiff import Diff, Patch
    old, new = random_bytes(600), random_bytes(700, seed=5)
    ms = io.BytesIO()
    Diff.create(old, new, ms, sorter)
    buf = ms.getvalue()

    class Pipe(io.BytesIO):
        def seekable(self):
            return False

    class WriteOnly(io.BytesIO):
        def readable(self):
            return False

    def opener(kind=io.BytesIO, data=buf):
        return lambda start, length: kind(data[start:start + length] if length > 0 else data[start:])

    with pytest.raises(ValueError, match="Patch stream must be seekable"):
        Patch.apply(io.BytesIO(old.tobytes()), opener(Pipe), io.BytesIO())
    with pytest.raises(ValueError, match="Patch stream must be readable"):
        Patch.apply(io.BytesIO(old.tobytes()), opener(WriteOnly), io.BytesIO())
    with pytest.raises(ValueError, match="Input stream must be seekable"):
        Patch.apply(Pipe(old.tobytes()), opener(), io.BytesIO())
    with pytest.raises(ValueError, match="Input stream must be readable"):
        Patch.apply(WriteOnly(old.tobytes()), opener(), io.BytesIO())

    class ReadOnly(io.BytesIO):
        def writable(self):
            return False

    with pytest.raises(ValueError, match="Output stream must be writable"):
        Patch.apply(io.BytesIO(old.tobytes()), opener(), ReadOnly())
    with pytest.raises(RuntimeError, match="Corrupt patch"):
        Patch.apply(io.BytesIO(old.tobytes()), opener(data=b"BSDIFF41" + buf[8:]), io.BytesIO())
    negative = buf[:15] + bytes([buf[15] | 0x80]) + buf[16:]          # ctrl length with the sign bit set
    with pytest.raises(RuntimeError, match="Corrupt patch"):
        Patch.apply(io.BytesIO(old.tobytes()), opener(data=negative), io.BytesIO())
    out = io.BytesIO()
    Patch.apply(io.BytesIO(old.tobytes()), opener(), out)
    assert out.getvalue() == new.tobytes()
