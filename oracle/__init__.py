"""ctypes binding of the CPU oracle (oracle/*.c).  TEST INFRASTRUCTURE ONLY.

Importable only from tests/, __graft_entry__.smoke() and bench.py's CPU-baseline
legs; the product package never imports this module.
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "liboracle.so")


def build(force=False):
    srcs = [os.path.join(_HERE, f) for f in ("sais.c", "divsufsort.c", "sufcheck.c", "bsdiff.c", "search_rank.c")]
    stale = force or not os.path.exists(_LIB_PATH) or any(
        os.path.getmtime(s) > os.path.getmtime(_LIB_PATH) for s in srcs)
    if stale:
        subprocess.check_call(["make", "-s", "-C", _HERE, "-B", "liboracle.so"])
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        try:
            build()
        except Exception:
            if not os.path.exists(_LIB_PATH):
                raise
        L = ctypes.CDLL(_LIB_PATH)
        u8p = ctypes.c_void_p
        i32p = ctypes.c_void_p
        L.oracle_sais.argtypes = [u8p, ctypes.c_int32, i32p]
        L.oracle_sais.restype = ctypes.c_int
        L.oracle_divsufsort.argtypes = [u8p, ctypes.c_int32, i32p]
        L.oracle_divsufsort.restype = ctypes.c_int
        L.oracle_sufcheck.argtypes = [u8p, ctypes.c_int32, i32p, ctypes.c_int32]
        L.oracle_sufcheck.restype = ctypes.c_int
        L.oracle_verify_sorted.argtypes = [u8p, ctypes.c_int32, i32p]
        L.oracle_verify_sorted.restype = ctypes.c_int32
        L.oracle_lcp_kasai.argtypes = [u8p, ctypes.c_int32, i32p, i32p, i32p]
        L.oracle_lcp_kasai.restype = None
        L.oracle_verify_pairs.argtypes = [u8p, ctypes.c_int32, i32p, ctypes.c_void_p, ctypes.c_int64]
        L.oracle_verify_pairs.restype = ctypes.c_int64
        L.oracle_sa_naive.argtypes = [u8p, ctypes.c_int32, i32p]
        L.oracle_sa_naive.restype = None
        L.oracle_search.argtypes = [i32p, u8p, ctypes.c_int32, u8p, ctypes.c_int32,
                                    ctypes.c_int32, ctypes.c_int32, ctypes.POINTER(ctypes.c_int32)]
        L.oracle_search.restype = ctypes.c_int32
        L.oracle_search_all.argtypes = [i32p, u8p, ctypes.c_int32, u8p, ctypes.c_int32,
                                        ctypes.c_int32, ctypes.c_int32, i32p, i32p]
        L.oracle_search_all.restype = None
        L.oracle_search_table.argtypes = [u8p, ctypes.c_int32, u8p, ctypes.c_int32,
                                          ctypes.c_int32, ctypes.c_int32, i32p, i32p]
        L.oracle_search_table.restype = ctypes.c_int
        L.oracle_write_packed_long.argtypes = [u8p, ctypes.c_int64]
        L.oracle_write_packed_long.restype = None
        L.oracle_bsdiff_run.argtypes = [u8p, ctypes.c_int32, u8p, ctypes.c_int32, i32p, i32p, i32p]
        L.oracle_bsdiff_run.restype = ctypes.c_void_p
        L.oracle_bsdiff_free.argtypes = [ctypes.c_void_p]
        L.oracle_bsdiff_free.restype = None
        _lib = L
    return _lib


class _BsdiffResult(ctypes.Structure):
    _fields_ = [("ctrl", ctypes.c_void_p), ("diff", ctypes.c_void_p), ("extra", ctypes.c_void_p),
                ("ctrl_len", ctypes.c_int64), ("diff_len", ctypes.c_int64), ("extra_len", ctypes.c_int64),
                ("search_calls", ctypes.c_int64)]


def _u8(a):
    a = np.ascontiguousarray(np.frombuffer(a, dtype=np.uint8) if not isinstance(a, np.ndarray) else a,
                             dtype=np.uint8)
    return a


def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data) if a.size else ctypes.c_void_p(0)


def sais(text):
    """SAIS.Sort(text) restated (oracle/sais.c)."""
    t = _u8(text)
    sa = np.empty(t.size, dtype=np.int32)
    rc = lib().oracle_sais(_ptr(t), t.size, _ptr(sa))
    if rc != 0:
        raise MemoryError("oracle_sais failed")
    return sa


def divsufsort(text):
    """LibDivSufSort.Sort(text) restated (oracle/divsufsort.c) -- the reference's default sorter."""
    t = _u8(text)
    sa = np.empty(t.size, dtype=np.int32)
    rc = lib().oracle_divsufsort(_ptr(t), t.size, _ptr(sa))
    if rc != 0:
        raise MemoryError("oracle_divsufsort failed")
    return sa


def sa_naive(text):
    t = _u8(text)
    sa = np.empty(t.size, dtype=np.int32)
    lib().oracle_sa_naive(_ptr(t), t.size, _ptr(sa))
    return sa


def sufcheck(text, sa):
    """LDSSChecker.Check: 0 Done, -1 BadArguments, -2 OutOfRange, -3 WrongOrder, -4 WrongPosition."""
    t = _u8(text)
    s = np.ascontiguousarray(sa, dtype=np.int32)
    return lib().oracle_sufcheck(_ptr(t), t.size, _ptr(s), s.size)


def verify(text, sa):
    """LibDivSufSortTests.Verify: raises AssertionError unless sa is THE suffix array of text."""
    t = _u8(text)
    s = np.ascontiguousarray(sa, dtype=np.int32)
    rc = sufcheck(t, s)
    assert rc == 0, f"sufcheck returned {rc}"
    bad = lib().oracle_verify_sorted(_ptr(t), t.size, _ptr(s))
    assert bad < 0, f"Input was unsorted at i={bad}"


def verify_pairs(text, sa, idx):
    """Number of sampled adjacent pairs (sa[i], sa[i+1]), i in idx, that are out of order or out of range."""
    t = _u8(text)
    s = np.ascontiguousarray(sa, dtype=np.int32)
    ix = np.ascontiguousarray(idx, dtype=np.int64)
    return int(lib().oracle_verify_pairs(_ptr(t), t.size, _ptr(s), _ptr(ix), ix.size))


def lcp_array(text, sa):
    """LCP[r] = longest common prefix of suffixes sa[r-1], sa[r]; LCP[0] = 0 (definition; Kasai's evaluation order)."""
    t = _u8(text)
    s = np.ascontiguousarray(sa, dtype=np.int32)
    out = np.zeros(t.size, dtype=np.int32)
    rank = np.empty(t.size, dtype=np.int32)
    if t.size:
        lib().oracle_lcp_kasai(_ptr(t), t.size, _ptr(s), _ptr(rank), _ptr(out))
    return out


def make_I(sa):
    """The (n+1)-entry buffer Diff.Create hands to Search: I[..n] = SA, I[n] = 0 (Diff.cs:78,90)."""
    s = np.ascontiguousarray(sa, dtype=np.int32)
    I = np.zeros(s.size + 1, dtype=np.int32)
    I[:s.size] = s
    return I


def search(I, old, query):
    """Diff.Search(I, old, query, 0, n) -> (pos, len)."""
    o = _u8(old)
    q = _u8(query)
    Ic = np.ascontiguousarray(I, dtype=np.int32)
    assert Ic.size == o.size + 1
    pos = ctypes.c_int32(0)
    ln = lib().oracle_search(_ptr(Ic), _ptr(o), o.size, _ptr(q), q.size, 0, o.size, ctypes.byref(pos))
    return pos.value, ln


def search_all(I, old, new, scan_begin=0, count=None):
    o = _u8(old)
    w = _u8(new)
    Ic = np.ascontiguousarray(I, dtype=np.int32)
    assert Ic.size == o.size + 1
    if count is None:
        count = w.size - scan_begin
    pos = np.empty(count, dtype=np.int32)
    ln = np.empty(count, dtype=np.int32)
    lib().oracle_search_all(_ptr(Ic), _ptr(o), o.size, _ptr(w), w.size, scan_begin, count, _ptr(pos), _ptr(ln))
    return pos, ln


def search_table(old, new, scan_begin=0, count=None):
    """What search_all returns for I = make_I(sais(old)), computed from the ranks of a generalized suffix array in
    linear time (oracle/search_rank.c): every scan position of inputs too large for the literal replay."""
    o = _u8(old)
    w = _u8(new)
    if count is None:
        count = w.size - scan_begin
    pos = np.empty(count, dtype=np.int32)
    ln = np.empty(count, dtype=np.int32)
    rc = lib().oracle_search_table(_ptr(o), o.size, _ptr(w), w.size, scan_begin, count, _ptr(pos), _ptr(ln))
    if rc == -2:
        raise MemoryError("oracle_search_table failed")
    if rc != 0:
        raise ValueError(f"oracle_search_table: bad arguments (n={o.size}, m={w.size}, {scan_begin}, {count})")
    return pos, ln


def packed_long(y):
    b = np.zeros(8, dtype=np.uint8)
    lib().oracle_write_packed_long(_ptr(b), int(y))
    return b.tobytes()


def bsdiff_streams(old, new, I=None, trace=False):
    """Diff.Create's loop restated: returns dict(ctrl, diff, extra, search_calls[, trace_pos, trace_len]).

    Streams are the UNCOMPRESSED bytes the reference feeds its three bzip2 streams."""
    o = _u8(old)
    w = _u8(new)
    if I is None:
        I = make_I(sais(o))
    Ic = np.ascontiguousarray(I, dtype=np.int32)
    assert Ic.size == o.size + 1 and Ic[o.size] == 0
    tp = tl = None
    if trace:
        tp = np.full(w.size, -1, dtype=np.int32)
        tl = np.full(w.size, -1, dtype=np.int32)
    h = lib().oracle_bsdiff_run(_ptr(o), o.size, _ptr(w), w.size, _ptr(Ic),
                                _ptr(tp) if trace else None, _ptr(tl) if trace else None)
    if not h:
        raise MemoryError("oracle_bsdiff_run failed")
    try:
        r = _BsdiffResult.from_address(h)
        out = {
            "ctrl": ctypes.string_at(r.ctrl, r.ctrl_len) if r.ctrl_len else b"",
            "diff": ctypes.string_at(r.diff, r.diff_len) if r.diff_len else b"",
            "extra": ctypes.string_at(r.extra, r.extra_len) if r.extra_len else b"",
            "search_calls": r.search_calls,
        }
    finally:
        lib().oracle_bsdiff_free(h)
    if trace:
        out["trace_pos"] = tp
        out["trace_len"] = tl
    return out
