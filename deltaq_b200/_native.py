"""ctypes binding of libdeltaq_cuda (include/deltaq_cuda.h).

The product loads exactly one library: deltaq_b200/libdeltaq_cuda.so, built in-tree by
``python -m deltaq_b200.build`` (nvcc, sm_100a).  If it is missing, or no CUDA device is present,
every entry point raises -- there is no CPU fallback.
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdeltaq_cuda.so")

DQ_OK = 0
DQ_ERR_INVALID_ARGUMENT = -1
DQ_ERR_OUT_OF_MEMORY = -2
DQ_ERR_CUDA = -3
DQ_ERR_NO_DEVICE = -4
DQ_ERR_INTERNAL = -5
DQ_ERR_CORRUPT_PATCH = -6


class DqStats(ctypes.Structure):
    _fields_ = [("n", ctypes.c_int32), ("rounds", ctypes.c_int32), ("radix_passes", ctypes.c_int32),
                ("kernel_launches", ctypes.c_int32), ("active_sum", ctypes.c_int64),
                ("algorithmic_bytes", ctypes.c_int64), ("device_ms", ctypes.c_float),
                ("pass_ms", ctypes.c_float), ("pass_pairs", ctypes.c_int64),
                ("search_queries", ctypes.c_int32), ("search_ms", ctypes.c_float),
                ("table_fallbacks", ctypes.c_int32), ("table_heads", ctypes.c_int32),
                ("search_index_ms", ctypes.c_float)]

    def as_dict(self):
        return {k: getattr(self, k) for k, _ in self._fields_}


class DqDiffStreams(ctypes.Structure):
    _fields_ = [("ctrl", ctypes.c_void_p), ("ctrl_len", ctypes.c_int64),
                ("diff", ctypes.c_void_p), ("diff_len", ctypes.c_int64),
                ("extra", ctypes.c_void_p), ("extra_len", ctypes.c_int64),
                ("search_visits", ctypes.c_int64)]


class NativeError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(f"libdeltaq_cuda error {status}: {message}")
        self.status = status


EXPORTS = [
    "dq_cuda_create", "dq_cuda_destroy", "dq_cuda_last_error", "dq_cuda_get_stats", "dq_cuda_set_timing",
    "dq_cuda_get_pass_times", "dq_cuda_get_round_times",
    "dq_cuda_host_alloc", "dq_cuda_host_free", "dq_cuda_suffix_sort", "dq_cuda_suffix_sort_device",
    "dq_cuda_suffix_sort_batch", "dq_cuda_suffix_sort_lcp_batch",
    "dq_cuda_bsdiff_search", "dq_cuda_bsdiff_search_device", "dq_cuda_bsdiff_search_batch", "dq_cuda_lcp", "dq_cuda_lcp_device", "dq_cuda_bsdiff_streams", "dq_cuda_greedy_emit",
    "dq_cuda_patch_apply", "dq_cuda_bz2_bound", "dq_cuda_bz2_compress", "dq_cuda_bsdiff_patch",
    "dq_cuda_bz2_decompress", "dq_cuda_bspatch",
    "dq_cuda_radix_sort_pairs", "dq_cuda_radix_sort_pairs_device",
]


class Library:
    """One loaded copy of the C ABI."""

    def __init__(self, path=LIB_PATH):
        if not os.path.exists(path):
            raise ImportError(
                f"{path} not found: build it with `python -m deltaq_b200.build` (needs nvcc). "
                "deltaq_b200 has no CPU fallback.")
        self.path = path
        L = ctypes.CDLL(path)
        vp, i32, i64 = ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64
        L.dq_cuda_create.argtypes = [ctypes.POINTER(vp), ctypes.POINTER(ctypes.c_int), ctypes.c_int]
        L.dq_cuda_destroy.argtypes = [vp]
        L.dq_cuda_last_error.argtypes = [vp]
        L.dq_cuda_last_error.restype = ctypes.c_char_p
        L.dq_cuda_get_stats.argtypes = [vp, ctypes.POINTER(DqStats)]
        L.dq_cuda_set_timing.argtypes = [vp, ctypes.c_int]
        L.dq_cuda_get_pass_times.argtypes = [vp, vp, vp, vp, ctypes.c_int]
        L.dq_cuda_get_round_times.argtypes = [vp, vp, vp, vp, ctypes.c_int]
        L.dq_cuda_host_alloc.argtypes = [ctypes.POINTER(vp), ctypes.c_size_t]
        L.dq_cuda_host_free.argtypes = [vp]
        L.dq_cuda_suffix_sort.argtypes = [vp, vp, i32, vp]
        L.dq_cuda_suffix_sort_device.argtypes = [vp, vp, i32, vp]
        L.dq_cuda_suffix_sort_batch.argtypes = [vp, vp, vp, i32, vp]
        L.dq_cuda_suffix_sort_lcp_batch.argtypes = [vp, vp, vp, i32, vp, vp]
        L.dq_cuda_bsdiff_search.argtypes = [vp, vp, i32, vp, vp, i32, i32, i32, vp, vp]
        L.dq_cuda_bsdiff_search_device.argtypes = [vp, vp, i32, vp, vp, i32, i32, i32, vp, vp]
        L.dq_cuda_bsdiff_search_batch.argtypes = [vp, vp, vp, vp, vp, i32, vp, vp]
        L.dq_cuda_lcp.argtypes = [vp, vp, i32, vp, vp]
        L.dq_cuda_lcp_device.argtypes = [vp, vp, i32, vp, vp]
        L.dq_cuda_bsdiff_streams.argtypes = [vp, vp, i32, vp, i32, ctypes.POINTER(DqDiffStreams)]
        L.dq_cuda_greedy_emit.argtypes = [vp, vp, i32, vp, i32, vp, vp, ctypes.POINTER(DqDiffStreams)]
        L.dq_cuda_patch_apply.argtypes = [vp, i64, vp, i64, vp, i64, vp, i64, vp, i64]
        L.dq_cuda_bz2_bound.argtypes = [i64]
        L.dq_cuda_bz2_compress.argtypes = [vp, vp, ctypes.c_int, ctypes.c_int, ctypes.c_int, vp, vp, vp, vp]
        L.dq_cuda_bz2_decompress.argtypes = [vp, i64, ctypes.c_int, vp, i64, ctypes.POINTER(i64), vp]
        L.dq_cuda_bspatch.argtypes = [vp, i64, vp, i64, ctypes.c_int, vp, i64, ctypes.POINTER(i64)]
        L.dq_cuda_bsdiff_patch.argtypes = [vp, vp, i32, vp, i32, ctypes.c_int, ctypes.POINTER(vp),
                                           ctypes.POINTER(i64)]
        L.dq_cuda_radix_sort_pairs.argtypes = [vp, vp, vp, i32, i32]
        L.dq_cuda_radix_sort_pairs_device.argtypes = [vp, vp, vp, i32, i32, i32, vp]
        for name in EXPORTS:
            if name not in ("dq_cuda_last_error", "dq_cuda_bz2_bound"):
                getattr(L, name).restype = ctypes.c_int
        L.dq_cuda_bz2_bound.restype = i64
        self.L = L


_default = None


def default_library():
    global _default
    if _default is None:
        _default = Library(LIB_PATH)
    return _default


def _addr(a):
    if a is None:
        return None
    return ctypes.c_void_p(a.ctypes.data) if a.size else ctypes.c_void_p(0)


def patch_apply(old, ctrl, diff, extra, new_size, lib=None):
    """dq_cuda_patch_apply: Patch.ApplyInternal on uncompressed streams -> bytes of the new file (numpy uint8).
    Raises RuntimeError("Corrupt patch") where the reference throws InvalidOperationException."""
    lib = lib or default_library()
    o, c, d, e = (np.ascontiguousarray(np.frombuffer(x, dtype=np.uint8) if not isinstance(x, np.ndarray) else x)
                  for x in (old, ctrl, diff, extra))
    if new_size < 0:
        raise RuntimeError("Corrupt patch")
    out = np.empty(int(new_size), dtype=np.uint8)
    rc = lib.L.dq_cuda_patch_apply(_addr(o), o.size, _addr(c), c.size, _addr(d), d.size, _addr(e), e.size, _addr(out),
                                   int(new_size))
    if rc == DQ_ERR_CORRUPT_PATCH:
        raise RuntimeError("Corrupt patch")
    if rc != DQ_OK:
        raise NativeError(rc, "dq_cuda_patch_apply: bad arguments")
    return out


def bz2_compress(sections, level=0, threads=0, lib=None, info=None):
    """dq_cuda_bz2_compress: every section (bytes-like / uint8 arrays) as one ordinary bzip2 stream, blocks compressed
    in parallel by one crew of host threads.  level 1..9 = bzip2's; 0 = chosen per section for the thread count.
    Returns a list of bytes.  info (a list, optional) receives (level, blocks, serial_fallback) per section."""
    lib = lib or default_library()
    arrs = [np.ascontiguousarray(np.frombuffer(x, dtype=np.uint8) if not isinstance(x, np.ndarray) else x)
            for x in sections]
    k = len(arrs)
    if k == 0:
        return []
    outs = [np.empty(int(lib.L.dq_cuda_bz2_bound(a.size)), dtype=np.uint8) for a in arrs]
    src = (ctypes.c_void_p * k)(*[a.ctypes.data if a.size else None for a in arrs])
    dst = (ctypes.c_void_p * k)(*[o.ctypes.data for o in outs])
    lens = (ctypes.c_int64 * k)(*[a.size for a in arrs])
    caps = (ctypes.c_int64 * k)(*[o.size for o in outs])
    got = (ctypes.c_int64 * k)()
    inf = (ctypes.c_int32 * (3 * k))()
    rc = lib.L.dq_cuda_bz2_compress(src, lens, k, int(level), int(threads), dst, caps, got, inf)
    if rc != DQ_OK:
        raise NativeError(rc, "dq_cuda_bz2_compress failed (bad arguments, or libbz2 missing)")
    if info is not None:
        info[:] = [(inf[3 * i], inf[3 * i + 1], inf[3 * i + 2]) for i in range(k)]
    return [outs[i][:got[i]].tobytes() for i in range(k)]


def bz2_decompress(data, threads=0, lib=None, info=None, size_hint=0):
    """dq_cuda_bz2_decompress: one bzip2 stream, its blocks decoded in parallel -> bytes.  info (a list, optional) receives
    (blocks, serial_fallback).  Raises RuntimeError("Corrupt patch") for a damaged stream."""
    lib = lib or default_library()
    a = np.ascontiguousarray(np.frombuffer(data, dtype=np.uint8) if not isinstance(data, np.ndarray) else data)
    got = ctypes.c_int64()
    inf = (ctypes.c_int32 * 2)()
    out = np.empty(max(int(size_hint), 0), dtype=np.uint8)
    for _ in range(2):
        rc = lib.L.dq_cuda_bz2_decompress(_addr(a), a.size, int(threads), _addr(out), out.size, ctypes.byref(got), inf)
        if rc == DQ_ERR_INVALID_ARGUMENT and got.value > out.size:
            out = np.empty(got.value, dtype=np.uint8)     # now the size is known
            continue
        break
    if rc == DQ_ERR_CORRUPT_PATCH:
        raise RuntimeError("Corrupt patch")
    if rc != DQ_OK:
        raise NativeError(rc, "dq_cuda_bz2_decompress failed")
    if info is not None:
        info[:] = [inf[0], inf[1]]
    return out[:got.value].tobytes()


def bspatch(old, patch, threads=0, lib=None):
    """dq_cuda_bspatch: Patch.Apply on a BSDIFF40 file -> the new file (numpy uint8)."""
    lib = lib or default_library()
    o, p = (np.ascontiguousarray(np.frombuffer(x, dtype=np.uint8) if not isinstance(x, np.ndarray) else x)
            for x in (old, patch))
    size = ctypes.c_int64(-1)
    rc = lib.L.dq_cuda_bspatch(_addr(o), o.size, _addr(p), p.size, int(threads), None, 0, ctypes.byref(size))
    if rc == DQ_ERR_CORRUPT_PATCH:
        raise RuntimeError("Corrupt patch")
    if size.value < 0:
        raise NativeError(rc, "dq_cuda_bspatch: bad arguments")
    out = np.empty(size.value, dtype=np.uint8)
    rc = lib.L.dq_cuda_bspatch(_addr(o), o.size, _addr(p), p.size, int(threads), _addr(out), out.size, ctypes.byref(size))
    if rc == DQ_ERR_CORRUPT_PATCH:
        raise RuntimeError("Corrupt patch")
    if rc != DQ_OK:
        raise NativeError(rc, "dq_cuda_bspatch failed")
    return out


class PinnedArray:
    """numpy view over cudaHostAlloc memory (what the C# provider's MemoryManager<int> would own)."""

    def __init__(self, lib, shape, dtype):
        self._lib = lib
        dtype = np.dtype(dtype)
        count = int(np.prod(shape)) if not np.isscalar(shape) else int(shape)
        nbytes = max(1, count * dtype.itemsize)
        p = ctypes.c_void_p()
        rc = lib.L.dq_cuda_host_alloc(ctypes.byref(p), nbytes)
        if rc != DQ_OK:
            raise NativeError(rc, lib.L.dq_cuda_last_error(None).decode())
        self._ptr = p
        buf = (ctypes.c_uint8 * nbytes).from_address(p.value)
        self.array = np.frombuffer(buf, dtype=dtype, count=count).reshape(shape)

    def free(self):
        if self._ptr is not None:
            self.array = None
            self._lib.L.dq_cuda_host_free(self._ptr)
            self._ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Context:
    """dq_ctx wrapper: one call at a time.  `device`: None (current device), one CUDA ordinal, or a list of ordinals
    -- a device GROUP driven by this one context: inputs of at least DQ_SHARD_MIN bytes (default 128 MiB) are sorted
    and searched by all of them (the same ordinal may be listed several times: logical shards on one GPU)."""

    def __init__(self, device=None, lib=None):
        import threading
        self.lib = lib or default_library()
        self._gate = threading.Lock()   # held while context-owned result buffers are read (bsdiff_streams, greedy_emit)
        self._h = ctypes.c_void_p()
        if device is None:
            rc = self.lib.L.dq_cuda_create(ctypes.byref(self._h), None, 0)
        else:
            devs = [int(d) for d in device] if isinstance(device, (list, tuple)) else [int(device)]
            dev = (ctypes.c_int * len(devs))(*devs)
            rc = self.lib.L.dq_cuda_create(ctypes.byref(self._h), dev, len(devs))
        if rc != DQ_OK:
            raise NativeError(rc, self.lib.L.dq_cuda_last_error(None).decode())

    def close(self):
        if self._h:
            self.lib.L.dq_cuda_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != DQ_OK:
            raise NativeError(rc, self.lib.L.dq_cuda_last_error(self._h).decode())

    def stats(self):
        st = DqStats()
        self._check(self.lib.L.dq_cuda_get_stats(self._h, ctypes.byref(st)))
        return st.as_dict()

    def pass_times(self):
        """[(ms, pairs, shift)] of every onesweep launch of the last sort (timing must be on)."""
        cap = 4096
        ms = np.zeros(cap, dtype=np.float32)
        pairs = np.zeros(cap, dtype=np.int64)
        shift = np.zeros(cap, dtype=np.int32)
        n = self.lib.L.dq_cuda_get_pass_times(self._h, _addr(ms), _addr(pairs), _addr(shift), cap)
        if n < 0:
            self._check(n)
        n = min(n, cap)
        return [(float(ms[i]), int(pairs[i]), int(shift[i])) for i in range(n)]

    def round_times(self):
        """[(ms, active, passes)] of every doubling round of the last single-device sort (timing must be on)."""
        cap = 256
        ms = np.zeros(cap, dtype=np.float32)
        active = np.zeros(cap, dtype=np.int64)
        passes = np.zeros(cap, dtype=np.int32)
        n = self.lib.L.dq_cuda_get_round_times(self._h, _addr(ms), _addr(active), _addr(passes), cap)
        if n < 0:
            self._check(n)
        n = min(n, cap)
        return [(float(ms[i]), int(active[i]), int(passes[i])) for i in range(n)]

    def set_timing(self, on):
        self._check(self.lib.L.dq_cuda_set_timing(self._h, 1 if on else 0))

    def pinned(self, shape, dtype):
        return PinnedArray(self.lib, shape, dtype)

    # ---- host-pointer entry points -------------------------------------------------------------
    def suffix_sort(self, text, sa_out):
        assert text.dtype == np.uint8 and sa_out.dtype == np.int32
        assert text.flags.c_contiguous and sa_out.flags.c_contiguous and sa_out.size >= text.size
        self._check(self.lib.L.dq_cuda_suffix_sort(self._h, _addr(text), text.size, _addr(sa_out)))

    def suffix_sort_batch(self, data, offsets, sa_out):
        """dq_cuda_suffix_sort_batch: text i is data[offsets[i]:offsets[i+1]], its suffix array (local indices) lands in
        sa_out[offsets[i]:offsets[i+1]].  offsets: int32, count+1 entries."""
        assert data.dtype == np.uint8 and offsets.dtype == np.int32 and sa_out.dtype == np.int32
        assert data.flags.c_contiguous and offsets.flags.c_contiguous and sa_out.flags.c_contiguous
        assert offsets.size >= 1 and data.size >= offsets[-1] and sa_out.size >= offsets[-1]
        self._check(self.lib.L.dq_cuda_suffix_sort_batch(self._h, _addr(data), _addr(offsets), offsets.size - 1,
                                                         _addr(sa_out)))

    def suffix_sort_lcp_batch(self, data, offsets, sa_out, lcp_out):
        """dq_cuda_suffix_sort_lcp_batch: suffix_sort_batch, and the LCP array of text i (lcp[0] = 0) in
        lcp_out[offsets[i]:offsets[i+1]]."""
        assert lcp_out.dtype == np.int32 and lcp_out.flags.c_contiguous and lcp_out.size >= offsets[-1]
        assert data.dtype == np.uint8 and offsets.dtype == np.int32 and sa_out.dtype == np.int32
        assert data.flags.c_contiguous and offsets.flags.c_contiguous and sa_out.flags.c_contiguous
        assert offsets.size >= 1 and data.size >= offsets[-1] and sa_out.size >= offsets[-1]
        self._check(self.lib.L.dq_cuda_suffix_sort_lcp_batch(self._h, _addr(data), _addr(offsets), offsets.size - 1,
                                                             _addr(sa_out), _addr(lcp_out)))

    def bsdiff_search(self, old, I, new, scan_begin, count, pos_out, len_out):
        assert old.dtype == np.uint8 and new.dtype == np.uint8
        assert pos_out.dtype == np.int32 and len_out.dtype == np.int32
        if I is not None:
            assert I.dtype == np.int32 and I.flags.c_contiguous and I.size >= old.size
        self._check(self.lib.L.dq_cuda_bsdiff_search(self._h, _addr(old), old.size, _addr(I), _addr(new), new.size,
                                                     scan_begin, count, _addr(pos_out), _addr(len_out)))

    def bsdiff_search_batch(self, olds, old_offsets, news, new_offsets, pos_out, len_out):
        """dq_cuda_bsdiff_search_batch: pair i is (olds[old_offsets[i]:old_offsets[i+1]], news[new_offsets[i]:
        new_offsets[i+1]]); its (pos, len) table of every scan position lands in pos_out / len_out[new_offsets[i]:
        new_offsets[i+1]].  Both offset arrays: int32, count+1 entries."""
        for a, dt in ((olds, np.uint8), (news, np.uint8), (old_offsets, np.int32), (new_offsets, np.int32),
                      (pos_out, np.int32), (len_out, np.int32)):
            assert a.dtype == dt and a.flags.c_contiguous
        assert old_offsets.size >= 1 and new_offsets.size == old_offsets.size
        assert olds.size >= old_offsets[-1] and news.size >= new_offsets[-1]
        assert pos_out.size >= new_offsets[-1] and len_out.size >= new_offsets[-1]
        self._check(self.lib.L.dq_cuda_bsdiff_search_batch(self._h, _addr(olds), _addr(old_offsets), _addr(news),
                                                           _addr(new_offsets), old_offsets.size - 1, _addr(pos_out),
                                                           _addr(len_out)))

    def greedy_emit(self, old, new, pos, ln):
        out = DqDiffStreams()
        with self._gate:
            self._check(self.lib.L.dq_cuda_greedy_emit(self._h, _addr(old), old.size, _addr(new), new.size,
                                                       _addr(pos), _addr(ln), ctypes.byref(out)))
            return self._streams(out)

    def bsdiff_streams(self, old, new, copy=True):
        """copy=False returns numpy views of the context-owned buffers (valid until the next call on this
        context) -- what a C caller of dq_cuda_bsdiff_streams gets; copy=True returns bytes objects."""
        out = DqDiffStreams()
        if copy:
            # the buffers belong to the context: copy them out before another thread's call can overwrite them
            with self._gate:
                self._check(self.lib.L.dq_cuda_bsdiff_streams(self._h, _addr(old), old.size, _addr(new), new.size,
                                                              ctypes.byref(out)))
                return self._streams(out)
        self._check(self.lib.L.dq_cuda_bsdiff_streams(self._h, _addr(old), old.size, _addr(new), new.size,
                                                      ctypes.byref(out)))
        if not copy:
            def view(ptr, n):
                if not n:
                    return np.zeros(0, dtype=np.uint8)
                return np.frombuffer((ctypes.c_uint8 * n).from_address(ptr), dtype=np.uint8)
            return {"ctrl": view(out.ctrl, out.ctrl_len), "diff": view(out.diff, out.diff_len),
                    "extra": view(out.extra, out.extra_len), "search_visits": out.search_visits}
        return self._streams(out)

    def lcp(self, text, I=None, out=None):
        """dq_cuda_lcp: LCP array (int32, n entries, lcp[0] = 0) of `text` under the suffix array I, or under the
        context's resident index (I=None; include/deltaq_cuda.h, "the resident index")."""
        n = text.size
        if out is None:
            out = np.empty(n, dtype=np.int32)
        assert out.dtype == np.int32 and out.size == n
        self._check(self.lib.L.dq_cuda_lcp(self._h, _addr(text), n, _addr(I) if I is not None else None, _addr(out)))
        return out

    def lcp_device(self, d_text, n, d_I, d_out):
        self._check(self.lib.L.dq_cuda_lcp_device(self._h, d_text, n, d_I, d_out))

    def bsdiff_patch(self, old, new, level=0):
        """dq_cuda_bsdiff_patch: the complete BSDIFF40 file for (old, new) as bytes -- sort, search and greedy loop as
        bsdiff_streams, then the three bzip2 sections produced block-parallel on the host."""
        p = ctypes.c_void_p()
        n = ctypes.c_int64()
        with self._gate:   # the patch buffer belongs to the context: copy it out before another call can replace it
            self._check(self.lib.L.dq_cuda_bsdiff_patch(self._h, _addr(old), old.size, _addr(new), new.size, int(level),
                                                        ctypes.byref(p), ctypes.byref(n)))
            return ctypes.string_at(p.value, n.value)

    @staticmethod
    def _streams(out):
        return {
            "ctrl": ctypes.string_at(out.ctrl, out.ctrl_len) if out.ctrl_len else b"",
            "diff": ctypes.string_at(out.diff, out.diff_len) if out.diff_len else b"",
            "extra": ctypes.string_at(out.extra, out.extra_len) if out.extra_len else b"",
            "search_visits": out.search_visits,
        }

    def radix_sort_pairs(self, keys, vals, key_bits=64):
        assert keys.dtype == np.uint64 and vals.dtype == np.uint32 and keys.size == vals.size
        self._check(self.lib.L.dq_cuda_radix_sort_pairs(self._h, _addr(keys), _addr(vals), keys.size, key_bits))

    # ---- multi-GPU building blocks (raw device addresses) ----------------------------------------
    def radix_sort_pairs_device(self, d_keys, d_vals, count, bit_lo, nbits, want_hist=False):
        hist = np.zeros(256, dtype=np.int64) if want_hist else None
        self._check(self.lib.L.dq_cuda_radix_sort_pairs_device(self._h, ctypes.c_void_p(d_keys), ctypes.c_void_p(d_vals),
                                                               count, bit_lo, nbits, _addr(hist)))
        return hist

    # ---- device-pointer entry points (raw addresses, e.g. torch.Tensor.data_ptr()) ---------------
    def suffix_sort_device(self, d_text, n, d_sa_out):
        self._check(self.lib.L.dq_cuda_suffix_sort_device(self._h, ctypes.c_void_p(d_text), n, ctypes.c_void_p(d_sa_out)))

    def bsdiff_search_device(self, d_old, n, d_I, d_new, m, scan_begin, count, d_pos, d_len):
        self._check(self.lib.L.dq_cuda_bsdiff_search_device(
            self._h, ctypes.c_void_p(d_old), n, ctypes.c_void_p(d_I) if d_I else None, ctypes.c_void_p(d_new), m,
            scan_begin, count, ctypes.c_void_p(d_pos), ctypes.c_void_p(d_len)))
