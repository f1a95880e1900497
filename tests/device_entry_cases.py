"""Checks of the device-pointer entry points (dq_cuda_*_device), shared by the emulator and the GPU tests.

Every check takes `mem`, which places arrays where the library reads device pointers: CUDA tensors on the GPU
(CudaMem), numpy arrays on the emulator (HostMem: there a device pointer is a host address).  Every output buffer is
larger than the result and filled with a sentinel, so a check sees both what a call wrote and what it must not touch."""
import ctypes

import numpy as np

import oracle

SENTINEL = -7

# radix fields (bit_lo, nbits): every plan shape -- one pass of 1..8 bits, uneven splits (9, 12, 13, 63 bits), fields
# that start inside a byte, at bit 32 and at the top of the key
RADIX_FIELDS = [(0, 64), (0, 1), (0, 7), (0, 8), (0, 9), (0, 13), (3, 9), (8, 12), (29, 3), (32, 32), (56, 8), (60, 4),
                (1, 63)]
RADIX_DISTRIBUTIONS = ["uniform", "few_digits", "constant", "sorted", "reverse", "one_value_99pct"]


class HostMem:
    """numpy arrays: the emulator's device pointers are host addresses."""

    def put(self, a):
        return np.array(a, copy=True)

    def ptr(self, buf, byte_offset=0):
        return buf.ctypes.data + byte_offset

    def get(self, buf):
        return np.array(buf, copy=True)


class CudaMem:
    """CUDA tensors, passed by data_ptr() as bench.py does.  The library works on its own non-blocking stream, so an
    upload is finished before its pointer is handed over."""
    _VIEW = {np.dtype(np.uint8): np.uint8, np.dtype(np.int32): np.int32, np.dtype(np.uint32): np.int32,
             np.dtype(np.int64): np.int64, np.dtype(np.uint64): np.int64}

    def __init__(self):
        import torch
        self.torch = torch

    def put(self, a):
        a = np.ascontiguousarray(a)
        t = self.torch.from_numpy(a.view(self._VIEW[a.dtype]).copy()).cuda()
        self.torch.cuda.synchronize()
        return t, a.dtype

    def ptr(self, buf, byte_offset=0):
        return buf[0].data_ptr() + byte_offset

    def get(self, buf):
        self.torch.cuda.synchronize()
        return buf[0].cpu().numpy().view(buf[1])


def text_buffer(mem, t, offset, pad=16):
    """`t` at byte `offset` of a larger buffer of other bytes -> (buffer, pointer to t)."""
    raw = np.random.default_rng(offset).integers(0, 256, t.size + offset + pad, dtype=np.uint8)
    raw[offset:offset + t.size] = t
    buf = mem.put(raw)
    return buf, mem.ptr(buf, offset)


def out_buffer(mem, count, front=1, back=8):
    """int32 output of `count` entries at element `front` of a sentinel-filled buffer -> (buffer, pointer)."""
    buf = mem.put(np.full(front + count + back, SENTINEL, np.int32))
    return buf, mem.ptr(buf, 4 * front)


def written(mem, buf, count, front=1):
    """The `count` entries a call wrote; asserts that every other slot still holds the sentinel."""
    a = mem.get(buf)
    assert np.all(a[:front] == SENTINEL) and np.all(a[front + count:] == SENTINEL), "wrote outside its output"
    return a[front:front + count]


# ---- dq_cuda_suffix_sort_device ---------------------------------------------------------------------------------
def check_suffix_sort(ctx, mem, t, offsets=(0,), ref=None):
    """suffix_sort_device of `t` placed at each byte offset, into an output at int32 offset 1, against SA-IS."""
    ref = oracle.sais(t) if ref is None else ref
    for off in offsets:
        text_buf, p_text = text_buffer(mem, t, off)
        sa_buf, p_sa = out_buffer(mem, t.size)
        ctx.suffix_sort_device(p_text, t.size, p_sa)
        assert np.array_equal(written(mem, sa_buf, t.size), ref), f"text offset {off}"
    return ref


# ---- dq_cuda_bsdiff_search_device ------------------------------------------------------------------------------
def scan_ranges(m):
    """(scan_begin, count): the whole scan, a middle sub-range, the last position alone, nothing."""
    out = [(0, m), (m // 3, m // 2), (m - 1, 1), (m // 2, 0)]
    return [(b, c) for b, c in out if b >= 0 and b + c <= m]


def search_into(ctx, mem, p_old, n, p_I, p_new, m, b, c):
    pos_buf, p_pos = out_buffer(mem, c)
    len_buf, p_len = out_buffer(mem, c)
    ctx.bsdiff_search_device(p_old, n, p_I, p_new, m, b, c, p_pos, p_len)
    assert ctx.stats()["search_queries"] == c
    return written(mem, pos_buf, c), written(mem, len_buf, c)


def check_search(ctx, mem, old, new, old_offset=3):
    """Sort `old` (device pointers), then search every scan range with the index the sort left (I = NULL) and with a
    caller suffix array of exactly n entries, against the literal replay of Diff.Search."""
    n, m = old.size, new.size
    old_buf, p_old = text_buffer(mem, old, old_offset)
    new_buf = mem.put(new if m else np.zeros(1, np.uint8))
    p_new = mem.ptr(new_buf)
    sa = check_suffix_sort(ctx, mem, old, (old_offset,))
    rp, rl = oracle.search_all(oracle.make_I(sa), old, new)
    I_buf = mem.put(sa if n else np.zeros(1, np.int32))            # n entries: nothing follows the last one
    for b, c in scan_ranges(m):
        pos, ln = search_into(ctx, mem, p_old, n, None, p_new, m, b, c)
        assert np.array_equal(pos, rp[b:b + c]) and np.array_equal(ln, rl[b:b + c]), ("resident index", b, c)
    for b, c in scan_ranges(m):
        pos, ln = search_into(ctx, mem, p_old, n, mem.ptr(I_buf) if n else None, p_new, m, b, c)
        assert np.array_equal(pos, rp[b:b + c]) and np.array_equal(ln, rl[b:b + c]), ("caller I", b, c)


# ---- dq_cuda_lcp_device ----------------------------------------------------------------------------------------
def check_lcp(ctx, mem, old, new):
    """lcp_device under the resident index and under a caller array of n entries; a following search with I = NULL
    still equals the oracle."""
    n, m = old.size, new.size
    old_buf, p_old = text_buffer(mem, old, 5)
    sa = check_suffix_sort(ctx, mem, old, (5,))
    ref = oracle.lcp_array(old, sa)
    lcp_buf, p_lcp = out_buffer(mem, n)
    ctx.lcp_device(p_old, n, None, p_lcp)
    assert np.array_equal(written(mem, lcp_buf, n), ref), "resident index"
    rp, rl = oracle.search_all(oracle.make_I(sa), old, new)
    new_buf = mem.put(new)
    pos, ln = search_into(ctx, mem, p_old, n, None, mem.ptr(new_buf), m, 0, m)
    assert np.array_equal(pos, rp) and np.array_equal(ln, rl), "search after lcp (resident)"
    I_buf = mem.put(sa)
    lcp_buf, p_lcp = out_buffer(mem, n)
    ctx.lcp_device(p_old, n, mem.ptr(I_buf), p_lcp)
    assert np.array_equal(written(mem, lcp_buf, n), ref), "caller I"
    pos, ln = search_into(ctx, mem, p_old, n, None, mem.ptr(new_buf), m, 0, m)
    assert np.array_equal(pos, rp) and np.array_equal(ln, rl), "search after lcp (caller I)"


# ---- dq_cuda_radix_sort_pairs_device ---------------------------------------------------------------------------
def radix_keys(count, bit_lo, nbits, dist, seed):
    """Random 64-bit keys whose field [bit_lo, bit_lo+nbits) follows `dist`; the bits outside it stay random."""
    rng = np.random.default_rng(seed)
    fmask = (1 << nbits) - 1
    if dist == "uniform":
        field = rng.integers(0, 1 << 63, count, dtype=np.uint64) ^ (rng.integers(0, 2, count, dtype=np.uint64) << np.uint64(63))
    elif dist == "few_digits":      # at most 8 distinct values, so at most 8 distinct digits in every pass: MATCH ranking
        field = rng.choice(rng.integers(0, 1 << 63, 8, dtype=np.uint64) * np.uint64(3), count)
    elif dist == "constant":
        field = np.full(count, rng.integers(0, 1 << 63, dtype=np.uint64), np.uint64)
    elif dist in ("sorted", "reverse"):
        field = np.sort(rng.integers(0, 1 << 63, count, dtype=np.uint64) & np.uint64(fmask))
        if dist == "reverse":
            field = field[::-1].copy()
    elif dist == "one_value_99pct":
        field = np.full(count, rng.integers(0, 1 << 63, dtype=np.uint64), np.uint64)
        few = rng.random(count) < 0.01
        field[few] = rng.integers(0, 1 << 63, int(few.sum()), dtype=np.uint64)
    else:
        raise ValueError(dist)
    field &= np.uint64(fmask)
    keep = np.uint64(~(fmask << bit_lo) & ((1 << 64) - 1))
    return (rng.integers(0, 1 << 63, count, dtype=np.uint64) * np.uint64(2) + np.uint64(1)) & keep | \
        (field << np.uint64(bit_lo))


def radix_sort_device(ctx, d_keys, d_vals, count, bit_lo, nbits, hist_fill=None):
    """dq_cuda_radix_sort_pairs_device with a histogram buffer pre-filled with `hist_fill` (None: no histogram)."""
    hist = None if hist_fill is None else np.full(256, hist_fill, np.int64)
    rc = ctx.lib.L.dq_cuda_radix_sort_pairs_device(ctx._h, ctypes.c_void_p(d_keys), ctypes.c_void_p(d_vals), count,
                                                  bit_lo, nbits, None if hist is None else hist.ctypes.data)
    ctx._check(rc)
    return hist


def check_radix(ctx, mem, count, bit_lo, nbits, dist, seed=0, pad=5):
    """Stable sort of (key, value) pairs by the field, against np.argsort(kind="stable"): whole keys move, the first
    digit's histogram is the header's, and nothing past `count` is touched."""
    keys = radix_keys(count, bit_lo, nbits, dist, seed)
    vals = np.random.default_rng(seed + 1).permutation(count).astype(np.uint32)
    kbuf = mem.put(np.concatenate([keys, np.full(pad, 0xDEADBEEFDEADBEEF, np.uint64)]))
    vbuf = mem.put(np.concatenate([vals, np.full(pad, 0xFEEDF00D, np.uint32)]))
    hist = radix_sort_device(ctx, mem.ptr(kbuf), mem.ptr(vbuf), count, bit_lo, nbits, hist_fill=-1)
    field = (keys >> np.uint64(bit_lo)) & np.uint64((1 << nbits) - 1)
    order = np.argsort(field, kind="stable")
    k2, v2 = mem.get(kbuf), mem.get(vbuf)
    what = (count, bit_lo, nbits, dist)
    assert np.all(k2[count:] == np.uint64(0xDEADBEEFDEADBEEF)) and np.all(v2[count:] == 0xFEEDF00D), what
    assert np.array_equal(k2[:count], keys[order]), what
    assert np.array_equal(v2[:count], vals[order]), what
    w = min(nbits, 8)
    digit = ((keys >> np.uint64(bit_lo)) & np.uint64((1 << w) - 1)).astype(np.int64)
    assert np.array_equal(hist, np.bincount(digit, minlength=256)), ("histogram",) + what


def check_radix_noop(ctx, mem):
    """nbits = 0 and count = 0 leave the arrays as they were and report an all-zero histogram."""
    keys = radix_keys(1000, 0, 64, "uniform", 9)
    vals = np.arange(1000, dtype=np.uint32)[::-1].copy()
    kbuf, vbuf = mem.put(keys), mem.put(vals)
    for count, bit_lo, nbits in [(1000, 0, 0), (1000, 64, 0), (1000, 17, 0), (0, 0, 64), (0, 5, 9)]:
        hist = radix_sort_device(ctx, mem.ptr(kbuf), mem.ptr(vbuf), count, bit_lo, nbits, hist_fill=-1)
        assert np.all(hist == 0), (count, bit_lo, nbits)
        assert np.array_equal(mem.get(kbuf), keys) and np.array_equal(mem.get(vbuf), vals), (count, bit_lo, nbits)
    hist = radix_sort_device(ctx, 0, 0, 0, 3, 9, hist_fill=-1)      # null arrays are fine when there is nothing to sort
    assert np.all(hist == 0)


def check_radix_keeps_resident_index(ctx, mem, old, new):
    """sort -> radix_sort_pairs_device -> search with I = NULL: the radix sort works in its own scratch and leaves the
    suffix array of `old` resident."""
    n, m = old.size, new.size
    old_buf, p_old = text_buffer(mem, old, 2)
    sa = check_suffix_sort(ctx, mem, old, (2,))
    count = 3 * 4096 + 7
    keys = radix_keys(count, 0, 64, "uniform", 4)
    kbuf, vbuf = mem.put(keys), mem.put(np.arange(count, dtype=np.uint32))
    radix_sort_device(ctx, mem.ptr(kbuf), mem.ptr(vbuf), count, 0, 64, hist_fill=-1)
    assert np.array_equal(mem.get(kbuf), np.sort(keys))
    new_buf = mem.put(new)
    pos, ln = search_into(ctx, mem, p_old, n, None, mem.ptr(new_buf), m, 0, m)
    rp, rl = oracle.search_all(oracle.make_I(sa), old, new)
    assert np.array_equal(pos, rp) and np.array_equal(ln, rl)


# ---- a device group of logical shards --------------------------------------------------------------------------
def check_group(ctx, mem, old, new):
    """On a group whose shard threshold is below n: suffix_sort_device runs the group sort, bsdiff_search_device with
    I = NULL the sharded search, lcp_device the group's LCP array -- all on device pointers."""
    n, m = old.size, new.size
    old_buf, p_old = text_buffer(mem, old, 1)
    sa = check_suffix_sort(ctx, mem, old, (1,))
    rp, rl = oracle.search_all(oracle.make_I(sa), old, new)
    new_buf = mem.put(new)
    for b, c in scan_ranges(m):
        pos, ln = search_into(ctx, mem, p_old, n, None, mem.ptr(new_buf), m, b, c)
        assert np.array_equal(pos, rp[b:b + c]) and np.array_equal(ln, rl[b:b + c]), (b, c)
    lcp_buf, p_lcp = out_buffer(mem, n)
    ctx.lcp_device(p_old, n, None, p_lcp)
    assert np.array_equal(written(mem, lcp_buf, n), oracle.lcp_array(old, sa))
