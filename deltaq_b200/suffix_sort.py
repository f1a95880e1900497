"""CudaSuffixSort -- host-side mirror of the reference's suffix-sort provider contract.

Mirrors ``DeltaQ.SuffixSorting.ISuffixSort`` (/root/reference/src/DeltaQ.SuffixSorting.Abstractions/
ISuffixSort.cs:9-28) as the reference's providers implement it (LibDivSufSort.cs:10-32, SAIS.cs:11-45):

    Sort(ReadOnlySpan<byte> text) -> IMemoryOwner<int>          ->  sort(text) -> SuffixArrayOwner
    Sort(ReadOnlySpan<byte> text, Span<int> suffixes)           ->  sort(text, suffixes)

and, for many texts in one call (no counterpart in the reference): sort_many(texts) -> SuffixArraysOwner and
sort_many(texts, suffixes), with their LCP arrays too when lcp is given.

Same argument meaning and error behaviour: the two-buffer overload raises ``ValueError("Text and suffix
buffers should have the same length")`` (ArgumentException, LibDivSufSort.cs:23-31); empty input yields
an empty owner; only ``suffixes[0:n]`` is written.  The C# provider that binds the same C ABI is in
csharp/DeltaQ.SuffixSorting.Cuda/ (see INTEGRATION.md).
"""
import numpy as np

from . import _native

LENGTH_MISMATCH = "Text and suffix buffers should have the same length"  # LibDivSufSort.cs:31, SAIS.cs:44


def as_bytes_array(buf, name="text"):
    if buf is None:
        raise TypeError(f"{name} must not be None")  # ArgumentNullException
    if isinstance(buf, np.ndarray):
        if buf.dtype != np.uint8:
            raise TypeError(f"{name} must be a uint8 buffer")
        return np.ascontiguousarray(buf).reshape(-1)
    return np.frombuffer(bytes(buf) if not isinstance(buf, (bytes, bytearray, memoryview)) else buf, dtype=np.uint8)


class SuffixArrayOwner:
    """IMemoryOwner<int> analogue: ``.memory`` is an int32 array of length n over pinned host memory;
    ``dispose()`` (or the context manager) releases it (README.md:108-110 of the reference)."""

    def __init__(self, pinned, n, release=None):
        self._pinned = pinned
        self._release = release        # hands the buffer back to the provider's pool; None: free it
        self.memory = pinned.array[:n]

    def dispose(self):
        if self._pinned is not None:
            self.memory = None
            pinned, self._pinned = self._pinned, None
            if self._release is not None:
                self._release(pinned)
            else:
                pinned.free()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.dispose()


class SuffixArraysOwner(SuffixArrayOwner):
    """What sort_many(texts) returns: one pinned int32 buffer holding the suffix arrays of all texts back to back.
    ``.memory`` is the flat array, ``.offsets`` (int32, count+1 entries) where each text's array starts, and
    ``.arrays`` the per-text views.  With lcp=True the same buffer holds the LCP arrays after them: ``.lcp_memory``
    (flat) and ``.lcp_arrays`` (per text), else both are None.  ``dispose()`` releases the buffer."""

    def __init__(self, pinned, offsets, release=None, lcp=False):
        total = int(offsets[-1])
        super().__init__(pinned, total, release)
        self.offsets = offsets
        self.arrays = self._split(self.memory)
        self.lcp_memory = pinned.array[total:2 * total] if lcp else None
        self.lcp_arrays = self._split(self.lcp_memory) if lcp else None

    def _split(self, flat):
        return [flat[self.offsets[i]:self.offsets[i + 1]] for i in range(self.offsets.size - 1)]

    def dispose(self):
        self.arrays = self.lcp_arrays = self.lcp_memory = None
        super().dispose()


class CudaSuffixSort:
    """ISuffixSort provider backed by libdeltaq_cuda.  Holds a native context (device, stream, scratch);
    disposable; one call in flight per instance.  Raises if the CUDA library or device is missing."""

    # The owners Sort(text) hands out sit on pinned host memory, and pinning is dear (cudaHostAlloc of a few MiB costs as
    # much as sorting them).  The reference rents its owners from a pool (MemoryOwner<int>.Allocate -> ArrayPool,
    # LibDivSufSort.cs:14), so Sort(asset).Dispose() in a loop -- its benchmark, SuffixSortingBenchmarks.cs:63-73 -- reuses
    # one array; so does this provider: a disposed owner's buffer is kept (a few, of moderate size) for the next Sort.
    _POOL_KEEP = 4
    _POOL_MAX_BYTES = 256 << 20

    def __init__(self, device=None, _lib=None):
        import threading
        self._ctx = _native.Context(device=device, lib=_lib)
        self._pool = []
        self._pool_lock = threading.Lock()
        self._closed = False

    def _rent(self, n):
        """A pinned int32 buffer of at least n entries: the smallest kept one that fits without being more than twice too
        big, else a new one (capacities below 16 Mi entries are rounded up to a power of two, like ArrayPool's buckets)."""
        with self._pool_lock:
            fit = [b for b in self._pool if n <= b.array.size <= max(2 * n, 1024)]
            if fit:
                best = min(fit, key=lambda b: b.array.size)
                self._pool.remove(best)
                return best
        cap = max(1, n)
        if cap < (16 << 20):
            cap = 1 << (cap - 1).bit_length()
        return self._ctx.pinned(cap, np.int32)

    def _give_back(self, pinned):
        with self._pool_lock:
            if not self._closed and pinned.array.nbytes <= self._POOL_MAX_BYTES and len(self._pool) < self._POOL_KEEP:
                self._pool.append(pinned)
                return
        pinned.free()

    # -- IDisposable
    def dispose(self):
        with self._pool_lock:
            self._closed = True
            pool, self._pool = self._pool, []
        for b in pool:
            b.free()
        self._ctx.close()

    close = dispose

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.dispose()

    @property
    def context(self):
        return self._ctx

    def stats(self):
        return self._ctx.stats()

    def sort(self, text, suffixes=None):
        t = as_bytes_array(text)
        if suffixes is None:
            # overload 1: ISuffixSort.cs:18 -- allocate, sort, hand the owner to the caller
            pinned = self._rent(t.size)
            owner = SuffixArrayOwner(pinned, t.size, release=self._give_back)
            try:
                self._ctx.suffix_sort(t, pinned.array)
            except BaseException:
                owner.dispose()
                raise
            return owner
        # overload 2: ISuffixSort.cs:27
        if suffixes is None or not isinstance(suffixes, np.ndarray) or suffixes.dtype != np.int32:
            raise TypeError("suffixes must be an int32 numpy array")
        if suffixes.size != t.size:
            raise ValueError(LENGTH_MISMATCH)
        if not suffixes.flags.c_contiguous:
            raise ValueError("suffixes must be contiguous")
        self._ctx.suffix_sort(t, suffixes)
        return None

    def sort_many(self, texts, suffixes=None, lcp=None):
        """Suffix arrays of many texts in one native call (dq_cuda_suffix_sort_batch), mirroring the two sort overloads:
        without `suffixes` it returns a SuffixArraysOwner over one pinned buffer rented from the pool; with `suffixes`
        (int32, the total length of the texts) the arrays are written there back to back and None is returned.  Every
        array holds indices local to its text and equals what sort(text) gives.
        `lcp` asks for the LCP array of every text as well (dq_cuda_suffix_sort_lcp_batch), each equal to what
        lcp_array(text) gives: lcp=True without `suffixes` (the owner's .lcp_arrays), or an int32 array like `suffixes`
        that receives them back to back."""
        if texts is None:
            raise TypeError("texts must not be None")
        arrs = [as_bytes_array(t, "texts[%d]" % i) for i, t in enumerate(texts)]
        offsets = np.zeros(len(arrs) + 1, dtype=np.int64)
        np.cumsum([a.size for a in arrs], out=offsets[1:])
        if offsets[-1] > np.iinfo(np.int32).max:
            raise ValueError("the texts of one batch must hold fewer than 2**31 bytes in all")
        offsets = offsets.astype(np.int32)
        data = np.concatenate(arrs) if arrs else np.zeros(0, np.uint8)
        total = int(offsets[-1])
        if suffixes is None:
            if isinstance(lcp, np.ndarray):
                raise TypeError("without suffixes, lcp must be True or False")
            pinned = self._rent(2 * total if lcp else total)
            owner = SuffixArraysOwner(pinned, offsets, release=self._give_back, lcp=bool(lcp))
            try:
                if lcp:
                    self._ctx.suffix_sort_lcp_batch(data, offsets, pinned.array, owner.lcp_memory)
                else:
                    self._ctx.suffix_sort_batch(data, offsets, pinned.array)
            except BaseException:
                owner.dispose()
                raise
            return owner
        if lcp is False:
            lcp = None
        for name, buf in (("suffixes", suffixes), ("lcp", lcp)):
            if buf is None and name == "lcp":
                continue
            if not isinstance(buf, np.ndarray) or buf.dtype != np.int32:
                raise TypeError(f"{name} must be an int32 numpy array")
            if buf.size != total:
                raise ValueError(LENGTH_MISMATCH)
            if not buf.flags.c_contiguous:
                raise ValueError(f"{name} must be contiguous")
        if lcp is None:
            self._ctx.suffix_sort_batch(data, offsets, suffixes)
        else:
            self._ctx.suffix_sort_lcp_batch(data, offsets, suffixes, lcp)
        return None

    def lcp_array(self, text, suffixes=None):
        """LCP array of `text` (int32, lcp[0] = 0, lcp[r] = common prefix of suffixes r-1 and r in sorted order): the
        extension SURVEY.md 8(f) rank 4 proposes for ISuffixSort providers.  suffixes=None uses the suffix array this
        provider's last sort(text, ...) left on the device; otherwise any suffix array of `text` (validated)."""
        t = as_bytes_array(text)
        I = None
        if suffixes is not None:
            I = np.ascontiguousarray(suffixes, dtype=np.int32)
            if I.size != t.size:
                raise ValueError(LENGTH_MISMATCH)
        return self._ctx.lcp(t, I)
