"""Host-side mirror of DeltaQ.BsDiff.Diff / Patch for the accelerated path.

``Diff.create(old, new, output, suffix_sort)`` mirrors ``Diff.Create(ReadOnlySpan<byte> oldData,
ReadOnlySpan<byte> newData, Stream output, ISuffixSort suffixSort)``
(/root/reference/src/DeltaQ.BsDiff/Diff.cs:27-242): same argument checks and error classes, same BSDIFF40
container (Diff.cs:54-70, :226-241, Constants.cs:5-12).  The suffix sort (Diff.cs:90) and every
``Search`` call (Diff.cs:106) run on the GPU; the greedy scan/emit loop (Diff.cs:100-223) runs on the
host inside libdeltaq_cuda (csrc/dq_diff_host.h), consuming the bulk (pos, len) table.

The three streams are compressed by libbz2, block-parallel on the host (csrc/dq_bz2_host.h: the bytes equal what
serial libbz2 writes at the chosen level).  The reference uses SharpZipLib 1.4.2 (un-vendored third party);
compressed bytes are not claimed identical to it -- the uncompressed ctrl/diff/extra streams and the header fields
are (tests/test_bsdiff_gpu.py).

``Patch.apply`` mirrors Patch.Apply (Patch.cs:25-168) through dq_cuda_bspatch (sections decoded block-parallel on the
host, native add loop); it is not on the hot path and serves the reference's round-trip tests (BsDiffTests.cs:30-78).
"""
import bz2
import io

import numpy as np

from . import _native
from .suffix_sort import CudaSuffixSort, as_bytes_array

HEADER_SIZE = 32                      # Constants.cs:7
SIGNATURE = 0x3034464649445342        # "BSDIFF40", Constants.cs:12


def write_packed_long(y):
    """SpanExtensions.WritePackedLong (SpanExtensions.cs:7-30): sign-magnitude, little-endian."""
    u = -y if y < 0 else y
    b = bytearray(u.to_bytes(8, "little"))
    if y < 0:
        b[7] |= 0x80
    return bytes(b)


def read_packed_long(b):
    """SpanExtensions.ReadPackedLong (SpanExtensions.cs:32-44)."""
    y = int.from_bytes(b[:7], "little") | ((b[7] & 0x7F) << 56)
    return -y if b[7] & 0x80 else y


_search_engine = None


def _engine():
    """The CudaSuffixSort whose context serves the match search when Diff.create is handed some OTHER
    ISuffixSort provider (the reference's Diff.Create accepts any, Diff.cs:27)."""
    global _search_engine
    if _search_engine is None:
        _search_engine = CudaSuffixSort()
    return _search_engine


def create_streams(old, new, suffix_sort):
    """Uncompressed ctrl / diff / extra streams of Diff.Create for (old, new).

    With a CudaSuffixSort: sort + search on the GPU in one native call (the suffix array never leaves the device),
    greedy loop on the host.  With any other provider exposing ``sort(text, suffixes)`` (the ISuffixSort contract):
    that provider sorts (Diff.cs:90), the GPU answers every Search (Diff.cs:106) over its suffix array, and the
    same host loop consumes the table."""
    o = as_bytes_array(old, "oldData")
    w = as_bytes_array(new, "newData")
    if isinstance(suffix_sort, CudaSuffixSort):
        return suffix_sort.context.bsdiff_streams(o, w)
    if not hasattr(suffix_sort, "sort"):
        raise TypeError("suffixSort must implement sort(text, suffixes)")
    I = np.zeros(o.size + 1, dtype=np.int32)          # Diff.cs:78: n+1 entries, cleared
    suffix_sort.sort(o, I[:o.size])                    # Diff.cs:90
    ctx = _engine().context
    pos = np.empty(w.size, dtype=np.int32)
    ln = np.empty(w.size, dtype=np.int32)
    ctx.bsdiff_search(o, I, w, 0, w.size, pos, ln)
    return ctx.greedy_emit(o, w, pos, ln)


def search_all(old, new, suffix_sort, I=None, scan_begin=0, count=None):
    """(pos, len) of Diff.Search at every scan position in [scan_begin, scan_begin+count).  I: the (n+1)-entry
    buffer of Diff.cs:78, or None to sort `old` with suffix_sort first."""
    o = as_bytes_array(old, "oldData")
    w = as_bytes_array(new, "newData")
    ctx = suffix_sort.context
    if count is None:
        count = w.size - scan_begin
    if I is None:
        I = np.zeros(o.size + 1, dtype=np.int32)
        suffix_sort.sort(o, I[:o.size])
        I_arg = None        # the suffix array is still resident on the device
    else:
        I_arg = np.ascontiguousarray(I, dtype=np.int32)
        if I_arg.size != o.size + 1:
            raise ValueError("I must have oldData.Length + 1 entries (Diff.cs:78)")
    pos = np.empty(count, dtype=np.int32)
    ln = np.empty(count, dtype=np.int32)
    ctx.bsdiff_search(o, I_arg, w, scan_begin, count, pos, ln)
    return pos, ln


def _flatten(arrays):
    """Concatenation of uint8 arrays and its int32 offsets (count + 1 entries)."""
    offsets = np.zeros(len(arrays) + 1, dtype=np.int64)
    np.cumsum([a.size for a in arrays], out=offsets[1:])
    if offsets[-1] > np.iinfo(np.int32).max:
        raise ValueError("the batch holds more than 2^31 - 1 bytes")
    flat = np.concatenate(arrays) if arrays else np.zeros(0, dtype=np.uint8)
    return np.ascontiguousarray(flat, dtype=np.uint8), offsets.astype(np.int32)


def search_many(pairs, suffix_sort):
    """search_all(old, new, suffix_sort) for every (old, new) in `pairs`, in one native call
    (dq_cuda_bsdiff_search_batch): a list of per-pair (pos, len) arrays, views of one flat buffer each."""
    if not isinstance(suffix_sort, CudaSuffixSort):
        raise TypeError("search_many needs a CudaSuffixSort: the pairs are sorted and searched on its device")
    olds = [as_bytes_array(o, "oldData") for o, _ in pairs]
    news = [as_bytes_array(w, "newData") for _, w in pairs]
    old_flat, old_offsets = _flatten(olds)
    new_flat, new_offsets = _flatten(news)
    pos = np.empty(int(new_offsets[-1]), dtype=np.int32)
    ln = np.empty(int(new_offsets[-1]), dtype=np.int32)
    suffix_sort.context.bsdiff_search_batch(old_flat, old_offsets, new_flat, new_offsets, pos, ln)
    return [(pos[new_offsets[i]:new_offsets[i + 1]], ln[new_offsets[i]:new_offsets[i + 1]]) for i in range(len(pairs))]


def _patch_file(new_size, streams, lib):
    """The BSDIFF40 file of Diff.create (Diff.cs:54-70, :226-241): header, then the three bzip2 sections."""
    ctrl, diff, extra = _native.bz2_compress([streams["ctrl"], streams["diff"], streams["extra"]], lib=lib)
    header = bytearray(HEADER_SIZE)
    header[0:8] = write_packed_long(SIGNATURE)
    header[8:16] = write_packed_long(len(ctrl))
    header[16:24] = write_packed_long(len(diff))
    header[24:32] = write_packed_long(new_size)
    return bytes(header) + ctrl + diff + extra


class Diff:
    @staticmethod
    def create_many(pairs, suffix_sort):
        """Diff.create for every (old, new) in `pairs`: a list of BSDIFF40 files (bytes), each identical to what
        Diff.create writes for that pair.  The sorts and searches of all pairs are one search_many; the greedy loop and
        the bzip2 sections run per pair."""
        olds = [as_bytes_array(o, "oldData") for o, _ in pairs]
        news = [as_bytes_array(w, "newData") for _, w in pairs]
        tables = search_many(list(zip(olds, news)), suffix_sort)
        ctx = suffix_sort.context
        return [_patch_file(w.size, ctx.greedy_emit(o, w, pos, ln), ctx.lib) for o, w, (pos, ln) in zip(olds, news, tables)]

    @staticmethod
    def create(old_data, new_data, output, suffix_sort):
        # argument checks: Diff.cs:29-52
        if output is None:
            raise TypeError("output must not be None")          # ArgumentNullException(nameof(output))
        if suffix_sort is None:
            raise TypeError("suffixSort must not be None")      # ArgumentNullException(nameof(suffixSort))
        if not (hasattr(output, "seekable") and output.seekable()):
            raise ValueError("Output stream must be seekable.")  # ArgumentException
        if not (hasattr(output, "writable") and output.writable()):
            raise ValueError("Output stream must be writable.")
        o = as_bytes_array(old_data, "oldData")
        w = as_bytes_array(new_data, "newData")

        if isinstance(suffix_sort, CudaSuffixSort):
            # one native call: streams as create_streams(), header and sections assembled in the library
            # (dq_cuda_bsdiff_patch); the bytes and the final stream position are those of the general path below
            output.write(suffix_sort.context.bsdiff_patch(o, w))
            # the reference ends with Seek calls (Diff.cs:237-241), which push a buffering stream's bytes down: its own
            # test reads the wrapped MemoryStream right after Create (BsPatchTests.cs:25-29)
            if hasattr(output, "flush"):
                output.flush()
            return

        header = bytearray(HEADER_SIZE)
        header[0:8] = write_packed_long(SIGNATURE)
        header[24:32] = write_packed_long(w.size)
        start = output.tell()
        output.write(bytes(header))

        streams = create_streams(o, w, suffix_sort)
        # Diff.cs:85-87: three bzip2 sections -- here one crew of host threads over the blocks of all three
        ctrl, diff, extra = _native.bz2_compress([streams["ctrl"], streams["diff"], streams["extra"]])

        output.write(ctrl)
        header[8:16] = write_packed_long(len(ctrl))
        output.write(diff)
        header[16:24] = write_packed_long(len(diff))
        output.write(extra)
        end = output.tell()
        output.seek(start)
        output.write(bytes(header))
        output.seek(end)


class Patch:
    @staticmethod
    def apply(old_data, patch, output):
        """Patch.Apply, both overloads (Patch.cs:25-50):
        (input bytes, patch bytes, output stream) -- Patch.cs:25-36;
        (input stream, open_patch_stream(offset, length) -> stream, output stream) -- Patch.cs:44-50, where length 0 means
        "the rest of the patch" (Patch.cs:15-17) and the streams must be readable and seekable (:60-63, :97-100)."""
        if output is None:
            raise TypeError("output must not be None")
        if hasattr(output, "writable") and not output.writable():
            raise ValueError("Output stream must be writable")          # Patch.cs:101-102
        if callable(patch):
            old_data, patch = Patch._read_streams(old_data, patch)
        o = as_bytes_array(old_data, "input")
        # header checks (:52-70), the three sections un-bzip2'ed block-parallel, the add loop (:95-168): one native call
        out = _native.bspatch(o, np.frombuffer(bytes(patch), dtype=np.uint8))
        output.write(out.tobytes())
        if hasattr(output, "flush"):
            output.flush()

    @staticmethod
    def _read_streams(input_stream, open_patch_stream):
        """The stream overload's reading side: CreatePatchStreams (Patch.cs:52-93) up to the compressed sections."""
        if input_stream is None:
            raise TypeError("input must not be None")
        with open_patch_stream(0, HEADER_SIZE) as hs:
            if not hs.readable():
                raise ValueError("Patch stream must be readable")       # ArgumentException, Patch.cs:60-61
            if not hs.seekable():
                raise ValueError("Patch stream must be seekable")       # Patch.cs:62-63
            header = hs.read(HEADER_SIZE)
        if len(header) < HEADER_SIZE or read_packed_long(header[0:8]) != SIGNATURE:
            raise RuntimeError("Corrupt patch")                         # InvalidOperationException, Patch.cs:68-70
        ctrl_len = read_packed_long(header[8:16])
        diff_len = read_packed_long(header[16:24])
        if ctrl_len < 0 or diff_len < 0 or read_packed_long(header[24:32]) < 0:
            raise RuntimeError("Corrupt patch")                         # Patch.cs:77-78
        parts = [bytes(header)]
        for off, ln in ((HEADER_SIZE, ctrl_len), (HEADER_SIZE + ctrl_len, diff_len), (HEADER_SIZE + ctrl_len + diff_len, 0)):
            with open_patch_stream(off, ln) as st:                      # Patch.cs:82-85
                part = st.read() if ln == 0 else st.read(ln)
            if ln and len(part) != ln:
                raise RuntimeError("Corrupt patch")
            parts.append(part)
        if not input_stream.readable():
            raise ValueError("Input stream must be readable")           # Patch.cs:97-98
        if not input_stream.seekable():
            raise ValueError("Input stream must be seekable")           # Patch.cs:99-100
        return np.frombuffer(input_stream.read(), dtype=np.uint8), b"".join(parts)

    @staticmethod
    def apply_reference_order(old_data, patch, output):
        """The same with the sections decoded by Python's bz2 (serial libbz2) and the header parsed here: an independent
        reader of the files Diff.create writes, used by the tests."""
        o = as_bytes_array(old_data, "input")
        p = bytes(patch)
        header = p[:HEADER_SIZE]
        if len(header) < HEADER_SIZE or read_packed_long(header[0:8]) != SIGNATURE:
            raise RuntimeError("Corrupt patch")                 # InvalidOperationException, Patch.cs:68-70
        ctrl_len = read_packed_long(header[8:16])
        diff_len = read_packed_long(header[16:24])
        new_size = read_packed_long(header[24:32])
        if ctrl_len < 0 or diff_len < 0 or new_size < 0:
            raise RuntimeError("Corrupt patch")
        ctrl = bz2.decompress(p[HEADER_SIZE:HEADER_SIZE + ctrl_len])
        diff = bz2.decompress(p[HEADER_SIZE + ctrl_len:HEADER_SIZE + ctrl_len + diff_len])
        extra = bz2.decompress(p[HEADER_SIZE + ctrl_len + diff_len:])
        out = apply_streams(o, ctrl, diff, extra, new_size)
        output.write(out)
        if hasattr(output, "flush"):
            output.flush()


def apply_streams(old, ctrl, diff, extra, new_size, lib=None):
    """Patch.ApplyInternal (Patch.cs:95-168) on uncompressed streams: the native add loop (dq_cuda_patch_apply).
    Returns the bytes of the new file; raises RuntimeError("Corrupt patch") like the reference."""
    o = as_bytes_array(old, "input")
    return _native.patch_apply(o, ctrl, diff, extra, new_size, lib=lib).tobytes()
