// CudaDiff.Create -- sibling of DeltaQ.BsDiff.Diff.Create (src/DeltaQ.BsDiff/Diff.cs:27-243) that runs the whole hot
// path inside libdeltaq_cuda: suffix sort of oldData (Diff.cs:90), Search at every scan position (Diff.cs:106) and the
// greedy scan / extend / emit loop (Diff.cs:100-223) in ONE native call, dq_cuda_bsdiff_streams, which returns the
// three UNCOMPRESSED streams.  What stays managed is what the reference does around them: the 32-byte header
// (Constants.cs:5-12, Diff.cs:54-70, :226-241) and the three BZip2OutputStream sections (Diff.cs:85-87) -- so the file
// is byte-identical to the reference's whenever the streams are, which tests/test_bsdiff_gpu.py checks.
//
// Source only (no .NET SDK in this repository's build image); see INTEGRATION.md section 6.
using System;
using System.IO;
using System.Runtime.InteropServices;
using ICSharpCode.SharpZipLib.BZip2;

namespace DeltaQ.SuffixSorting.Cuda;

[StructLayout(LayoutKind.Sequential)]
internal unsafe struct DqDiffStreams
{
    public byte* ctrl; public long ctrlLen;
    public byte* diff; public long diffLen;
    public byte* extra; public long extraLen;
    public long searchVisits;
}

internal static unsafe partial class Native
{
    [LibraryImport("deltaq_cuda")]
    internal static partial int dq_cuda_bsdiff_streams(IntPtr ctx, byte* old, int n, byte* @new, int m, DqDiffStreams* streams);

    // the whole file: streams + header + the three bzip2 sections produced block-parallel by the library (level 0 = chosen
    // for the machine's thread count; 9 = the bytes serial libbz2 -9 writes)
    [LibraryImport("deltaq_cuda")]
    internal static partial int dq_cuda_bsdiff_patch(IntPtr ctx, byte* old, int n, byte* @new, int m, int level, byte** patch, long* patchLen);

    // the (pos, len) tables of many pairs in one call: the sort and search of Diff.Create for a tree of files
    [LibraryImport("deltaq_cuda")]
    internal static partial int dq_cuda_bsdiff_search_batch(IntPtr ctx, byte* olds, int* oldOffsets, byte* news, int* newOffsets,
                                                            int count, int* posOut, int* lenOut);
}

/// <summary>Sibling of DeltaQ.BsDiff.Patch.Apply(ReadOnlyMemory&lt;byte&gt; input, ReadOnlyMemory&lt;byte&gt; diff, Stream output)
/// (Patch.cs:25-36): header checks, the three bzip2 sections decoded block-parallel and the add loop of Patch.cs:143-144 in
/// one native call, dq_cuda_bspatch.  Needs no device and no context.</summary>
public static unsafe class CudaPatch
{
    [DllImport("deltaq_cuda")]
    private static extern int dq_cuda_bspatch(byte* old, long n, byte* patch, long patchLen, int threads, byte* @out, long outCap, long* newSize);

    public static void Apply(ReadOnlyMemory<byte> input, ReadOnlyMemory<byte> diff, Stream output)
    {
        if (output == null) throw new ArgumentNullException(nameof(output));
        fixed (byte* o = input.Span) fixed (byte* p = diff.Span)
        {
            long size = -1;
            int rc = dq_cuda_bspatch(o, input.Length, p, diff.Length, 0, null, 0, &size);   // the header's newSize
            if (rc == -6 || size < 0) throw new InvalidOperationException("Corrupt patch");
            var result = new byte[size];
            fixed (byte* r = result)
                Native.Check(IntPtr.Zero, dq_cuda_bspatch(o, input.Length, p, diff.Length, 0, r, size, &size));
            output.Write(result);
        }
    }
}

public static unsafe class CudaDiff
{
    private const long Signature = 0x3034464649445342;   // "BSDIFF40", Constants.cs
    private const int HeaderSize = 32;

    /// <summary>Same contract as Diff.Create(oldData, newData, output, suffixSort): writes a BSDIFF40 delta to a
    /// seekable, writable stream.  The provider's native context does the sort, the search and the loop.</summary>
    public static void Create(ReadOnlySpan<byte> oldData, ReadOnlySpan<byte> newData, Stream output, CudaSuffixSort provider)
    {
        if (output == null) throw new ArgumentNullException(nameof(output));           // Diff.cs:29-52
        if (provider == null) throw new ArgumentNullException(nameof(provider));
        if (!output.CanSeek) throw new ArgumentException("Output stream must be seekable.", nameof(output));
        if (!output.CanWrite) throw new ArgumentException("Output stream must be writable.", nameof(output));

        Span<byte> header = stackalloc byte[HeaderSize];
        WritePackedLong(header, Signature);
        WritePackedLong(header[24..], newData.Length);
        long start = output.Position;
        output.Write(header);

        // The three buffers belong to the context and stay valid only until its next call, so the provider's gate is
        // held across the native call AND the compression: a second Create / Sort / SearchAll on the same provider
        // waits instead of overwriting streams that are still being read.
        lock (provider.Gate)
        {
            DqDiffStreams s;
            fixed (byte* o = oldData) fixed (byte* w = newData)
                Native.Check(provider.Handle, Native.dq_cuda_bsdiff_streams(provider.Handle, o, oldData.Length, w, newData.Length, &s));

            WriteSection(output, s.ctrl, s.ctrlLen);
            WritePackedLong(header[8..], output.Position - start - HeaderSize);              // Diff.cs:226-233
            long afterCtrl = output.Position;
            WriteSection(output, s.diff, s.diffLen);
            WritePackedLong(header[16..], output.Position - afterCtrl);
            WriteSection(output, s.extra, s.extraLen);
        }

        long end = output.Position;
        output.Position = start;
        output.Write(header);
        output.Position = end;
    }

    /// <summary>As Create, but the header and the three bzip2 sections are produced inside the library as well
    /// (dq_cuda_bsdiff_patch): the sections are cut where serial libbz2 would start its blocks, compressed on all
    /// cores and stitched into one ordinary stream each, which Patch.Apply's BZip2InputStream (Patch.cs:52-93) reads
    /// like any other.  On BASELINE's 16 MiB pair the managed sections above cost about a second; this call, tens of
    /// milliseconds.  The compressed bytes are libbz2's, not SharpZipLib's: the file differs from Diff.Create's in its
    /// compressed sections and decodes to the same streams.</summary>
    public static void CreateNative(ReadOnlySpan<byte> oldData, ReadOnlySpan<byte> newData, Stream output, CudaSuffixSort provider, int level = 0)
    {
        if (output == null) throw new ArgumentNullException(nameof(output));
        if (provider == null) throw new ArgumentNullException(nameof(provider));
        if (!output.CanSeek) throw new ArgumentException("Output stream must be seekable.", nameof(output));
        if (!output.CanWrite) throw new ArgumentException("Output stream must be writable.", nameof(output));
        lock (provider.Gate)
        {
            byte* patch;
            long len;
            fixed (byte* o = oldData) fixed (byte* w = newData)
                Native.Check(provider.Handle, Native.dq_cuda_bsdiff_patch(provider.Handle, o, oldData.Length, w, newData.Length, level, &patch, &len));
            const int chunk = 1 << 20;
            for (long at = 0; at < len; at += chunk)
                output.Write(new ReadOnlySpan<byte>(patch + at, (int)Math.Min(chunk, len - at)));
        }
    }

    /// <summary>Search(I, oldData, newData[scan..], 0, oldData.Length, out pos) of Diff.Create (Diff.cs:106) at every scan
    /// position of many pairs, in one native call (dq_cuda_bsdiff_search_batch).  Pair i is olds[oldOffsets[i] ..
    /// oldOffsets[i+1]) and news[newOffsets[i] .. newOffsets[i+1]); both offset spans have count + 1 entries, start at 0
    /// and never decrease.  pos / len[newOffsets[i] + k] receive what the search returns for scan position k of pair i,
    /// equal to sorting old_i alone and searching new_i against it.  The greedy loop and the sections stay per pair.</summary>
    public static void SearchMany(ReadOnlySpan<byte> olds, ReadOnlySpan<int> oldOffsets, ReadOnlySpan<byte> news,
                                  ReadOnlySpan<int> newOffsets, Span<int> pos, Span<int> len, CudaSuffixSort provider)
    {
        if (provider == null) throw new ArgumentNullException(nameof(provider));
        if (oldOffsets.Length == 0 || newOffsets.Length != oldOffsets.Length)
            throw new ArgumentException("Both offset spans must have count + 1 entries.", nameof(newOffsets));
        int total = newOffsets[^1];
        if (oldOffsets[^1] > olds.Length || total > news.Length || pos.Length < total || len.Length < total)
            throw new ArgumentException("The offsets reach past a buffer.");
        lock (provider.Gate)
        {
            fixed (byte* o = olds) fixed (int* oo = oldOffsets) fixed (byte* w = news) fixed (int* wo = newOffsets)
            fixed (int* p = pos) fixed (int* l = len)
                Native.Check(provider.Handle, Native.dq_cuda_bsdiff_search_batch(provider.Handle, o, oo, w, wo,
                                                                                  oldOffsets.Length - 1, p, l));
        }
    }

    private static void WriteSection(Stream output, byte* p, long len)
    {
        using var bz = new BZip2OutputStream(output) { IsStreamOwner = false };           // Diff.cs:85-87
        const int chunk = 1 << 20;
        for (long at = 0; at < len; at += chunk)
            bz.Write(new ReadOnlySpan<byte>(p + at, (int)Math.Min(chunk, len - at)));
    }

    // sign-magnitude, little endian: SpanExtensions.cs:7-30
    private static void WritePackedLong(Span<byte> b, long y)
    {
        ulong u = y < 0 ? (ulong)(-y) : (ulong)y;
        for (int i = 0; i < 8; ++i) b[i] = (byte)(u >> (8 * i));
        if (y < 0) b[7] |= 0x80;
    }
}
