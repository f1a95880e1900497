// DeltaQ.SuffixSorting.Cuda -- ISuffixSort provider backed by libdeltaq_cuda (B200, sm_100a).
//
// Source only: this repository's build image has no .NET SDK, so this project is compiled wherever one
// exists (see INTEGRATION.md).  It implements the reference's plug-in contract unchanged
// (src/DeltaQ.SuffixSorting.Abstractions/ISuffixSort.cs:9-28) with the same argument checks as the
// reference's own providers (LibDivSufSort.cs:21-31, SAIS.cs:25-45), and adds the one optional hook the
// reference lacks (Diff.Search is private static, Diff.cs:267): ISuffixSearch.
using System;
using System.Buffers;
using System.Collections.Generic;
using System.Runtime.InteropServices;

namespace DeltaQ.SuffixSorting.Cuda;

/// <summary>Optional companion of ISuffixSort: bulk evaluation of Diff.Search (Diff.cs:267-298) for every
/// scan position. Diff.Create probes `suffixSort is ISuffixSearch` and, when present, replaces the call at
/// Diff.cs:106 by reads of (pos[scan], len[scan]).</summary>
public interface ISuffixSearch
{
    void SearchAll(ReadOnlySpan<int> I, ReadOnlySpan<byte> oldData, ReadOnlySpan<byte> newData,
                   Span<int> pos, Span<int> len);
}

internal static unsafe partial class Native
{
    private const string Lib = "deltaq_cuda"; // libdeltaq_cuda.so

    [LibraryImport(Lib)] internal static partial int dq_cuda_create(out IntPtr ctx, int* devices, int ndev);
    [LibraryImport(Lib)] internal static partial int dq_cuda_destroy(IntPtr ctx);
    [LibraryImport(Lib)] internal static partial IntPtr dq_cuda_last_error(IntPtr ctx);
    [LibraryImport(Lib)] internal static partial int dq_cuda_host_alloc(out IntPtr p, nuint bytes);
    [LibraryImport(Lib)] internal static partial int dq_cuda_host_free(IntPtr p);
    [LibraryImport(Lib)] internal static partial int dq_cuda_suffix_sort(IntPtr ctx, byte* text, int n, int* saOut);
    [LibraryImport(Lib)] internal static partial int dq_cuda_suffix_sort_batch(IntPtr ctx, byte* texts, int* offsets,
        int count, int* saOut);
    [LibraryImport(Lib)] internal static partial int dq_cuda_suffix_sort_lcp_batch(IntPtr ctx, byte* texts, int* offsets,
        int count, int* saOut, int* lcpOut);
    [LibraryImport(Lib)] internal static partial int dq_cuda_bsdiff_search(IntPtr ctx, byte* old, int n, int* iOrNull,
        byte* @new, int m, int scanBegin, int count, int* posOut, int* lenOut);
    [LibraryImport(Lib)] internal static partial int dq_cuda_lcp(IntPtr ctx, byte* text, int n, int* iOrNull, int* lcpOut);
    [LibraryImport(Lib)] internal static partial int dq_cuda_patch_apply(byte* old, long n, byte* ctrl, long ctrlLen,
        byte* diff, long diffLen, byte* extra, long extraLen, byte* @out, long newSize);

    internal static void Check(IntPtr ctx, int status)
    {
        if (status == 0) return;
        var msg = Marshal.PtrToStringUTF8(dq_cuda_last_error(ctx)) ?? "libdeltaq_cuda error";
        throw status switch
        {
            -1 => new ArgumentException(msg),
            -2 => new OutOfMemoryException(msg),
            -6 => new InvalidOperationException("Corrupt patch"),   // Patch.cs:68-70, :128, :151
            _ => new InvalidOperationException(msg), // -3 CUDA, -4 no device (there is no CPU fallback), -5 internal
        };
    }
}

/// <summary>IMemoryOwner&lt;int&gt; over cudaHostAlloc memory: the D2H copy of the suffix array lands in it
/// directly (no staging copy).</summary>
internal sealed unsafe class PinnedSuffixOwner : MemoryManager<int>
{
    private IntPtr _p;
    private readonly int _length;
    private readonly int _capacity;
    private readonly PinnedPool? _pool;

    public PinnedSuffixOwner(int length, PinnedPool? pool = null)
    {
        _length = length;
        _pool = pool;
        (_p, _capacity) = pool?.Rent(length) ?? PinnedPool.Allocate(length);
    }

    public override Span<int> GetSpan() => new((void*)_p, _length);
    public override MemoryHandle Pin(int elementIndex = 0) => new((int*)_p + elementIndex);
    public override void Unpin() { }

    protected override void Dispose(bool disposing)
    {
        if (_p == IntPtr.Zero) return;
        if (_pool is null || !_pool.Return(_p, _capacity)) Native.dq_cuda_host_free(_p);
        _p = IntPtr.Zero;
    }
}

/// <summary>The provider's ArrayPool: the reference rents its owners from one (MemoryOwner&lt;int&gt;.Allocate,
/// LibDivSufSort.cs:14), so Sort(asset).Dispose() in a loop (SuffixSortingBenchmarks.cs:63-73) reuses one array. Pinning is
/// dear -- cudaHostAlloc of a few MiB costs as much as sorting them -- so a disposed owner's buffer is kept (a few, of
/// moderate size) for the next Sort. Same policy as deltaq_b200/suffix_sort.py.</summary>
internal sealed unsafe class PinnedPool
{
    private const int Keep = 4;
    private const long MaxBytes = 256L << 20;
    private readonly List<(IntPtr p, int capacity)> _free = new();
    private bool _closed;

    public static (IntPtr, int) Allocate(int length)
    {
        int cap = Math.Max(1, length);
        if (cap < (16 << 20)) cap = (int)System.Numerics.BitOperations.RoundUpToPowerOf2((uint)cap);
        Native.Check(IntPtr.Zero, Native.dq_cuda_host_alloc(out var p, (nuint)cap * sizeof(int)));
        return (p, cap);
    }

    public (IntPtr, int) Rent(int length)
    {
        lock (_free)
        {
            int best = -1;
            for (int i = 0; i < _free.Count; i++)
                if (_free[i].capacity >= length && _free[i].capacity <= Math.Max(2L * length, 1024) &&
                    (best < 0 || _free[i].capacity < _free[best].capacity)) best = i;
            if (best >= 0) { var hit = _free[best]; _free.RemoveAt(best); return hit; }
        }
        return Allocate(length);
    }

    public bool Return(IntPtr p, int capacity)
    {
        lock (_free)
        {
            if (_closed || (long)capacity * sizeof(int) > MaxBytes || _free.Count >= Keep) return false;
            _free.Add((p, capacity));
            return true;
        }
    }

    public void Close()
    {
        lock (_free)
        {
            _closed = true;
            foreach (var (p, _) in _free) Native.dq_cuda_host_free(p);
            _free.Clear();
        }
    }
}

public sealed unsafe class CudaSuffixSort : ISuffixSort, ISuffixSearch, IDisposable
{
    private IntPtr _ctx;
    internal IntPtr Handle => _ctx;   // CudaDiff.Create drives the same native context
    private readonly PinnedPool _pool = new();
    private readonly object _gate = new();
    internal object Gate => _gate;    // CudaDiff.Create holds it while it reads the context-owned streams

    public CudaSuffixSort(int device = -1)
    {
        int dev = device;
        Native.Check(IntPtr.Zero, device < 0 ? Native.dq_cuda_create(out _ctx, null, 0)
                                             : Native.dq_cuda_create(out _ctx, &dev, 1));
    }

    /// <summary>A device GROUP: this one provider, in this one process, drives all listed GPUs (dq_cuda_create with
    /// ndev &gt; 1). Nothing else changes for the caller: texts of at least DQ_SHARD_MIN bytes (default 128 MiB) are
    /// sorted by all of them, SearchAll shards the scan positions, smaller inputs stay on devices[0].</summary>
    public CudaSuffixSort(ReadOnlySpan<int> devices)
    {
        fixed (int* d = devices)
            Native.Check(IntPtr.Zero, Native.dq_cuda_create(out _ctx, d, devices.Length));
    }

    public IMemoryOwner<int> Sort(ReadOnlySpan<byte> textBuffer)
    {
        var owner = new PinnedSuffixOwner(textBuffer.Length, _pool);
        try { Sort(textBuffer, owner.GetSpan()); }
        catch { ((IDisposable)owner).Dispose(); throw; }
        return owner;
    }

    public void Sort(ReadOnlySpan<byte> textBuffer, Span<int> suffixBuffer)
    {
        if (textBuffer.Length != suffixBuffer.Length)
            throw new ArgumentException("Text and suffix buffers should have the same length");
        lock (_gate)
            fixed (byte* t = textBuffer)
            fixed (int* sa = suffixBuffer)
                Native.Check(_ctx, Native.dq_cuda_suffix_sort(_ctx, t, textBuffer.Length, sa));
    }

    /// <summary>Suffix arrays of many texts in one native call (dq_cuda_suffix_sort_batch). Text i is
    /// packedTexts[offsets[i]..offsets[i+1]); its suffix array, with indices local to text i, is written to
    /// suffixes[offsets[i]..offsets[i+1]) and equals what Sort gives for that text alone. offsets has one entry more
    /// than there are texts, starts at 0, never decreases and ends at packedTexts.Length.</summary>
    public void SortMany(ReadOnlySpan<byte> packedTexts, ReadOnlySpan<int> offsets, Span<int> suffixes)
    {
        if (packedTexts.Length != suffixes.Length)
            throw new ArgumentException("Text and suffix buffers should have the same length");
        if (offsets.Length == 0 || offsets[^1] != packedTexts.Length)
            throw new ArgumentException("offsets must have count + 1 entries and end at packedTexts.Length");
        lock (_gate)
            fixed (byte* t = packedTexts) fixed (int* o = offsets) fixed (int* sa = suffixes)
                Native.Check(_ctx, Native.dq_cuda_suffix_sort_batch(_ctx, t, o, offsets.Length - 1, sa));
    }

    /// <summary>SortMany, and the LCP array of every text as well (dq_cuda_suffix_sort_lcp_batch):
    /// lcp[offsets[i] + r] is the common prefix length of suffixes r-1 and r of text i alone (0 for r = 0), what
    /// LcpArray gives for that text.</summary>
    public void SortMany(ReadOnlySpan<byte> packedTexts, ReadOnlySpan<int> offsets, Span<int> suffixes, Span<int> lcp)
    {
        if (packedTexts.Length != suffixes.Length || packedTexts.Length != lcp.Length)
            throw new ArgumentException("Text, suffix and LCP buffers should have the same length");
        if (offsets.Length == 0 || offsets[^1] != packedTexts.Length)
            throw new ArgumentException("offsets must have count + 1 entries and end at packedTexts.Length");
        lock (_gate)
            fixed (byte* t = packedTexts) fixed (int* o = offsets) fixed (int* sa = suffixes) fixed (int* l = lcp)
                Native.Check(_ctx, Native.dq_cuda_suffix_sort_lcp_batch(_ctx, t, o, offsets.Length - 1, sa, l));
    }

    /// <summary>Suffix arrays of many texts in one native call, back to back in one owner rented from the pinned pool:
    /// text i's array is Memory.Slice(s_i, texts[i].Length) with s_i the sum of the lengths of the texts before it.</summary>
    public IMemoryOwner<int> SortMany(IReadOnlyList<ReadOnlyMemory<byte>> texts) => SortManyPacked(texts, default, false);

    /// <summary>The same, and the LCP arrays of the texts, back to back in lcp (the total length of the texts) at the
    /// same positions as the suffix arrays in the owner.</summary>
    public IMemoryOwner<int> SortMany(IReadOnlyList<ReadOnlyMemory<byte>> texts, Span<int> lcp) =>
        SortManyPacked(texts, lcp, true);

    private IMemoryOwner<int> SortManyPacked(IReadOnlyList<ReadOnlyMemory<byte>> texts, Span<int> lcp, bool withLcp)
    {
        ArgumentNullException.ThrowIfNull(texts);
        var offsets = new int[texts.Count + 1];
        long total = 0;
        for (int i = 0; i < texts.Count; i++)
        {
            total += texts[i].Length;
            if (total > int.MaxValue) throw new ArgumentException("the texts of one batch must hold fewer than 2^31 bytes");
            offsets[i + 1] = (int)total;
        }
        var packed = ArrayPool<byte>.Shared.Rent((int)total);
        try
        {
            for (int i = 0; i < texts.Count; i++) texts[i].Span.CopyTo(packed.AsSpan(offsets[i]));
            var owner = new PinnedSuffixOwner((int)total, _pool);
            try
            {
                if (withLcp) SortMany(packed.AsSpan(0, (int)total), offsets, owner.GetSpan(), lcp);
                else SortMany(packed.AsSpan(0, (int)total), offsets, owner.GetSpan());
            }
            catch { ((IDisposable)owner).Dispose(); throw; }
            return owner;
        }
        finally { ArrayPool<byte>.Shared.Return(packed); }
    }

    public void SearchAll(ReadOnlySpan<int> I, ReadOnlySpan<byte> oldData, ReadOnlySpan<byte> newData,
                          Span<int> pos, Span<int> len)
    {
        if (I.Length != oldData.Length + 1) throw new ArgumentException("I must have oldData.Length + 1 entries");
        if (pos.Length != newData.Length || len.Length != newData.Length)
            throw new ArgumentException("pos/len must have newData.Length entries");
        lock (_gate)
            fixed (int* i = I) fixed (byte* o = oldData) fixed (byte* w = newData)
            fixed (int* p = pos) fixed (int* l = len)
                Native.Check(_ctx, Native.dq_cuda_bsdiff_search(_ctx, o, oldData.Length, i, w, newData.Length,
                                                                0, newData.Length, p, l));
    }

    /// <summary>LCP array of textBuffer under suffixBuffer (any suffix array of it; validated natively):
    /// lcp[0] = 0, lcp[r] = common prefix length of suffixes suffixBuffer[r-1] and suffixBuffer[r].  An empty
    /// suffixBuffer means "the array my last Sort of this text left on the device".</summary>
    public void LcpArray(ReadOnlySpan<byte> textBuffer, ReadOnlySpan<int> suffixBuffer, Span<int> lcp)
    {
        if (lcp.Length != textBuffer.Length || (suffixBuffer.Length != 0 && suffixBuffer.Length != textBuffer.Length))
            throw new ArgumentException("Text, suffix and LCP buffers should have the same length");
        lock (_gate)
            fixed (byte* t = textBuffer) fixed (int* i = suffixBuffer) fixed (int* l = lcp)
                Native.Check(_ctx, Native.dq_cuda_lcp(_ctx, t, textBuffer.Length, suffixBuffer.Length == 0 ? null : i, l));
    }

    public void Dispose()
    {
        _pool.Close();
        if (_ctx != IntPtr.Zero) { Native.dq_cuda_destroy(_ctx); _ctx = IntPtr.Zero; }
    }
}
