"""Suffix and LCP arrays of many texts, one call: dq_cuda_suffix_sort_lcp_batch against a loop of dq_cuda_suffix_sort +
dq_cuda_lcp (I == NULL) per text, and against dq_cuda_suffix_sort_batch alone, so that the LCP step's own cost shows.

    python scripts/bench_batch_lcp.py [--reps R] [--only W1,W2,W3,W4] [--out results.jsonl]

Prints one JSON line per workload (and appends it to --out): the card's name and power limit (read in this run), the
per-text microseconds of the loop, of the LCP batch call and of the plain batch sort (host clock around calls that
synchronise before they return; median, min and max of R repetitions after one warm-up of each shape, the three arms
alternated), the loop / LCP-batch ratio, both batch calls' device_ms, and how many texts' suffix or LCP arrays differ
between the LCP batch and the loop (must be 0).  Texts, offsets and outputs sit in pinned buffers for every arm.  The
loop's figure includes two Python ctypes calls per text (a few microseconds each).

    W1  4,096 random texts of 16 B .. 8 KiB (one row per size)
    W2  random texts of 64 KiB and of 1 MiB, K = 64 MiB / size of them
    W3  the file-tree mix of bench_batch_sort.py: 2,000 texts, 16 B .. 1 MiB log-uniform, half random, half slices of
        the C2 exe-like old text
    W4  300 slices of the C2 exe-like old text, 16 B .. 1 MiB log-uniform: zero runs at many text ends and starts
"""
import argparse
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_batch_sort import MIB, file_tree_mix, gpu_info  # noqa: E402
from deltaq_b200 import CudaSuffixSort, workloads  # noqa: E402


class Batch:
    """The texts back to back in pinned memory, their offsets, and pinned suffix and LCP outputs for every arm."""

    def __init__(self, ctx, texts):
        self.count = len(texts)
        offs = np.zeros(self.count + 1, np.int64)
        np.cumsum([t.size for t in texts], out=offs[1:])
        self.total = t = int(offs[-1])
        size = max(t, 1)
        self._bufs = [ctx.pinned(size, np.uint8), ctx.pinned(self.count + 1, np.int32)] + \
            [ctx.pinned(size, np.int32) for _ in range(5)]
        self.data = self._bufs[0].array[:t]
        self.offsets = self._bufs[1].array
        self.sa_loop, self.lcp_loop, self.sa_batch, self.lcp_batch, self.sa_plain = (b.array[:t] for b in self._bufs[2:])
        self.offsets[:] = offs
        for i, x in enumerate(texts):
            self.data[offs[i]:offs[i + 1]] = x
        self.views = [(self.data[offs[i]:offs[i + 1]], self.sa_loop[offs[i]:offs[i + 1]],
                       self.lcp_loop[offs[i]:offs[i + 1]]) for i in range(self.count)]

    def free(self):
        for b in self._bufs:
            b.free()

    def mismatches(self):
        o = self.offsets
        return sum(not (np.array_equal(self.sa_loop[o[i]:o[i + 1]], self.sa_batch[o[i]:o[i + 1]]) and
                        np.array_equal(self.lcp_loop[o[i]:o[i + 1]], self.lcp_batch[o[i]:o[i + 1]]))
                   for i in range(self.count))


def measure(ctx, texts, reps):
    b = Batch(ctx, texts)
    try:
        def run_loop():
            t0 = time.perf_counter()
            for text, sa, lcp in b.views:
                ctx.suffix_sort(text, sa)
                if text.size:
                    ctx.lcp(text, None, lcp)
            return time.perf_counter() - t0

        def run_lcp_batch():
            t0 = time.perf_counter()
            ctx.suffix_sort_lcp_batch(b.data, b.offsets, b.sa_batch, b.lcp_batch)
            return time.perf_counter() - t0

        def run_sort_batch():
            t0 = time.perf_counter()
            ctx.suffix_sort_batch(b.data, b.offsets, b.sa_plain)
            return time.perf_counter() - t0

        run_loop()   # warm-up of every shape
        run_lcp_batch()
        run_sort_batch()
        loop_s, lcp_s, sort_s, lcp_ms, sort_ms = [], [], [], [], []
        for _ in range(reps):   # alternated, so drift on a shared host hits every arm
            loop_s.append(run_loop())
            lcp_s.append(run_lcp_batch())
            st = ctx.stats()
            lcp_ms.append(st["device_ms"])
            sort_s.append(run_sort_batch())
            sort_ms.append(ctx.stats()["device_ms"])
        per = lambda xs: {"median": round(float(np.median(xs)) * 1e6 / max(b.count, 1), 3),  # noqa: E731
                          "min": round(min(xs) * 1e6 / max(b.count, 1), 3),
                          "max": round(max(xs) * 1e6 / max(b.count, 1), 3)}
        ms = lambda xs: {"median": round(float(np.median(xs)), 3), "min": round(min(xs), 3),  # noqa: E731
                         "max": round(max(xs), 3)}
        return {"texts": b.count, "bytes": b.total, "loop_us_per_text": per(loop_s),
                "lcp_batch_us_per_text": per(lcp_s), "sort_batch_us_per_text": per(sort_s),
                "speedup": round(float(np.median(loop_s) / np.median(lcp_s)), 2),
                "lcp_batch_device_ms": ms(lcp_ms), "sort_batch_device_ms": ms(sort_ms),
                "rounds": st["rounds"], "kernel_launches": st["kernel_launches"],
                "mismatching_texts": int(b.mismatches())}
    finally:
        b.free()


def exe_slices(rng, count=300):
    old, _ = workloads.c2_exe_pair()
    sizes = np.exp(rng.uniform(np.log(16), np.log(MIB), count)).astype(np.int64)
    return [np.ascontiguousarray(old[p:p + int(n)]) for n, p in
            ((n, int(rng.integers(0, old.size - int(n)))) for n in sizes)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--only", default="W1,W2,W3,W4")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    only = set(args.only.split(","))
    name, power = gpu_info()
    out = open(args.out, "a") if args.out else None

    def emit(rec):
        rec = {"gpu": name, "power_limit": power, **rec}
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    with CudaSuffixSort(device=0) as sorter:
        ctx = sorter.context
        if "W1" in only:
            for size in (16, 64, 256, 1024, 4096, 8192):
                rng = np.random.default_rng(size)
                emit({"workload": "W1", "size": size,
                      **measure(ctx, list(rng.integers(0, 256, (4096, size), dtype=np.uint8)), args.reps)})
        if "W2" in only:
            for size in (64 * 1024, MIB):
                rng = np.random.default_rng(size)
                texts = list(rng.integers(0, 256, ((64 * MIB) // size, size), dtype=np.uint8))
                emit({"workload": "W2", "size": size, **measure(ctx, texts, args.reps)})
        if "W3" in only:
            emit({"workload": "W3", **measure(ctx, file_tree_mix(np.random.default_rng(2)), args.reps)})
        if "W4" in only:
            emit({"workload": "W4", **measure(ctx, exe_slices(np.random.default_rng(5)), args.reps)})
    if out:
        out.close()


if __name__ == "__main__":
    main()
