"""Many texts, one call: dq_cuda_suffix_sort_batch against a loop of dq_cuda_suffix_sort over the same texts.

    python scripts/bench_batch_sort.py [--reps R] [--only W1,W2,W3,W4] [--out results.jsonl]

Prints one JSON line per workload (and appends it to --out): the card's name and power limit (read in this run), the
per-text microseconds of the loop and of the batch call (host clock around calls that synchronise before they return;
median, min and max of R repetitions after one warm-up of each shape), their ratio, the batch call's device_ms, and how
many texts' arrays differ between the two (must be 0).  Texts, offsets and outputs sit in pinned buffers for both.
The loop's figure includes the Python ctypes call of every text (a few microseconds each).

    W1  for every size of `python -m deltaq_b200 bench`: K random texts, K = min(4096, max(1, 64 MiB / size))
    W2  a file-tree mix: 2,000 texts, 16 B .. 1 MiB log-uniform, half random, half slices of the C2 exe-like old text
    W3  W2 plus three random texts of 16, 24 and 40 MiB, above DQ_BATCH_SINGLE_MIN: both sides of the dispatch
    W4  the dispatch threshold: K = max(2, 128 / MiB) texts of 1 .. 64 MiB, random or slices of a 64 MiB exe-like text,
        with every text forced through the batched chunks
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from deltaq_b200 import CudaSuffixSort, workloads  # noqa: E402
from deltaq_b200.__main__ import benchmark_sizes  # noqa: E402

MIB = 1 << 20


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True, check=True).stdout.strip().splitlines()[0]
    name, power = [x.strip() for x in out.split(",")]
    return name, power


class Batch:
    """The texts back to back in pinned memory, their offsets, and pinned outputs for the loop and for the batch."""

    def __init__(self, ctx, texts):
        self.count = len(texts)
        offs = np.zeros(self.count + 1, np.int64)
        np.cumsum([t.size for t in texts], out=offs[1:])
        self.total = int(offs[-1])
        self._bufs = [ctx.pinned(max(self.total, 1), np.uint8), ctx.pinned(max(self.total, 1), np.int32),
                      ctx.pinned(max(self.total, 1), np.int32), ctx.pinned(self.count + 1, np.int32)]
        self.data = self._bufs[0].array[:self.total]
        self.sa_loop = self._bufs[1].array[:self.total]
        self.sa_batch = self._bufs[2].array[:self.total]
        self.offsets = self._bufs[3].array
        self.offsets[:] = offs
        for i, t in enumerate(texts):
            self.data[offs[i]:offs[i + 1]] = t
        self.views = [(self.data[offs[i]:offs[i + 1]], self.sa_loop[offs[i]:offs[i + 1]]) for i in range(self.count)]

    def free(self):
        for b in self._bufs:
            b.free()

    def mismatches(self):
        o = self.offsets
        return sum(not np.array_equal(self.sa_loop[o[i]:o[i + 1]], self.sa_batch[o[i]:o[i + 1]]) for i in range(self.count))


def measure(ctx, texts, reps, env=None):
    env = env or {}
    saved = {k: os.environ.get(k) for k in env}
    b = Batch(ctx, texts)
    try:
        def run_loop():
            t0 = time.perf_counter()
            for text, sa in b.views:
                ctx.suffix_sort(text, sa)
            return time.perf_counter() - t0

        def run_batch():
            os.environ.update(env)
            try:
                t0 = time.perf_counter()
                ctx.suffix_sort_batch(b.data, b.offsets, b.sa_batch)
                return time.perf_counter() - t0
            finally:
                for k, v in saved.items():
                    if v is None:
                        os.environ.pop(k, None)
                    else:
                        os.environ[k] = v

        run_loop()   # warm-up of every shape
        run_batch()
        loop_s, batch_s, dev_ms = [], [], []
        for _ in range(reps):   # alternated, so drift on a shared host hits both
            loop_s.append(run_loop())
            batch_s.append(run_batch())
            dev_ms.append(ctx.stats()["device_ms"])
        stats = ctx.stats()
        per = lambda xs: {"median": round(float(np.median(xs)) * 1e6 / max(b.count, 1), 3),  # noqa: E731
                          "min": round(min(xs) * 1e6 / max(b.count, 1), 3),
                          "max": round(max(xs) * 1e6 / max(b.count, 1), 3)}
        return {"texts": b.count, "bytes": b.total, "loop_us_per_text": per(loop_s), "batch_us_per_text": per(batch_s),
                "speedup": round(float(np.median(loop_s) / np.median(batch_s)), 2),
                "device_ms": {"median": round(float(np.median(dev_ms)), 3), "min": round(min(dev_ms), 3),
                              "max": round(max(dev_ms), 3)},
                "rounds": stats["rounds"], "kernel_launches": stats["kernel_launches"],
                "mismatching_texts": int(b.mismatches())}
    finally:
        b.free()


def file_tree_mix(rng, count=2000):
    old, _ = workloads.c2_exe_pair()
    sizes = np.exp(rng.uniform(np.log(16), np.log(MIB), count)).astype(np.int64)
    texts = []
    for i, n in enumerate(sizes):
        n = int(n)
        if i % 2:
            p = int(rng.integers(0, old.size - n))
            texts.append(np.ascontiguousarray(old[p:p + n]))
        else:
            texts.append(rng.integers(0, 256, n, dtype=np.uint8))
    return texts


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
            for size in benchmark_sizes():
                k = min(4096, max(1, (64 * MIB) // size)) if size else 4096
                rng = np.random.default_rng(size)
                texts = list(rng.integers(0, 256, (k, size), dtype=np.uint8))
                emit({"workload": "W1", "size": size, **measure(ctx, texts, args.reps)})
        if "W2" in only or "W3" in only:
            w2 = file_tree_mix(np.random.default_rng(2))
            if "W2" in only:
                emit({"workload": "W2", **measure(ctx, w2, args.reps)})
            if "W3" in only:
                rng = np.random.default_rng(3)
                big = [rng.integers(0, 256, n, dtype=np.uint8) for n in (16 * MIB, 24 * MIB, 40 * MIB)]
                emit({"workload": "W3", **measure(ctx, w2[:1000] + big + w2[1000:], args.reps)})
        if "W4" in only:
            exe = workloads.c2_exe_pair(64 * MIB, 64 * MIB + 1)[0]
            for kind in ("random", "exe"):
                for mib in (1, 2, 4, 8, 16, 32, 64):
                    k = max(2, 128 // mib)
                    rng = np.random.default_rng(mib)
                    if kind == "random":
                        texts = list(rng.integers(0, 256, (k, mib * MIB), dtype=np.uint8))
                    else:   # slices of an exe-like text: zero runs, which the single-text path refines by run length
                        starts = rng.integers(0, exe.size - mib * MIB + 1, k)
                        texts = [np.ascontiguousarray(exe[p:p + mib * MIB]) for p in starts]
                    emit({"workload": "W4", "kind": kind, "size": mib * MIB, "forced": "chunks",
                          **measure(ctx, texts, args.reps, env={"DQ_BATCH_SINGLE_MIN": str(2 ** 31 - 1)})})
    if out:
        out.close()


if __name__ == "__main__":
    main()
