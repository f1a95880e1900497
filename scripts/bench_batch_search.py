"""The (pos, len) tables of many file pairs, one call: dq_cuda_bsdiff_search_batch against a loop of dq_cuda_suffix_sort +
dq_cuda_bsdiff_search (I == NULL) per pair; and whole patches, Diff.create_many against a loop of Diff.create.

    python scripts/bench_batch_search.py [--reps R] [--only W1,W2,W3,W4,W5] [--out results.jsonl]

Prints one JSON line per workload (and appends it to --out): the card's name and power limit (read in this run), the
per-pair microseconds of the search loop, of the batch call, of the Diff.create loop and of Diff.create_many (host clock
around calls that synchronise before they return; median, min and max of R repetitions after one warm-up of each shape,
the arms alternated), the loop / batch ratios, the batch's device_ms (sorts) and search_ms, and how many pairs' tables
or patch files differ between the batch and the loop (must be 0).  Inputs and the search tables sit in pinned buffers.
The loops' figures include Python ctypes calls per pair (a few microseconds each); both Diff arms run the host greedy
loop and bzip2 per pair.

    W1  4,096 pairs of 16 B .. 8 KiB (one row per size): random olds, news mutated from them
    W2  mutated pairs of 64 KiB and of 1 MiB, K = 64 MiB / size of them
    W3  the file-tree mix of bench_batch_sort.py (2,000 olds, 16 B .. 1 MiB, half random, half exe-like), mutated news
    W4  identical pairs (new == old) of 64 KiB and of 1 MiB, K = 64 MiB / size: every super of the head level starts
        cold inside a match as long as the pair (the batch has no seed level)
    W5  unrelated pairs: 4,096 random olds and news of 4 KiB
"""
import argparse
import io
import json
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_batch_sort import MIB, file_tree_mix, gpu_info  # noqa: E402
from deltaq_b200 import CudaSuffixSort, workloads  # noqa: E402
from deltaq_b200.bsdiff import Diff  # noqa: E402


def pinned_flat(ctx, arrays, keep):
    offs = np.zeros(len(arrays) + 1, np.int64)
    np.cumsum([a.size for a in arrays], out=offs[1:])
    buf = ctx.pinned(max(int(offs[-1]), 1), np.uint8)
    ob = ctx.pinned(len(arrays) + 1, np.int32)
    keep += [buf, ob]
    data, o = buf.array[:int(offs[-1])], ob.array
    o[:] = offs
    for i, a in enumerate(arrays):
        data[offs[i]:offs[i + 1]] = a
    return data, o


def measure(sorter, pairs, reps, diffs=True):
    ctx = sorter.context
    keep = []
    try:
        olds, oo = pinned_flat(ctx, [p[0] for p in pairs], keep)
        news, no = pinned_flat(ctx, [p[1] for p in pairs], keep)
        total = int(no[-1])
        bufs = [ctx.pinned(max(total, 1), np.int32) for _ in range(4)]
        keep += bufs
        pos_loop, len_loop, pos_batch, len_batch = (b.array[:total] for b in bufs)
        scratch = ctx.pinned(max(int(max((p[0].size for p in pairs), default=1)), 1), np.int32)
        keep.append(scratch)
        views = [(olds[oo[i]:oo[i + 1]], news[no[i]:no[i + 1]], pos_loop[no[i]:no[i + 1]], len_loop[no[i]:no[i + 1]])
                 for i in range(len(pairs))]

        def run_loop():
            t0 = time.perf_counter()
            for o, w, p, ln in views:
                ctx.suffix_sort(o, scratch.array[:o.size])
                ctx.bsdiff_search(o, None, w, 0, w.size, p, ln)
            return time.perf_counter() - t0

        def run_batch():
            t0 = time.perf_counter()
            ctx.bsdiff_search_batch(olds, oo, news, no, pos_batch, len_batch)
            return time.perf_counter() - t0

        files = {}

        def run_create_loop():
            t0 = time.perf_counter()
            out = []
            for o, w, _, _ in views:
                f = io.BytesIO()
                Diff.create(o, w, f, sorter)
                out.append(f.getvalue())
            files["loop"] = out
            return time.perf_counter() - t0

        def run_create_many():
            t0 = time.perf_counter()
            files["many"] = Diff.create_many([(o, w) for o, w, _, _ in views], sorter)
            return time.perf_counter() - t0

        arms = [run_loop, run_batch] + ([run_create_loop, run_create_many] if diffs else [])
        for arm in arms:   # warm-up of every shape
            arm()
        times = {arm.__name__: [] for arm in arms}
        dev_ms, search_ms = [], []
        for _ in range(reps):   # alternated, so drift on a shared host hits every arm
            for arm in arms:
                times[arm.__name__].append(arm())
                if arm is run_batch:
                    st = ctx.stats()
                    dev_ms.append(st["device_ms"])
                    search_ms.append(st["search_ms"])
        n = max(len(pairs), 1)
        per = lambda xs: {"median": round(float(np.median(xs)) * 1e6 / n, 3), "min": round(min(xs) * 1e6 / n, 3),  # noqa: E731
                          "max": round(max(xs) * 1e6 / n, 3)}
        ms = lambda xs: {"median": round(float(np.median(xs)), 3), "min": round(min(xs), 3), "max": round(max(xs), 3)}  # noqa: E731
        bad = sum(not (np.array_equal(pos_loop[no[i]:no[i + 1]], pos_batch[no[i]:no[i + 1]]) and
                       np.array_equal(len_loop[no[i]:no[i + 1]], len_batch[no[i]:no[i + 1]])) for i in range(len(pairs)))
        rec = {"pairs": len(pairs), "old_bytes": int(oo[-1]), "new_bytes": total,
               "loop_us_per_pair": per(times["run_loop"]), "batch_us_per_pair": per(times["run_batch"]),
               "speedup": round(float(np.median(times["run_loop"]) / np.median(times["run_batch"])), 2),
               "batch_device_ms": ms(dev_ms), "batch_search_ms": ms(search_ms), "rounds": st["rounds"],
               "kernel_launches": st["kernel_launches"], "mismatching_pairs": int(bad)}
        if diffs:
            rec.update({"create_loop_us_per_pair": per(times["run_create_loop"]),
                        "create_many_us_per_pair": per(times["run_create_many"]),
                        "create_speedup": round(float(np.median(times["run_create_loop"]) /
                                                      np.median(times["run_create_many"])), 2),
                        "mismatching_files": int(sum(a != b for a, b in zip(files["loop"], files["many"])))})
        return rec
    finally:
        for b in keep:
            b.free()


def mutated(rng, olds):
    return [workloads._mutate(o, rng, max(1, o.size + int(rng.integers(-8, 9))), regions=max(1, o.size // 4096))
            for o in olds]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--only", default="W1,W2,W3,W4,W5")
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
        if "W1" in only:
            for size in (16, 256, 1024, 8192):
                rng = np.random.default_rng(size)
                olds = list(rng.integers(0, 256, (4096, size), dtype=np.uint8))
                emit({"workload": "W1", "size": size, **measure(sorter, list(zip(olds, mutated(rng, olds))), args.reps)})
        if "W2" in only:
            for size in (64 * 1024, MIB):
                rng = np.random.default_rng(size)
                olds = list(rng.integers(0, 256, ((64 * MIB) // size, size), dtype=np.uint8))
                emit({"workload": "W2", "size": size, **measure(sorter, list(zip(olds, mutated(rng, olds))), args.reps)})
        if "W3" in only:
            rng = np.random.default_rng(2)
            olds = file_tree_mix(rng)
            emit({"workload": "W3", **measure(sorter, list(zip(olds, mutated(rng, olds))), args.reps)})
        if "W4" in only:
            for size in (64 * 1024, MIB):
                rng = np.random.default_rng(size + 1)
                olds = list(rng.integers(0, 256, ((64 * MIB) // size, size), dtype=np.uint8))
                emit({"workload": "W4", "size": size,
                      **measure(sorter, [(o, o.copy()) for o in olds], args.reps, diffs=False)})
        if "W5" in only:
            rng = np.random.default_rng(9)
            olds = list(rng.integers(0, 256, (4096, 4096), dtype=np.uint8))
            news = list(rng.integers(0, 256, (4096, 4096), dtype=np.uint8))
            emit({"workload": "W5", **measure(sorter, list(zip(olds, news)), args.reps)})
    if out:
        out.close()


if __name__ == "__main__":
    main()
