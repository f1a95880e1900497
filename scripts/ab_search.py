"""A/B of compile-time variants of the search kernels on the same box: builds the library once per set of -D flags and
times the search of C2 and of two repetitive inputs.   python scripts/ab_search.py "" "-DDQ_SCRATCH_BATCH=1" ..."""
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from deltaq_b200 import _native, build, workloads as w  # noqa: E402


def tiled(n, blk, seed=5):
    rng = np.random.default_rng(seed)
    base = w.c2_exe_pair(blk, blk + 1)[0]
    old = np.concatenate([base if k % 3 else rng.integers(0, 256, base.size, dtype=np.uint8) for k in range(n // blk)])
    new = old.copy()
    for c in rng.integers(0, old.size - (1 << 20), max(4, n >> 22)):
        new[c:c + int(rng.integers(64, 1 << 20))] = rng.integers(0, 256, 1, dtype=np.uint8)
    return old, new


inputs = {"c2": w.c2_exe_pair(), "rep16MiB/4MiB": tiled(16 << 20, 4 << 20), "rep128MiB/32MiB": tiled(128 << 20, 32 << 20)}
for vi, flags in enumerate(sys.argv[1:]):
    out = os.path.join(ROOT, "gpurun_out", f"libdq_ab{vi}.so")
    subprocess.check_call([build.nvcc_path()] + build.NVCC_FLAGS + flags.split() + ["-I", build.INCLUDE, "-o", out,
                                                                                      os.path.join(build.CSRC, "deltaq_cuda.cu")])
    ctx = _native.Context(lib=_native.Library(out))
    res = []
    for name, (old, new) in inputs.items():
        sa = ctx.pinned(old.size, np.int32)
        pos = ctx.pinned(new.size, np.int32)
        ln = ctx.pinned(new.size, np.int32)
        best = None
        for _ in range(4):
            ctx.suffix_sort(old, sa.array)
            ctx.bsdiff_search(old, None, new, 0, new.size, pos.array, ln.array)
            ms = ctx.stats()["search_ms"]
            best = ms if best is None else min(best, ms)
        res.append(f"{name} {best:.3f} ms (chk {int(pos.array.sum()) ^ int(ln.array.sum()):x})")
        del sa, pos, ln
    print(f"[{flags or 'default'}] " + " | ".join(res), flush=True)
    ctx.close()
    os.remove(out)
