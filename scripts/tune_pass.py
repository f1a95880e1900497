"""Build variants of the onesweep pass (items/thread, min CTAs/SM) on the GPU box and time them."""
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from deltaq_b200 import _native, build, workloads as w  # noqa: E402

variants = [(16, 4), (16, 3), (16, 2), (12, 4), (12, 5), (8, 6), (20, 3)]
if len(sys.argv) > 1:
    variants = [tuple(int(x) for x in v.split("x")) for v in sys.argv[1:]]
variants = [tuple(list(v) + [8][len(v) - 2:]) if len(v) < 3 else v for v in variants]
texts = {"uniform16M": w.c1_uniform(16 << 20, 9), "c2_old": w.c2_exe_pair()[0]}
if os.environ.get("TUNE_SMALL"):
    texts = {"c1_1MiB": w.c1_uniform(), "u256K": w.c1_uniform(256 << 10, 3), "u4MiB": w.c1_uniform(4 << 20, 4)}
res = {}
lib_dir = tempfile.mkdtemp(prefix="tune_pass_")  # one throwaway library per variant
for items, minb, window in variants:
    out = os.path.join(lib_dir, f"libdq_{items}_{minb}_{window}.so")
    cmd = [build.nvcc_path()] + build.NVCC_FLAGS + [f"-DDQ_PASS_ITEMS={items}", f"-DDQ_PASS_MIN_BLOCKS={minb}", f"-DDQ_LOOK_WINDOW={window}",  "-Xptxas", "-v",
           "-I", build.INCLUDE, "-o", out, os.path.join(build.CSRC, "deltaq_cuda.cu")]
    p = subprocess.run(cmd, capture_output=True, text=True)
    info = [l for l in p.stderr.splitlines() if "onesweep_pass_kernelIj" in l or "spill" in l or "Used" in l]
    regs = ""
    for i, l in enumerate(p.stderr.splitlines()):
        if "onesweep_pass_kernelIj" in l:
            regs = " | ".join(x.strip() for x in p.stderr.splitlines()[i + 1:i + 3])
    if p.returncode != 0:
        print(items, minb, "BUILD FAILED", p.stderr[-500:])
        continue
    lib = _native.Library(out)
    ctx = _native.Context(lib=lib)
    ctx.set_timing(True)
    for name, t in texts.items():
        pin = ctx.pinned(t.size, np.int32)
        best = None
        for _ in range(12):
            ctx.suffix_sort(t, pin.array)
            st = ctx.stats()
            if best is None or st["device_ms"] < best["device_ms"]:
                best = st
        if "--passes" in os.environ.get("TUNE_FLAGS", ""):
            for ms, pairs, shift in ctx.pass_times()[:40]:
                print(f"      shift={shift:2d} pairs={pairs:9d} {ms*1e3:8.1f} us  {pairs*24/ms/1e6:7.0f} GB/s")
        gbs = best["pass_pairs"] * 24 / best["pass_ms"] / 1e6
        res[f"{items}x{minb}x{window}:{name}"] = dict(device_ms=best["device_ms"], pass_ms=best["pass_ms"], pass_GBps=gbs)
        print(f"items={items} minb={minb} window={window} {name}: device {best['device_ms']:.3f} ms, passes {best['pass_ms']:.3f} ms, {gbs:.0f} GB/s   [{regs}]", flush=True)
        pin.free()
    ctx.close()
json.dump(res, open(os.path.join(ROOT, "gpurun_out", "tune_pass.json"), "w"), indent=1)
