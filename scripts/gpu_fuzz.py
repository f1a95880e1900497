"""Randomised parity sweep on the GPU: suffix sort and match search vs the oracle (many small/medium inputs)."""
import os
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import oracle  # noqa: E402
from deltaq_b200 import CudaSuffixSort, bsdiff  # noqa: E402

seed = int(sys.argv[1]) if len(sys.argv) > 1 else 0
budget = float(sys.argv[2]) if len(sys.argv) > 2 else 60.0
rng = np.random.default_rng(seed)
s = CudaSuffixSort()
t0 = time.time()
n_sort = n_search = 0
bad = 0


def gen_text(n):
    kind = rng.integers(0, 6)
    if kind == 0:
        return rng.integers(0, 256, n, dtype=np.uint8)
    if kind == 1:
        return rng.integers(0, int(rng.integers(1, 5)), n, dtype=np.uint8)
    if kind == 2:      # periodic with noise
        p = rng.integers(0, 256, int(rng.integers(1, 40)), dtype=np.uint8)
        t = np.tile(p, n // p.size + 1)[:n].copy()
        k = int(rng.integers(0, max(1, n // 50) + 1))
        if k and n:
            t[rng.integers(0, n, k)] = rng.integers(0, 256, k, dtype=np.uint8)
        return t
    if kind == 3:      # runs
        t = np.zeros(n, np.uint8)
        i = 0
        while i < n:
            L = int(rng.integers(1, 2000))
            t[i:i + L] = rng.integers(0, 3)
            i += L
        return t
    if kind == 4:      # repeated blocks
        b = rng.integers(0, 256, int(rng.integers(10, 3000)), dtype=np.uint8)
        return np.tile(b, n // b.size + 1)[:n].copy()
    t = rng.integers(0, 256, n, dtype=np.uint8)   # ends in zeros (end-of-text rule)
    z = int(rng.integers(0, min(n, 20) + 1))
    if z:
        t[n - z:] = 0
    return t


def mutate(old):
    new = bytearray(old.tobytes())
    for _ in range(int(rng.integers(0, 8))):
        p = int(rng.integers(0, len(new) + 1))
        k = int(rng.integers(1, 200))
        op = int(rng.integers(0, 3))
        if op == 0:
            new[p:p + k] = rng.integers(0, 256, k, dtype=np.uint8).tobytes()
        elif op == 1:
            new[p:p] = rng.integers(0, 4, k, dtype=np.uint8).tobytes()
        else:
            del new[p:p + k]
    return np.frombuffer(bytes(new), dtype=np.uint8)


while time.time() - t0 < budget:
    n = int(rng.choice([rng.integers(0, 64), rng.integers(64, 5000), rng.integers(5000, 300000)]))
    t = gen_text(n)
    ref = oracle.sais(t)
    with s.sort(t) as owner:
        got = owner.memory.copy()
    n_sort += 1
    if not np.array_equal(got, ref):
        bad += 1
        np.save(f"gpurun_out/fuzz_bad_sort_{seed}_{n_sort}.npy", t)
        print("SORT MISMATCH n=", n, flush=True)
        continue
    if n <= 20000:
        new = mutate(t) if rng.integers(0, 4) else gen_text(int(rng.integers(0, 3000)))
        I = oracle.make_I(ref)
        pos, ln = bsdiff.search_all(t, new, s, I=I if rng.integers(0, 2) else None)
        rp, rl = oracle.search_table(t, new)
        ok = np.array_equal(pos, rp) and np.array_equal(ln, rl)
        st = bsdiff.create_streams(t, new, s)
        r = oracle.bsdiff_streams(t, new, I, trace=True)
        v = r["trace_len"] >= 0
        ok = ok and all(st[k] == r[k] for k in ("ctrl", "diff", "extra")) and np.array_equal(pos[v], r["trace_pos"][v]) \
            and np.array_equal(ln[v], r["trace_len"][v])
        n_search += 1
        if not ok:
            bad += 1
            np.save(f"gpurun_out/fuzz_bad_search_old_{seed}_{n_search}.npy", t)
            np.save(f"gpurun_out/fuzz_bad_search_new_{seed}_{n_search}.npy", new)
            print("SEARCH MISMATCH n=", n, "m=", new.size, flush=True)
print(f"fuzz seed={seed}: {n_sort} sorts, {n_search} searches, {bad} mismatches in {time.time()-t0:.0f}s", flush=True)
sys.exit(1 if bad else 0)
