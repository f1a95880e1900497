#!/usr/bin/env python
"""bench.py -- the hot path of DeltaQ's `dq bsdiff` on B200: ISuffixSort.Sort(old) + Diff.Search at every
scan position of new, on BASELINE.json's config #2 (synthetic 16 MiB -> 17 MiB executable-like pair).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One step = one pass of the hot path over one (old, new) pair:
  value  : inputs and outputs resident in HBM (dq_cuda_suffix_sort_device + dq_cuda_bsdiff_search_device)
  e2e    : dq_cuda_bsdiff_streams through the C ABI with pinned HOST buffers: H2D of old and new, sort,
           search, D2H of the (pos, len) table, and the reference's greedy scan/emit loop on the host,
           returning the uncompressed ctrl/diff/extra streams (everything of Diff.Create except bzip2).
Unit: MB/s = 1e6 bytes of `new` per second (SURVEY.md section 8(d)); whole-job aggregate over ranks.
N > 1: every rank diffs its own pair (independent objects, no data-path collective) -> weak scaling.  The same line
then carries a `sharded` record: rank 0 alone drives ALL N GPUs through one device-group context (dq_cuda_create
with ndev = N) -- BASELINE config #4 (512 MiB genome-like text, one suffix sort by N GPUs, sufcheck asserted in the
run), the match search of a 256 MiB executable-like pair sharded by new-range (table asserted equal to the one-GPU
table), and at N = 8 BASELINE config #5's 1.9 GiB text; the other ranks hold no GPU work meanwhile.

--impl reference times the CPU restatement of the reference's path (oracle/: the faster of its LibDivSufSort and
SA-IS restatements + Diff.Create's loop with its inline Search) on one host core -- the reference is single-threaded --
on the same C2 pair at full size.

--dump-outputs DIR writes what the last timed step returned for rank 0's pair, so that two builds (or the two arms)
can be compared output for output on identical seeded inputs: suffix_array in float64 and the ctrl / diff / extra
stream bytes in float32 (both arms; on the GPU, the streams of the e2e arm), plus match_pos / match_len, the device
arm's (pos, len) table, in float64.  An array longer than 2^20 entries is written as a seeded sample (dump_sample).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "bsdiff Diff.Create hot path (ISuffixSort.Sort + Diff.Search at every scan position) input MB/s"
UNIT = "MB/s"
WORKLOAD = "C2: synthetic 16 MiB -> 17 MiB executable-like pair, ~13% mutated regions (workloads.c2_exe_pair)"
NOMINAL_HBM_GBS = 8000.0   # BASELINE.json north_star: "~8 TB/s"; reported beside the measured peak
MIB = 1 << 20


def pass_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of one round-0 onesweep launch from the committed ncu --set full
    capture (profiles/); per launch, like `achieved`."""
    for name in ("r02_pass_traffic.json", "r01_pass_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                return float(json.load(f)["traffic_bytes_round0_launch"])
        except Exception:
            continue
    return None


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def host_cores_per_rank(world):
    """The share of the host's cores one rank keeps (main() pins to it when there are two or more per rank)."""
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 0)
    per = cores // max(world, 1)
    return per if (world > 1 and per >= 2) else cores


def cores_by_physical_core(cpus, topology=None):
    """The logical CPUs this process may run on, ordered (package, physical core, cpu): hyper-thread siblings end up side by
    side, so when the list is dealt out in equal runs every rank gets whole physical cores -- and the cores of one
    package -- instead of sharing a core's two threads with another rank's spinning host loop.  Without sibling pairs in
    the set (or without sysfs) the order is the plain one."""
    def read(c, name):
        with open(f"/sys/devices/system/cpu/cpu{c}/topology/{name}") as f:
            return int(f.read().strip())
    keyed = []
    for c in sorted(cpus):
        try:
            pkg, core = topology[c] if topology is not None else (read(c, "physical_package_id"), read(c, "core_id"))
        except Exception:
            return sorted(cpus)
        keyed.append((pkg, core, c))
    return [c for _, _, c in sorted(keyed)]


def workload_config(world, n, m, cores_per_rank):
    """`config` of the JSON line: the same dict from both arms (the driver compares them)."""
    return {"workload": WORKLOAD, "old_bytes": n, "new_bytes": m, "pairs_per_step": world,
            "l2": "working set (>= 24 B x 16.7 M pairs per radix pass, 400 MB) exceeds the 126 MB L2; no flush",
            "parallelism": f"{world} x independent pairs (one process and context per GPU)",
            "host_cores_per_rank": cores_per_rank}


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self.index)],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return None
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if not sm:
            return None
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "reasons": sorted(reasons),
                "samples": len(sm)}


# ---- CPU arm ---------------------------------------------------------------------------------------------------

def cpu_sorters():
    """The reference's sorters as restated in oracle/ (name -> callable).  LibDivSufSort is the reference's default
    (Defaults.cs:9); SA-IS is what its bsdiff tests use."""
    import oracle
    out = {"sais": oracle.sais}
    if hasattr(oracle, "divsufsort"):
        out["divsufsort"] = oracle.divsufsort
    return out


# --dump-outputs: arrays longer than this are written as a seeded sample of this many entries, so that the six arrays
# of a dump stay under 64 MB in all (3 x 8 MB in float64, 3 x 4 MB in float32)
DUMP_MAX_ELEMENTS = 1 << 20


def dump_sample(a, dtype):
    """All of `a` when it has at most DUMP_MAX_ELEMENTS entries, else its entries at sorted positions drawn with a fixed
    seed (the same positions in every run for the same length), converted to `dtype`."""
    a = np.asarray(a).reshape(-1)
    if a.size > DUMP_MAX_ELEMENTS:
        a = a[np.unique(np.random.default_rng(0).integers(0, a.size, DUMP_MAX_ELEMENTS))]
    return a.astype(dtype)


def stream_outputs(streams):
    """The uncompressed ctrl / diff / extra streams, byte values as float32."""
    return {k: dump_sample(np.frombuffer(streams[k], dtype=np.uint8), np.float32) for k in ("ctrl", "diff", "extra")}


def write_outputs(dirname, arrays):
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(dirname, name + ".npy"), a)


def stream_digests(streams):
    """Digest of each uncompressed stream (ctrl / diff / extra): how the GPU arm's result is compared with the CPU arm's."""
    import hashlib
    return {k: hashlib.blake2b(bytes(streams[k]) if not isinstance(streams[k], bytes) else streams[k],
                               digest_size=16).hexdigest() for k in ("ctrl", "diff", "extra")}


def cpu_step_times(old, new, reps):
    """Seconds per sorter for the sort, and for the Diff.Create loop (inline Search), best of `reps`; the digests of the
    streams the loop produced; whether the reference's sorters gave the same suffix array."""
    import oracle
    sort_s = {}
    sa = None
    agree = True
    for name, fn in cpu_sorters().items():
        best = None
        for _ in range(reps):
            t0 = time.perf_counter()
            got = fn(old)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        sort_s[name] = best
        if sa is not None and not np.array_equal(sa, got):
            agree = False
        sa = got
    I = oracle.make_I(sa)
    loop = None
    streams = None
    for _ in range(reps):
        t0 = time.perf_counter()
        streams = oracle.bsdiff_streams(old, new, I)
        dt = time.perf_counter() - t0
        loop = dt if loop is None else min(loop, dt)
    return sort_s, loop, stream_digests(streams), agree


def run_reference(args, rank):
    """CPU arm: the oracle's restatement of the reference's path on the full C2 pair, one core."""
    if rank != 0:
        return
    import oracle
    from deltaq_b200 import workloads as w
    world = int(os.environ.get("WORLD_SIZE", "1"))
    oracle.build()
    old, new = w.c2_exe_pair()
    sorters = cpu_sorters()
    # the faster of the reference's sorters on this input carries the arm (one untimed probe each)
    probe = {}
    agree, first = True, None
    for name, fn in sorters.items():
        t0 = time.perf_counter()
        got = fn(old)
        probe[name] = time.perf_counter() - t0
        if first is None:
            first = got
        elif not np.array_equal(first, got):
            agree = False
    del first, got
    best = min(probe, key=probe.get)
    sort = sorters[best]

    def step():
        sa = sort(old)
        return sa, oracle.bsdiff_streams(old, new, oracle.make_I(sa))

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        sa, streams = step()
    dt = (time.perf_counter() - t0) / args.steps
    if args.dump_outputs:
        write_outputs(args.dump_outputs, {"suffix_array": dump_sample(sa, np.float64), **stream_outputs(streams)})
    v = new.size / dt / 1e6
    sample = (f"the full C2 pair ({old.size} -> {new.size} bytes); per step: suffix sort of old with the faster of the "
              f"reference's sorters as restated in oracle/ ({best}; one probe each: "
              + ", ".join(f"{k} {v_:.2f} s" for k, v_ in probe.items()) +
              ") + Diff.Create loop with inline Search (oracle/bsdiff.c ~ Diff.cs:92-298), no bzip2; gcc -O2, "
              "single thread as the reference is single-threaded")
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8/int32", "data": "synthetic",
        "config": workload_config(world, int(old.size), int(new.size), host_cores_per_rank(world)),
        "cpu_baseline": {"value": v, "unit": UNIT, "cores": 1, "kind": "port", "sorter": best, "sorters_agree": agree,
                         "sample": sample},
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }), flush=True)


def cpu_baseline_once():
    import oracle
    from deltaq_b200 import workloads as w
    oracle.build()
    old, new = w.c2_exe_pair()
    sort_s, loop, digests, agree = cpu_step_times(old, new, 2)
    best = min(sort_s, key=sort_s.get)
    dt = sort_s[best] + loop
    return {"value": new.size / dt / 1e6, "unit": UNIT, "cores": 1, "kind": "port", "sorter": best,
            "sorters_agree": agree, "stream_digests": digests,
            "sort_only_MBps": {k: old.size / v / 1e6 for k, v in sort_s.items()},
            "loop_only_MBps": new.size / loop / 1e6,
            "sample": f"the full C2 pair ({old.size} -> {new.size} bytes), best of 2 per part; oracle restatements of the "
                      "reference's sorters + Diff.Create loop with inline Search, no bzip2, gcc -O2, 1 thread"}


# ---- per-round roofline (north_star: fraction of HBM bandwidth per doubling round) ----------------------------------

def round_records(acc_rounds, steps, peak):
    out = []
    for r, (ms, active, passes) in enumerate(acc_rounds):
        ms /= steps
        alg = active * ((41 if r == 0 else 52) + 24 * passes)
        gbs = alg / (ms * 1e-3) / 1e9 if ms > 0 else None
        out.append({"round": r, "active": active, "passes": passes, "ms": ms, "algorithmic_bytes": alg, "GBps": gbs,
                    "frac_measured_peak": gbs / peak if gbs else None,
                    "frac_nominal_8TBps": gbs / NOMINAL_HBM_GBS if gbs else None})
    return out


def abi_sort_record(ctx, text, reps):
    """ISuffixSort.Sort as the caller sees it (SURVEY 8(d): wall seconds through the C ABI): dq_cuda_suffix_sort with
    pinned host buffers, H2D of the text and D2H of the suffix array inside.  Reported, never fatal."""
    n = int(text.size)
    try:
        p_t = ctx.pinned(n, np.uint8)
        p_sa = ctx.pinned(n, np.int32)
        try:
            p_t.array[:] = text
            abi = None
            for it in range(reps + 1):
                t0 = time.perf_counter()
                ctx.suffix_sort(p_t.array, p_sa.array)
                dt = time.perf_counter() - t0
                if it and (abi is None or dt < abi):
                    abi = dt
            import oracle
            # the array that call delivered, under the reference's own checker (LDSSChecker.cs:23-119 restated), untimed
            bad = int(oracle.sufcheck(np.ascontiguousarray(text), p_sa.array))
            return {"abi_ms": abi * 1e3, "input_MBps_abi": n / abi / 1e6, "sufcheck": bad,
                    "abi_note": "dq_cuda_suffix_sort, pinned host text in, pinned host suffix array out (4n bytes over PCIe); "
                                "sufcheck = the reference's checker on the delivered array (0 = a correct suffix array)"}
        finally:
            p_t.free()
            p_sa.free()
    except Exception as e:
        return {"abi_error": repr(e)}


def sort_config_record(ctx, torch, text, name, peak, reps=3):
    """Device-resident sort of one of BASELINE's other single-GPU configs: ms, MB/s, per-round roofline."""
    n = int(text.size)
    d_t = torch.from_numpy(text).cuda()
    d_sa = torch.empty(max(n, 1), dtype=torch.int32, device="cuda")
    ctx.set_timing(False)
    best = None
    for it in range(reps + 1):
        ctx.suffix_sort_device(d_t.data_ptr(), n, d_sa.data_ptr())
        st = ctx.stats()
        if it and (best is None or st["device_ms"] < best):
            best = st["device_ms"]
    ctx.set_timing(True)          # per-round times from one more run (the extra event records cost a few microseconds)
    ctx.suffix_sort_device(d_t.data_ptr(), n, d_sa.data_ptr())
    rounds = ctx.round_times()
    st = ctx.stats()
    ctx.set_timing(False)
    del d_t, d_sa
    rec = {"config": name, "n": n, "device_ms": best, "input_MBps_device": n / (best * 1e-3) / 1e6 if best else None,
           "rounds": st["rounds"], "launches": st["kernel_launches"],
           "algorithmic_GBps": st["algorithmic_bytes"] / (best * 1e-3) / 1e9 if best else None,
           "per_round": round_records(rounds, 1, peak)}
    rec.update(abi_sort_record(ctx, text, reps))
    return rec


# ---- one device group over all GPUs, driven by rank 0 (N > 1) ---------------------------------------------------------

def diff_create_record(ctx, old, new, reps=3):
    """Diff.Create as a whole (Diff.cs:27-242): dq_cuda_bsdiff_patch = streams + header + the three bzip2 sections
    produced block-parallel on the host, against the same streams compressed serially (what a BZip2OutputStream per
    section costs with libbz2).  One record beside the headline; never inside a timed region of `value` / `e2e`."""
    import bz2
    try:
        times = []
        patch = None
        for _ in range(reps + 1):
            t0 = time.perf_counter()
            patch = ctx.bsdiff_patch(old, new)
            times.append(time.perf_counter() - t0)
        streams = ctx.bsdiff_streams(old, new)
        t0 = time.perf_counter()
        serial = [bz2.compress(streams[k]) for k in ("ctrl", "diff", "extra")]
        serial_s = time.perf_counter() - t0
        cl = int.from_bytes(patch[8:16], "little")
        dl = int.from_bytes(patch[16:24], "little")
        same = (bz2.decompress(patch[32:32 + cl]) == streams["ctrl"] and
                bz2.decompress(patch[32 + cl:32 + cl + dl]) == streams["diff"] and
                bz2.decompress(patch[32 + cl + dl:]) == streams["extra"])
        best = min(times[1:])
        # the way back: Patch.Apply on that file, sections decoded block-parallel (dq_cuda_bspatch), against the three
        # sections through serial libbz2 + the same native add loop
        from deltaq_b200 import _native
        from deltaq_b200.bsdiff import apply_streams
        apply_times = []
        rebuilt = None
        for _ in range(3):
            t0 = time.perf_counter()
            rebuilt = _native.bspatch(old, patch)
            apply_times.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        parts = [bz2.decompress(patch[32:32 + cl]), bz2.decompress(patch[32 + cl:32 + cl + dl]),
                 bz2.decompress(patch[32 + cl + dl:])]
        serial_new = apply_streams(old, parts[0], parts[1], parts[2], new.size)
        serial_apply_s = time.perf_counter() - t0
        applied = {"call": "dq_cuda_bspatch (patch file in, new file out; host code)", "ms": min(apply_times) * 1e3,
                   "serial_bz2_decode_and_apply_ms": serial_apply_s * 1e3,
                   "reproduces_new": bool(rebuilt.tobytes() == new.tobytes() == serial_new)}
        return {"call": "dq_cuda_bsdiff_patch (pageable host buffers in, BSDIFF40 file out)", "ms": best * 1e3,
                "patch_apply": applied,
                "new_MBps": new.size / best / 1e6, "patch_bytes": len(patch),
                "serial_bz2_ms": serial_s * 1e3, "serial_bz2_bytes": 32 + sum(len(x) for x in serial),
                "sections_decode_to_the_streams": bool(same), "host_threads": len(os.sched_getaffinity(0))}
    except Exception as e:   # reported, not fatal: the headline line must still print
        return {"error": repr(e)}


def sharded_record(devices, workers, lib=None, scale=1.0):
    """`lib`/`scale`: the CPU tests run this function on the logic emulator with tiny inputs."""
    import oracle
    from deltaq_b200 import CudaSuffixSort, workloads as w
    G = len(devices)
    rec = {"devices": devices,
           "what": "ONE context over all GPUs (dq_cuda_create, ndev = N) in rank 0's process; host buffers (pinned) in and "
                   "out through the ordinary C ABI calls; MB/s = 1e6 input bytes / wall second"}

    def timed(fn, reps=2):
        fn()
        best = None
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
        return best

    one = CudaSuffixSort(device=devices[0], _lib=lib)
    grp = CudaSuffixSort(device=devices, _lib=lib)
    try:
        # -- BASELINE config #4: 512 MiB genome-like text, one suffix sort
        t = w.c4_genome(max(64, int(512 * MIB * scale)))
        n = int(t.size)
        p_t = grp.context.pinned(n, np.uint8)
        p_t.array[:] = t
        p_sa = grp.context.pinned(n, np.int32)
        dt_g = timed(lambda: grp.context.suffix_sort(p_t.array, p_sa.array))
        st = grp.stats()
        bad = int(oracle.sufcheck(t, p_sa.array))
        assert bad == 0, f"sharded C4 suffix array fails sufcheck ({bad})"
        dt_1 = timed(lambda: one.context.suffix_sort(p_t.array, p_sa.array))
        rec["sort_c4"] = {"config": "C4: 512 MiB iid {A,C,G,T} + 1 % tandem repeats (workloads.c4_genome)", "n": n,
                          "ms": dt_g * 1e3, "input_MBps": n / dt_g / 1e6, "rounds": st["rounds"],
                          "launches": st["kernel_launches"], "sufcheck": bad,
                          "one_gpu_ms": dt_1 * 1e3, "one_gpu_input_MBps": n / dt_1 / 1e6,
                          "speedup_vs_one_gpu": dt_1 / dt_g, "strong_scaling_efficiency": dt_1 / dt_g / G}
        p_t.free()
        p_sa.free()
        del t

        # -- match search sharded by new-range: 256 MiB executable-like pair (C5's recipe at 1/8 scale)
        old, new = w.c5_pair(max(4096, int(256 * MIB * scale)), workers=workers)
        n, m = int(old.size), int(new.size)
        p_o = grp.context.pinned(n, np.uint8)
        p_o.array[:] = old
        p_n = grp.context.pinned(m, np.uint8)
        p_n.array[:] = new
        p_sa = grp.context.pinned(n, np.int32)
        pos_g = grp.context.pinned(m, np.int32)
        len_g = grp.context.pinned(m, np.int32)
        pos_1 = grp.context.pinned(m, np.int32)
        len_1 = grp.context.pinned(m, np.int32)

        def both(c, pos, ln):
            c.suffix_sort(p_o.array, p_sa.array)
            c.bsdiff_search(p_o.array, None, p_n.array, 0, m, pos.array, ln.array)

        dt_g = timed(lambda: both(grp.context, pos_g, len_g), reps=1)
        sg = grp.stats()
        dt_1 = timed(lambda: both(one.context, pos_1, len_1), reps=1)
        s1 = one.stats()
        same = bool(np.array_equal(pos_g.array, pos_1.array) and np.array_equal(len_g.array, len_1.array))
        assert same, "sharded search table differs from the one-GPU table"
        rec["sort_search_256MiB"] = {
            "config": "C5 recipe at 1/8 scale: 256 MiB executable-like old -> 272 MiB new (workloads.c5_pair); sort(old) "
                      "by all GPUs + Diff.Search at every scan position sharded by new-range",
            "old_bytes": n, "new_bytes": m, "ms": dt_g * 1e3, "input_MBps": m / dt_g / 1e6,
            "search_device_ms": sg["search_ms"], "one_gpu_ms": dt_1 * 1e3, "one_gpu_input_MBps": m / dt_1 / 1e6,
            "one_gpu_search_device_ms": s1["search_ms"], "speedup_vs_one_gpu": dt_1 / dt_g,
            "table_equals_one_gpu_table": same}
        for p in (p_o, p_n, p_sa, pos_g, len_g, pos_1, len_1):
            p.free()
        del old, new

        # -- BASELINE config #5's text (near the int32 suffix-array limit) over 8 GPUs
        if G >= 8:
            t = w.c5_old(max(4096, int(2_040_109_466 * scale)), workers=workers)
            n = int(t.size)
            p_t = grp.context.pinned(n, np.uint8)
            p_t.array[:] = t
            p_sa = grp.context.pinned(n, np.int32)
            dt_g = timed(lambda: grp.context.suffix_sort(p_t.array, p_sa.array), reps=1)
            st = grp.stats()
            sa_g = np.array(p_sa.array, copy=True)
            dt_1 = timed(lambda: one.context.suffix_sort(p_t.array, p_sa.array), reps=1)
            same = bool(np.array_equal(sa_g, p_sa.array))
            # a full sufcheck of 2 G suffixes takes minutes on one core (tests/ runs it at this size): here the result
            # is compared with the one-GPU path's (different code: run-aware rounds, no exchanges) and sampled
            idx = np.sort(np.random.default_rng(0).integers(0, max(1, n - 1), min(n, 200_000)))
            sample_bad = int(oracle.verify_pairs(t, sa_g, idx))
            assert same, "sharded C5 suffix array differs from the one-GPU suffix array"
            assert sample_bad == 0, "sharded C5 suffix array has adjacent suffixes out of order"
            rec["sort_c5"] = {"config": "C5 text: 2,040,109,466 B executable-like (workloads.c5_old)", "n": n,
                              "ms": dt_g * 1e3, "input_MBps": n / dt_g / 1e6, "rounds": st["rounds"],
                              "one_gpu_ms": dt_1 * 1e3, "one_gpu_input_MBps": n / dt_1 / 1e6,
                              "speedup_vs_one_gpu": dt_1 / dt_g, "equals_one_gpu_suffix_array": same,
                              "sampled_adjacent_pairs_out_of_order": sample_bad}
    except Exception as e:  # the record reports, the bench line survives
        rec["error"] = f"{type(e).__name__}: {e}"
    finally:
        one.dispose()
        grp.dispose()
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="deltaq_b200")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the other configs / the sharded record")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step computed for rank 0's pair as "
                         "DIR/<name>.npy: suffix_array, match_pos, match_len (float64) and ctrl, diff, extra (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl != "reference" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    from deltaq_b200 import CudaSuffixSort, workloads as w

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: deltaq_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    host_group = None
    pinned_cores = None
    cores_per_rank = host_cores_per_rank(world)   # before this rank pins itself
    if world > 1 and hasattr(os, "sched_setaffinity"):
        # one process per GPU: every rank's host threads (the greedy loop's scan / extender / writers, the CUDA worker
        # threads) stay on their own share of the cores, so the ranks do not preempt each other; the library sizes its
        # thread crew by the CPUs the process may run on
        cores = cores_by_physical_core(os.sched_getaffinity(0))
        per = len(cores) // world
        if per >= 2:
            pinned_cores = cores[local_rank * per:(local_rank + 1) * per]
            os.sched_setaffinity(0, pinned_cores)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        host_group = dist.new_group(backend="gloo")   # host-side waits that keep the GPUs free

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # every rank diffs its own pair (same recipe, rank-specific seeds)
    old, new = w.c2_exe_pair(seed_old=1 + 1000 * rank, seed_new=2 + 1000 * rank)
    n, m = int(old.size), int(new.size)
    sorter = CudaSuffixSort(device=local_rank)
    ctx = sorter.context

    # ---- device-resident arm -----------------------------------------------------------------------
    d_old = torch.from_numpy(old).cuda()
    d_new = torch.from_numpy(new).cuda()
    d_sa = torch.empty(n, dtype=torch.int32, device="cuda")
    d_pos = torch.empty(m, dtype=torch.int32, device="cuda")
    d_len = torch.empty(m, dtype=torch.int32, device="cuda")
    torch.cuda.synchronize()

    acc = {"launches": 0, "device_ms": 0.0, "pass_ms": 0.0, "pass_pairs": 0, "search_ms": 0.0, "passes": 0,
           "rounds": 0, "alg_bytes": 0, "round_times": None}

    def step_device(record):
        ctx.suffix_sort_device(d_old.data_ptr(), n, d_sa.data_ptr())
        if record:
            rt = ctx.round_times()
            if acc["round_times"] is None:
                acc["round_times"] = [[0.0, a, p] for _, a, p in rt]
            for slot, (ms, _, _) in zip(acc["round_times"], rt):
                slot[0] += ms
        ctx.bsdiff_search_device(d_old.data_ptr(), n, None, d_new.data_ptr(), m, 0, m, d_pos.data_ptr(), d_len.data_ptr())
        if record:
            st = ctx.stats()
            acc["launches"] += st["kernel_launches"]
            acc["device_ms"] += st["device_ms"]
            acc["search_ms"] += st["search_ms"]
            acc["pass_ms"] += st["pass_ms"]
            acc["pass_pairs"] += st["pass_pairs"]
            acc["passes"] += st["radix_passes"]
            acc["rounds"] = st["rounds"]
            acc["alg_bytes"] = st["algorithmic_bytes"]

    ctx.set_timing(True)
    for _ in range(args.warmup):
        step_device(False)
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_device(True)
    barrier()
    dt = time.perf_counter() - t0
    outputs = {}
    if args.dump_outputs and rank == 0:
        outputs.update({name: dump_sample(t.cpu().numpy(), np.float64)
                        for name, t in (("suffix_array", d_sa), ("match_pos", d_pos), ("match_len", d_len))})

    # ---- end-to-end arm: host buffers through the C ABI ------------------------------------------------
    ctx.set_timing(False)
    p_old = ctx.pinned(n, np.uint8)
    p_new = ctx.pinned(m, np.uint8)
    p_old.array[:] = old
    p_new.array[:] = new
    streams = None
    for _ in range(args.warmup):
        streams = ctx.bsdiff_streams(p_old.array, p_new.array, copy=False)
    barrier()
    t1 = time.perf_counter()
    for _ in range(args.steps):
        streams = ctx.bsdiff_streams(p_old.array, p_new.array, copy=False)   # the C ABI's own result: pointers + lengths
    barrier()
    dt_e2e = time.perf_counter() - t1
    e2e_stats = ctx.stats()
    stream_sizes = [len(streams["ctrl"]), len(streams["diff"]), len(streams["extra"])]
    if args.dump_outputs and rank == 0:
        outputs.update(stream_outputs(streams))
    streams = None
    clocks = sampler.stop() if rank == 0 else None   # sampled over both timed regions (device arm + e2e arm)

    # the same call with ordinary (pageable) numpy buffers: what a managed caller's `fixed` spans are (Diff.cs:78,90)
    for _ in range(2):
        ctx.bsdiff_streams(old, new, copy=False)
    barrier()
    t2 = time.perf_counter()
    for _ in range(args.steps):
        ctx.bsdiff_streams(old, new, copy=False)
    barrier()
    dt_pageable = time.perf_counter() - t2

    # what the call returned for this pair, for the comparison with the CPU arm's streams below (untimed)
    gpu_digests = stream_digests(ctx.bsdiff_streams(old, new, copy=True)) if rank == 0 else None

    # max over ranks
    if world > 1:
        tt = torch.tensor([dt, dt_e2e, dt_pageable], dtype=torch.float64, device="cuda")
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt, dt_e2e, dt_pageable = float(tt[0]), float(tt[1]), float(tt[2])

    peak, peak_src = measured_peak()
    extras = None
    sharded = None
    diff_create = None
    if not args.no_extras:
        if world == 1:
            diff_create = diff_create_record(ctx, old, new)
            # BASELINE's other single-GPU configs, device-resident sort only (bounded: a few hundred ms in all)
            extras = []
            for make, name, reps in ((w.c1_uniform, "C1: 1 MiB uniform random bytes", 5),
                                     (w.c3_repetitive, "C3: 64 MiB repetitive text", 2),
                                     (lambda: w.c4_genome(64 * MIB), "C4 recipe, 64 MiB slice", 2)):
                try:
                    extras.append(sort_config_record(ctx, torch, make(), name, peak, reps=reps))
                except Exception as e:   # the record reports, the bench line survives
                    extras.append({"config": name, "error": repr(e)})
        else:
            # free this rank's GPU memory, then rank 0 drives all GPUs; the others wait on the host
            del d_old, d_new, d_sa, d_pos, d_len
            p_old.free()
            p_new.free()
            sorter.dispose()
            sorter = None
            torch.cuda.empty_cache()
            torch.cuda.synchronize()
            dist.barrier(group=host_group)
            if rank == 0:
                if pinned_cores:
                    os.sched_setaffinity(0, cores)   # this process now drives every GPU: all cores again
                os.environ["DQ_SHARD_MIN"] = str(32 * MIB)
                sharded = sharded_record(list(range(world)), workers=min(8, max(1, (os.cpu_count() or 8) // 2)))
            dist.barrier(group=host_group)

    if rank == 0:
        ms_step = dt / args.steps * 1e3
        value = world * m / (dt / args.steps) / 1e6
        e2e_value = world * m / (dt_e2e / args.steps) / 1e6
        pass_gbs = acc["pass_pairs"] * 24 / (acc["pass_ms"] * 1e-3) / 1e9 if acc["pass_ms"] > 0 else None
        cpu = None if args.no_cpu_baseline else cpu_baseline_once()
        sort_ms = acc["device_ms"] / args.steps
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8/int32", "data": "synthetic",
            "config": workload_config(world, n, m, cores_per_rank),
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": dt_e2e / args.steps * 1e3,
                    "h2d_bytes_per_step": n + m,
                    # the (pos,len) table crosses PCIe coded: 1 B/position + 12 B/match head + 8 B per 1024 positions
                    "d2h_bytes_per_step": (8 * m if e2e_stats["table_fallbacks"] else
                                           m + 12 * e2e_stats["table_heads"] + 8 * ((m + 1023) // 1024)),
                    "includes": "H2D old+new, sort, search, D2H of the coded (pos,len) table in slices, host greedy "
                                "scan/extend/emit loop on host threads overlapped with the slices; result = "
                                "context-owned ctrl/diff/extra buffers; streams "
                                f"ctrl/diff/extra = {stream_sizes[0]}/{stream_sizes[1]}/{stream_sizes[2]} B",
                    "pageable_buffers": {"value": world * m / (dt_pageable / args.steps) / 1e6, "unit": UNIT,
                                         "ms_per_step": dt_pageable / args.steps * 1e3,
                                         "note": "the same call with ordinary numpy (pageable) old/new buffers"}},
            "gpu_launches": acc["launches"],
            "roofline": {"bound": "hbm", "kernel": "dq::radix::onesweep_pass_kernel",
                         "achieved": pass_gbs, "peak": peak, "unit": "GB/s",
                         "frac": (pass_gbs / peak) if pass_gbs else None, "peak_source": peak_src,
                         "frac_nominal_8TBps": (pass_gbs / NOMINAL_HBM_GBS) if pass_gbs else None,
                         "algorithmic_bytes_per_pair": 24, "launches_timed": acc["passes"],
                         "share_of_device_time": acc["pass_ms"] / (acc["device_ms"] + acc["search_ms"])
                         if acc["device_ms"] else None,
                         "traffic": pass_traffic(),
                         "traffic_note": "ncu capture of a round-0 launch (16,777,216 pairs, 402,653,184 algorithmic B); "
                                         "achieved averages all launches of the step (round 0 and the smaller doubling rounds)",
                         "per_round": round_records(acc["round_times"] or [], args.steps, peak),
                         "per_round_note": "north_star's yardstick: SURVEY 8(d) algorithmic bytes of the round / CUDA-event "
                                           "time from the round's first launch to the next round's (all kernels of the "
                                           "round, not only the radix passes)"},
            "device_ms_per_step": {"sort": sort_ms, "search": acc["search_ms"] / args.steps},
            "sort": {"rounds": acc["rounds"], "algorithmic_bytes": acc["alg_bytes"],
                     "input_MBps_device": n / (sort_ms * 1e-3) / 1e6 if sort_ms else None,
                     "algorithmic_GBps": acc["alg_bytes"] / (sort_ms * 1e-3) / 1e9 if sort_ms else None,
                     "algorithmic_frac_measured_peak": acc["alg_bytes"] / (sort_ms * 1e-3) / 1e9 / peak if sort_ms else None},
            "clocks": clocks,
            "cpu_baseline": cpu,
        }
        if cpu is not None and "stream_digests" in cpu:
            # in-run parity at the bench's own size: the streams dq_cuda_bsdiff_streams returned for this pair against the
            # streams of the CPU restatement of Diff.Create that was just timed on the same pair (oracle/ as the checker)
            line["parity"] = {"streams_identical_to_cpu_baseline": gpu_digests == cpu["stream_digests"],
                              "what": "blake2b digests of the uncompressed ctrl / diff / extra streams of the C2 pair: "
                                      "dq_cuda_bsdiff_streams (GPU arm) vs oracle.bsdiff_streams (cpu_baseline)",
                              "gpu": gpu_digests, "cpu": cpu["stream_digests"]}
        if diff_create is not None:
            line["diff_create"] = diff_create
        if extras is not None:
            line["other_configs"] = extras
        if sharded is not None:
            line["sharded"] = sharded
        if args.dump_outputs:
            write_outputs(args.dump_outputs, outputs)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
