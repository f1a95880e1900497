"""bench.py's contract with the driver: the reference arm (CPU: runs here) prints one JSON line with the agreed keys,
and the committed line of the GPU arm (profiles/r01_bench_n1.json) carries the same ones plus roofline / cpu_baseline."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e"}


def load_dump(dirname):
    """--dump-outputs DIR as {name: array}; every file float32 or float64, all of them under 64 MB."""
    import numpy as np
    out = {f[:-4]: np.load(os.path.join(dirname, f)) for f in os.listdir(dirname)}
    assert all(a.dtype in (np.float32, np.float64) for a in out.values())
    assert sum(os.path.getsize(os.path.join(dirname, f)) for f in os.listdir(dirname)) <= 64 << 20
    return out


def test_reference_arm_prints_one_json_line(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--dump-outputs", str(tmp_path / "dump")],
                       capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip().startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and BASE_KEYS <= set(d)
    assert d["config"]["workload"].startswith("C2") and d["value"] > 0 and d["higher_is_better"] is True
    assert d["cpu_baseline"]["kind"] in ("port", "reference") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["e2e"]["value"] == d["value"] and d["cpu_baseline"]["value"] == d["value"]
    # the same `config` as the GPU arm's line (the driver compares the two arms' configs); what this run sampled is
    # said in cpu_baseline
    gpu = json.loads(open(os.path.join(ROOT, "profiles", "r02_bench_n1.json")).read())["config"]
    assert set(d["config"]) == set(gpu)
    assert {k: v for k, v in d["config"].items() if k != "host_cores_per_rank"} == \
           {k: v for k, v in gpu.items() if k != "host_cores_per_rank"}
    assert "full C2 pair" in d["cpu_baseline"]["sample"]
    assert d["cpu_baseline"]["sorters_agree"] is True      # LibDivSufSort and SA-IS restatements: the same suffix array
    # the full-size arrays are written as a seeded sample of the last step's suffix array and streams
    dump = load_dump(tmp_path / "dump")
    assert set(dump) == {"suffix_array", "ctrl", "diff", "extra"}
    sa = dump["suffix_array"]
    assert 0 < sa.size <= 1 << 20 and sa.min() >= 0 and sa.max() < d["config"]["old_bytes"] and sa.dtype == "float64"
    assert sum(dump[k].size for k in ("ctrl", "diff", "extra")) > 0


import pytest


@pytest.mark.parametrize("name", ["r01_bench_n1.json", "r02_bench_n1.json"])
def test_committed_gpu_line_has_the_contract_keys(name):
    d = json.loads(open(os.path.join(ROOT, "profiles", name)).read())
    assert BASE_KEYS | {"gpu_launches", "clocks", "roofline", "cpu_baseline"} <= set(d)
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(d["roofline"])
    assert {"value", "unit", "cores", "kind", "sample"} <= set(d["cpu_baseline"])
    assert {"value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step"} <= set(d["e2e"])
    assert d["gpu_launches"] > 0 and d["n_gpus"] == 1 and abs(d["roofline"]["frac"] - d["roofline"]["achieved"] / d["roofline"]["peak"]) < 1e-9
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])


def test_sharded_record_on_the_emulator(monkeypatch):
    """bench.py's `sharded` record (what rank 0 does at N > 1), run on the CPU logic emulator with tiny inputs and 8
    logical shards: the C4 sort with its in-run sufcheck, the sharded search with its table comparison, the C5 text."""
    import importlib.util
    monkeypatch.setenv("DQ_SHARD_MIN", "1")
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import emu
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    rec = bench.sharded_record([0] * 8, workers=1, lib=emu.library(), scale=2e-5)
    assert "error" not in rec, rec.get("error")
    assert rec["sort_c4"]["sufcheck"] == 0 and rec["sort_c4"]["input_MBps"] > 0
    assert rec["sort_search_256MiB"]["table_equals_one_gpu_table"] is True
    assert rec["sort_c5"]["equals_one_gpu_suffix_array"] is True
    assert rec["sort_c5"]["sampled_adjacent_pairs_out_of_order"] == 0


def test_rank_core_shares_hold_whole_physical_cores():
    """bench.py deals the host's logical CPUs out to the ranks in runs of the (package, core, cpu) order: with sibling
    threads numbered i and i + 4 on two packages, two ranks get one package each and no physical core is shared."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    topo = {0: (0, 0), 1: (0, 1), 2: (1, 0), 3: (1, 1), 4: (0, 0), 5: (0, 1), 6: (1, 0), 7: (1, 1)}
    order = bench.cores_by_physical_core(range(8), topo)
    assert order == [0, 4, 1, 5, 2, 6, 3, 7]
    shares = [order[r * 4:(r + 1) * 4] for r in range(2)]
    assert {topo[c][0] for c in shares[0]} == {0} and {topo[c][0] for c in shares[1]} == {1}
    assert bench.cores_by_physical_core([3, 1, 2], {}) == [1, 2, 3]          # no topology: the plain order
    assert sorted(bench.cores_by_physical_core(os.sched_getaffinity(0))) == sorted(os.sched_getaffinity(0))


def test_bench_main_runs_on_the_emulator(tmp_path):
    """Every line of bench.py's GPU arm (N = 1) executed here, on the emulator with small inputs (tests/bench_on_emulator.py):
    the line carries the contract keys, the in-run parity record holds, no extra record reports an error, and
    --dump-outputs writes the last timed step's arrays, whole at this size and equal to the oracle's."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "bench_on_emulator.py"), "--steps", "2", "--warmup", "3",
                        "--dump-outputs", str(tmp_path / "dump")],
                       capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip().startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert BASE_KEYS | {"gpu_launches", "clocks", "roofline", "cpu_baseline", "parity"} <= set(d)
    assert d["steps"] == 2 and d["warmup"] == 3 and d["n_gpus"] == 1 and d["gpu_launches"] > 0
    assert d["parity"]["streams_identical_to_cpu_baseline"] is True
    assert d["cpu_baseline"]["sorters_agree"] is True
    assert d["e2e"]["h2d_bytes_per_step"] == d["config"]["old_bytes"] + d["config"]["new_bytes"]
    assert "error" not in d["diff_create"], d["diff_create"]
    assert d["diff_create"]["sections_decode_to_the_streams"] and d["diff_create"]["patch_apply"]["reproduces_new"]
    assert len(d["other_configs"]) == 3
    for rec in d["other_configs"]:
        assert "error" not in rec and "abi_error" not in rec, rec
        assert rec["sufcheck"] == 0 and rec["rounds"] >= 1
    import numpy as np
    import oracle
    from deltaq_b200 import workloads as w
    old, new = w.c2_exe_pair(d["config"]["old_bytes"], d["config"]["new_bytes"])   # the pair bench_on_emulator.py gives rank 0
    dump = load_dump(tmp_path / "dump")
    assert set(dump) == {"suffix_array", "match_pos", "match_len", "ctrl", "diff", "extra"}
    sa = oracle.sais(old)
    pos, ln = oracle.search_all(oracle.make_I(sa), old, new)
    ref = oracle.bsdiff_streams(old, new)
    assert np.array_equal(dump["suffix_array"], sa) and dump["suffix_array"].dtype == np.float64
    assert np.array_equal(dump["match_pos"], pos) and np.array_equal(dump["match_len"], ln)
    for k in ("ctrl", "diff", "extra"):
        assert np.array_equal(dump[k], np.frombuffer(ref[k], np.uint8)) and dump[k].dtype == np.float32, k


def test_dump_sample_is_a_fixed_sample():
    """--dump-outputs writes an array longer than DUMP_MAX_ELEMENTS as its entries at seeded positions: the same positions
    in every run, sorted, no more than DUMP_MAX_ELEMENTS of them."""
    import importlib.util
    import numpy as np
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    a = np.arange(3 * bench.DUMP_MAX_ELEMENTS, dtype=np.int32)
    s = bench.dump_sample(a, np.float64)
    assert s.dtype == np.float64 and 0.8 * bench.DUMP_MAX_ELEMENTS < s.size <= bench.DUMP_MAX_ELEMENTS
    assert np.all(np.diff(s) > 0) and np.array_equal(s, bench.dump_sample(a.copy(), np.float64))
    small = np.arange(1000, dtype=np.int32)
    assert np.array_equal(bench.dump_sample(small, np.float32), small)


def test_in_run_parity_digests():
    """bench.py's `parity` record compares digests of the GPU arm's streams with the CPU baseline's: the same function on
    the emulator's streams and the oracle's, for a small pair, must give equal digests (and differ for another pair)."""
    import importlib.util
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import emu
    import oracle
    from deltaq_b200 import CudaSuffixSort
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    rng = np.random.default_rng(5)
    old = rng.integers(0, 4, 30000, dtype=np.uint8)
    new = np.concatenate([old[:9000], rng.integers(0, 256, 77, dtype=np.uint8), old[9500:]])
    with CudaSuffixSort(_lib=emu.library()) as s:
        gpu = bench.stream_digests(s.context.bsdiff_streams(old, new, copy=True))
        view = bench.stream_digests(s.context.bsdiff_streams(old, new, copy=False))
    cpu = bench.stream_digests(oracle.bsdiff_streams(old, new))
    assert gpu == cpu == view and set(gpu) == {"ctrl", "diff", "extra"}
    assert bench.stream_digests(oracle.bsdiff_streams(old, new[:-1])) != cpu


def test_abi_sort_record_on_the_emulator():
    """other_configs' ABI-level timing (dq_cuda_suffix_sort with pinned host buffers) on the emulator, tiny input."""
    import importlib.util
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import emu
    from deltaq_b200 import CudaSuffixSort
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    with CudaSuffixSort(_lib=emu.library()) as s:
        rec = bench.abi_sort_record(s.context, np.random.default_rng(1).integers(0, 256, 20000, dtype=np.uint8), 2)
    assert "abi_error" not in rec, rec
    assert rec["abi_ms"] > 0 and rec["input_MBps_abi"] > 0 and rec["sufcheck"] == 0


def test_bench_main_n2_under_torchrun_on_the_emulator():
    """bench.py's N > 1 flow exactly as the driver launches it (torch.distributed.run, one process per rank), on the
    emulator: every rank pins itself and diffs its own pair, the timings are reduced over the ranks, every rank drops its
    work, all meet on a HOST barrier, rank 0 alone drives the device group (`sharded` record with its in-run checks), all
    meet again; rank 0 prints the one line.  gloo stands in for NCCL, logical shards for the GPUs."""
    import socket
    with socket.socket() as sk:
        sk.bind(("127.0.0.1", 0))
        port = sk.getsockname()[1]
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
                        "--master-addr", "127.0.0.1", "--master-port", str(port),
                        os.path.join(ROOT, "tests", "bench_on_emulator.py"), "--gpus", "2", "--steps", "2", "--warmup", "3"],
                       capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip().startswith("{")]
    assert len(lines) == 1                      # rank 0 alone prints
    d = json.loads(lines[0])
    assert BASE_KEYS | {"gpu_launches", "roofline", "cpu_baseline", "parity", "sharded"} <= set(d)
    assert d["n_gpus"] == 2 and d["scaling"] == "weak" and d["config"]["pairs_per_step"] == 2
    assert d["parity"]["streams_identical_to_cpu_baseline"] is True
    rec = d["sharded"]
    assert "error" not in rec, rec.get("error")
    assert rec["devices"] == [0, 0] and rec["sort_c4"]["sufcheck"] == 0
    assert rec["sort_search_256MiB"]["table_equals_one_gpu_table"] is True


def test_diff_create_record_on_the_emulator():
    """bench.py's `diff_create` record (dq_cuda_bsdiff_patch against serial bzip2 of the same streams), on the CPU logic
    emulator with a small pair."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import emu
    import bench
    from deltaq_b200 import CudaSuffixSort, workloads as w
    sorter = CudaSuffixSort(_lib=emu.library())
    try:
        old, new = w.c2_exe_pair(200_000, 210_000)
        rec = bench.diff_create_record(sorter.context, old, new, reps=1)
    finally:
        sorter.dispose()
    assert "error" not in rec, rec.get("error")
    assert rec["sections_decode_to_the_streams"] is True and rec["patch_bytes"] > 32
    assert rec["patch_apply"]["reproduces_new"] is True
