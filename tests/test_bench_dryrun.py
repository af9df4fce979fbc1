"""Rehearsal of bench.py's own Python on the CPU: main() runs end to end against a stand-in for elprep_b200.device.Context whose
phases are the ORACLE (so --verify compares like with like) and a stand-in for the handful of torch.cuda calls.  Nothing here measures
or proves anything about the GPU path -- it only keeps the bench script's control flow, its pipelined e2e ring and the JSON line it prints
from breaking unnoticed between GPU sessions (the contract: one JSON line with metric / value / e2e / roofline / cpu_baseline / clocks)."""
import io
import json
import os
import sys
import time
from contextlib import redirect_stdout

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


class FakeContext:
    SO_COORDINATE = 4
    live = 0

    def __init__(self, header, device=0, profile=False, **kw):
        self.header, self.batch, self.ref, self.sites = header, None, {}, {}
        self.n, self._launches, self._t0, self.res = 0, 0, None, None
        FakeContext.live += 1

    # side inputs / lifecycle
    def set_reference(self, ci, bases): self.ref[ci] = bases
    def set_known_sites(self, ci, se, already_flat=False): self.sites[ci] = se
    def reserve(self, *a): pass
    def reset(self): self.batch, self.res, self.n = None, None, 0
    def synchronize(self): pass
    def reset_stats(self): self._launches = 0
    def launch_count(self): return self._launches
    def kernel_stats(self): return {"bqsr_apply": dict(launches=3, ms=3.0, alg_bytes=3e6), "bqsr_g_count": dict(launches=3, ms=2.0, alg_bytes=2e6), "radix_onesweep_u64": dict(launches=30, ms=1.0, alg_bytes=5e6)}
    def timer_start(self): self._t0 = time.perf_counter()
    def timer_stop(self): return 1e3 * (time.perf_counter() - self._t0) + 1e-3
    def close(self): pass

    # ingest
    def append(self, b): self.batch = b; self.n = b.n
    def append_async(self, b): self.append(b)
    def append_wait(self): pass

    # phases: the oracle
    def sort_markdup(self, order, markdup):
        import oracle
        self._launches += 40
        b = self.batch.copy()
        if markdup:
            oracle.mark_duplicates(b, self.header, n_threads=2)
        self.perm = oracle.coordinate_sort(b, n_threads=2)
        self.srt = b.take(self.perm)

    def bqsr_gather(self):
        import oracle
        self._launches += 8
        contig_bases = [self.ref[i] for i in range(len(self.header.SQ))]
        sites = [self.sites[i] for i in range(len(self.header.SQ))]
        self.oref = oracle.Reference(self.header, contig_bases, sites)
        self.t = oracle.bqsr_gather(self.srt, self.header, self.oref, n_threads=2)

    def bqsr_finalize(self, path):
        import oracle
        oracle.bqsr_finalize(self.t)

    def bqsr_apply(self):
        import oracle
        self._launches += 1
        oracle.bqsr_apply(self.srt, self.header, self.t, n_threads=2)

    def tables_get(self):
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from util import oracle_tables_dense
        return oracle_tables_dense(self.t)[0]

    def empirical_get(self):
        from util import oracle_tables_dense
        return oracle_tables_dense(self.t)[1]

    # egress
    def fetch_async(self, out, first=0, n=None):
        idx, flag, qoff, qual = out
        idx[:self.n] = self.perm.astype(np.uint32); flag[:self.n] = self.srt.flag; qoff[:self.n + 1] = self.srt.qual_off; qual[:self.srt.qual.size] = self.srt.qual

    def fetch_wait(self): pass


class FakeEvent:
    def __init__(self, enable_timing=True): self.t = None
    def record(self): self.t = time.perf_counter()
    def synchronize(self): pass
    def elapsed_time(self, other): return 1e3 * (other.t - self.t)


def _fake_gpu_bench(monkeypatch):
    """bench.py with the fake device, its torch.cuda calls stubbed and a ~1 Mbp genome"""
    import torch
    sys.path.insert(0, ROOT)
    import bench
    from elprep_b200 import device
    real_empty, real_tensor = torch.empty, torch.tensor
    monkeypatch.setattr(torch, "empty", lambda *a, pin_memory=False, **k: real_empty(*a, **k))
    monkeypatch.setattr(torch, "tensor", lambda *a, device=None, **k: real_tensor(*a, **k))
    monkeypatch.setattr(torch.cuda, "set_device", lambda *a: None)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a: None)
    monkeypatch.setattr(torch.cuda, "Event", FakeEvent)
    monkeypatch.setattr(torch.cuda, "mem_get_info", lambda *a: (100 * 10**9, 180 * 10**9))
    monkeypatch.setattr(device, "Context", FakeContext)
    monkeypatch.setattr(device, "SO_COORDINATE", 4, raising=False)
    monkeypatch.setattr(bench.ClockSampler, "start", lambda self: None)
    monkeypatch.setattr(bench.ClockSampler, "stop", lambda self: {"sm_mhz": 1965.0, "sm_max_mhz": 1965.0, "reasons": [], "samples": 3})
    monkeypatch.setattr(bench, "GENOME_SCALE", 3000.0)              # a ~1 Mbp genome for 12 k reads
    for k in ("RANK", "WORLD_SIZE", "LOCAL_RANK"):
        monkeypatch.delenv(k, raising=False)
    return bench


def _run_bench(monkeypatch, bench, argv):
    monkeypatch.setattr(sys, "argv", ["bench.py"] + argv)
    buf = io.StringIO()
    with redirect_stdout(buf):
        bench.main()
    lines = [ln for ln in buf.getvalue().splitlines() if ln.strip()]
    assert len(lines) == 1, lines                                   # exactly one JSON line on stdout
    return json.loads(lines[0])


@pytest.mark.parametrize("extra", [[], ["--e2e-contexts", "1", "--steps", "1"]])
def test_bench_main_runs_and_prints_one_contract_line(monkeypatch, extra):
    bench = _fake_gpu_bench(monkeypatch)
    d = _run_bench(monkeypatch, bench, ["--reads", "12000", "--steps", "4", "--warmup", "1", "--cpu-sample", "6000"] + extra)
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config",
                "e2e", "roofline", "roofline_graded", "cpu_baseline", "clocks", "gpu_launches", "verified"):
        assert key in d, key
    assert d["n_gpus"] == 1 and d["unit"] == "reads/s" and d["higher_is_better"] is True and d["config"]["workload"]
    assert d["verified"] is True and all(d["verify"]["checks"].values())
    e = d["e2e"]
    assert e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["value"] > 0 and e["contexts"] == (1 if extra else 3)
    assert (e["steady_ms_per_step"] is None) == bool(extra)         # needs >= 3 pipelined steps
    assert d["roofline"]["kernel"] == "bqsr_apply" and 0 < d["roofline"]["frac"] and set(d["roofline_graded"]) == {"radix_sort", "covariate_histogram"}
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["value"] > 0 and d["gpu_launches"] > 0


def test_bench_steps_and_dump_outputs(monkeypatch, tmp_path):
    """--steps is the number of timed steps (the fake launches 49 kernels a step); --dump-outputs writes, as float arrays under 64 MB, the
    outputs the last timed step fetched (a seeded sample of output positions, QUAL cut at DUMP_QUAL_MAX bytes), the same on every run"""
    bench = _fake_gpu_bench(monkeypatch)
    monkeypatch.setattr(bench, "DUMP_ROWS", 3000)
    monkeypatch.setattr(bench, "DUMP_QUAL_MAX", 300_000)            # 3000 records x 150 B: the cut applies
    fetched = []
    real_dump = bench.dump_outputs

    def spy(path, out_np, n_reads, tables, emp, suffix=""):
        fetched.append(([a.copy() for a in out_np], tables.copy(), emp.copy()))
        real_dump(path, out_np, n_reads, tables, emp, suffix)
    monkeypatch.setattr(bench, "dump_outputs", spy)
    dumps = []
    for k in (2, 5):
        out = tmp_path / f"steps{k}"
        d = _run_bench(monkeypatch, bench, ["--reads", "12000", "--steps", str(k), "--warmup", "1", "--no-cpu-baseline", "--dump-outputs", str(out)])
        assert d["steps"] == k and d["gpu_launches"] == 49 * k and d["verified"] is True
        files = sorted(os.listdir(out))
        assert files == sorted(f"{n}.npy" for n in ("rows", "order", "flag", "qual_len", "qual", "bqsr_tables", "empirical_quality"))
        assert sum(os.path.getsize(out / f) for f in files) <= 64 << 20
        a = {f[:-4]: np.load(out / f) for f in files}
        assert all(x.dtype in (np.float32, np.float64) for x in a.values())
        dumps.append(a)
    assert dumps[0].keys() == dumps[1].keys() and all(np.array_equal(dumps[0][n], dumps[1][n]) for n in dumps[0])
    (idx, flag, qoff, qual), tables, emp = fetched[-1]
    a = dumps[-1]
    rows = a["rows"].astype(np.int64)
    assert 0 < rows.size < 3000 and np.all(np.diff(rows) > 0) and a["qual"].size == a["qual_len"].sum() <= 300_000
    assert np.array_equal(a["order"], idx[rows]) and np.array_equal(a["flag"], flag[rows])
    assert np.array_equal(a["qual"], np.concatenate([qual[qoff[r]:qoff[r + 1]] for r in rows]))
    assert np.array_equal(a["bqsr_tables"], tables) and np.array_equal(a["empirical_quality"], emp) and tables.sum() > 0


def _rank_main(rank, world, port, out_dir):
    """one rank of `torchrun bench.py --gpus 2`, with gloo standing in for NCCL and the fake device"""
    import torch
    import torch.distributed as dist
    sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
    import bench
    from elprep_b200 import device
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    real_empty, real_tensor, real_init = torch.empty, torch.tensor, dist.init_process_group
    torch.empty = lambda *a, pin_memory=False, **k: real_empty(*a, **k)
    torch.tensor = lambda *a, device=None, **k: real_tensor(*a, **k)
    torch.cuda.set_device = lambda *a: None
    torch.cuda.synchronize = lambda *a: None
    torch.cuda.Event = FakeEvent
    torch.cuda.mem_get_info = lambda *a: (100 * 10**9, 180 * 10**9)
    dist.init_process_group = lambda backend=None, device_id=None, **k: real_init("gloo", rank=rank, world_size=world)

    class Ctx(FakeContext):
        @staticmethod
        def comm_unique_id(): return b"\0" * 128
        def comm_init(self, uid, r, w): assert (r, w) == (rank, world) and len(uid) == 128
        def comm_set_partition(self, owner): self.owner = np.asarray(owner)
        def tables_allreduce(self): pass
        def bqsr_gather(self):             # a rank only has the reference of its own contigs: the fake skips BQSR
            self._launches += 8
        def bqsr_finalize(self, path): pass
        def bqsr_apply(self): self._launches += 1
    device.Context = Ctx
    device.SO_COORDINATE = 4
    bench.ClockSampler.start = lambda self: None
    bench.ClockSampler.stop = lambda self: {"sm_mhz": 1965.0, "sm_max_mhz": 1965.0, "reasons": [], "samples": 3}
    bench.GENOME_SCALE = 3000.0
    sys.argv = ["bench.py", "--gpus", str(world), "--reads", "12000", "--steps", "3", "--warmup", "1", "--cpu-sample", "3000"]
    buf = io.StringIO()
    with redirect_stdout(buf):
        bench.main()
    open(os.path.join(out_dir, f"stdout_{rank}.txt"), "w").write(buf.getvalue())


def test_bench_two_ranks_over_gloo(tmp_path):
    """the N > 1 control flow of bench.py: one genome split over two ranks, per-rank phase times gathered, only rank 0 prints"""
    import torch.multiprocessing as mp
    port = 29100 + (os.getpid() % 300)
    mp.spawn(_rank_main, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    out0 = [ln for ln in open(tmp_path / "stdout_0.txt").read().splitlines() if ln.strip()]
    out1 = [ln for ln in open(tmp_path / "stdout_1.txt").read().splitlines() if ln.strip()]
    assert len(out0) == 1 and out1 == []
    d = json.loads(out0[0])
    assert d["n_gpus"] == 2 and d["scaling"] == "weak" and d["verified"] is None
    assert [p["rank"] for p in d["phases_per_rank"]] == [0, 1] and all(p["device_ms"] > 0 for p in d["phases_per_rank"])
    assert "2 contig group(s)" in d["config"]["workload"] and d["e2e"]["contexts"] == 3 and d["value"] > 0
