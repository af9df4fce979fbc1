#!/usr/bin/env python
"""bench.py -- reads/sec through coordinate sort + mark duplicates + BQSR gather/finalize/apply on B200.

One "step" = one pass of the whole hot path over one batch of synthetic 150-bp paired reads:
  value : whole-job reads/s with the reads already resident in HBM when the timed region starts
          (elp_sort_markdup + elp_bqsr_gather + [allreduce of the tables at N>1] + elp_bqsr_finalize + elp_bqsr_apply)
  e2e   : the same metric through the C ABI with HOST buffers: elp_append_batch (H2D from pinned memory) ... elp_fetch (D2H)
Timing: CUDA events on the library's own stream (elp_timer_start/stop), barrier + synchronize on both sides, max over ranks.
Each step re-ingests ~270 B/read (>> the 126 MB L2), so no kernel ever sees a warm L2 from the previous step.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--reads R] [--impl reference] [--dump-outputs DIR]
--dump-outputs DIR writes what the last timed step returned to its caller as DIR/<name>.npy (float32/float64, < 64 MB; see dump_outputs).
N>1 is launched by torchrun (one rank per GPU): ONE hg38-shaped genome is partitioned over the ranks by contig group (sfm-style,
cmd/sfm.go); 1 % of the pairs span two groups.  All cross-GPU traffic of the hot path is NCCL inside the library (C ABI): the spread-pair
exchange of elp_sort_markdup (grouped ncclSend/ncclRecv of 128-byte mate records) and one ncclAllReduce of the integer BQSR tables.  --impl reference times the CPU restatement of the reference algorithm (oracle/, the Go
toolchain being absent) on the host cores, on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

# NCCL's own banner (printed when the box sets NCCL_DEBUG) must not land on stdout, which carries exactly one JSON line
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True      # the benchmark leaves the source tree as it found it (it may be read-only)

METRIC = "reads/sec through sort+markdup+BQSR"
DEFAULT_READS = 30_000_000          # configs[1] scale (WES-scale 30M reads), with the full sort+markdup+BQSR path of configs[2]
GENOME_SCALE = 20.0                 # hg38 / 20 = 155 Mbp  ->  30 M x 150 bp = 29x coverage, WGS-30x-like group statistics
DUMP_ROWS = 1 << 16                 # --dump-outputs: output records in the seeded sample (all of them below this)
DUMP_QUAL_MAX = 10_000_000          # --dump-outputs: QUAL bytes at most (40 MB as float32)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.index, self.rows, self.p = index, [], None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                                      stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.p = None

    def _read(self):
        for line in self.p.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.p:
            self.p.terminate()
        sm, mx, reasons = [], 0, set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except Exception:
                pass
        busy = [x for x in sm if x > 0]
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def pinned(batch):
    """copy the batch columns into page-locked host memory so H2D runs at PCIe speed"""
    import torch
    from elprep_b200 import sam
    kw = {}
    for f in sam.AlignmentBatch.FIELDS:
        a = getattr(batch, f)
        t = torch.empty(a.shape, dtype=getattr(torch, str(a.dtype)) if str(a.dtype) not in ("uint16", "uint32", "uint64") else {"uint16": torch.int16, "uint32": torch.int32, "uint64": torch.int64}[str(a.dtype)], pin_memory=True)
        v = t.numpy().view(a.dtype)
        v[...] = a
        kw[f] = v
        kw.setdefault("_keep", []).append(t)
    keep = kw.pop("_keep")
    b = sam.AlignmentBatch(**kw)
    b._pinned = keep
    return b


def contig_groups(contigs, n):
    from elprep_b200 import multi
    return multi.contig_groups(contigs, n)


def cpu_pipeline(w, n_reads, threads):
    """the CPU restatement (oracle) over the first n_reads reads: markdup -> sort -> gather -> finalize -> apply"""
    import oracle
    from elprep_b200 import synth
    b = synth.take(w.batch, np.arange(min(n_reads, w.batch.n)), threads=threads)
    t0 = time.perf_counter()
    oracle.mark_duplicates(b, w.header, n_threads=threads)
    perm = oracle.coordinate_sort(b, n_threads=threads)
    t1 = time.perf_counter()
    srt = synth.take(b, perm, threads=threads)            # (*sam.Sam) sorts pointers; materialising the order is not part of the reference's work
    t2 = time.perf_counter()
    ref = oracle.Reference(w.header, [b if b is not None else np.zeros(0, np.uint8) for b in w.contig_bases], w.sites)
    t3 = time.perf_counter()
    tb = oracle.bqsr_gather(srt, w.header, ref, n_threads=threads)
    oracle.bqsr_finalize(tb)
    oracle.bqsr_apply(srt, w.header, tb, n_threads=threads)
    t4 = time.perf_counter()
    return b.n, (t1 - t0) + (t4 - t3)


def verify_against_oracle(ctx, w, out_np, n_reads, threads):
    """untimed: the output of the LAST timed step (still in the pinned fetch buffers and in the context) against the oracle run on
    the same reads: output permutation, FLAG of every record, BQSR table counters, EmpiricalQuality, every QUAL byte"""
    import hashlib
    import oracle
    from elprep_b200 import synth
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from util import oracle_tables_dense
    t0 = time.time()
    idx, flag, qoff, qual = out_np
    g_tables, g_emp = ctx.tables_get(), ctx.empirical_get()
    b = w.batch                                   # in place: the timed steps are over
    oracle.mark_duplicates(b, w.header, n_threads=threads)
    perm = oracle.coordinate_sort(b, n_threads=threads)
    srt = synth.take(b, perm, threads=threads)
    ref = oracle.Reference(w.header, w.contig_bases, w.sites)
    tb = oracle.bqsr_gather(srt, w.header, ref, n_threads=threads)
    oracle.bqsr_finalize(tb)
    oracle.bqsr_apply(srt, w.header, tb, n_threads=threads)
    o_tables, o_emp = oracle_tables_dense(tb)
    nq = int(qoff[n_reads])
    checks = {"order": bool(np.array_equal(idx[:n_reads].astype(np.uint64), perm.astype(np.uint64))), "flag": bool(np.array_equal(flag[:n_reads], srt.flag)),
              "tables": bool(np.array_equal(g_tables, o_tables)), "empirical_quality": bool(np.array_equal(g_emp, o_emp)),
              "qual": bool(nq == srt.qual.size and np.array_equal(qual[:nq], srt.qual))}
    return {"ok": all(checks.values()), "checks": checks, "reads": int(n_reads), "duplicates": int(((flag[:n_reads] & 0x400) != 0).sum()),
            "observations": int(g_tables[:, :, 0, 0].sum()), "mismatches": int(g_tables[:, :, 0, 1].sum()),
            "flag_sha256": hashlib.sha256(flag[:n_reads].tobytes()).hexdigest()[:16], "qual_sha256": hashlib.sha256(qual[:nq].tobytes()).hexdigest()[:16],
            "against": "oracle/ (C restatement of the reference) on the same reads", "seconds": round(time.time() - t0, 1)}


def dump_outputs(path, out_np, n_reads, tables, emp, suffix=""):
    """what a caller of the timed path receives after a step, as path/<name><suffix>.npy for output-by-output comparison of two builds:
    the BQSR table counters and EmpiricalQuality in full, and for a fixed seeded sample of output positions (every position when there
    are at most DUMP_ROWS) the input record index, FLAG and QUAL there.  qual holds the QUAL bytes of the sampled records back to back
    (qual_len of each), cut at DUMP_QUAL_MAX bytes; integers are exact in the float type they are stored as."""
    idx, flag, qoff, qual = out_np
    rows = np.arange(n_reads) if n_reads <= DUMP_ROWS else np.unique(np.random.default_rng(20260924).integers(0, n_reads, DUMP_ROWS))
    lo, hi = qoff[rows].astype(np.int64), qoff[rows + 1].astype(np.int64)
    keep = np.cumsum(hi - lo) <= DUMP_QUAL_MAX
    rows, lo, lens = rows[keep], lo[keep], (hi - lo)[keep]
    at = np.repeat(lo - (np.cumsum(lens) - lens), lens) + np.arange(int(lens.sum()))
    arrays = {"rows": rows.astype(np.float64), "order": idx[rows].astype(np.float64), "flag": flag[rows].astype(np.float32),
              "qual_len": lens.astype(np.float32), "qual": qual[at].astype(np.float32),
              "bqsr_tables": np.asarray(tables).astype(np.float64), "empirical_quality": np.asarray(emp).astype(np.float32)}
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, f"{name}{suffix}.npy"), a)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reads", type=int, default=DEFAULT_READS, help="reads per GPU")
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--cpu-sample", type=int, default=3_000_000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-contexts", type=int, default=3, choices=(1, 3), help="contexts in the e2e pipeline ring (1: sequential, for runs where one context fills the HBM)")
    ap.add_argument("--verify", dest="verify", action="store_true", default=None, help="check the last step's output against the oracle (default: on at --gpus 1)")
    ap.add_argument("--no-verify", dest="verify", action="store_false")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    from elprep_b200 import synth
    all_contigs = synth.scaled_hg38(GENOME_SCALE / world)     # weak scaling: the genome grows with the number of GPUs, ~155 Mbp (29x coverage) per contig group
    groups = contig_groups(all_contigs, world)
    contigs = groups[rank]
    threads = min(os.cpu_count() or 1, 64)
    workload_name = (f"one hg38/{GENOME_SCALE / world:g}-shaped genome partitioned into {world} contig group(s) (1 % of the pairs span two groups), "
                     f"{args.reads} synthetic 150-bp paired reads per GPU, sort+markdup+BQSR(gather,finalize,apply)")

    if args.impl == "reference":
        if rank != 0:
            return
        n_sample = min(args.cpu_sample, args.reads)
        w = synth.make_workload(args.reads // 2, contigs, seed=20260924, threads=threads)   # the same workload as our arm; each step processes its first n_sample reads
        times = []
        for i in range(args.warmup + args.steps):
            n, t = cpu_pipeline(w, n_sample, threads)
            if i >= args.warmup:
                times.append(t)
        tt = float(np.sum(times))
        v = n * len(times) / tt
        print(json.dumps({"metric": METRIC, "value": v, "unit": "reads/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                          "ms_per_step": 1e3 * tt / len(times), "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/int64",
                          "data": "synthetic", "impl": "reference", "config": {"workload": workload_name, "flush": "inputs >> L2"},
                          "cpu_baseline": {"value": v, "unit": "reads/s", "cores": threads, "kind": "port",
                                           "sample": f"first {n} reads of the workload per step; C restatement of the elPrep 5.1.3 algorithm (oracle/), not the Go binary"},
                          "e2e": {"value": v, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    import torch
    from elprep_b200 import device
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    t0 = time.time()
    owner = None
    if world == 1:
        w = synth.make_workload(args.reads // 2, contigs, seed=20260924, threads=max(4, threads))
        header, batch, my_contigs = w.header, w.batch, list(range(len(contigs)))
    else:
        # ONE genome partitioned over the ranks by contig group (sfm-style): each rank generates the pairs whose fragment starts in its group; the
        # mates of its cross-contig pairs (1 % of the pairs) land on any contig, so pairs span ranks.  The split step hands every read to the
        # rank that owns its contig (host-side setup, untimed) -- after it a rank holds exactly the reads `elprep split` would have put in its file.
        from elprep_b200 import multi
        header = synth.make_header(all_contigs)
        owner = multi.owner_table(header, groups)
        my_contigs = [i for i in range(len(all_contigs)) if owner[i] == rank]
        home = np.array([1 if owner[i] == rank else 0 for i in range(len(all_contigs))], np.uint8)
        w = synth.make_workload(args.reads // 2, all_contigs, seed=20260924 + rank, home=home, pair_id_base=rank * 10**10, genome_seed=20260924,
                                reference_for=my_contigs, threads=max(4, threads // max(1, world)))
        gen_threads = max(4, threads // max(1, world))
        batch = multi.redistribute(w.batch, owner, rank, world, multi.torch_gather_objects(), take=lambda b, idx: synth.take(b, idx, threads=gen_threads))
        w.batch = batch
    log(f"[rank {rank}] {batch.n} reads on {len(my_contigs)} of {len(all_contigs)} contigs, generated in {time.time() - t0:.1f}s")
    hb = pinned(batch)
    w.batch = batch = hb           # one host copy of the reads from here on (the page-locked one): the CPU legs and --verify read the same arrays
    n_reads = hb.n
    h2d = sum(getattr(hb, f).nbytes for f in hb.FIELDS)

    def make_ctx():
        cx = device.Context(header, device=local, profile=True)
        for ci in my_contigs:
            cx.set_reference(ci, w.contig_bases[ci])
            cx.set_known_sites(ci, w.sites[ci], already_flat=True)
        cx.reserve(n_reads, int(hb.qual.size), int(hb.cigar.size), int(hb.qname.size))
        if world > 1:     # NCCL behind the C ABI: communicator per context, contig -> rank table
            uid = [device.Context.comm_unique_id() if rank == 0 else None]
            dist.broadcast_object_list(uid, src=0)
            cx.comm_init(uid[0], rank, world); cx.comm_set_partition(owner)
        return cx
    ctx = make_ctx()
    # pinned output buffers for the fetch: 32-bit record indices, FLAG, QUAL offsets, QUAL bytes
    out = tuple(torch.empty(s, dtype=dt, pin_memory=True) for s, dt in ((n_reads, torch.int32), (n_reads, torch.int16), (n_reads + 1, torch.int64), (int(hb.qual.size), torch.uint8)))
    out_np = (out[0].numpy().view(np.uint32), out[1].numpy().view(np.uint16), out[2].numpy().view(np.uint64), out[3].numpy())
    d2h = sum(a.nbytes for a in out_np)


    def barrier(cx):
        cx.synchronize(); torch.cuda.synchronize()
        if dist:
            dist.barrier(); torch.cuda.synchronize()

    def phases(cx):
        """the device-resident hot path of one step; returns the time this rank spent in the collective (ms, host clock around a synchronised allreduce)"""
        cx.sort_markdup(device.SO_COORDINATE, True)
        cx.bqsr_gather()
        t_coll = 0.0
        if dist:
            cx.synchronize()
            t0 = time.perf_counter()
            cx.tables_allreduce(); cx.synchronize()           # ncclAllReduce(sum, int64) inside the library, on the context's stream
            t_coll = 1e3 * (time.perf_counter() - t0)
        cx.bqsr_finalize(None)
        cx.bqsr_apply()
        return t_coll

    def step():
        """one step with nothing overlapped: upload | barrier | device-resident region (the `value` clock) | download"""
        ctx.reset()
        barrier(ctx)
        ctx.timer_start()
        ctx.append(hb)
        t_in = ctx.timer_stop()
        barrier(ctx)                            # every rank's reads are resident before any rank starts the device-resident clock
        ctx.timer_start()
        t_coll = phases(ctx)
        t_dev = ctx.timer_stop()
        ctx.timer_start()
        ctx.fetch_async(out_np); ctx.fetch_wait()
        t_out = ctx.timer_stop()
        return t_dev, t_in, t_out, t_coll

    for _ in range(args.warmup):
        step()
    ctx.reset_stats()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    dev_ms, in_ms, out_ms, coll_ms = [], [], [], []
    for _ in range(args.steps):
        a, b, c_, d_ = step()
        dev_ms.append(a); in_ms.append(b); out_ms.append(c_); coll_ms.append(d_)
    launches = ctx.launch_count()
    stats = ctx.kernel_stats()
    if args.dump_outputs:           # untimed, before the e2e run below reuses the context and the output buffers
        dump_outputs(args.dump_outputs, out_np, n_reads, ctx.tables_get(), ctx.empirical_get(), f"_rank{rank}" if world > 1 else "")
    # ---- e2e: the same K steps through the public API with host buffers, software-pipelined over a ring of three contexts: while the
    # batch of step s uploads into one context, the context of step s-1 runs its device phases and starts its download, and the download of
    # step s-2 drains into the other of two page-locked output buffers.  The host->device copy engine -- the longest stage -- never waits.
    # Every step still moves its full input and its full output.
    ring = args.e2e_contexts
    cs = (ctx,) + tuple(make_ctx() for _ in range(ring - 1))
    outs = (out_np, out_np)
    if ring > 1:
        out_b = tuple(torch.empty(s_, dtype=dt, pin_memory=True) for s_, dt in ((n_reads, torch.int32), (n_reads, torch.int16), (n_reads + 1, torch.int64), (int(hb.qual.size), torch.uint8)))
        outs = (out_np, (out_b[0].numpy().view(np.uint32), out_b[1].numpy().view(np.uint16), out_b[2].numpy().view(np.uint64), out_b[3].numpy()))

    trace = {}
    marks = []

    def timed(name, fn):
        t0 = time.perf_counter(); fn(); trace[name] = trace.get(name, 0.0) + 1e3 * (time.perf_counter() - t0)

    def e2e_run(k_steps):
        if ring == 1:                        # capacity runs (one context fills the HBM): no overlap, the same calls in sequence
            for s in range(k_steps):
                timed("reset+append_async", lambda: (ctx.reset(), ctx.append_async(hb))); timed("append_wait", ctx.append_wait)
                timed("phases", lambda: phases(ctx)); timed("fetch_async", lambda: ctx.fetch_async(out_np)); timed("fetch_wait", ctx.fetch_wait)
                marks.append(time.perf_counter())
            return
        for s in range(k_steps + 2):
            cur = cs[s % 3] if s < k_steps else None
            prev = cs[(s - 1) % 3] if 1 <= s <= k_steps else None
            prev2 = cs[(s - 2) % 3] if s >= 2 else None
            if cur is not None:
                timed("reset+append_async", lambda: (cur.reset(), cur.append_async(hb)))
            if prev is not None:
                timed("phases", lambda: phases(prev)); timed("fetch_async", lambda: prev.fetch_async(outs[(s - 1) % 2]))
            if prev2 is not None:
                timed("fetch_wait", prev2.fetch_wait)
            if cur is not None:
                timed("append_wait", cur.append_wait)
            marks.append(time.perf_counter())
    e2e_run(ring)                                # warm-up (allocations of the other contexts)
    trace.clear(); marks.clear()
    barrier(ctx); [c_.synchronize() for c_ in cs]
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    e2e_run(args.steps)
    [c_.synchronize() for c_ in cs]; torch.cuda.synchronize()
    ev1.record(); ev1.synchronize()
    e2e_ms_total = ev0.elapsed_time(ev1)
    mid = np.diff(np.array(marks[:args.steps]))                    # iterations that both upload and run phases
    steady_ms = float(np.median(mid[1:]) * 1e3) if mid.size >= 2 else None
    free_b, total_b = torch.cuda.mem_get_info(local)
    hbm_used_gb = (total_b - free_b) / 1e9                 # all contexts of the ring resident
    clocks = sampler.stop() if rank == 0 else None
    tot = torch.tensor([float(np.sum(dev_ms)), float(e2e_ms_total)], device=f"cuda:{local}", dtype=torch.float64)
    cnt = torch.tensor([float(n_reads)], device=f"cuda:{local}", dtype=torch.float64)
    ph = torch.tensor([float(np.mean(in_ms)), float(np.mean(dev_ms)), float(np.mean(coll_ms)), float(np.mean(out_ms))], device=f"cuda:{local}", dtype=torch.float64)
    ph_all = [ph]
    if dist:
        dist.all_reduce(tot, op=dist.ReduceOp.MAX); dist.all_reduce(cnt, op=dist.ReduceOp.SUM)
        ph_all = [torch.zeros_like(ph) for _ in range(world)]
        dist.all_gather(ph_all, ph)
    dev_total_ms, e2e_total_ms = tot.tolist()
    total_reads = cnt.item()
    phases_per_rank = [{"rank": r, "append_ms": p[0], "device_ms": p[1], "collective_ms": p[2], "fetch_ms": p[3]} for r, p in enumerate(x.tolist() for x in ph_all)]
    if rank != 0:
        if dist:
            dist.barrier(); dist.destroy_process_group()
        return
    value = total_reads * args.steps / (dev_total_ms / 1e3)
    e2e = total_reads * args.steps / (e2e_total_ms / 1e3)
    # roofline of the dominant kernel (largest summed device time over the timed steps)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak, peak_src = (peaks.get("hbm_gbs"), "measured (MEASURED_PEAKS.json hbm_gbs)") if peaks.get("hbm_gbs") else (6650.0, "fallback (B200_PROFILING.md)")
    def roof_of(names, label, traffic_key=None):
        ks = [stats[nm] for nm in names if nm in stats]
        if not ks:
            return None
        ms, by, ln = sum(k["ms"] for k in ks), sum(k["alg_bytes"] for k in ks), sum(k["launches"] for k in ks)
        ach = by / (ms / 1e3) / 1e9 if ms > 0 else None
        traffic = None
        try:   # DRAM bytes per launch from an `ncu --set full` capture of this same workload and build (profiles/r02_traffic.json names the capture)
            tr = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
            ent = tr["kernels"].get(traffic_key or names[0])
            if ent and abs(tr["reads"] - n_reads) <= 0.01 * n_reads and world == 1:
                traffic = ent["dram_bytes_per_launch"]
        except Exception:
            pass
        return {"bound": "hbm", "kernel": label, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak if ach else None, "traffic": traffic, "peak_source": peak_src,
                "launches": ln, "avg_launch_ms": ms / max(1, ln), "alg_bytes_per_launch": by / max(1, ln), "ms_per_step": ms / args.steps}
    dom = max(stats.items(), key=lambda kv: kv[1]["ms"]) if stats else (None, None)
    roof = roof_of([dom[0]], dom[0]) if dom[0] else None
    gather_names = [k for k in stats if k.startswith("bqsr_g_")]
    graded = {"radix_sort": roof_of(["radix_onesweep_u64"], "radix_onesweep_u64 (one digit pass: N*2*(8+4) B)"),
              "covariate_histogram": roof_of(gather_names, "elp_bqsr_gather: " + "+".join(sorted(gather_names)) + " (N_eligible*(19+4+4c+L/2+L) + genome once)", "bqsr_g_count")}
    kern = {n: {"ms_per_step": v["ms"] / args.steps, "launches_per_step": v["launches"] / args.steps,
                "GBps": (v["alg_bytes"] / (v["ms"] / 1e3) / 1e9) if v["ms"] > 0 and v["alg_bytes"] > 0 else None} for n, v in sorted(stats.items(), key=lambda kv: -kv[1]["ms"])}
    cpu = None
    if not args.no_cpu_baseline:
        n_s, t_s = cpu_pipeline(w, args.cpu_sample, threads)
        cpu = {"value": n_s / t_s, "unit": "reads/s", "cores": threads, "kind": "port",
               "sample": f"first {n_s} reads of rank 0's workload, one pass; C restatement of the elPrep 5.1.3 algorithm (oracle/), not the Go binary"}
    verified = None
    if args.verify if args.verify is not None else world == 1:

        ctx.reset(); ctx.append(w.batch); phases(ctx); ctx.fetch_async(out_np); ctx.fetch_wait()      # one more (untimed) pass whose outputs are checked
        verified = verify_against_oracle(ctx, w, out_np, n_reads, threads)
    line = {"metric": METRIC, "value": value, "unit": "reads/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8/int64", "data": "synthetic",
            "config": {"workload": workload_name, "cpu_arm": f"CPU arm runs a sample: the first {args.cpu_sample} reads per step", "reads_per_gpu": n_reads, "parallelism": f"contig-group x{world}; NCCL inside the C ABI: spread-pair exchange (ncclSend/Recv) in elp_sort_markdup + one ncclAllReduce of the BQSR tables", "flush": "inputs >> L2 (re-ingested every step)"},
            "e2e": {"value": e2e, "unit": "reads/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": e2e_total_ms / args.steps,
                    "how": ("K steps through elp_append_batch_async / phases / elp_fetch_async with pinned host buffers, " +
                            ("software-pipelined over a ring of three contexts and two output buffers (upload of step s overlaps the phases of step s-1 and the download of steps s-1 / s-2)" if ring > 1 else "one context, the calls in sequence (no overlap)")),
                    "unpipelined_ms_per_step": float(np.mean(in_ms) + np.mean(dev_ms) + np.mean(out_ms)),
                    "host_ms_per_step_in_call": {k: v / args.steps for k, v in trace.items()}, "contexts": ring, "hbm_used_gb_all_contexts": hbm_used_gb,
                    "steady_ms_per_step": steady_ms, "note": "ms_per_step = the K timed steps including pipeline fill (first upload) and drain (last phases + download); steady_ms_per_step = median host interval between consecutive steps in the middle of the run"},
            "phases_per_rank": phases_per_rank, "roofline_graded": graded,
            "gpu_launches": launches, "verified": (verified or {}).get("ok"), "verify": verified, "roofline": roof, "cpu_baseline": cpu, "clocks": clocks, "kernels": kern}
    print(json.dumps(line))
    if dist:
        dist.barrier(); dist.destroy_process_group()


if __name__ == "__main__":
    main()
