#!/usr/bin/env python3
"""Headline benchmark: genome Gbp/s scanned + scored (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                  [--workload arabidopsis|sorghum|maize|sugarcane|sample] [--no-extra] [--no-cpu-baseline]
                  [--dump-outputs DIR]

A "step" is one pass of the hot path (PAM scan both strands + ordered compaction + Rule-Set-1
scoring of every candidate) over one synthetic genome (tools/workloads.py).  K steps are timed,
after W >= 3 untimed ones; the end-to-end leg below times K steps of its own.

  --dump-outputs DIR   after the timed steps, write what the last one computed as float64 .npy files
          (dump_outputs below): the per-segment candidate counts, and of each strand stream a fixed,
          seeded sample of at most 2^19 rows (row index, pos, fp64 x, packed 30-mer as two 32-bit
          halves).  The inputs are seeded, so two builds run with the same arguments can be compared
          file by file.

  N = 1   configs[1] (Arabidopsis-scale); the other single-GPU configs ride along as extra keys
  N > 1   STRONG scaling: ONE genome (configs[3], maize-scale; at N = 8 also configs[4], sugarcane-
          scale, under "largest") is cut into N contiguous tile-aligned shards, one process and one
          GPU per shard.  The one exchange step -- the NCCL all-gather of the per-segment candidate
          counts -- runs inside the library on the scan's stream, so the CUDA events that time a step
          bracket kernel + collective.  Rank 0 also scans the whole genome alone in the same run
          ("strong_scaling.single_gpu_ms"): the denominator an efficiency needs.

  value   whole-job Gbp/s with the packed genome already resident in HBM, CUDA events on the
          library's stream, mean over the timed steps, max over ranks; L2 flushed between steps
  e2e     the same metric through the C ABI from pinned HOST buffers (crp_scan_segments): ASCII
          tokens -> H2D -> pack -> scan+score+logistic -> D2H of the rows a CSV writer needs
          (pos u32 + score f64), wall clock between barriers, count exchange included
  roofline / cpu_baseline / clocks / link_ceiling: DESIGN.md "Measurement".

Launch for N > 1: `python -m torch.distributed.run --nproc-per-node N ... bench.py --gpus N` (or any
launcher that sets RANK / LOCAL_RANK / WORLD_SIZE / MASTER_ADDR / MASTER_PORT); ranks find each other
over the TCP rendezvous of cropsr_b200/launch.py -- no PyTorch in this process.
"""
import argparse
import faulthandler
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "tools")):
    if _p not in sys.path:
        sys.path.insert(0, _p)
faulthandler.enable()

import workloads as W      # noqa: E402  (tools/workloads.py)

METRIC = "genome Gbp/s scanned+scored"
CONFIG_NAME = W.CONFIG_NAME


# round 1 imported these from here; the generators now live in tools/workloads.py
WORKLOADS = {k: (v["seed"], v["lengths"], v["gc"], v["lower"]) for k, v in W.WORKLOADS.items() if v["lengths"] is not None}


def synth_tokens(name, only=None, copies=1):
    assert copies == 1
    return W.tokens(name, only)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                      "-i", str(self.index)], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([c.strip() for c in out.strip().split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.1)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        sm = [float(r[0]) for r in self.rows if len(r) == 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) == 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({n for r in self.rows if len(r) == 6 for n, v in zip(names, r[2:]) if v == "Active"})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def measured_traffic(workload):
    """dram__bytes_read.sum + dram__bytes_write.sum of one scan launch on this workload, from the
    committed `ncu --set full` capture (profiles/traffic.json)."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f)[workload]["dram_bytes_per_launch"]
    except Exception:
        return None


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ---------------------------------------------------------------------------------- CPU arm
_SAMPLE_CACHE = {}


def _reference_sample_files(workload, per, n_rec):
    """The sample FASTA / GFF of a workload, written once per process (generating five chromosomes costs
    seconds; the reference arm runs the same sample every step)."""
    key = (workload, per, n_rec)
    if key not in _SAMPLE_CACHE:
        wd = tempfile.mkdtemp(prefix="cropsr_ref_sample_")
        fa, gff = os.path.join(wd, "sample.fa"), os.path.join(wd, "sample.gff")
        W.write_fasta(workload, fa, records=range(n_rec), prefix_bases=per)
        W.write_gff(workload, gff, records=range(n_rec), prefix_bases=per)
        _SAMPLE_CACHE[key] = (fa, gff)
    return _SAMPLE_CACHE[key]


def reference_sample(workload, seconds_target):
    """One run of the reference's CPU implementation on a bounded MULTI-RECORD sample of the
    workload: the first `per` bases of each of its first (up to) 5 records, written as the same
    80-column FASTA our arm's tokens stand for.  The unmodified reference (baseline/_ref, see
    oracle/install_reference.py) when it is installed, else the oracle's literal port.
    -> (cpu_baseline dict, seconds, bases)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import run_reference
    n_rec = min(5, len(W.lengths(workload)))
    # ~0.19 Mbp/s in-program on this class of host, cumulative re-emission of earlier records included
    per = int(max(20_000, min(min(W.lengths(workload)[:n_rec]), seconds_target * 0.17e6 / n_rec)))
    fa, gff = _reference_sample_files(workload, per, n_rec)
    with tempfile.TemporaryDirectory() as wd:
        n_bases = per * n_rec
        what = (f"first {per} bp of each of the first {n_rec} records of the {workload} workload "
                f"({n_bases} bp, 80-column FASTA + synthetic GFF)")
        if run_reference.available():
            r = run_reference.run(fa, gff, os.path.join(wd, "out.csv"), wd)
            dt = r["program_s"] or r["main_s"]
            rows = sum(1 for _ in open(os.path.join(wd, "out.csv"))) - 1
            cb = {"value": n_bases / dt / 1e9, "unit": "Gbp/s", "cores": r["blas_threads"] or (os.cpu_count() or 1),
                  "kind": "reference",
                  "sample": what + f"; UNMODIFIED reference CLI (baseline/_ref/CROPSR.py --cas9, time.sleep stubbed): "
                            f"{rows} CSV rows, in-program time {dt:.1f} s (its own time.txt), wall {r['wall_s']:.1f} s with "
                            f"imports; single-threaded Python, {r['blas_threads']} OpenBLAS threads inside np.matmul only",
                  "program_s": dt, "wall_s": r["wall_s"]}
            return cb, dt, n_bases
        import cropsr_oracle as oracle
        with open(fa) as f:
            text = f.read()
        np.random.seed(0)
        dt, nb, rows = oracle.timed_reference_pass(text, 20)
        threads = int(os.environ.get("OPENBLAS_NUM_THREADS", os.cpu_count() or 1))
        cb = {"value": n_bases / dt / 1e9, "unit": "Gbp/s", "cores": threads, "kind": "port",
              "sample": what + f"; baseline/_ref is not installed here, so the oracle's literal port ran "
                        f"(oracle/cropsr_oracle.py, {rows} rows, {dt:.1f} s)"}
        return cb, dt, n_bases


def run_reference_arm(args, rank):
    """bench.py --impl reference: the reference's own CPU path on the host cores, rank 0 only."""
    if rank != 0:
        return
    workload = args.workload or ("arabidopsis" if args.gpus <= 1 else "maize")
    per_step = max(4.0, min(60.0, 150.0 / (args.warmup + args.steps)))
    times, nb, cb = [], 0, None
    for i in range(args.warmup + args.steps):
        cb, dt, nb = reference_sample(workload, per_step)
        if i >= args.warmup:
            times.append(dt)
    t = float(np.mean(times))
    v = nb / t / 1e9
    cb["value"] = v
    print(json.dumps({"impl": "reference", "metric": METRIC, "value": v, "unit": "Gbp/s", "n_gpus": args.gpus,
                      "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3, "higher_is_better": True,
                      "scaling": "strong" if args.gpus > 1 else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                      "config": {"workload": CONFIG_NAME[workload], "guide_len": 20,
                                 "note": "bounded multi-record sample of the workload per step (cpu_baseline.sample)"},
                      "cpu_baseline": cb,
                      "e2e": {"value": v, "unit": "Gbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


# ---------------------------------------------------------------------------------- our arm
class Shard:
    """This rank's part of a workload: pinned token buffers + the packed genome in HBM."""

    def __init__(self, engine, shard_mod, workload, rank, world, pinned=True):
        self.engine, self.workload, self.rank, self.world = engine, workload, rank, world
        self.lengths = W.token_lengths(workload)
        self.n_bases_total = sum(self.lengths)
        self.plans = shard_mod.plan(self.lengths, world)
        self.mine = self.plans[rank]
        self.slots = max(1, max(len(p) for p in self.plans))
        self.host_tokens = {}
        self._pinned = []
        for k in sorted({k for k, _, _ in self.mine}):
            t = W.token(workload, k)
            if pinned:
                buf = engine.PinnedBuffer(len(t))
                buf.array[:] = t
                self._pinned.append(buf)
                t = buf.array
            self.host_tokens[k] = t
        self.my_bases = sum(b - a for _, a, b in self.mine)
        # one genome handle addresses 2^32 positions: a bigger shard (10 Gbp on one GPU) becomes several
        # handles scanned back to back, exactly as the product path does (pipeline.scan_token_bytes)
        self.groups, acc = [[]], 0
        for seg in self.mine:
            n = seg[2] - seg[1]
            if self.groups[-1] and acc + n > (1 << 31):
                self.groups.append([])
                acc = 0
            self.groups[-1].append(seg)
            acc += n
        if len(self.groups) > 1 and world > 1:
            raise SystemExit(f"{workload}: {self.my_bases} positions per GPU need several genome handles; the sharded "
                             "scan of this benchmark takes one per rank -- run it on more GPUs")
        self.genomes = [self.build(g) for g in self.groups]
        self.genome = self.genomes[0]

    def build(self, group=None):
        g = self.engine.Genome()
        for k, a, b in (self.mine if group is None else group):
            g.add_segment(k, self.host_tokens[k], a, b)
        return g.commit()

    def scan(self):
        if self.world > 1:
            return self.genome.scan_sharded(self.slots, 20)
        if len(self.genomes) == 1:
            return self.genome.scan(20)
        return _ManyResults([g.scan(20) for g in self.genomes])

    def free(self):
        for g in self.genomes:
            g.free()
        for b in self._pinned:
            b.free()
        self._pinned, self.host_tokens = [], {}


class _ManyResults:
    """the scans of the several genome handles of one oversized shard, timed as one step"""

    def __init__(self, results):
        self.results = results
        self.n_plus = sum(r.n_plus for r in results)
        self.n_minus = sum(r.n_minus for r in results)

    def timing_detail(self):
        ds = [r.timing_detail() for r in self.results]
        return {"kernel_ms": sum(d["kernel_ms"] for d in ds), "total_ms": sum(d["total_ms"] for d in ds),
                "launches": sum(d["launches"] for d in ds) - len(ds) + 1}

    def free(self):
        for r in self.results:
            r.free()


def time_scans(engine, sh, steps, warmup, sampler_index=None, keep_last=False):
    """-> dict(ms mean of kernel(+collective) per step on this rank, kernel_ms, candidates, launches, wall_ms, clocks,
    last: the result of the last step if keep_last, else None; the caller frees it)"""
    total_ms, kernel_ms, n_cand, last = [], [], 0, None
    launches0, sampler, t_wall0, relaunched = 0, None, 0.0, 0
    for i in range(warmup + steps):
        if i == warmup:
            engine.comm_barrier()
            launches0 = engine.launch_count()
            if sampler_index is not None:
                sampler = ClockSampler(sampler_index)
                sampler.start()
            t_wall0 = time.perf_counter()
        engine.flush_l2()                         # a 512 MiB memset, waited for: no scan finds its records in L2
        engine.comm_barrier()                     # barrier + device synchronize on both sides of every step
        res = sh.scan()
        if i >= warmup:
            d = res.timing_detail()
            total_ms.append(d["total_ms"])
            kernel_ms.append(d["kernel_ms"])
            relaunched += d["launches"] - 1
        n_cand = res.n_plus + res.n_minus
        if keep_last and i == warmup + steps - 1:
            last = res
        else:
            res.free()
    engine.comm_barrier()
    wall_ms = (time.perf_counter() - t_wall0) * 1e3 / steps
    return {"ms": float(np.mean(total_ms)), "kernel_ms": float(np.mean(kernel_ms)), "candidates": int(n_cand),
            "launches": engine.launch_count() - launches0, "wall_ms": wall_ms, "capacity_reruns": relaunched,
            "sampler": sampler, "last": last}


DUMP_ROWS = 1 << 19        # rows per strand, shared by all ranks: 2 strands x 5 float64 columns x 2^19 rows = 40 MiB


def dump_outputs(res, out_dir, rank, world):
    """What a caller of the scan gets back (ScanResult.fetch of both strands, per-segment counts), as float64
    .npy files under out_dir: every count, and of each strand a sample of rows drawn with a fixed seed from
    the row count alone, so two builds that agree on the counts sample the same rows.  Exact in float64:
    pos and the two halves of the packed 30-mer are 32-bit integers.  Several ranks: files rank<r>_*.npy."""
    os.makedirs(out_dir, exist_ok=True)
    prefix = f"rank{rank}_" if world > 1 else ""
    parts = res.results if isinstance(res, _ManyResults) else [res]

    def save(name, a):
        np.save(os.path.join(out_dir, prefix + name + ".npy"), np.asarray(a, dtype=np.float64))

    save("seg_counts", [np.concatenate([r.seg_plus for r in parts]), np.concatenate([r.seg_minus for r in parts])])
    for strand, name in (("+", "plus"), ("-", "minus")):
        rows = [r.fetch(strand) for r in parts]
        pos, packed, x = (np.concatenate([f[k] for f in rows]) for k in ("pos", "packed", "x"))
        n = len(pos)
        keep = DUMP_ROWS // world
        idx = np.arange(n) if n <= keep else np.sort(np.random.default_rng(20).choice(n, keep, replace=False))
        save(f"{name}_row", idx)
        save(f"{name}_pos", pos[idx])
        save(f"{name}_x", x[idx])
        save(f"{name}_packed_lo", packed[idx] & np.uint64(0xFFFFFFFF))
        save(f"{name}_packed_hi", packed[idx] >> np.uint64(32))


def roofline(my_bases, n_cand, kernel_ms, workload, world):
    peak, peak_src = measured_peak()
    alg_bytes = 0.5 * my_bases + 20.0 * n_cand          # SURVEY 8d, this rank's launch
    achieved = alg_bytes / (kernel_ms * 1e-3) / 1e9
    return {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
            "traffic": measured_traffic(workload) if world == 1 else None, "peak_source": peak_src,
            "kernel_ms": kernel_ms,
            "algorithmic_bytes": "0.5 B/base read + 20 B/candidate written (pos u32, packed u64, x f64)"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=None, choices=sorted(W.WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the ride-along workloads / single-GPU denominator")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step computed to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup     # timing rule: W >= 3

    from cropsr_b200 import launch
    rank, world, local = launch.env_rank()
    if args.impl == "reference":
        return run_reference_arm(args, rank)

    from cropsr_b200 import engine, shard, _native as N
    cpus_before = os.sched_getaffinity(0)
    numa_node = engine.bind_host_near(local)      # before any pinned allocation: staging buffers next to the GPU
    engine.init(local)
    rdv = launch.Rendezvous(rank, world)
    launch.init_comm(rdv, engine)

    workload = args.workload or ("arabidopsis" if world == 1 else "maize")
    sh = Shard(engine, shard, workload, rank, world)
    n_bases_total = sh.n_bases_total

    # ---- device-resident metric: kernel (+ all-gather of the counts for N > 1) between CUDA events
    # nvidia-smi is polled by rank 0 only: eight pollers at 10 Hz each take driver locks that every rank's CUDA calls need
    t = time_scans(engine, sh, args.steps, args.warmup, sampler_index=local if rank == 0 else None,
                   keep_last=args.dump_outputs is not None)
    if t["last"] is not None:
        dump_outputs(t["last"], args.dump_outputs, rank, world)
        t["last"].free()
    sampler = t["sampler"]
    ms = float(engine.comm_max([t["ms"]])[0])                      # the slowest rank sets the step
    value = n_bases_total / (ms * 1e-3) / 1e9
    n_cand_total = int(engine.comm_sum([t["candidates"]])[0])
    per_rank = rdv.all_gather({"rank": rank, "tiles": sum(-(-(b - a) // engine.TILE) for _, a, b in sh.mine),
                               "candidates": t["candidates"], "kernel_ms": t["kernel_ms"], "step_ms": t["ms"]})

    # ---- end to end from host buffers (pinned in, pinned out), through the pipelined C-ABI call:
    # per segment H2D -> pack -> scan+score+logistic -> D2H of (pos, score), then the count exchange
    segs = [(k, sh.host_tokens[k], a, b) for k, a, b in sh.mine]
    want = ("pos", "x")
    arena, e2e_ms, h2d, d2h = None, [], 0, 0
    e2e_warmup = max(args.warmup, 5)           # the block cache of the pipelined call settles within the first calls
    for i in range(e2e_warmup + args.steps):
        engine.comm_barrier()
        t0 = time.perf_counter()
        arena, n_plus, n_minus, _ = engine.scan_segments(segs, 20, flags=N.CRP_SCAN_LOGISTIC, arena=arena, want=want)
        counts = np.zeros(2 * sh.slots, dtype=np.uint64)
        counts[:len(n_plus)] = n_plus
        counts[sh.slots:sh.slots + len(n_minus)] = n_minus
        gathered = engine.comm_allgather(counts).reshape(world, 2, sh.slots)      # the exchange step (NCCL)
        shard.global_offsets(sh.plans, [(gathered[r, 0, :len(sh.plans[r])], gathered[r, 1, :len(sh.plans[r])])
                                        for r in range(world)])
        engine.comm_barrier()
        dt = (time.perf_counter() - t0) * 1e3
        if i >= e2e_warmup:
            e2e_ms.append(dt)
        h2d = sum(min(b + 32, sh.lengths[k]) - max(a - 32, 0) for k, a, b in sh.mine)
        d2h = 12 * int(n_plus.sum() + n_minus.sum())
    clocks = sampler.summary() if sampler is not None else None      # sampled from the first timed scan to the last end-to-end step
    e2e = float(engine.comm_max([float(np.mean(e2e_ms))])[0])
    h2d_total, d2h_total = (int(v) for v in engine.comm_sum([float(h2d), float(d2h)]))

    # ---- what the link allows: the same bytes both ways at once, nothing else (all ranks together)
    engine.comm_barrier()
    link_ms = float(engine.comm_max([engine.link_probe(h2d, d2h, 5)])[0])
    if True:
        link = {"ms_per_step": link_ms, "value": n_bases_total / (link_ms * 1e-3) / 1e9, "unit": "Gbp/s",
                "what": "concurrent pinned H2D + D2H cudaMemcpyAsync of exactly the e2e byte counts on every rank, no kernels"}
    if arena is not None:
        arena.free()
    g = sh.build(sh.groups[0])       # a warm commit (the first one of a process pays lazy module loading)
    ingest_timing = g.timing()
    g.free()

    line = None
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": "Gbp/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong" if world > 1 else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": CONFIG_NAME[workload], "bases": n_bases_total, "candidates": n_cand_total,
                       "guide_len": 20, "sharding": f"ONE genome, {world} contiguous shard(s), tile-aligned, halo 32/32",
                       "collective": "ncclAllGather of per-segment counts inside the library, on the scan stream, "
                                     "inside the timed events" if world > 1 else "none (1 GPU)",
                       "l2": "flushed between steps (512 MiB memset)", "host_numa_node": numa_node,
                       "resident": "the packed genome as k_pack leaves it: tile records (0.5 B/base), PAM records, and 48-byte tile "
                                   "headers with the PAM hit counts of every 2,048-position chunk under the guide-independent bounds "
                                   "(the scan's count phase reads the headers; building them is part of `ingest` and of `e2e`)"},
            "e2e": {"value": n_bases_total / (e2e * 1e-3) / 1e9, "unit": "Gbp/s", "ms_per_step": e2e,
                    "ms_each_step_this_rank": [round(v, 3) for v in e2e_ms],
                    "h2d_bytes_per_step": h2d_total, "d2h_bytes_per_step": d2h_total,
                    "rows": "pos u32 + score f64 (CRP_SCAN_LOGISTIC) per candidate; the packed 30-mer stays on the device",
                    "link_ceiling": link},
            "gpu_launches": t["launches"],
            "capacity_reruns": t["capacity_reruns"],
            "wall_ms_per_step_incl_flush_barriers": t["wall_ms"],
            "clocks": clocks,
            "roofline": roofline(sh.my_bases, t["candidates"], t["kernel_ms"], workload, world),
            "ingest": ingest_timing,
        }
        if world > 1:
            line["collective_ms"] = t["ms"] - t["kernel_ms"]
            line["per_rank"] = per_rank         # what sets the step: equal tiles, unequal candidates (soft-masked repeats carry none)
    # ---- N > 1: the same steps with the other exchange (the default is the fused one when peers map)
    if world > 1:
        fused, why = engine.comm_exchange_info()
        other = "nccl" if fused else None
        alt = None
        if other:
            engine.comm_set_exchange(other)
            ta = time_scans(engine, sh, min(args.steps, 10), 3)
            alt_ms = float(engine.comm_max([ta["ms"]])[0])
            alt = {"ms_per_step": alt_ms, "value": n_bases_total / (alt_ms * 1e-3) / 1e9, "kernel_ms": ta["kernel_ms"],
                   "collective_ms": ta["ms"] - ta["kernel_ms"]}
            engine.comm_set_exchange("fused")
        if rank == 0:
            line["exchange"] = {"timed": "fused into k_scan_score (peer stores over NVLink, CUDA IPC)" if fused
                                else "ncclAllGather behind the kernel", "note": why, "nccl_all_gather": alt}
            line["config"]["collective"] = ("per-segment counts all-gathered INSIDE k_scan_score: peer stores over NVLink after the "
                                            "count phase, flags, wait at the kernel's end; inside the timed events "
                                            "(ncclAllGather variant timed beside it: exchange.nccl_all_gather)") if fused else \
                line["config"]["collective"]
    sh.free()

    # ---- N > 1: the single-GPU time of the SAME genome, measured by rank 0 in this run
    if world > 1 and not args.no_extra:
        single = None
        if rank == 0:
            one = Shard(engine, shard, workload, 0, 1, pinned=False)
            t1 = time_scans_local(engine, one, min(args.steps, 5), 3)
            single = {"workload": CONFIG_NAME[workload], "single_gpu_ms": t1["ms"],
                      "single_gpu_value": n_bases_total / (t1["ms"] * 1e-3) / 1e9, "n_gpu_ms": ms,
                      "speedup": t1["ms"] / ms, "note": "whole genome on rank 0's GPU alone, same process, same run"}
            one.free()
        engine.comm_barrier()
        if rank == 0:
            line["strong_scaling"] = single
        if world >= 8 and workload != "sugarcane":
            big = Shard(engine, shard, "sugarcane", rank, world, pinned=False)
            tb = time_scans(engine, big, min(args.steps, 5), 3)
            big_ms = float(engine.comm_max([tb["ms"]])[0])
            kernel_all = rdv.all_gather(tb["kernel_ms"])
            cand = int(engine.comm_sum([tb["candidates"]])[0])
            if rank == 0:
                line["largest"] = {"workload": CONFIG_NAME["sugarcane"], "bases": big.n_bases_total, "candidates": cand,
                                   "segments_per_rank": big.slots, "ms_per_step": big_ms,
                                   "value": big.n_bases_total / (big_ms * 1e-3) / 1e9, "unit": "Gbp/s",
                                   "kernel_ms_per_rank": kernel_all,
                                   "sum_of_kernels_over_n_ms": float(np.sum(kernel_all)) / world,
                                   "roofline": roofline(big.my_bases, tb["candidates"], tb["kernel_ms"], "sugarcane", world)}
            big.free()

    # ---- N = 1: the other single-GPU configs ride along
    if world == 1 and not args.no_extra and args.workload is None:
        line["workloads"] = {}
        for other in ("sorghum", "maize"):
            o = Shard(engine, shard, other, 0, 1, pinned=False)
            to = time_scans_local(engine, o, min(args.steps, 5), 3)
            line["workloads"][other] = {"workload": CONFIG_NAME[other], "bases": o.n_bases_total, "candidates": to["candidates"],
                                        "ms_per_step": to["ms"], "value": o.n_bases_total / (to["ms"] * 1e-3) / 1e9,
                                        "roofline": roofline(o.my_bases, to["candidates"], to["kernel_ms"], other, 1)}
            o.free()

    if rank == 0:
        if not args.no_cpu_baseline and world == 1:
            os.sched_setaffinity(0, cpus_before)          # the CPU baseline may use every core of the host
            line["cpu_baseline"] = reference_sample(workload, 20.0)[0]
        line["perf_report"] = engine.perf_report()
        print(json.dumps(line))
    engine.comm_barrier()
    engine.comm_shutdown()
    rdv.close()


def time_scans_local(engine, sh, steps, warmup):
    """time_scans for a shard that only this rank scans (no collective calls inside)."""
    total_ms, kernel_ms, n_cand = [], [], 0
    for i in range(warmup + steps):
        engine.flush_l2()
        engine.device_synchronize()
        res = sh.scan() if sh.world == 1 else sh.genome.scan(20)
        if i >= warmup:
            d = res.timing_detail()
            total_ms.append(d["total_ms"])
            kernel_ms.append(d["kernel_ms"])
        n_cand = res.n_plus + res.n_minus
        res.free()
    return {"ms": float(np.mean(total_ms)), "kernel_ms": float(np.mean(kernel_ms)), "candidates": int(n_cand)}


if __name__ == "__main__":
    main()
