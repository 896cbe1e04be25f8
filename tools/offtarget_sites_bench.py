#!/usr/bin/env python3
"""Cost of the off-target listing (csrc/offtarget.cuh: k_ot_sites<true>, k_ot_join<OtList>) on the benchmark genomes:

    python tools/offtarget_sites_bench.py [--tsv-max-mbp N] [workload ...]     (default: arabidopsis maize)

Per workload: commit every chromosome (as many genome handles as the 32-bit limits ask for) and scan it; build one
index without loci and one with loci over all handles (ms_sites of each, and the device bytes per site of each); then,
at k = 0, 1, 2, 3, count every candidate of both strands (ms_count) and list every candidate whose counts sum to at
most 1,000 (ms_list: device time of every list call, the same ten counting sorts and the join; listing calls are
batched as engine.OffTargetIndex.list_candidates batches them).  One JSON line per (workload, k) with the pairs and
bytes listed, list/count ratio, and the device with its power limit and maximum SM clock (nvidia-smi, read only, in
the same call).  For genomes of at most --tsv-max-mbp (default 200: configs[1]) the host time of
pipeline.write_offtarget_sites at k = 3 is measured separately (counts given, so it is listing + host work), written
to a temporary directory that is removed afterwards.
"""
import json
import os
import shutil
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tools")]
import numpy as np                                     # noqa: E402
import workloads as W                                  # noqa: E402
from cropsr_b200 import engine, pipeline               # noqa: E402

MAX_SITES = 1000


def device_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        name, power, clock = [x.strip() for x in r.stdout.splitlines()[0].split(",")]
        return {"device": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:                             # the numbers are still device times; say what is missing
        return {"device": None, "nvidia_smi": str(e)}


def list_timed(index, result, strand, k, counts):
    """list every candidate with 0 < total <= MAX_SITES; -> (pairs, device ms summed over the list calls)"""
    ok = counts[:, 0] != index.NO_COUNT
    tot = np.where(ok, counts.astype(np.int64).sum(axis=1), 0)
    rows = np.nonzero((tot > 0) & (tot <= MAX_SITES))[0]
    pairs, ms, lo = 0, 0.0, 0
    csum = np.cumsum(tot[rows])
    while lo < len(rows):                              # one library call per batch, as list_candidates batches
        base = csum[lo - 1] if lo else 0
        hi = max(int(np.searchsorted(csum, base + engine.LIST_BATCH_SITES, side="right")), lo + 1)
        _, first, _ = index.list_candidates(result, strand, k, rows=rows[lo:hi], counts=counts)
        ms += index.timing()["ms_count"]
        pairs += int(first[-1])
        lo = hi
    return pairs, ms


def run(workload, info, tsv_max_mbp):
    t0 = time.time()
    lengths = W.token_lengths(workload)
    parts = []
    for first, cnt in pipeline._groups(lengths):
        g = engine.Genome()
        for k in range(first, first + cnt):
            g.add_token(W.token(workload, k))
        g.commit()
        parts.append((g, g.scan(20), first, cnt))
    plain = engine.OffTargetIndex([g for g, _, _, _ in parts])
    ms_sites_plain = plain.timing()["ms_sites"]
    plain.free()
    index = engine.OffTargetIndex([g for g, _, _, _ in parts], loci=True)
    ms_sites_loci = index.timing()["ms_sites"]
    n_sites = index.num_sites()
    queries = sum(r.n_plus + r.n_minus for _, r, _, _ in parts)
    setup_s = time.time() - t0
    for k in range(4):
        ms_count = ms_list = 0.0
        pairs = 0
        wall = time.time()
        for _, r, _, _ in parts:
            for strand in "+-":
                counts = index.count_candidates(r, strand, k)
                ms_count += index.timing()["ms_count"]
                p, ms = list_timed(index, r, strand, k, counts)
                pairs += p
                ms_list += ms
        line = {"workload": workload, "config": W.CONFIG_NAME[workload], "k": k, "max_sites": MAX_SITES,
                "sites": n_sites, "queries": int(queries), "ms_sites": round(ms_sites_plain, 3),
                "ms_sites_loci": round(ms_sites_loci, 3), "index_bytes_per_site": 8, "index_bytes_per_site_loci": 16,
                "ms_count": round(ms_count, 3), "ms_list": round(ms_list, 3),
                "list_over_count": round(ms_list / ms_count, 3) if ms_count else None,
                "pairs": pairs, "pair_bytes": 4 * pairs, "wall_s": round(time.time() - wall, 3),
                "setup_s": round(setup_s, 1), **info}
        print(json.dumps(line), flush=True)
    if sum(lengths) <= tsv_max_mbp * 1_000_000:
        token_bytes = [W.token(workload, k).tobytes() for k in range(len(lengths))]
        tokens = {">" + W.record_name(workload, k): None for k in range(len(lengths))}
        scan = pipeline.ScanOutput(token_bytes, parts, 20)
        counts = pipeline.offtarget_counts(index, scan, 3)
        tmp = tempfile.mkdtemp(prefix="offtarget_sites_bench_")
        try:
            path = os.path.join(tmp, "sites.tsv")
            wall = time.time()
            pairs, capped = pipeline.write_offtarget_sites(path, tokens, scan, 3, MAX_SITES, index=index, counts=counts)
            print(json.dumps({"workload": workload, "config": W.CONFIG_NAME[workload], "k": 3, "max_sites": MAX_SITES,
                              "tsv_pairs": pairs, "tsv_capped": capped, "tsv_bytes": os.path.getsize(path),
                              "tsv_wall_s": round(time.time() - wall, 3), **info}), flush=True)
        finally:
            shutil.rmtree(tmp, ignore_errors=True)
    index.free()
    for g, r, _, _ in parts:
        r.free()
        g.free()


def main(argv):
    tsv_max_mbp = 200
    if argv[:1] == ["--tsv-max-mbp"]:
        tsv_max_mbp, argv = float(argv[1]), argv[2:]
    engine.init(0)
    info = device_info()
    for workload in argv or ["arabidopsis", "maize"]:
        run(workload, info, tsv_max_mbp)


if __name__ == "__main__":
    main(sys.argv[1:])
