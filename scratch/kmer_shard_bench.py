"""k-mer rarefaction over a table sharded across contexts: counting time per batch, reads/s over the pass, and the time of
fq_kmer_end_pass_all (host clock around the call, which synchronises), with the distinct k-mers each context held before
the merge.  Configurations: 1 and 2 contexts on one GPU, then 1/2/4/8 GPUs in one process (those that are visible).

Workload: random 150-base pairs (synth.c2: nearly every 31-mer distinct, the merge's worst case), B distinct batches of
2^19 pairs (~1 M reads, ~126 M k-mers each), dealt round robin.  Writes one JSON (default profiles/r3_kmer_shard_bench.json).

    python scratch/kmer_shard_bench.py [--batches 6] [--out PATH]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from faqcs_b200 import dist_stats, synth  # noqa: E402
from faqcs_b200.api import Engine, Options  # noqa: E402

PAIRS = 1 << 19


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit", "--format=csv,noheader"], stdout=subprocess.PIPE,
                       stderr=subprocess.PIPE, text=True)
    return [ln.strip() for ln in q.stdout.splitlines() if ln.strip()]


def sync_all(devices):
    for d in set(devices):
        torch.cuda.synchronize(d)


def own_distinct(devices, data, opt, k=31, split=10 ** 12, subset=10):
    """Distinct k-mers in each context's own table before the merge: context i's batches (every n-th) counted alone, at
    consecutive positions, in a one-context pass of their own (untimed)."""
    out = []
    for i, d in enumerate(devices):
        mine = data[i::len(devices)]
        with Engine(opt, device=d) as e:
            e.kmer_enable(k, split, 2 * subset)
            e.autodetect(mine[0][0], mine[0][1])
            for j, (r1, r2) in enumerate(mine):
                e.process(r1, r2, j * PAIRS, j == len(mine) - 1)
            e.kmer_end_pass()
            out.append(int(e.kmer_results()[0][-1][1]))
    return out


def warm_up(devices, opt):
    """Modules and first allocations on every device, in contexts of their own."""
    w = synth.c2(32768, seed=1234)
    engines = [Engine(opt, device=d) for d in devices]
    try:
        for j, e in enumerate(engines):
            e.kmer_enable(31, 10 ** 12, 20)
            e.autodetect(w.r1, w.r2)
        for e in engines:
            e.process(w.r1, w.r2, 0, True)
            e.kmer_end_pass()
    finally:
        for e in engines:
            e.close()


def run(devices, data, opt, kmer=True, k=31, split=10 ** 12, subset=10):
    """One pass over `data` with one context per entry of `devices`; split_size so large that every batch is counted."""
    engines = [Engine(opt, device=d) for d in devices]
    try:
        for e in engines:
            if kmer:
                e.kmer_enable(k, split, 2 * subset)
            e.autodetect(data[0][0], data[0][1])
        per_batch = []
        sync_all(devices)
        t_pass = time.perf_counter()
        for j, (r1, r2) in enumerate(data):
            e = engines[j % len(engines)]
            t = time.perf_counter()
            e.process(r1, r2, j * PAIRS, j == len(data) - 1)          # returns after its stream has synchronised
            seg = e.last_timing()
            per_batch.append({"batch": j, "device": devices[j % len(devices)], "host_s": time.perf_counter() - t,
                              "device_ms_all": seg["all"], "device_ms_kmer_route_scan": seg["emit"]})
        sync_all(devices)
        t_count = time.perf_counter() - t_pass
        n_reads = 2 * PAIRS * len(data)
        r = {"devices": devices, "contexts": len(devices), "kmer": kmer, "batches": len(data), "reads": n_reads,
             "pass_s": t_count, "reads_per_s": n_reads / t_count,
             "median_device_ms_kmer_route_scan": float(np.median([b["device_ms_kmer_route_scan"] for b in per_batch])),
             "per_batch": per_batch}
        if kmer:
            t = time.perf_counter()
            dist_stats.kmer_end_pass_local(engines)
            r["end_pass_all_s"] = time.perf_counter() - t
            rare, _ = engines[0].kmer_results()
            r["distinct_total"], r["kmer_instances"] = int(rare[-1][1]), int(rare[-1][2])
        return r
    finally:
        for e in engines:
            e.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, default=6)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_kmer_shard_bench.json"))
    a = ap.parse_args()
    n_gpu = torch.cuda.device_count()
    if n_gpu == 0:
        raise SystemExit("no CUDA device: this benchmark measures the GPU path only")
    data = []
    for j in range(a.batches):
        w = synth.c2(PAIRS, seed=100 + j, start=j * PAIRS)
        data.append((w.r1, w.r2))
    opt = Options(qc_only=True)
    configs = [[0], [0, 0]] + [list(range(g)) for g in (2, 4, 8) if g <= n_gpu]
    warm_up(list(range(n_gpu)), opt)
    results = [run([0], data, opt, kmer=False)]             # the same batches without k-mer counting
    for devs in configs:
        r = run(devs, data, opt)
        r["distinct_per_context_before_merge"] = own_distinct(devs, data, opt)
        print(json.dumps({k: v for k, v in r.items() if k != "per_batch"}), flush=True)
        results.append(r)
    out = {"what": "k-mer rarefaction, table sharded over contexts: counting and fq_kmer_end_pass_all",
           "gpus": gpu_info(), "torch": torch.__version__, "pairs_per_batch": PAIRS, "read_length": 150, "k": 31,
           "workload": "synth.c2 random pairs, distinct seeds per batch", "results": results}
    os.makedirs(os.path.dirname(a.out), exist_ok=True)
    with open(a.out, "w") as fh:
        json.dump(out, fh, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
