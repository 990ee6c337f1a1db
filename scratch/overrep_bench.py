"""Cost of overrepresented sequences (fq_overrep_*): added device time per 2 M-pair batch resident in HBM on three inputs --
C2 (nearly every prefix distinct: every insert claims a slot), 20 000 distinct pairs x 100, and one primer dimer in 30 % of
the reads (the case the warp aggregation is for) -- and the end of a pass over two contexts on one device.  The device time
is the library's CUDA-event segment "all" of each batch; runs with the feature off and on alternate, one batch each, after
warm-up.

  python scratch/overrep_bench.py [--pairs 2000000] [--reps 10] [--out DIR]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from faqcs_b200 import dist_stats, synth  # noqa: E402
from faqcs_b200.api import Engine, Options  # noqa: E402

DIMER = "ACACTCTTTCCCTACACGACGCTCTTCCGATCTAGATCGGAAGAGCACACGTCTGAACTCCAGTCAC"


def device_batch(r1, r2):
    return torch.from_numpy(np.asarray(r1)).cuda(0), torch.from_numpy(np.asarray(r2)).cuda(0)


def run_ms(eng, d1, d2, on):
    eng.process_device(d1.data_ptr(), d1.numel(), d2.data_ptr(), d2.numel(), 0, True)
    ms = eng.last_timing()["all"]
    if on:
        eng.overrep_end_pass()             # a cleared table for the next batch: every key is new again
    return ms


def compare(name, d1, d2, reps):
    opt = Options(input_quality_offset=33)
    with Engine(opt) as off, Engine(opt) as on:
        on.overrep_enable()
        for _ in range(3):
            run_ms(off, d1, d2, False)
            run_ms(on, d1, d2, True)
        t_off, t_on = [], []
        for _ in range(reps):
            t_off.append(run_ms(off, d1, d2, False))
            t_on.append(run_ms(on, d1, d2, True))
        run_ms(on, d1, d2, False)
        on.overrep_end_pass()
        res = on.overrep_results()
    med_off, med_on = statistics.median(t_off), statistics.median(t_on)
    return {"input": name, "ms_off_median": med_off, "ms_on_median": med_on, "added_ms_median": med_on - med_off,
            "ms_off_range": [min(t_off), max(t_off)], "ms_on_range": [min(t_on), max(t_on)],
            "reads": res["reads"], "listed": len(res["seqs"]), "top_count": res["seqs"][0][2] if res["seqs"] else 0}


def merge_time(d1, d2, reps):
    """Two contexts on device 0, one batch each (the same pairs, so every key has entries in both to merge)."""
    opt = Options(input_quality_offset=33)
    engines = [Engine(opt) for _ in range(2)]
    try:
        for e in engines:
            e.overrep_enable()
        times = []
        for k in range(reps + 1):
            for e in engines:
                e.process_device(d1.data_ptr(), d1.numel(), d2.data_ptr(), d2.numel(), 0, True)
            torch.cuda.synchronize()
            t = time.perf_counter()
            dist_stats.overrep_end_pass_local(engines)
            if k:
                times.append((time.perf_counter() - t) * 1e3)
        res = engines[0].overrep_results()
        return {"merge_2ctx_ms_median": statistics.median(times), "merge_2ctx_ms_range": [min(times), max(times)],
                "reads": res["reads"], "listed": len(res["seqs"])}
    finally:
        for e in engines:
            e.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=2_000_000)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()[0]
    block = 250_000
    parts = [synth.c2(block, start=s) for s in range(0, a.pairs, block)]
    r1 = np.concatenate([w.r1 for w in parts])
    r2 = np.concatenate([w.r2 for w in parts])
    d1, d2 = device_batch(r1, r2)
    out = {"gpu": gpu, "pairs": a.pairs, "c2": compare("c2", d1, d2, a.reps)}
    o1 = np.concatenate([[0], np.flatnonzero(r1 == 10)[3::4] + 1])
    o2 = np.concatenate([[0], np.flatnonzero(r2 == 10)[3::4] + 1])
    k = a.pairs // 100
    h1, h2 = device_batch(np.tile(r1[:o1[k]], 100), np.tile(r2[:o2[k]], 100))
    out["high_dup"] = compare("c2 first %d pairs x 100" % k, h1, h2, a.reps)
    del h1, h2
    n_dimer = int(a.pairs * 0.3)
    dparts = [synth.overrepresented(block, plants=[(DIMER, int(block * 0.3), 0, True)], start=s) for s in range(0, a.pairs, block)]
    g1, g2 = device_batch(np.concatenate([w.r1 for w in dparts]), np.concatenate([w.r2 for w in dparts]))
    out["dimer_30pct"] = compare("one %d-base dimer in %d of %d reads of each mate" % (len(DIMER), n_dimer, a.pairs), g1, g2, a.reps)
    del g1, g2
    out["merge"] = merge_time(d1, d2, a.reps)
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        open(os.path.join(a.out, "overrep_bench.json"), "w").write(line + "\n")


if __name__ == "__main__":
    main()
