"""Cost of the insert size and overlap error profile (fq_overlap_*): added device time per 2 M-pair 2x150 batch, for C2
(unrelated mates: almost every candidate is rejected within its first 32 positions) and for synth.fragments (most pairs
overlap, so one candidate per pair is counted to its end), plus the time of k_overlap alone from torch.profiler.  Batches
are resident in HBM (fq_process_device, outputs left on the device); the device time is the library's CUDA-event segment
"all" of each batch.  Runs with the profile off and on alternate, one batch each, after warm-up.  On C2 the kernel is also
timed at min_overlap 90 and 150 (121 candidates and 1 candidate per pair instead of 241), which separates the cost that every
pair pays (record and base loads, packing, reductions, counters) from the cost of testing candidates.

  python scratch/insert_bench.py [--pairs 2000000] [--reps 10] [--out DIR]
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

from faqcs_b200 import synth  # noqa: E402
from faqcs_b200.api import Engine, Options  # noqa: E402


def device_batch(r1, r2):
    return torch.from_numpy(np.asarray(r1)).cuda(0), torch.from_numpy(np.asarray(r2)).cuda(0)


def run_ms(eng, d1, d2, on):
    eng.process_device(d1.data_ptr(), d1.numel(), d2.data_ptr(), d2.numel(), 0, True)
    ms = eng.last_timing()["all"]
    if on:
        eng.overlap_end_pass()
    return ms


def compare(name, d1, d2, reps):
    opt = Options(input_quality_offset=33)
    with Engine(opt) as off, Engine(opt) as on:
        on.overlap_enable()
        for _ in range(3):
            run_ms(off, d1, d2, False)
            run_ms(on, d1, d2, True)
        t_off, t_on = [], []
        for _ in range(reps):
            t_off.append(run_ms(off, d1, d2, False))
            t_on.append(run_ms(on, d1, d2, True))
        res = on.overlap_results()
        kernel_ms = profile_kernel(on, d1, d2)
    med_off, med_on = statistics.median(t_off), statistics.median(t_on)
    return {"input": name, "ms_off_median": med_off, "ms_on_median": med_on, "added_ms_median": med_on - med_off,
            "ms_off_range": [min(t_off), max(t_off)], "ms_on_range": [min(t_on), max(t_on)], "k_overlap_ms": kernel_ms,
            "pairs": res["pairs"], "overlapped": res["overlapped"], "too_short": res["too_short"],
            "mismatch_bases": res["mismatch_bases"]}


def profile_kernel(eng, d1, d2, reps=5):
    """Mean device time of the k_overlap launches of `reps` batches, from torch.profiler's CUDA activity."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            run_ms(eng, d1, d2, True)
        torch.cuda.synchronize()
    times = [e.device_time_total for e in prof.key_averages() if "k_overlap" in e.key]
    return sum(times) / reps / 1e3 if times else None


def kernel_ms_at(d1, d2, min_overlap):
    with Engine(Options(input_quality_offset=33)) as e:
        e.overlap_enable(min_overlap, 5, 20)
        for _ in range(2):
            run_ms(e, d1, d2, True)
        return profile_kernel(e, d1, d2)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=2_000_000)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()[0]
    block = 250_000
    out = {"gpu": gpu, "pairs": a.pairs}
    for name, gen in (("c2", synth.c2), ("fragments", synth.fragments)):
        parts = [gen(block, start=s) for s in range(0, a.pairs, block)]
        d1, d2 = device_batch(np.concatenate([w.r1 for w in parts]), np.concatenate([w.r2 for w in parts]))
        out[name] = compare(name, d1, d2, a.reps)
        if name == "c2":
            out["c2_k_overlap_ms_by_min_overlap"] = {str(O): kernel_ms_at(d1, d2, O) for O in (30, 90, 150)}
        del d1, d2
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        open(os.path.join(a.out, "insert_bench.json"), "w").write(line + "\n")


if __name__ == "__main__":
    main()
