"""Cost of per flowcell tile quality (fq_tile_qual_*): added device time per 2 M-pair 2x150 batch resident in HBM on three
inputs -- synth.tiled in (lane, tile) order as a sequencer writes it, the same reads shuffled (every warp run crosses many
tiles), and C2 (every read untiled: the header parse alone) -- and the end of a pass over two contexts on one device.  The
device time is the library's CUDA-event segment "all" of each batch; runs with the feature off and on alternate, one batch
each, after warm-up.  The feature reads every header and quality byte once more: the bytes are counted here too.

  python scratch/tile_bench.py [--pairs 2000000] [--reps 10] [--out DIR]
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


def device_batch(r1, r2):
    return torch.from_numpy(np.asarray(r1)).cuda(0), torch.from_numpy(np.asarray(r2)).cuda(0)


def run_ms(eng, d1, d2, on):
    eng.process_device(d1.data_ptr(), d1.numel(), d2.data_ptr(), d2.numel(), 0, True)
    ms = eng.last_timing()["all"]
    if on:
        eng.tile_qual_end_pass()
    return ms


def header_and_quality_bytes(buf):
    nl = np.flatnonzero(buf == 10)
    start = np.concatenate([[0], nl[:-1] + 1])
    return int((nl[0::4] - start[0::4]).sum() + (nl[3::4] - start[3::4]).sum())


def compare(name, r1, r2, reps):
    d1, d2 = device_batch(r1, r2)
    opt = Options(input_quality_offset=33)
    with Engine(opt) as off, Engine(opt) as on:
        on.tile_qual_enable()
        for _ in range(3):
            run_ms(off, d1, d2, False)
            run_ms(on, d1, d2, True)
        t_off, t_on = [], []
        for _ in range(reps):
            t_off.append(run_ms(off, d1, d2, False))
            t_on.append(run_ms(on, d1, d2, True))
        run_ms(on, d1, d2, False)
        on.tile_qual_end_pass()
        res = on.tile_qual_results()
    med_off, med_on = statistics.median(t_off), statistics.median(t_on)
    return {"input": name, "ms_off_median": med_off, "ms_on_median": med_on, "added_ms_median": med_on - med_off,
            "ms_off_range": [min(t_off), max(t_off)], "ms_on_range": [min(t_on), max(t_on)],
            "header_and_quality_bytes": header_and_quality_bytes(r1) + header_and_quality_bytes(r2),
            "tiles": res["n_tiles"], "untiled": [int(x) for x in res["untiled"]]}


def merge_time(r1, r2, reps):
    """Two contexts on device 0, one batch each (the same pairs, so every tile has counts in both to sum)."""
    d1, d2 = device_batch(r1, r2)
    opt = Options(input_quality_offset=33)
    engines = [Engine(opt) for _ in range(2)]
    try:
        for e in engines:
            e.tile_qual_enable()
        times = []
        for k in range(reps + 1):
            for e in engines:
                e.process_device(d1.data_ptr(), d1.numel(), d2.data_ptr(), d2.numel(), 0, True)
            torch.cuda.synchronize()
            t = time.perf_counter()
            dist_stats.tile_qual_end_pass_local(engines)
            if k:
                times.append((time.perf_counter() - t) * 1e3)
        res = engines[0].tile_qual_results()
        return {"merge_2ctx_ms_median": statistics.median(times), "merge_2ctx_ms_range": [min(times), max(times)],
                "tiles": res["n_tiles"], "reads": [int(x) for x in res["reads"]]}
    finally:
        for e in engines:
            e.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=2_000_000)
    ap.add_argument("--lanes", type=int, default=4)
    ap.add_argument("--tiles-per-lane", type=int, default=128)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         stdout=subprocess.PIPE, text=True).stdout.strip().splitlines()[0]
    out = {"gpu": gpu, "pairs": a.pairs, "tiles": a.lanes * a.tiles_per_lane}
    for order in ("sorted", "shuffled"):
        w = synth.tiled(a.pairs, lanes=a.lanes, tiles_per_lane=a.tiles_per_lane, order=order)
        out["tiled_" + order] = compare("synth.tiled %s, %d tiles" % (order, a.lanes * a.tiles_per_lane), w.r1, w.r2, a.reps)
        if order == "sorted":
            out["merge"] = merge_time(w.r1, w.r2, a.reps)
        del w
        torch.cuda.empty_cache()
    block = 250_000
    parts = [synth.c2(block, start=s) for s in range(0, a.pairs, block)]
    out["c2"] = compare("c2 (every read untiled)", np.concatenate([p.r1 for p in parts]), np.concatenate([p.r2 for p in parts]), a.reps)
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        open(os.path.join(a.out, "tile_bench.json"), "w").write(line + "\n")


if __name__ == "__main__":
    main()
