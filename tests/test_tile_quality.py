"""Per flowcell tile quality (fq_tile_qual_*, --tile_quality): every read's (lane, tile) from its name, and per (tile, mate)
the reads, whole-read bases and score sums, and the bases and score sum at each cycle.  The restatement below follows the
definition in include/faqcs_b200.h; the library must give exactly its integers, and the command line exactly its text."""
import gzip
import os
import shutil
import subprocess
import tempfile

import numpy as np
import pytest

from faqcs_b200 import dist_stats, synth
from faqcs_b200.api import Engine, FaqcsError, Options
from test_dup_stats import _as_u8, cut, fuzz_workload, run_batches, seq_lines, shuffled

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CLI = os.path.join(ROOT, "faqcs_b200", "host", "faqcs_b200")
FQ_ERR_ARG, FQ_ERR_FORMAT, FQ_ERR_STATE, FQ_ERR_QUALITY = 1, 4, 8, 5
MAX_KEYS, MAX_CYCLES = 16384, 1024


# ---- the restatement ---------------------------------------------------------------------------------------------------
def _value(f):
    return int(f) if 1 <= len(f) <= 9 and all(48 <= c <= 57 for c in f) else None


def name_key(header_line: bytes):
    """(lane, tile) of one header line (with its '@'), or None when the read is untiled."""
    name = header_line[1:]
    for i, c in enumerate(name):
        if c in b" \t\r\n":
            name = name[:i]
            break
    f = name.split(b":")
    if len(f) >= 7:
        lane, tile = _value(f[3]), _value(f[4])
    elif len(f) in (5, 6):
        lane, tile = _value(f[1]), _value(f[2])
    else:
        return None
    return None if lane is None or tile is None else (lane, tile)


def _mate_reads(buf, off):
    """Keys, lengths as framed, and every base's (read, cycle, score) of one mate."""
    b = np.asarray(buf, np.uint8)
    nl = np.flatnonzero(b == 10)
    line_start = np.concatenate([[0], nl[:-1] + 1])
    keys = [name_key(bytes(b[s:e])) for s, e in zip(line_start[0::4].tolist(), nl[0::4].tolist())]
    _, lens = seq_lines(b)
    qs = line_start[3::4]
    read = np.repeat(np.arange(lens.size), lens)
    cyc = np.arange(read.size) - np.repeat(np.cumsum(lens) - lens, lens)
    score = np.maximum(0, b[qs[read] + cyc].astype(np.int64) - off)
    return keys, lens, read, cyc, score


def restate(r1, r2=None, off=33):
    mates = [_mate_reads(x, off) for x in (r1, r2) if x is not None]
    M = len(mates)
    reads = np.zeros(2, np.uint64)
    untiled = np.zeros(2, np.uint64)
    longest = 0
    keys = set()
    for m, (k, lens, _, _, _) in enumerate(mates):
        reads[m] = len(k)
        untiled[m] = sum(x is None for x in k)
        keys.update(x for x in k if x is not None)
        longest = max(longest, int(lens.max()) if lens.size else 0)
    C = min(longest, MAX_CYCLES)
    out = {"n_mates": M, "overflow": int(len(keys) > MAX_KEYS), "cycles": C, "reads": reads, "untiled": untiled}
    keys = [] if out["overflow"] else sorted(keys)
    T = len(keys)
    out["n_tiles"] = T
    out["lane"] = np.array([k[0] for k in keys], np.uint32)
    out["tile"] = np.array([k[1] for k in keys], np.uint32)
    for name in ("tile_reads", "tile_bases", "tile_qsum"):
        out[name] = np.zeros((T, M), np.uint64)
    for name in ("cycle_bases", "cycle_qsum"):
        out[name] = np.zeros((T, M, C), np.uint64)
    index = {k: i for i, k in enumerate(keys)}
    for m, (k, lens, read, cyc, score) in enumerate(mates):
        if not T:
            continue
        t = np.array([index.get(x, -1) if x is not None else -1 for x in k], np.int64)
        ok = t >= 0
        out["tile_reads"][:, m] = np.bincount(t[ok], minlength=T)
        out["tile_bases"][:, m] = np.bincount(t[ok], weights=lens[ok], minlength=T).astype(np.uint64)
        tb = t[read]
        sel = tb >= 0
        out["tile_qsum"][:, m] = np.bincount(tb[sel], weights=score[sel], minlength=T).astype(np.uint64)
        sel &= cyc < C
        flat = tb[sel] * C + cyc[sel]
        out["cycle_bases"][:, m, :] = np.bincount(flat, minlength=T * C).reshape(T, C)
        out["cycle_qsum"][:, m, :] = np.bincount(flat, weights=score[sel], minlength=T * C).astype(np.uint64).reshape(T, C)
    return out


ARRAYS = ("reads", "untiled", "lane", "tile", "tile_reads", "tile_bases", "tile_qsum", "cycle_bases", "cycle_qsum")


def assert_same(got, want):
    for k in ("n_mates", "overflow", "n_tiles", "cycles"):
        assert got[k] == want[k], (k, got[k], want[k])
    for k in ARRAYS:
        assert got[k].shape == want[k].shape and np.array_equal(got[k].astype(np.uint64), want[k].astype(np.uint64)), k


def _fmt(x):
    return "%.2f" % x


def report(res, paired):
    """The block the command line writes for one pass."""
    M, C, T = (2 if paired else 1), res["cycles"], res["n_tiles"]
    out = [f"pass\t{'paired' if paired else 'unpaired'}\ttiles\t{T}\tcycles\t{C}\toverflow\t{res['overflow']}", "#mate\treads\ttiled\tuntiled"]
    for m in range(M):
        r, u = int(res["reads"][m]), int(res["untiled"][m])
        out.append(f"{m + 1}\t{r}\t{r - u}\t{u}")
    if res["overflow"]:
        return "\n".join(out) + "\n"
    nm = res["n_mates"]

    def col(name, m):
        return res[name][:, m] if m < nm else np.zeros((T,) + res[name].shape[2:], np.uint64)
    out.append("#mate\tmean_by_cycle")
    allm = []
    for m in range(M):
        b, q = col("cycle_bases", m).sum(0) if T else np.zeros(C, np.uint64), col("cycle_qsum", m).sum(0) if T else np.zeros(C, np.uint64)
        means = [float(int(q[c])) / float(int(b[c])) if b[c] else None for c in range(C)]
        allm.append(means)
        out.append("\t".join([str(m + 1)] + [_fmt(x) if x is not None else "NA" for x in means]))
    out.append("#lane\ttile\tmate\treads\tbases\tmean\tworst_cycle\tworst_delta\tdelta_by_cycle")
    for t in range(T):
        for m in range(M):
            reads, bases, qsum = (int(col(k, m)[t]) for k in ("tile_reads", "tile_bases", "tile_qsum"))
            cb, cq = col("cycle_bases", m)[t], col("cycle_qsum", m)[t]
            deltas, worst = [], None
            for c in range(C):
                if not cb[c]:
                    deltas.append("NA")
                    continue
                d = float(int(cq[c])) / float(int(cb[c])) - allm[m][c]
                if worst is None or d < worst[1]:
                    worst = (c + 1, d)
                deltas.append(_fmt(d))
            row = [str(int(res["lane"][t])), str(int(res["tile"][t])), str(m + 1), str(reads), str(bases),
                   _fmt(float(qsum) / float(bases)) if bases else "NA"]
            row += [str(worst[0]), _fmt(worst[1])] if worst else ["NA", "NA"]
            out.append("\t".join(row + deltas))
    return "\n".join(out) + "\n"


# ---- CPU: the restatement on hand-written headers, the command line's usage ----------------------------------------------
HEADER_CASES = [
    (b"@A00123:456:HXXXXXXXX:1:1101:12345:67890 1:N:0:ACGT", (1, 1101)),                 # 7 fields
    (b"@A00123:456:HXXXXXXXX:2:2207:12345:67890:ACGTACGT 2:N:0:ACGT", (2, 2207)),        # 8 fields: a UMI
    (b"@HWUSI-EAS100R:6:73:941:1973#0/1", (6, 73)),                                      # 5 fields, older names
    (b"@HWUSI-EAS100R:6:73:941:1973:5#0/1", (6, 73)),                                    # 6 fields
    (b"@SYN:C2:1:0000:00013:00000 1:N:0:1", None),                                       # synthetic: the lane field is C2
    (b"@A:1:FC:3:1101:5:6 1:N:0:ACGT", (3, 1101)),
    (b"@A 1:FC:3:1101:5:6", None),                                                       # a space before the colons
    (b"@A\t1:FC:3:1101:5:6", None),                                                      # a tab before the colons
    (b"@A:1:FC:3:1101:5:6\r", (3, 1101)),                                                # CRLF
    (b"@A:1:FC:3:11\r01:5:6", None),                                                     # a lone '\r' ends the name
    (b"@", None), (b"@ 1:2:3:4:5:6:7", None),                                            # empty names
    (b"@A:1:FC:3:1234567890:5:6", None), (b"@A:1:FC:3:123456789:5:6", (3, 123456789)),  # 10 and 9 digits
    (b"@A:1:FC:+3:1101:5:6", None), (b"@A:1:FC:3:-1101:5:6", None),                      # signs
    (b"@A:1:FC:03:01101:5:6", (3, 1101)), (b"@A:1:FC:0:0:5:6", (0, 0)),                 # leading zeros, zero
    (b"@A:1:FC::1101:5:6", None), (b"@a:b:c:d", None), (b"@a:1:2", None),               # empty field, 4 and 3 fields
]


@pytest.mark.parametrize("header, key", HEADER_CASES)
def test_name_key(header, key):
    assert name_key(header) == key


def test_restatement_counts():
    recs = [("@A:1:FC:1:1101:1:1", "ACGT", "IIII"), ("@A:1:FC:1:1101:1:2", "AC", "#I"), ("@A:1:FC:1:01101:1:3", "A", "5"),
            ("@A:1:FC:2:5:1:1", "ACGTA", "!!!!I"), ("@SYN:C2:1:0000:00013:00000", "AC", "II")]
    got = restate(np.frombuffer(synth.fastq_bytes(recs), np.uint8))
    assert got["n_mates"] == 1 and got["cycles"] == 5 and got["n_tiles"] == 2 and got["overflow"] == 0
    assert got["reads"].tolist() == [5, 0] and got["untiled"].tolist() == [1, 0]
    assert got["lane"].tolist() == [1, 2] and got["tile"].tolist() == [1101, 5]
    assert got["tile_reads"][:, 0].tolist() == [3, 1] and got["tile_bases"][:, 0].tolist() == [7, 5]
    assert got["tile_qsum"][:, 0].tolist() == [40 * 4 + 2 + 40 + 20, 40]
    assert got["cycle_bases"][0, 0].tolist() == [3, 2, 1, 1, 0] and got["cycle_qsum"][0, 0].tolist() == [40 + 2 + 20, 80, 40, 40, 0]
    assert got["cycle_qsum"][1, 0].tolist() == [0, 0, 0, 0, 40]


def test_synth_tiled_plants_the_bubble():
    w = synth.tiled(4000, lanes=2, tiles_per_lane=4, order="shuffled")
    got = restate(w.r1, w.r2)
    assert got["n_tiles"] == 8 and got["untiled"].tolist() == [0, 0] and got["tile_reads"].sum() == 8000
    mean = got["cycle_qsum"] / got["cycle_bases"]
    bad = list(zip(got["lane"].tolist(), got["tile"].tolist())).index((1, 1102))
    assert (mean[bad, :, 49:80].mean() + 10) < np.delete(mean, bad, 0)[:, :, 49:80].mean()
    assert abs(mean[bad, :, :40].mean() - np.delete(mean, bad, 0)[:, :, :40].mean()) < 1


cli = pytest.mark.skipif(not os.path.exists(CLI), reason="CLI not built")


@cli
def test_cli_usage_lists_the_flag():
    p = subprocess.run([CLI], stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=60)
    assert b"--tile_quality" in p.stderr and b"prefix.tile_quality.txt" in p.stderr


# ---- GPU: the library ------------------------------------------------------------------------------------------------
def run_tq(r1, r2, opt, size, n_ctx=1, order=None, deal=None, mode="host"):
    """One pass through the API: batches of `size` records, permuted by `order`, dealt to n_ctx contexts on device 0
    (deal(j) picks the context of the j-th batch; default round robin).  Returns every context's tile_qual_results()."""
    r1, r2 = _as_u8(r1), _as_u8(r2)
    todo = cut(r1, r2, size)
    if order is not None:
        todo = [todo[i] for i in order(len(todo))]
    engines = [Engine(opt) for _ in range(n_ctx)]
    try:
        for e in engines:
            if mode == "pieces":
                e.set_output_pieces(True)
            e.tile_qual_enable()
        for c in range(n_ctx):
            mine = [b for j, b in enumerate(todo) if (deal(j) if deal else j % n_ctx) == c]
            if mine:
                run_batches(engines[c], mine, mode)
        if n_ctx == 1:
            engines[0].tile_qual_end_pass()
        else:
            dist_stats.tile_qual_end_pass_local(engines)
        return [e.tile_qual_results() for e in engines]
    finally:
        for e in engines:
            e.close()


def _mates(w, off):
    return w.r1, w.r2, off


def tiled_names(buf, mate, every=7):
    """The records of one mate under tiled names: 7-, 8- and 5-field names, leading zeros, every `every`-th read untiled
    (as in real runs with a second naming scheme).  A header's trailing '\\r' (CRLF input) stays."""
    lines = bytes(buf).split(b"\n")
    for i in range(0, len(lines) - 1, 4):
        r, cr = i // 4, b"\r" if lines[i].endswith(b"\r") else b""
        kind = r % every
        if kind == 0:
            name = b"@SYN:C2:1:%d:1:1 %d:N:0:1" % (r, mate)
        elif kind == 1:
            name = b"@M:7:FC:%d:%05d:%d:1:AACC %d:N:0:1" % (r % 3 + 1, 1100 + r % 5, r, mate)
        elif kind == 2:
            name = b"@HW:%d:%d:%d:1#0/%d" % (r % 3 + 1, 1100 + r % 5, r, mate)
        else:
            name = b"@M:7:FC:%d:%d:%d:1 %d:N:0:1" % (r % 3 + 1, 1100 + (r // 1000) % 5, r, mate)
        lines[i] = name + cr
    return np.frombuffer(b"\n".join(lines), np.uint8)


def low_bytes(buf, off, seed, frac=0.03):
    """A share of the quality bytes (never a line's '\\r') set below the offset: 33..off-1 at offset 64, 20..32 at offset
    33 (no '\\n' or '\\r'); their score is 0."""
    b = np.array(buf, np.uint8)
    nl = np.flatnonzero(b == 10)
    start = np.concatenate([[0], nl[:-1] + 1])
    qs, qe = start[3::4], nl[3::4]
    lens = qe - qs
    pos = np.repeat(qs, lens) + (np.arange(lens.sum()) - np.repeat(np.cumsum(lens) - lens, lens))
    pos = pos[b[pos] != 13]
    rng = np.random.default_rng(seed)
    pick = pos[rng.random(pos.size) < frac]
    b[pick] = rng.integers(33 if off == 64 else 20, off, size=pick.size)
    return b


def _renamed(r1, r2, off, low=False, seed=0):
    bufs = [None if x is None else tiled_names(x, m + 1) for m, x in enumerate((r1, r2))]
    if low:
        bufs = [None if x is None else low_bytes(x, off, seed + m) for m, x in enumerate(bufs)]
    return bufs[0], bufs[1], off


WORKLOADS = {
    "tiled_sorted": lambda: _mates(synth.tiled(30000, lanes=2, tiles_per_lane=24), 33),
    "tiled_shuffled": lambda: _mates(synth.tiled(30000, lanes=3, tiles_per_lane=20, order="shuffled", seed=3), 33),
    "tiled_single": lambda: _mates(synth.tiled(30000, lanes=1, tiles_per_lane=30, paired=False, L=100, seed=4), 33),
    "c2_untiled": lambda: _mates(synth.c2(20000), 33),
    "c2_renamed": lambda: _renamed(synth.c2(20000).r1, synth.c2(20000).r2, 33),
    "c5_phred64_ragged": lambda: _renamed(synth.c5(20000).r1, None, 64, low=True, seed=1),
    "fuzz_paired_crlf": lambda: _renamed(*fuzz_workload(1, True), 33, low=True, seed=2),
    "fuzz_single": lambda: _renamed(*fuzz_workload(2, False), 33, low=True, seed=3),
}


def _below_offset(buf, off):
    """Quality bytes below the offset in tiled reads, as framed."""
    keys, lens, read, cyc, _ = _mate_reads(buf, off)
    b = np.asarray(buf, np.uint8)
    nl = np.flatnonzero(b == 10)
    qs = np.concatenate([[0], nl[:-1] + 1])[3::4]
    tiled = np.array([k is not None for k in keys])
    return int(((b[qs[read] + cyc] < off) & tiled[read]).sum())


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(WORKLOADS))
def test_matches_restatement(name):
    r1, r2, off = WORKLOADS[name]()
    want = restate(r1, r2, off)
    if name.startswith("tiled"):
        assert want["n_tiles"] > 1 and not want["untiled"].any()
    if name == "c2_untiled":
        assert want["n_tiles"] == 0 and want["untiled"][0] == want["reads"][0]
    else:
        assert want["n_tiles"] > 1 and want["cycle_qsum"].sum() > 0
    if name in ("c5_phred64_ragged", "fuzz_paired_crlf", "fuzz_single"):
        # scores below the offset go through the accumulator as 0, and the restatement sees ragged and '\r'-cut reads
        assert _below_offset(r1, off) > 1000 and want["untiled"][0] > 0 and want["tile_reads"].sum() > want["untiled"].sum()
    for k, size in enumerate([1000, 7777, 1 << 20]):
        assert_same(run_tq(r1, r2, Options(input_quality_offset=off), size, order=shuffled(k))[0], want)


@pytest.mark.gpu
def test_header_cases_through_the_library():
    """Every hand-written name of test_name_key in one batch, tiled or not on the device as in the restatement, with quality
    bytes below the offset."""
    recs = b"".join(h + b"\nACGTA\n+\nI5 #!\n" for h, _ in HEADER_CASES * 3)
    r1 = np.frombuffer(recs, np.uint8)
    want = restate(r1)
    assert want["n_tiles"] == len({k for _, k in HEADER_CASES if k is not None})
    assert want["untiled"][0] == 3 * sum(k is None for _, k in HEADER_CASES)
    assert_same(run_tq(r1, None, Options(input_quality_offset=33), 1000)[0], want)


@pytest.mark.gpu
def test_reads_longer_than_1024_bases():
    rng = np.random.default_rng(5)
    lens = [1, 1023, 1024, 1025, 3000, 150, 2048, 0, 1100]
    recs = [(f"@X:1:FC:{1 + i % 2}:{1101 + i % 3}:1:{i}", "".join(rng.choice(list("ACGT"), size=n)),
             "".join(chr(33 + int(v)) for v in rng.integers(2, 42, size=n))) for i, n in enumerate(lens * 40)]
    r1 = np.frombuffer(synth.fastq_bytes(recs), np.uint8)
    want = restate(r1)
    assert want["cycles"] == 1024 and want["tile_bases"].sum() > want["cycle_bases"].sum()
    for size in (7, 100, 1000):
        assert_same(run_tq(r1, None, Options(input_quality_offset=33), size)[0], want)


def _keys_input(n_keys, seed=6, reps=2):
    """reps reads of each of n_keys distinct (lane, tile) keys, in random order."""
    rng = np.random.default_rng(seed)
    ks = np.repeat(np.arange(n_keys), reps)[rng.permutation(n_keys * reps)]
    recs = [(f"@K:1:FC:{1 + k % 9}:{k}:1:{i}", "ACGTACGTAC"[:1 + k % 10], "IIII#IIII5"[:1 + k % 10]) for i, k in enumerate(ks.tolist())]
    return np.frombuffer(synth.fastq_bytes(recs), np.uint8)


@pytest.mark.gpu
def test_full_table_and_overflow():
    opt = Options(input_quality_offset=33)
    full = _keys_input(MAX_KEYS)
    want = restate(full)
    assert want["n_tiles"] == MAX_KEYS and want["overflow"] == 0
    assert_same(run_tq(full, None, opt, 5000)[0], want)
    assert_same(run_tq(full, None, opt, 5000, n_ctx=3)[0], want)
    over = _keys_input(MAX_KEYS + 1, seed=7)
    want = restate(over)
    assert want["overflow"] == 1 and want["n_tiles"] == 0 and want["reads"][0] == 2 * (MAX_KEYS + 1)
    for n_ctx in (1, 2, 3):
        # split over 2 or 3 contexts, no single context sees more than the limit: the union still overflows
        for got in run_tq(over, None, opt, 4000, n_ctx=n_ctx):
            assert_same(got, want)
    # far more keys than the table has slots: the table never fills
    many = _keys_input(3 * 2 ** 15, seed=8, reps=1)
    assert_same(run_tq(many, None, opt, 1 << 20)[0], restate(many))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["pieces", "pipelined", "device"])
def test_batch_paths_match_process_host(mode):
    w = synth.tiled(30000, lanes=2, tiles_per_lane=10, order="shuffled", seed=8)
    want = restate(w.r1, w.r2)
    assert_same(run_tq(w.r1, w.r2, Options(input_quality_offset=33), 7000, mode=mode)[0], want)


@pytest.mark.gpu
def test_results_do_not_depend_on_options():
    w = synth.tiled(20000, lanes=2, tiles_per_lane=6, seed=9)
    want = restate(w.r1, w.r2)
    for opt in (Options(input_quality_offset=33, qc_only=True), Options(input_quality_offset=33, min_read_length=140, trim_5=10, discard_output=True)):
        assert_same(run_tq(w.r1, w.r2, opt, 6000)[0], want)


@pytest.mark.gpu
@pytest.mark.parametrize("n_ctx", [2, 3])
def test_contexts_with_uneven_deals_and_differing_tile_sets(n_ctx):
    w = synth.tiled(40000, lanes=4, tiles_per_lane=12, seed=10)        # sorted: each batch holds few tiles
    want = restate(w.r1, w.r2)
    deal_a = lambda j: 0 if j % 4 == 0 else (1 + j % (n_ctx - 1))
    deal_b = lambda j: 0 if j % 5 else n_ctx - 1
    for deal in (None, deal_a, deal_b):
        for got in run_tq(w.r1, w.r2, Options(input_quality_offset=33), 3000, n_ctx=n_ctx, deal=deal, order=shuffled(n_ctx)):
            assert_same(got, want)


@pytest.mark.gpu
def test_scores_above_41():
    """A score above 41 fails the batch with or without qc_only, unless terminal-N masking covers the base; then the batch
    passes and the base counts with its score as read."""
    bad = np.frombuffer(synth.fastq_bytes([("@A:1:FC:1:1101:1:1", "ACGT", "II~I")]), np.uint8)
    masked = np.frombuffer(synth.fastq_bytes([("@A:1:FC:1:1101:1:1", "NACGTN", "~IIII~"), ("@A:1:FC:1:1101:1:2", "AC", "II")]), np.uint8)
    for qc_only in (False, True):
        opt = Options(input_quality_offset=33, qc_only=qc_only)
        with Engine(opt) as e:
            e.tile_qual_enable()
            with pytest.raises(FaqcsError) as ex:
                e.process(bad)
            assert ex.value.status == FQ_ERR_QUALITY
        got = run_tq(masked, None, opt, 10)[0]
        assert_same(got, restate(masked))
        assert got["cycle_qsum"][0, 0, 0] == 93 + 40


@pytest.mark.gpu
def test_failed_batch_drops_the_pass():
    """A batch that fails after its keys were counted (|seq| != |qual| at framing, a score above 41 in k_trim) leaves no
    partial result: the end of the pass fails, and the next pass is exact."""
    w = synth.tiled(3000, lanes=1, tiles_per_lane=3, seed=16, paired=False)
    bad_len = np.frombuffer(synth.fastq_bytes([("@A:1:FC:9:9999:1:1", "ACGT", "III")]), np.uint8)
    bad_q = np.frombuffer(synth.fastq_bytes([("@A:1:FC:9:9998:1:1", "ACGT", "II~I")]), np.uint8)
    opt = Options(input_quality_offset=33)
    for bad, status in ((bad_len, FQ_ERR_FORMAT), (bad_q, FQ_ERR_QUALITY)):
        with Engine(opt) as a, Engine(opt) as b:
            for e in (a, b):
                e.tile_qual_enable()
            a.process(w.r1)
            assert _status(lambda: b.process(bad)) == status
            assert _status(lambda: dist_stats.tile_qual_end_pass_local([a, b])) == FQ_ERR_STATE
            got = a.tile_qual_results()
            assert got["n_mates"] == 0 and got["n_tiles"] == 0            # no pass finished
            b.process(w.r1)
            dist_stats.tile_qual_end_pass_local([a, b])
            assert_same(a.tile_qual_results(), restate(w.r1))
            a.process(w.r1)
            assert _status(lambda: a.process(bad)) == status
            assert _status(a.tile_qual_end_pass) == FQ_ERR_STATE
            a.process(w.r1)
            a.tile_qual_end_pass()
            assert_same(a.tile_qual_results(), restate(w.r1))


@pytest.mark.gpu
def test_two_passes_and_empty_pass():
    a = synth.tiled(5000, lanes=1, tiles_per_lane=3, seed=11)
    b = synth.tiled(3000, lanes=2, tiles_per_lane=2, seed=12, paired=False, L=80)
    with Engine(Options(input_quality_offset=33)) as e:
        e.tile_qual_enable()
        e.tile_qual_end_pass()
        got = e.tile_qual_results()
        assert got["n_mates"] == 0 and got["n_tiles"] == 0 and got["cycles"] == 0 and not got["reads"].any()
        e.process(a.r1, a.r2)
        e.tile_qual_end_pass()
        assert_same(e.tile_qual_results(), restate(a.r1, a.r2))
        e.process(b.r1)                                         # a single-end pass after a paired one
        e.tile_qual_end_pass()
        assert_same(e.tile_qual_results(), restate(b.r1))


def _status(fn):
    with pytest.raises(FaqcsError) as ex:
        fn()
    return ex.value.status


@pytest.mark.gpu
def test_refusals():
    w = synth.tiled(100, lanes=1, tiles_per_lane=2, seed=13)
    opt = Options(input_quality_offset=33)
    with Engine(opt) as a, Engine(opt) as b:
        assert _status(a.tile_qual_end_pass) == FQ_ERR_STATE
        assert _status(a.tile_qual_results) == FQ_ERR_STATE
        assert _status(lambda: dist_stats.tile_qual_end_pass_local([a, b])) == FQ_ERR_STATE
        a.tile_qual_enable()
        a.process(w.r1, w.r2)
        assert _status(a.tile_qual_enable) == FQ_ERR_STATE                                # in the middle of a pass
        assert _status(lambda: a.process(w.r1)) == FQ_ERR_ARG                             # single-end in a paired pass
        assert _status(lambda: dist_stats.tile_qual_end_pass_local([a, b])) == FQ_ERR_ARG  # enabled on one context only
        b.tile_qual_enable()
        b.process(w.r1)
        assert _status(lambda: dist_stats.tile_qual_end_pass_local([a, b])) == FQ_ERR_ARG  # paired on one, single-end on the other
    with Engine(opt) as a, Engine(opt) as b:
        for e in (a, b):
            e.tile_qual_enable()
        a.process(w.r1, w.r2)
        dist_stats.tile_qual_end_pass_local([a, b])
        assert_same(b.tile_qual_results(), restate(w.r1, w.r2))


# ---- the command line --------------------------------------------------------------------------------------------------
def run_cli(files, flags):
    tmp = tempfile.mkdtemp(prefix="faqcs_tile_")
    try:
        args = []
        for flag, (name, data) in files.items():
            path = os.path.join(tmp, name)
            if name.endswith(".gz"):
                with gzip.open(path, "wb", compresslevel=1) as fh:
                    fh.write(bytes(data))
            else:
                open(path, "wb").write(bytes(data))
            args += [flag, path]
        out = os.path.join(tmp, "out")
        p = subprocess.run([CLI, "-d", out] + args + flags, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=600)
        assert p.returncode == 0, p.stderr.decode(errors="replace")[-600:]
        return {n: open(os.path.join(out, n), "rb").read() for n in sorted(os.listdir(out))}
    finally:
        shutil.rmtree(tmp, ignore_errors=True)


@pytest.mark.gpu
@cli
@pytest.mark.parametrize("devices, gz", [("0,0", True), ("0", False)], ids=["devices_0_0_gzip", "one_device"])
def test_cli_tile_quality_file(devices, gz):
    w = synth.tiled(60000, lanes=2, tiles_per_lane=8)
    u = synth.tiled(30000, lanes=1, tiles_per_lane=5, paired=False, order="shuffled", seed=14, L=120)
    ext = ".fq.gz" if gz else ".fq"
    files = {"-1": ("r1" + ext, w.r1), "-2": ("r2" + ext, w.r2), "-u": ("u" + ext, u.r1)}
    flags = ["--batch_mb", "4", "--devices", devices, "--debug"]
    without = run_cli(files, flags)
    with_flag = run_cli(files, flags + ["--tile_quality"])
    got = with_flag.pop("QC.tile_quality.txt").decode()
    assert got == report(restate(w.r1, w.r2), True) + report(restate(u.r1), False)
    assert "QC.tile_quality.txt" not in without and sorted(without) == sorted(with_flag)
    for name in without:
        assert without[name] == with_flag[name], name


def test_report_of_an_overflowed_pass():
    res = {"n_mates": 1, "overflow": 1, "n_tiles": 0, "cycles": 4, "reads": np.array([10, 0], np.uint64), "untiled": np.array([3, 0], np.uint64)}
    assert report(res, False) == "pass\tunpaired\ttiles\t0\tcycles\t4\toverflow\t1\n#mate\treads\ttiled\tuntiled\n1\t10\t7\t3\n"


# ---- several GPUs ------------------------------------------------------------------------------------------------------
def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count() if torch.cuda.is_available() else 0
    except Exception:
        return 0


@pytest.mark.gpu
@pytest.mark.skipif(_n_gpus() < 2, reason="needs at least two GPUs")
def test_two_devices_in_one_process():
    w = synth.tiled(40000, lanes=3, tiles_per_lane=10, order="shuffled", seed=15)
    want = restate(w.r1, w.r2)
    todo = cut(_as_u8(w.r1), _as_u8(w.r2), 7000)
    engines = [Engine(Options(input_quality_offset=33), device=d) for d in (0, 1)]
    try:
        for e in engines:
            e.tile_qual_enable()
        for j, (first, final, a1, a2) in enumerate(todo):
            engines[j % 2].process(a1, a2, first, final)
        dist_stats.tile_qual_end_pass_local(engines)
        for e in engines:
            assert_same(e.tile_qual_results(), want)
    finally:
        for e in engines:
            e.close()
