"""Overrepresented sequences (fq_overrep_*, --overrep): each read's prefix (the first prefix_len bytes of its sequence line as
framed) counted per mate in a hash table per context, the bytes of the sequences above min_ppm of a mate's reads kept by a
capture rule, everything merged at the end of a pass.  The restatement below is a Counter over (mate, prefix bytes) with the
threshold and order of the definition; the library must give exactly its list."""
import collections
import gzip
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from faqcs_b200 import dist_stats, synth
from faqcs_b200.api import BUILTIN_ADAPTERS, POLYA_ADAPTER, Engine, FaqcsError, Options
from test_dup_stats import _as_u8, _fq, cut, fuzz_workload, run_batches, seq_lines, shuffled

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CLI = os.path.join(ROOT, "faqcs_b200", "host", "faqcs_b200")
FQ_ERR_ARG, FQ_ERR_STATE = 1, 8


# ---- the restatement ---------------------------------------------------------------------------------------------------
def restate(r1, r2=None, prefix_len=50, min_ppm=1000):
    """{"reads", "min_count", "seqs": [(mate, prefix bytes, count)]} of one pass, in the definition's order."""
    counts = collections.Counter()
    reads = [0, 0]
    for m, buf in enumerate((r1, r2)):
        if buf is None:
            continue
        b = bytes(np.asarray(buf, np.uint8))
        starts, lengths = seq_lines(buf)
        reads[m] = int(starts.size)
        for s, n in zip(starts.tolist(), lengths.tolist()):
            if n:
                counts[(m + 1, b[s:s + min(n, prefix_len)])] += 1
    min_count = [max(2, -(-min_ppm * n // 10**6)) for n in reads]
    seqs = [(m, s, c) for (m, s), c in counts.items() if c * 10**6 >= min_ppm * reads[m - 1] and c >= 2]
    seqs.sort(key=lambda t: (-t[2], t[0], t[1]))          # bytes compare as memcmp on the common length, shorter first
    return {"reads": reads, "min_count": min_count, "seqs": seqs}


def assert_same(got, want):
    assert got["reads"] == want["reads"] and got["min_count"] == want["min_count"], (got["reads"], want["reads"])
    assert len(got["seqs"]) == len(want["seqs"]), (len(got["seqs"]), len(want["seqs"]), got["seqs"][:5], want["seqs"][:5])
    assert got["seqs"] == want["seqs"]


# ---- CPU: the restatement on hand cases, the command line's usage and refusals -------------------------------------------
def test_threshold_boundary():
    """4000 reads at 1000 ppm: min_count 4, so 4 copies are listed and 3 are not; at 10 ppm min_count is 2, never 1."""
    seqs = ["AAAA"] * 4 + ["CCCC"] * 3 + [f"G{i:05d}" for i in range(3993)]
    got = restate(_fq(seqs))
    assert got["reads"] == [4000, 0] and got["min_count"] == [4, 2]
    assert got["seqs"] == [(1, b"AAAA", 4)]
    got = restate(_fq(["AAAA", "CCCC", "CCCC"]), min_ppm=10)
    assert got["min_count"] == [2, 2] and got["seqs"] == [(1, b"CCCC", 2)]


def test_prefix_collapse_case_and_line_ends():
    # equal in the first 4 bytes: one sequence; case counts; a read shorter than the prefix is its own sequence
    got = restate(_fq(["ACGTAA", "ACGTCC", "acgtAA", "acgt", "ACG", "ACG"]), prefix_len=4, min_ppm=10)
    assert got["seqs"] == [(1, b"ACG", 2), (1, b"ACGT", 2), (1, b"acgt", 2)]
    # CRLF ends the line at '\r'; a lone '\r' inside the line ends it too
    buf = np.frombuffer(synth.fastq_bytes([("@a", "AC\rGT", "II\rII"), ("@b", "AC", "II"), ("@c", "ACGT", "IIII")], "\r\n"), np.uint8)
    assert restate(buf, prefix_len=4, min_ppm=10)["seqs"] == [(1, b"AC", 2)]


def test_empty_reads_count_but_are_not_listed():
    got = restate(_fq(["", "", "", "A", "A"]), min_ppm=10)
    assert got["reads"] == [5, 0] and got["seqs"] == [(1, b"A", 2)]


def test_order_ties():
    """Count descending, then mate, then bytes (shorter first on a common prefix)."""
    r1 = _fq(["AG", "AG", "ACG", "ACG", "AC", "AC", "T", "T", "T"])
    r2 = _fq(["AA", "AA", "C", "C", "C", "G", "G", "G", "X"])
    got = restate(r1, r2, min_ppm=10)
    assert got["seqs"] == [(1, b"T", 3), (2, b"C", 3), (2, b"G", 3), (1, b"AC", 2), (1, b"ACG", 2), (1, b"AG", 2), (2, b"AA", 2)]


def test_synth_plants():
    n = 20000
    plants = [("ACGT" * 15, 20, 1, False), ("TTGCA" * 10, 19, 1, False), ("GATTACA" * 10, 30, 0, True), ("CCA" * 5, 25, 2, True)]
    w = synth.overrepresented(n, plants)
    got = restate(w.r1, w.r2)
    assert got["min_count"] == [20, 20]
    listed = {(m, s): c for m, s, c in got["seqs"]}
    assert listed[(1, ("ACGT" * 15)[:50].encode())] == 20                 # exactly at min_count
    assert (1, ("TTGCA" * 10).encode()) not in listed                     # one below
    assert listed[(1, ("GATTACA" * 10)[:50].encode())] == 30 and listed[(2, ("GATTACA" * 10)[:50].encode())] == 30
    assert listed[(2, b"CCA" * 5)] == 25                                  # shorter than the prefix
    d = restate(synth.overrepresented(n).r1)
    assert (1, synth.TRUSEQ_FRAGMENT[:50].encode(), n // 50) in d["seqs"]


cli = pytest.mark.skipif(not os.path.exists(CLI), reason="CLI not built")


def _cli(args):
    return subprocess.run([CLI] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=60)


@cli
def test_cli_usage_lists_the_flags():
    err = _cli([]).stderr
    for flag in (b"--overrep", b"--overrep_len", b"--overrep_ppm"):
        assert flag in err


@cli
@pytest.mark.parametrize("args, message", [
    (["--overrep_len", "0"], b"--overrep_len as an integer in the range 1 <= length <= 256"),
    (["--overrep_len", "257"], b"--overrep_len as an integer in the range 1 <= length <= 256"),
    (["--overrep_ppm", "9"], b"10 <= ppm <= 1000000"),
    (["--overrep_ppm", "1000001"], b"10 <= ppm <= 1000000"),
    (["--overrep_ppm", "1e3"], b"10 <= ppm <= 1000000"),
    (["--overrep", "--overrep_len", "0", "--lc", "2"], b"low complexity cutoff"),          # the reference's check comes first
], ids=["len_0", "len_257", "ppm_9", "ppm_1000001", "not_a_number", "reference_first"])
def test_cli_refusals(args, message):
    p = _cli(["-u", "X", "--overrep"] + args + ["-d", tempfile.gettempdir()])
    assert p.returncode != 0
    assert message in p.stderr, p.stderr.decode(errors="replace")[-400:]


# ---- GPU: the library ------------------------------------------------------------------------------------------------
def run_ovr(r1, r2, opt, size, n_ctx=1, order=None, deal=None, mode="host", prefix_len=50, min_ppm=1000):
    """One pass through the API: batches of `size` records, permuted by `order`, dealt to n_ctx contexts on device 0
    (deal(j) picks the context of the j-th batch; default round robin).  Returns every context's overrep_results()."""
    r1, r2 = _as_u8(r1), _as_u8(r2)
    todo = cut(r1, r2, size)
    if order is not None:
        todo = [todo[i] for i in order(len(todo))]
    engines = [Engine(opt) for _ in range(n_ctx)]
    try:
        for e in engines:
            if mode == "pieces":
                e.set_output_pieces(True)
            e.overrep_enable(prefix_len, min_ppm)
        for c in range(n_ctx):
            mine = [b for j, b in enumerate(todo) if (deal(j) if deal else j % n_ctx) == c]
            if mine:
                run_batches(engines[c], mine, mode)
        if n_ctx == 1:
            engines[0].overrep_end_pass()
        else:
            dist_stats.overrep_end_pass_local(engines)
        return [e.overrep_results() for e in engines]
    finally:
        for e in engines:
            e.close()


def _mates(w, off):
    return w.r1, w.r2, off


WORKLOADS = {
    "overrep_paired": lambda: _mates(synth.overrepresented(40000), 33),
    "overrep_single": lambda: _mates(synth.overrepresented(40000, seed=5, paired=False), 33),
    "c2": lambda: _mates(synth.c2(30000), 33),
    "c3": lambda: _mates(synth.c3(30000), 33),
    "shotgun": lambda: _mates(synth.shotgun(40000), 33),
    "fuzz_paired_crlf": lambda: fuzz_workload(1, True) + (33,),
    "fuzz_single": lambda: fuzz_workload(2, False) + (33,),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(WORKLOADS))
def test_matches_restatement(name):
    r1, r2, off = WORKLOADS[name]()
    for prefix_len, ppm in ((50, 1000), (20, 100)):
        want = restate(r1, r2, prefix_len, ppm)
        for k, size in enumerate([1000, 7777, 1 << 20]):
            got = run_ovr(r1, r2, Options(input_quality_offset=off), size, order=shuffled(k), prefix_len=prefix_len, min_ppm=ppm)[0]
            assert got["prefix_len"] == prefix_len and got["min_ppm"] == ppm
            assert_same(got, want)


def _background(n, seed, L=60):
    rng = np.random.default_rng(seed)
    return ["".join(rng.choice(list("ACGT"), size=L)) for _ in range(n)]


def _capture_case():
    """100 000 single-end reads, batches of 1000 in input order, 1000 ppm (min_count 100):
    FIRST: 150 copies in the first batch only, then diluted far below the running threshold;
    LAST: 100 copies, all in the last batch;
    EVEN: 100 copies, one per batch: exactly at the running threshold after every batch;
    BELOW: 99 copies, one per batch but the last."""
    n = 100000
    seqs = _background(n, 11)
    first, last, even, below = "A" * 10 + "C" * 50, "G" * 10 + "T" * 50, "ACGTTGCA" * 8, "TGCAACGT" * 8
    for i in range(150):
        seqs[3 + 6 * i] = first
    for i in range(100):
        seqs[n - 1000 + 7 * i] = last
        seqs[1000 * i + 500] = even
    for i in range(99):
        seqs[1000 * i + 501] = below
    return _fq(seqs), {first[:50], last[:50], even[:50]}, below[:50]


@pytest.mark.gpu
def test_capture_first_batch_last_batch_and_exact_threshold():
    r1, listed, below = _capture_case()
    want = restate(r1)
    assert {s.decode() for _, s, _ in want["seqs"]} == listed and want["min_count"] == [100, 2]
    assert_same(run_ovr(r1, None, Options(input_quality_offset=33), 1000)[0], want)
    assert_same(run_ovr(r1, None, Options(input_quality_offset=33), 1000, order=lambda n: list(range(n))[::-1])[0], want)


@pytest.mark.gpu
@pytest.mark.parametrize("n_ctx", [2, 3])
def test_capture_over_contexts(n_ctx):
    """CONC sits in batches that all go to context 0 (its share of context 0's reads is large); THIN is spread over every
    batch at one copy per batch, so no context holds much of it; uneven deals give some contexts few batches."""
    n, size = 60000, 500
    seqs = _background(n, 12)
    conc, thin = "CA" * 30, "GGT" * 20
    for i in range(120):
        seqs[size * (4 * (i % 6)) + 10 + i] = conc                         # batches 0, 4, ..., 20: context 0 under deal_a
    for b in range(n // size):
        seqs[size * b + 250] = thin
    r1 = _fq(seqs)
    want = restate(r1, None, 50, 1000)
    assert {s for _, s, _ in want["seqs"]} == {conc[:50].encode(), thin[:50].encode()}
    deal_a = lambda j: 0 if j % 4 == 0 else (1 + j % (n_ctx - 1))
    deal_b = lambda j: 0 if j % 5 else n_ctx - 1
    for deal in (None, deal_a, deal_b):
        for got in run_ovr(r1, None, Options(input_quality_offset=33), size, n_ctx=n_ctx, deal=deal):
            assert_same(got, want)


@pytest.mark.gpu
def test_results_do_not_depend_on_options():
    w = synth.overrepresented(20000, seed=7)
    want = restate(w.r1, w.r2)
    assert want["seqs"]
    adapters = list(BUILTIN_ADAPTERS) + [POLYA_ADAPTER]
    for opt in (Options(input_quality_offset=33), Options(input_quality_offset=33, qc_only=True),
                Options(input_quality_offset=33, filter_adapter=True, adapters=adapters, discard_output=True),
                Options(input_quality_offset=33, min_read_length=140, trim_5=10)):
        assert_same(run_ovr(w.r1, w.r2, opt, 6000)[0], want)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["pieces", "pipelined", "device"])
def test_batch_paths_match_process_host(mode):
    w = synth.overrepresented(30000, seed=8)
    want = run_ovr(w.r1, w.r2, Options(input_quality_offset=33), 7000)[0]
    assert_same(want, restate(w.r1, w.r2))
    assert_same(run_ovr(w.r1, w.r2, Options(input_quality_offset=33), 7000, mode=mode)[0], want)


@pytest.mark.gpu
def test_table_and_store_grow():
    """At 10 ppm every repeated prefix of the shotgun reads is listed (min_count 2) and early batches capture nearly every
    read: the count table (2^16 slots) and the capture store grow many times, contents kept."""
    w = synth.shotgun(60000)
    want = restate(w.r1, w.r2, 50, 10)
    assert len(want["seqs"]) > 1000
    assert_same(run_ovr(w.r1, w.r2, Options(input_quality_offset=33), 2500, min_ppm=10)[0], want)
    assert_same(run_ovr(w.r1, w.r2, Options(input_quality_offset=33), 2500, min_ppm=10, prefix_len=256, order=shuffled(3))[0],
                restate(w.r1, w.r2, 256, 10))


@pytest.mark.gpu
def test_two_passes_and_empty_pass():
    a = synth.overrepresented(10000, seed=9, paired=False).r1
    b = _fq(["AAAA", "AAAA", "C", ""])
    with Engine(Options(input_quality_offset=33)) as e:
        e.overrep_enable(50, 10)
        e.overrep_end_pass()
        got = e.overrep_results()
        assert got["reads"] == [0, 0] and got["min_count"] == [2, 2] and got["seqs"] == []
        e.process(a)
        e.overrep_end_pass()
        assert_same(e.overrep_results(), restate(a, None, 50, 10))
        e.overrep_enable(3, 20)                                         # between passes: new parameters
        e.process(b)
        e.overrep_end_pass()
        assert_same(e.overrep_results(), restate(b, None, 3, 20))


def _status(fn):
    with pytest.raises(FaqcsError) as ex:
        fn()
    return ex.value.status


@pytest.mark.gpu
def test_refusals():
    r1, r2 = _fq(["ACGT", "ACGT"]), _fq(["TT", "GG"])
    opt = Options(input_quality_offset=33)
    with Engine(opt) as a, Engine(opt) as b:
        assert _status(a.overrep_end_pass) == FQ_ERR_STATE
        assert _status(a.overrep_results) == FQ_ERR_STATE
        assert _status(lambda: dist_stats.overrep_end_pass_local([a, b])) == FQ_ERR_STATE
        for bad in ((0, 1000), (257, 1000), (50, 9), (50, 1000001)):
            assert _status(lambda: a.overrep_enable(*bad)) == FQ_ERR_ARG
        a.overrep_enable()
        a.process(r1, r2)
        assert _status(lambda: a.overrep_enable(40, 1000)) == FQ_ERR_STATE       # in the middle of a pass
        assert _status(lambda: dist_stats.overrep_end_pass_local([a, b])) == FQ_ERR_ARG   # enabled on one context only
        b.overrep_enable(40, 1000)
        assert _status(lambda: dist_stats.overrep_end_pass_local([a, b])) == FQ_ERR_ARG   # parameters differ
        b.overrep_enable(50, 1000)
        dist_stats.overrep_end_pass_local([a, b])
        assert_same(b.overrep_results(), restate(r1, r2))


# ---- the command line --------------------------------------------------------------------------------------------------
def parse_overrep_file(txt):
    """[(pass, prefix_len, ppm, {mate: (reads, min_count)}, [(mate, count, percent, sequence, source)])]"""
    passes = []
    section = None
    for ln in txt.decode().splitlines():
        f = ln.split("\t")
        if f[0] == "pass":
            assert f[2] == "prefix_len" and f[4] == "ppm"
            passes.append((f[1], int(f[3]), int(f[5]), {}, []))
        elif f[0] == "#mate":
            section = "reads" if f[1] == "reads" else "seqs"
            assert f == (["#mate", "reads", "min_count"] if section == "reads" else ["#mate", "count", "percent", "sequence", "source"])
        elif section == "reads":
            passes[-1][3][int(f[0])] = (int(f[1]), int(f[2]))
        else:
            passes[-1][4].append((int(f[0]), int(f[1]), f[2], f[3], f[4]))
    return passes


def check_block(block, name, want, prefix_len, ppm, mates):
    assert block[0] == name and block[1] == prefix_len and block[2] == ppm
    assert block[3] == {m + 1: (want["reads"][m], want["min_count"][m]) for m in range(mates)}
    assert [(m, c, s) for m, c, _, s, _ in block[4]] == [(m, c, s.decode()) for m, s, c in want["seqs"]]
    for m, c, pct, _, _ in block[4]:
        assert pct == "%.4f" % (100.0 * c / want["reads"][m - 1])


def run_cli(files, flags):
    tmp = tempfile.mkdtemp(prefix="faqcs_overrep_")
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


PRIMER = "GATTACAGATTACAGGCCTTAAGG"


def _rc(s):
    return s[::-1].translate(str.maketrans("ACGT", "TGCA"))


def _cli_inputs(gz):
    w = synth.overrepresented(60000)
    u = synth.overrepresented(30000, seed=78, paired=False, plants=[(synth.phix174()[2000:2100][::-1], 600, 1, True),
                                                                     ("acgtacgtacgt", 300, 1, True), (PRIMER, 200, 1, True)])
    ext = ".fq.gz" if gz else ".fq"
    return {"-1": ("r1" + ext, w.r1), "-2": ("r2" + ext, w.r2), "-u": ("u" + ext, u.r1)}, w, u


@pytest.mark.gpu
@cli
@pytest.mark.parametrize("devices, gz", [("0,0", False), ("0", True)], ids=["devices_0_0", "gzip"])
def test_cli_overrepresented_file(devices, gz):
    files, w, u = _cli_inputs(gz)
    got = parse_overrep_file(run_cli(files, ["--overrep", "--batch_mb", "4", "--devices", devices])["QC.overrepresented.txt"])
    assert len(got) == 2
    check_block(got[0], "paired", restate(w.r1, w.r2), 50, 1000, 2)
    check_block(got[1], "unpaired", restate(u.r1), 50, 1000, 1)
    src = {(m, s): source for m, _, _, s, source in got[0][4]}
    truseq = synth.TRUSEQ_FRAGMENT[:50]
    assert src[(1, truseq)] == "TruSeq-adapter-1" and src[(2, truseq)] == "TruSeq-adapter-1"
    phix = synth.phix174()[1000:1050]
    assert src[(1, phix)] == "PhiX174"
    assert src[(1, "ACACTCTTTCCCTACACGACGCTCTTCCGA")] == "Nextera-primer-adapter-2"     # on its reverse strand
    usrc = {s: source for _, _, _, s, source in got[1][4]}
    assert usrc[synth.phix174()[2000:2100][::-1][:50]] == "No Hit"              # reversed, not reverse-complemented
    assert usrc["acgtacgtacgt"] == "No Hit" and usrc[PRIMER] == "No Hit"


@pytest.mark.gpu
@cli
def test_cli_source_column_and_other_files_unchanged():
    """--overrep_len / --overrep_ppm, and --artifactFile entries: one matched on its reverse strand, one by a sequence shorter
    than 20 bases; every other output file is byte for byte the same as without --overrep."""
    files, w, u = _cli_inputs(False)
    tmp = tempfile.mkdtemp(prefix="faqcs_overrep_art_")
    try:
        fa = os.path.join(tmp, "art.fa")
        open(fa, "w").write(">my-primer\nTTTTT" + _rc(PRIMER).lower() + "\n>short\nTTACGTACGTACGTTT\n")
        flags = ["--batch_mb", "16", "--debug", "--discard", "--artifactFile", fa]
        without = run_cli(files, flags)
        with_flag = run_cli(files, flags + ["--overrep", "--overrep_len", "40", "--overrep_ppm", "500"])
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    got = parse_overrep_file(with_flag.pop("QC.overrepresented.txt"))
    check_block(got[0], "paired", restate(w.r1, w.r2, 40, 500), 40, 500, 2)
    check_block(got[1], "unpaired", restate(u.r1, None, 40, 500), 40, 500, 1)
    src = {(m, s): source for m, _, _, s, source in got[0][4]}
    assert src[(1, "ACACTCTTTCCCTACACGACGCTCTTCCGA")] == "Nextera-primer-adapter-2"     # built-in entries come first
    usrc = {s: source for _, _, _, s, source in got[1][4]}
    assert usrc[PRIMER] == "my-primer"                                       # reverse strand of a lower-case entry
    assert usrc["acgtacgtacgt"] == "short"                                   # upper-cased, shorter than 20: the whole of it
    assert "QC.overrepresented.txt" not in without
    assert sorted(without) == sorted(with_flag)
    for name in without:
        assert without[name] == with_flag[name], name


# ---- several GPUs ------------------------------------------------------------------------------------------------------
def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count() if torch.cuda.is_available() else 0
    except Exception:
        return 0


multi_gpu = pytest.mark.skipif(_n_gpus() < 2, reason="needs at least two GPUs")


@pytest.mark.gpu
@multi_gpu
def test_two_devices_in_one_process():
    w = synth.overrepresented(40000, seed=10)
    want = restate(w.r1, w.r2, 50, 100)
    todo = cut(_as_u8(w.r1), _as_u8(w.r2), 7000)
    engines = [Engine(Options(input_quality_offset=33), device=d) for d in (0, 1)]
    try:
        for e in engines:
            e.overrep_enable(50, 100)
        for j, (first, final, a1, a2) in enumerate(todo):
            engines[j % 2].process(a1, a2, first, final)
        dist_stats.overrep_end_pass_local(engines)
        for e in engines:
            assert_same(e.overrep_results(), want)
    finally:
        for e in engines:
            e.close()


def _rank_worker(rank, world, port, q):
    sys.path.insert(0, HERE)
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    w = synth.overrepresented(40000, seed=10)
    todo = cut(_as_u8(w.r1), _as_u8(w.r2), 7000)
    with Engine(Options(input_quality_offset=33), device=rank) as eng:
        eng.overrep_enable(50, 100)
        for j, (first, final, a1, a2) in enumerate(todo):
            if j % world == rank:
                eng.process(a1, a2, first, final)
        dist_stats.overrep_end_pass_ranks(eng, dist, dev)
        q.put((rank, eng.overrep_results()))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.gpu
@multi_gpu
def test_one_process_per_gpu_over_nccl():
    import socket
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    w = synth.overrepresented(40000, seed=10)
    want = restate(w.r1, w.r2, 50, 100)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_rank_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = [q.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for _, res in got:
        assert_same(res, want)


@pytest.mark.gpu
@multi_gpu
@cli
def test_cli_overrepresented_file_on_two_devices():
    files, w, u = _cli_inputs(False)
    got = parse_overrep_file(run_cli(files, ["--overrep", "--batch_mb", "4", "--devices", "0,1"])["QC.overrepresented.txt"])
    check_block(got[0], "paired", restate(w.r1, w.r2), 50, 1000, 2)
    check_block(got[1], "unpaired", restate(u.r1), 50, 1000, 1)
