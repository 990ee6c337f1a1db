"""Sequence duplication statistics (fq_dup_*, --dup_stats): one key per read (single-end) or pair, from the bytes of the
sequence line(s) as framed, counted in a hash table per context and merged at the end of a pass.  The numpy restatement
below computes the same fingerprint (fq_dup.cuh), so every comparison with it is exact."""
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

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CLI = os.path.join(ROOT, "faqcs_b200", "host", "faqcs_b200")
FQ_ERR_ARG, FQ_ERR_STATE = 1, 8
M64 = (1 << 64) - 1
WORD_MUL, LEN_MUL, PAIR_XOR = 0x9e3779b97f4a7c15, 0xc2b2ae3d27d4eb4f, 0x165667b19e3779f9


# ---- the restatement ---------------------------------------------------------------------------------------------------
def fmix64(x):
    x = np.asarray(x, np.uint64)
    with np.errstate(over="ignore"):
        x = x ^ (x >> np.uint64(33))
        x = x * np.uint64(0xff51afd7ed558ccd)
        x = x ^ (x >> np.uint64(33))
        x = x * np.uint64(0xc4ceb9fe1a85ec53)
        return x ^ (x >> np.uint64(33))


def seq_lines(buf):
    """(start, length) of every record's sequence line as framed: its bytes up to the first '\\r' or '\\n'."""
    buf = np.asarray(buf, np.uint8)
    nl = np.flatnonzero(buf == 10)
    assert nl.size % 4 == 0
    starts = np.concatenate([[0], nl[:-1] + 1])[1::4]
    ends = nl[1::4]
    cr = np.flatnonzero(buf == 13)
    if cr.size:
        j = np.searchsorted(cr, starts)
        ends = np.minimum(ends, np.where(j < cr.size, cr[np.minimum(j, cr.size - 1)], ends))
    return starts.astype(np.int64), (ends - starts).astype(np.int64)


def line_hash(buf, starts, lengths):
    """h(s) = fmix64(sum_i fmix64(w_i + (i + 1) * WORD_MUL) + len * LEN_MUL), w_i little-endian 8-byte words, the last zero-padded."""
    buf = np.asarray(buf, np.uint8)
    acc = np.zeros(starts.size, np.uint64)
    n_words = (lengths + 7) // 8
    for i in range(int(n_words.max()) if starts.size else 0):
        idx = np.flatnonzero(n_words > i)
        w = np.zeros(idx.size, np.uint64)
        for b in range(8):
            ok = lengths[idx] > 8 * i + b
            v = np.zeros(idx.size, np.uint64)
            v[ok] = buf[starts[idx[ok]] + 8 * i + b]
            w |= v << np.uint64(8 * b)
        with np.errstate(over="ignore"):
            acc[idx] += fmix64(w + np.uint64(((i + 1) * WORD_MUL) & M64))
    with np.errstate(over="ignore"):
        return fmix64(acc + lengths.astype(np.uint64) * np.uint64(LEN_MUL))


def unit_keys(r1, r2=None):
    key = line_hash(r1, *seq_lines(r1))
    if r2 is not None:
        with np.errstate(over="ignore"):
            key = fmix64(key + fmix64(line_hash(r2, *seq_lines(r2)) ^ np.uint64(PAIR_XOR)))
    key[key == np.uint64(M64)] = np.uint64(M64 - 1)
    return key


def summarize(keys):
    _, counts = np.unique(keys, return_counts=True)
    mult, n_keys = np.unique(counts, return_counts=True)
    return {"units": int(keys.size), "distinct": int(counts.size), "levels": np.stack([mult, n_keys], 1).astype(np.uint64).reshape(-1, 2)}


def restate(r1, r2=None):
    return summarize(unit_keys(r1, r2))


def assert_same(got, want):
    assert got["units"] == want["units"] and got["distinct"] == want["distinct"], (got, want)
    assert np.array_equal(got["levels"], want["levels"]), (got["levels"][:10], want["levels"][:10])


# ---- CPU: the restatement against hand-computed keys, the command line's usage text ----------------------------------
LINE150 = "".join("ACGT"[(i * 7 + i // 3) % 4] for i in range(150))
HAND_KEYS = [("", 0x0000000000000000), ("A", 0x8ae08db2af3248d1), ("ACGTACGT", 0x9e5cbc1d1d23a0fa), ("ACGTACGTN", 0xa1841ad195e65da7),
             (LINE150, 0x865212cad9963cc3)]


def _fq(seqs, eol="\n"):
    return np.frombuffer(synth.fastq_bytes([(f"@r{i}", s, "I" * len(s)) for i, s in enumerate(seqs)], eol), np.uint8)


def test_fingerprint_matches_hand_computed_keys():
    seqs = [s for s, _ in HAND_KEYS]
    assert [int(k) for k in unit_keys(_fq(seqs))] == [k for _, k in HAND_KEYS]
    assert [int(k) for k in unit_keys(_fq(seqs, "\r\n"))] == [k for _, k in HAND_KEYS]       # CRLF: the line ends at '\r'
    assert int(unit_keys(_fq(["ACGTACGTN"]), _fq(["TTGCA"]))[0]) == 0x03a5f04184f99bb2
    assert int(unit_keys(_fq(["TTGCA"]), _fq(["ACGTACGTN"]))[0]) != 0x03a5f04184f99bb2       # mates are ordered


def test_restatement_histogram():
    got = restate(_fq(["AC", "AC", "ac", "AC", "G", "G", "T"]))
    assert got["units"] == 7 and got["distinct"] == 4
    assert got["levels"].tolist() == [[1, 2], [2, 1], [3, 1]]


@pytest.mark.skipif(not os.path.exists(CLI), reason="CLI not built")
def test_cli_usage_lists_dup_stats():
    p = subprocess.run([CLI], stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=60)
    assert b"--dup_stats" in p.stderr


# ---- GPU: the library ------------------------------------------------------------------------------------------------
def record_offsets(buf):
    nl = np.flatnonzero(np.asarray(buf, np.uint8) == 10)
    return np.concatenate([[0], nl[3::4] + 1]).astype(np.int64)


def cut(r1, r2, size):
    """The input as batches of `size` records (the last one takes the rest): [(first_record_index, is_final, r1, r2)]."""
    o1 = record_offsets(r1)
    o2 = record_offsets(r2) if r2 is not None else None
    n = o1.size - 1
    starts = list(range(0, max(n, 1), size))
    out = []
    for j, a in enumerate(starts):
        b = min(n, a + size)
        out.append((a, j == len(starts) - 1, r1[o1[a]:o1[b]], r2[o2[a]:o2[b]] if r2 is not None else None))
    return out


def _as_u8(b):
    return None if b is None else np.frombuffer(bytes(b), np.uint8)


def run_batches(eng, todo, mode):
    if mode == "pipelined":
        tickets = []
        for i, (first, final, a1, a2) in enumerate(todo):
            tickets.append(eng.submit(a1, a2, first, final))
            if i >= 1:
                eng.run(tickets[i - 1])
            if i >= 2:
                eng.wait(tickets[i - 2])
        eng.run(tickets[-1])
        for t in tickets[max(0, len(tickets) - 2):]:
            eng.wait(t)
        return
    for first, final, a1, a2 in todo:
        if mode == "device":
            import torch
            d1 = torch.from_numpy(np.array(a1)).cuda(0)
            d2 = torch.from_numpy(np.array(a2)).cuda(0) if a2 is not None else None
            eng.process_device(d1.data_ptr(), d1.numel(), d2.data_ptr() if d2 is not None else None, d2.numel() if d2 is not None else 0, first, final)
            torch.cuda.synchronize()
        else:
            eng.process(a1, a2, first, final)


def run_dup(r1, r2, opt, size, n_ctx=1, order=None, deal=None, mode="host"):
    """One pass through the API: batches of `size` records, permuted by `order`, dealt to n_ctx contexts on device 0
    (deal(j) picks the context of the j-th batch run; default round robin).  Returns every context's dup_results()."""
    r1, r2 = _as_u8(r1), _as_u8(r2)
    todo = cut(r1, r2, size)
    if order is not None:
        todo = [todo[i] for i in order(len(todo))]
    engines = [Engine(opt) for _ in range(n_ctx)]
    try:
        for e in engines:
            if mode == "pieces":
                e.set_output_pieces(True)
            e.dup_enable()
        for c in range(n_ctx):
            mine = [b for j, b in enumerate(todo) if (deal(j) if deal else j % n_ctx) == c]
            if mine:
                run_batches(engines[c], mine, mode)
        if n_ctx == 1:
            engines[0].dup_end_pass()
        else:
            dist_stats.dup_end_pass_local(engines)
        return [e.dup_results() for e in engines]
    finally:
        for e in engines:
            e.close()


def shuffled(seed):
    return lambda n: list(np.random.default_rng(seed).permutation(n))


def planted(paired, seed=3):
    """1000 keys once, 200 twice, 50 seven times, one key 70 000 times (past the dense histogram) -- in random order.  Paired:
    every pair shares its R1 with the pair of another key, so only the R2 tells them apart."""
    rng = np.random.default_rng(seed)
    groups = [(1000, 1), (200, 2), (50, 7), (1, 70000)]
    seqs = ["".join(rng.choice(list("ACGT"), size=int(rng.integers(20, 160)))) for _ in range(sum(k for k, _ in groups))]
    ids = np.concatenate([np.repeat(np.arange(k) + sum(g[0] for g in groups[:gi]), m) for gi, (k, m) in enumerate(groups)])
    ids = ids[rng.permutation(ids.size)]
    want = {"units": int(ids.size), "distinct": len(seqs), "levels": np.array([[1, 1000], [2, 200], [7, 50], [70000, 1]], np.uint64)}
    if not paired:
        return _fq([seqs[i] for i in ids]), None, want
    r1 = _fq(["ACGT" * 10 if i % 2 else "TTTTGGGGCC" for i in ids])
    return r1, _fq([seqs[i] for i in ids]), want


@pytest.mark.gpu
@pytest.mark.parametrize("paired", [False, True], ids=["single", "paired"])
def test_planted_multiplicities(paired):
    r1, r2, want = planted(paired)
    assert_same(restate(r1, r2), want)
    opt = Options(input_quality_offset=33)
    assert_same(run_dup(r1, r2, opt, 10000, order=shuffled(1))[0], want)


def fuzz_workload(seed, paired):
    """tests/fuzz.py records (lengths 1..420, lower case, IUPAC, N runs), CRLF for odd seeds, a lone '\\r' at the same
    position of the sequence and quality lines of some records (the line ends there), copies of earlier records."""
    from fuzz import fuzz_reads
    rng = np.random.default_rng(900 + seed)
    n = 12000
    recs = [fuzz_reads(rng, n, 33, str(m + 1) if paired else None) for m in range(2 if paired else 1)]
    src = rng.integers(0, n, size=n // 3)                       # a third of the units repeat another one
    for m in range(len(recs)):
        for d, s in zip(range(n - src.size, n), src):
            recs[m][d] = (recs[m][d][0], recs[m][s][1], recs[m][s][2])
        for i in rng.integers(0, n, size=300):
            h, s, q = recs[m][i]
            if len(s) > 3:
                p = int(rng.integers(1, len(s) - 1))
                recs[m][i] = (h, s[:p] + "\r" + s[p + 1:], q[:p] + "\r" + q[p + 1:])
    eol = "\r\n" if seed % 2 else "\n"
    bufs = [np.frombuffer(synth.fastq_bytes(r, eol), np.uint8) for r in recs]
    return bufs[0], bufs[1] if paired else None


def _mates(w, off):
    return w.r1, w.r2, off


WORKLOADS = {
    "c2": lambda: _mates(synth.c2(30000), 33),
    "c5": lambda: _mates(synth.c5(30000), 64),
    "shotgun": lambda: _mates(synth.shotgun(40000), 33),
    "shotgun_unpaired": lambda: _mates(synth.shotgun(40000, seed=78, paired=False, L=100), 33),
    "fuzz_paired_crlf": lambda: fuzz_workload(1, True) + (33,),
    "fuzz_single": lambda: fuzz_workload(2, False) + (33,),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(WORKLOADS))
def test_matches_restatement(name):
    r1, r2, off = WORKLOADS[name]()
    want = restate(r1, r2)
    for k, size in enumerate([1000, 7777, 1 << 20]):
        assert_same(run_dup(r1, r2, Options(input_quality_offset=off), size, order=shuffled(k))[0], want)


@pytest.mark.gpu
def test_counts_do_not_depend_on_options():
    w = synth.c3(20000)
    dup_half = lambda b: np.concatenate([b, b[:record_offsets(b)[5000]]])         # 5000 pairs twice
    r1, r2 = dup_half(w.r1), dup_half(w.r2)
    want = restate(r1, r2)
    assert want["units"] - want["distinct"] >= 5000
    adapters = list(BUILTIN_ADAPTERS) + [POLYA_ADAPTER] + list(w.artifacts)
    for opt in (Options(input_quality_offset=33), Options(input_quality_offset=33, qc_only=True),
                Options(input_quality_offset=33, filter_adapter=True, adapters=adapters, discard_output=True)):
        assert_same(run_dup(r1, r2, opt, 6000)[0], want)


@pytest.mark.gpu
def test_table_grows():
    """Almost every pair distinct, 10 000 pairs per batch into a table of 2^16 slots grown at half load: it grows before
    batches 4, 7 and 13; the single batch grows it once, straight to its size."""
    w = synth.c2(120000)
    want = restate(w.r1, w.r2)
    assert want["distinct"] > 110000
    assert_same(run_dup(w.r1, w.r2, Options(input_quality_offset=33), 10000)[0], want)
    assert_same(run_dup(w.r1, w.r2, Options(input_quality_offset=33), 1 << 20)[0], want)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["pieces", "pipelined", "device"])
def test_batch_paths_match_process_host(mode):
    w = synth.shotgun(40000)
    want = run_dup(w.r1, w.r2, Options(input_quality_offset=33), 9000)[0]
    assert_same(want, restate(w.r1, w.r2))
    assert_same(run_dup(w.r1, w.r2, Options(input_quality_offset=33), 9000, mode=mode)[0], want)


@pytest.mark.gpu
@pytest.mark.parametrize("n_ctx", [2, 3])
@pytest.mark.parametrize("paired", [True, False], ids=["paired", "single"])
def test_several_contexts_on_one_device(n_ctx, paired):
    w = synth.shotgun(50000, paired=paired)
    r2 = w.r2 if paired else None
    want = run_dup(w.r1, r2, Options(input_quality_offset=33), 6000)[0]
    assert_same(want, restate(w.r1, r2))
    for deal in (None, lambda j: 0 if j % 4 else 1):            # round robin; uneven (the last context may get nothing)
        for got in run_dup(w.r1, r2, Options(input_quality_offset=33), 6000, n_ctx=n_ctx, order=shuffled(5), deal=deal):
            assert_same(got, want)


@pytest.mark.gpu
def test_two_passes_and_empty_pass():
    """The end of a pass clears the table: the second pass counts alone; a pass without batches gives zeros."""
    a, b = planted(False)[0], _fq(["AAAA", "AAAA", "C"])
    with Engine(Options(input_quality_offset=33)) as e:
        e.dup_enable()
        e.dup_end_pass()
        got = e.dup_results()
        assert got["units"] == 0 and got["distinct"] == 0 and got["levels"].shape == (0, 2)
        e.process(a)
        e.dup_end_pass()
        e.process(b)
        e.dup_end_pass()
        assert_same(e.dup_results(), restate(b))


# ---- refusals ----------------------------------------------------------------------------------------------------------
def _status(fn):
    with pytest.raises(FaqcsError) as ex:
        fn()
    return ex.value.status


@pytest.mark.gpu
def test_refusals():
    r1, r2 = _fq(["ACGT", "ACGT"]), _fq(["TT", "GG"])
    opt = Options(input_quality_offset=33)
    with Engine(opt) as a, Engine(opt) as b:
        assert _status(a.dup_end_pass) == FQ_ERR_STATE
        assert _status(a.dup_results) == FQ_ERR_STATE
        assert _status(lambda: dist_stats.dup_end_pass_local([a, b])) == FQ_ERR_STATE
        a.dup_enable()
        a.process(r1, r2)
        assert _status(lambda: dist_stats.dup_end_pass_local([a, b])) == FQ_ERR_ARG       # enabled on one context only
        b.dup_enable()
        b.process(r1)
        assert _status(lambda: dist_stats.dup_end_pass_local([a, b])) == FQ_ERR_ARG       # pairs on one, reads on the other
        assert _status(lambda: a.process(r1)) == FQ_ERR_ARG                             # reads after pairs in one pass
    with Engine(opt) as a:
        a.dup_enable()
        a.process(r1, r2)
        a.dup_end_pass()
        a.process(r1)                                                                   # a new pass may count reads
        a.dup_end_pass()
        assert_same(a.dup_results(), restate(r1))


# ---- the command line --------------------------------------------------------------------------------------------------
def parse_dup_file(txt):
    passes = []
    for ln in txt.decode().splitlines():
        f = ln.split("\t")
        if f[0] == "pass":
            assert f[2] == "units" and f[4] == "distinct" and f[6] == "duplicates" and int(f[7]) == int(f[3]) - int(f[5])
            passes.append((f[1], {"units": int(f[3]), "distinct": int(f[5]), "levels": []}))
        else:
            passes[-1][1]["levels"].append([int(f[0]), int(f[1])])
    for _, p in passes:
        p["levels"] = np.array(p["levels"], np.uint64).reshape(-1, 2)
    return passes


def run_cli(files, flags):
    tmp = tempfile.mkdtemp(prefix="faqcs_dup_")
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


cli = pytest.mark.skipif(not os.path.exists(CLI), reason="CLI not built")


def _cli_inputs(gz):
    w = synth.shotgun(50000)
    u = synth.shotgun(30000, seed=78, paired=False, L=100)
    ext = ".fq.gz" if gz else ".fq"
    files = {"-1": ("r1" + ext, w.r1), "-2": ("r2" + ext, w.r2), "-u": ("u" + ext, u.r1)}
    return files, [("paired", restate(w.r1, w.r2)), ("unpaired", restate(u.r1))]


@pytest.mark.gpu
@cli
@pytest.mark.parametrize("devices, gz", [("0", False), ("0,0", False), ("0", True)], ids=["one", "devices_0_0", "gzip"])
def test_cli_duplication_file(devices, gz):
    files, want = _cli_inputs(gz)
    outs = run_cli(files, ["--dup_stats", "--batch_mb", "4", "--devices", devices])
    got = parse_dup_file(outs["QC.duplication.txt"])
    assert [k for k, _ in got] == [k for k, _ in want]
    for (_, g), (_, w) in zip(got, want):
        assert_same(g, w)


@pytest.mark.gpu
@cli
def test_cli_without_flag_writes_no_duplication_file_and_the_same_files():
    files, _ = _cli_inputs(False)
    flags = ["--batch_mb", "16", "--debug", "--discard", "--adapter"]       # adapters: batches of whole 32768-record chunks
    without = run_cli(files, flags)
    with_flag = run_cli(files, flags + ["--dup_stats"])
    assert "QC.duplication.txt" not in without
    assert with_flag.pop("QC.duplication.txt")
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
    w = synth.shotgun(40000)
    want = restate(w.r1, w.r2)
    todo = cut(_as_u8(w.r1), _as_u8(w.r2), 7000)
    engines = [Engine(Options(input_quality_offset=33), device=d) for d in (0, 1)]
    try:
        for e in engines:
            e.dup_enable()
        for j, (first, final, a1, a2) in enumerate(todo):
            engines[j % 2].process(a1, a2, first, final)
        dist_stats.dup_end_pass_local(engines)
        for e in engines:
            assert_same(e.dup_results(), want)
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
    w = synth.shotgun(40000)
    todo = cut(_as_u8(w.r1), _as_u8(w.r2), 7000)
    with Engine(Options(input_quality_offset=33), device=rank) as eng:
        eng.dup_enable()
        for j, (first, final, a1, a2) in enumerate(todo):
            if j % world == rank:
                eng.process(a1, a2, first, final)
        dist_stats.dup_end_pass_ranks(eng, dist, dev)
        got = eng.dup_results()
    q.put((rank, got["units"], got["distinct"], got["levels"].tolist()))
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
    w = synth.shotgun(40000)
    want = restate(w.r1, w.r2)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_rank_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = [q.get(timeout=300) for _ in procs]
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for _, units, distinct, levels in got:
        assert_same({"units": units, "distinct": distinct, "levels": np.array(levels, np.uint64).reshape(-1, 2)}, want)


@pytest.mark.gpu
@multi_gpu
@cli
def test_cli_duplication_file_on_two_devices():
    files, want = _cli_inputs(False)
    got = parse_dup_file(run_cli(files, ["--dup_stats", "--batch_mb", "4", "--devices", "0,1"])["QC.duplication.txt"])
    assert [k for k, _ in got] == [k for k, _ in want]
    for (_, g), (_, w) in zip(got, want):
        assert_same(g, w)
