"""k-mer rarefaction with the table sharded over several contexts (fq_kmer_end_pass_all): batches of one pass are dealt
to several contexts -- in any order, unevenly -- each counts into its own table, and the end of the pass merges the tables by
owner.  The files must be the reference's (tests/golden/kmer/), the single context's and the CPU oracle's."""
import ast
import glob
import os
import sys

import numpy as np
import pytest

from faqcs_b200 import dist_stats, synth
from faqcs_b200.api import Engine, FaqcsError, Options
from oracle_binding import OracleEngine
from parity import kmer_files, run_kmer

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
FIXTURES = sorted(glob.glob(os.path.join(HERE, "golden", "kmer", "*.npz")))
IDS = [os.path.basename(p)[:-4] for p in FIXTURES]
REF_BATCH = 32768
FQ_ERR_ARG = 1

pytestmark = pytest.mark.gpu


def _n_gpus():
    try:
        import torch
        return torch.cuda.device_count() if torch.cuda.is_available() else 0
    except Exception:
        return 0


def load(path):
    z = np.load(path)
    w = eval(bytes(z["paired"]).decode(), {"synth": synth})
    u = eval(bytes(z["unpaired"]).decode(), {"synth": synth})
    opt = Options(**ast.literal_eval(bytes(z["options"]).decode()))
    k, split, subset = (int(x) for x in z["params"])
    return [(w.r1, w.r2), (u.r1, None)], opt, k, split, subset, bytes(z["kmercount"]), bytes(z["kmerh"])


def fixture(name):
    return load(os.path.join(HERE, "golden", "kmer", name + ".npz"))


def record_offsets(buf):
    """Byte offset of every record start, and of the end."""
    nl = np.flatnonzero(buf == 10)
    assert nl.size % 4 == 0
    return np.concatenate([[0], nl[3::4] + 1]).astype(np.int64)


def batches(r1, r2, sizes=None):
    """The pass cut into batches of `sizes` records (default 32768 each; the last one takes the rest):
    [(index, first_record_index, is_final, r1 slice, r2 slice)]."""
    o1 = record_offsets(r1)
    o2 = record_offsets(r2) if r2 is not None else None
    n = o1.size - 1
    starts = [0]
    for s in (sizes or []):
        if starts[-1] + s >= n:
            break
        starts.append(starts[-1] + s)
    if not sizes:
        starts = list(range(0, max(n, 1), REF_BATCH))
    bounds = starts + [n]
    out = []
    for j in range(len(starts)):
        a, b = bounds[j], bounds[j + 1]
        out.append((j, a, j == len(starts) - 1, r1[o1[a]:o1[b]], r2[o2[a]:o2[b]] if r2 is not None else None))
    return out


def run_sharded(engines, passes, k, split, subset, sizes=None, order=None, owner=None, end_pass=None):
    """The k-mer API over `passes` with the batches dealt to `engines`: `order` permutes a pass's batch list, `owner(j, n)` picks
    the engine of batch j (default: round robin in the order run).  Returns every engine's (Kmercount, kmerH)."""
    end_pass = end_pass or dist_stats.kmer_end_pass_local
    for e in engines:
        e.kmer_enable(k, split, 2 * subset)
    first = True
    for r1, r2 in passes:
        r1 = np.frombuffer(bytes(r1), np.uint8)
        r2 = np.frombuffer(bytes(r2), np.uint8) if r2 is not None else None
        if first:
            for e in engines:
                e.autodetect(r1, r2)
            first = False
        todo = batches(r1, r2, sizes)
        if order:
            todo = order(todo)
        for t, (j, first_index, final, a1, a2) in enumerate(todo):
            eng = engines[owner(j, len(engines)) if owner else t % len(engines)]
            eng.process(a1, a2, first_index, final)
        end_pass(engines)
    return [kmer_files(*e.kmer_results()) for e in engines]


def with_engines(opt, devices, fn):
    engines = [Engine(opt, device=d) for d in devices]
    try:
        return fn(engines)
    finally:
        for e in engines:
            e.close()


# ---- 1. the reference's files, 2 and 3 contexts on one device -------------------------------------------------------
@pytest.mark.parametrize("n_ctx", [2, 3])
@pytest.mark.parametrize("path", FIXTURES, ids=IDS)
def test_sharded_reproduces_reference_kmer_files(path, n_ctx):
    passes, opt, k, split, subset, kc, kh = load(path)
    got = with_engines(opt, [0] * n_ctx, lambda es: run_sharded(es, passes, k, split, subset))
    for g in got:
        assert g == (kc, kh)


# ---- 2. batch order does not matter -----------------------------------------------------------------------------------
def _final_first(todo):
    return todo[-1:] + todo[:-1]


@pytest.mark.parametrize("order", [lambda t: t[::-1], _final_first], ids=["reversed", "final_first"])
@pytest.mark.parametrize("name", ["qc_only_early_stop", "qc_only_one_point"])
def test_sharded_batch_order_does_not_matter(name, order):
    passes, opt, k, split, subset, kc, kh = fixture(name)
    got = with_engines(opt, [0, 0], lambda es: run_sharded(es, passes, k, split, subset, order=order))
    for g in got:
        assert g == (kc, kh)
    # one context, batches out of order: the same files too
    got = with_engines(opt, [0], lambda es: run_sharded(es, passes, k, split, subset, order=order))
    assert got[0] == (kc, kh)


# ---- 3. unbalanced contexts, counts above 65535 ------------------------------------------------------------------------
def repeat_workload(n_pairs, seed=11):
    """Mate 1 of every pair is one of a few repeats (each of their k-mers is counted ~10^6 times: the list of large counts,
    spread over the owners), mate 2 a random read."""
    rng = np.random.default_rng(seed)
    motifs = ["A", "C", "AC", "AG", "CG", "AAC", "ACG", "AATT", "GGCA"]
    pick = rng.integers(0, len(motifs), n_pairs)
    rnd = rng.choice(np.array(list("ACGT")), size=(n_pairs, 150))
    r1 = [(f"@p{i}/1", (motifs[m] * 150)[:150], "I" * 150) for i, m in enumerate(pick)]
    r2 = [(f"@p{i}/2", "".join(rnd[i]), "I" * 150) for i in range(n_pairs)]
    return (np.frombuffer(synth.fastq_bytes(r1), np.uint8), np.frombuffer(synth.fastq_bytes(r2), np.uint8))


def test_sharded_unbalanced_contexts_and_large_counts():
    r1, r2 = repeat_workload(70000)
    passes = [(r1, r2)]
    opt = Options(qc_only=True, input_quality_offset=33)      # every quality is 'I': valid at both offsets, nothing to detect
    k, split, subset = 31, 30000, 3
    with Engine(opt) as one, OracleEngine(opt) as ora:
        want = run_kmer(one, passes, k, split, subset)
        assert run_kmer(ora, passes, k, split, subset) == want
    big = [int(c) for c, _ in [ln.split() for ln in want[1].decode().splitlines()] if int(c) > 65535]
    assert len(big) >= 4                                  # several k-mers counted more than 65535 times
    got = with_engines(opt, [0, 0], lambda es: run_sharded(es, passes, k, split, subset, owner=lambda j, n: 1 if j == 1 else 0))
    for g in got:
        assert g == want


# ---- 4. every table grows; the merged table grows ----------------------------------------------------------------------
def test_sharded_tables_grow():
    """Random reads (~120 distinct 31-mers per read): every context's table grows between batches, and in the uneven split
    the context that ran one batch (a table of 2^24 slots) owns about half of the 47 M distinct k-mers, so the table it
    merges into must be grown first."""
    w = synth.c2(6 * REF_BATCH)
    passes = [(w.r1, w.r2)]
    opt = Options(qc_only=True)
    k, split, subset = 31, 100000, 4
    with OracleEngine(opt) as ora:
        want = run_kmer(ora, passes, k, split, subset)
    got = with_engines(opt, [0, 0, 0], lambda es: run_sharded(es, passes, k, split, subset))
    for g in got:
        assert g == want
    got = with_engines(opt, [0, 0], lambda es: run_sharded(es, passes, k, split, subset, owner=lambda j, n: 1 if j == 2 else 0))
    for g in got:
        assert g == want


# ---- 5. fuzz -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("seed", range(8))
def test_sharded_kmer_fuzz_against_single_context_and_oracle(seed):
    from fuzz import fuzz_bytes, fuzz_options, fuzz_reads
    rng = np.random.default_rng(7000 + seed)
    in_off = 64 if seed % 4 == 3 else 33
    paired = seed % 2 == 0
    eol = "\r\n" if seed % 5 == 4 else "\n"
    n = 2 * REF_BATCH + int(rng.integers(1, 3000))
    r1 = fuzz_bytes(fuzz_reads(rng, n, in_off, "1" if paired else None), rng, eol)
    r2 = fuzz_bytes(fuzz_reads(rng, n, in_off, "2"), rng, eol) if paired else None
    kw = fuzz_options(rng, in_off, adapters=seed % 3 == 1)
    if seed % 2:
        kw["replace_to_N_q"] = 20
        kw["qc_only"] = False
    k = int(rng.choice([2, 5, 11, 21, 31]))
    split = int(rng.choice([5000, 30000, 100000, 1000000]))
    subset = int(rng.integers(1, 5))
    sizes = [REF_BATCH * int(rng.integers(1, 3)) for _ in range(4)]
    n_ctx = int(rng.integers(2, 4))
    perm = rng.permutation(8)
    passes = [(r1, r2)]
    with Engine(Options(**kw)) as one, OracleEngine(Options(**kw)) as ora:
        want = run_kmer(one, passes, k, split, subset)
        assert run_kmer(ora, passes, k, split, subset) == want
    got = with_engines(Options(**kw), [0] * n_ctx,
                       lambda es: run_sharded(es, passes, k, split, subset, sizes=sizes, order=lambda t: [t[i] for i in perm if i < len(t)]))
    for g in got:
        assert g == want


# ---- 6. refusals -------------------------------------------------------------------------------------------------------
def _three_batches():
    w = synth.c4(3 * REF_BATCH)
    r1 = np.frombuffer(bytes(w.r1), np.uint8)
    return batches(r1, None)


def _refusal(engines, runs, k=(31, 31), split=(1000, 1000)):
    for e, kk, ss in zip(engines, k, split):
        e.kmer_enable(kk, ss, 4)
    todo = _three_batches()
    for e in engines:
        e.autodetect(todo[0][3], None)
    for ctx_i, j, first_index in runs:
        _, _, final, a1, _ = todo[j]
        engines[ctx_i].process(a1, None, first_index, final)
    with pytest.raises(FaqcsError) as ex:
        dist_stats.kmer_end_pass_local(engines)
    assert ex.value.status == FQ_ERR_ARG
    return ex.value.message


def test_sharded_refuses_a_batch_run_twice():
    msg = with_engines(Options(qc_only=True), [0, 0], lambda es: _refusal(es, [(0, 0, 0), (1, 0, 0), (0, 1, REF_BATCH), (1, 2, 2 * REF_BATCH)]))
    assert "call 0 " in msg and "2 times" in msg


def test_sharded_refuses_a_missing_batch():
    msg = with_engines(Options(qc_only=True), [0, 0], lambda es: _refusal(es, [(0, 0, 0), (1, 2, 2 * REF_BATCH)]))
    assert "call 1 " in msg and "never run" in msg


@pytest.mark.parametrize("k, split", [((31, 21), (1000, 1000)), ((31, 31), (1000, 2000))], ids=["k", "split_size"])
def test_sharded_refuses_contexts_that_disagree(k, split):
    msg = with_engines(Options(qc_only=True), [0, 0], lambda es: _refusal(es, [(0, 0, 0), (1, 1, REF_BATCH), (0, 2, 2 * REF_BATCH)], k=k, split=split))
    assert "context 1" in msg and f"k = {k[1]}" in msg and f"split_size = {split[1]}" in msg


# ---- 7. command line: several contexts on one device -------------------------------------------------------------------
CLI_FLAGS = [["--qc_only", "--split_size", "30000", "--subset", "2"], ["--split_size", "10000", "--subset", "3", "-q", "20"]]


def _cli_available():
    import refcli
    return refcli.available() and os.path.exists(os.path.join(ROOT, "faqcs_b200", "host", "faqcs_b200"))


def _cli_kmer_files(devices, flags):
    from test_cli_dropin import assert_same_files, run_both
    w = synth.shotgun(70000)
    u = synth.shotgun(40000, seed=78, paired=False, L=100)
    outs = run_both({"-1": ("r1.fq", w.r1), "-2": ("r2.fq", w.r2), "-u": ("u.fq", u.r1)}, ["--kmer_rarefaction"] + flags, threads=3,
                    extra_cli=["--batch_mb", "16", "--devices", devices])
    assert "QC.Kmercount.txt" in outs["ref"] and "QC.kmerH.txt" in outs["ref"]
    assert_same_files(outs)


@pytest.mark.skipif(not _cli_available(), reason="reference binary / recorded runs or the CLI not present")
@pytest.mark.parametrize("devices", ["0,0", "0,0,0"])
@pytest.mark.parametrize("flags", CLI_FLAGS, ids=["qc_only", "trimmed"])
def test_cli_kmer_rarefaction_on_several_contexts(flags, devices):
    _cli_kmer_files(devices, flags)


# ---- 8. several GPUs ---------------------------------------------------------------------------------------------------
multi_gpu = pytest.mark.skipif(_n_gpus() < 2, reason="needs at least two GPUs")


@multi_gpu
@pytest.mark.parametrize("name", ["qc_only", "trimmed"])
def test_sharded_over_two_devices_in_one_process(name):
    passes, opt, k, split, subset, kc, kh = fixture(name)
    got = with_engines(opt, [0, 1], lambda es: run_sharded(es, passes, k, split, subset))
    for g in got:
        assert g == (kc, kh)


def _rank_worker(rank, world, port, name, q):
    sys.path.insert(0, HERE)
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    passes, opt, k, split, subset, _, _ = fixture(name)
    with Engine(opt, device=rank) as eng:
        got = run_sharded([eng], passes, k, split, subset, owner=lambda j, n: 0,
                          order=lambda t: [b for b in t if b[0] % world == rank],
                          end_pass=lambda es: dist_stats.kmer_end_pass_ranks(es[0], dist, dev))
    q.put((rank, got[0]))
    dist.barrier()
    dist.destroy_process_group()


@multi_gpu
def test_sharded_one_process_per_gpu_over_nccl():
    import socket
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    name = "qc_only_early_stop"
    _, _, _, _, _, kc, kh = fixture(name)
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_rank_worker, args=(r, 2, port, name, q)) for r in range(2)]
    for p in procs:
        p.start()
    got = dict(q.get(timeout=300) for _ in procs)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    assert got[0] == (kc, kh) and got[1] == (kc, kh)


@multi_gpu
@pytest.mark.skipif(not _cli_available(), reason="reference binary / recorded runs or the CLI not present")
@pytest.mark.parametrize("flags", CLI_FLAGS, ids=["qc_only", "trimmed"])
def test_cli_kmer_rarefaction_on_two_devices(flags):
    _cli_kmer_files("0,1", flags)
