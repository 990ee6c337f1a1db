"""Paired-end insert size and overlap error profile (fq_overlap_*, --insert_size): for every pair, the overlap of R1 with the
reverse complement of R2, as defined in fq_overlap.cuh and include/faqcs_b200.h.  A scalar pure-Python statement of the
definition checks a numpy restatement (vectorised over the candidate insert sizes of the pairs with the same mate lengths),
and the library is compared with the numpy restatement exactly."""
import gzip
import os
import shutil
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from faqcs_b200 import dist_stats, synth
from faqcs_b200.api import BUILTIN_ADAPTERS, MODE_HARD, OVERLAP_CYCLE_ARRAYS, OVERLAP_SCALARS, POLYA_ADAPTER, Engine, FaqcsError, Options
from test_dup_stats import _as_u8, _status, cut, fuzz_workload, run_batches, seq_lines, shuffled

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CLI = os.path.join(ROOT, "faqcs_b200", "host", "faqcs_b200")
FQ_ERR_ARG, FQ_ERR_STATE = 1, 8
DEFAULT = (30, 5, 20)

# 2-bit codes of the known bases (either case); -1 for every other byte
CODE = np.full(256, -1, np.int8)
for i, ch in enumerate(b"ACGT"):
    CODE[ch] = CODE[ch | 0x20] = i


# ---- the scalar statement ------------------------------------------------------------------------------------------------
def scalar_pair(a, r2, O, D, P):
    """(m, o, s) of the pair's accepted overlap, None when there is none, "short" when a mate is shorter than O."""
    L1, L2 = len(a), len(r2)
    if L1 < O or L2 < O:
        return "short"
    fa = [int(CODE[c]) for c in a]
    fb = [3 - int(CODE[r2[L2 - 1 - j]]) if CODE[r2[L2 - 1 - j]] >= 0 else -1 for j in range(L2)]
    best = None
    for s in range(O, L1 + L2 - O + 1):
        x0, x1 = max(0, s - L2), min(L1, s)
        o = x1 - x0
        m = sum(1 for x in range(x0, x1) if fa[x] < 0 or fa[x] != fb[x - s + L2])
        if m <= min(D, o * P // 100) and (best is None or (m, -o, s) < (best[0], -best[1], best[2])):
            best = (m, o, s)
    return best


def empty_result():
    return {k: 0 for k in OVERLAP_SCALARS}, {}, {k: {} for k in OVERLAP_CYCLE_ARRAYS}


def finish(sc, ins, cyc):
    out = dict(sc)
    n_ins = max(ins) + 1 if ins else 0
    out["insert_hist"] = np.zeros(n_ins, np.uint64)
    for s, v in ins.items():
        out["insert_hist"][s] = v
    n_cyc = max([max(d) + 1 for d in cyc.values() if d] or [0])
    for k, d in cyc.items():
        out[k] = np.zeros(n_cyc, np.uint64)
        for x, v in d.items():
            out[k][x] = v
    return out


def scalar_restate(pairs, O=30, D=5, P=20):
    """The definition, one pair and one candidate at a time: pairs = [(r1 sequence bytes, r2 sequence bytes)]."""
    sc, ins, cyc = empty_result()
    for a, r2 in pairs:
        sc["pairs"] += 1
        got = scalar_pair(a, r2, O, D, P)
        if got == "short":
            sc["too_short"] += 1
            continue
        if got is None:
            continue
        m, o, s = got
        L1, L2 = len(a), len(r2)
        sc["overlapped"] += 1
        sc["r1_adapter"] += s < L1
        sc["r2_adapter"] += s < L2
        sc["overlap_bases"] += o
        sc["mismatch_bases"] += m
        ins[s] = ins.get(s, 0) + 1
        for x in range(max(0, s - L2), min(L1, s)):
            y = s - 1 - x
            ca, cb = int(CODE[a[x]]), int(CODE[r2[y]])
            hit = ca < 0 or cb < 0 or ca != 3 - cb
            for k, i in (("r1_overlap", x), ("r2_overlap", y)) + ((("r1_mismatch", x), ("r2_mismatch", y)) if hit else ()):
                cyc[k][i] = cyc[k].get(i, 0) + 1
    return finish(sc, ins, cyc)


# ---- the numpy restatement -----------------------------------------------------------------------------------------------
def mate_codes(buf):
    """Every record's sequence line as framed, as 2-bit codes (-1 unknown): (list of arrays)."""
    buf = np.asarray(buf, np.uint8)
    starts, lengths = seq_lines(buf)
    return starts, lengths, CODE[buf]


def restate(r1, r2, O=30, D=5, P=20):
    """The definition over whole FASTQ buffers: pairs grouped by (L1, L2), every candidate s of a group tested on all its
    pairs at once."""
    s1, l1, c1 = mate_codes(r1)
    s2, l2, c2 = mate_codes(r2)
    assert s1.size == s2.size
    n = s1.size
    out = {k: 0 for k in OVERLAP_SCALARS}
    out["pairs"] = n
    short = (l1 < O) | (l2 < O)
    out["too_short"] = int(short.sum())
    maxlen = int(max(l1.max(initial=0), l2.max(initial=0)))
    ins = np.zeros(2 * maxlen + 1, np.uint64)
    cyc = {k: np.zeros(maxlen + 1, np.int64) for k in OVERLAP_CYCLE_ARRAYS}
    keys = np.stack([l1, l2], 1)[~short]
    idx_ok = np.flatnonzero(~short)
    for L1, L2 in np.unique(keys, axis=0) if keys.size else []:
        L1, L2 = int(L1), int(L2)
        sel = idx_ok[(l1[idx_ok] == L1) & (l2[idx_ok] == L2)]
        A = c1[s1[sel, None] + np.arange(L1)[None, :]]
        B = c2[s2[sel, None] + (L2 - 1 - np.arange(L2))[None, :]]          # reverse complement of R2
        B = np.where(B >= 0, 3 - B, -1)
        cands = np.arange(O, L1 + L2 - O + 1)
        x0 = np.maximum(0, cands - L2)
        x1 = np.minimum(L1, cands)
        o = x1 - x0
        lim = np.minimum(D, o * P // 100)

        def mism(k):
            s = int(cands[k])
            a = A[:, x0[k]:x1[k]]
            b = B[:, x0[k] - s + L2:x1[k] - s + L2]
            return (a < 0) | (a != b)
        M = np.stack([mism(k).sum(1) for k in range(cands.size)], 1)
        ok = M <= lim[None, :]
        cost = np.where(ok, (M.astype(np.int64) << 42) + ((2 ** 21 - o[None, :]) << 21) + cands[None, :], np.iinfo(np.int64).max)
        win = cost.argmin(1)
        has = ok[np.arange(sel.size), win]
        for k in np.unique(win[has]):
            rows = np.flatnonzero(has & (win == k))
            s = int(cands[k])
            out["overlapped"] += rows.size
            out["r1_adapter"] += rows.size * (s < L1)
            out["r2_adapter"] += rows.size * (s < L2)
            out["overlap_bases"] += rows.size * int(o[k])
            mm = mism(k)[rows].sum(0)
            out["mismatch_bases"] += int(mm.sum())
            ins[s] += rows.size
            xs = np.arange(x0[k], x1[k])
            cyc["r1_overlap"][xs] += rows.size
            cyc["r2_overlap"][s - 1 - xs] += rows.size
            cyc["r1_mismatch"][xs] += mm
            cyc["r2_mismatch"][s - 1 - xs] += mm
    nz = np.flatnonzero(ins)
    out["insert_hist"] = ins[:nz[-1] + 1] if nz.size else np.zeros(0, np.uint64)
    n_cyc = max([int(np.flatnonzero(v)[-1]) + 1 if v.any() else 0 for v in cyc.values()])
    for k, v in cyc.items():
        out[k] = v[:n_cyc].astype(np.uint64)
    return out


def assert_same(got, want):
    for k in OVERLAP_SCALARS:
        assert got[k] == want[k], (k, got[k], want[k])
    for k in ("insert_hist",) + OVERLAP_CYCLE_ARRAYS:
        assert np.array_equal(np.asarray(got[k], np.uint64), np.asarray(want[k], np.uint64)), (k, got[k][:20], want[k][:20])


# ---- CPU: the restatements on hand-built pairs -----------------------------------------------------------------------
COMP = bytes.maketrans(b"ACGTacgt", b"TGCAtgca")


def rc(s):
    return s.translate(COMP)[::-1]


def _fq(seqs, eol="\n"):
    return np.frombuffer(synth.fastq_bytes([(f"@r{i}", s, "I" * len(s)) for i, s in enumerate(seqs)], eol), np.uint8)


def both(pairs, O=30, D=5, P=20):
    """Both restatements of the same pairs (sequences as str), checked equal; returns the result."""
    want = scalar_restate([(a.encode(), b.encode()) for a, b in pairs], O, D, P)
    got = restate(_fq([a for a, _ in pairs]), _fq([b for _, b in pairs]), O, D, P)
    assert_same(got, want)
    return got


def randseq(rng, n, alphabet="ACGT"):
    return "".join(rng.choice(list(alphabet), size=n))


def one(a, b, O=30, D=5, P=20):
    return scalar_pair(a.encode(), b.encode(), O, D, P)


def test_full_overlap():
    frag = randseq(np.random.default_rng(1), 150)
    assert one(frag, rc(frag)) == (0, 150, 150)
    got = both([(frag, rc(frag))])
    assert got["overlapped"] == 1 and got["r1_adapter"] == 0 and got["r2_adapter"] == 0
    assert got["insert_hist"].size == 151 and got["insert_hist"][150] == 1
    assert got["r1_overlap"].tolist() == [1] * 150 and got["r2_overlap"].tolist() == [1] * 150


def test_fragment_shorter_than_both_mates():
    rng = np.random.default_rng(2)
    frag = randseq(rng, 80)
    ad1, ad2 = dict(BUILTIN_ADAPTERS)["Nextera-primer-adapter-1"], dict(BUILTIN_ADAPTERS)["Nextera-primer-adapter-2"]
    r1 = (frag + ad1 + randseq(rng, 100))[:150]
    r2 = (rc(frag) + ad2 + randseq(rng, 100))[:150]
    assert one(r1, r2) == (0, 80, 80)
    got = both([(r1, r2)])
    assert got["r1_adapter"] == 1 and got["r2_adapter"] == 1 and got["overlap_bases"] == 80
    assert got["r1_overlap"].tolist() == [1] * 80 and got["r2_overlap"].tolist() == [1] * 80


def test_mismatch_limit_d_accepted_d_plus_one_rejected():
    rng = np.random.default_rng(3)
    frag = randseq(rng, 200)
    r1, r2 = frag[:150], rc(frag[50:])
    def flip(s, pos):
        s = list(s)
        for p in pos:
            s[p] = {"A": "C", "C": "G", "G": "T", "T": "A"}[s[p]]
        return "".join(s)
    five = flip(r1, [60, 70, 80, 90, 100])
    assert one(five, r2) == (5, 100, 200)
    got = both([(five, r2)])
    assert got["r1_mismatch"].nonzero()[0].tolist() == [60, 70, 80, 90, 100]
    assert got["r2_mismatch"].nonzero()[0].tolist() == sorted(199 - x for x in [60, 70, 80, 90, 100])
    six = flip(r1, [60, 70, 80, 90, 100, 110])
    assert one(six, r2) != (6, 100, 200)
    assert one(six, r2, D=6) == (6, 100, 200)
    both([(six, r2)])


def test_percent_limit_with_small_min_overlap():
    # 10 positions of overlap allow floor(10 * 20 / 100) = 2 mismatches, 9 positions only 1
    assert one("ACGTACGTAC", rc("ACGTACGTAC"), O=5) == (0, 10, 10)
    two = "ACCTACGAAC"                         # 2 mismatches against ACGTACGTAC over 10
    assert one(two, rc("ACGTACGTAC"), O=10) == (2, 10, 10)
    three = "ACCTACGAAA"
    assert one(three, rc("ACGTACGTAC"), O=10) is None
    assert one("ACCTACGAA", rc("ACGTACGTA"), O=9) is None          # 2 mismatches > floor(9 * 0.2) = 1
    both([(two, rc("ACGTACGTAC")), (three, rc("ACGTACGTAC")), ("ACCTACGAA", rc("ACGTACGTA"))], O=9)
    both([("ACGTACGTAC", rc("ACGTACGTAC")), ("ACGTTGCAACGGGGG", rc("TTACGTTGCAAC"))], O=5)


def test_ties_by_overlap_then_by_insert_size():
    # period-4 sequences: every shift by a multiple of 4 is a perfect match; the longest overlap wins (rule 2)
    a = "ACGT" * 10
    assert one(a, rc(a), O=8) == (0, 40, 40)
    # equal overlaps on both sides of the plateau: L1 = 40, L2 = 44, s = 40 and s = 44 both overlap 40 positions
    b = rc("ACGT" * 11)
    assert one(a, b, O=8) == (0, 40, 40)                          # rule 3: the smaller s
    both([(a, rc(a)), (a, b)], O=8)


def test_n_against_n_and_lowercase():
    frag = randseq(np.random.default_rng(5), 100)
    withn = frag[:40] + "N" + frag[41:]
    assert one(withn, rc(withn)) == (1, 100, 100)                # N against N: a mismatch
    low = frag.lower()
    assert one(low, rc(frag)) == (0, 100, 100) and one(frag, rc(frag).lower()) == (0, 100, 100)
    iupac = frag[:10] + "R" + frag[11:]
    assert one(iupac, rc(iupac)) == (1, 100, 100)
    both([(withn, rc(withn)), (low, rc(frag)), (iupac, rc(iupac)), ("N" * 50, "N" * 50)])


def test_mate_shorter_than_min_overlap_and_uneven_mates():
    rng = np.random.default_rng(6)
    frag = randseq(rng, 300)
    got = both([(frag[:29], rc(frag)[:150]), (frag[:150], rc(frag)[:29]), (frag[:150], rc(frag)[:30]), (frag[:250], rc(frag)[:90])])
    assert got["too_short"] == 2
    assert one(frag[:250], rc(frag)[:90]) == (0, 40, 300)              # b covers [210, 300) of the fragment
    assert one(frag[:150], rc(frag)[:30]) is None                 # the mates do not overlap: 300 > 150 + 30 - 30


def test_numpy_restatement_matches_scalar_on_random_pairs():
    rng = np.random.default_rng(7)
    pairs = []
    for _ in range(300):
        f = int(rng.integers(20, 260))
        frag = randseq(rng, f, "ACGTNacgt")
        L1, L2 = int(rng.integers(1, 130)), int(rng.integers(1, 130))
        r1 = (frag + randseq(rng, 200))[:L1]
        r2 = (rc(frag) + randseq(rng, 200))[:L2]
        r2 = "".join(c if rng.random() > 0.02 else "A" for c in r2)
        pairs.append((r1, r2))
    for prm in ((30, 5, 20), (5, 3, 50), (12, 0, 0), (1, 100, 100)):
        both(pairs, *prm)


def test_numpy_restatement_on_crlf_and_lone_cr():
    frag = randseq(np.random.default_rng(8), 120)
    r1 = _fq([frag[:100], frag[:60] + "\r" + frag[61:100]], "\r\n")
    r2q = [rc(frag)[:100], rc(frag)[:100]]
    r2 = _fq(r2q, "\r\n")
    got = restate(r1, r2)
    want = scalar_restate([(frag[:100].encode(), r2q[0].encode()), (frag[:60].encode(), r2q[1].encode())])
    assert_same(got, want)


# ---- CPU: the command line's refusals (they come before any device is touched) ----------------------------------------
cli = pytest.mark.skipif(not os.path.exists(CLI), reason="CLI not built")


def _cli(args):
    return subprocess.run([CLI] + args, stdout=subprocess.PIPE, stderr=subprocess.PIPE, timeout=60)


@cli
def test_cli_usage_lists_the_flags():
    err = _cli([]).stderr
    for flag in (b"--insert_size", b"--insert_min_overlap", b"--insert_diff_limit", b"--insert_diff_pct"):
        assert flag in err


@cli
@pytest.mark.parametrize("args, message", [
    (["-u", "X", "--insert_size"], b"--insert_size needs paired reads"),
    (["-1", "X", "-2", "Y", "--insert_min_overlap", "0"], b"--insert_min_overlap as an integer >= 1"),
    (["-1", "X", "-2", "Y", "--insert_diff_pct", "101"], b"in the range 0 <= percent <= 100"),
    (["-1", "X", "-2", "Y", "--insert_diff_limit", "-1"], b"--insert_diff_limit as an integer >= 0"),
    (["-1", "X", "-2", "Y", "--insert_min_overlap", "3x"], b"--insert_min_overlap as an integer >= 1"),
    (["-1", "X", "--insert_size"], b"Please specify a read one file (-2 <file>)"),           # the reference's check comes first
    (["-1", "X", "-2", "Y", "--insert_size", "--lc", "2"], b"low complexity cutoff"),
], ids=["unpaired_only", "min_overlap_0", "pct_101", "limit_negative", "not_a_number", "reference_first", "reference_lc_first"])
def test_cli_refusals(args, message):
    p = _cli(args + ["-d", tempfile.gettempdir()])
    assert p.returncode != 0
    assert message in p.stderr, p.stderr.decode(errors="replace")[-400:]


# ---- GPU: the library ------------------------------------------------------------------------------------------------
def run_ovl(r1, r2, opt, size, n_ctx=1, order=None, deal=None, mode="host", params=DEFAULT):
    """One pass through the API: batches of `size` records, permuted by `order`, dealt to n_ctx contexts on device 0
    (deal(j) picks the context of the j-th batch; default round robin).  Returns every context's overlap_results()."""
    r1, r2 = _as_u8(r1), _as_u8(r2)
    todo = cut(r1, r2, size)
    if order is not None:
        todo = [todo[i] for i in order(len(todo))]
    engines = [Engine(opt) for _ in range(n_ctx)]
    try:
        for e in engines:
            if mode == "pieces":
                e.set_output_pieces(True)
            e.overlap_enable(*params)
        for c in range(n_ctx):
            mine = [b for j, b in enumerate(todo) if (deal(j) if deal else j % n_ctx) == c]
            if mine:
                run_batches(engines[c], mine, mode)
        if n_ctx == 1:
            engines[0].overlap_end_pass()
        else:
            dist_stats.overlap_end_pass_local(engines)
        return [e.overlap_results() for e in engines]
    finally:
        for e in engines:
            e.close()


def long_mates(n, L1, L2, seed):
    """Fragments around the mates' length, so that long overlaps are found; some too long to overlap."""
    rng = np.random.default_rng(seed)
    r1, r2 = [], []
    for _ in range(n):
        f = int(rng.integers(max(L1, L2) // 2, L1 + L2 + 50))
        frag = randseq(rng, f + 100)
        a = (frag[:f] + randseq(rng, L1))[:L1]
        b = (rc(frag[:f]) + randseq(rng, L2))[:L2]
        b = "".join(c if rng.random() > 0.003 else "N" for c in b)
        r1.append(a)
        r2.append(b)
    return _fq(r1), _fq(r2)


WORKLOADS = {
    "fragments": lambda: synth.fragments(60000),
    "c2": lambda: synth.c2(30000),
    "c3": lambda: synth.c3(30000),
    "shotgun": lambda: synth.shotgun(40000),
}


@pytest.mark.gpu
@pytest.mark.parametrize("name", list(WORKLOADS))
def test_matches_restatement(name):
    w = WORKLOADS[name]()
    want = restate(w.r1, w.r2)
    if name == "fragments":
        assert want["overlapped"] > 0.75 * want["pairs"] and want["r1_adapter"] > 0.1 * want["pairs"] and want["mismatch_bases"] > 0
    for k, size in enumerate([1000, 7777, 1 << 20]):
        assert_same(run_ovl(w.r1, w.r2, Options(input_quality_offset=33), size, order=shuffled(k))[0], want)


@pytest.mark.gpu
@pytest.mark.parametrize("seed", [1, 2])
def test_fuzz_inputs_with_cr(seed):
    r1, r2 = fuzz_workload(seed, True)
    for params in (DEFAULT, (5, 3, 50)):
        want = restate(r1, r2, *params)
        assert want["overlapped"] > 0 or params == DEFAULT
        assert_same(run_ovl(r1, r2, Options(input_quality_offset=33), 5000, order=shuffled(seed), params=params)[0], want)


@pytest.mark.gpu
@pytest.mark.parametrize("L1, L2, n", [(600, 450, 400), (2100, 2000, 60), (9000, 7000, 6)], ids=["600", "2000", "9000"])
def test_long_mates(L1, L2, n):
    """600 and 2000+ bases keep the planes in shared memory; 9000 bases put them in global memory."""
    r1, r2 = long_mates(n, L1, L2, seed=L1)
    for params in (DEFAULT, (30, 40, 5)):
        want = restate(r1, r2, *params)
        assert want["overlapped"] > 0
        assert_same(run_ovl(r1, r2, Options(input_quality_offset=33), max(1, n // 3), order=shuffled(3), params=params)[0], want)


@pytest.mark.gpu
def test_counts_do_not_depend_on_options():
    w = synth.c3(20000)
    f = synth.fragments(20000, seed=5)
    r1, r2 = np.concatenate([w.r1, f.r1]), np.concatenate([w.r2, f.r2])
    want = restate(r1, r2)
    adapters = list(BUILTIN_ADAPTERS) + [POLYA_ADAPTER] + list(w.artifacts)
    for opt in (Options(input_quality_offset=33, qc_only=True), Options(input_quality_offset=33, mode=MODE_HARD, quality=20),
                Options(input_quality_offset=33, filter_adapter=True, adapters=adapters, discard_output=True)):
        assert_same(run_ovl(r1, r2, opt, 6000)[0], want)


@pytest.mark.gpu
def test_outputs_and_stats_unchanged_by_the_profile():
    from parity import assert_engines_equal, run_engine
    f = synth.fragments(30000, seed=6)
    opt = Options(input_quality_offset=33, discard_output=True)
    with Engine(opt) as off, Engine(opt) as on:
        on.overlap_enable()
        streams_off, _ = run_engine(off, f.r1, f.r2, 7000)
        streams_on, _ = run_engine(on, f.r1, f.r2, 7000)
        assert_engines_equal(streams_off, off.stats(), streams_on, on.stats())
        on.overlap_end_pass()
        assert on.overlap_results()["pairs"] == 30000


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["pieces", "pipelined", "device"])
def test_batch_paths_match_process_host(mode):
    w = synth.fragments(40000, seed=7)
    want = run_ovl(w.r1, w.r2, Options(input_quality_offset=33), 9000)[0]
    assert_same(want, restate(w.r1, w.r2))
    assert_same(run_ovl(w.r1, w.r2, Options(input_quality_offset=33), 9000, mode=mode)[0], want)


@pytest.mark.gpu
@pytest.mark.parametrize("n_ctx", [2, 3])
def test_several_contexts_on_one_device(n_ctx):
    w = synth.fragments(50000, seed=8)
    want = restate(w.r1, w.r2)
    for deal in (None, lambda j: 0 if j % 4 else 1):            # round robin; uneven (the last context may get nothing)
        for got in run_ovl(w.r1, w.r2, Options(input_quality_offset=33), 6000, n_ctx=n_ctx, order=shuffled(5), deal=deal):
            assert_same(got, want)


@pytest.mark.gpu
def test_single_end_batches_are_not_counted_and_passes_are_separate():
    f = synth.fragments(5000, seed=9)
    with Engine(Options(input_quality_offset=33)) as e:
        e.overlap_enable()
        e.overlap_end_pass()
        got = e.overlap_results()
        assert got["pairs"] == 0 and got["insert_hist"].size == 0 and got["r1_overlap"].size == 0
        e.process(f.r1, f.r2)
        e.process(f.r1)                                          # single-end: neither counted nor refused
        e.overlap_end_pass()
        assert_same(e.overlap_results(), restate(f.r1, f.r2))
        g = synth.fragments(3000, seed=10)
        e.process(g.r1, g.r2)
        e.overlap_end_pass()
        assert_same(e.overlap_results(), restate(g.r1, g.r2))


@pytest.mark.gpu
def test_refusals():
    f = synth.fragments(100, seed=11)
    opt = Options(input_quality_offset=33)
    with Engine(opt) as a, Engine(opt) as b:
        assert _status(a.overlap_end_pass) == FQ_ERR_STATE
        assert _status(a.overlap_results) == FQ_ERR_STATE
        assert _status(lambda: dist_stats.overlap_end_pass_local([a, b])) == FQ_ERR_STATE
        assert _status(lambda: a.overlap_enable(0, 5, 20)) == FQ_ERR_ARG
        assert _status(lambda: a.overlap_enable(30, 5, 101)) == FQ_ERR_ARG
        a.overlap_enable()
        a.process(f.r1, f.r2)
        assert _status(lambda: a.overlap_enable()) == FQ_ERR_STATE                       # in the middle of a pass
        assert _status(lambda: dist_stats.overlap_end_pass_local([a, b])) == FQ_ERR_ARG  # enabled on one context only
        b.overlap_enable(31, 5, 20)
        assert _status(lambda: dist_stats.overlap_end_pass_local([a, b])) == FQ_ERR_ARG  # different parameters
        b.overlap_enable(30, 5, 20)                                                      # no pass under way on b yet
        dist_stats.overlap_end_pass_local([a, b])
        assert_same(b.overlap_results(), restate(f.r1, f.r2))
        a.overlap_enable(20, 2, 10)                                                      # between passes
        a.process(f.r1, f.r2)
        a.overlap_end_pass()
        assert_same(a.overlap_results(), restate(f.r1, f.r2, 20, 2, 10))


# ---- the command line --------------------------------------------------------------------------------------------------
def parse_insert_file(txt):
    out, ins, rows, section = {}, {}, [], None
    for ln in txt.decode().splitlines():
        f = ln.split("\t")
        if ln.startswith("#"):
            section = f[0]
            continue
        if section is None:
            out[f[0]] = int(f[1])
        elif section == "#insert_size":
            ins[int(f[0])] = int(f[1])
        else:
            rows.append([int(v) for v in f])
    out["insert_hist"] = np.zeros(max(ins) + 1 if ins else 0, np.uint64)
    for s, v in ins.items():
        out["insert_hist"][s] = v
    rows = np.array(rows, np.uint64).reshape(-1, 5)
    assert rows[:, 0].tolist() == list(range(1, rows.shape[0] + 1))
    for j, k in enumerate(OVERLAP_CYCLE_ARRAYS):
        out[k] = rows[:, j + 1]
    assert list(out)[:7] == list(OVERLAP_SCALARS)
    return out


def run_cli(files, flags):
    tmp = tempfile.mkdtemp(prefix="faqcs_ins_")
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
def test_cli_insert_size_file_and_other_files_unchanged():
    w = synth.fragments(60000, seed=12)
    u = synth.shotgun(20000, seed=78, paired=False, L=100)
    files = {"-1": ("r1.fq.gz", w.r1), "-2": ("r2.fq.gz", w.r2), "-u": ("u.fq.gz", u.r1)}
    flags = ["--batch_mb", "4", "--devices", "0,0", "--debug", "--discard"]
    without = run_cli(files, flags)
    with_flag = run_cli(files, flags + ["--insert_size"])
    assert_same(parse_insert_file(with_flag.pop("QC.insert_size.txt")), restate(w.r1, w.r2))
    assert "QC.insert_size.txt" not in without
    assert sorted(without) == sorted(with_flag)
    for name in without:
        assert without[name] == with_flag[name], name
    got = parse_insert_file(run_cli(files, flags + ["--insert_size", "--insert_min_overlap", "12", "--insert_diff_limit", "3",
                                                    "--insert_diff_pct", "10"])["QC.insert_size.txt"])
    assert_same(got, restate(w.r1, w.r2, 12, 3, 10))


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
    w = synth.fragments(40000, seed=13)
    want = restate(w.r1, w.r2)
    todo = cut(_as_u8(w.r1), _as_u8(w.r2), 7000)
    engines = [Engine(Options(input_quality_offset=33), device=d) for d in (0, 1)]
    try:
        for e in engines:
            e.overlap_enable()
        for j, (first, final, a1, a2) in enumerate(todo):
            engines[j % 2].process(a1, a2, first, final)
        dist_stats.overlap_end_pass_local(engines)
        for e in engines:
            assert_same(e.overlap_results(), want)
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
    w = synth.fragments(40000, seed=13)
    todo = cut(_as_u8(w.r1), _as_u8(w.r2), 7000 if rank else 3000)      # the ranks see different mate lengths first
    with Engine(Options(input_quality_offset=33), device=rank) as eng:
        eng.overlap_enable()
        for j, (first, final, a1, a2) in enumerate(todo):
            if j % world == rank:
                eng.process(a1, a2, first, final)
        dist_stats.overlap_end_pass_ranks(eng, dist, dev)
        got = eng.overlap_results()
    q.put((rank, {k: (v.tolist() if isinstance(v, np.ndarray) else v) for k, v in got.items()}))
    dist.barrier()
    dist.destroy_process_group()


@pytest.mark.gpu
@multi_gpu
def test_one_process_per_gpu_over_nccl():
    """Rank 0 runs the even batches of 3000 pairs, rank 1 the odd batches of 7000: together not the whole input, so the
    expected result is the restatement of exactly those batches."""
    import socket
    import torch.multiprocessing as mp
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    w = synth.fragments(40000, seed=13)
    parts = [b for j, b in enumerate(cut(_as_u8(w.r1), _as_u8(w.r2), 3000)) if j % 2 == 0]
    parts += [b for j, b in enumerate(cut(_as_u8(w.r1), _as_u8(w.r2), 7000)) if j % 2 == 1]
    want = restate(np.concatenate([p[2] for p in parts]), np.concatenate([p[3] for p in parts]))
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
        assert_same({k: (np.array(v, np.uint64) if isinstance(v, list) else v) for k, v in res.items()}, want)
