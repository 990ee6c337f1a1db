"""Seeded synthetic Illumina-like FASTQ for the BASELINE.json workloads
(SURVEY.md section 8(d), labels C2-C5).  Pure numpy, vectorised, so that a
million-pair block is generated in seconds.

Generator constraints that the reference would otherwise abort on
(BASELINE.md section 3): Q <= 41 (fastq.h:15,31-33); a quality char < 59
(ASCII-33 sets) or > 74 (ASCII-64 set) within the first 32768 reads
(trim.cpp:599-617); headers do not start with ``@NS`` (trim.cpp:619-626);
R1/R2 ids equal up to the first space (trim.cpp:188-222); LF line endings,
bare ``+`` line, final newline, no blank lines (fastq.cpp:34-66).
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import List, Optional, Tuple

import numpy as np

from .api import BUILTIN_ADAPTERS

SEEDS = {"C2": 20261017, "C3": 20261018, "C4": 20261019, "C5": 5}
_BASES = np.frombuffer(b"ACGT", dtype=np.uint8)


@dataclass
class Workload:
    """A named workload: reads plus the FaQCs flags it is meant to be run with."""
    name: str
    r1: np.ndarray                      # uint8 FASTQ bytes
    r2: Optional[np.ndarray]            # None for single-end
    cli_flags: List[str]                # reference command-line flags (without -1/-2/-u/-d)
    artifacts: Optional[List[Tuple[str, str]]] = None   # extra adapters (--artifactFile contents)


def _headers(n: int, tag: str, mate: int, start: int = 0) -> np.ndarray:
    """Fixed-width 34-byte headers '@SYN:<tag>:1:TTTT:XXXXX:YYYYY <mate>:N:0:1'."""
    idx = np.arange(start, start + n, dtype=np.int64)
    tile = (idx // 100000) % 10000
    x = (idx * 7919 + 13) % 100000
    y = idx % 100000
    prefix = f"@SYN:{tag}:1:".encode()
    suffix = f" {mate}:N:0:1".encode()
    w = len(prefix) + 4 + 1 + 5 + 1 + 5 + len(suffix)
    h = np.empty((n, w), dtype=np.uint8)
    c = 0
    h[:, c:c + len(prefix)] = np.frombuffer(prefix, dtype=np.uint8); c += len(prefix)

    def digits(v, k):
        out = np.empty((n, k), dtype=np.uint8)
        for d in range(k):
            out[:, k - 1 - d] = 48 + (v // (10 ** d)) % 10
        return out

    h[:, c:c + 4] = digits(tile, 4); c += 4
    h[:, c] = ord(":"); c += 1
    h[:, c:c + 5] = digits(x, 5); c += 5
    h[:, c] = ord(":"); c += 1
    h[:, c:c + 5] = digits(y, 5); c += 5
    h[:, c:c + len(suffix)] = np.frombuffer(suffix, dtype=np.uint8)
    return h


def _qualities(rng, n, L, base_lo, base_hi, slope_hi, sigma, qmin, qmax, tail_frac, tail_max):
    base = rng.integers(base_lo, base_hi + 1, size=(n, 1)).astype(np.float32)
    slope = rng.uniform(0.0, slope_hi, size=(n, 1)).astype(np.float32)
    pos = np.arange(L, dtype=np.float32)[None, :]
    q = base - slope * pos + rng.normal(0.0, sigma, size=(n, L)).astype(np.float32)
    q = np.clip(np.rint(q), qmin, qmax).astype(np.uint8)
    if tail_frac > 0:
        has_tail = rng.random(n) < tail_frac
        tail_len = rng.integers(1, tail_max + 1, size=n)
        tail_len = np.where(has_tail, tail_len, 0)
        cut = (L - tail_len)[:, None]
        q = np.where(np.arange(L)[None, :] >= cut, np.uint8(2), q)
    return q


def _bases(rng, n, L, p_n, lowcomp_frac):
    s = _BASES[rng.integers(0, 4, size=(n, L))]
    if p_n > 0:
        s = np.where(rng.random((n, L)) < p_n, np.uint8(ord("N")), s)
    if lowcomp_frac > 0:
        lc = np.flatnonzero(rng.random(n) < lowcomp_frac)
        kind = rng.integers(0, 3, size=lc.size)
        for i, k in zip(lc, kind):
            if k == 0:                                    # poly-G (NextSeq style)
                s[i, :] = ord("G")
            elif k == 1:                                  # dinucleotide repeat
                a, b = rng.choice(4, size=2, replace=False)
                s[i, 0::2] = _BASES[a]
                s[i, 1::2] = _BASES[b]
            else:                                         # 90 % mono + noise
                s[i, :] = np.where(rng.random(L) < 0.9, _BASES[rng.integers(0, 4)], s[i, :])
    return s


def _assemble(hdr: np.ndarray, seq: np.ndarray, qual_chars: np.ndarray, lengths: Optional[np.ndarray] = None) -> np.ndarray:
    """Lay records out as header LF seq LF + LF qual LF; ragged lengths via a keep-mask."""
    n, hw = hdr.shape
    L = seq.shape[1]
    w = hw + 1 + L + 1 + 2 + L + 1
    rec = np.empty((n, w), dtype=np.uint8)
    c = 0
    rec[:, c:c + hw] = hdr; c += hw
    rec[:, c] = 10; c += 1
    s0 = c
    rec[:, c:c + L] = seq; c += L
    rec[:, c] = 10; c += 1
    rec[:, c] = ord("+"); c += 1
    rec[:, c] = 10; c += 1
    q0 = c
    rec[:, c:c + L] = qual_chars; c += L
    rec[:, c] = 10
    if lengths is None:
        return rec.reshape(-1)
    keep = np.ones((n, w), dtype=bool)
    col = np.arange(L)[None, :]
    drop = col >= lengths[:, None]
    keep[:, s0:s0 + L] = ~drop
    keep[:, q0:q0 + L] = ~drop
    return rec[keep]


def _mutate(rng, s: np.ndarray, k: int) -> np.ndarray:
    s = s.copy()
    if k and s.size:
        for p in rng.integers(0, s.size, size=k):
            s[p] = _BASES[rng.integers(0, 4)]
    return s


def make_primers(seed: int = SEEDS["C3"], n: int = 64) -> List[Tuple[str, str]]:
    rng = np.random.default_rng(seed ^ 0x5EED)
    out = []
    for i in range(n):
        L = int(rng.integers(20, 31))
        out.append((f"P{i:02d}", _BASES[rng.integers(0, 4, size=L)].tobytes().decode()))
    return out


def _inject_adapters(rng, s: np.ndarray, primers: List[Tuple[str, str]], mate: int):
    n, L = s.shape
    nextera = np.frombuffer(dict(BUILTIN_ADAPTERS)[f"Nextera-primer-adapter-{mate}"].encode(), dtype=np.uint8)
    r = rng.random(n)
    short = np.flatnonzero(r < 0.05)
    for i in short:                      # short insert: 3' end runs into the Nextera adapter
        k = int(rng.integers(20, L - 10))
        ad = _mutate(rng, nextera, int(rng.integers(0, 4)))
        m = min(L - k, ad.size)
        s[i, k:k + m] = ad[:m]
    polya = np.flatnonzero((r >= 0.05) & (r < 0.06))
    for i in polya:
        k = int(rng.integers(18, 41))
        s[i, L - k:] = ord("A")
    prim = np.flatnonzero((r >= 0.06) & (r < 0.08))
    for i in prim:
        p = np.frombuffer(primers[int(rng.integers(0, len(primers)))][1].encode(), dtype=np.uint8)
        s[i, :p.size] = p


def c2(n_pairs: int, seed: int = SEEDS["C2"], start: int = 0, L: int = 150) -> Workload:
    """configs[1]: 2x150 PE, ASCII-33, default trim + filters + full stats (other L: the same recipe at another read length)."""
    rng = np.random.default_rng(seed + start)
    mates = []
    for mate in (1, 2):
        q = _qualities(rng, n_pairs, L, 30, 40, 0.12, 3.0, 2, 41, 0.10, 59)
        s = _bases(rng, n_pairs, L, 0.002, 0.01)
        mates.append(_assemble(_headers(n_pairs, "C2", mate, start), s, q + 33))
    return Workload("C2", mates[0], mates[1], [])


def c3(n_pairs: int, seed: int = SEEDS["C3"], start: int = 0) -> Workload:
    """configs[2]: C2-style reads + adapters / poly-A / 64 primers (seq_overlap path)."""
    rng = np.random.default_rng(seed + start)
    L = 150
    primers = make_primers(seed)
    mates = []
    for mate in (1, 2):
        q = _qualities(rng, n_pairs, L, 30, 40, 0.12, 3.0, 2, 41, 0.10, 59)
        s = _bases(rng, n_pairs, L, 0.002, 0.01)
        _inject_adapters(rng, s, primers, mate)
        mates.append(_assemble(_headers(n_pairs, "C3", mate, start), s, q + 33))
    return Workload("C3", mates[0], mates[1], ["--adapter", "--rate", "0.2", "--polyA"], artifacts=primers)


def c4(n_reads: int, seed: int = SEEDS["C4"], start: int = 0) -> Workload:
    """configs[3]: --qc_only statistics pass over 1x100 SE reads."""
    rng = np.random.default_rng(seed + start)
    L = 100
    q = _qualities(rng, n_reads, L, 30, 40, 0.12, 3.0, 2, 41, 0.0, 0)
    s = _bases(rng, n_reads, L, 0.002, 0.01)
    return Workload("C4", _assemble(_headers(n_reads, "C4", 1, start), s, q + 33), None, ["--qc_only"])


def c5(n_reads: int, seed: int = SEEDS["C5"], start: int = 0) -> Workload:
    """configs[4]: mixed 50-300 bp SE, ASCII-64 autodetect, HARD -q 20 --avg_q 25 --replace_to_N_q 10 --discard."""
    rng = np.random.default_rng(seed + start)
    Lmax = 300
    lengths = rng.integers(50, Lmax + 1, size=n_reads)
    q = _qualities(rng, n_reads, Lmax, 22, 40, 0.08, 4.0, 0, 41, 0.0, 0)
    s = _bases(rng, n_reads, Lmax, 0.003, 0.01)
    if n_reads:
        q[0, 0] = 40          # 'h' (104) > 74 right away so autodetect says 64
    return Workload("C5", _assemble(_headers(n_reads, "C5", 1, start), s, q + 64, lengths), None,
                    ["--mode", "HARD", "-q", "20", "--avg_q", "25", "--replace_to_N_q", "10", "--discard"])


def shotgun(n_pairs: int, genome_len: int = 60000, seed: int = 77, start: int = 0, paired: bool = True, L: int = 150) -> Workload:
    """Reads drawn from a small random genome (both strands, 0.5 % substitutions, a few N): the workload of
    --kmer_rarefaction, where k-mers must repeat for the curve and the frequency histogram to mean anything."""
    g = _BASES[np.random.default_rng(seed).integers(0, 4, size=genome_len + 2 * L)]
    comp = np.zeros(256, dtype=np.uint8)
    comp[list(b"ACGTN")] = list(b"TGCAN")
    rng = np.random.default_rng(seed + 1 + start)
    mates = []
    pos = rng.integers(0, genome_len, size=n_pairs)
    for mate in (1, 2) if paired else (1,):
        off = pos if mate == 1 else (pos + rng.integers(0, L, size=n_pairs)) % genome_len
        s = g[off[:, None] + np.arange(L)[None, :]]
        rev = rng.random(n_pairs) < 0.5
        s = np.where(rev[:, None], comp[s][:, ::-1], s)
        err = rng.random((n_pairs, L)) < 0.005
        s = np.where(err, _BASES[rng.integers(0, 4, size=(n_pairs, L))], s)
        s = np.where(rng.random((n_pairs, L)) < 0.001, np.uint8(ord("N")), s)
        lower = rng.random(n_pairs) < 0.01                 # soft-masked reads: update_kmer folds case (trim.cpp:903-918)
        s = np.where(lower[:, None], s | 0x20, s)
        q = _qualities(rng, n_pairs, L, 30, 40, 0.12, 3.0, 2, 41, 0.10, 59)
        mates.append(_assemble(_headers(n_pairs, "SG", mate, start), s, q + 33))
    return Workload("shotgun", mates[0], mates[1] if paired else None, ["--kmer_rarefaction"])


def fragments(n_pairs: int, seed: int = 91, start: int = 0, L: int = 150, mean: float = 200.0, sd: float = 50.0) -> Workload:
    """Paired reads sequenced from both ends of fragments, the workload of --insert_size: R1 is the fragment's start, R2 the
    reverse complement of its end.  Insert sizes: 70 % normal(mean, sd), 15 % shorter than the read (both mates run into
    their Nextera adapter, then random bases), 10 % between L and 2L, 5 % too long for the mates to overlap.  Then 0.5 %
    substitutions and 0.2 % N per mate, 2 % lowercase mates, and 5 % of the pairs with one mate cut to 1..L bases."""
    rng = np.random.default_rng(seed + start)
    kind = rng.random(n_pairs)
    f = np.rint(rng.normal(mean, sd, size=n_pairs)).astype(np.int64)
    f = np.where(kind >= 0.70, rng.integers(10, L, size=n_pairs), f)
    f = np.where(kind >= 0.85, rng.integers(L, 2 * L, size=n_pairs), f)
    f = np.where(kind >= 0.95, rng.integers(2 * L, 3 * L, size=n_pairs), f)
    f = np.clip(f, 10, 3 * L)
    W = 3 * L
    frag = _BASES[rng.integers(0, 4, size=(n_pairs, W))]
    comp = np.zeros(256, dtype=np.uint8)
    comp[list(b"ACGT")] = list(b"TGCA")
    col = np.arange(L)[None, :]
    rows = np.arange(n_pairs)[:, None]
    mates = []
    for mate in (1, 2):
        ad = np.frombuffer(dict(BUILTIN_ADAPTERS)[f"Nextera-primer-adapter-{mate}"].encode(), dtype=np.uint8)
        tail = np.concatenate([np.broadcast_to(ad, (n_pairs, ad.size)), _BASES[rng.integers(0, 4, size=(n_pairs, L))]], 1)
        inside = col < f[:, None]
        if mate == 1:
            body = frag[rows, np.minimum(col, W - 1)]
        else:
            body = comp[frag[rows, np.clip(f[:, None] - 1 - col, 0, W - 1)]]
        s = np.where(inside, body, tail[rows, np.clip(col - f[:, None], 0, tail.shape[1] - 1)])
        s = np.where(rng.random((n_pairs, L)) < 0.005, _BASES[rng.integers(0, 4, size=(n_pairs, L))], s)
        s = np.where(rng.random((n_pairs, L)) < 0.002, np.uint8(ord("N")), s)
        s = np.where((rng.random(n_pairs) < 0.02)[:, None], s | 0x20, s)
        lengths = np.where((rng.random(n_pairs) < 0.025), rng.integers(1, L + 1, size=n_pairs), L)
        q = _qualities(rng, n_pairs, L, 30, 40, 0.12, 3.0, 2, 41, 0.10, 59)
        mates.append(_assemble(_headers(n_pairs, "FR", mate, start), s, q + 33, lengths))
    return Workload("fragments", mates[0], mates[1], [])


def phix174() -> str:
    """The PhiX174 genome the command-line driver carries (faqcs_b200/host/phix174.inc)."""
    import os
    import re
    txt = open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "host", "phix174.inc")).read()
    return "".join(re.findall(r'"([^"]*)"', txt))


TRUSEQ_FRAGMENT = dict(BUILTIN_ADAPTERS)["TruSeq-adapter-1"][:60]


def overrepresented(n_pairs: int, plants=None, seed: int = 93, start: int = 0, paired: bool = True, L: int = 150) -> Workload:
    """C2-like reads with planted sequences, the workload of --overrep.  A plant is (sequence, copies, mate, whole): `copies`
    reads of `mate` (1, 2, or 0 for both mates of the same pairs) start with `sequence`; with whole=True the read is exactly
    the sequence (a read shorter than the prefix when the sequence is), otherwise the rest of the read stays random (reads
    equal in their first len(sequence) bases only).  Plants take disjoint reads of a mate.  The default plants a 60-base
    TruSeq-adapter fragment in 2 % of both mates, a 150-base PhiX fragment in 1 % of R1 and a 30-base primer dimer read in
    0.5 % of R1."""
    if plants is None:
        plants = [(TRUSEQ_FRAGMENT, n_pairs // 50, 0, False), (phix174()[1000:1000 + L], n_pairs // 100, 1, True),
                  ("ACACTCTTTCCCTACACGACGCTCTTCCGA", n_pairs // 200, 1, True)]
    rng = np.random.default_rng(seed + start)
    mates = []
    rows_both = {}
    for mate in (1, 2) if paired else (1,):
        q = _qualities(rng, n_pairs, L, 30, 40, 0.12, 3.0, 2, 41, 0.10, 59)
        s = _bases(rng, n_pairs, L, 0.002, 0.01)
        lengths = np.full(n_pairs, L, dtype=np.int64)
        free = np.ones(n_pairs, dtype=bool)
        for k, (seq, copies, pm, whole) in enumerate(plants):
            if pm not in (0, mate):
                continue
            b = np.frombuffer(seq.encode(), dtype=np.uint8)
            assert b.size <= L, "a plant longer than the reads"
            if pm == 0 and k in rows_both:
                rows = rows_both[k]
            else:
                rows = rng.choice(np.flatnonzero(free), size=copies, replace=False)
                rows_both[k] = rows
            assert free[rows].all(), "plants overlap"
            free[rows] = False
            s[rows, :b.size] = b
            if whole:
                lengths[rows] = b.size
        mates.append(_assemble(_headers(n_pairs, "OR", mate, start), s, q + 33, lengths))
    return Workload("overrepresented", mates[0], mates[1] if paired else None, [])


def _digits(v: np.ndarray, k: int) -> np.ndarray:
    out = np.empty((v.size, k), dtype=np.uint8)
    for d in range(k):
        out[:, k - 1 - d] = 48 + (v // (10 ** d)) % 10
    return out


def tile_numbers(tiles_per_lane: int) -> List[int]:
    """Flowcell tile numbers in the NovaSeq style: 1101, 1102, ..., 64 tiles per swath, then the next swath (1201, ...)."""
    return [1101 + 100 * (k // 64) + k % 64 for k in range(tiles_per_lane)]


def tiled(n_pairs: int, lanes: int = 2, tiles_per_lane: int = 16, order: str = "sorted", bad_tiles=None, seed: int = 95,
          paired: bool = True, L: int = 150) -> Workload:
    """C2-like reads under Casava 1.8 names '@B200SIM:1:FC:{lane}:{tile}:{x}:{y} {mate}:N:0:ACGT', the workload of
    --tile_quality.  The pairs are spread evenly over lanes x tiles_per_lane flowcell tiles (tile_numbers(), zero-padded to
    one width when they need more than 4 digits; lanes <= 9), in (lane, tile) order as a sequencer writes them
    (order="sorted") or in random order ("shuffled").  bad_tiles = [(lane, tile, first_cycle, last_cycle, drop)]: the
    scores of cycles first..last (1-based, inclusive) of both mates of that tile's reads drop by `drop` (at least 2 stays).
    Default: one bubble on lane 1's second tile, cycles 50-80, 15 lower."""
    assert 1 <= lanes <= 9 and tiles_per_lane >= 1 and order in ("sorted", "shuffled")
    tnum = np.array(tile_numbers(tiles_per_lane), dtype=np.int64)
    if bad_tiles is None:
        bad_tiles = [(1, int(tnum[1]), 50, 80, 15)] if tiles_per_lane > 1 else []
    rng = np.random.default_rng(seed)
    n_keys = lanes * tiles_per_lane
    key = np.arange(n_pairs, dtype=np.int64) * n_keys // max(n_pairs, 1)
    if order == "shuffled":
        key = key[rng.permutation(n_pairs)]
    lane = 1 + key // tiles_per_lane
    tile = tnum[key % tiles_per_lane]
    x = rng.integers(10000, 100000, size=n_pairs)
    y = rng.integers(10000, 100000, size=n_pairs)
    tw = max(4, len(str(int(tnum.max()))))
    mates = []
    for mate in (1, 2) if paired else (1,):
        q = _qualities(rng, n_pairs, L, 30, 40, 0.12, 3.0, 2, 41, 0.10, 59).astype(np.int16)
        for bl, bt, c0, c1, drop in bad_tiles:
            rows = np.flatnonzero((lane == bl) & (tile == bt))
            q[rows[:, None], np.arange(c0 - 1, min(c1, L))[None, :]] -= drop
        q = np.clip(q, 2, 41).astype(np.uint8)
        s = _bases(rng, n_pairs, L, 0.002, 0.01)
        head = np.frombuffer(b"@B200SIM:1:FC:", dtype=np.uint8)
        tail = np.frombuffer(f" {mate}:N:0:ACGT".encode(), dtype=np.uint8)
        colon = np.full((n_pairs, 1), ord(":"), dtype=np.uint8)
        hdr = np.concatenate([np.broadcast_to(head, (n_pairs, head.size)), _digits(lane, 1), colon, _digits(tile, tw), colon,
                              _digits(x, 5), colon, _digits(y, 5), np.broadcast_to(tail, (n_pairs, tail.size))], 1)
        mates.append(_assemble(np.ascontiguousarray(hdr), s, q + 33))
    return Workload("tiled", mates[0], mates[1] if paired else None, [])


def fastq_bytes(records: List[Tuple[str, str, str]], eol: str = "\n") -> bytes:
    """Hand-written records -> FASTQ bytes (micro-cases)."""
    return "".join(f"{h}{eol}{s}{eol}+{eol}{q}{eol}" for h, s, q in records).encode()


def algorithmic_bytes(r1: np.ndarray, r2: Optional[np.ndarray], out_bytes: List[int]) -> int:
    """SURVEY 8(d): B_in + B_out, summed over the batch."""
    return int(r1.size + (0 if r2 is None else r2.size) + sum(out_bytes))
