"""Host-side I/O of the command-line driver without a GPU (SURVEY 8(f) N1 / N2): the batch reader on plain, gzip and blocked
gzip (BGZF) input -- members inflated by several threads straight into the batch buffer, ordinary members after blocked ones
handed to zlib, pipes read through zlib -- the blocked-gzip writer of --gz_out, the mapped and pieces writers, and fork_join.
tests/host_io_harness.cpp includes faqcs_cli.cpp and drives its Source / writers the way the driver does."""
import contextlib
import gzip
import os
import random
import struct
import subprocess
import threading
import zlib

import pytest

from faqcs_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIBDIR = os.path.join(ROOT, "faqcs_b200")


def bgzf_bytes(data: bytes, block: int = 0xff00, level: int = 1, eof_marker: bool = True) -> bytes:
    out = bytearray()
    chunks = [data[i:i + block] for i in range(0, len(data), block)] + ([b""] if eof_marker else [])
    for c in chunks:
        z = zlib.compressobj(level, zlib.DEFLATED, -15)
        payload = z.compress(c) + z.flush()
        out += struct.pack("<4BI2BH2BHH", 0x1f, 0x8b, 8, 4, 0, 0, 0xff, 6, 66, 67, 2, len(payload) + 25)
        out += payload + struct.pack("<II", zlib.crc32(c), len(c))
    return bytes(out)


@contextlib.contextmanager
def fifo(path, feed=None):
    """A FIFO at `path` served by a thread: it writes `feed` into the FIFO, or (feed None) reads what arrives into the list
    it yields."""
    os.mkfifo(path)
    got = []

    def serve():
        try:
            if feed is None:
                with open(path, "rb") as f:
                    got.append(f.read())
            else:
                with open(path, "wb") as f:
                    f.write(feed)
        except BrokenPipeError:
            pass

    t = threading.Thread(target=serve, daemon=True)
    t.start()
    try:
        yield got
    finally:
        try:        # a harness that stopped before opening its end leaves the thread waiting in open(): give it the other end
            os.close(os.open(path, (os.O_WRONLY if feed is None else os.O_RDONLY) | os.O_NONBLOCK))
        except OSError:
            pass
        t.join(timeout=60)


@pytest.fixture(scope="module")
def harness(tmp_path_factory):
    if not os.path.exists(os.path.join(LIBDIR, "libfaqcs_b200.so")):
        pytest.skip("libfaqcs_b200.so not built")
    exe = str(tmp_path_factory.mktemp("hostio") / "host_io_harness")
    subprocess.check_call(["/usr/bin/g++", "-O2", "-std=c++17", "-I" + os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "host_io_harness.cpp"),
                           "-o", exe, "-L" + LIBDIR, "-lfaqcs_b200", "-lz", "-lpthread", "-Wl,-rpath," + LIBDIR])
    return exe


@pytest.fixture(scope="module")
def fastq():
    return bytes(synth.c2(12000).r1)


@pytest.mark.parametrize("shape", ["plain", "gzip", "bgzf", "bgzf_no_eof_member", "bgzf_small_members", "bgzf_then_gzip"])
@pytest.mark.parametrize("buffer_kib", [150, 3000, 100000])
def test_reader_delivers_the_file(harness, fastq, tmp_path, shape, buffer_kib):
    cut = fastq.index(b"\n", len(fastq) // 2) + 1
    data = {"plain": fastq, "gzip": gzip.compress(fastq, 1), "bgzf": bgzf_bytes(fastq), "bgzf_no_eof_member": bgzf_bytes(fastq, eof_marker=False),
            "bgzf_small_members": bgzf_bytes(fastq, block=777),
            "bgzf_then_gzip": bgzf_bytes(fastq[:cut], eof_marker=False) + gzip.compress(fastq[cut:], 1)}[shape]
    src, dst = tmp_path / "in.bin", tmp_path / "out.bin"
    src.write_bytes(data)
    p = subprocess.run([harness, "read", str(src), str(dst), str(buffer_kib)], capture_output=True)
    assert p.returncode == 0, p.stderr.decode()
    assert dst.read_bytes() == fastq
    assert f"lines {fastq.count(10)}".encode() in p.stdout


@pytest.mark.parametrize("shape", ["plain", "gzip", "bgzf"])
def test_reader_on_a_pipe(harness, fastq, tmp_path, shape):
    """A FIFO cannot be read twice: the format is left to zlib, which passes plain text through (the reference's gzopen)."""
    data = {"plain": fastq, "gzip": gzip.compress(fastq, 1), "bgzf": bgzf_bytes(fastq)}[shape]
    src, dst = tmp_path / "in.fifo", tmp_path / "out.bin"
    with fifo(src, feed=data):
        p = subprocess.run([harness, "read", str(src), str(dst), "150"], capture_output=True, timeout=120)
    assert p.returncode == 0, p.stderr.decode()
    assert dst.read_bytes() == fastq
    assert f"lines {fastq.count(10)} mode zlib".encode() in p.stdout


def test_reader_rejects_a_corrupt_member(harness, fastq, tmp_path):
    data = bytearray(bgzf_bytes(fastq))
    data[len(data) // 2] ^= 0x55
    src = tmp_path / "bad.gz"
    src.write_bytes(bytes(data))
    p = subprocess.run([harness, "read", str(src), str(tmp_path / "out.bin"), "100000"], capture_output=True)
    assert p.returncode == 5 and b"Unable to read" in p.stderr


def test_blocked_gzip_writer_round_trips(harness, fastq, tmp_path):
    src, dst = tmp_path / "in.fq", tmp_path / "out.gz"
    src.write_bytes(fastq)
    p = subprocess.run([harness, "write", str(src), str(dst)], capture_output=True)
    assert p.returncode == 0, p.stderr.decode()
    z = dst.read_bytes()
    assert z[:4] == b"\x1f\x8b\x08\x04" and z.endswith(b"\x1b\x00\x03\x00" + b"\x00" * 8)
    assert gzip.decompress(z) == fastq
    back = tmp_path / "back.bin"                      # and through the driver's own parallel reader
    p = subprocess.run([harness, "read", str(dst), str(back), "2048"], capture_output=True)
    assert p.returncode == 0 and back.read_bytes() == fastq


def _pieces(fastq, bad_source=False):
    """(R1, R2, literal bytes, piece list text, the stream the pieces spell): pieces of both mates mixed with literal bytes."""
    rng = random.Random(11)
    bufs = (fastq, fastq[::-1], bytes(rng.randrange(256) for _ in range(20000)))
    lines, want = [], bytearray()
    for _ in range(4000):
        s = rng.randrange(3)
        o = rng.randrange(len(bufs[s]))
        n = rng.randrange(min(len(bufs[s]) - o, 3000) + 1)
        lines.append(f"{s} {o} {n}")
        want += bufs[s][o:o + n]
    if bad_source:
        lines[len(lines) * 3 // 4] = "3 0 10"
    return bufs, "\n".join(lines) + "\n", bytes(want)


@pytest.mark.parametrize("target", ["file", "fifo"])
@pytest.mark.parametrize("writer", ["mapped", "pieces", "pieces_bad_source"])
def test_plain_writers(harness, fastq, tmp_path, writer, target):
    """write_mapped (the byte streams) and write_pieces (pieces mode) append in two calls: into a mapping of a regular file
    (FAQCS_B200_IO_SLICE_MIN=1000 lets write_mapped take it), and with write(2) / writev(2) into a FIFO."""
    dst = tmp_path / ("out.fifo" if target == "fifo" else "out.bin")
    if writer == "mapped":
        (tmp_path / "in.fq").write_bytes(fastq)
        args, want = [str(tmp_path / "in.fq")], fastq
    else:
        bufs, listing, want = _pieces(fastq, bad_source=writer == "pieces_bad_source")
        args = []
        for name, b in zip(("r1", "r2", "lit"), bufs):
            (tmp_path / name).write_bytes(b)
            args.append(str(tmp_path / name))
        (tmp_path / "list.txt").write_text(listing)
        args.append(str(tmp_path / "list.txt"))
    cmd = [harness, writer.replace("_bad_source", "")] + args + [str(dst)]
    env = dict(os.environ, FAQCS_B200_IO_SLICE_MIN="1000")
    with fifo(dst) if target == "fifo" else contextlib.nullcontext([]) as got:
        p = subprocess.run(cmd, capture_output=True, env=env, timeout=120)
    if writer == "pieces_bad_source":
        assert p.returncode == 5 and b"pieces of a stream do not add up to its size" in p.stderr
        return
    assert p.returncode == 0, p.stderr.decode()
    assert (got[0] if target == "fifo" else dst.read_bytes()) == want


@pytest.mark.parametrize("kind", ["str", "bad_alloc"])
@pytest.mark.parametrize("n,k", [(1, 0), (2, 0), (2, 1), (8, 0), (8, 7)])
def test_fork_join_hands_a_job_exception_to_the_caller(harness, n, k, kind):
    """A job that throws (first or last, on a thread or on the caller's) ends up as the I/O worker's error message, after
    every other job has finished, instead of ending the process."""
    p = subprocess.run([harness, "fork_join", str(n), str(k), kind], capture_output=True, timeout=60)
    msg = "job failed" if kind == "str" else "I/O worker failed (std::exception)"
    assert p.returncode == 5, p.stderr.decode()
    assert f"error: {msg} (other jobs finished: {n - 1})".encode() in p.stderr


# ---- ordinary gzip, inflated by several threads (faqcs_b200/host/pgzip.hpp) -----------------------------------------------
@pytest.fixture(scope="module")
def big_fastq():
    return bytes(synth.c2(40000).r1)          # 13.6 MB: its gzip is above the 4 MiB below which the reader stays with zlib


def _shape(d, name):
    """(gzip bytes, what they inflate to) -- only the requested one is built."""
    import numpy as np
    tiny = b"@x\nACGT\n+\nIIII\n"
    if name.startswith("level"):
        return gzip.compress(d, int(name[5:])), d
    if name == "two_members":
        return gzip.compress(d[:6_000_000], 6) + gzip.compress(d[6_000_000:], 1), d
    if name == "member_then_tiny_member":
        return gzip.compress(d, 6) + gzip.compress(tiny, 6), d + tiny
    if name == "trailing_zeros":
        return gzip.compress(d, 6) + b"\0" * 100, d
    if name == "full_flush_inside":
        co = zlib.compressobj(6, zlib.DEFLATED, 31)
        return co.compress(d[:7_000_000]) + co.flush(zlib.Z_FULL_FLUSH) + co.compress(d[7_000_000:]) + co.flush(), d
    if name == "incompressible":                  # stored blocks: nothing to enter, one thread inflates it all
        rnd = np.random.default_rng(1).integers(0, 256, size=6_000_000, dtype=np.uint8).tobytes()
        return gzip.compress(rnd, 6), rnd
    if name == "stored_level0":
        return gzip.compress(d[:8_000_000], 0), d[:8_000_000]
    raise KeyError(name)


@pytest.mark.parametrize("shape", ["level1", "level6", "level9", "two_members", "member_then_tiny_member", "trailing_zeros", "full_flush_inside",
                                   "incompressible", "stored_level0"])
def test_parallel_gzip_reader_delivers_the_file(harness, big_fastq, tmp_path, shape):
    z, want = _shape(big_fastq, shape)
    src, dst = tmp_path / "in.gz", tmp_path / "out.bin"
    src.write_bytes(z)
    for buffer_kib, env in ((3000, {}), (65536, {}), (65536, {"FAQCS_B200_PGZIP": "0"})):
        p = subprocess.run([harness, "read", str(src), str(dst), str(buffer_kib)], capture_output=True, env=dict(os.environ, **env))
        assert p.returncode == 0, p.stderr.decode()
        assert dst.read_bytes() == want
        assert (b"mode zlib" if env else b"mode pgzip") in p.stdout


def test_parallel_gzip_reader_rejects_damage(harness, big_fastq, tmp_path):
    z = bytearray(gzip.compress(big_fastq, 6))
    for where, what in ((len(z) // 2, "a flipped byte in the deflate stream"), (len(z) - 6, "a wrong CRC-32"), (len(z) - 2, "a wrong length")):
        bad = bytearray(z)
        bad[where] ^= 0x41
        src = tmp_path / "bad.gz"
        src.write_bytes(bytes(bad))
        p = subprocess.run([harness, "read", str(src), str(tmp_path / "out.bin"), "65536"], capture_output=True)
        assert p.returncode == 5 and b"Unable to read" in p.stderr, what


def test_parallel_gzip_reader_on_a_truncated_file(harness, big_fastq, tmp_path):
    """A gzip file that is cut short: gzread / gzgets (the reference's reader, fastq.cpp:8-30) hand out everything up to the last
    byte present and then report the end of the file; the parallel reader must deliver exactly the same bytes."""
    z = gzip.compress(big_fastq, 6)
    for cut in (len(z) * 2 // 3, len(z) - 1000, len(z) - 4):
        src = tmp_path / "cut.gz"
        src.write_bytes(z[:cut])
        got = []
        for env in ({}, {"FAQCS_B200_PGZIP": "0"}):
            p = subprocess.run([harness, "read", str(src), str(tmp_path / "out.bin"), "65536"], capture_output=True, env=dict(os.environ, **env))
            assert p.returncode == 0, p.stderr.decode()
            assert (b"mode zlib" if env else b"mode pgzip") in p.stdout
            got.append((tmp_path / "out.bin").read_bytes())
        assert got[0] == got[1] and big_fastq.startswith(got[0]) and len(got[0]) > len(big_fastq) // 2
