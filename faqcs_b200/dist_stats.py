"""Multi-GPU merge of the statistics through the library's own collective (fq_allreduce_stats: one
ncclAllReduce(u64, sum) over NVLink + a max of the row counters; include/faqcs_b200.h), and the end of a k-mer
rarefaction, sequence duplication or overrepresented-sequence pass over a table sharded across contexts (fq_kmer_end_pass_all,
fq_dup_end_pass_all, fq_overrep_end_pass_all), and of an insert-size or per flowcell tile quality pass (fq_overlap_end_pass_all,
fq_tile_qual_end_pass_all).

Two launch shapes, both ending in the same C call:
  * one process per GPU (torchrun): rank 0 draws the NCCL id (fq_comm_unique_id), the launcher's process group
    broadcasts those 128 bytes, every rank joins (fq_comm_init_rank) and calls the library on its one context;
  * one process, several GPUs: fq_comm_init_all over the contexts (statistics) or no communicator at all (k-mer,
    duplication, insert-size, overrepresented-sequence and tile quality passes), one call for all of them.
The reference's counterpart is the `omp critical` merge at the end of trim() (trim.cpp:120-154).
"""
from __future__ import annotations

import ctypes as C
from typing import Sequence

import numpy as np

from .api import Engine, FaqcsError

COMM_ID_BYTES = 128


def _check(eng: Engine, st: int):
    if st != 0:
        raise FaqcsError(st, eng.lib.fq_last_error(eng.ctx).decode(errors="replace"))


def _rank_comm(eng: Engine, dist, dev) -> C.c_void_p:
    """This rank's communicator: rank 0 draws the NCCL id, the launcher's group broadcasts it, every rank joins."""
    import torch
    ident = torch.zeros(COMM_ID_BYTES, dtype=torch.uint8, device=dev)
    if dist.get_rank() == 0:
        buf = (C.c_uint8 * COMM_ID_BYTES)()
        _check(eng, eng.lib.fq_comm_unique_id(buf))
        ident = torch.tensor(list(buf), dtype=torch.uint8, device=dev)
    dist.broadcast(ident, src=0)
    raw = (C.c_uint8 * COMM_ID_BYTES)(*ident.cpu().tolist())
    comm = C.c_void_p()
    _check(eng, eng.lib.fq_comm_init_rank(eng.ctx, dist.get_world_size(), dist.get_rank(), raw, C.byref(comm)))
    return comm


def allreduce_engine_stats(eng: Engine, dist, dev) -> float:
    """One context per process: merge over the ranks of `dist` (torch.distributed).  Returns the device ms of the collective."""
    comm = _rank_comm(eng, dist, dev)
    try:
        ctxs = (C.c_void_p * 1)(eng.ctx)
        comms = (C.c_void_p * 1)(comm)
        _check(eng, eng.lib.fq_allreduce_stats(ctxs, 1, comms))
        return float(eng.lib.fq_last_allreduce_ms(eng.ctx))
    finally:
        eng.lib.fq_comm_destroy(comm)


def allreduce_local_engines(engines: Sequence[Engine]) -> float:
    """One process, one context per device: merge all of them in place.  Returns the device ms seen by the first context."""
    n = len(engines)
    e0 = engines[0]
    ctxs = (C.c_void_p * n)(*[e.ctx for e in engines])
    comms = (C.c_void_p * n)()
    _check(e0, e0.lib.fq_comm_init_all(ctxs, n, comms))
    try:
        _check(e0, e0.lib.fq_allreduce_stats(ctxs, n, comms))
        return float(e0.lib.fq_last_allreduce_ms(e0.ctx))
    finally:
        for c in comms:
            e0.lib.fq_comm_destroy(c)


def kmer_end_pass_local(engines: Sequence[Engine]):
    """End of a k-mer rarefaction pass whose batches ran on these contexts (one process, any devices, a device may repeat):
    the per-context tables are merged, and every engine's kmer_results() returns the whole run's curve and histogram."""
    n = len(engines)
    e0 = engines[0]
    ctxs = (C.c_void_p * n)(*[e.ctx for e in engines])
    _check(e0, e0.lib.fq_kmer_end_pass_all(ctxs, n, None))


def kmer_end_pass_ranks(eng: Engine, dist, dev):
    """The same with one context per process: the tables are merged over the ranks of `dist` (torch.distributed)."""
    comm = _rank_comm(eng, dist, dev)
    try:
        ctxs = (C.c_void_p * 1)(eng.ctx)
        comms = (C.c_void_p * 1)(comm)
        _check(eng, eng.lib.fq_kmer_end_pass_all(ctxs, 1, comms))
    finally:
        eng.lib.fq_comm_destroy(comm)


def dup_end_pass_local(engines: Sequence[Engine]):
    """End of a duplication-statistics pass whose batches ran on these contexts (one process, any devices, a device may
    repeat): the per-context tables are merged, and every engine's dup_results() returns the whole pass's result."""
    n = len(engines)
    e0 = engines[0]
    ctxs = (C.c_void_p * n)(*[e.ctx for e in engines])
    _check(e0, e0.lib.fq_dup_end_pass_all(ctxs, n, None))


def dup_end_pass_ranks(eng: Engine, dist, dev):
    """The same with one context per process: the tables are merged over the ranks of `dist` (torch.distributed)."""
    comm = _rank_comm(eng, dist, dev)
    try:
        ctxs = (C.c_void_p * 1)(eng.ctx)
        comms = (C.c_void_p * 1)(comm)
        _check(eng, eng.lib.fq_dup_end_pass_all(ctxs, 1, comms))
    finally:
        eng.lib.fq_comm_destroy(comm)


def overlap_end_pass_local(engines: Sequence[Engine]):
    """End of an insert-size pass whose batches ran on these contexts (one process, any devices, a device may repeat): the
    accumulators are summed, and every engine's overlap_results() returns the whole pass's result."""
    n = len(engines)
    e0 = engines[0]
    ctxs = (C.c_void_p * n)(*[e.ctx for e in engines])
    _check(e0, e0.lib.fq_overlap_end_pass_all(ctxs, n, None))


def overlap_end_pass_ranks(eng: Engine, dist, dev):
    """The same with one context per process: the accumulators are summed over the ranks of `dist` (torch.distributed)."""
    comm = _rank_comm(eng, dist, dev)
    try:
        ctxs = (C.c_void_p * 1)(eng.ctx)
        comms = (C.c_void_p * 1)(comm)
        _check(eng, eng.lib.fq_overlap_end_pass_all(ctxs, 1, comms))
    finally:
        eng.lib.fq_comm_destroy(comm)


def overrep_end_pass_local(engines: Sequence[Engine]):
    """End of an overrepresented-sequence pass whose batches ran on these contexts (one process, any devices, a device may
    repeat): the count tables are merged, and every engine's overrep_results() returns the whole pass's list."""
    n = len(engines)
    e0 = engines[0]
    ctxs = (C.c_void_p * n)(*[e.ctx for e in engines])
    _check(e0, e0.lib.fq_overrep_end_pass_all(ctxs, n, None))


def overrep_end_pass_ranks(eng: Engine, dist, dev):
    """The same with one context per process: the tables are merged over the ranks of `dist` (torch.distributed)."""
    comm = _rank_comm(eng, dist, dev)
    try:
        ctxs = (C.c_void_p * 1)(eng.ctx)
        comms = (C.c_void_p * 1)(comm)
        _check(eng, eng.lib.fq_overrep_end_pass_all(ctxs, 1, comms))
    finally:
        eng.lib.fq_comm_destroy(comm)


def tile_qual_end_pass_local(engines: Sequence[Engine]):
    """End of a per flowcell tile quality pass whose batches ran on these contexts (one process, any devices, a device may
    repeat): the key lists are united and the counts summed, and every engine's tile_qual_results() returns the whole pass."""
    n = len(engines)
    e0 = engines[0]
    ctxs = (C.c_void_p * n)(*[e.ctx for e in engines])
    _check(e0, e0.lib.fq_tile_qual_end_pass_all(ctxs, n, None))


def tile_qual_end_pass_ranks(eng: Engine, dist, dev):
    """The same with one context per process: keys and counts are merged over the ranks of `dist` (torch.distributed)."""
    comm = _rank_comm(eng, dist, dev)
    try:
        ctxs = (C.c_void_p * 1)(eng.ctx)
        comms = (C.c_void_p * 1)(comm)
        _check(eng, eng.lib.fq_tile_qual_end_pass_all(ctxs, 1, comms))
    finally:
        eng.lib.fq_comm_destroy(comm)
