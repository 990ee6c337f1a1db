// fq_tile_qual.cuh -- per flowcell tile sequence quality (fq_tile_qual_*, --tile_quality).
//
// ("Flowcell tile" throughout: `tile` alone means an emit chunk in fq_emit.cuh.)
//
// Every framed record counts, whatever trimming, filtering or --qc_only later make of it; the mates of a pair count
// separately (mate m = 1, 2; a single-end batch has mate 1 only).
//
// A read's (lane, flowcell tile).  The name is the header-line bytes after '@' up to the first ' ', '\t', '\r' or '\n'; it is
// split at ':' into n fields f[0..n-1].  n >= 7 (Casava 1.8 / bcl-convert, with or without a UMI field): lane = f[3], tile =
// f[4]; n = 5 or 6 (@inst:lane:tile:x:y#idx/1): lane = f[1], tile = f[2]; otherwise, or when lane or tile is not 1..9 ASCII
// digits, the read is untiled.  Lane and tile compare as values (01101 is 1101); the key is (lane << 32) | tile.
//
// A base's score is max(0, byte - input_quality_offset) on the quality line as framed, before terminal-N masking, with no
// upper clamp.  (A score above 41 fails the batch with FQ_ERR_QUALITY, with or without --qc_only, unless the base lies in a
// leading or trailing run of 'N' that the masking covers; such a base counts here with its score as read.)
//
// Per (flowcell tile, mate): reads, a length histogram over 0..C (lengths above C in bin C; the bases at 0-based cycle c are
// the reads longer than c), the score sum at each cycle 1..C, and the bases and score sum of whole reads.  C = min(longest read
// of the pass, kTileMaxCycles); cycles beyond it count in the whole-read totals only.  Per mate: reads and untiled reads.
//
// Keys.  k_tile_keys parses each header with one thread and gives every tiled read the dense id of its key in a
// per-context open-addressing table of kTileSlots KmerSlots (key, id + 1 in `count`; 0 while the id is being published).  A
// new key needs a ticket before it may claim a slot: tickets counts claims made plus claims under way, and a ticket at or
// above kTileMaxKeys is handed back at once.  So at most kTileMaxKeys slots are ever claimed and the table never fills,
// whatever the input.  A thread whose key is absent while all kTileMaxKeys keys are claimed marks its reads overflowed: the
// context then saw more than kTileMaxKeys distinct keys, so the union over contexts did too.
//
// Accumulation.  k_tile_qual gives each warp a run of consecutive reads of one mate.  Lanes own cycles (lane l: l, l + 32,
// ...) and add scores into the warp's shared-memory row while the dense id stays the same, and lane 0 run-length codes the
// lengths; everything is added to the context's u64 block only when the id changes and at the end of the run.  Real FASTQ
// is written in flowcell tile order, so that is a few atomics per read; shuffled input is as exact, only slower.
#pragma once
#include "fq_kmer.cuh"

namespace fq {

constexpr uint32_t kTileMaxKeys = 16384;          // distinct (lane, flowcell tile) keys of one pass
constexpr uint32_t kTileSlots = 1u << 15;         // key table slots per context
constexpr uint32_t kTileMaxCycles = 1024;
constexpr uint16_t kTileUntiled = 0xffff, kTileOverflowed = 0xfffe;     // per-read ids that are not a dense id
constexpr int kTileKeyThreads = 256, kTileQualThreads = 256;
constexpr uint32_t kRegCycles = 160;              // k_tile_qual: cycles of a read whose quality bytes are loaded at once

// Per-context counters: the host reads {claims, overflow} after every batch, untiled[] at the end of a pass.
struct TileCounters {
    uint32_t claims;                // dense ids handed out
    uint32_t overflow;              // a read's key found no room
    uint32_t tickets;               // claims + claims under way (+ tickets about to be handed back)
    uint32_t pad;
    unsigned long long untiled[2];
};

// The accumulator block, u64, column d = n_mates * id + mate - 1 of D columns (n_mates of the pass), rows: whole-read bases,
// whole-read score sum, the length histogram [C + 1], the score sums of cycles 1..C.
struct TileLayout {
    uint32_t D, C;
    __host__ __device__ size_t rows() const { return 2 + (size_t)(C + 1) + C; }
    __host__ __device__ size_t total() const { return rows() * D; }
    __host__ __device__ size_t bases(uint32_t d) const { return d; }
    __host__ __device__ size_t qual(uint32_t d) const { return (size_t)D + d; }
    __host__ __device__ size_t hist(uint32_t len, uint32_t d) const { return (2 + (size_t)len) * D + d; }
    __host__ __device__ size_t cyc(uint32_t c, uint32_t d) const { return (3 + (size_t)C + c) * D + d; }      // c: 0-based
};

struct TileKeyArgs {
    const uint8_t *raw[2];
    const Rec *rec[2];
    uint32_t n_rec, n_mates;
    KmerTable T;
    TileCounters *cnt;
    uint16_t *id[2];                // [n_rec] per mate
};

struct TileQualArgs {
    const uint8_t *raw[2];
    const Rec *rec[2];
    const uint16_t *id[2];
    uint32_t n_rec, n_mates, run;   // reads per warp
    int32_t in_off;
    TileLayout L;
    unsigned long long *acc;
};

// A field being read: its value, its length and whether every byte so far is a digit.
struct TileField {
    uint32_t v = 0, len = 0;
    bool digits = true;
    __device__ __forceinline__ void add(uint32_t d)
    {
        digits &= d <= 9;
        ++len;
        v = v * 10 + d;            // wraps past 9 digits, which no key uses
    }
    __device__ __forceinline__ bool ok() const { return digits && len >= 1 && len <= 9; }
};

// The key of one header (h: the header line after '@', hl bytes before its '\n'); kKmerEmpty when untiled.  One thread reads
// the name in aligned 4-byte words and keeps fields 1..4 as it goes; it stops at the name's end or at the sixth ':' (n >= 7
// then, and fields 3 and 4 are complete).  A word holding a byte of the line lies inside the input buffer.
__device__ __forceinline__ unsigned long long tile_key(const uint8_t *h, uint32_t hl)
{
    TileField f1, f2, f3, f4;
    uint32_t fi = 0;
    const uintptr_t start = reinterpret_cast<uintptr_t>(h);
    bool done = false;
    for (uintptr_t w = start & ~(uintptr_t)3; !done; w += 4) {
        const uint32_t word = *reinterpret_cast<const uint32_t *>(w);
#pragma unroll
        for (uint32_t k = 0; k < 4; ++k) {
            const uintptr_t at = w + k;
            if (done || at < start) continue;
            const uint32_t c = at - start < hl ? (word >> (8 * k)) & 0xffu : '\n';
            if (c == ' ' || c == '\t' || c == '\r' || c == '\n') { done = true; continue; }
            if (c == ':') {
                done = ++fi >= 6;
                continue;
            }
            const uint32_t d = c - '0';
            if (fi == 1) f1.add(d);
            else if (fi == 2) f2.add(d);
            else if (fi == 3) f3.add(d);
            else if (fi == 4) f4.add(d);
        }
    }
    const TileField &lane = fi >= 6 ? f3 : f1, &tile = fi >= 6 ? f4 : f2;
    if (fi < 4 || !lane.ok() || !tile.ok()) return kKmerEmpty;
    return ((unsigned long long)lane.v << 32) | tile.v;
}

__device__ __forceinline__ void prefetch_l2(const void *p)
{
    asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}

__device__ __forceinline__ void prefetch_quality(const uint8_t *raw, const Rec &rc)
{
    for (uint32_t o = rc.qual & ~127u; o < rc.qual + rc.len; o += 128) prefetch_l2(raw + o);
}

__device__ __forceinline__ uint32_t tile_wait_id(KmerSlot *p)
{
    uint32_t v;
    while ((v = *reinterpret_cast<volatile uint32_t *>(&p->count)) == 0) {}
    return v - 1;
}

// First slot on the key's chain that holds the key (found = true) or is empty.
__device__ __forceinline__ KmerSlot *tile_probe(const KmerTable &T, unsigned long long key, bool &found)
{
    unsigned long long slot = kmer_hash(key) & T.cap_mask;
    for (;;) {
        KmerSlot *const p = &T.slots[slot];
        const unsigned long long k = *reinterpret_cast<volatile unsigned long long *>(&p->key);
        if (k == key || k == kKmerEmpty) {
            found = k == key;
            return p;
        }
        slot = (slot + 1) & T.cap_mask;
    }
}

// The dense id of a key, claiming a slot for a new one; kTileOverflowed when all kTileMaxKeys ids are taken by other keys.
__device__ uint32_t tile_insert(const KmerTable &T, TileCounters *cnt, unsigned long long key)
{
    for (;;) {
        bool found;
        KmerSlot *p = tile_probe(T, key, found);
        if (found) return tile_wait_id(p);
        if (*reinterpret_cast<volatile uint32_t *>(&cnt->claims) >= kTileMaxKeys) {
            __threadfence();                                  // every claim is in the table before its count
            p = tile_probe(T, key, found);
            return found ? tile_wait_id(p) : kTileOverflowed;
        }
        if (atomicAdd(&cnt->tickets, 1u) >= kTileMaxKeys) {
            atomicSub(&cnt->tickets, 1u);                     // claims under way may yet hand theirs back: look again
            continue;
        }
        unsigned long long slot = p - T.slots;
        for (;;) {
            KmerSlot *const q = &T.slots[slot];
            const unsigned long long prev = atomicCAS(&q->key, kKmerEmpty, key);
            if (prev == kKmerEmpty) {
                __threadfence();
                const uint32_t id = atomicAdd(&cnt->claims, 1u);
                atomicExch(&q->count, id + 1);
                return id;
            }
            if (prev == key) {
                atomicSub(&cnt->tickets, 1u);
                return tile_wait_id(q);
            }
            slot = (slot + 1) & T.cap_mask;
        }
    }
}

// One warp per 32 consecutive reads of one mate (mate-major), one thread per header.  Lanes with equal keys look them up
// once.
__global__ void __launch_bounds__(kTileKeyThreads) k_tile_keys(const TileKeyArgs a)
{
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t warp = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
    const uint32_t per_mate = (a.n_rec + 31) / 32;
    if (warp >= per_mate * a.n_mates) return;
    const uint32_t m = warp / per_mate, t = (warp - m * per_mate) * 32 + lane;
    const uint8_t *const raw = m ? a.raw[1] : a.raw[0];          // selected, not indexed: the arguments stay in constant memory
    uint16_t *const ids = m ? a.id[1] : a.id[0];
    const bool valid = t < a.n_rec;
    unsigned long long key = kKmerEmpty;
    if (valid) {
        const Rec rc = (m ? a.rec[1] : a.rec[0])[t];
        key = tile_key(raw + rc.hdr + 1, rc.seq - rc.hdr >= 2 ? rc.seq - rc.hdr - 2 : 0);
    }
    const bool tiled = valid && key != kKmerEmpty;
    const uint32_t untiled = __popc(__ballot_sync(0xffffffffu, valid && !tiled));
    if (lane == 0 && untiled) atomicAdd(&a.cnt->untiled[m ? 1 : 0], (unsigned long long)untiled);
    const uint32_t peers = __match_any_sync(0xffffffffu, key), leader = __ffs(peers) - 1;
    uint32_t id = kTileUntiled;
    if (tiled && lane == leader) {
        id = tile_insert(a.T, a.cnt, key);
        if (id == kTileOverflowed) atomicOr(&a.cnt->overflow, 1u);
    }
    id = __shfl_sync(0xffffffffu, id, leader);
    if (valid) ids[t] = (uint16_t)(tiled ? id : kTileUntiled);
}

// Reads [w * run, (w + 1) * run) of one mate per warp.  Dynamic shared memory: a row of L.C u32 score sums per warp.
__global__ void __launch_bounds__(kTileQualThreads) k_tile_qual(const TileQualArgs a)
{
    extern __shared__ uint32_t tq_smem[];
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t warp = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
    const uint32_t per_mate = (a.n_rec + a.run - 1) / a.run;
    if (warp >= per_mate * a.n_mates) return;
    const uint32_t m = warp / per_mate, r0 = (warp - m * per_mate) * a.run, r1 = min(a.n_rec, r0 + a.run);
    uint32_t *const row = tq_smem + (threadIdx.x / 32) * a.L.C;
    const uint8_t *const raw = m ? a.raw[1] : a.raw[0];
    const Rec *const rec = m ? a.rec[1] : a.rec[0];
    const uint16_t *const ids = m ? a.id[1] : a.id[0];
    const TileLayout L = a.L;
    for (uint32_t c = lane; c < L.C; c += 32) row[c] = 0;
    uint32_t cur = kTileUntiled, span = 0;                    // current id; cycles of the row in use
    unsigned long long tot_q = 0, tot_b = 0;                  // lane's share of the whole-read sums; bases (lane 0)
    uint32_t run_len = 0, run_n = 0;                          // lane 0: the current run of equal clamped lengths
    auto flush = [&]() {
        if (cur >= kTileMaxKeys) return;
        const uint32_t d = a.n_mates * cur + m;
        for (uint32_t c = lane; c < span; c += 32) {
            if (row[c]) atomicAdd(&a.acc[L.cyc(c, d)], (unsigned long long)row[c]);
            row[c] = 0;
        }
        for (int o = 16; o; o >>= 1) tot_q += __shfl_xor_sync(0xffffffffu, tot_q, o);
        if (lane == 0) {
            if (run_n) atomicAdd(&a.acc[L.hist(run_len, d)], (unsigned long long)run_n);
            if (tot_b) atomicAdd(&a.acc[L.bases(d)], tot_b);
            if (tot_q) atomicAdd(&a.acc[L.qual(d)], tot_q);
        }
        span = 0; tot_q = 0; tot_b = 0; run_n = 0;
    };
    // 32 reads at a time: lane j holds read j's id and record, the warp walks them with shuffles.  Records are loaded two
    // blocks ahead and the quality lines of the next block requested from the L2 one block ahead, so that the loads that
    // wait on a read are L2 hits.
    const Rec none{0, 0, 0, 0};
    Rec rc0 = r0 + lane < r1 ? rec[r0 + lane] : none, rc1 = r0 + 32 + lane < r1 ? rec[r0 + 32 + lane] : none;
    uint32_t id0 = r0 + lane < r1 ? ids[r0 + lane] : kTileUntiled, id1 = r0 + 32 + lane < r1 ? ids[r0 + 32 + lane] : kTileUntiled;
    if (id0 < kTileMaxKeys) prefetch_quality(raw, rc0);
    for (uint32_t b = r0; b < r1; b += 32) {
        const bool in2 = b + 64 + lane < r1;
        const Rec rc2 = in2 ? rec[b + 64 + lane] : none;
        const uint32_t id2 = in2 ? ids[b + 64 + lane] : kTileUntiled;
        if (id1 < kTileMaxKeys) prefetch_quality(raw, rc1);
        const uint32_t nb = min(32u, r1 - b);
        for (uint32_t j = 0; j < nb; ++j) {
            const uint32_t id = __shfl_sync(0xffffffffu, id0, j);
            if (id != cur) {
                flush();
                cur = id;
            }
            if (id >= kTileMaxKeys) continue;
            const uint8_t *const q = raw + __shfl_sync(0xffffffffu, rc0.qual, j);
            const uint32_t len = __shfl_sync(0xffffffffu, rc0.len, j), clamped = min(len, L.C);
            span = max(span, clamped);
            // the first kRegCycles cycles: every load issued before the first add
            uint32_t sc[kRegCycles / 32];
#pragma unroll
            for (uint32_t k = 0; k < kRegCycles / 32; ++k) {
                const uint32_t c = lane + 32 * k;
                sc[k] = c < len ? (uint32_t)max(0, (int)q[c] - a.in_off) : 0u;
            }
#pragma unroll
            for (uint32_t k = 0; k < kRegCycles / 32; ++k) {
                const uint32_t c = lane + 32 * k;
                tot_q += sc[k];
                if (c < L.C) row[c] += sc[k];
            }
            for (uint32_t c = kRegCycles + lane; c < len; c += 32) {
                const uint32_t s = (uint32_t)max(0, (int)q[c] - a.in_off);
                tot_q += s;
                if (c < L.C) row[c] += s;
            }
            if (lane == 0) {
                tot_b += len;
                if (run_n && run_len != clamped) {
                    atomicAdd(&a.acc[L.hist(run_len, a.n_mates * cur + m)], (unsigned long long)run_n);
                    run_n = 0;
                }
                run_len = clamped;
                ++run_n;
            }
        }
        rc0 = rc1; id0 = id1;
        rc1 = rc2; id1 = id2;
    }
    flush();
}

// Columns [0, from.D) and rows of `from` into the (larger, zeroed) block `to`: histogram bin b and cycle c keep their index.
__global__ void __launch_bounds__(256) k_tile_relay(const unsigned long long *src, TileLayout from, unsigned long long *dst, TileLayout to)
{
    const size_t n = from.total();
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const uint32_t d = (uint32_t)(i % from.D), r = (uint32_t)(i / from.D);
        size_t j;
        if (r < 2) j = (size_t)r * to.D + d;
        else if (r < 3 + from.C) j = to.hist(r - 2, d);
        else j = to.cyc(r - 3 - from.C, d);
        dst[j] = src[i];
    }
}

}  // namespace fq
