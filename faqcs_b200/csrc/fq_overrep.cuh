// fq_overrep.cuh -- overrepresented sequences (fq_overrep_*, --overrep).
//
// A unit is one read; the mates of a pair are counted separately (mate m = 1, 2; a single-end batch has mate 1 only).  Every
// framed record counts, whatever trimming and filtering later make of it.  A read's prefix is the first min(len, P) bytes of
// its sequence line as framed (up to the first '\r' or '\n': Rec::len after k_fix_lone_cr), case-sensitive, before masking,
// trimming and the G -> N replacement; P = prefix_len (1..256).  Reads with equal prefixes are one sequence; a read shorter than
// P is its own whole sequence; reads of length 0 count in N_m but are never keyed.
//
// Key.  h is the line fingerprint of fq_dup.cuh applied to the prefix (len = the prefix's length); key = (h & ~1) | (m - 1), so
// the mate is the key's low bit, and a key equal to kKmerEmpty becomes kKmerEmpty - 2 (still mate 2).  n distinct prefixes
// of one mate give about n^2 / 2^64 expected pairs of equal keys (0.05 at 10^9 prefixes); each would count two sequences
// as one.
//
// Report.  N_m = mate-m reads of the pass, ppm = min_ppm (10..10^6).  A sequence of mate m with count c is reported when
// c * 10^6 >= ppm * N_m and c >= 2, i.e. c >= min_count_m = max(2, ceil(ppm * N_m / 10^6)).
//
// Counting is exact: every key goes into an open-addressing table of KmerSlot (fq_kmer.cuh), merged at the end of a pass
// exactly as the duplication table is.  The bytes come from a small capture store per context: the thread whose increment
// leaves the key's count in this context at c_after writes the prefix into the store when
//     c_after * 10^6 >= ppm * n_{ctx,m}(b)                       (n_{ctx,m}(b): mate-m reads this context counted through batch b)
// and the key is not there yet.  Every reported key meets the threshold in some context i (otherwise summing the strict
// inequalities over the contexts would contradict it), and in the last batch of context i that holds the key one increment
// returns the final local count c_i >= ppm * n_i / 10^6 >= ppm * n_i(b) / 10^6: that increment captured it.  The c >= 2 rule
// belongs to the report only.  In one batch at most floor(10^6 / ppm) keys per mate meet the condition (their counts add up
// to at most n), which bounds the store's growth per batch.
#pragma once
#include "fq_dup.cuh"

namespace fq {

constexpr uint32_t kOverrepMaxPrefix = 256;

// The capture store: cap_mask + 1 entries of `stride` bytes {key (kKmerEmpty: free), len, mate - 1, prefix bytes}.
struct OverrepStore {
    uint8_t *e;
    unsigned long long cap_mask;
    uint32_t stride;
    unsigned long long *n;          // entries claimed (exact occupancy, read by the host before a batch when it matters)
};

struct OverrepArgs {
    const uint8_t *raw[2];
    const Rec *rec[2];
    uint32_t n_rec, n_mates, prefix_len;
    unsigned long long thr[2];      // ppm * n_{ctx,m}(b): the capture threshold of mate m, times 10^6
    KmerTable T;
    OverrepStore S;
};

__device__ __forceinline__ unsigned long long *overrep_entry(const OverrepStore &S, unsigned long long i)
{
    return reinterpret_cast<unsigned long long *>(S.e + i * S.stride);
}

// The prefix of a key into the store unless it is there already.  A plain load comes first, so a key that was captured long
// ago costs one read; only the thread that claims the entry writes it.
__device__ __forceinline__ void overrep_capture(const OverrepStore &S, unsigned long long key, uint32_t mate0, const uint8_t *s, uint32_t len)
{
    unsigned long long slot = kmer_hash(key) & S.cap_mask;
    for (;;) {
        unsigned long long *const p = overrep_entry(S, slot);
        unsigned long long prev = *reinterpret_cast<volatile unsigned long long *>(p);
        if (prev == kKmerEmpty) prev = atomicCAS(p, kKmerEmpty, key);
        if (prev == kKmerEmpty) {
            uint32_t *const h = reinterpret_cast<uint32_t *>(p + 1);
            h[0] = len;
            h[1] = mate0;
            uint8_t *const d = reinterpret_cast<uint8_t *>(p + 2);
            for (uint32_t i = 0; i < len; ++i) d[i] = s[i];
            atomicAdd(S.n, 1ull);
            return;
        }
        if (prev == key) return;
        slot = (slot + 1) & S.cap_mask;
    }
}

// One warp per 32 consecutive reads of one mate (mate-major).  A group of 8 lanes fingerprints one read's prefix (words i,
// i + 8, ... on lane i, at most 4 per lane) and reduces it with three shuffles; in 8 rounds the 4 groups key the warp's 32
// reads, and lane 8g + r keeps the key of read 4r + g.  Lanes with equal keys then insert once, adding their number: the
// count returned is the c_after of the last of them, which is what the capture rule needs.
__global__ void __launch_bounds__(256) k_overrep(const OverrepArgs a)
{
    const uint32_t lane = threadIdx.x & 31, g = lane >> 3, l = lane & 7;
    const uint32_t warp = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
    const uint32_t per_mate = (a.n_rec + 31) / 32;
    if (warp >= per_mate * a.n_mates) return;
    const uint32_t m = warp / per_mate, base = (warp - m * per_mate) * 32;
    const uint8_t *const raw = a.raw[m];
    const Rec *const rec = a.rec[m];
    unsigned long long key = 0;
    uint32_t my_len = 0, my_seq = 0;
#pragma unroll 1
    for (uint32_t r = 0; r < 8; ++r) {
        const uint32_t t = base + 4 * r + g;
        uint32_t len = 0, seq = 0;
        if (t < a.n_rec) {
            const Rec rc = rec[t];
            len = min(rc.len, a.prefix_len);
            seq = rc.seq;
        }
        unsigned long long acc = 0;
        for (uint32_t i = l; 8 * i < len; i += 8) acc += dup_word_term(raw + seq, len, i);
        acc += __shfl_xor_sync(0xffffffffu, acc, 4);
        acc += __shfl_xor_sync(0xffffffffu, acc, 2);
        acc += __shfl_xor_sync(0xffffffffu, acc, 1);
        if (l == r) {
            key = (kmer_hash(acc + (unsigned long long)len * kDupLenMul) & ~1ull) | m;
            if (key == kKmerEmpty) key = kKmerEmpty - 2;
            my_len = len;
            my_seq = seq;
        }
    }
    const bool keyed = my_len > 0;
    const uint32_t active = __ballot_sync(0xffffffffu, keyed);
    if (!keyed) return;
    const uint32_t peers = __match_any_sync(active, key);
    if (lane != (uint32_t)__ffs(peers) - 1) return;
    const uint32_t c_after = kmer_insert_add(a.T, key, __popc(peers));
    if ((unsigned long long)c_after * 1000000ull >= a.thr[m]) overrep_capture(a.S, key, m, raw + my_seq, my_len);
}

// End of a pass, on the owner shard: the slots that pass the report rule (count >= min_count of the key's mate), compacted.
__global__ void __launch_bounds__(256) k_overrep_select(KmerTable T, unsigned long long min1, unsigned long long min2, KmerSlot *out, uint32_t cap, uint32_t *n_out)
{
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i <= T.cap_mask; i += (unsigned long long)gridDim.x * blockDim.x) {
        const KmerSlot e = T.slots[i];
        if (e.key == kKmerEmpty || e.count < ((e.key & 1ull) ? min2 : min1)) continue;
        const uint32_t k = atomicAdd(n_out, 1u);
        if (k < cap) out[k] = e;
    }
}

__global__ void __launch_bounds__(256) k_overrep_store_clear(OverrepStore S)
{
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i <= S.cap_mask; i += (unsigned long long)gridDim.x * blockDim.x)
        *overrep_entry(S, i) = kKmerEmpty;
}

// Every entry of `from` into the (larger, cleared) store `to`; keys are distinct, so the first free slot takes each.
__global__ void __launch_bounds__(256) k_overrep_store_rehash(OverrepStore from, OverrepStore to)
{
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i <= from.cap_mask; i += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned long long *const src = overrep_entry(from, i);
        const unsigned long long key = src[0];
        if (key == kKmerEmpty) continue;
        unsigned long long slot = kmer_hash(key) & to.cap_mask;
        while (atomicCAS(overrep_entry(to, slot), kKmerEmpty, key) != kKmerEmpty) slot = (slot + 1) & to.cap_mask;
        unsigned long long *const dst = overrep_entry(to, slot);
        for (uint32_t w = 1; w < from.stride / 8; ++w) dst[w] = src[w];
    }
}

}  // namespace fq
