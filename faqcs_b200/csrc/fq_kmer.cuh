// fq_kmer.cuh -- k-mer rarefaction (--qc_only --kmer_rarefaction; SURVEY 8(f) N4).
//
// update_kmer (trim.cpp:887-931) counts the canonical k-mers (minimum of a k-mer and its reverse complement, two bits per
// base with A=0 T=1 C=2 G=3, FaQCs.h:35-42; any other character restarts the window) while the rarefaction curve is being
// collected: of every raw read under --qc_only (trim.cpp:260-262), of the trimmed sequence of every surviving read
// otherwise (trim.cpp:545-547), into one table per pass over an input (FaQCs.cpp:235, 588).  At the end of a
// trim() call whose running read count crossed another multiple of --split_size the reference records (reads so far,
// distinct k-mers, k-mer instances) (trim.cpp:157-185); at the end of the pass it turns the table into a histogram of
// counts (FaQCs.cpp:518-521, 737-740).
//
// Here the table is an open-addressing hash table in HBM (16-byte slots, linear probing).  Every slot also remembers the
// FIRST trim() call that produced its k-mer, and every call its number of instances, so all points of the curve follow from
// the final table: distinct(c) = #{slots first seen in a call <= c}, total(c) = sum of instances of the calls <= c.
// One thread walks one read with the same rolling update as the reference.
#pragma once
#include "fq_common.cuh"

namespace fq {

constexpr unsigned long long kKmerEmpty = ~0ull;
constexpr uint32_t kKmerMaxCalls = 1u << 16;         // trim() calls of one pass while the curve is collected
constexpr uint32_t kKmerSmallCounts = 1u << 16;      // counts below this go to a dense histogram, larger ones to a list

struct KmerSlot {                   // 16 bytes: key, count and first call of a k-mer share one 32-byte sector
    unsigned long long key;         // canonical k-mer or kKmerEmpty
    uint32_t count;
    uint32_t first_call;            // smallest call index that inserted the k-mer
};
struct KmerTable {
    KmerSlot *slots;                // [cap]
    unsigned long long cap_mask;    // cap - 1 (cap is a power of two)
};

struct KmerArgs {
    const uint8_t *raw[2];
    const Rec *rec[2];
    const uint2 *res[2];            // trim verdicts: count the trimmed sequence of surviving reads; null = the raw read (--qc_only)
    uint32_t n_rec, n_mates;
    uint32_t k;
    uint32_t replace_q;             // --replace_to_N_q of a trimming run: a 'G' below this score has become 'N' (trim.cpp:389-403)
    int32_t in_off;
    uint32_t first_call;            // call index of (mate 0, record 0) inside the pass
    uint32_t stop_call;             // calls >= this one do not count (the curve is complete)
    KmerTable T;
    unsigned long long *call_total; // [kKmerMaxCalls] instances per call
};

__device__ __forceinline__ unsigned long long kmer_hash(unsigned long long x)
{
    x ^= x >> 33; x *= 0xff51afd7ed558ccdull; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ull; x ^= x >> 33;
    return x;
}

__device__ __forceinline__ void kmer_insert(const KmerTable &T, unsigned long long key, uint32_t call)
{
    unsigned long long slot = kmer_hash(key) & T.cap_mask;
    for (;;) {
        KmerSlot *const p = &T.slots[slot];
        // most k-mers of real data are already in the table: look before claiming (a key never changes once it is set)
        unsigned long long prev = *reinterpret_cast<volatile unsigned long long *>(&p->key);
        if (prev == kKmerEmpty) prev = atomicCAS(&p->key, kKmerEmpty, key);
        if (prev == kKmerEmpty || prev == key) {
            atomicAdd(&p->count, 1u);
            if (call < *reinterpret_cast<volatile uint32_t *>(&p->first_call)) atomicMin(&p->first_call, call);
            return;
        }
        slot = (slot + 1) & T.cap_mask;
    }
}

// kmer_insert adding `add` to the key's count (first_call untouched): returns the count right after this increment.
__device__ __forceinline__ uint32_t kmer_insert_add(const KmerTable &T, unsigned long long key, uint32_t add)
{
    unsigned long long slot = kmer_hash(key) & T.cap_mask;
    for (;;) {
        KmerSlot *const p = &T.slots[slot];
        unsigned long long prev = *reinterpret_cast<volatile unsigned long long *>(&p->key);
        if (prev == kKmerEmpty) prev = atomicCAS(&p->key, kKmerEmpty, key);
        if (prev == kKmerEmpty || prev == key) return atomicAdd(&p->count, add) + add;
        slot = (slot + 1) & T.cap_mask;
    }
}

// One thread per read (mate-major).  The reference's trim() call of record r of mate m (batches of 32768 records, mate 1's
// call in front of mate 2's): first_call + (r / 32768) * n_mates + m.
__global__ void __launch_bounds__(256) k_kmer(const KmerArgs a)
{
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= a.n_rec * a.n_mates) return;
    const uint32_t mate = g >= a.n_rec ? 1u : 0u, r = g - mate * a.n_rec;
    const uint32_t call = a.first_call + (r / FQ_REF_BATCH) * a.n_mates + mate;
    if (call >= a.stop_call) return;
    const Rec rc = (mate ? a.rec[1] : a.rec[0])[r];
    const uint8_t *s = (mate ? a.raw[1] : a.raw[0]) + rc.seq;
    const signed char *q = reinterpret_cast<const signed char *>((mate ? a.raw[1] : a.raw[0]) + rc.qual);
    uint32_t len = rc.len, replace_q = 0;
    if (const uint2 *res = mate ? a.res[1] : a.res[0]) {
        const uint2 v = res[r];
        if (!((v.y >> kResLenBits) & FQ_RR_VALID)) return;
        s += v.x & ~kResPlusBad;
        q += v.x & ~kResPlusBad;
        len = v.y & kResLenMask;
        replace_q = a.replace_q;
    }
    const unsigned long long mask = (1ull << (2 * a.k)) - 1ull;
    const uint32_t comp_shift = 2 * (a.k - 1);
    unsigned long long w = 0, comp = 0;
    uint32_t word_len = 0, n_inst = 0;
    for (uint32_t i = 0; i < len; ++i) {
        ++word_len;
        uint32_t b;
        uint32_t ch = s[i];
        if (replace_q && ch == 'G' && max(0, (int)q[i] - a.in_off) < (int)replace_q) ch = 'N';
        switch (ch | 0x20u) {
            case 'a': b = 0; break;
            case 't': b = 1; break;
            case 'c': b = 2; break;
            case 'g': b = 3; break;
            default: b = 4; break;
        }
        if (b < 4) {
            w = (w << 2) | b;
            comp = (comp >> 2) | ((unsigned long long)(b ^ 1u) << comp_shift);        // A <-> T, C <-> G
        } else word_len = 0;
        if (word_len >= a.k) {
            const unsigned long long x = w & mask, y = comp & mask;
            kmer_insert(a.T, x < y ? x : y, call);
            ++n_inst;
        }
    }
    if (n_inst) atomicAdd(&a.call_total[call], (unsigned long long)n_inst);
}

__global__ void __launch_bounds__(256) k_kmer_clear(KmerTable T)
{
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i <= T.cap_mask; i += (unsigned long long)gridDim.x * blockDim.x) {
        T.slots[i] = KmerSlot{kKmerEmpty, 0u, 0xffffffffu};
    }
}

// Re-insert every entry of `from` into the (larger, cleared) table `to`.
__global__ void __launch_bounds__(256) k_kmer_rehash(KmerTable from, KmerTable to)
{
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i <= from.cap_mask; i += (unsigned long long)gridDim.x * blockDim.x) {
        const KmerSlot e = from.slots[i];
        if (e.key == kKmerEmpty) continue;
        unsigned long long slot = kmer_hash(e.key) & to.cap_mask;
        for (;;) {
            const unsigned long long prev = atomicCAS(&to.slots[slot].key, kKmerEmpty, e.key);
            if (prev == kKmerEmpty) {
                to.slots[slot].count = e.count;
                to.slots[slot].first_call = e.first_call;
                break;
            }
            slot = (slot + 1) & to.cap_mask;
        }
    }
}

// End of a pass: distinct k-mers per first call, histogram of counts (dense below kKmerSmallCounts, a list above).
__global__ void __launch_bounds__(256) k_kmer_summarize(KmerTable T, unsigned long long *call_distinct, unsigned long long *small_hist, uint32_t *big_list,
                                                        uint32_t big_cap, uint32_t *n_big, unsigned long long *n_distinct)
{
    unsigned long long mine = 0;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i <= T.cap_mask; i += (unsigned long long)gridDim.x * blockDim.x) {
        const KmerSlot e = T.slots[i];
        if (e.key == kKmerEmpty) continue;
        ++mine;
        const uint32_t c = e.count, f = e.first_call;
        if (f < kKmerMaxCalls) atomicAdd(&call_distinct[f], 1ull);
        if (c < kKmerSmallCounts) atomicAdd(&small_hist[c], 1ull);
        else {
            const uint32_t k = atomicAdd(n_big, 1u);
            if (k < big_cap) big_list[k] = c;
        }
    }
    if (mine) atomicAdd(n_distinct, mine);
}

// Occupied slots (load check before a batch).
__global__ void __launch_bounds__(256) k_kmer_count(KmerTable T, unsigned long long *n_distinct)
{
    unsigned long long mine = 0;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i <= T.cap_mask; i += (unsigned long long)gridDim.x * blockDim.x)
        mine += T.slots[i].key != kKmerEmpty;
#pragma unroll
    for (int o = 16; o; o >>= 1) mine += __shfl_xor_sync(0xffffffffu, mine, o);
    if ((threadIdx.x & 31) == 0 && mine) atomicAdd(n_distinct, mine);
}

// ---- a table sharded over n contexts: end of pass ---------------------------------------------------------------------
// Every context counted its own batches into its own table.  At the end of the pass each k-mer gets one owner context;
// every context sends its entries to their owners, and each owner merges what it receives into a cleared table (counts add,
// first calls take the minimum), so the owners' tables together hold the table one context would have built.
constexpr uint32_t kKmerMaxOwners = 1024;

// The slot index uses the low bits of the hash, the owner the high half: a shard's keys still spread over its whole table.
__device__ __forceinline__ uint32_t kmer_owner(unsigned long long key, uint32_t n)
{
    return (uint32_t)(((kmer_hash(key) >> 32) * n) >> 32);
}

// Occupied slots per owner (count[n], zeroed by the caller).
__global__ void __launch_bounds__(256) k_kmer_partition_count(KmerTable T, uint32_t n, unsigned long long *count)
{
    __shared__ uint32_t h[kKmerMaxOwners];
    for (uint32_t j = threadIdx.x; j < n; j += blockDim.x) h[j] = 0;
    __syncthreads();
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i <= T.cap_mask; i += (unsigned long long)gridDim.x * blockDim.x) {
        const unsigned long long key = T.slots[i].key;
        if (key != kKmerEmpty) atomicAdd(&h[kmer_owner(key, n)], 1u);
    }
    __syncthreads();
    for (uint32_t j = threadIdx.x; j < n; j += blockDim.x)
        if (h[j]) atomicAdd(&count[j], (unsigned long long)h[j]);
}

// The occupied slots into `out`, grouped by owner: cursor[j] starts at group j's offset.  The lanes of a warp that share an
// owner take their places with one atomic.  (The grid stride is a multiple of 32 and the capacity a power of two >= 32, so
// every lane of a warp makes the same number of trips.)
__global__ void __launch_bounds__(256) k_kmer_partition_scatter(KmerTable T, uint32_t n, unsigned long long *cursor, KmerSlot *out)
{
    const uint32_t lane = threadIdx.x & 31;
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i <= T.cap_mask; i += (unsigned long long)gridDim.x * blockDim.x) {
        const KmerSlot e = T.slots[i];
        const bool used = e.key != kKmerEmpty;
        const uint32_t active = __ballot_sync(0xffffffffu, used);
        if (!used) continue;
        const uint32_t owner = kmer_owner(e.key, n);
        const uint32_t peers = __match_any_sync(active, owner);
        const uint32_t leader = __ffs(peers) - 1;
        unsigned long long base = 0;
        if (lane == leader) base = atomicAdd(&cursor[owner], (unsigned long long)__popc(peers));
        base = __shfl_sync(peers, base, leader);
        out[base + __popc(peers & ((1u << lane) - 1u))] = e;
    }
}

// Entries of other tables into T: counts add, the first call is the smallest.
__global__ void __launch_bounds__(256) k_kmer_merge(KmerTable T, const KmerSlot *in, unsigned long long n)
{
    for (unsigned long long i = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (unsigned long long)gridDim.x * blockDim.x) {
        const KmerSlot e = in[i];
        unsigned long long slot = kmer_hash(e.key) & T.cap_mask;
        for (;;) {
            KmerSlot *const p = &T.slots[slot];
            unsigned long long prev = *reinterpret_cast<volatile unsigned long long *>(&p->key);
            if (prev == kKmerEmpty) prev = atomicCAS(&p->key, kKmerEmpty, e.key);
            if (prev == kKmerEmpty || prev == e.key) {
                atomicAdd(&p->count, e.count);
                if (e.first_call < *reinterpret_cast<volatile uint32_t *>(&p->first_call)) atomicMin(&p->first_call, e.first_call);
                break;
            }
            slot = (slot + 1) & T.cap_mask;
        }
    }
}

}  // namespace fq
