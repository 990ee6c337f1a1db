// fq_dup.cuh -- sequence duplication statistics (fq_dup_*, --dup_stats).
//
// A unit is a read of a single-end pass or a pair (records i of R1 and R2) of a paired pass.  Every framed record counts,
// whatever trimming and filtering later make of it.  Two units are copies when their sequence lines are byte for byte the
// same, exactly as framed: the bytes up to the line's first '\r' or '\n' (Rec::len after k_fix_lone_cr), case-sensitive,
// before terminal-N masking, trimming and the G -> N replacement.  Each unit is inserted once, as a 64-bit key, into an
// open-addressing table of KmerSlot (fq_kmer.cuh) whose count is then the key's multiplicity; the end of a pass merges the
// per-context tables exactly as the k-mer table's are merged, and the result is the histogram of the counts.
//
// Key.  fmix64 is kmer_hash (murmur3's 64-bit finalizer); w_i are the little-endian 8-byte words of a line of len bytes, the
// last one zero-padded; all arithmetic is mod 2^64:
//     h(s) = fmix64( sum_i fmix64(w_i + (i + 1) * 0x9e3779b97f4a7c15) + len * 0xc2b2ae3d27d4eb4f )
//     pair: key = fmix64(h(r1) + fmix64(h(r2) ^ 0x165667b19e3779f9))        single-end: key = h(r1)
// and a key equal to kKmerEmpty becomes kKmerEmpty - 1.  The words enter through a sum, so the lanes of a warp fingerprint
// their words independently and reduce them in any order; the position of a word enters through (i + 1), the length through
// its own term (lines that differ only in trailing zero bytes differ), and the pair form is not symmetric in its mates.
// Collisions: n distinct units give about n^2 / 2^65 expected pairs of equal keys (0.03 at 10^9 units); each would count two
// different units as copies.
#pragma once
#include "fq_kmer.cuh"

namespace fq {

constexpr unsigned long long kDupWordMul = 0x9e3779b97f4a7c15ull;
constexpr unsigned long long kDupLenMul = 0xc2b2ae3d27d4eb4full;
constexpr unsigned long long kDupPairXor = 0x165667b19e3779f9ull;

struct DupArgs {
    const uint8_t *raw[2];
    const Rec *rec[2];
    uint32_t n_rec, n_mates;
    KmerTable T;
};

// Term i of h's sum: the mixed little-endian word of bytes 8i .. 8i+7 of the line (zero-padded), 0 beyond its end.  The
// eight byte loads are independent, and the lanes of a warp taking consecutive words read one contiguous span of the line.
__device__ __forceinline__ unsigned long long dup_word_term(const uint8_t *s, uint32_t len, uint32_t i)
{
    const uint32_t k = 8 * i;
    if (k >= len) return 0ull;
    unsigned long long w = 0;
#pragma unroll
    for (uint32_t b = 0; b < 8; ++b)
        if (k + b < len) w |= (unsigned long long)s[k + b] << (8 * b);
    return kmer_hash(w + (unsigned long long)(i + 1) * kDupWordMul);
}

__device__ __forceinline__ unsigned long long dup_warp_sum(unsigned long long v)
{
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// One warp per unit: lane l takes words l, l + 32, ... of both mates' lines in the same loop (every load of a unit is in
// flight at once for lines up to 256 bytes), a butterfly sum gives h on every lane, and lane 0 inserts the key once.  The
// slot's first_call stays at its cleared value, so k_kmer_summarize's per-call array never sees this table.
__global__ void __launch_bounds__(256) k_dup(const DupArgs a)
{
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t u = blockIdx.x * (blockDim.x / 32) + threadIdx.x / 32;
    if (u >= a.n_rec) return;
    const Rec r1 = a.rec[0][u];
    const Rec r2 = a.n_mates == 2 ? a.rec[1][u] : Rec{0u, 0u, 0u, 0u};
    const uint8_t *s1 = a.raw[0] + r1.seq, *s2 = a.n_mates == 2 ? a.raw[1] + r2.seq : nullptr;
    unsigned long long acc1 = 0, acc2 = 0;
    for (uint32_t i = lane; 8 * i < max(r1.len, r2.len); i += 32) {
        acc1 += dup_word_term(s1, r1.len, i);
        acc2 += dup_word_term(s2, r2.len, i);
    }
    unsigned long long key = kmer_hash(dup_warp_sum(acc1) + (unsigned long long)r1.len * kDupLenMul);
    if (a.n_mates == 2)
        key = kmer_hash(key + kmer_hash(kmer_hash(dup_warp_sum(acc2) + (unsigned long long)r2.len * kDupLenMul) ^ kDupPairXor));
    if (key == kKmerEmpty) key = kKmerEmpty - 1;
    if (lane == 0) kmer_insert(a.T, key, 0xffffffffu);
}

}  // namespace fq
