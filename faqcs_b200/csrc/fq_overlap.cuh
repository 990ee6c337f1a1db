// fq_overlap.cuh -- paired-end insert size and overlap error profile (fq_overlap_*, --insert_size).
//
// Every pair of a paired batch (records i of R1 and R2, whatever trimming and filtering later make of it): a = R1's sequence
// line as framed (Rec::seq, Rec::len after k_fix_lone_cr), length L1; b = the reverse complement of R2's, length L2,
// b[j] = comp(R2[L2 - 1 - j]).  A, C, G, T in either case are known bases (case folded); every other byte is unknown, and a
// position matches only when both bases are known and equal (N against N is a mismatch).
//   Candidate insert size s: R1 covers fragment positions [0, L1), b covers [s - L2, s); the overlap is
//   [x0, x1) = [max(0, s - L2), min(L1, s)) of o(s) = x1 - x0 positions; candidates are the s with o(s) >= O.
//   m(s) = positions of the overlap that do not match; s is accepted when m(s) <= min(D, floor(o(s) * P / 100)).
//   The pair's insert size is the accepted s with the fewest mismatches, then the longest overlap, then the smallest s.
// Overlap position x is R1 cycle x and R2 cycle s - 1 - x (0-based).
//
// Kernel: one warp per pair.  The warp packs both mates into 32-base words of three bit planes {lo, hi, unknown} (one
// coalesced byte load per lane and word, three ballots), b reverse-complemented while it is packed and stored one word to
// the right so that a shifted fetch never reads in front of it.  Lane l tests the candidates s = O + l, O + l + 32, ...:
// per 32 positions of the overlap two 16-byte loads of b, three funnel shifts, three logic ops and a popcount, and the count
// stops as soon as it passes the candidate's limit (unrelated sequences pass a limit of 5 within the first word).  Three warp
// reductions pick the winner; the lanes then recompute its mismatch words to bump the per-cycle mismatch counters.  The
// per-cycle overlap counts are a difference array (+1 at the first cycle, -1 past the last), prefix-summed when the pass
// ends.  The counters live in shared memory per block (u32) and are added to the context's u64 block once per block; with
// mates too long for shared memory (kSmem == false) the planes go to a global scratch region per warp and the counters
// straight to the u64 block.
#pragma once
#include "fq_common.cuh"

namespace fq {

constexpr int kOvlThreads = 512;

// Indices of the accumulator block (u64 on the device, u32 in a block's shared copy) for a cycle capacity C: 8 scalars, the
// insert-size histogram [2C] (s <= L1 + L2 - O < 2C), the R1 and R2 overlap difference arrays [C + 1] each, the R1 and R2
// mismatch counts [C] each.
enum : uint32_t { kOvlTooShort, kOvlOverlapped, kOvlR1Adapter, kOvlR2Adapter, kOvlOverlapBases, kOvlMismatchBases, kOvlPairs, kOvlScalars = 8 };

struct OverlapLayout {
    uint32_t cyc, ins, d1, d2, m1, m2, total;
    __host__ __device__ static OverlapLayout make(uint32_t C)
    {
        OverlapLayout L;
        L.cyc = C;
        L.ins = kOvlScalars;
        L.d1 = L.ins + 2 * C;
        L.d2 = L.d1 + C + 1;
        L.m1 = L.d2 + C + 1;
        L.m2 = L.m1 + C;
        L.total = L.m2 + C;
        return L;
    }
};

struct OverlapArgs {
    const uint8_t *raw[2];
    const Rec *rec[2];
    uint32_t n_rec;
    uint32_t min_overlap, diff_limit, diff_percent;
    OverlapLayout L;
    unsigned long long *acc;       // the context's u64 block
    uint4 *scratch;                // kSmem == false: plane words of warp w at scratch + w * plane_words
    uint32_t wa, plane_words;      // words of a; words of a and b per warp
};

// A base as three plane bits: (c | 0x20) >> 1 & 3 codes a 0, c 1, g 3, t 2, so the complement flips the high bit.
__device__ __forceinline__ void ovl_code(uint32_t c, bool comp, uint32_t &lo, uint32_t &hi, uint32_t &un)
{
    c |= 0x20u;
    lo = (c >> 1) & 1u;
    hi = ((c >> 2) & 1u) ^ (comp ? 1u : 0u);
    // known: c is 0x60 + i with bit i of the mask set for a (1), c (3), g (7), t (0x14)
    un = (c >> 5) == 3u ? ((~0x10008Au >> (c & 31)) & 1u) : 1u;
}

// Mismatch bits of a's word w against b shifted so that b[j] faces a[j + s - L2]; e = L2 + 32 - s.  Only the bits of
// [x0, x1) are kept.
__device__ __forceinline__ uint32_t ovl_mismatch_word(const uint4 *A, const uint4 *B, uint32_t w, int32_t e, uint32_t x0, uint32_t x1)
{
    const uint4 av = A[w];
    const uint32_t jp = (uint32_t)((int32_t)(32 * w) + e), k = jp >> 5, sh = jp & 31;
    const uint4 b0 = B[k], b1 = B[k + 1];
    const uint32_t lo = __funnelshift_r(b0.x, b1.x, sh), hi = __funnelshift_r(b0.y, b1.y, sh), un = __funnelshift_r(b0.z, b1.z, sh);
    uint32_t mm = (av.x ^ lo) | (av.y ^ hi) | av.z | un;
    if (w == x0 >> 5) mm &= ~0u << (x0 & 31);
    if (w == (x1 - 1) >> 5) mm &= ~0u >> (31 - ((x1 - 1) & 31));
    return mm;
}

template <bool kSmem>
struct OvlAcc {
    uint32_t *s;
    unsigned long long *g;
    __device__ __forceinline__ void add(uint32_t i, uint32_t v) const
    {
        if (kSmem) atomicAdd(s + i, v);
        else atomicAdd(g + i, (unsigned long long)v);
    }
    // -1 at an entry of a difference array: a wrapped u32 in shared memory, sign-extended when the block is flushed
    __device__ __forceinline__ void dec(uint32_t i) const
    {
        if (kSmem) atomicAdd(s + i, ~0u);
        else atomicAdd(g + i, ~0ull);
    }
};

template <bool kSmem>
__device__ __forceinline__ void ovl_pair(const OverlapArgs &a, const OvlAcc<kSmem> &acc, uint4 *A, uint32_t p, uint32_t lane)
{
    const Rec r1 = a.rec[0][p], r2 = a.rec[1][p];
    const uint32_t L1 = r1.len, L2 = r2.len, O = a.min_overlap;
    if (L1 < O || L2 < O) {
        if (lane == 0) acc.add(kOvlTooShort, 1);
        return;
    }
    uint4 *B = A + a.wa;
    const uint8_t *s1 = a.raw[0] + r1.seq, *s2 = a.raw[1] + r2.seq;
    const uint32_t na = (L1 + 31) >> 5, nb = (L2 + 31) >> 5;
    // pack: eight words of each mate per round, every load of the round issued before the ballots
    for (uint32_t w0 = 0; w0 < max(na, nb); w0 += 8) {
        uint32_t c1[8], c2[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const uint32_t x = 32 * (w0 + k) + lane;
            c1[k] = x < L1 ? s1[x] : 0u;
            c2[k] = x < L2 ? s2[L2 - 1 - x] : 0u;
        }
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            if (w0 + k >= max(na, nb)) break;      // the same on every lane
            uint32_t lo, hi, un;
            ovl_code(c1[k], false, lo, hi, un);
            const uint4 va = make_uint4(__ballot_sync(~0u, lo), __ballot_sync(~0u, hi), __ballot_sync(~0u, un), 0u);
            ovl_code(c2[k], true, lo, hi, un);
            const uint4 vb = make_uint4(__ballot_sync(~0u, lo), __ballot_sync(~0u, hi), __ballot_sync(~0u, un), 0u);
            if (lane == 0 && w0 + k < na) A[w0 + k] = va;
            if (lane == 0 && w0 + k < nb) B[w0 + k + 1] = vb;
        }
    }
    __syncwarp();
    // candidates: the lane's best by (fewest mismatches, longest overlap, smallest s)
    uint32_t bm = 0xffffffffu, bo = 0, bs = 0xffffffffu;
    for (uint32_t s = O + lane; s <= L1 + L2 - O; s += 32) {
        const uint32_t x0 = s > L2 ? s - L2 : 0u, x1 = min(L1, s), o = x1 - x0;
        const uint32_t lim = min(a.diff_limit, o * a.diff_percent / 100u);       // o < 2^24, diff_percent <= 100
        const int32_t e = (int32_t)(L2 + 32) - (int32_t)s;
        uint32_t m = 0;
        for (uint32_t w = x0 >> 5; w <= (x1 - 1) >> 5 && m <= lim; ++w) m += __popc(ovl_mismatch_word(A, B, w, e, x0, x1));
        if (m <= lim && (m < bm || (m == bm && o > bo))) { bm = m; bo = o; bs = s; }
    }
    const uint32_t m = __reduce_min_sync(~0u, bm);
    if (m == 0xffffffffu) {
        __syncwarp();
        return;
    }
    const uint32_t o = __reduce_max_sync(~0u, bm == m ? bo : 0u);
    const uint32_t s = __reduce_min_sync(~0u, bm == m && bo == o ? bs : 0xffffffffu);
    const uint32_t x0 = s > L2 ? s - L2 : 0u, x1 = min(L1, s);
    if (lane == 0) {
        acc.add(kOvlOverlapped, 1);
        acc.add(a.L.ins + s, 1);
        if (s < L1) acc.add(kOvlR1Adapter, 1);
        if (s < L2) acc.add(kOvlR2Adapter, 1);
        acc.add(kOvlOverlapBases, o);
        acc.add(kOvlMismatchBases, m);
        acc.add(a.L.d1 + x0, 1);
        acc.dec(a.L.d1 + x1);
        acc.add(a.L.d2 + s - x1, 1);
        acc.dec(a.L.d2 + s - x0);
    }
    if (m) {
        const int32_t e = (int32_t)(L2 + 32) - (int32_t)s;
        for (uint32_t w = (x0 >> 5) + lane; w <= (x1 - 1) >> 5; w += 32) {
            for (uint32_t mm = ovl_mismatch_word(A, B, w, e, x0, x1); mm; mm &= mm - 1) {
                const uint32_t x = 32 * w + __ffs(mm) - 1;
                acc.add(a.L.m1 + x, 1);
                acc.add(a.L.m2 + s - 1 - x, 1);
            }
        }
    }
    __syncwarp();          // the planes are rewritten by the warp's next pair
}

// Dynamic shared memory (kSmem): the plane words of every warp, then the block's u32 copy of the accumulator block.
template <bool kSmem>
__global__ void __launch_bounds__(kOvlThreads) k_overlap(const OverlapArgs a)
{
    extern __shared__ uint4 ovl_smem[];
    const uint32_t lane = threadIdx.x & 31, wpb = blockDim.x >> 5, warp = threadIdx.x >> 5;
    uint32_t *cnt = reinterpret_cast<uint32_t *>(ovl_smem + (size_t)wpb * a.plane_words);
    uint4 *A = kSmem ? ovl_smem + (size_t)warp * a.plane_words : a.scratch + ((size_t)blockIdx.x * wpb + warp) * a.plane_words;
    const OvlAcc<kSmem> acc{cnt, a.acc};
    if (kSmem) {
        for (uint32_t i = threadIdx.x; i < a.L.total; i += blockDim.x) cnt[i] = 0;
        __syncthreads();
    }
    for (uint32_t p = blockIdx.x * wpb + warp; p < a.n_rec; p += gridDim.x * wpb) ovl_pair<kSmem>(a, acc, A, p, lane);
    if (kSmem) {
        __syncthreads();
        // the difference arrays [d1, m1) hold signed counts (a block's pairs are far fewer than 2^31); every other entry is a
        // plain count
        for (uint32_t i = threadIdx.x; i < a.L.total; i += blockDim.x)
            if (cnt[i]) atomicAdd(a.acc + i, i >= a.L.d1 && i < a.L.m1 ? (unsigned long long)(long long)(int32_t)cnt[i] : (unsigned long long)cnt[i]);
    }
}

}  // namespace fq
