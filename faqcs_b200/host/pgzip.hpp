// pgzip.hpp -- parallel inflate of ORDINARY gzip members (SURVEY 8(f) N1), on top of zlib.
//
// A deflate stream has no index, but it can be entered at any block boundary if the 32 KiB of output in front of it are
// known.  Here they are not known yet, so a chunk that starts in the middle of the stream is inflated twice with two
// different 32 KiB "marker" dictionaries: a byte of the output that is the same in both runs is a literal of the chunk,
// a byte that differs was copied (through any chain of matches) from position p of the unknown window, and the pair of
// values spells p.  Once the chunk in front has been resolved, its last 32 KiB are that window and the markers are
// replaced.  (The idea of resolving back-references after the fact is pugz's; the marker pair lets an unmodified zlib do
// the decoding.)
//
// Entering the stream: a candidate bit position must look like the header of a dynamic-Huffman block (block type, code
// counts, a COMPLETE code-length code: about one random position in 500 passes) and then inflate through two whole blocks.
// A false start cannot do harm: chunk i is only accepted if the chunk in front of it ends EXACTLY on chunk i's first bit
// (zlib reports block boundaries with Z_BLOCK), otherwise the stream is inflated on from where the accepted output ends;
// and every member's CRC-32 and length are checked as gzip defines them.
#pragma once
#include <zlib.h>

#include <algorithm>
#include <cstdint>
#include <cstring>
#include <memory>
#include <vector>

#include "fork_join.hpp"

namespace pgz {

constexpr size_t kWin = 32768;

// marker pair of window position p (0 = oldest byte, 32767 = the byte right in front of the chunk): a != b, injective
inline void marker_dictionaries(uint8_t *A, uint8_t *B)
{
    for (uint32_t p = 0; p < kWin; ++p) {
        const uint32_t a = p / 255, b0 = p % 255;
        A[p] = (uint8_t)a;
        B[p] = (uint8_t)(b0 >= a ? b0 + 1 : b0);
    }
}
inline uint32_t marker_position(uint8_t a, uint8_t b) { return (uint32_t)a * 255u + (b > a ? (uint32_t)b - 1u : (uint32_t)b); }

inline uint32_t peek_bits(const uint8_t *buf, size_t n, size_t bit, int count)       // LSB first, as deflate packs them
{
    uint64_t v = 0;
    const size_t byte = bit >> 3;
    for (int k = 0; k < 8 && byte + k < n; ++k) v |= (uint64_t)buf[byte + k] << (8 * k);
    return (uint32_t)((v >> (bit & 7)) & ((1ull << count) - 1));
}

// Header of a non-final dynamic block with a complete code-length code at this bit? (RFC 1951 3.2.7)
inline bool plausible_block_start(const uint8_t *buf, size_t n, size_t bit)
{
    if ((bit >> 3) + 12 > n) return false;
    if (peek_bits(buf, n, bit, 3) != 4u) return false;                  // BFINAL = 0, BTYPE = 2 (bits: 0, then 0 1)
    const uint32_t hlit = peek_bits(buf, n, bit + 3, 5), hdist = peek_bits(buf, n, bit + 8, 5), hclen = peek_bits(buf, n, bit + 13, 4) + 4;
    if (hlit > 29 || hdist > 29) return false;
    uint32_t kraft = 0, used = 0;
    for (uint32_t i = 0; i < hclen; ++i) {
        const uint32_t len = peek_bits(buf, n, bit + 17 + 3 * i, 3);
        if (len) { kraft += 128u >> len; ++used; }
    }
    return used >= 2 && kraft == 128u;                                    // complete prefix code (zlib rejects anything else)
}

enum class End { Boundary, StreamEnd, InputEnd, Error };

// Output bytes of one run: grows without zeroing (zlib overwrites every byte it reports).
struct Bytes {
    std::unique_ptr<uint8_t[]> p;
    size_t cap = 0, n = 0;
    uint8_t *data() { return p.get(); }
    const uint8_t *data() const { return p.get(); }
    size_t size() const { return n; }
    void reserve(size_t want)
    {
        if (want <= cap) return;
        std::unique_ptr<uint8_t[]> q(new uint8_t[want]);
        if (n) memcpy(q.get(), p.get(), n);
        p = std::move(q);
        cap = want;
    }
    void release() { p.reset(); cap = n = 0; }
};

struct Piece {
    size_t start_bit = 0, end_bit = 0;      // compressed range decoded: [start_bit, end_bit), end on a block boundary
    End end = End::Error;
    Bytes out, out_b;                       // out_b: the second marker run (empty for a run with the true window)
};

// Inflate raw deflate data from bit `start_bit` of comp[0..n) with dictionary dict[0..dict_len).  Stops at the first block
// boundary at or after `stop_bit`, at the end of the deflate stream, or -- when the input runs out -- at the last boundary
// seen (partial output is dropped).  max_blocks > 0: stop after that many blocks (start validation).
inline End inflate_from(const uint8_t *comp, size_t n, size_t start_bit, size_t stop_bit, const uint8_t *dict, size_t dict_len, int max_blocks,
                        Bytes &out, size_t &end_bit, size_t expect = 0)
{
    z_stream zs;
    memset(&zs, 0, sizeof(zs));
    if (inflateInit2(&zs, -15) != Z_OK) return End::Error;
    End result = End::Error;
    size_t byte = start_bit >> 3;
    const int k = (int)(start_bit & 7);
    bool ok = true;
    if (dict_len) ok = inflateSetDictionary(&zs, dict, (uInt)dict_len) == Z_OK;
    if (ok && k) {
        if (byte >= n) ok = false;
        else { ok = inflatePrime(&zs, 8 - k, comp[byte] >> k) == Z_OK; ++byte; }
    }
    const uint8_t *const in0 = comp + byte;
    size_t in_left = n - std::min(n, byte);
    zs.next_in = const_cast<uint8_t *>(in0);
    size_t produced = 0, last_out = 0, last_bit = start_bit;
    bool have_boundary = false;
    int blocks = 0;
    out.n = 0;
    out.reserve(std::max<size_t>(expect, 1u << 16));
    while (ok) {
        if (zs.avail_in == 0 && in_left) { const size_t take = std::min<size_t>(in_left, 1u << 30); zs.avail_in = (uInt)take; in_left -= take; }
        if (produced == out.cap) { out.n = produced; out.reserve(out.cap + out.cap / 2); }
        zs.next_out = out.data() + produced;
        const size_t room = std::min<size_t>(out.cap - produced, 1u << 30);
        zs.avail_out = (uInt)room;
        const int rc = inflate(&zs, Z_BLOCK);
        produced += room - zs.avail_out;
        if (rc == Z_STREAM_END) {
            end_bit = 8 * (size_t)(zs.next_in - comp);               // the trailer starts at the next byte boundary
            last_out = produced;
            result = End::StreamEnd;
            break;
        }
        if (rc != Z_OK && rc != Z_BUF_ERROR) break;                   // data error: not a deflate stream from here
        if ((zs.data_type & 128) && !(zs.data_type & 64) ) {
            // just finished a block (not inside the last one): bits still unused in the last byte taken = data_type & 7...63
            const size_t bit = 8 * (size_t)(zs.next_in - comp) - (size_t)(zs.data_type & 63);
            have_boundary = true;
            last_bit = bit;
            last_out = produced;
            ++blocks;
            if (bit >= stop_bit || (max_blocks > 0 && blocks >= max_blocks)) { end_bit = bit; result = End::Boundary; break; }
        }
        if (zs.avail_in == 0 && in_left == 0 && zs.avail_out != 0) {     // the input ran out inside a block
            if (have_boundary) { end_bit = last_bit; result = End::InputEnd; }
            else { end_bit = start_bit; last_out = 0; result = End::InputEnd; }
            break;
        }
    }
    inflateEnd(&zs);
    out.n = result == End::Error ? 0 : last_out;
    return result;
}

// What one zlib stream still gets out of a deflate stream that is cut short (a truncated file): everything up to the last
// byte present, as gzread hands it out before it reports the end of the file.  False: the data are not deflate data.
inline bool inflate_truncated_tail(const uint8_t *comp, size_t n, size_t start_bit, const uint8_t *dict, size_t dict_len, Bytes &out)
{
    z_stream zs;
    memset(&zs, 0, sizeof(zs));
    if (inflateInit2(&zs, -15) != Z_OK) return false;
    size_t byte = start_bit >> 3;
    const int k = (int)(start_bit & 7);
    bool ok = true;
    if (dict_len) ok = inflateSetDictionary(&zs, dict, (uInt)dict_len) == Z_OK;
    if (ok && k && byte < n) { ok = inflatePrime(&zs, 8 - k, comp[byte] >> k) == Z_OK; ++byte; }
    zs.next_in = const_cast<uint8_t *>(comp + std::min(byte, n));
    zs.avail_in = (uInt)(n - std::min(byte, n));
    out.n = 0;
    out.reserve(std::max<size_t>(6 * n, 1u << 16));
    size_t produced = 0;
    while (ok) {
        if (produced == out.cap) { out.n = produced; out.reserve(out.cap + out.cap / 2); }
        zs.next_out = out.data() + produced;
        const size_t room = std::min<size_t>(out.cap - produced, 1u << 30);
        zs.avail_out = (uInt)room;
        const int rc = inflate(&zs, Z_SYNC_FLUSH);
        produced += room - zs.avail_out;
        if (rc == Z_STREAM_END) break;
        if (rc == Z_BUF_ERROR || (rc == Z_OK && zs.avail_in == 0 && zs.avail_out != 0)) break;      // the input is used up
        if (rc != Z_OK) { ok = false; break; }
    }
    inflateEnd(&zs);
    out.n = ok ? produced : 0;
    return ok;
}

// First bit at or after `from_bit` (and before `limit_bit`) where a dynamic block starts and two blocks inflate cleanly.
inline size_t find_block_start(const uint8_t *comp, size_t n, size_t from_bit, size_t limit_bit, const uint8_t *dict)
{
    Bytes scratch;
    for (size_t bit = from_bit; bit < limit_bit; ++bit) {
        if (!plausible_block_start(comp, n, bit)) continue;
        size_t end = 0;
        const End e = inflate_from(comp, n, bit, ~(size_t)0, dict, kWin, 2, scratch, end);
        if (e == End::Boundary || e == End::StreamEnd) return bit;
    }
    return ~(size_t)0;
}

// Replace the markers of a speculative piece: out[j] (run A) and out_b[j] (run B) agree on literals; where they differ the
// byte is window[position], window = the 32 KiB of true output in front of the piece (shorter at the start of a member:
// aligned to the END of the window array).
inline void resolve(uint8_t *a, const uint8_t *b, size_t n, const uint8_t *window)
{
    for (size_t j = 0; j < n; ++j)
        if (a[j] != b[j]) a[j] = window[marker_position(a[j], b[j])];
}

// The last 32 KiB of `prev_window` followed by `out` (what a piece after them sees as its window).
inline void slide_window(std::vector<uint8_t> &window, const uint8_t *out, size_t n)
{
    if (n >= kWin) { memcpy(window.data(), out + n - kWin, kWin); return; }
    memmove(window.data(), window.data() + n, kWin - n);
    memcpy(window.data() + kWin - n, out, n);
}

struct Result {
    std::vector<Piece> pieces;      // accepted, resolved, in stream order (out holds true bytes)
    size_t end_bit = 0;             // where the accepted output ends in the compressed buffer
    bool stream_end = false;        // the deflate stream of the member ended there (end_bit is byte aligned)
    bool error = false;
};

// Inflate as much of comp[0..n) as ends on a block boundary, starting at `start_bit` with the true `window` (32 KiB, the valid
// part aligned to its end, `window_len` bytes of it valid).  `threads` pieces are tried in parallel.
inline Result inflate_parallel(const uint8_t *comp, size_t n, size_t start_bit, std::vector<uint8_t> &window, size_t window_len, int threads,
                               size_t min_piece = 256u << 10)
{
    Result R;
    static const struct Dicts { uint8_t A[kWin], B[kWin]; Dicts() { marker_dictionaries(A, B); } } D;
    const size_t total_bits = 8 * n;
    const int T = (int)std::max<size_t>(1, std::min<size_t>((size_t)threads, (n - (start_bit >> 3)) / std::max<size_t>(min_piece, 64)));   // >= 256 KiB per piece
    std::vector<size_t> start(T, ~(size_t)0);
    start[0] = start_bit;
    // the first piece knows its window and is inflated once, the others twice: it gets two shares of the span
    const size_t span = (total_bits - start_bit) / (T + 1);
    // 1. entry points of the pieces (blocks of a FASTQ file are tens of KiB of compressed data: a piece whose first quarter holds
    // no entry point is left to the piece in front of it)
    fork_join(T - 1, [&](int j) {
        const int i = j + 1;
        start[i] = find_block_start(comp, n, (start_bit + span * (i + 1) + 7) & ~(size_t)7, start_bit + span * (i + 1) + span / 4, D.A);
    });
    std::vector<int> idx;           // pieces with an entry point, in order
    for (int i = 0; i < T; ++i)
        if (start[i] != ~(size_t)0 && (idx.empty() || start[i] > start[idx.back()])) idx.push_back(i);
    std::vector<Piece> P(idx.size());
    // 2. every piece up to the entry point of the next one; the first with the true window, the others with both marker sets
    fork_join((int)idx.size(), [&](int q) {
        Piece &pc = P[q];
        pc.start_bit = start[idx[q]];
        const size_t stop = q + 1 < (int)idx.size() ? start[idx[q + 1]] : ~(size_t)0;
        const size_t guess = ((std::min(stop, total_bits) - pc.start_bit) >> 3) * 5 + (1u << 16);      // FASTQ deflates 2-4.5 x
        if (q == 0) pc.end = inflate_from(comp, n, pc.start_bit, stop, window.data() + (kWin - window_len), window_len, 0, pc.out, pc.end_bit, guess);
        else {
            pc.end = inflate_from(comp, n, pc.start_bit, stop, D.A, kWin, 0, pc.out, pc.end_bit, guess);
            size_t end_b = 0;
            const End eb = inflate_from(comp, n, pc.start_bit, stop, D.B, kWin, 0, pc.out_b, end_b, pc.out.size() + 64);
            if (eb != pc.end || end_b != pc.end_bit || pc.out_b.size() != pc.out.size()) pc.end = End::Error;
        }
    });
    // 3. stitch: a piece counts only if the accepted output ends exactly on its first bit
    if (P[0].end == End::Error) { R.error = true; return R; }
    size_t accepted = 1;
    while (accepted < P.size() && P[accepted - 1].end == End::Boundary && P[accepted - 1].end_bit == P[accepted].start_bit && P[accepted].end != End::Error) ++accepted;
    P.resize(accepted);
    // 4. windows in front of the accepted pieces (a chain over their last 32 KiB), then the markers of every piece
    std::vector<std::vector<uint8_t>> win(accepted);
    std::vector<uint8_t> w = window;
    for (size_t q = 0; q < accepted; ++q) {
        win[q] = w;
        Piece &pc = P[q];
        const size_t nq = pc.out.size(), tail = std::min(nq, kWin);
        if (q > 0) resolve(pc.out.data() + (nq - tail), pc.out_b.data() + (nq - tail), tail, win[q].data());
        // a marker in the tail may point at a byte of this piece's own window only: positions are relative to win[q]
        slide_window(w, pc.out.data(), nq);
    }
    fork_join((int)accepted - 1, [&](int j) {
        Piece &pc = P[j + 1];
        const size_t nq = pc.out.size(), tail = std::min(nq, kWin);
        resolve(pc.out.data(), pc.out_b.data(), nq - tail, win[j + 1].data());
        pc.out_b.release();
    });
    window = w;
    R.end_bit = P.back().end_bit;
    R.stream_end = P.back().end == End::StreamEnd;
    R.pieces = std::move(P);
    return R;
}

}  // namespace pgz
