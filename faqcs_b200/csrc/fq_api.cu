// fq_api.cu -- C ABI (include/faqcs_b200.h) over the sm_100a kernels.
//
// One fq_ctx = one CUDA device + one stream + the run's accumulators (the
// filter_stats / adaptor_stats / PlotInfo trio main() owns, FaQCs.cpp:67-69).
// A batch goes through: frame -> [pair-id check] -> [adapter pass] -> trim ->
// route -> scan -> emit.  There is no CPU implementation of any of these steps
// in this library: without a CUDA device fq_create fails.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <nccl.h>          // types and enums only: the library is loaded with dlopen, not linked

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <utility>
#include <vector>

#include "fq_adapter.cuh"
#include "fq_common.cuh"
#include "fq_dup.cuh"
#include "fq_emit.cuh"
#include "fq_frame.cuh"
#include "fq_kmer.cuh"
#include "fq_overlap.cuh"
#include "fq_overrep.cuh"
#include "fq_tile_qual.cuh"
#include "fq_trim.cuh"

using namespace fq;

#define FQ_STR2(x) #x
#define FQ_STR(x) FQ_STR2(x)

namespace {

std::string g_create_error;

// Device (cudaMalloc) or pinned host (cudaMallocHost) memory with one owner: move-only, freed by its destructor.
// ensure() grows it with 1/8 headroom and does not keep the contents.
template <bool Pinned>
struct Buf {
    void *p = nullptr;
    size_t cap = 0;
    Buf() = default;
    Buf(const Buf &) = delete;
    Buf &operator=(const Buf &) = delete;
    Buf(Buf &&o) noexcept : p(std::exchange(o.p, nullptr)), cap(std::exchange(o.cap, 0)) {}
    Buf &operator=(Buf &&o) noexcept
    {
        if (this != &o) {
            release();
            p = std::exchange(o.p, nullptr);
            cap = std::exchange(o.cap, 0);
        }
        return *this;
    }
    ~Buf() { release(); }
    cudaError_t ensure(size_t bytes)
    {
        if (bytes <= cap) return cudaSuccess;
        release();
        const size_t want = bytes + bytes / 8 + 256;
        cudaError_t e = Pinned ? cudaMallocHost(&p, want) : cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release()
    {
        if (p) {
            if (Pinned) cudaFreeHost(p);
            else cudaFree(p);
        }
        p = nullptr;
        cap = 0;
    }
    template <class T> T *as() const { return reinterpret_cast<T *>(p); }
};
using DevBuf = Buf<false>;
using HostBuf = Buf<true>;

// An open-addressing table of KmerSlot in device memory (fq_kmer.cuh) with the buffers of its end-of-pass exchange: the k-mer
// table, the duplication table and the overrepresented-sequence count table of a context.
struct HashTable {
    unsigned long long min_cap = 1ull << 20;       // slots of a new table (a power of two)
    unsigned long long cap = 0, occupied_bound = 0;
    DevBuf d_slots, d_scalars;
    DevBuf d_send, d_recv;                         // end of a sharded pass: entries grouped by owner, one received group
};

const char *kPhiX = "__PhiX174_NC_001422__";                       // FaQCs.h:29-30
const char *kPhiXComplement = "__PhiX174_NC_001422_complement__";

int na_bits_host(char c)
{
    switch (c | 0x20) {
        case 'a': return 1;  case 'c': return 2;  case 'g': return 4;  case 't': return 8;
        case 'm': return 3;  case 'r': return 5;  case 's': return 6;  case 'v': return 7;
        case 'w': return 9;  case 'y': return 10; case 'h': return 11; case 'k': return 12;
        case 'd': return 13; case 'b': return 14; case 'n': return 15;
        default: return c == '-' ? 16 : -1;
    }
}

}  // namespace

struct fq_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    fq_options opt{};
    DevOpts dopt{};
    std::vector<std::string> adapter_names, adapter_seqs;
    AdapterSet aset{};
    DevBuf d_adp_codes, d_adp_off, d_adp_or;

    DevBuf d_raw[2], d_chunk[2], d_nl[2], d_rec[2], d_canon[2], d_adp[2], d_adp_best[2], d_res[2], d_dbg[2], d_tile, d_out[2][4];
    DevBuf d_raw_slot[2][2];           // pipelined submit: raw input slots
    DevBuf d_info, d_stats, d_rows;
    HostBuf h_info;                    // one BatchInfo
    StatsLayout L{};
    HostBuf h_out[2][4], h_dbg[2], h_stats, h_pieces[2][4];
    DevBuf d_pieces[2][4];
    bool pieces = false;               // fq_set_output_pieces
    cudaStream_t s_in = nullptr, s_out = nullptr;
    cudaEvent_t ev_in[2] = {nullptr, nullptr}, ev_comp[2] = {nullptr, nullptr}, ev_out[2] = {nullptr, nullptr};
    // pipelined path: an input slot is busy from submit until run returns, an output slot from run until wait
    struct Submitted { bool busy = false; size_t n1 = 0, n2 = 0; bool paired = false; uint64_t first = 0; int is_final = 0; uint64_t ticket = 0; } sub[2];
    struct Finished { bool busy = false; uint64_t ticket = 0; fq_batch_out out{}; } fin[2];
    uint64_t next_ticket = 0;
    bool debug_results = false;
    bool check_pair_ids = true;
    bool frame_exact[2] = {false, false};      // this mate's input is not plain LF text: skip the fast framing instance

    // k-mer rarefaction (fq_kmer_*): Options::kmer_rarefaction / kmer / split_size / num_subsample, PlotInfo::kmer_*
    struct Kmer {
        bool enabled = false, collecting = false;
        uint32_t k = 31, num_subsample = 0;
        uint64_t split_size = 1;
        uint64_t total_reads = 0;                  // TOTAL_NUMBER
        std::vector<fq_rarefaction> samples;       // finished points
        std::map<uint64_t, uint64_t> freq;         // kmer_frequency_histogram
        // current pass: what this context's batches covered (call numbers follow from first_record_index)
        std::vector<uint64_t> call_reads;          // [kKmerMaxCalls] reads of each call run here
        std::vector<uint64_t> call_runs;           // [kKmerMaxCalls] times each call was run here
        uint64_t calls_beyond = 0;                 // calls >= kKmerMaxCalls run here (the curve is complete by then)
        uint64_t call_end = 0;                     // 1 + the highest call run here
        uint64_t pass_reads = 0;
        HashTable T;
        DevBuf d_call_total, d_call_distinct, d_small, d_big;
        std::vector<uint64_t> flat;                // fq_kmer_view::frequency
    } kmer;

    // duplication statistics (fq_dup_*, fq_dup.cuh): one key per read or pair
    struct Dup {
        bool enabled = false;
        uint32_t n_mates = 0;                      // mates per unit in the current pass (0: no batch yet)
        uint64_t units = 0;                        // units of the current pass counted here
        HashTable T{1ull << 16};                   // small, so that modest inputs already exercise the growth
        DevBuf d_small, d_big;                     // end of a pass: the histogram of counts
        uint64_t res_units = 0, res_distinct = 0;  // the last finished pass (fq_dup_view)
        std::vector<uint64_t> levels;
    } dup;

    // insert size and overlap error profile (fq_overlap_*, fq_overlap.cuh): per-pair overlap of R1 with reverse-complemented R2
    struct Overlap {
        bool enabled = false;
        uint32_t min_overlap = 30, diff_limit = 5, diff_percent = 20;
        uint32_t cyc = 0;                          // cycle capacity of d_acc (OverlapLayout; 0: nothing allocated yet)
        uint64_t pairs = 0;                        // pairs of the current pass counted here
        DevBuf d_acc, d_scratch;
        // the last finished pass (fq_overlap_view): scalars, insert-size histogram, per-cycle arrays
        uint64_t res[kOvlPairs + 1] = {};
        std::vector<uint64_t> ins, r1o, r1m, r2o, r2m;
    } ovl;

    // overrepresented sequences (fq_overrep_*, fq_overrep.cuh): one key per read's prefix, the bytes in a capture store
    struct Overrep {
        bool enabled = false;
        uint32_t prefix_len = 50, min_ppm = 1000;
        uint64_t reads[2] = {0, 0};                // mate-m reads of the current pass counted here
        HashTable T{1ull << 16};
        DevBuf d_store, d_sel;                     // capture store (OverrepStore); end of a pass: the selected slots
        uint64_t store_cap = 0, store_bound = 0;   // entries, and a bound on the occupied ones
        // the last finished pass (fq_overrep_view)
        uint32_t res_prefix_len = 50, res_min_ppm = 1000;
        uint64_t res_reads[2] = {0, 0}, res_min_count[2] = {2, 2};
        std::vector<fq_overrep_seq> seqs;
        std::vector<uint8_t> bytes;
    } ovr;

    // per flowcell tile quality (fq_tile_qual_*, fq_tile_qual.cuh): a key table and an accumulator block per context
    struct TileQual {
        bool enabled = false;
        uint32_t n_mates = 0;                      // mates of the current pass's batches (0: no batch yet)
        uint64_t reads[2] = {0, 0};                // reads of the current pass counted here
        uint32_t longest = 0;                      // longest read of the current pass here
        uint32_t claims = 0, overflow = 0;         // TileCounters after the last batch
        // a batch counted its keys and has not returned FQ_OK yet; set when the next batch starts: a batch of this pass
        // failed part-way (its keys are in the table, its reads only partly counted), so the pass has no result
        bool batch_open = false, failed = false;
        TileLayout L{0, 0};                        // of d_acc (D == 0: nothing allocated yet)
        DevBuf d_slots, d_cnt, d_id[2], d_acc;
        HostBuf h_cnt;                             // {claims, overflow}, read back with the batch's BatchInfo
        // the last finished pass (fq_tile_qual_view)
        uint32_t res_mates = 0, res_overflow = 0, res_cycles = 0;
        uint64_t res_reads[2] = {0, 0}, res_untiled[2] = {0, 0};
        std::vector<uint32_t> lane, tile;
        std::vector<uint64_t> t_reads, t_bases, t_qsum, c_bases, c_qsum;
    } tq;

    // host-side stats views handed out by fq_stats
    std::vector<uint64_t> v_adapter_reads, v_adapter_bases, v_pre_q, v_post_q, v_pre_b, v_post_b, v_hist[4], v_pre_comp,
        v_post_comp, v_pre_len, v_post_len;

    std::string error;
    uint64_t launches = 0;
    cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};
    float t_seg[5] = {0, 0, 0, 0, 0};
    int sm_count = 0;
    size_t smem_optin = 0;
    float allreduce_ms = 0.0f;
    const void *last_dev_out[4] = {nullptr, nullptr, nullptr, nullptr};

    // The buffers free themselves after this; fq_destroy makes the device current first.
    ~fq_ctx()
    {
        for (cudaEvent_t e : {ev_in[0], ev_in[1], ev_comp[0], ev_comp[1], ev_out[0], ev_out[1], ev[0], ev[1], ev[2], ev[3], ev[4]})
            if (e) cudaEventDestroy(e);
        for (cudaStream_t s : {s_in, s_out, stream})
            if (s) cudaStreamDestroy(s);
    }
};

namespace {

fq_status fail(fq_ctx *c, fq_status code, const std::string &msg)
{
    if (c) c->error = msg; else g_create_error = msg;
    return code;
}

#define CK(call)                                                                                           \
    do {                                                                                                   \
        cudaError_t e__ = (call);                                                                          \
        if (e__ != cudaSuccess)                                                                            \
            return fail(ctx, FQ_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));           \
    } while (0)

uint32_t round_up(uint32_t v, uint32_t m) { return (v + m - 1) / m * m; }

// (Re)allocate the stats block for at least `rows` position rows, keeping the contents.
// The dynamic shared-memory limit of a kernel is state of the device's (primary) CUDA context, shared by every fq_ctx on
// that device -- and contexts on one device run on different host threads.  It is therefore raised ONCE per kernel and
// device to the opt-in maximum and never lowered: a per-launch value would race with the other context's launch.
cudaError_t allow_dynamic_smem(fq_ctx *ctx, const void *kernel)
{
    static std::mutex mu;
    static std::map<std::pair<int, const void *>, bool> done;
    std::lock_guard<std::mutex> lk(mu);
    bool &d = done[std::make_pair(ctx->device, kernel)];
    if (d) return cudaSuccess;
    cudaFuncAttributes fa{};
    cudaError_t e = cudaFuncGetAttributes(&fa, kernel);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(ctx->smem_optin - fa.sharedSizeBytes));      // static + dynamic <= opt-in
    if (e == cudaSuccess) d = true;
    return e;
}

__global__ void __launch_bounds__(256) k_merge_stats(unsigned long long *dst, unsigned long long *src, size_t n, uint32_t *dst_rows, uint32_t *src_rows)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        dst[i] += src[i];
        src[i] = 0;
    }
    if (blockIdx.x == 0 && threadIdx.x < 4) {
        dst_rows[threadIdx.x] = max(dst_rows[threadIdx.x], src_rows[threadIdx.x]);
        src_rows[threadIdx.x] = 0;
    }
}

fq_status ensure_stats_rows(fq_ctx *ctx, uint32_t rows)
{
    rows = std::max(64u, round_up(rows, 64));
    if (ctx->d_stats.p && rows <= ctx->L.rows) return FQ_OK;
    const StatsLayout oldL = ctx->L;
    const StatsLayout newL = StatsLayout::make(rows, ctx->opt.n_adapters);
    std::vector<unsigned long long> oldv, newv(newL.total, 0);
    if (ctx->d_stats.p) {
        oldv.resize(oldL.total);
        CK(cudaStreamSynchronize(ctx->stream));
        CK(cudaMemcpy(oldv.data(), ctx->d_stats.p, oldL.total * 8, cudaMemcpyDeviceToHost));
        auto copy = [&](size_t so, size_t dso, size_t n) { std::copy(oldv.begin() + so, oldv.begin() + so + n, newv.begin() + dso); };
        copy(oldL.filter, newL.filter, 32);
        copy(oldL.adapter_reads, newL.adapter_reads, oldL.n_adapters);
        copy(oldL.adapter_bases, newL.adapter_bases, oldL.n_adapters);
        copy(oldL.pre_rq, newL.pre_rq, 4 * kQualCols);
        copy(oldL.pre_comp, newL.pre_comp, 12 * (size_t)kCompBins);
        for (int c = 0; c < kQualCols; ++c) {
            copy(oldL.pre_q + (size_t)c * oldL.rows, newL.pre_q + (size_t)c * newL.rows, oldL.rows);
            copy(oldL.rem_q + (size_t)c * oldL.rows, newL.rem_q + (size_t)c * newL.rows, oldL.rows);
        }
        for (int c = 0; c < kBaseCols; ++c) {
            copy(oldL.pre_b + (size_t)c * oldL.rows, newL.pre_b + (size_t)c * newL.rows, oldL.rows);
            copy(oldL.rem_b + (size_t)c * oldL.rows, newL.rem_b + (size_t)c * newL.rows, oldL.rows);
        }
        copy(oldL.g2n, newL.g2n, oldL.rows);
        copy(oldL.pre_len, newL.pre_len, oldL.rows + 1);
        copy(oldL.post_len, newL.post_len, oldL.rows + 1);
    }
    DevBuf nb;
    CK(nb.ensure(newL.total * 8));
    CK(cudaMemcpy(nb.p, newv.data(), newL.total * 8, cudaMemcpyHostToDevice));
    ctx->d_stats = std::move(nb);
    ctx->L = newL;
    return FQ_OK;
}

fq_status upload_adapters(fq_ctx *ctx)
{
    const uint32_t n = ctx->opt.n_adapters;
    std::vector<uint8_t> codes, orb(n ? n : 1, 0);
    std::vector<uint32_t> off(n + 1, 0);
    for (uint32_t j = 0; j < n; ++j) {
        off[j] = (uint32_t)codes.size();
        for (char ch : ctx->adapter_seqs[j]) {
            const int b = na_bits_host(ch);
            if (b < 0) return fail(ctx, FQ_ERR_BASE, "seq_overlap.cpp:na_to_bits: Unknown base!");
            codes.push_back((uint8_t)b);
            orb[j] |= (uint8_t)b;
        }
    }
    off[n] = (uint32_t)codes.size();
    CK(ctx->d_adp_codes.ensure(codes.size() + 16));
    CK(ctx->d_adp_off.ensure(off.size() * 4));
    CK(ctx->d_adp_or.ensure(orb.size()));
    if (!codes.empty()) CK(cudaMemcpy(ctx->d_adp_codes.p, codes.data(), codes.size(), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(ctx->d_adp_off.p, off.data(), off.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(ctx->d_adp_or.p, orb.data(), orb.size(), cudaMemcpyHostToDevice));
    ctx->aset.codes = ctx->d_adp_codes.as<uint8_t>();
    ctx->aset.offset = ctx->d_adp_off.as<uint32_t>();
    ctx->aset.or_bits = ctx->d_adp_or.as<uint8_t>();
    ctx->aset.n = n;
    ctx->aset.total = (uint32_t)codes.size();
    ctx->aset.any_bits = 0;
    return FQ_OK;
}

void refresh_dev_opts(fq_ctx *ctx)
{
    const fq_options &o = ctx->opt;
    DevOpts &d = ctx->dopt;
    d.mode = o.mode;
    d.quality = (int)(signed char)o.quality;
    d.trim_5 = o.trim_5;
    d.trim_3 = o.trim_3;
    d.min_len = o.min_read_length;
    d.max_poly_n = o.max_num_poly_N;
    d.avg_q = o.average_quality;
    d.lc = o.low_complexity_cutoff_ratio;
    d.match_rate = (float)(1.0 - (double)o.adapter_mismatch_rate);     // trim.cpp:969
    d.in_off = (int)(signed char)o.input_quality_offset;
    d.out_off = (int)(signed char)o.output_quality_offset;
    d.replace_q = o.replace_to_N_q;
    d.qc_only = o.qc_only;
    d.protect_5 = o.protect_5;
    d.filter_adapter = o.filter_adapter && o.n_adapters > 0;
    d.discard = o.discard_output;
    d.num_thread = o.num_thread;
    d.n_adapters = o.n_adapters;
}

// A fresh BatchInfo on the device, through the pinned mirror, ahead of the batch's kernels.
cudaError_t reset_info(fq_ctx *ctx)
{
    BatchInfo init{};
    init.err_record = 0xffffffffu;
    init.detect_key = ~0ull;
    *ctx->h_info.as<BatchInfo>() = init;
    return cudaMemcpyAsync(ctx->d_info.p, ctx->h_info.p, sizeof(BatchInfo), cudaMemcpyHostToDevice, ctx->stream);
}

// The device's BatchInfo once the stream has caught up with it.
cudaError_t read_info(fq_ctx *ctx, BatchInfo *hi)
{
    cudaError_t e = cudaMemcpyAsync(ctx->h_info.p, ctx->d_info.p, sizeof(BatchInfo), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e == cudaSuccess) *hi = *ctx->h_info.as<BatchInfo>();
    return e;
}

// Every context's stream drained, each with its device current.  Like the rest of an entry point over several contexts,
// a failure is reported on ctxs[0].
fq_status sync_all(fq_ctx *const *ctxs, int n)
{
    fq_ctx *const ctx = ctxs[0];
    for (int i = 0; i < n; ++i) {
        CK(cudaSetDevice(ctxs[i]->device));
        CK(cudaStreamSynchronize(ctxs[i]->stream));
    }
    return FQ_OK;
}

// Framing of one mate: count -> scan -> (sync) -> scatter -> records.
fq_status frame_mate(fq_ctx *ctx, int m, const uint8_t *d_raw, size_t n, uint32_t *n_rec_out)
{
    *n_rec_out = 0;
    if (n == 0) return FQ_OK;
    if (n >= (1ull << 30)) return fail(ctx, FQ_ERR_ARG, "batch larger than 1 GiB per mate: split it");
    if ((reinterpret_cast<uintptr_t>(d_raw) & 15) != 0) return fail(ctx, FQ_ERR_ARG, "device input must be 16-byte aligned");
    BatchInfo *info = ctx->d_info.as<BatchInfo>();
    BatchInfo hi{};
    // single-pass segmented line index: one contiguous segment per resident warp, no cross-warp dependency
    int frame_ctas = 4;                                     // resident CTAs per SM -> exactly one wave of segments
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&frame_ctas, k_frame_lines<false>, kFrameThreads, 0));
    const uint32_t want_warps = (uint32_t)ctx->sm_count * (uint32_t)std::max(frame_ctas, 1) * (kFrameThreads / 32);
    uint32_t seg_bytes = (uint32_t)((n + want_warps - 1) / want_warps);
    seg_bytes = std::max<uint32_t>(kChunkBytes, (seg_bytes + kChunkBytes - 1) / kChunkBytes * kChunkBytes);
    const uint32_t n_seg = (uint32_t)((n + seg_bytes - 1) / seg_bytes);
    CK(ctx->d_chunk[m].ensure(((size_t)n_seg * 2 + 2) * 4));
    uint32_t *seg_count = ctx->d_chunk[m].as<uint32_t>();
    uint32_t *seg_base = seg_count + n_seg;
    uint32_t n_lines = 0;
    uint32_t seg_cap = seg_bytes / 24 + 64;                 // lines per segment region: >= 24 bytes per line on average
    for (int attempt = 0; attempt < 2; ++attempt) {
        CK(ctx->d_nl[m].ensure((size_t)n_seg * seg_cap * 4));
        const int grid = (n_seg + kFrameThreads / 32 - 1) / (kFrameThreads / 32);
        if (attempt) {
            CK(cudaMemsetAsync(&info->n_cr[m], 0, 4, ctx->stream));
            CK(cudaMemsetAsync(&info->n_cr_eol[m], 0, 4, ctx->stream));
            CK(cudaMemsetAsync(&info->seg_overflow, 0, 4, ctx->stream));
        }
        // the fast instance first (plain LF text); the exact instance redoes the mate only if the fast one met a control
        // character other than '\n' (CRLF input: remembered, later batches go straight to the exact instance)
        for (int pass = 0; pass < 2; ++pass) {
            const bool exact = ctx->frame_exact[m];
            if (exact) k_frame_lines<false><<<grid, kFrameThreads, 0, ctx->stream>>>(d_raw, n, seg_bytes, n_seg, ctx->d_nl[m].as<uint32_t>(), seg_cap, seg_count, info, m, 0);
            else k_frame_lines<true><<<grid, kFrameThreads, 0, ctx->stream>>>(d_raw, n, seg_bytes, n_seg, ctx->d_nl[m].as<uint32_t>(), seg_cap, seg_count, info, m, 0);
            k_scan_segments<<<1, 1024, 0, ctx->stream>>>(seg_count, n_seg, seg_base, info, m);
            ctx->launches += 2;
            CK(read_info(ctx, &hi));
            if (exact || !hi.frame_exact[m]) break;
            ctx->frame_exact[m] = true;                   // the fast instance gave up: run the exact one
        }
        n_lines = hi.n_lines[m];
        if (hi.seg_overflow == 0) break;
        seg_cap = hi.seg_overflow + 64;           // very short lines: repeat once with the exact need
    }
    const bool had_cr = hi.n_cr[m] != 0;
    if (had_cr) {
        // CRLF input (or stray CRs): exact CR count, to be compared with the CRs that sit right before a '\n'
        CK(cudaMemsetAsync(&info->n_cr[m], 0, 4, ctx->stream));
        k_count_byte<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(d_raw, n, '\r', &info->n_cr[m]);
        ctx->launches++;
    }
    if (n_lines % 4 != 0) {
        static const char *msg[4] = {"", "fastq.cpp:next_read: Unable to read sequence", "fastq.cpp:next_read: Unable to read '+'",
                                     "fastq.cpp:next_read: Unable to read quality"};
        return fail(ctx, FQ_ERR_FORMAT, msg[n_lines % 4]);
    }
    const uint32_t n_rec = n_lines / 4;
    if (n_rec == 0) return FQ_OK;
    CK(ctx->d_rec[m].ensure((size_t)n_rec * sizeof(Rec)));
    CK(ctx->d_canon[m].ensure((size_t)n_rec));
    const LineIndex li{ctx->d_nl[m].as<uint32_t>(), seg_base, seg_cap, n_seg};
    k_build_records<<<(n_rec + 255) / 256, 256, 0, ctx->stream>>>(li, n_rec, ctx->d_rec[m].as<Rec>(), ctx->d_canon[m].as<uint8_t>(), info, m);
    ctx->launches++;
    if (had_cr) {
        // exact CR count against the CRs that close a line: any other one cuts its line short (strpbrk, fastq.cpp:44)
        CK(read_info(ctx, &hi));
        if (hi.n_cr[m] != hi.n_cr_eol[m]) {
            // the lengths (and a possible |seq| != |qual| verdict) of k_build_records are void for such lines: redo them
            if ((hi.err & ~kErrLenMismatch) == 0) {
                const uint32_t zero = 0, none = 0xffffffffu;
                CK(cudaMemcpyAsync(&info->err, &zero, 4, cudaMemcpyHostToDevice, ctx->stream));
                CK(cudaMemcpyAsync(&info->err_record, &none, 4, cudaMemcpyHostToDevice, ctx->stream));
            }
            k_fix_lone_cr<<<(n_rec + 255) / 256, 256, 0, ctx->stream>>>(d_raw, ctx->d_rec[m].as<Rec>(), ctx->d_canon[m].as<uint8_t>(), n_rec, info, m);
            ctx->launches++;
        }
    }
    *n_rec_out = n_rec;
    return FQ_OK;
}

fq_status map_device_error(fq_ctx *ctx, const BatchInfo &hi)
{
    if (!hi.err) return FQ_OK;
    char where[64];
    snprintf(where, sizeof where, " (record %u)", hi.err_record);
    if (hi.err & kErrLenMismatch) return fail(ctx, FQ_ERR_FORMAT, std::string("fastq.cpp:next_read: |Sequence| != |Quality|") + where);
    if (hi.err & kErrPairId) return fail(ctx, FQ_ERR_FORMAT, std::string("FaQCs.cpp:trim: I/O error") + where);
    if (hi.err & kErrUnknownBase) return fail(ctx, FQ_ERR_BASE, std::string("seq_overlap.cpp:na_to_bits: Unknown base!") + where);
    if (hi.err & kErrQualGt41)
        return fail(ctx, FQ_ERR_QUALITY,
                    std::string("fastq.h:quality_score: Found a quality score value that is greater than the maximum allowed quality score") + where);
    if (hi.err & kErrReencode) return fail(ctx, FQ_ERR_QUALITY, std::string("trim.cpp: quality error!") + where);
    if (hi.err & kErrInternal) return fail(ctx, FQ_ERR_CUDA, "internal: a bulk copy did not complete");
    return fail(ctx, FQ_ERR_STATE, "unknown device error");
}

// ---- the hash tables (k-mer rarefaction, duplication statistics, overrepresented sequences): host side of fq_kmer.cuh ----
KmerTable table_of(const HashTable &T)
{
    return KmerTable{T.d_slots.as<KmerSlot>(), T.cap - 1};
}

// (Re)allocate the table for at least `slots` slots (a power of two), keeping its entries (or, with keep == false, empty).
fq_status table_resize(fq_ctx *ctx, HashTable &T, unsigned long long slots, bool keep = true)
{
    unsigned long long cap = T.min_cap;
    while (cap < slots) cap <<= 1;
    if (cap <= T.cap) return FQ_OK;
    if (!keep) {
        CK(cudaStreamSynchronize(ctx->stream));
        T.d_slots.release();
        T.cap = 0;
    }
    DevBuf ns;
    CK(ns.ensure(cap * sizeof(KmerSlot)));
    KmerTable to{ns.as<KmerSlot>(), cap - 1};
    k_kmer_clear<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(to);
    if (T.cap) k_kmer_rehash<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(table_of(T), to);
    ctx->launches += T.cap ? 2 : 1;
    CK(cudaStreamSynchronize(ctx->stream));
    T.d_slots = std::move(ns);
    T.cap = cap;
    return FQ_OK;
}

// Room for `adding` more keys at a load factor <= 1/2, before a batch; the bound on the occupied slots is made exact when it
// matters.
fq_status table_reserve(fq_ctx *ctx, HashTable &T, unsigned long long adding)
{
    unsigned long long need = T.occupied_bound + adding;
    if (2 * need > T.cap && T.cap) {
        CK(cudaMemsetAsync(T.d_scalars.p, 0, 16, ctx->stream));
        k_kmer_count<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(table_of(T), T.d_scalars.as<unsigned long long>());
        ctx->launches++;
        unsigned long long occ = 0;
        CK(cudaMemcpyAsync(&occ, T.d_scalars.p, 8, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        T.occupied_bound = occ;
        need = occ + adding;
    }
    if (2 * need > T.cap) {
        fq_status st = table_resize(ctx, T, 2 * need);
        if (st != FQ_OK) return st;
    }
    T.occupied_bound = need;
    return FQ_OK;
}

// The reference's sequence of trim() calls in one pass (trim.cpp:157-185), from the state at the start of the pass:
// reads(c) is the number of reads of call c.  A call feeds the table while the curve is collected (trim.cpp:260-262); at
// its end a point is taken if the running read count crossed another multiple of split_size.  The call that follows the
// last point still feeds the table: `collecting` is cleared only after the point is pushed.
struct KmerWalk {
    std::vector<std::pair<uint32_t, uint64_t>> points;     // (call, TOTAL_NUMBER)
    uint32_t counted = 0;                                  // calls [0, counted) feed the table
    bool collecting = false;                               // still collecting after the last call walked
};

template <class Reads>
fq_status kmer_walk(fq_ctx *ctx, const fq_ctx::Kmer &K, uint64_t n_calls, Reads reads, KmerWalk *w)
{
    w->points.clear();
    w->counted = 0;
    w->collecting = K.collecting;
    uint64_t total = K.total_reads;
    for (uint64_t call = 0; call < n_calls && w->collecting; ++call) {
        if (call >= kKmerMaxCalls) return fail(ctx, FQ_ERR_ARG, "k-mer rarefaction: more than 65536 trim() batches while the curve is collected");
        w->counted = (uint32_t)call + 1;
        total += reads((uint32_t)call);
        const uint64_t index = total / K.split_size;
        const uint64_t n_points = K.samples.size() + w->points.size();
        if (index > n_points && n_points < K.num_subsample) w->points.push_back(std::make_pair((uint32_t)call, total));
        if (n_points >= K.num_subsample) w->collecting = false;
    }
    return FQ_OK;
}

// One batch: which trim() calls of the reference it spans (from its position in the input, so batches may run in any order
// and on any context of a sharded table), which of them still feed the table, then the counting kernel.
fq_status kmer_batch(fq_ctx *ctx, const uint8_t *d_r1, const uint8_t *d_r2, uint32_t n, int n_mates, uint32_t max_len, uint64_t first_record_index, int is_final, bool trimmed)
{
    fq_ctx::Kmer &K = ctx->kmer;
    if ((first_record_index % FQ_REF_BATCH) != 0 || (!is_final && (n % FQ_REF_BATCH) != 0))
        return fail(ctx, FQ_ERR_ARG, "k-mer rarefaction needs batches that start on a 32768-record boundary and hold a multiple of 32768 records");
    // call = (first_record_index / 32768 + chunk) * n_mates + mate; only the final batch may end in a partial chunk, so every
    // call in front of this batch holds 32768 reads
    const uint64_t first_call = first_record_index / FQ_REF_BATCH * (uint64_t)n_mates;
    const uint64_t n_calls = (uint64_t)(n + FQ_REF_BATCH - 1) / FQ_REF_BATCH * (uint64_t)n_mates;
    auto reads_of = [&](uint64_t call) -> uint32_t {
        if (call < first_call) return FQ_REF_BATCH;
        const uint64_t b0 = (call - first_call) / (uint64_t)n_mates * FQ_REF_BATCH;
        return (uint32_t)std::min<uint64_t>(FQ_REF_BATCH, n - b0);
    };
    KmerWalk w;
    fq_status st = kmer_walk(ctx, K, first_call + n_calls, reads_of, &w);
    if (st != FQ_OK) return st;
    if (K.call_reads.size() != kKmerMaxCalls) {
        K.call_reads.assign(kKmerMaxCalls, 0);
        K.call_runs.assign(kKmerMaxCalls, 0);
    }
    uint64_t counted_reads = 0;
    for (uint64_t call = first_call; call < first_call + n_calls; ++call) {
        const uint32_t reads = reads_of(call);
        if (call < kKmerMaxCalls) {
            K.call_reads[call] += reads;
            K.call_runs[call] += 1;
        } else K.calls_beyond += 1;
        if (call < w.counted) counted_reads += reads;
        K.pass_reads += reads;
    }
    K.call_end = std::max(K.call_end, first_call + n_calls);
    if (w.counted <= first_call || counted_reads == 0) return FQ_OK;
    // room for every k-mer this batch can add
    const unsigned long long per_read = max_len >= K.k ? (unsigned long long)(max_len - K.k + 1) : 0ull;
    st = table_reserve(ctx, K.T, counted_reads * per_read);
    if (st != FQ_OK) return st;
    KmerArgs ka{};
    ka.raw[0] = d_r1; ka.raw[1] = d_r2;
    ka.rec[0] = ctx->d_rec[0].as<Rec>(); ka.rec[1] = ctx->d_rec[1].as<Rec>();
    ka.res[0] = trimmed ? ctx->d_res[0].as<uint2>() : nullptr;
    ka.res[1] = trimmed ? ctx->d_res[1].as<uint2>() : nullptr;
    ka.n_rec = n; ka.n_mates = (uint32_t)n_mates; ka.k = K.k;
    ka.replace_q = ctx->dopt.replace_q; ka.in_off = ctx->dopt.in_off;
    ka.first_call = (uint32_t)first_call; ka.stop_call = w.counted;
    ka.T = table_of(K.T);
    ka.call_total = K.d_call_total.as<unsigned long long>();
    k_kmer<<<(n * n_mates + 255) / 256, 256, 0, ctx->stream>>>(ka);
    ctx->launches++;
    return FQ_OK;
}

// One batch of duplication statistics: room for one key per unit, then one insert per unit.
fq_status dup_batch(fq_ctx *ctx, const uint8_t *d_r1, const uint8_t *d_r2, uint32_t n, int n_mates)
{
    fq_ctx::Dup &D = ctx->dup;
    fq_status st = table_reserve(ctx, D.T, n);
    if (st != FQ_OK) return st;
    DupArgs da{};
    da.raw[0] = d_r1; da.raw[1] = d_r2;
    da.rec[0] = ctx->d_rec[0].as<Rec>(); da.rec[1] = ctx->d_rec[1].as<Rec>();
    da.n_rec = n; da.n_mates = (uint32_t)n_mates;
    da.T = table_of(D.T);
    k_dup<<<(n + 7) / 8, 256, 0, ctx->stream>>>(da);
    ctx->launches++;
    D.n_mates = (uint32_t)n_mates;
    D.units += n;
    return FQ_OK;
}

// Host copy of an accumulator block of capacity `from` added into one of capacity `to` >= from, section by section.
void overlap_add_relaid(const uint64_t *src, uint32_t from, uint64_t *dst, uint32_t to)
{
    const OverlapLayout a = OverlapLayout::make(from), b = OverlapLayout::make(to);
    const uint32_t so[6] = {0, a.ins, a.d1, a.d2, a.m1, a.m2}, dO[6] = {0, b.ins, b.d1, b.d2, b.m1, b.m2};
    const uint32_t len[6] = {kOvlScalars, 2 * from, from + 1, from + 1, from, from};
    for (int k = 0; k < 6; ++k)
        for (uint32_t i = 0; i < len[k]; ++i) dst[dO[k] + i] += src[so[k] + i];
}

// One paired batch of the overlap profile: the accumulators grown (contents kept) to the batch's longest mate, then k_overlap.
fq_status overlap_batch(fq_ctx *ctx, const uint8_t *d_r1, const uint8_t *d_r2, uint32_t n, uint32_t max_len)
{
    fq_ctx::Overlap &V = ctx->ovl;
    if (!V.d_acc.p || max_len > V.cyc) {
        const uint32_t C = std::max(64u, round_up(max_len, 64));
        const OverlapLayout L = OverlapLayout::make(C);
        std::vector<uint64_t> h(L.total, 0);
        if (V.cyc) {
            std::vector<uint64_t> old(OverlapLayout::make(V.cyc).total);
            CK(cudaMemcpyAsync(old.data(), V.d_acc.p, old.size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            overlap_add_relaid(old.data(), V.cyc, h.data(), C);
        }
        DevBuf nb;
        CK(nb.ensure((size_t)L.total * 8));
        CK(cudaMemcpy(nb.p, h.data(), h.size() * 8, cudaMemcpyHostToDevice));
        V.d_acc = std::move(nb);
        V.cyc = C;
    }
    OverlapArgs oa{};
    oa.raw[0] = d_r1; oa.raw[1] = d_r2;
    oa.rec[0] = ctx->d_rec[0].as<Rec>(); oa.rec[1] = ctx->d_rec[1].as<Rec>();
    oa.n_rec = n;
    oa.min_overlap = V.min_overlap; oa.diff_limit = V.diff_limit; oa.diff_percent = V.diff_percent;
    oa.L = OverlapLayout::make(V.cyc);
    oa.acc = V.d_acc.as<unsigned long long>();
    oa.wa = (max_len + 31) / 32;
    oa.plane_words = 2 * oa.wa + 2;                // b: one word of padding in front, one behind
    const size_t per_warp = (size_t)oa.plane_words * sizeof(uint4), counters = (size_t)oa.L.total * 4;
    const size_t budget = std::min<size_t>(ctx->smem_optin, 200 * 1024);
    int warps = kOvlThreads / 32;
    while (warps > 1 && counters + warps * per_warp > budget) warps >>= 1;
    if (counters + warps * per_warp <= budget) {
        const size_t smem = counters + warps * per_warp;
        CK(allow_dynamic_smem(ctx, reinterpret_cast<const void *>(k_overlap<true>)));
        int per_sm = 1;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_overlap<true>, warps * 32, smem));
        const int grid = std::max(1, std::min<int>((n + warps - 1) / warps, ctx->sm_count * std::max(per_sm, 1)));
        k_overlap<true><<<grid, warps * 32, smem, ctx->stream>>>(oa);
    } else {
        // mates too long for shared memory: planes in global scratch (at most 256 MiB of it), counters straight to the block
        const uint32_t total_warps = (uint32_t)std::max<size_t>(1, std::min<size_t>({(size_t)n, (size_t)ctx->sm_count * 32, ((size_t)256 << 20) / per_warp}));
        CK(V.d_scratch.ensure(total_warps * per_warp));
        oa.scratch = V.d_scratch.as<uint4>();
        k_overlap<false><<<total_warps, 32, 0, ctx->stream>>>(oa);
    }
    ctx->launches++;
    V.pairs += n;
    return FQ_OK;
}

size_t overrep_stride(uint32_t prefix_len) { return 16 + ((size_t)prefix_len + 7) / 8 * 8; }

OverrepStore overrep_store_of(fq_ctx::Overrep &R)
{
    return OverrepStore{R.d_store.as<uint8_t>() + 64, R.store_cap - 1, (uint32_t)overrep_stride(R.prefix_len), R.d_store.as<unsigned long long>()};
}

// Room for `adding` more entries in the capture store at a load factor <= 1/2, contents kept (as table_reserve does).  The
// store's first 64 bytes hold its exact occupancy.
fq_status overrep_store_reserve(fq_ctx *ctx, fq_ctx::Overrep &R, uint64_t adding)
{
    uint64_t need = R.store_bound + adding;
    if (2 * need > R.store_cap && R.store_cap) {
        uint64_t occ = 0;
        CK(cudaMemcpyAsync(&occ, R.d_store.p, 8, cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        need = occ + adding;
    }
    if (2 * need > R.store_cap) {
        uint64_t cap = 1024;
        while (cap < 4 * need) cap <<= 1;           // headroom: the exact occupancy is read back rarely
        const size_t stride = overrep_stride(R.prefix_len);
        DevBuf nb;
        CK(nb.ensure(64 + cap * stride));
        OverrepStore to{nb.as<uint8_t>() + 64, cap - 1, (uint32_t)stride, nb.as<unsigned long long>()};
        if (R.store_cap) CK(cudaMemcpyAsync(nb.p, R.d_store.p, 8, cudaMemcpyDeviceToDevice, ctx->stream));
        else CK(cudaMemsetAsync(nb.p, 0, 8, ctx->stream));
        k_overrep_store_clear<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(to);
        if (R.store_cap) k_overrep_store_rehash<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(overrep_store_of(R), to);
        ctx->launches += R.store_cap ? 2 : 1;
        CK(cudaStreamSynchronize(ctx->stream));
        R.d_store = std::move(nb);
        R.store_cap = cap;
    }
    R.store_bound = need;
    return FQ_OK;
}

// One batch of overrepresented sequences: room for one key per read in the count table and, per mate, for the keys that can
// meet the capture condition in this batch (at most floor(10^6 / ppm), and at most the batch's reads), then k_overrep.
fq_status overrep_batch(fq_ctx *ctx, const uint8_t *d_r1, const uint8_t *d_r2, uint32_t n, int n_mates)
{
    fq_ctx::Overrep &R = ctx->ovr;
    fq_status st = table_reserve(ctx, R.T, (uint64_t)n * n_mates);
    if (st != FQ_OK) return st;
    st = overrep_store_reserve(ctx, R, (uint64_t)n_mates * std::min<uint64_t>(n, 1000000u / R.min_ppm));
    if (st != FQ_OK) return st;
    OverrepArgs oa{};
    oa.raw[0] = d_r1; oa.raw[1] = d_r2;
    oa.rec[0] = ctx->d_rec[0].as<Rec>(); oa.rec[1] = ctx->d_rec[1].as<Rec>();
    oa.n_rec = n; oa.n_mates = (uint32_t)n_mates; oa.prefix_len = R.prefix_len;
    for (int m = 0; m < n_mates; ++m) {
        R.reads[m] += n;
        oa.thr[m] = (unsigned long long)R.min_ppm * R.reads[m];
    }
    oa.T = table_of(R.T);
    oa.S = overrep_store_of(R);
    const uint64_t warps = (uint64_t)(n + 31) / 32 * n_mates;
    k_overrep<<<(unsigned)((warps + 7) / 8), 256, 0, ctx->stream>>>(oa);
    ctx->launches++;
    return FQ_OK;
}

KmerTable tile_table_of(fq_ctx::TileQual &Q) { return KmerTable{Q.d_slots.as<KmerSlot>(), kTileSlots - 1}; }

// Per flowcell tile quality, first half of a batch (right after framing): every read's key into the table and its dense id
// into d_id; {claims, overflow} travel back with the batch's BatchInfo, so the host knows the tiles without a sync of its own.
fq_status tile_keys_batch(fq_ctx *ctx, const uint8_t *d_r1, const uint8_t *d_r2, uint32_t n, int n_mates)
{
    fq_ctx::TileQual &Q = ctx->tq;
    Q.failed |= Q.batch_open;
    Q.batch_open = true;
    TileKeyArgs ka{};
    ka.raw[0] = d_r1; ka.raw[1] = d_r2;
    ka.rec[0] = ctx->d_rec[0].as<Rec>(); ka.rec[1] = ctx->d_rec[1].as<Rec>();
    ka.n_rec = n; ka.n_mates = (uint32_t)n_mates;
    ka.T = tile_table_of(Q);
    ka.cnt = Q.d_cnt.as<TileCounters>();
    for (int m = 0; m < n_mates; ++m) {
        CK(Q.d_id[m].ensure((size_t)n * sizeof(uint16_t)));
        ka.id[m] = Q.d_id[m].as<uint16_t>();
        Q.reads[m] += n;
    }
    const uint64_t warps = (uint64_t)(n + 31) / 32 * n_mates;
    k_tile_keys<<<(unsigned)((warps + kTileKeyThreads / 32 - 1) / (kTileKeyThreads / 32)), kTileKeyThreads, 0, ctx->stream>>>(ka);
    ctx->launches++;
    CK(cudaMemcpyAsync(Q.h_cnt.p, Q.d_cnt.p, 8, cudaMemcpyDeviceToHost, ctx->stream));
    Q.n_mates = (uint32_t)n_mates;
    return FQ_OK;
}

// Second half, once the BatchInfo is back: the block grown to the tiles seen and the batch's longest read (contents relaid on
// the device), then k_tile_qual.  A context that overflowed accumulates nothing more: its pass reports no table.
fq_status tile_qual_batch(fq_ctx *ctx, const uint8_t *d_r1, const uint8_t *d_r2, uint32_t n, int n_mates, uint32_t max_len, int32_t in_off)
{
    fq_ctx::TileQual &Q = ctx->tq;
    const uint32_t *h = Q.h_cnt.as<uint32_t>();
    Q.claims = h[0];
    Q.overflow |= h[1];
    Q.longest = std::max(Q.longest, max_len);
    if (Q.overflow || Q.claims == 0) return FQ_OK;
    uint32_t D = 64;
    while (D < (uint32_t)n_mates * Q.claims) D <<= 1;
    const uint32_t C = std::min(kTileMaxCycles, round_up(std::max(Q.longest, 1u), 32));
    if (D > Q.L.D || C > Q.L.C) {
        const TileLayout nl{std::max(D, Q.L.D), std::max(C, Q.L.C)};
        DevBuf nb;
        CK(nb.ensure(nl.total() * 8));
        CK(cudaMemsetAsync(nb.p, 0, nl.total() * 8, ctx->stream));
        if (Q.L.D) {
            k_tile_relay<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(Q.d_acc.as<unsigned long long>(), Q.L, nb.as<unsigned long long>(), nl);
            ctx->launches++;
        }
        CK(cudaStreamSynchronize(ctx->stream));
        Q.d_acc = std::move(nb);
        Q.L = nl;
    }
    TileQualArgs qa{};
    qa.raw[0] = d_r1; qa.raw[1] = d_r2;
    qa.rec[0] = ctx->d_rec[0].as<Rec>(); qa.rec[1] = ctx->d_rec[1].as<Rec>();
    qa.id[0] = Q.d_id[0].as<uint16_t>(); qa.id[1] = Q.d_id[1].as<uint16_t>();
    qa.n_rec = n; qa.n_mates = (uint32_t)n_mates; qa.in_off = in_off;
    // one wave of warps: runs as long as that allows, so that a run spans few id changes of sorted input
    const size_t smem = (size_t)(kTileQualThreads / 32) * Q.L.C * 4;
    int per_sm = 1;
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_tile_qual, kTileQualThreads, smem));
    const uint64_t wave = std::max<uint64_t>(1, (uint64_t)ctx->sm_count * std::max(per_sm, 1) * (kTileQualThreads / 32) / (uint64_t)n_mates);
    qa.run = (uint32_t)std::max<uint64_t>(32, ((uint64_t)n + wave - 1) / wave);
    qa.L = Q.L;
    qa.acc = Q.d_acc.as<unsigned long long>();
    const uint64_t warps = (uint64_t)((n + qa.run - 1) / qa.run) * n_mates;
    k_tile_qual<<<(unsigned)((warps + kTileQualThreads / 32 - 1) / (kTileQualThreads / 32)), kTileQualThreads, smem, ctx->stream>>>(qa);
    ctx->launches++;
    return FQ_OK;
}

// Outputs go to the d_out / h_out set `slot`.  With async_copy the D2H runs on s_out and the caller waits on ev_out.
fq_status process_common(fq_ctx *ctx, const uint8_t *d_r1, size_t n1, const uint8_t *d_r2, size_t n2, bool paired,
                         uint64_t first_record_index, int is_final, int copy_out, int slot, bool async_copy, fq_batch_out *out)
{
    memset(out, 0, sizeof(*out));
    for (auto &p : ctx->last_dev_out) p = nullptr;
    if (ctx->opt.input_quality_offset == FQ_OFFSET_AUTO)
        return fail(ctx, FQ_ERR_STATE, "quality offset not set; call fq_autodetect on the first batch");
    refresh_dev_opts(ctx);
    ctx->dopt.paired = paired ? 1 : 0;
    const DevOpts o = ctx->dopt;
    if (o.filter_adapter && o.num_thread && (first_record_index % FQ_REF_BATCH) != 0)
        return fail(ctx, FQ_ERR_ARG, "thread-count emulation needs batches that start on a 32768-record boundary");
    if (ctx->dup.enabled && ctx->dup.n_mates && ctx->dup.n_mates != (paired ? 2u : 1u))
        return fail(ctx, FQ_ERR_ARG, "duplication statistics: paired and single-end batches in one pass");
    if (ctx->tq.enabled && ctx->tq.n_mates && ctx->tq.n_mates != (paired ? 2u : 1u))
        return fail(ctx, FQ_ERR_ARG, "per flowcell tile quality: paired and single-end batches in one pass");
    BatchInfo *info = ctx->d_info.as<BatchInfo>();
    CK(reset_info(ctx));
    CK(cudaEventRecord(ctx->ev[0], ctx->stream));

    uint32_t n_rec[2] = {0, 0};
    fq_status st = frame_mate(ctx, 0, d_r1, n1, &n_rec[0]);
    if (st != FQ_OK) return st;
    if (paired) {
        st = frame_mate(ctx, 1, d_r2, n2, &n_rec[1]);
        if (st != FQ_OK) return st;
        if (n_rec[0] != n_rec[1]) return fail(ctx, FQ_ERR_FORMAT, "FaQCs.cppI/O error");   // FaQCs.cpp:370-380 (sic)
    }
    const uint32_t n = n_rec[0];
    const int n_mates = paired ? 2 : 1;
    out->n_records = n;
    if (o.filter_adapter && o.num_thread && !is_final && (n % FQ_REF_BATCH) != 0)
        return fail(ctx, FQ_ERR_ARG, "thread-count emulation needs non-final batches of a multiple of 32768 records");
    if (n == 0) {
        CK(cudaStreamSynchronize(ctx->stream));
        return FQ_OK;
    }
    // ---- per flowcell tile quality, first half: the keys, while the host waits for the framing scalars anyway
    if (ctx->tq.enabled) {
        st = tile_keys_batch(ctx, d_r1, d_r2, n, n_mates);
        if (st != FQ_OK) return st;
    }
    // second look at the framing scalars: max length, CR accounting, |seq| != |qual|
    BatchInfo hi;
    CK(read_info(ctx, &hi));
    st = map_device_error(ctx, hi);
    if (st != FQ_OK) return st;
    CK(cudaEventRecord(ctx->ev[4], ctx->stream));
    const uint32_t max_len = std::max(hi.max_len[0], hi.max_len[1]);
    if (max_len > kResLenMask) return fail(ctx, FQ_ERR_ARG, "read longer than 16 Mi bases");
    st = ensure_stats_rows(ctx, max_len);
    if (st != FQ_OK) return st;
    unsigned long long *S = ctx->d_stats.as<unsigned long long>();

    // read ids of the two mates (FaQCs.cpp:383-389): k_emit compares them while both headers pass through it;
    // --qc_only emits nothing, so it keeps the stand-alone kernel
    if (paired && ctx->check_pair_ids && o.qc_only) {
        k_check_pair_ids<<<(n + 255) / 256, 256, 0, ctx->stream>>>(d_r1, ctx->d_rec[0].as<Rec>(), d_r2, ctx->d_rec[1].as<Rec>(), n, info);
        ctx->launches++;
    }
    for (int m = 0; m < n_mates; ++m) {
        CK(ctx->d_res[m].ensure((size_t)n * sizeof(uint2)));
        if (ctx->debug_results) CK(ctx->d_dbg[m].ensure((size_t)n * sizeof(fq_read_result)));
    }

    // ---- adapter pass
    if (o.filter_adapter) {
        AdapterArgs aa{};
        for (int m = 0; m < n_mates; ++m) {
            CK(ctx->d_adp[m].ensure((size_t)n * sizeof(uint2)));
            CK(ctx->d_adp_best[m].ensure((size_t)n * sizeof(int32_t)));
            aa.raw[m] = m ? d_r2 : d_r1;
            aa.rec[m] = ctx->d_rec[m].as<Rec>();
            aa.adp[m] = ctx->d_adp[m].as<uint2>();
            aa.adp_best[m] = ctx->d_adp_best[m].as<int32_t>();
        }
        aa.n_rec = n;
        aa.n_mates = n_mates;
        aa.max_len = max_len;
        aa.stats = S;
        aa.L = ctx->L;
        aa.info = info;
        aa.first_index = first_record_index;
        aa.end_index = is_final ? first_record_index + n : ~0ull;
        // shared memory plan: offsets, codes, [adapter bit planes], per warp read codes + mask (+ read planes)
        const size_t smem_cap = ctx->smem_optin - 2048;          // the kernel also has 1 KiB of static shared memory
        const uint32_t mask_words = (max_len + 31) >> 5;
        uint32_t plane_words = 0, has_gap = 0, rpad = 1;
        for (uint32_t j = 0; j < ctx->aset.n; ++j) {
            const uint32_t wt = ((uint32_t)ctx->adapter_seqs[j].size() + 31) / 32;
            plane_words += 5 * wt;
            rpad = std::max(rpad, wt + 1);
            if (ctx->adapter_seqs[j].find('-') != std::string::npos) has_gap = 1;
        }
        aa.rpad = rpad;
        const size_t base_fixed = (size_t)(ctx->aset.n + 1) * 8 + ((ctx->aset.total + 3) & ~3u);
        const size_t per_warp_plain = ((max_len + 3) & ~3u) + 4 * (size_t)mask_words;
        const size_t per_warp_planes = per_warp_plain + 20 * ((size_t)mask_words + 2 * rpad);
        // segment sweep: four more read masks, the candidate bits and per-read bounds per warp; two 16-byte mask sets + 8 bytes per segment of the adapters
        uint32_t n_seg = 0, sweep_pure = 1;
        for (uint32_t j = 0; j < ctx->aset.n; ++j) {
            const size_t T = ctx->adapter_seqs[j].size();
            if (T && T <= kSweepMaxLen) {
                n_seg += (uint32_t)((T + 31) / 32);
                if (ctx->adapter_seqs[j].find_first_not_of("ACGTacgt") != std::string::npos) sweep_pure = 0;
            }
        }
        const size_t per_warp_sweep = 16 * ((size_t)mask_words + 2 * rpad) + 4 * (((size_t)ctx->aset.n + 31) / 32) + (((size_t)n_seg + 3) & ~(size_t)3);
        const size_t fixed_sweep = 40 * (size_t)n_seg + 16 + 8 + 4 * (((size_t)ctx->aset.n + 31) / 32);          // + alignment, + unswept bits, + origin / longest
        aa.use_planes = base_fixed + (size_t)plane_words * 4 + 4 * per_warp_planes <= smem_cap ? 1 : 0;
        aa.sweep = aa.use_planes && n_seg && base_fixed + (size_t)plane_words * 4 + fixed_sweep + 4 * (per_warp_planes + per_warp_sweep) <= smem_cap ? 1 : 0;
        aa.n_seg = aa.sweep ? n_seg : 0;
        aa.sweep_pure = sweep_pure;
        aa.plane_words = aa.use_planes ? plane_words : 0;
        aa.has_gap = has_gap;
        const size_t fixed = base_fixed + (size_t)aa.plane_words * 4 + (aa.sweep ? fixed_sweep : 0);
        const size_t per_warp = (aa.use_planes ? per_warp_planes : per_warp_plain) + (aa.sweep ? per_warp_sweep : 0);
        int warps = 8;
        while (warps > 1 && fixed + warps * per_warp > smem_cap) warps >>= 1;
        const size_t smem = fixed + warps * per_warp;
        if (smem > smem_cap) return fail(ctx, FQ_ERR_ARG, "adapter set + read length exceed shared memory");
        CK(allow_dynamic_smem(ctx, reinterpret_cast<const void *>(k_adapter)));
        int per_sm = 1;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_adapter, warps * 32, smem));
        const int grid = std::max(1, std::min<int>((n * n_mates + warps - 1) / warps, ctx->sm_count * std::max(per_sm, 1)));
        k_adapter<<<grid, warps * 32, smem, ctx->stream>>>(aa, o, ctx->aset);
        ctx->launches++;
    }

    // ---- trim / filter / statistics
    CK(cudaEventRecord(ctx->ev[1], ctx->stream));
    {
        TrimArgs ta{};
        for (int m = 0; m < n_mates; ++m) {
            ta.raw[m] = m ? d_r2 : d_r1;
            ta.rec[m] = ctx->d_rec[m].as<Rec>();
            ta.adp[m] = o.filter_adapter ? ctx->d_adp[m].as<uint2>() : nullptr;
            ta.adp_best[m] = o.filter_adapter ? ctx->d_adp_best[m].as<int32_t>() : nullptr;
            ta.res[m] = ctx->d_res[m].as<uint2>();
            ta.dbg[m] = ctx->debug_results ? ctx->d_dbg[m].as<fq_read_result>() : nullptr;
        }
        ta.n_rec = n;
        ta.n_mates = n_mates;
        ta.stats = S;
        ta.L = ctx->L;
        ta.rows = ctx->d_rows.as<StatsRows>();
        ta.info = info;
        // shared histogram rows: cover the longest read if it fits next to the composition tables
        ta.comp_key_len = max_len <= 1023 ? max_len : 0xffffffffu;
        const size_t budget = std::min<size_t>(ctx->smem_optin, 200 * 1024);
        uint32_t rows = round_up(std::max(max_len, 1u), 32);
        while (rows > 32 && SmemHist::words(rows, ta.comp_key_len) * 4 > budget) rows -= 32;
        rows = std::min(rows, ctx->L.rows);
        ta.smem_rows = rows;
        const size_t smem = SmemHist::words(rows, ta.comp_key_len) * 4;
        // instance with only the phase-1 width(s) this batch needs (smaller hot loop)
        using TrimKernel = void (*)(const TrimArgs, const DevOpts);
        const bool plain = o.mode == FQ_MODE_BWA_PLUS && !o.trim_5 && !o.trim_3 && !o.replace_q && !o.qc_only && !o.filter_adapter && o.in_off == o.out_off;
        // width-specialised instances have no generic path: every read of the batch must fit the shared-memory rows
        const int ksel = rows < max_len ? 0 : max_len <= 128 ? 4 : max_len <= 160 ? 5 : 0;
        const TrimKernel kern = plain ? (ksel == 4 ? (TrimKernel)k_trim<4, true> : ksel == 5 ? (TrimKernel)k_trim<5, true> : (TrimKernel)k_trim<0, true>)
                                      : (ksel == 4 ? (TrimKernel)k_trim<4, false> : ksel == 5 ? (TrimKernel)k_trim<5, false> : (TrimKernel)k_trim<0, false>);
        CK(allow_dynamic_smem(ctx, reinterpret_cast<const void *>(kern)));
        const int threads = kTrimThreads;
        int per_sm = 1;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem));
        per_sm = std::max(per_sm, 1);
        {   // tuning knob: cap the resident k_trim CTAs per SM (room for another context's kernels on the same device)
            static const int cap = [] { const char *e = getenv("FAQCS_B200_TRIM_CTAS_PER_SM"); return e ? atoi(e) : 0; }();
            if (cap > 0) per_sm = std::min(per_sm, cap);
        }
        const uint32_t groups = ((n + 31) / 32) * n_mates;
        const int grid = std::max(1, std::min<int>((groups + threads / 32 - 1) / (threads / 32), ctx->sm_count * per_sm));
        kern<<<grid, threads, smem, ctx->stream>>>(ta, o);
        ctx->launches++;
    }
    CK(cudaEventRecord(ctx->ev[2], ctx->stream));

    // ---- k-mer rarefaction: raw reads under --qc_only (trim.cpp:260-262), trimmed survivors otherwise (trim.cpp:545-547)
    if (ctx->kmer.enabled) {
        st = kmer_batch(ctx, d_r1, d_r2, n, n_mates, max_len, first_record_index, is_final, !o.qc_only);
        if (st != FQ_OK) return st;
    }
    // ---- duplication statistics: the sequence lines as framed
    if (ctx->dup.enabled) {
        st = dup_batch(ctx, d_r1, d_r2, n, n_mates);
        if (st != FQ_OK) return st;
    }
    // ---- insert size and overlap error profile: paired batches, the sequence lines as framed
    if (ctx->ovl.enabled && paired) {
        st = overlap_batch(ctx, d_r1, d_r2, n, max_len);
        if (st != FQ_OK) return st;
    }
    // ---- overrepresented sequences: the prefixes of the sequence lines as framed, each mate on its own
    if (ctx->ovr.enabled) {
        st = overrep_batch(ctx, d_r1, d_r2, n, n_mates);
        if (st != FQ_OK) return st;
    }
    // ---- per flowcell tile quality, second half: the quality lines as framed, each mate on its own
    if (ctx->tq.enabled) {
        st = tile_qual_batch(ctx, d_r1, d_r2, n, n_mates, max_len, o.in_off);
        if (st != FQ_OK) return st;
    }

    // ---- route / scan / emit
    EmitArgs ea{};
    ea.n_rec = n;
    ea.n_tiles = (n + kTile - 1) / kTile;
    ea.check_ids = paired && ctx->check_pair_ids && !o.qc_only;
    {   // rounds in which a warp stages its 32 records: the smallest split whose average slab leaves 8 % headroom
        const double avg = (double)std::max(n1, n2) / (double)std::max<uint32_t>(n, 1u);
        ea.parts = 1;
        while (ea.parts < 8 && (32.0 / ea.parts) * avg * 1.08 + 32.0 > (double)kEmitSlab) ea.parts *= 2;
    }
    const bool pieces = ctx->pieces && !o.qc_only;
    ea.prefetch_tiles = (uint32_t)(ctx->sm_count * FQ_EMIT_MIN_CTAS);      // one wave of k_emit CTAs
    if (const char *pf = getenv("FAQCS_B200_EMIT_PREFETCH_TILES")) ea.prefetch_tiles = (uint32_t)atoi(pf);
    CK(ctx->d_tile.ensure((size_t)ea.n_tiles * (pieces ? 12 : 4) * 4));
    ea.tile_sum = ctx->d_tile.as<uint32_t>();
    ea.info = info;
    ea.stats = S;
    ea.filter_off = ctx->L.filter;
    for (int m = 0; m < n_mates; ++m) {
        ea.raw[m] = m ? d_r2 : d_r1;
        ea.raw_bytes[m] = m ? n2 : n1;
        ea.rec[m] = ctx->d_rec[m].as<Rec>();
        ea.res[m] = ctx->d_res[m].as<uint2>();
        ea.canon[m] = ctx->d_canon[m].as<uint8_t>();
    }
    if (!o.qc_only) {
        // a trimmed record is never longer than its raw record, so the inputs bound the outputs; the unpaired stream of a
        // paired run takes mate 1 OR mate 2 of each pair, i.e. up to sum_i max(rec1_i, rec2_i) <= n1 + n2 bytes
        const size_t cap[4] = {paired ? n1 : 0, paired ? n2 : 0, paired ? n1 + n2 : n1, o.discard ? n1 + n2 : 0};
        for (int s = 0; s < 4; ++s) {
            if (cap[s]) CK(ctx->d_out[slot][s].ensure(cap[s] + 16));
            ea.out[s] = ctx->d_out[slot][s].as<uint8_t>();
            if (pieces && cap[s]) {       // at most one piece per record and mate
                CK(ctx->d_pieces[slot][s].ensure(((size_t)n * (s == 3 && paired ? 2 : 1) + 1) * sizeof(fq_out_piece)));
                ea.pieces[s] = ctx->d_pieces[slot][s].as<fq_out_piece>();
            }
        }
    }
    if (pieces) {
        k_route_pieces<<<ea.n_tiles, kTile, 0, ctx->stream>>>(ea, o);
        k_scan_tiles<<<12, 1024, 0, ctx->stream>>>(ea.tile_sum, ea.n_tiles, info);
        using EmitKernel = void (*)(const EmitArgs, const DevOpts);
        const EmitKernel kern = (!o.replace_q && o.in_off == o.out_off) ? (EmitKernel)k_emit_pieces<true> : (EmitKernel)k_emit_pieces<false>;
        kern<<<ea.n_tiles, kTile, 0, ctx->stream>>>(ea, o);
        ctx->launches += 3;
    } else {
    k_route<<<ea.n_tiles, kTile, 0, ctx->stream>>>(ea, o);
    k_scan_tiles<<<4, 1024, 0, ctx->stream>>>(ea.tile_sum, ea.n_tiles, info);
    ctx->launches += 2;
    }
    if (!o.qc_only && !pieces) {
        using EmitKernel = void (*)(const EmitArgs, const DevOpts);
        const EmitKernel kern = (!o.replace_q && o.in_off == o.out_off) ? (EmitKernel)k_emit<true> : (EmitKernel)k_emit<false>;
        CK(allow_dynamic_smem(ctx, reinterpret_cast<const void *>(kern)));
        kern<<<ea.n_tiles, kTile, kEmitSmem, ctx->stream>>>(ea, o);
        ctx->launches++;
    }
    CK(cudaEventRecord(ctx->ev[3], ctx->stream));
    CK(read_info(ctx, &hi));
    CK(cudaGetLastError());
    cudaEventElapsedTime(&ctx->t_seg[0], ctx->ev[0], ctx->ev[3]);
    cudaEventElapsedTime(&ctx->t_seg[1], ctx->ev[0], ctx->ev[4]);
    cudaEventElapsedTime(&ctx->t_seg[2], ctx->ev[4], ctx->ev[1]);
    cudaEventElapsedTime(&ctx->t_seg[3], ctx->ev[1], ctx->ev[2]);
    cudaEventElapsedTime(&ctx->t_seg[4], ctx->ev[2], ctx->ev[3]);
    st = map_device_error(ctx, hi);
    if (st != FQ_OK) return st;
    out->n_valid[0] = hi.n_valid[0];
    out->n_valid[1] = hi.n_valid[1];
    out->paired_read_number = hi.paired_reads;
    out->paired_base_length = hi.paired_bases;
    for (int s = 0; s < 4; ++s) {
        out->bytes[s] = o.qc_only ? 0 : hi.out_bytes[s];
        ctx->last_dev_out[s] = out->bytes[s] ? ctx->d_out[slot][s].p : nullptr;
        out->n_pieces[s] = pieces ? hi.out_pieces[s] : 0;
        out->literal_bytes[s] = pieces ? hi.out_literal[s] : 0;
    }
    if (copy_out) {
        // D2H of the four streams: on the compute stream (synchronous API) or, pipelined, on the copy-out
        // stream behind an event so that it overlaps the next batch's kernels
        cudaStream_t cs = ctx->stream;
        if (async_copy) {
            CK(cudaEventRecord(ctx->ev_comp[slot], ctx->stream));
            CK(cudaStreamWaitEvent(ctx->s_out, ctx->ev_comp[slot], 0));
            cs = ctx->s_out;
        }
        for (int s = 0; s < 4; ++s) {
            if (!out->bytes[s]) continue;
            // pieces mode: only the literal bytes and the piece list travel
            const size_t nb = pieces ? out->literal_bytes[s] : out->bytes[s];
            if (nb) {
                CK(ctx->h_out[slot][s].ensure(nb));
                CK(cudaMemcpyAsync(ctx->h_out[slot][s].p, ctx->d_out[slot][s].p, nb, cudaMemcpyDeviceToHost, cs));
                out->data[s] = static_cast<const uint8_t *>(ctx->h_out[slot][s].p);
            }
            if (pieces && out->n_pieces[s]) {
                const size_t pb = out->n_pieces[s] * sizeof(fq_out_piece);
                CK(ctx->h_pieces[slot][s].ensure(pb));
                CK(cudaMemcpyAsync(ctx->h_pieces[slot][s].p, ctx->d_pieces[slot][s].p, pb, cudaMemcpyDeviceToHost, cs));
                out->pieces[s] = static_cast<const fq_out_piece *>(ctx->h_pieces[slot][s].p);
            }
        }
        if (async_copy) CK(cudaEventRecord(ctx->ev_out[slot], ctx->s_out));
    }
    if (ctx->debug_results) {
        for (int m = 0; m < n_mates; ++m) {
            CK(ctx->h_dbg[m].ensure((size_t)n * sizeof(fq_read_result)));
            CK(cudaMemcpyAsync(ctx->h_dbg[m].p, ctx->d_dbg[m].p, (size_t)n * sizeof(fq_read_result), cudaMemcpyDeviceToHost, ctx->stream));
            out->results[m] = static_cast<const fq_read_result *>(ctx->h_dbg[m].p);
        }
    }
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->tq.batch_open = false;
    return FQ_OK;
}

}  // namespace

extern "C" {

int fq_abi_version(void) { return FQ_ABI_VERSION; }

const char *fq_build_info(void) { return "faqcs_b200 " __DATE__ " sm_100a (nvcc " FQ_STR(__CUDACC_VER_MAJOR__) "." FQ_STR(__CUDACC_VER_MINOR__) ")"; }

fq_status fq_create(const fq_options *opt, int device, fq_ctx **out)
{
    fq_ctx *ctx = nullptr;
    if (!opt || !out) return fail(nullptr, FQ_ERR_ARG, "fq_create: null argument");
    int n_dev = 0;
    if (cudaGetDeviceCount(&n_dev) != cudaSuccess || n_dev == 0)
        return fail(nullptr, FQ_ERR_NO_DEVICE, "no CUDA device: faqcs_b200 has no CPU fallback");
    if (device < 0 || device >= n_dev) return fail(nullptr, FQ_ERR_ARG, "fq_create: bad device index");
    if (cudaSetDevice(device) != cudaSuccess) return fail(nullptr, FQ_ERR_CUDA, "cudaSetDevice failed");
    ctx = new fq_ctx();
    ctx->device = device;
    ctx->opt = *opt;
    for (uint32_t i = 0; i < opt->n_adapters; ++i) {
        ctx->adapter_names.push_back(opt->adapters[i].name ? opt->adapters[i].name : "");
        ctx->adapter_seqs.push_back(opt->adapters[i].seq ? opt->adapters[i].seq : "");
    }
    ctx->opt.adapters = nullptr;
    cudaDeviceProp prop{};
    fq_status st = FQ_OK;
    auto boot = [&]() -> fq_status {
        CK(cudaGetDeviceProperties(&prop, device));
        ctx->sm_count = prop.multiProcessorCount;
        ctx->smem_optin = prop.sharedMemPerBlockOptin;
        CK(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&ctx->s_in, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&ctx->s_out, cudaStreamNonBlocking));
        for (int k = 0; k < 2; ++k) {
            CK(cudaEventCreateWithFlags(&ctx->ev_in[k], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&ctx->ev_comp[k], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&ctx->ev_out[k], cudaEventDisableTiming));
        }
        for (auto &e : ctx->ev) CK(cudaEventCreate(&e));
        CK(ctx->h_info.ensure(sizeof(BatchInfo)));
        CK(ctx->d_info.ensure(sizeof(BatchInfo)));
        CK(ctx->d_rows.ensure(sizeof(StatsRows)));
        CK(cudaMemset(ctx->d_rows.p, 0, sizeof(StatsRows)));
        fq_status s2 = upload_adapters(ctx);
        if (s2 != FQ_OK) return s2;
        return ensure_stats_rows(ctx, 320);
    };
    st = boot();
    if (st != FQ_OK) {
        g_create_error = ctx->error;
        fq_destroy(ctx);
        return st;
    }
    refresh_dev_opts(ctx);
    *out = ctx;
    return FQ_OK;
}

void fq_destroy(fq_ctx *ctx)
{
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    // copies queued by fq_submit_host / fq_run may still target buffers the destructor frees
    for (cudaStream_t s : {ctx->stream, ctx->s_in, ctx->s_out})
        if (s) cudaStreamSynchronize(s);
    delete ctx;
}

const char *fq_last_error(const fq_ctx *ctx) { return ctx ? ctx->error.c_str() : g_create_error.c_str(); }

fq_status fq_set_debug_results(fq_ctx *ctx, int enable)
{
    if (!ctx) return FQ_ERR_ARG;
    ctx->debug_results = enable != 0;
    return FQ_OK;
}

fq_status fq_set_output_pieces(fq_ctx *ctx, int enable)
{
    if (!ctx) return FQ_ERR_ARG;
    ctx->pieces = enable != 0;
    return FQ_OK;
}

fq_status fq_set_check_pair_ids(fq_ctx *ctx, int enable)
{
    if (!ctx) return FQ_ERR_ARG;
    ctx->check_pair_ids = enable != 0;
    return FQ_OK;
}

fq_status fq_set_quality(fq_ctx *ctx, int32_t quality)
{
    if (!ctx) return FQ_ERR_ARG;
    ctx->opt.quality = quality;
    refresh_dev_opts(ctx);
    return FQ_OK;
}

void *fq_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaMallocHost(&p, bytes ? bytes : 1) != cudaSuccess) return nullptr;
    return p;
}

void fq_host_free(void *p) { if (p) cudaFreeHost(p); }

fq_status fq_autodetect(fq_ctx *ctx, const uint8_t *r1, size_t n1, const uint8_t *r2, size_t n2,
                        int32_t *input_quality_offset, int32_t *quality)
{
    if (!ctx || (!r1 && n1) || (!r2 && n2)) return FQ_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    const bool paired = r2 != nullptr;
    if (ctx->opt.input_quality_offset == FQ_OFFSET_AUTO) {
        int detected[2] = {0, 0};
        for (int m = 0; m < (paired ? 2 : 1); ++m) {
            const uint8_t *h = m ? r2 : r1;
            const size_t n = m ? n2 : n1;
            CK(reset_info(ctx));
            uint32_t n_rec = 0;
            if (n) {
                CK(ctx->d_raw[m].ensure(n + 16));
                CK(cudaMemcpyAsync(ctx->d_raw[m].p, h, n, cudaMemcpyHostToDevice, ctx->stream));
                fq_status st = frame_mate(ctx, m, ctx->d_raw[m].as<uint8_t>(), n, &n_rec);
                if (st != FQ_OK) return st;
            }
            const uint32_t look = std::min<uint32_t>(n_rec, FQ_REF_BATCH);
            if (look) {
                k_detect_offset<<<(look * 32 + 255) / 256, 256, 0, ctx->stream>>>(ctx->d_raw[m].as<uint8_t>(), ctx->d_rec[m].as<Rec>(), look,
                                                                                 ctx->d_info.as<BatchInfo>());
                ctx->launches++;
            }
            BatchInfo hi;
            CK(read_info(ctx, &hi));
            fq_status st = map_device_error(ctx, hi);
            if (st != FQ_OK) return st;
            if (hi.detect_key == ~0ull)
                return fail(ctx, FQ_ERR_OFFSET, "trim.cpp:auto_detect_quality_offset: Unknown quality format!");
            detected[m] = (int)(hi.detect_key & 0xff);
        }
        if (paired && detected[0] != detected[1])
            return fail(ctx, FQ_ERR_OFFSET, "FaQCs.cpp:process_paired: I/O Error (inconsistent quality offset detection between reads one and two)");
        ctx->opt.input_quality_offset = detected[0];
    }
    // auto_detect_next_seq (trim.cpp:619-626): header of the first read starts with "@NS"
    if (ctx->opt.quality < 20 && n1 >= 3 && r1[0] == '@' && r1[1] == 'N' && r1[2] == 'S') {
        bool first_line = true;     // "@NS" must sit inside the first header line
        for (int i = 0; i < 3; ++i) first_line &= (r1[i] != '\n' && r1[i] != '\r');
        if (first_line) ctx->opt.quality = 20;
    }
    refresh_dev_opts(ctx);
    if (input_quality_offset) *input_quality_offset = ctx->opt.input_quality_offset;
    if (quality) *quality = ctx->opt.quality;
    return FQ_OK;
}

fq_status fq_process_host(fq_ctx *ctx, const uint8_t *r1, size_t n1, const uint8_t *r2, size_t n2,
                          uint64_t first_record_index, int is_final, fq_batch_out *out)
{
    if (!ctx || !out || (!r1 && n1) || (!r2 && n2)) return FQ_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    const bool paired = r2 != nullptr;
    CK(ctx->d_raw[0].ensure(n1 + 16));
    if (n1) CK(cudaMemcpyAsync(ctx->d_raw[0].p, r1, n1, cudaMemcpyHostToDevice, ctx->stream));
    if (paired) {
        CK(ctx->d_raw[1].ensure(n2 + 16));
        if (n2) CK(cudaMemcpyAsync(ctx->d_raw[1].p, r2, n2, cudaMemcpyHostToDevice, ctx->stream));
    }
    return process_common(ctx, ctx->d_raw[0].as<uint8_t>(), n1, paired ? ctx->d_raw[1].as<uint8_t>() : nullptr, n2, paired,
                          first_record_index, is_final, 1, 0, false, out);
}

// ---- pipelined host path: submit (H2D on its own stream) / run (kernels) / wait (D2H on its own stream) ----
fq_status fq_submit_host(fq_ctx *ctx, const uint8_t *r1, size_t n1, const uint8_t *r2, size_t n2,
                         uint64_t first_record_index, int is_final, uint64_t *ticket)
{
    if (!ctx || !ticket || (!r1 && n1) || (!r2 && n2)) return FQ_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    const uint64_t t = ctx->next_ticket;
    const int slot = (int)(t & 1);
    if (ctx->sub[slot].busy) return fail(ctx, FQ_ERR_STATE, "fq_submit_host: the batch submitted two tickets ago has not been run yet");
    fq_ctx::Submitted &p = ctx->sub[slot];
    p = fq_ctx::Submitted{};
    p.busy = true;
    p.n1 = n1; p.n2 = n2; p.paired = r2 != nullptr; p.first = first_record_index; p.is_final = is_final; p.ticket = t;
    CK(ctx->d_raw_slot[slot][0].ensure(n1 + 16));
    if (n1) CK(cudaMemcpyAsync(ctx->d_raw_slot[slot][0].p, r1, n1, cudaMemcpyHostToDevice, ctx->s_in));
    if (p.paired) {
        CK(ctx->d_raw_slot[slot][1].ensure(n2 + 16));
        if (n2) CK(cudaMemcpyAsync(ctx->d_raw_slot[slot][1].p, r2, n2, cudaMemcpyHostToDevice, ctx->s_in));
    }
    CK(cudaEventRecord(ctx->ev_in[slot], ctx->s_in));
    ctx->next_ticket++;
    *ticket = t;
    return FQ_OK;
}

fq_status fq_run(fq_ctx *ctx, uint64_t ticket)
{
    if (!ctx) return FQ_ERR_ARG;
    const int slot = (int)(ticket & 1);
    fq_ctx::Submitted &p = ctx->sub[slot];
    if (!p.busy || p.ticket != ticket) return fail(ctx, FQ_ERR_STATE, "fq_run: unknown or already processed ticket");
    if (ctx->fin[slot].busy) return fail(ctx, FQ_ERR_STATE, "fq_run: the outputs of the ticket two submissions ago have not been collected with fq_wait");
    // the per-read debug verdicts live in one buffer per mate, not one per output slot
    if (ctx->debug_results) return fail(ctx, FQ_ERR_STATE, "fq_run: per-read debug results are only available through the synchronous entry points");
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_in[slot], 0));
    fq_ctx::Finished &f = ctx->fin[slot];
    fq_status st = process_common(ctx, ctx->d_raw_slot[slot][0].as<uint8_t>(), p.n1, p.paired ? ctx->d_raw_slot[slot][1].as<uint8_t>() : nullptr,
                                  p.n2, p.paired, p.first, p.is_final, 1, slot, true, &f.out);
    p.busy = false;                       // the kernels are done with the raw input slot
    if (st != FQ_OK) return st;
    f.busy = true;
    f.ticket = ticket;
    return FQ_OK;
}

fq_status fq_wait(fq_ctx *ctx, uint64_t ticket, fq_batch_out *out)
{
    if (!ctx || !out) return FQ_ERR_ARG;
    const int slot = (int)(ticket & 1);
    fq_ctx::Finished &f = ctx->fin[slot];
    if (!f.busy || f.ticket != ticket) return fail(ctx, FQ_ERR_STATE, "fq_wait: ticket has not been run");
    CK(cudaSetDevice(ctx->device));
    bool any = false;
    for (int s = 0; s < 4; ++s) any |= f.out.bytes[s] != 0;
    if (any) CK(cudaEventSynchronize(ctx->ev_out[slot]));
    *out = f.out;
    f.busy = false;
    return FQ_OK;
}

fq_status fq_process_device(fq_ctx *ctx, const void *d_r1, size_t n1, const void *d_r2, size_t n2,
                            uint64_t first_record_index, int is_final, int copy_out, fq_batch_out *out)
{
    if (!ctx || !out || (!d_r1 && n1) || (!d_r2 && n2)) return FQ_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    return process_common(ctx, static_cast<const uint8_t *>(d_r1), n1, static_cast<const uint8_t *>(d_r2), n2, d_r2 != nullptr,
                          first_record_index, is_final, copy_out, 0, false, out);
}

fq_status fq_device_outputs(fq_ctx *ctx, const void *d_out[FQ_NUM_STREAM])
{
    if (!ctx || !d_out) return FQ_ERR_ARG;
    for (int s = 0; s < 4; ++s) d_out[s] = ctx->last_dev_out[s];
    return FQ_OK;
}

fq_status fq_last_timing(fq_ctx *ctx, float *ms, int n)
{
    if (!ctx || !ms) return FQ_ERR_ARG;
    for (int i = 0; i < n && i < 5; ++i) ms[i] = ctx->t_seg[i];
    return FQ_OK;
}

uint64_t fq_launch_count(const fq_ctx *ctx) { return ctx ? ctx->launches : 0; }

void *fq_stream(fq_ctx *ctx) { return ctx ? static_cast<void *>(ctx->stream) : nullptr; }

fq_status fq_stats_reserve_rows(fq_ctx *ctx, uint32_t rows)
{
    if (!ctx) return FQ_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    return ensure_stats_rows(ctx, rows);
}

fq_status fq_stats_device_buffer(fq_ctx *ctx, void **d_u64, size_t *n_u64, void **d_rows_u32x4)
{
    if (!ctx) return FQ_ERR_ARG;
    CK(cudaStreamSynchronize(ctx->stream));
    if (d_u64) *d_u64 = ctx->d_stats.p;
    if (n_u64) *n_u64 = ctx->L.total;
    if (d_rows_u32x4) *d_rows_u32x4 = ctx->d_rows.p;
    return FQ_OK;
}

fq_status fq_kmer_enable(fq_ctx *ctx, uint32_t k, uint64_t split_size, uint32_t num_subsample)
{
    if (!ctx || k < 2 || k > 31 || split_size == 0 || num_subsample == 0) return FQ_ERR_ARG;      // options.cpp:537-568
    CK(cudaSetDevice(ctx->device));
    fq_ctx::Kmer &K = ctx->kmer;
    K.enabled = K.collecting = true;
    K.k = k; K.split_size = split_size; K.num_subsample = num_subsample;
    CK(K.d_call_total.ensure((size_t)kKmerMaxCalls * 8));
    CK(K.d_call_distinct.ensure((size_t)kKmerMaxCalls * 8));
    CK(K.d_small.ensure((size_t)kKmerSmallCounts * 8));
    CK(K.d_big.ensure((size_t)(1u << 20) * 4));
    CK(K.T.d_scalars.ensure(64));
    CK(cudaMemset(K.d_call_total.p, 0, (size_t)kKmerMaxCalls * 8));
    return table_resize(ctx, K.T, 1ull << 24);
}

fq_status fq_kmer_end_pass(fq_ctx *ctx)
{
    if (!ctx) return FQ_ERR_ARG;
    fq_ctx *const ctxs[1] = {ctx};
    return fq_kmer_end_pass_all(ctxs, 1, nullptr);
}

fq_status fq_kmer_results(fq_ctx *ctx, fq_kmer_view *view)
{
    if (!ctx || !view) return FQ_ERR_ARG;
    fq_ctx::Kmer &K = ctx->kmer;
    K.flat.clear();
    for (const auto &kv : K.freq) { K.flat.push_back(kv.first); K.flat.push_back(kv.second); }
    view->n_rarefaction = (uint32_t)K.samples.size();
    view->rarefaction = K.samples.data();
    view->n_frequency = K.flat.size() / 2;
    view->frequency = K.flat.data();
    return FQ_OK;
}

fq_status fq_reset_stats(fq_ctx *ctx)
{
    if (!ctx) return FQ_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaMemset(ctx->d_stats.p, 0, ctx->L.total * 8));
    CK(cudaMemset(ctx->d_rows.p, 0, sizeof(StatsRows)));
    return FQ_OK;
}

fq_status fq_stats(fq_ctx *ctx, fq_stats_view *v)
{
    if (!ctx || !v) return FQ_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    const StatsLayout &L = ctx->L;
    CK(ctx->h_stats.ensure(L.total * 8 + sizeof(StatsRows)));
    uint64_t *S = static_cast<uint64_t *>(ctx->h_stats.p);
    StatsRows rows{};
    CK(cudaMemcpy(S, ctx->d_stats.p, L.total * 8, cudaMemcpyDeviceToHost));
    CK(cudaMemcpy(&rows, ctx->d_rows.p, sizeof(StatsRows), cudaMemcpyDeviceToHost));
    memset(v, 0, sizeof(*v));
    for (int i = 0; i < FQ_NUM_STAT; ++i) v->filter_stats[i] = S[L.filter + i];
    const uint32_t na = L.n_adapters;
    ctx->v_adapter_reads.assign(S + L.adapter_reads, S + L.adapter_reads + na);
    ctx->v_adapter_bases.assign(S + L.adapter_bases, S + L.adapter_bases + na);
    // main(): phiX pseudo-adapters -> READ_PHIX/BASE_PHIX, the rest -> READ_ADAPTER/BASE_ADAPTER (FaQCs.cpp:92-127)
    for (uint32_t j = 0; j < na; ++j) {
        const bool phix = ctx->adapter_names[j] == kPhiX || ctx->adapter_names[j] == kPhiXComplement;
        v->filter_stats[phix ? FQ_READ_PHIX : FQ_READ_ADAPTER] += ctx->v_adapter_reads[j];
        v->filter_stats[phix ? FQ_BASE_PHIX : FQ_BASE_ADAPTER] += ctx->v_adapter_bases[j];
    }
    v->n_adapters = na;
    v->adapter_reads = ctx->v_adapter_reads.data();
    v->adapter_bases = ctx->v_adapter_bases.data();
    const uint32_t pr = std::min(rows.pre_rows, L.rows), qr = std::min(rows.post_rows, L.rows);
    v->pre_rows = pr;
    v->post_rows = qr;
    ctx->v_pre_q.assign((size_t)pr * kQualCols, 0);
    ctx->v_post_q.assign((size_t)qr * kQualCols, 0);
    ctx->v_pre_b.assign((size_t)pr * kBaseCols, 0);
    ctx->v_post_b.assign((size_t)qr * kBaseCols, 0);
    for (uint32_t p = 0; p < pr; ++p) {
        for (int c = 0; c < kQualCols; ++c) ctx->v_pre_q[(size_t)p * kQualCols + c] = S[L.pre_q + (size_t)c * L.rows + p];
        for (int c = 0; c < kBaseCols; ++c) ctx->v_pre_b[(size_t)p * kBaseCols + c] = S[L.pre_b + (size_t)c * L.rows + p];
    }
    for (uint32_t p = 0; p < qr; ++p) {          // post = pre - removed (+ G->N into column N)
        for (int c = 0; c < kQualCols; ++c)
            ctx->v_post_q[(size_t)p * kQualCols + c] = S[L.pre_q + (size_t)c * L.rows + p] - S[L.rem_q + (size_t)c * L.rows + p];
        for (int c = 0; c < kBaseCols; ++c)
            ctx->v_post_b[(size_t)p * kBaseCols + c] = S[L.pre_b + (size_t)c * L.rows + p] - S[L.rem_b + (size_t)c * L.rows + p] +
                                                       (c == 4 ? S[L.g2n + p] : 0);
    }
    v->pre_quality_matrix = ctx->v_pre_q.data();
    v->post_quality_matrix = ctx->v_post_q.data();
    v->pre_base_matrix = ctx->v_pre_b.data();
    v->post_base_matrix = ctx->v_post_b.data();
    const size_t hist_off[4] = {L.pre_rq, L.pre_bq, L.post_rq, L.post_bq};
    for (int h = 0; h < 4; ++h) ctx->v_hist[h].assign(S + hist_off[h], S + hist_off[h] + kQualCols);
    v->pre_read_quality_hist = ctx->v_hist[0].data();
    v->pre_base_quality_hist = ctx->v_hist[1].data();
    v->post_read_quality_hist = ctx->v_hist[2].data();
    v->post_base_quality_hist = ctx->v_hist[3].data();
    ctx->v_pre_comp.assign(S + L.pre_comp, S + L.pre_comp + 6 * (size_t)kCompBins);
    ctx->v_post_comp.assign(S + L.post_comp, S + L.post_comp + 6 * (size_t)kCompBins);
    v->pre_composition = ctx->v_pre_comp.data();
    v->post_composition = ctx->v_post_comp.data();
    v->pre_len_size = std::min(rows.pre_len_size, L.rows + 1);
    v->post_len_size = std::min(rows.post_len_size, L.rows + 1);
    ctx->v_pre_len.assign(S + L.pre_len, S + L.pre_len + v->pre_len_size);
    ctx->v_post_len.assign(S + L.post_len, S + L.post_len + v->post_len_size);
    v->pre_length_hist = ctx->v_pre_len.data();
    v->post_length_hist = ctx->v_post_len.data();
    return FQ_OK;
}


// ---- multi-GPU merge: NCCL, loaded at run time --------------------------------------------------------
namespace {
struct NcclApi {
    void *handle = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommInitAll)(ncclComm_t *, int, const int *) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    ncclResult_t (*Send)(const void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Recv)(void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    bool ok = false;
};
NcclApi &nccl()
{
    static NcclApi api = [] {
        NcclApi a;
        for (const char *name : {"libnccl.so.2", "libnccl.so"}) {
            a.handle = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
            if (a.handle) break;
        }
        if (!a.handle) return a;
        auto sym = [&](const char *n) { return dlsym(a.handle, n); };
        a.GetUniqueId = reinterpret_cast<decltype(a.GetUniqueId)>(sym("ncclGetUniqueId"));
        a.CommInitRank = reinterpret_cast<decltype(a.CommInitRank)>(sym("ncclCommInitRank"));
        a.CommInitAll = reinterpret_cast<decltype(a.CommInitAll)>(sym("ncclCommInitAll"));
        a.CommDestroy = reinterpret_cast<decltype(a.CommDestroy)>(sym("ncclCommDestroy"));
        a.AllReduce = reinterpret_cast<decltype(a.AllReduce)>(sym("ncclAllReduce"));
        a.GroupStart = reinterpret_cast<decltype(a.GroupStart)>(sym("ncclGroupStart"));
        a.GroupEnd = reinterpret_cast<decltype(a.GroupEnd)>(sym("ncclGroupEnd"));
        a.Send = reinterpret_cast<decltype(a.Send)>(sym("ncclSend"));
        a.Recv = reinterpret_cast<decltype(a.Recv)>(sym("ncclRecv"));
        a.AllGather = reinterpret_cast<decltype(a.AllGather)>(sym("ncclAllGather"));
        a.GetErrorString = reinterpret_cast<decltype(a.GetErrorString)>(sym("ncclGetErrorString"));
        a.ok = a.GetUniqueId && a.CommInitRank && a.CommInitAll && a.CommDestroy && a.AllReduce && a.GroupStart && a.GroupEnd && a.GetErrorString &&
               a.Send && a.Recv && a.AllGather;
        return a;
    }();
    return api;
}
}  // namespace

struct fq_comm {
    ncclComm_t comm = nullptr;
    int device = 0;
    int n_ranks = 1, rank = 0;
};

#define NK(ctx_, call)                                                                                          \
    do {                                                                                                        \
        ncclResult_t r__ = (call);                                                                              \
        if (r__ != ncclSuccess) return fail(ctx_, FQ_ERR_CUDA, std::string(#call) + ": " + nccl().GetErrorString(r__)); \
    } while (0)

fq_status fq_comm_unique_id(uint8_t id[FQ_COMM_ID_BYTES])
{
    static_assert(sizeof(ncclUniqueId) == FQ_COMM_ID_BYTES, "ncclUniqueId is 128 bytes");
    if (!id) return FQ_ERR_ARG;
    if (!nccl().ok) return fail(nullptr, FQ_ERR_STATE, "NCCL (libnccl.so.2) could not be loaded");
    ncclUniqueId u;
    NK(nullptr, nccl().GetUniqueId(&u));
    memcpy(id, &u, FQ_COMM_ID_BYTES);
    return FQ_OK;
}

fq_status fq_comm_init_rank(fq_ctx *ctx, int n_ranks, int rank, const uint8_t id[FQ_COMM_ID_BYTES], fq_comm **out)
{
    if (!ctx || !id || !out || n_ranks < 1 || rank < 0 || rank >= n_ranks) return FQ_ERR_ARG;
    if (!nccl().ok) return fail(ctx, FQ_ERR_STATE, "NCCL (libnccl.so.2) could not be loaded");
    CK(cudaSetDevice(ctx->device));
    ncclUniqueId u;
    memcpy(&u, id, FQ_COMM_ID_BYTES);
    fq_comm *c = new fq_comm();
    c->device = ctx->device;
    c->n_ranks = n_ranks;
    c->rank = rank;
    ncclResult_t r = nccl().CommInitRank(&c->comm, n_ranks, u, rank);
    if (r != ncclSuccess) { delete c; return fail(ctx, FQ_ERR_CUDA, std::string("ncclCommInitRank: ") + nccl().GetErrorString(r)); }
    *out = c;
    return FQ_OK;
}

fq_status fq_comm_init_all(fq_ctx *const *ctxs, int n, fq_comm **out)
{
    if (!ctxs || !out || n < 1) return FQ_ERR_ARG;
    fq_ctx *ctx = ctxs[0];
    if (!nccl().ok) return fail(ctx, FQ_ERR_STATE, "NCCL (libnccl.so.2) could not be loaded");
    std::vector<int> devs(n);
    std::vector<ncclComm_t> comms(n);
    for (int i = 0; i < n; ++i) devs[i] = ctxs[i]->device;
    NK(ctx, nccl().CommInitAll(comms.data(), n, devs.data()));
    for (int i = 0; i < n; ++i) {
        out[i] = new fq_comm();
        out[i]->comm = comms[i];
        out[i]->device = devs[i];
        out[i]->n_ranks = n;
        out[i]->rank = i;
    }
    return FQ_OK;
}

void fq_comm_destroy(fq_comm *c)
{
    if (!c) return;
    if (c->comm && nccl().ok) {
        cudaSetDevice(c->device);
        nccl().CommDestroy(c->comm);
    }
    delete c;
}

fq_status fq_allreduce_stats(fq_ctx *const *ctxs, int n, fq_comm *const *comms)
{
    if (!ctxs || !comms || n < 1) return FQ_ERR_ARG;
    fq_ctx *ctx = ctxs[0];
    if (!nccl().ok) return fail(ctx, FQ_ERR_STATE, "NCCL (libnccl.so.2) could not be loaded");
    for (int i = 0; i < n; ++i)
        if (!ctxs[i] || !comms[i] || comms[i]->device != ctxs[i]->device) return fail(ctx, FQ_ERR_ARG, "fq_allreduce_stats: communicator and context are on different devices");
    fq_status st = sync_all(ctxs, n);
    if (st != FQ_OK) return st;
    // 1. every rank must use the same layout: agree on the row capacity (MAX), grow where needed
    std::vector<DevBuf> d_cap(n);
    std::vector<uint32_t> cap(n);
    for (int i = 0; i < n; ++i) {
        CK(cudaSetDevice(ctxs[i]->device));
        CK(d_cap[i].ensure(4));
        cap[i] = ctxs[i]->L.rows;
        CK(cudaMemcpyAsync(d_cap[i].p, &cap[i], 4, cudaMemcpyHostToDevice, ctxs[i]->stream));
    }
    NK(ctx, nccl().GroupStart());
    for (int i = 0; i < n; ++i) NK(ctx, nccl().AllReduce(d_cap[i].p, d_cap[i].p, 1, ncclUint32, ncclMax, comms[i]->comm, ctxs[i]->stream));
    NK(ctx, nccl().GroupEnd());
    for (int i = 0; i < n; ++i) {
        CK(cudaSetDevice(ctxs[i]->device));
        CK(cudaMemcpyAsync(&cap[i], d_cap[i].p, 4, cudaMemcpyDeviceToHost, ctxs[i]->stream));
        CK(cudaStreamSynchronize(ctxs[i]->stream));
        st = ensure_stats_rows(ctxs[i], cap[i]);
        if (st != FQ_OK) return st;
        if (ctxs[i]->L.rows != cap[i] && ctxs[i]->L.rows != std::max(64u, round_up(cap[i], 64)))
            return fail(ctx, FQ_ERR_STATE, "fq_allreduce_stats: row capacities disagree");
    }
    // 2. the merge: SUM of the flat u64 block, MAX of the four row counters (timed: the first collective above also carries
    //    NCCL's one-off connection set-up)
    for (int i = 0; i < n; ++i) {
        CK(cudaSetDevice(ctxs[i]->device));
        CK(cudaEventRecord(ctxs[i]->ev[0], ctxs[i]->stream));
    }
    NK(ctx, nccl().GroupStart());
    for (int i = 0; i < n; ++i) {
        NK(ctx, nccl().AllReduce(ctxs[i]->d_stats.p, ctxs[i]->d_stats.p, ctxs[i]->L.total, ncclUint64, ncclSum, comms[i]->comm, ctxs[i]->stream));
        NK(ctx, nccl().AllReduce(ctxs[i]->d_rows.p, ctxs[i]->d_rows.p, 4, ncclUint32, ncclMax, comms[i]->comm, ctxs[i]->stream));
    }
    NK(ctx, nccl().GroupEnd());
    for (int i = 0; i < n; ++i) {
        CK(cudaSetDevice(ctxs[i]->device));
        CK(cudaEventRecord(ctxs[i]->ev[1], ctxs[i]->stream));
        CK(cudaStreamSynchronize(ctxs[i]->stream));
        cudaEventElapsedTime(&ctxs[i]->allreduce_ms, ctxs[i]->ev[0], ctxs[i]->ev[1]);
        d_cap[i].release();
    }
    return FQ_OK;
}

// Contexts that share a device (one in-flight batch each, so that consecutive batches overlap on the device): dst += src,
// src = 0.  The same merge as the all-reduce (sum of the block, max of the row counters) without a communicator.
fq_status fq_merge_stats(fq_ctx *dst, fq_ctx *src)
{
    if (!dst || !src || dst == src) return FQ_ERR_ARG;
    if (dst->device != src->device) return fail(dst, FQ_ERR_ARG, "fq_merge_stats: contexts on different devices (use fq_allreduce_stats)");
    if (dst->opt.n_adapters != src->opt.n_adapters) return fail(dst, FQ_ERR_ARG, "fq_merge_stats: contexts with different adapter lists");
    fq_ctx *const ctx = dst;
    CK(cudaSetDevice(dst->device));
    CK(cudaStreamSynchronize(src->stream));
    CK(cudaStreamSynchronize(dst->stream));
    const uint32_t rows = std::max(dst->L.rows, src->L.rows);
    fq_status st = ensure_stats_rows(dst, rows);
    if (st == FQ_OK) st = ensure_stats_rows(src, rows);
    if (st != FQ_OK) return st;
    if (dst->L.total != src->L.total) return fail(dst, FQ_ERR_STATE, "fq_merge_stats: row capacities disagree");
    k_merge_stats<<<dst->sm_count * 4, 256, 0, dst->stream>>>(dst->d_stats.as<unsigned long long>(), src->d_stats.as<unsigned long long>(), dst->L.total,
                                                           dst->d_rows.as<uint32_t>(), src->d_rows.as<uint32_t>());
    dst->launches++;
    CK(cudaStreamSynchronize(dst->stream));
    return FQ_OK;
}

float fq_last_allreduce_ms(const fq_ctx *ctx) { return ctx ? ctx->allreduce_ms : 0.0f; }

// ---- k-mer rarefaction: end of a pass, over one context or a table sharded over several ------------------------------
namespace {

constexpr uint32_t kKmerBigCap = 1u << 20;         // counts >= kKmerSmallCounts listed per context

// What one context contributes to the end of a pass, as one flat u64 block: summed over the contexts (on the host, or one
// ncclAllReduce across ranks).  Per-context scalars have one entry per context, zero in the others' blocks.
struct KmerSum {
    size_t call_total, call_distinct, call_reads, call_runs, small, n_distinct, pass_reads, calls_beyond, n_big, call_end, total;
    explicit KmerSum(size_t n_shards)
    {
        size_t o = 0;
        call_total = o;    o += kKmerMaxCalls;      // k-mer instances per call
        call_distinct = o; o += kKmerMaxCalls;      // k-mers first seen in each call (of the context's share of the keys)
        call_reads = o;    o += kKmerMaxCalls;      // reads per call
        call_runs = o;     o += kKmerMaxCalls;      // times each call was run
        small = o;         o += kKmerSmallCounts;   // k-mers per count, counts below kKmerSmallCounts
        n_distinct = o++;
        pass_reads = o++;
        calls_beyond = o++;                         // calls >= kKmerMaxCalls run
        n_big = o;         o += n_shards;           // per context: k-mers with a larger count (listed separately)
        call_end = o;      o += n_shards;           // per context: 1 + its highest call
        total = o;
    }
};

// Occupied slots of the context's table per owner.
fq_status table_owner_counts(fq_ctx *ctx, HashTable &T, uint32_t n_shards, uint64_t *counts)
{
    CK(cudaSetDevice(ctx->device));
    CK(T.d_scalars.ensure(64 + (size_t)n_shards * 8));
    CK(cudaMemsetAsync(T.d_scalars.p, 0, (size_t)n_shards * 8, ctx->stream));
    k_kmer_partition_count<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(table_of(T), n_shards, T.d_scalars.as<unsigned long long>());
    ctx->launches++;
    CK(cudaMemcpyAsync(counts, T.d_scalars.p, (size_t)n_shards * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return FQ_OK;
}

// The table's entries into d_send grouped by owner (group j at offsets[j]); the table is then cleared -- first grown, empty,
// if `incoming` entries need more than half of it -- and takes back the context's own group.
fq_status table_scatter(fq_ctx *ctx, HashTable &T, uint32_t n_shards, uint32_t me, const uint64_t *counts, uint64_t incoming, std::vector<uint64_t> *offsets)
{
    CK(cudaSetDevice(ctx->device));
    offsets->assign(n_shards + 1, 0);
    for (uint32_t j = 0; j < n_shards; ++j) (*offsets)[j + 1] = (*offsets)[j] + counts[j];
    CK(T.d_send.ensure(std::max<uint64_t>(offsets->back(), 1) * sizeof(KmerSlot)));
    CK(cudaMemcpyAsync(T.d_scalars.p, offsets->data(), (size_t)n_shards * 8, cudaMemcpyHostToDevice, ctx->stream));
    k_kmer_partition_scatter<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(table_of(T), n_shards, T.d_scalars.as<unsigned long long>(), T.d_send.as<KmerSlot>());
    k_kmer_clear<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(table_of(T));
    ctx->launches += 2;
    fq_status st = table_resize(ctx, T, 2 * incoming, false);
    if (st != FQ_OK) return st;
    if (counts[me]) {
        k_kmer_merge<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(table_of(T), T.d_send.as<KmerSlot>() + (*offsets)[me], counts[me]);
        ctx->launches++;
    }
    CK(cudaGetLastError());
    return FQ_OK;
}

fq_status table_merge_received(fq_ctx *ctx, HashTable &T, uint64_t n)
{
    if (!n) return FQ_OK;
    k_kmer_merge<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(table_of(T), T.d_recv.as<KmerSlot>(), n);
    ctx->launches++;
    CK(cudaGetLastError());
    return FQ_OK;
}

// The context's share of the table -> its summary block; `big` gets its list of counts >= kKmerSmallCounts.
fq_status kmer_summarize(fq_ctx *ctx, const KmerSum &S, uint32_t me, std::vector<uint64_t> *flat, std::vector<uint32_t> *big)
{
    fq_ctx::Kmer &K = ctx->kmer;
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemsetAsync(K.d_call_distinct.p, 0, (size_t)kKmerMaxCalls * 8, ctx->stream));
    CK(cudaMemsetAsync(K.d_small.p, 0, (size_t)kKmerSmallCounts * 8, ctx->stream));
    CK(cudaMemsetAsync(K.T.d_scalars.p, 0, 64, ctx->stream));
    k_kmer_summarize<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(table_of(K.T), K.d_call_distinct.as<unsigned long long>(), K.d_small.as<unsigned long long>(),
                                                              K.d_big.as<uint32_t>(), kKmerBigCap, reinterpret_cast<uint32_t *>(K.T.d_scalars.as<uint8_t>() + 16),
                                                              K.T.d_scalars.as<unsigned long long>());
    ctx->launches++;
    flat->assign(S.total, 0);
    uint64_t *F = flat->data();
    uint32_t n_big = 0;
    CK(cudaMemcpyAsync(F + S.call_total, K.d_call_total.p, (size_t)kKmerMaxCalls * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(F + S.call_distinct, K.d_call_distinct.p, (size_t)kKmerMaxCalls * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(F + S.small, K.d_small.p, (size_t)kKmerSmallCounts * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(F + S.n_distinct, K.T.d_scalars.p, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&n_big, K.T.d_scalars.as<uint8_t>() + 16, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (!K.call_reads.empty()) {
        std::copy(K.call_reads.begin(), K.call_reads.end(), F + S.call_reads);
        std::copy(K.call_runs.begin(), K.call_runs.end(), F + S.call_runs);
    }
    F[S.pass_reads] = K.pass_reads;
    F[S.calls_beyond] = K.calls_beyond;
    F[S.n_big + me] = n_big;
    F[S.call_end + me] = K.call_end;
    if (big) {
        big->resize(std::min(n_big, kKmerBigCap));
        if (!big->empty()) CK(cudaMemcpy(big->data(), K.d_big.p, big->size() * 4, cudaMemcpyDeviceToHost));
    }
    return FQ_OK;
}

// The whole pass's summary -> the pass's points, histogram and end state (FaQCs.cpp:518-537, 737-756); every context of
// the run computes the same from the same summary.  Then a new table for the next pass.
fq_status kmer_finish(fq_ctx *ctx, const KmerSum &S, uint32_t n_shards, const std::vector<uint64_t> &sum, const std::vector<uint32_t> &big)
{
    fq_ctx::Kmer &K = ctx->kmer;
    const uint64_t *F = sum.data();
    uint64_t call_end = 0;
    for (uint32_t j = 0; j < n_shards; ++j) {
        if (F[S.n_big + j] > kKmerBigCap) return fail(ctx, FQ_ERR_ARG, "k-mer rarefaction: more than 2^20 k-mers with counts above 65535");
        call_end = std::max(call_end, F[S.call_end + j]);
    }
    // every call up to the highest one run must have been run exactly once, on one of the contexts
    const uint32_t nc = (uint32_t)std::min<uint64_t>(call_end, kKmerMaxCalls);
    for (uint32_t c = 0; c < nc; ++c) {
        const uint64_t runs = F[S.call_runs + c];
        if (runs != 1) {
            char msg[200];
            if (runs == 0) snprintf(msg, sizeof msg, "k-mer rarefaction: trim() call %u of the pass was never run: a batch in front of the last one is missing", c);
            else snprintf(msg, sizeof msg, "k-mer rarefaction: trim() call %u of the pass was run %llu times: batches with the same first_record_index", c,
                          (unsigned long long)runs);
            return fail(ctx, FQ_ERR_ARG, msg);
        }
    }
    if (F[S.calls_beyond] != (call_end > kKmerMaxCalls ? call_end - kKmerMaxCalls : 0))
        return fail(ctx, FQ_ERR_ARG, "k-mer rarefaction: the trim() calls beyond the 65536th were not each run once");
    KmerWalk w;
    fq_status st = kmer_walk(ctx, K, call_end, [&](uint32_t c) { return F[S.call_reads + c]; }, &w);
    if (st != FQ_OK) return st;
    // points of the curve taken in this pass (trim.cpp:165-178): table size and instances after their call
    unsigned long long run_d = 0, run_t = 0;
    size_t next = 0;
    for (uint32_t c = 0; c < nc; ++c) {
        run_d += F[S.call_distinct + c];
        run_t += F[S.call_total + c];
        while (next < w.points.size() && w.points[next].first == c) {
            K.samples.push_back(fq_rarefaction{w.points[next].second, run_d, run_t});
            ++next;
        }
    }
    // FaQCs.cpp:518-537 / 737-756: frequency histogram of the table, and one point if the curve is still empty
    for (uint32_t c = 1; c < kKmerSmallCounts; ++c)
        if (F[S.small + c]) K.freq[c] += F[S.small + c];
    for (uint32_t c : big) K.freq[c] += 1;
    K.total_reads += F[S.pass_reads];
    K.collecting = w.collecting;
    if (K.collecting && K.samples.empty()) K.samples.push_back(fq_rarefaction{K.total_reads, F[S.n_distinct], run_t});
    // a new table for the next pass
    if (!K.call_reads.empty()) {
        std::fill(K.call_reads.begin(), K.call_reads.end(), 0);
        std::fill(K.call_runs.begin(), K.call_runs.end(), 0);
    }
    K.calls_beyond = K.call_end = K.pass_reads = 0;
    K.T.occupied_bound = 0;
    CK(cudaSetDevice(ctx->device));
    k_kmer_clear<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(table_of(K.T));
    ctx->launches++;
    CK(cudaMemsetAsync(K.d_call_total.p, 0, (size_t)kKmerMaxCalls * 8, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    K.T.d_send.release();
    K.T.d_recv.release();
    return FQ_OK;
}

fq_status nccl_allgather_u64(fq_ctx *ctx, const fq_comm *c, const std::vector<uint64_t> &mine, std::vector<uint64_t> *all)
{
    const size_t m = mine.size();
    DevBuf d;
    CK(d.ensure((size_t)(c->n_ranks + 1) * m * 8));
    uint64_t *send = d.as<uint64_t>() + (size_t)c->n_ranks * m;
    all->assign((size_t)c->n_ranks * m, 0);
    CK(cudaMemcpyAsync(send, mine.data(), m * 8, cudaMemcpyHostToDevice, ctx->stream));
    NK(ctx, nccl().AllGather(send, d.p, m, ncclUint64, c->comm, ctx->stream));
    CK(cudaMemcpyAsync(all->data(), d.p, all->size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return FQ_OK;
}

fq_status nccl_sum_u64(fq_ctx *ctx, const fq_comm *c, std::vector<uint64_t> *v)
{
    DevBuf d;
    CK(d.ensure(v->size() * 8));
    CK(cudaMemcpyAsync(d.p, v->data(), v->size() * 8, cudaMemcpyHostToDevice, ctx->stream));
    NK(ctx, nccl().AllReduce(d.p, d.p, v->size(), ncclUint64, ncclSum, c->comm, ctx->stream));
    CK(cudaMemcpyAsync(v->data(), d.p, v->size() * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return FQ_OK;
}

// Every rank's list of large counts (n_big[j] of rank j, at d_big on each) on every rank.
fq_status nccl_gather_big(fq_ctx *ctx, const fq_comm *c, const void *d_big, const uint64_t *n_big, std::vector<uint32_t> *big)
{
    uint64_t most = 1;
    for (int j = 0; j < c->n_ranks; ++j) most = std::max(most, n_big[j]);
    DevBuf d;
    CK(d.ensure((size_t)c->n_ranks * most * 4));
    NK(ctx, nccl().AllGather(d_big, d.p, most, ncclUint32, c->comm, ctx->stream));
    std::vector<uint32_t> all((size_t)c->n_ranks * most);
    CK(cudaMemcpyAsync(all.data(), d.p, all.size() * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    big->clear();
    for (int j = 0; j < c->n_ranks; ++j) big->insert(big->end(), all.begin() + (size_t)j * most, all.begin() + (size_t)j * most + n_big[j]);
    return FQ_OK;
}

// Steps 3 and 4 of the end of a sharded pass, for either table (tab(ctx) is the context's table): the contexts' groups go to
// their owners in n_shards - 1 rounds (round r: shard s sends to s + r, receives from s - r), and each owner merges them into
// its cleared table.  head[s * H + kHeadCounts + j] = entries of shard s owned by shard j.
constexpr size_t kHeadCounts = 4;

using TableOf = HashTable &(*)(fq_ctx *);

fq_status table_exchange(fq_ctx *const *ctxs, int n, const fq_comm *cm, uint32_t rank0, uint32_t n_shards, TableOf tab, const std::vector<uint64_t> &head, size_t H)
{
    auto counts = [&](uint32_t from, uint32_t to) { return head[(size_t)from * H + kHeadCounts + to]; };
    std::vector<std::vector<uint64_t>> offsets(n);
    for (int i = 0; i < n; ++i) {
        fq_ctx *const ctx = ctxs[i];
        const uint32_t me = rank0 + i;
        uint64_t incoming = 0, largest = 1;
        for (uint32_t j = 0; j < n_shards; ++j) {
            incoming += counts(j, me);
            if (j != me) largest = std::max(largest, counts(j, me));
        }
        fq_status st = table_scatter(ctx, tab(ctx), n_shards, me, head.data() + (size_t)me * H + kHeadCounts, incoming, &offsets[i]);
        if (st != FQ_OK) return st;
        CK(tab(ctx).d_recv.ensure(largest * sizeof(KmerSlot)));
    }
    fq_status st = sync_all(ctxs, n);       // every send buffer is complete before another context reads it
    if (st != FQ_OK) return st;
    for (uint32_t r = 1; r < n_shards; ++r) {
        for (int i = 0; i < n; ++i) {
            fq_ctx *const ctx = ctxs[i];
            HashTable &T = tab(ctx);
            const uint32_t me = rank0 + i, dst = (me + r) % n_shards, src = (me + n_shards - r) % n_shards;
            const uint64_t n_out = counts(me, dst), n_in = counts(src, me);
            CK(cudaSetDevice(ctx->device));
            if (cm) {
                if (!n_out && !n_in) continue;      // both ends know the counts: neither posts a transfer
                NK(ctx, nccl().GroupStart());
                if (n_out) NK(ctx, nccl().Send(T.d_send.as<KmerSlot>() + offsets[i][dst], 2 * n_out, ncclUint64, (int)dst, cm->comm, ctx->stream));
                if (n_in) NK(ctx, nccl().Recv(T.d_recv.p, 2 * n_in, ncclUint64, (int)src, cm->comm, ctx->stream));
                NK(ctx, nccl().GroupEnd());
            } else if (n_in) {
                fq_ctx *const from = ctxs[src];
                CK(cudaMemcpyPeerAsync(T.d_recv.p, ctx->device, tab(from).d_send.as<KmerSlot>() + offsets[src][me], from->device,
                                       n_in * sizeof(KmerSlot), ctx->stream));
            }
            st = table_merge_received(ctx, T, n_in);
            if (st != FQ_OK) return st;
        }
    }
    return FQ_OK;
}

// The arguments and the error reporting of an end of pass over n contexts, shared by both tables: impl runs the pass, with
// ctxs[0] as shard rank0 of n_shards.
using EndPassImpl = fq_status (*)(fq_ctx *const *ctxs, int n, const fq_comm *cm, uint32_t n_shards, uint32_t rank0);

fq_status end_pass_entry(fq_ctx *const *ctxs, int n, fq_comm *const *comm, const char *name, EndPassImpl impl)
{
    if (!ctxs || n < 1) return FQ_ERR_ARG;
    for (int i = 0; i < n; ++i) {
        if (!ctxs[i]) return FQ_ERR_ARG;
        for (int j = 0; j < i; ++j)
            if (ctxs[j] == ctxs[i]) return fail(ctxs[0], FQ_ERR_ARG, std::string(name) + ": a context is listed twice");
    }
    if (comm && !comm[0]) return fail(ctxs[0], FQ_ERR_ARG, std::string(name) + ": null communicator");
    fq_status st = FQ_OK;
    fq_ctx *const ctx0 = ctxs[0];
    const fq_comm *cm = comm ? comm[0] : nullptr;
    const uint32_t n_shards = cm ? (uint32_t)cm->n_ranks : (uint32_t)n;
    if (cm && (n != 1 || cm->device != ctx0->device)) st = fail(ctx0, FQ_ERR_ARG, std::string(name) + ": with a communicator, pass this process's one context on its device");
    else if (cm && !nccl().ok) st = fail(ctx0, FQ_ERR_STATE, "NCCL (libnccl.so.2) could not be loaded");
    else if (n_shards > kKmerMaxOwners) st = fail(ctx0, FQ_ERR_ARG, std::string(name) + ": more than 1024 contexts");
    else {
        for (int i = 0; i < n; ++i) ctxs[i]->error.clear();
        st = impl(ctxs, n, cm, n_shards, cm ? (uint32_t)cm->rank : 0u);
    }
    if (st != FQ_OK) {          // the verdict is the run's: every context reports it
        std::string msg;
        for (int i = 0; i < n && msg.empty(); ++i) msg = ctxs[i]->error;
        for (int i = 0; i < n; ++i) ctxs[i]->error = msg;
    }
    return st;
}

fq_status kmer_end_pass_impl(fq_ctx *const *ctxs, int n, const fq_comm *cm, uint32_t n_shards, uint32_t rank0)
{
    fq_ctx *const ctx0 = ctxs[0];
    fq_status st = sync_all(ctxs, n);
    if (st != FQ_OK) return st;
    // 1. agree on the parameters; 2. occupied slots per owner: header {enabled, k, split_size, num_subsample, counts[n_shards]}
    const size_t H = 4 + n_shards;
    std::vector<uint64_t> head((size_t)n_shards * H, 0);
    for (int i = 0; i < n; ++i) {
        const fq_ctx::Kmer &K = ctxs[i]->kmer;
        uint64_t *h = head.data() + (size_t)(rank0 + i) * H;
        h[0] = K.enabled; h[1] = K.k; h[2] = K.split_size; h[3] = K.num_subsample;
        if (K.enabled && n_shards > 1) {
            st = table_owner_counts(ctxs[i], ctxs[i]->kmer.T, n_shards, h + kHeadCounts);
            if (st != FQ_OK) return st;
        }
    }
    if (cm) {
        const std::vector<uint64_t> mine(head.begin() + (size_t)rank0 * H, head.begin() + (size_t)(rank0 + 1) * H);
        st = nccl_allgather_u64(ctx0, cm, mine, &head);
        if (st != FQ_OK) return st;
    }
    for (uint32_t j = 1; j < n_shards; ++j)
        if (head[(size_t)j * H] != head[0]) return fail(ctx0, FQ_ERR_ARG, "fq_kmer_end_pass_all: k-mer rarefaction is enabled on some contexts only");
    if (!head[0]) return FQ_OK;
    for (uint32_t j = 1; j < n_shards; ++j) {
        const uint64_t *a = head.data(), *b = head.data() + (size_t)j * H;
        if (a[1] != b[1] || a[2] != b[2] || a[3] != b[3]) {
            char msg[240];
            snprintf(msg, sizeof msg, "fq_kmer_end_pass_all: context %u counts k = %llu, split_size = %llu, num_subsample = %llu; context 0 k = %llu, "
                     "split_size = %llu, num_subsample = %llu", j, (unsigned long long)b[1], (unsigned long long)b[2], (unsigned long long)b[3],
                     (unsigned long long)a[1], (unsigned long long)a[2], (unsigned long long)a[3]);
            return fail(ctx0, FQ_ERR_ARG, msg);
        }
    }
    // 3, 4. exchange the groups and merge
    if (n_shards > 1) {
        st = table_exchange(ctxs, n, cm, rank0, n_shards, [](fq_ctx *c) -> HashTable & { return c->kmer.T; }, head, H);
        if (st != FQ_OK) return st;
    }
    // 5. summarise each shard; 6. combine
    const KmerSum S(n_shards);
    std::vector<uint64_t> sum, flat;
    std::vector<uint32_t> big, part;
    for (int i = 0; i < n; ++i) {
        st = kmer_summarize(ctxs[i], S, rank0 + i, &flat, cm ? nullptr : &part);
        if (st != FQ_OK) return st;
        if (sum.empty()) sum.assign(S.total, 0);
        for (size_t k = 0; k < S.total; ++k) sum[k] += flat[k];
        big.insert(big.end(), part.begin(), part.end());
    }
    if (cm) {
        st = nccl_sum_u64(ctx0, cm, &sum);
        if (st == FQ_OK) {
            for (uint32_t j = 0; j < n_shards; ++j)
                if (sum[S.n_big + j] > kKmerBigCap) return fail(ctx0, FQ_ERR_ARG, "k-mer rarefaction: more than 2^20 k-mers with counts above 65535");
            st = nccl_gather_big(ctx0, cm, ctx0->kmer.d_big.p, sum.data() + S.n_big, &big);
        }
        if (st != FQ_OK) return st;
    }
    // 7. the pass's points and histogram, identically on every context
    for (int i = 0; i < n; ++i) {
        st = kmer_finish(ctxs[i], S, n_shards, sum, big);
        if (st != FQ_OK) return st;
    }
    return FQ_OK;
}

// ---- duplication statistics: end of a pass, over one context or a table sharded over several -------------------------
// The summary block of one shard: {histogram of counts below kKmerSmallCounts, distinct keys, per shard: keys with a larger
// count (listed separately)}.
constexpr size_t kDupDistinct = kKmerSmallCounts, kDupBig = kKmerSmallCounts + 1;

fq_status dup_summarize(fq_ctx *ctx, uint32_t n_shards, uint32_t me, std::vector<uint64_t> *flat, std::vector<uint32_t> *big)
{
    fq_ctx::Dup &D = ctx->dup;
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemsetAsync(D.d_small.p, 0, (size_t)kKmerSmallCounts * 8, ctx->stream));
    CK(cudaMemsetAsync(D.T.d_scalars.p, 0, 64, ctx->stream));
    // no slot of this table has a first call (fq_dup.cuh), so the per-call array is never written
    k_kmer_summarize<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(table_of(D.T), nullptr, D.d_small.as<unsigned long long>(), D.d_big.as<uint32_t>(), kKmerBigCap,
                                                              reinterpret_cast<uint32_t *>(D.T.d_scalars.as<uint8_t>() + 16), D.T.d_scalars.as<unsigned long long>());
    ctx->launches++;
    flat->assign(kDupBig + n_shards, 0);
    uint64_t *F = flat->data();
    uint32_t n_big = 0;
    CK(cudaMemcpyAsync(F, D.d_small.p, (size_t)kKmerSmallCounts * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(F + kDupDistinct, D.T.d_scalars.p, 8, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaMemcpyAsync(&n_big, D.T.d_scalars.as<uint8_t>() + 16, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    F[kDupBig + me] = n_big;
    if (big) {
        big->resize(std::min(n_big, kKmerBigCap));
        if (!big->empty()) CK(cudaMemcpy(big->data(), D.d_big.p, big->size() * 4, cudaMemcpyDeviceToHost));
    }
    return FQ_OK;
}

// The pass's result on one context, then a cleared table for the next pass.
fq_status dup_finish(fq_ctx *ctx, uint64_t units, const std::vector<uint64_t> &sum, const std::vector<uint32_t> &big)
{
    fq_ctx::Dup &D = ctx->dup;
    std::map<uint64_t, uint64_t> levels;
    for (uint32_t c = 1; c < kKmerSmallCounts; ++c)
        if (sum[c]) levels[c] += sum[c];
    for (uint32_t c : big) levels[c] += 1;
    D.levels.clear();
    for (const auto &kv : levels) { D.levels.push_back(kv.first); D.levels.push_back(kv.second); }
    D.res_units = units;
    D.res_distinct = sum[kDupDistinct];
    D.units = 0;
    D.n_mates = 0;
    D.T.occupied_bound = 0;
    CK(cudaSetDevice(ctx->device));
    k_kmer_clear<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(table_of(D.T));
    ctx->launches++;
    CK(cudaStreamSynchronize(ctx->stream));
    D.T.d_send.release();
    D.T.d_recv.release();
    return FQ_OK;
}

fq_status dup_end_pass_impl(fq_ctx *const *ctxs, int n, const fq_comm *cm, uint32_t n_shards, uint32_t rank0)
{
    fq_ctx *const ctx0 = ctxs[0];
    fq_status st = sync_all(ctxs, n);
    if (st != FQ_OK) return st;
    // 1. agree on the units; 2. occupied slots per owner: header {enabled, mates per unit (0: no batch), units, -, counts[n_shards]}
    const size_t H = kHeadCounts + n_shards;
    std::vector<uint64_t> head((size_t)n_shards * H, 0);
    for (int i = 0; i < n; ++i) {
        fq_ctx::Dup &D = ctxs[i]->dup;
        uint64_t *h = head.data() + (size_t)(rank0 + i) * H;
        h[0] = D.enabled; h[1] = D.n_mates; h[2] = D.units;
        if (D.enabled && n_shards > 1) {
            st = table_owner_counts(ctxs[i], D.T, n_shards, h + kHeadCounts);
            if (st != FQ_OK) return st;
        }
    }
    if (cm) {
        const std::vector<uint64_t> mine(head.begin() + (size_t)rank0 * H, head.begin() + (size_t)(rank0 + 1) * H);
        st = nccl_allgather_u64(ctx0, cm, mine, &head);
        if (st != FQ_OK) return st;
    }
    uint64_t enabled = 0, n_mates = 0, units = 0;
    for (uint32_t j = 0; j < n_shards; ++j) {
        const uint64_t *h = head.data() + (size_t)j * H;
        enabled += h[0];
        if (h[1] && n_mates && h[1] != n_mates) return fail(ctx0, FQ_ERR_ARG, "fq_dup_end_pass_all: some contexts counted pairs, others single reads");
        if (h[1]) n_mates = h[1];
        units += h[2];
    }
    if (!enabled) return fail(ctx0, FQ_ERR_STATE, "fq_dup_end_pass_all: duplication statistics are not enabled (fq_dup_enable)");
    if (enabled != n_shards) return fail(ctx0, FQ_ERR_ARG, "fq_dup_end_pass_all: duplication statistics are enabled on some contexts only");
    // 3, 4. exchange the groups and merge
    if (n_shards > 1) {
        st = table_exchange(ctxs, n, cm, rank0, n_shards, [](fq_ctx *c) -> HashTable & { return c->dup.T; }, head, H);
        if (st != FQ_OK) return st;
    }
    // 5. summarise each shard; 6. combine
    std::vector<uint64_t> sum(kDupBig + n_shards, 0), flat;
    std::vector<uint32_t> big, part;
    for (int i = 0; i < n; ++i) {
        st = dup_summarize(ctxs[i], n_shards, rank0 + i, &flat, cm ? nullptr : &part);
        if (st != FQ_OK) return st;
        for (size_t k = 0; k < sum.size(); ++k) sum[k] += flat[k];
        big.insert(big.end(), part.begin(), part.end());
    }
    if (cm) {
        st = nccl_sum_u64(ctx0, cm, &sum);
        if (st != FQ_OK) return st;
    }
    for (uint32_t j = 0; j < n_shards; ++j)
        if (sum[kDupBig + j] > kKmerBigCap) return fail(ctx0, FQ_ERR_ARG, "duplication statistics: more than 2^20 sequences with more than 65535 copies in one shard");
    if (cm) {
        st = nccl_gather_big(ctx0, cm, ctx0->dup.d_big.p, sum.data() + kDupBig, &big);
        if (st != FQ_OK) return st;
    }
    // 7. the same result on every context
    for (int i = 0; i < n; ++i) {
        st = dup_finish(ctxs[i], units, sum, big);
        if (st != FQ_OK) return st;
    }
    return FQ_OK;
}

// ---- insert size and overlap error profile: end of a pass, over one context or several ---------------------------------
// Every context's block, laid out for the largest capacity of any of them, is summed (on the host, or one ncclAllReduce
// across ranks); the sum is published on every context and the accumulators are cleared.
fq_status overlap_end_pass_impl(fq_ctx *const *ctxs, int n, const fq_comm *cm, uint32_t n_shards, uint32_t rank0)
{
    fq_ctx *const ctx0 = ctxs[0];
    fq_status st = sync_all(ctxs, n);
    if (st != FQ_OK) return st;
    // 1. agree on the parameters and the capacity: header {enabled, min_overlap, diff_limit, diff_percent, capacity}
    const size_t H = 5;
    std::vector<uint64_t> head((size_t)n_shards * H, 0);
    for (int i = 0; i < n; ++i) {
        const fq_ctx::Overlap &V = ctxs[i]->ovl;
        uint64_t *h = head.data() + (size_t)(rank0 + i) * H;
        h[0] = V.enabled; h[1] = V.min_overlap; h[2] = V.diff_limit; h[3] = V.diff_percent; h[4] = V.cyc;
    }
    if (cm) {
        const std::vector<uint64_t> mine(head.begin() + (size_t)rank0 * H, head.begin() + (size_t)(rank0 + 1) * H);
        st = nccl_allgather_u64(ctx0, cm, mine, &head);
        if (st != FQ_OK) return st;
    }
    uint64_t enabled = 0, cap = 0;
    for (uint32_t j = 0; j < n_shards; ++j) {
        const uint64_t *h = head.data() + (size_t)j * H;
        enabled += h[0];
        cap = std::max(cap, h[4]);
    }
    if (!enabled) return fail(ctx0, FQ_ERR_STATE, "fq_overlap_end_pass_all: the overlap profile is not enabled (fq_overlap_enable)");
    if (enabled != n_shards) return fail(ctx0, FQ_ERR_ARG, "fq_overlap_end_pass_all: the overlap profile is enabled on some contexts only");
    for (uint32_t j = 1; j < n_shards; ++j) {
        const uint64_t *a = head.data(), *b = head.data() + (size_t)j * H;
        if (a[1] != b[1] || a[2] != b[2] || a[3] != b[3]) {
            char msg[240];
            snprintf(msg, sizeof msg, "fq_overlap_end_pass_all: context %u has min_overlap = %llu, diff_limit = %llu, diff_percent = %llu; context 0 "
                     "min_overlap = %llu, diff_limit = %llu, diff_percent = %llu", j, (unsigned long long)b[1], (unsigned long long)b[2],
                     (unsigned long long)b[3], (unsigned long long)a[1], (unsigned long long)a[2], (unsigned long long)a[3]);
            return fail(ctx0, FQ_ERR_ARG, msg);
        }
    }
    // 2. sum the blocks
    const uint32_t C = (uint32_t)cap;
    const OverlapLayout L = OverlapLayout::make(C);
    std::vector<uint64_t> sum(L.total, 0), blk;
    for (int i = 0; i < n; ++i) {
        fq_ctx *const ctx = ctxs[i];
        fq_ctx::Overlap &V = ctx->ovl;
        sum[kOvlPairs] += V.pairs;
        if (!V.cyc) continue;
        blk.assign(OverlapLayout::make(V.cyc).total, 0);
        CK(cudaSetDevice(ctx->device));
        CK(cudaMemcpy(blk.data(), V.d_acc.p, blk.size() * 8, cudaMemcpyDeviceToHost));
        overlap_add_relaid(blk.data(), V.cyc, sum.data(), C);
    }
    if (cm) {
        st = nccl_sum_u64(ctx0, cm, &sum);
        if (st != FQ_OK) return st;
    }
    // 3. the result: difference arrays prefix-summed, trailing zero entries dropped; the same on every context
    std::vector<uint64_t> ins(sum.begin() + L.ins, sum.begin() + L.ins + 2 * C), r1o(C), r2o(C), r1m(sum.begin() + L.m1, sum.begin() + L.m1 + C),
        r2m(sum.begin() + L.m2, sum.begin() + L.m2 + C);
    for (uint32_t x = 0; x < C; ++x) {
        r1o[x] = (x ? r1o[x - 1] : 0) + sum[L.d1 + x];
        r2o[x] = (x ? r2o[x - 1] : 0) + sum[L.d2 + x];
    }
    auto trimmed = [](std::vector<uint64_t> &v) { while (!v.empty() && !v.back()) v.pop_back(); return v.size(); };
    trimmed(ins);
    const size_t n_cyc = std::max({trimmed(r1o), trimmed(r2o), trimmed(r1m), trimmed(r2m)});
    for (auto *v : {&r1o, &r2o, &r1m, &r2m}) v->resize(n_cyc, 0);
    for (int i = 0; i < n; ++i) {
        fq_ctx *const ctx = ctxs[i];
        fq_ctx::Overlap &V = ctx->ovl;
        std::copy(sum.begin(), sum.begin() + kOvlPairs + 1, V.res);
        V.ins = ins; V.r1o = r1o; V.r1m = r1m; V.r2o = r2o; V.r2m = r2m;
        V.pairs = 0;
        if (V.cyc) {
            CK(cudaSetDevice(ctx->device));
            CK(cudaMemset(V.d_acc.p, 0, (size_t)OverlapLayout::make(V.cyc).total * 8));
        }
    }
    return FQ_OK;
}

// ---- overrepresented sequences: end of a pass, over one context or a table sharded over several ------------------------
// Every rank's u64 list on every rank, concatenated in rank order: the sizes, then the lists padded to the longest.
fq_status nccl_allgather_var(fq_ctx *ctx, const fq_comm *c, std::vector<uint64_t> mine, std::vector<uint64_t> *all)
{
    std::vector<uint64_t> sizes, padded;
    fq_status st = nccl_allgather_u64(ctx, c, std::vector<uint64_t>{mine.size()}, &sizes);
    if (st != FQ_OK) return st;
    const uint64_t most = std::max<uint64_t>(1, *std::max_element(sizes.begin(), sizes.end()));
    mine.resize(most, 0);
    st = nccl_allgather_u64(ctx, c, mine, &padded);
    if (st != FQ_OK) return st;
    all->clear();
    for (int j = 0; j < c->n_ranks; ++j) all->insert(all->end(), padded.begin() + (size_t)j * most, padded.begin() + (size_t)j * most + sizes[j]);
    return FQ_OK;
}

// The owner shard's keys that pass the report rule, appended to `sel` as {key, count} word pairs.
fq_status overrep_select(fq_ctx *ctx, const uint64_t min_count[2], std::vector<uint64_t> *sel)
{
    fq_ctx::Overrep &R = ctx->ovr;
    const uint32_t cap = 2 * (1000000u / R.min_ppm);            // at most floor(10^6 / ppm) keys per mate pass
    CK(cudaSetDevice(ctx->device));
    CK(R.d_sel.ensure((size_t)cap * sizeof(KmerSlot)));
    CK(cudaMemsetAsync(R.T.d_scalars.p, 0, 8, ctx->stream));
    uint32_t *const d_n = R.T.d_scalars.as<uint32_t>();
    k_overrep_select<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(table_of(R.T), min_count[0], min_count[1], R.d_sel.as<KmerSlot>(), cap, d_n);
    ctx->launches++;
    uint32_t n_sel = 0;
    CK(cudaMemcpyAsync(&n_sel, d_n, 4, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (n_sel > cap) return fail(ctx, FQ_ERR_STATE, "overrepresented sequences: more keys pass the threshold than the reads allow");
    std::vector<KmerSlot> e(n_sel);
    if (n_sel) CK(cudaMemcpy(e.data(), R.d_sel.p, (size_t)n_sel * sizeof(KmerSlot), cudaMemcpyDeviceToHost));
    for (const KmerSlot &x : e) { sel->push_back(x.key); sel->push_back(x.count); }
    return FQ_OK;
}

// The context's captured entries whose key is in `keys`, appended to `out` as whole store entries (stride / 8 words each).
fq_status overrep_captured(fq_ctx *ctx, const std::map<uint64_t, uint64_t> &keys, std::vector<uint64_t> *out)
{
    fq_ctx::Overrep &R = ctx->ovr;
    if (!R.store_cap || keys.empty()) return FQ_OK;
    const size_t words = overrep_stride(R.prefix_len) / 8;
    std::vector<uint64_t> h(R.store_cap * words);
    CK(cudaSetDevice(ctx->device));
    CK(cudaMemcpy(h.data(), R.d_store.as<uint8_t>() + 64, h.size() * 8, cudaMemcpyDeviceToHost));
    for (uint64_t i = 0; i < R.store_cap; ++i) {
        const uint64_t *const e = h.data() + i * words;
        if (e[0] != kKmerEmpty && keys.count(e[0])) out->insert(out->end(), e, e + words);
    }
    return FQ_OK;
}

// A cleared count table and capture store for the next pass.
fq_status overrep_clear(fq_ctx *ctx)
{
    fq_ctx::Overrep &R = ctx->ovr;
    R.reads[0] = R.reads[1] = 0;
    R.T.occupied_bound = 0;
    R.store_bound = 0;
    CK(cudaSetDevice(ctx->device));
    k_kmer_clear<<<ctx->sm_count * 8, 256, 0, ctx->stream>>>(table_of(R.T));
    ctx->launches++;
    if (R.store_cap) {
        CK(cudaMemsetAsync(R.d_store.p, 0, 8, ctx->stream));
        k_overrep_store_clear<<<ctx->sm_count * 4, 256, 0, ctx->stream>>>(overrep_store_of(R));
        ctx->launches++;
    }
    CK(cudaStreamSynchronize(ctx->stream));
    R.T.d_send.release();
    R.T.d_recv.release();
    return FQ_OK;
}

fq_status overrep_end_pass_impl(fq_ctx *const *ctxs, int n, const fq_comm *cm, uint32_t n_shards, uint32_t rank0)
{
    fq_ctx *const ctx0 = ctxs[0];
    fq_status st = sync_all(ctxs, n);
    if (st != FQ_OK) return st;
    // 1. agree on the parameters; occupied slots per owner: header {enabled, prefix_len << 32 | min_ppm, reads of mate 1, of mate 2, counts[n_shards]}
    const size_t H = kHeadCounts + n_shards;
    std::vector<uint64_t> head((size_t)n_shards * H, 0);
    for (int i = 0; i < n; ++i) {
        fq_ctx::Overrep &R = ctxs[i]->ovr;
        uint64_t *h = head.data() + (size_t)(rank0 + i) * H;
        h[0] = R.enabled; h[1] = (uint64_t)R.prefix_len << 32 | R.min_ppm; h[2] = R.reads[0]; h[3] = R.reads[1];
        if (R.enabled && n_shards > 1) {
            st = table_owner_counts(ctxs[i], R.T, n_shards, h + kHeadCounts);
            if (st != FQ_OK) return st;
        }
    }
    if (cm) {
        const std::vector<uint64_t> mine(head.begin() + (size_t)rank0 * H, head.begin() + (size_t)(rank0 + 1) * H);
        st = nccl_allgather_u64(ctx0, cm, mine, &head);
        if (st != FQ_OK) return st;
    }
    uint64_t enabled = 0, reads[2] = {0, 0};
    for (uint32_t j = 0; j < n_shards; ++j) {
        const uint64_t *h = head.data() + (size_t)j * H;
        enabled += h[0];
        reads[0] += h[2];
        reads[1] += h[3];
    }
    if (!enabled) return fail(ctx0, FQ_ERR_STATE, "fq_overrep_end_pass_all: overrepresented sequences are not enabled (fq_overrep_enable)");
    if (enabled != n_shards) return fail(ctx0, FQ_ERR_ARG, "fq_overrep_end_pass_all: overrepresented sequences are enabled on some contexts only");
    for (uint32_t j = 1; j < n_shards; ++j) {
        const uint64_t a = head[1], b = head[(size_t)j * H + 1];
        if (a != b) {
            char msg[200];
            snprintf(msg, sizeof msg, "fq_overrep_end_pass_all: context %u has prefix_len = %llu, min_ppm = %llu; context 0 prefix_len = %llu, min_ppm = %llu", j,
                     (unsigned long long)(b >> 32), (unsigned long long)(b & 0xffffffffu), (unsigned long long)(a >> 32), (unsigned long long)(a & 0xffffffffu));
            return fail(ctx0, FQ_ERR_ARG, msg);
        }
    }
    const uint32_t prefix_len = (uint32_t)(head[1] >> 32), ppm = (uint32_t)(head[1] & 0xffffffffu);
    uint64_t min_count[2];
    for (int m = 0; m < 2; ++m) min_count[m] = std::max<uint64_t>(2, (ppm * reads[m] + 999999) / 1000000);
    // 2. exchange the groups and merge
    if (n_shards > 1) {
        st = table_exchange(ctxs, n, cm, rank0, n_shards, [](fq_ctx *c) -> HashTable & { return c->ovr.T; }, head, H);
        if (st != FQ_OK) return st;
    }
    // 3. select on each owner; 4. the selected {key, count} and the captured entries of those keys, from every shard
    std::vector<uint64_t> sel, all;
    for (int i = 0; i < n; ++i) {
        st = overrep_select(ctxs[i], min_count, &sel);
        if (st != FQ_OK) return st;
    }
    if (cm) {
        st = nccl_allgather_var(ctx0, cm, sel, &all);
        if (st != FQ_OK) return st;
        sel.swap(all);
    }
    std::map<uint64_t, uint64_t> count;
    for (size_t k = 0; k < sel.size(); k += 2) count[sel[k]] = sel[k + 1];
    std::vector<uint64_t> cap;
    for (int i = 0; i < n; ++i) {
        st = overrep_captured(ctxs[i], count, &cap);
        if (st != FQ_OK) return st;
    }
    if (cm) {
        st = nccl_allgather_var(ctx0, cm, cap, &all);
        if (st != FQ_OK) return st;
        cap.swap(all);
    }
    // 5. join and order: count descending, mate ascending, bytes ascending (memcmp on the common length, shorter first)
    const size_t words = overrep_stride(prefix_len) / 8;
    std::map<uint64_t, const uint8_t *> entry;
    for (size_t k = 0; k < cap.size(); k += words) entry.emplace(cap[k], reinterpret_cast<const uint8_t *>(cap.data() + k));
    struct Seq { uint64_t count; uint32_t mate, len; const uint8_t *s; };
    std::vector<Seq> seqs;
    for (const auto &kv : count) {
        const auto it = entry.find(kv.first);
        if (it == entry.end()) {
            char msg[200];
            snprintf(msg, sizeof msg, "fq_overrep_end_pass_all: key %016llx (mate %llu, %llu reads) passed the threshold, but no context captured its bytes",
                     (unsigned long long)kv.first, (unsigned long long)(kv.first & 1) + 1, (unsigned long long)kv.second);
            return fail(ctx0, FQ_ERR_STATE, msg);
        }
        uint32_t hdr[2];
        memcpy(hdr, it->second + 8, 8);
        seqs.push_back(Seq{kv.second, (uint32_t)(kv.first & 1) + 1, hdr[0], it->second + 16});
    }
    std::sort(seqs.begin(), seqs.end(), [](const Seq &a, const Seq &b) {
        if (a.count != b.count) return a.count > b.count;
        if (a.mate != b.mate) return a.mate < b.mate;
        const int c = memcmp(a.s, b.s, std::min(a.len, b.len));
        return c ? c < 0 : a.len < b.len;
    });
    std::vector<fq_overrep_seq> out;
    std::vector<uint8_t> bytes;
    for (const Seq &q : seqs) {
        out.push_back(fq_overrep_seq{q.count, q.mate, q.len, bytes.size()});
        bytes.insert(bytes.end(), q.s, q.s + q.len);
    }
    // 6. the same result on every context, then a cleared table and store
    for (int i = 0; i < n; ++i) {
        fq_ctx::Overrep &R = ctxs[i]->ovr;
        R.res_prefix_len = prefix_len;
        R.res_min_ppm = ppm;
        for (int m = 0; m < 2; ++m) { R.res_reads[m] = reads[m]; R.res_min_count[m] = min_count[m]; }
        R.seqs = out;
        R.bytes = bytes;
        st = overrep_clear(ctxs[i]);
        if (st != FQ_OK) return st;
    }
    return FQ_OK;
}

// ---- per flowcell tile quality: end of a pass, over one context or several ---------------------------------------------
// The contexts' key lists are united (gathered on the host, or NCCL all-gathers across ranks) and sorted by (lane, tile);
// every context's block is laid out in union order for the largest cycle capacity of any, and the blocks are summed (on
// the host, or one ncclAllReduce).  The same result goes to every context, then the tables and blocks are cleared.
fq_status tile_qual_clear(fq_ctx *ctx)
{
    fq_ctx::TileQual &Q = ctx->tq;
    CK(cudaSetDevice(ctx->device));
    k_kmer_clear<<<ctx->sm_count * 2, 256, 0, ctx->stream>>>(tile_table_of(Q));
    ctx->launches++;
    CK(cudaMemsetAsync(Q.d_cnt.p, 0, sizeof(TileCounters), ctx->stream));
    if (Q.L.D) CK(cudaMemsetAsync(Q.d_acc.p, 0, Q.L.total() * 8, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    Q.n_mates = 0;
    Q.reads[0] = Q.reads[1] = 0;
    Q.longest = Q.claims = Q.overflow = 0;
    Q.batch_open = Q.failed = false;
    return FQ_OK;
}

fq_status tile_qual_end_pass_impl(fq_ctx *const *ctxs, int n, const fq_comm *cm, uint32_t n_shards, uint32_t rank0)
{
    fq_ctx *const ctx0 = ctxs[0];
    fq_status st = sync_all(ctxs, n);
    if (st != FQ_OK) return st;
    // 1. header {enabled, mates (0: no batch), overflow, longest, cycle capacity, reads[2], untiled[2], a batch failed};
    //    each context's keys by dense id
    const size_t H = 10;
    std::vector<uint64_t> head((size_t)n_shards * H, 0), all_keys;
    std::vector<std::vector<uint64_t>> key_of(n);
    std::vector<KmerSlot> slots(kTileSlots);
    for (int i = 0; i < n; ++i) {
        fq_ctx *const ctx = ctxs[i];
        fq_ctx::TileQual &Q = ctx->tq;
        uint64_t *h = head.data() + (size_t)(rank0 + i) * H;
        h[0] = Q.enabled;
        if (!Q.enabled) continue;
        TileCounters tc{};
        CK(cudaSetDevice(ctx->device));
        CK(cudaMemcpy(&tc, Q.d_cnt.p, sizeof tc, cudaMemcpyDeviceToHost));
        CK(cudaMemcpy(slots.data(), Q.d_slots.p, slots.size() * sizeof(KmerSlot), cudaMemcpyDeviceToHost));
        key_of[i].assign(tc.claims, kKmerEmpty);
        for (const KmerSlot &e : slots)
            if (e.key != kKmerEmpty && e.count >= 1 && e.count <= tc.claims) key_of[i][e.count - 1] = e.key;
        h[1] = Q.n_mates; h[2] = tc.overflow; h[3] = Q.longest; h[4] = Q.L.C;
        h[5] = Q.reads[0]; h[6] = Q.reads[1]; h[7] = tc.untiled[0]; h[8] = tc.untiled[1];
        h[9] = Q.failed || Q.batch_open;
        all_keys.insert(all_keys.end(), key_of[i].begin(), key_of[i].end());
    }
    if (cm) {
        const std::vector<uint64_t> mine(head.begin() + (size_t)rank0 * H, head.begin() + (size_t)(rank0 + 1) * H);
        st = nccl_allgather_u64(ctx0, cm, mine, &head);
        if (st != FQ_OK) return st;
        st = nccl_allgather_var(ctx0, cm, std::vector<uint64_t>(all_keys), &all_keys);
        if (st != FQ_OK) return st;
    }
    uint64_t enabled = 0, n_mates = 0, overflow = 0, longest = 0, cap = 0, reads[2] = {0, 0}, untiled[2] = {0, 0}, failed = 0;
    for (uint32_t j = 0; j < n_shards; ++j) {
        const uint64_t *h = head.data() + (size_t)j * H;
        enabled += h[0];
        if (h[1] && n_mates && h[1] != n_mates) return fail(ctx0, FQ_ERR_ARG, "fq_tile_qual_end_pass_all: some contexts counted paired batches, others single-end ones");
        if (h[1]) n_mates = h[1];
        overflow |= h[2];
        longest = std::max(longest, h[3]);
        cap = std::max(cap, h[4]);
        for (int m = 0; m < 2; ++m) { reads[m] += h[5 + m]; untiled[m] += h[7 + m]; }
        failed |= h[9];
    }
    if (!enabled) return fail(ctx0, FQ_ERR_STATE, "fq_tile_qual_end_pass_all: per flowcell tile quality is not enabled (fq_tile_qual_enable)");
    if (enabled != n_shards) return fail(ctx0, FQ_ERR_ARG, "fq_tile_qual_end_pass_all: per flowcell tile quality is enabled on some contexts only");
    if (failed) {           // no partial result: the pass is dropped and the contexts are ready for the next one
        for (int i = 0; i < n; ++i) {
            st = tile_qual_clear(ctxs[i]);
            if (st != FQ_OK) return st;
        }
        return fail(ctx0, FQ_ERR_STATE, "fq_tile_qual_end_pass_all: a batch of this pass failed, so the pass has no result");
    }
    // 2. the union, ascending by (lane, tile); more than kTileMaxKeys keys: no table
    std::sort(all_keys.begin(), all_keys.end());
    all_keys.erase(std::unique(all_keys.begin(), all_keys.end()), all_keys.end());
    if (all_keys.size() > kTileMaxKeys) overflow = 1;
    if (overflow) all_keys.clear();
    const uint32_t U = (uint32_t)all_keys.size(), cycles = (uint32_t)std::min<uint64_t>(longest, kTileMaxCycles);
    // 3. the blocks in union order, summed
    const uint32_t M = (uint32_t)n_mates;
    const TileLayout S{M * U, (uint32_t)cap};
    std::vector<uint64_t> sum(U ? S.total() : 0, 0), blk;
    for (int i = 0; i < n && U; ++i) {
        fq_ctx *const ctx = ctxs[i];
        const TileLayout L = ctx->tq.L;
        if (!ctx->tq.n_mates) continue;                   // no batch here this pass
        if ((uint64_t)M * key_of[i].size() > L.D) return fail(ctx0, FQ_ERR_STATE, "fq_tile_qual_end_pass_all: internal: a context's block is smaller than its keys");
        blk.resize(L.total());
        CK(cudaSetDevice(ctx->device));
        CK(cudaMemcpy(blk.data(), ctx->tq.d_acc.p, blk.size() * 8, cudaMemcpyDeviceToHost));
        for (uint32_t id = 0; id < key_of[i].size(); ++id) {
            const uint32_t u = (uint32_t)(std::lower_bound(all_keys.begin(), all_keys.end(), key_of[i][id]) - all_keys.begin());
            for (uint32_t m = 0; m < M; ++m) {
                const uint32_t d = M * id + m, e = M * u + m;
                sum[S.bases(e)] += blk[L.bases(d)];
                sum[S.qual(e)] += blk[L.qual(d)];
                for (uint32_t b = 0; b <= L.C; ++b) sum[S.hist(b, e)] += blk[L.hist(b, d)];
                for (uint32_t c = 0; c < L.C; ++c) sum[S.cyc(c, e)] += blk[L.cyc(c, d)];
            }
        }
    }
    if (cm && U) {
        st = nccl_sum_u64(ctx0, cm, &sum);
        if (st != FQ_OK) return st;
    }
    // 4. the result, [tile][mate] and [tile][mate][cycle]; bases at cycle c are the reads longer than c
    std::vector<uint32_t> lane(U), tile(U);
    std::vector<uint64_t> t_reads((size_t)U * M), t_bases((size_t)U * M), t_qsum((size_t)U * M), c_bases((size_t)U * M * cycles),
        c_qsum((size_t)U * M * cycles);
    for (uint32_t u = 0; u < U; ++u) {
        lane[u] = (uint32_t)(all_keys[u] >> 32);
        tile[u] = (uint32_t)all_keys[u];
        for (uint32_t m = 0; m < M; ++m) {
            const uint32_t e = M * u + m;
            const size_t k = (size_t)u * M + m;
            uint64_t longer = 0;
            for (uint32_t b = S.C + 1; b-- > 0;) {
                if (b < cycles && b < S.C) {          // cycles past every tiled read stay 0
                    c_bases[k * cycles + b] = longer;
                    c_qsum[k * cycles + b] = sum[S.cyc(b, e)];
                }
                longer += sum[S.hist(b, e)];
            }
            t_reads[k] = longer;
            t_bases[k] = sum[S.bases(e)];
            t_qsum[k] = sum[S.qual(e)];
        }
    }
    for (int i = 0; i < n; ++i) {
        fq_ctx::TileQual &Q = ctxs[i]->tq;
        Q.res_mates = M;
        Q.res_overflow = (uint32_t)overflow;
        Q.res_cycles = cycles;
        for (int m = 0; m < 2; ++m) { Q.res_reads[m] = reads[m]; Q.res_untiled[m] = untiled[m]; }
        Q.lane = lane; Q.tile = tile;
        Q.t_reads = t_reads; Q.t_bases = t_bases; Q.t_qsum = t_qsum; Q.c_bases = c_bases; Q.c_qsum = c_qsum;
        st = tile_qual_clear(ctxs[i]);
        if (st != FQ_OK) return st;
    }
    return FQ_OK;
}

}  // namespace

fq_status fq_kmer_end_pass_all(fq_ctx *const *ctxs, int n, fq_comm *const *comm)
{
    return end_pass_entry(ctxs, n, comm, "fq_kmer_end_pass_all", kmer_end_pass_impl);
}

fq_status fq_dup_enable(fq_ctx *ctx)
{
    if (!ctx) return FQ_ERR_ARG;
    fq_ctx::Dup &D = ctx->dup;
    if (D.enabled) return D.units ? fail(ctx, FQ_ERR_STATE, "fq_dup_enable: a pass is under way") : FQ_OK;
    CK(cudaSetDevice(ctx->device));
    CK(D.T.d_scalars.ensure(64));
    CK(D.d_small.ensure((size_t)kKmerSmallCounts * 8));
    CK(D.d_big.ensure((size_t)kKmerBigCap * 4));
    const fq_status st = table_resize(ctx, D.T, D.T.min_cap);
    if (st == FQ_OK) D.enabled = true;
    return st;
}

fq_status fq_dup_end_pass_all(fq_ctx *const *ctxs, int n, fq_comm *const *comm)
{
    return end_pass_entry(ctxs, n, comm, "fq_dup_end_pass_all", dup_end_pass_impl);
}

fq_status fq_dup_results(fq_ctx *ctx, fq_dup_view *view)
{
    if (!ctx || !view) return FQ_ERR_ARG;
    const fq_ctx::Dup &D = ctx->dup;
    if (!D.enabled) return fail(ctx, FQ_ERR_STATE, "fq_dup_results: duplication statistics are not enabled (fq_dup_enable)");
    view->units = D.res_units;
    view->distinct = D.res_distinct;
    view->n_levels = D.levels.size() / 2;
    view->levels = D.levels.data();
    return FQ_OK;
}

fq_status fq_overlap_enable(fq_ctx *ctx, uint32_t min_overlap, uint32_t diff_limit, uint32_t diff_percent)
{
    if (!ctx) return FQ_ERR_ARG;
    if (min_overlap == 0 || diff_percent > 100)
        return fail(ctx, FQ_ERR_ARG, "fq_overlap_enable: min_overlap must be at least 1 and diff_percent at most 100");
    fq_ctx::Overlap &V = ctx->ovl;
    if (V.enabled && V.pairs) return fail(ctx, FQ_ERR_STATE, "fq_overlap_enable: a pass is under way");
    V.enabled = true;
    V.min_overlap = min_overlap; V.diff_limit = diff_limit; V.diff_percent = diff_percent;
    return FQ_OK;
}

fq_status fq_overlap_end_pass_all(fq_ctx *const *ctxs, int n, fq_comm *const *comm)
{
    return end_pass_entry(ctxs, n, comm, "fq_overlap_end_pass_all", overlap_end_pass_impl);
}

fq_status fq_overlap_results(fq_ctx *ctx, fq_overlap_view *view)
{
    if (!ctx || !view) return FQ_ERR_ARG;
    const fq_ctx::Overlap &V = ctx->ovl;
    if (!V.enabled) return fail(ctx, FQ_ERR_STATE, "fq_overlap_results: the overlap profile is not enabled (fq_overlap_enable)");
    view->pairs = V.res[kOvlPairs];
    view->too_short = V.res[kOvlTooShort];
    view->overlapped = V.res[kOvlOverlapped];
    view->r1_adapter = V.res[kOvlR1Adapter];
    view->r2_adapter = V.res[kOvlR2Adapter];
    view->overlap_bases = V.res[kOvlOverlapBases];
    view->mismatch_bases = V.res[kOvlMismatchBases];
    view->n_insert = (uint32_t)V.ins.size();
    view->insert_hist = V.ins.data();
    view->n_cycles = (uint32_t)V.r1o.size();
    view->r1_overlap = V.r1o.data();
    view->r1_mismatch = V.r1m.data();
    view->r2_overlap = V.r2o.data();
    view->r2_mismatch = V.r2m.data();
    return FQ_OK;
}

fq_status fq_overrep_enable(fq_ctx *ctx, uint32_t prefix_len, uint32_t min_ppm)
{
    if (!ctx) return FQ_ERR_ARG;
    if (prefix_len < 1 || prefix_len > kOverrepMaxPrefix || min_ppm < 10 || min_ppm > 1000000)
        return fail(ctx, FQ_ERR_ARG, "fq_overrep_enable: prefix_len must be in 1..256 and min_ppm in 10..1000000");
    fq_ctx::Overrep &R = ctx->ovr;
    if (R.enabled && (R.reads[0] || R.reads[1])) return fail(ctx, FQ_ERR_STATE, "fq_overrep_enable: a pass is under way");
    CK(cudaSetDevice(ctx->device));
    CK(R.T.d_scalars.ensure(64));
    fq_status st = table_resize(ctx, R.T, R.T.min_cap);
    if (st != FQ_OK) return st;
    if (prefix_len != R.prefix_len) {              // the store's entries have another size: a new one at the first batch
        R.d_store.release();
        R.store_cap = R.store_bound = 0;
    }
    R.prefix_len = prefix_len;
    R.min_ppm = min_ppm;
    if (!R.enabled) { R.res_prefix_len = prefix_len; R.res_min_ppm = min_ppm; }
    R.enabled = true;
    return FQ_OK;
}

fq_status fq_overrep_end_pass_all(fq_ctx *const *ctxs, int n, fq_comm *const *comm)
{
    return end_pass_entry(ctxs, n, comm, "fq_overrep_end_pass_all", overrep_end_pass_impl);
}

fq_status fq_overrep_results(fq_ctx *ctx, fq_overrep_view *view)
{
    if (!ctx || !view) return FQ_ERR_ARG;
    const fq_ctx::Overrep &R = ctx->ovr;
    if (!R.enabled) return fail(ctx, FQ_ERR_STATE, "fq_overrep_results: overrepresented sequences are not enabled (fq_overrep_enable)");
    view->prefix_len = R.res_prefix_len;
    view->min_ppm = R.res_min_ppm;
    for (int m = 0; m < 2; ++m) { view->reads[m] = R.res_reads[m]; view->min_count[m] = R.res_min_count[m]; }
    view->n_seqs = R.seqs.size();
    view->seqs = R.seqs.data();
    view->bytes = R.bytes.data();
    return FQ_OK;
}

fq_status fq_tile_qual_enable(fq_ctx *ctx)
{
    if (!ctx) return FQ_ERR_ARG;
    fq_ctx::TileQual &Q = ctx->tq;
    if (Q.enabled) return Q.reads[0] || Q.reads[1] ? fail(ctx, FQ_ERR_STATE, "fq_tile_qual_enable: a pass is under way") : FQ_OK;
    CK(cudaSetDevice(ctx->device));
    CK(Q.d_slots.ensure((size_t)kTileSlots * sizeof(KmerSlot)));
    CK(Q.d_cnt.ensure(sizeof(TileCounters)));
    CK(Q.h_cnt.ensure(8));
    const fq_status st = tile_qual_clear(ctx);
    if (st == FQ_OK) Q.enabled = true;
    return st;
}

fq_status fq_tile_qual_end_pass_all(fq_ctx *const *ctxs, int n, fq_comm *const *comm)
{
    return end_pass_entry(ctxs, n, comm, "fq_tile_qual_end_pass_all", tile_qual_end_pass_impl);
}

fq_status fq_tile_qual_results(fq_ctx *ctx, fq_tile_qual_view *view)
{
    if (!ctx || !view) return FQ_ERR_ARG;
    const fq_ctx::TileQual &Q = ctx->tq;
    if (!Q.enabled) return fail(ctx, FQ_ERR_STATE, "fq_tile_qual_results: per flowcell tile quality is not enabled (fq_tile_qual_enable)");
    view->n_mates = Q.res_mates;
    view->overflow = Q.res_overflow;
    view->n_tiles = (uint32_t)Q.lane.size();
    view->cycles = Q.res_cycles;
    for (int m = 0; m < 2; ++m) { view->reads[m] = Q.res_reads[m]; view->untiled[m] = Q.res_untiled[m]; }
    view->lane = Q.lane.data();
    view->tile = Q.tile.data();
    view->tile_reads = Q.t_reads.data();
    view->tile_bases = Q.t_bases.data();
    view->tile_qsum = Q.t_qsum.data();
    view->cycle_bases = Q.c_bases.data();
    view->cycle_qsum = Q.c_qsum.data();
    return FQ_OK;
}

}  // extern "C"
