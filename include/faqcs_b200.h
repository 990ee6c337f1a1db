/*
 * faqcs_b200.h -- C ABI of the B200-native FaQCs trim / filter / statistics path.
 *
 * FaQCs (v2.10) has no plugin or FFI layer.  The narrowest seam the hot path
 * sits behind is the C++ function
 *
 *     void trim(std::vector<Read>&, std::vector<size_t>& filter_stats,
 *               MAP<std::string, std::pair<size_t,size_t>>& adapter_stats,
 *               MAP<Word,size_t>& kmer_table, PlotInfo&, Options&);   (FaQCs.h:245-248)
 *
 * called once per mate per batch from process_paired (FaQCs.cpp:287-291,424-428)
 * and process_unpaired (FaQCs.cpp:628,692), followed by the pair-routing / emit
 * loops (FaQCs.cpp:296-361,431-496,634-659,696-720).  This header is the C
 * restatement of that seam with record parsing moved across it: the caller
 * hands over raw FASTQ record bytes (what fastq.cpp:next_read would have
 * consumed) and gets back the bytes write_read (fastq.cpp:127-138) would have
 * produced for each of the four output files, plus the integer statistics that
 * write_stats (FaQCs.cpp:759-1034) and plot (plot.cpp:31-78) print.
 *
 * Conventions: plain pointers and sizes, no C++ / torch types, no exceptions.
 * Every entry point returns an fq_status; fq_last_error() gives the message
 * (for reference-defined failures, the reference's own text).  A context is
 * bound to one CUDA device and one host thread; contexts are independent.
 * There is NO CPU fallback: fq_create fails if no CUDA device is usable.
 */
#ifndef FAQCS_B200_H
#define FAQCS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define FQ_ABI_VERSION 4

/* ---- FilterStat (FaQCs.h:46-75), same order, same meaning ---------------- */
enum fq_filter_stat {
    FQ_TOTAL_COUNT = 0,
    FQ_TOTAL_NUMBER,
    FQ_TOTAL_LENGTH,
    FQ_TOTAL_TRIMMED_NUMBER,
    FQ_TOTAL_TRIMMED_LENGTH,
    FQ_PAIRED_READ_NUMBER,
    FQ_PAIRED_BASE_LENGTH,
    FQ_READ_LENGTH,
    FQ_BASE_LENGTH,
    FQ_READ_NN,
    FQ_BASE_NN,
    FQ_READ_PHIX,
    FQ_BASE_PHIX,
    FQ_READ_ADAPTER,
    FQ_BASE_ADAPTER,
    FQ_READ_AVG_Q,
    FQ_BASE_AVG_Q,
    FQ_READ_QUAL_TRIM,
    FQ_BASE_QUAL_TRIM,
    FQ_READ_LOW_COMPLEXITY,
    FQ_BASE_LOW_COMPLEXITY,
    FQ_N_TO_A,
    FQ_N_TO_T,
    FQ_N_TO_G,
    FQ_N_TO_C,
    FQ_NUM_STAT
};

#define FQ_MAX_QUALITY_SCORE   41     /* fastq.h:15 */
#define FQ_NUM_QUAL            42     /* columns of the quality matrices */
#define FQ_NUM_BASE            5      /* A,T,C,G,N   (FaQCs.h:35-42) */
#define FQ_NUM_COMPOSITION_BIN 10001  /* FaQCs.h:20 */
#define FQ_NUM_COMPOSITION     6      /* A,T,C,G,N,GC (NucleotideCount, FaQCs.h:167-192) */
#define FQ_REF_BATCH           32768  /* reads per trim() call in the reference (FaQCs.cpp:232,585) */
#define FQ_OFFSET_AUTO         (-128) /* AUTO_DETECT_QUALITY_OFFSET = SCHAR_MIN (FaQCs.h:13) */

/* Options::Mode (FaQCs.h:90-97) */
enum fq_mode { FQ_MODE_HARD = 0, FQ_MODE_BWA = 1, FQ_MODE_BWA_PLUS = 2 };

/* Output streams, in the order FaQCs names its files (options.cpp:696-741). */
enum fq_stream { FQ_OUT_R1 = 0, FQ_OUT_R2 = 1, FQ_OUT_UNPAIRED = 2, FQ_OUT_DISCARD = 3, FQ_NUM_STREAM = 4 };

typedef enum fq_status {
    FQ_OK = 0,
    FQ_ERR_ARG = 1,          /* bad argument */
    FQ_ERR_CUDA = 2,         /* CUDA runtime failure (message has the CUDA error string) */
    FQ_ERR_NO_DEVICE = 3,    /* no usable CUDA device: there is no CPU fallback */
    FQ_ERR_FORMAT = 4,       /* FASTQ grammar error (fastq.cpp:34-122 messages) */
    FQ_ERR_QUALITY = 5,      /* quality > 41 (fastq.h:31-33) or re-encode overflow (trim.cpp:521-523) */
    FQ_ERR_OFFSET = 6,       /* "Unknown quality format!" / inconsistent R1-R2 (trim.cpp:615, FaQCs.cpp:265-269) */
    FQ_ERR_BASE = 7,         /* "Unknown base!" in the aligner (seq_overlap.cpp:409) */
    FQ_ERR_STATE = 8         /* call order violated */
} fq_status;

/* One adapter / artifact target, in reference order (options.cpp:576-694). */
typedef struct fq_adapter {
    const char *name;
    const char *seq;
} fq_adapter;

/*
 * The subset of struct Options (FaQCs.h:77-144) that trim() reads.
 * Field meaning and C types follow the reference exactly (float stays float).
 */
typedef struct fq_options {
    int32_t  mode;                        /* fq_mode; Options::mode */
    int32_t  quality;                     /* -q, char in the reference */
    uint32_t trim_5;                      /* --5end */
    uint32_t trim_3;                      /* --3end */
    uint32_t min_read_length;             /* --min_L */
    uint32_t max_num_poly_N;              /* -n */
    float    average_quality;             /* --avg_q */
    float    low_complexity_cutoff_ratio; /* --lc */
    float    adapter_mismatch_rate;       /* --rate (filterAdapterMismatchRate) */
    int32_t  input_quality_offset;        /* --ascii; FQ_OFFSET_AUTO until detected */
    int32_t  output_quality_offset;       /* --out_ascii */
    uint32_t replace_to_N_q;              /* --replace_to_N_q */
    int32_t  qc_only;                     /* --qc_only */
    int32_t  protect_5;                   /* --5trim_off */
    int32_t  filter_adapter;              /* adapter pass enabled (filter_adapter || filter_phiX, trim.cpp:86) */
    int32_t  discard_output;              /* --discard: emit raw records of invalid reads */
    /*
     * Thread-count emulation for the adapter match threshold (SURVEY Q3,
     * trim.cpp:985,996-1008,1074-1082): the reference's threshold depends on
     * how libgomp's static schedule cuts each 32768-read batch into per-thread
     * chunks and 8-read SIMD groups.  num_thread = the -t the reference would
     * run with (>=1).  0 disables the emulation: every read uses
     * int(float(1-rate) * min(own length, |adapter|)), which equals the
     * reference whenever every read is at least as long as every adapter.
     */
    uint32_t num_thread;
    uint32_t n_adapters;
    const fq_adapter *adapters;
} fq_options;

/* Per-read verdict, for tests and debugging (one entry per record per mate). */
typedef struct fq_read_result {
    uint32_t offset_5;   /* bases removed from the 5' end, original coordinates (trim.cpp:236) */
    uint32_t length;     /* final length (0 if the read is invalid) */
    uint16_t flags;      /* FQ_RR_* */
    int16_t  adapter;    /* index of the best matching adapter, -1 if none (trim.cpp:1036-1040) */
    float    avg_q;      /* average_quality of the trimmed read (trim.cpp:374) */
} fq_read_result;

#define FQ_RR_VALID          0x0001  /* trim_read returned true */
#define FQ_RR_F_LENGTH       0x0002  /* counted in READ_LENGTH */
#define FQ_RR_F_NN           0x0004  /* counted in READ_NN */
#define FQ_RR_F_AVGQ         0x0008  /* counted in READ_AVG_Q */
#define FQ_RR_F_LOWCOMP      0x0010  /* counted in READ_LOW_COMPLEXITY */
#define FQ_RR_QUAL_TRIMMED   0x0020  /* counted in READ_QUAL_TRIM */
#define FQ_RR_ADAPTER        0x0040  /* an adapter clipped this read */

/* One piece of an output stream (pieces mode, fq_set_output_pieces): `length` bytes starting at `offset` of
 * source 0 = the r1 buffer handed to this batch, 1 = the r2 buffer, 2 = this stream's literal bytes (fq_batch_out.data). */
typedef struct fq_out_piece {
    uint64_t offset;
    uint32_t length;
    uint32_t source;
} fq_out_piece;

/* Result of one batch.  Host pointers are owned by the context and stay valid
 * until the next fq_process_* / fq_submit on the same context. */
typedef struct fq_batch_out {
    const uint8_t *data[FQ_NUM_STREAM];   /* emitted FASTQ bytes per stream (NULL if empty / qc_only); pieces mode: the literal bytes */
    uint64_t       bytes[FQ_NUM_STREAM];  /* size of each stream (in pieces mode too) */
    uint64_t       n_records;             /* records per mate in this batch */
    uint64_t       n_valid[2];            /* surviving reads per mate */
    uint64_t       paired_read_number;    /* PAIRED_READ_NUMBER increment (FaQCs.cpp:304-308) */
    uint64_t       paired_base_length;
    const fq_read_result *results[2];     /* per-read verdicts (only if debug results were requested) */
    /* pieces mode: each stream as a list of pieces in stream order (concatenating them gives the `bytes[s]` stream bytes) */
    const fq_out_piece *pieces[FQ_NUM_STREAM];
    uint64_t       n_pieces[FQ_NUM_STREAM];
    uint64_t       literal_bytes[FQ_NUM_STREAM];
} fq_batch_out;

/* Flattened statistics (SURVEY Appendix D).  All counters are u64 like the
 * reference's size_t.  Pointers are host memory owned by the context. */
typedef struct fq_stats_view {
    uint64_t filter_stats[FQ_NUM_STAT];
    uint32_t n_adapters;
    const uint64_t *adapter_reads;        /* [n_adapters], index = adapter order */
    const uint64_t *adapter_bases;        /* [n_adapters] */
    uint32_t pre_rows, post_rows;         /* rows of the position-indexed matrices (matrix.h growth rule) */
    uint32_t pre_len_size, post_len_size; /* size() of the length histograms (trim.cpp:877-885) */
    const uint64_t *pre_quality_matrix;   /* [pre_rows][42]  (trim.cpp:795-808) */
    const uint64_t *post_quality_matrix;  /* [post_rows][42] */
    const uint64_t *pre_base_matrix;      /* [pre_rows][5] A,T,C,G,N (trim.cpp:810-858) */
    const uint64_t *post_base_matrix;     /* [post_rows][5] */
    const uint64_t *pre_read_quality_hist;  /* [42] (trim.cpp:254-258) */
    const uint64_t *pre_base_quality_hist;  /* [42] */
    const uint64_t *post_read_quality_hist; /* [42] (trim.cpp:539-543) */
    const uint64_t *post_base_quality_hist; /* [42] */
    const uint64_t *pre_composition;      /* [6][10001]: A,T,C,G,N,GC (trim.cpp:860-874) */
    const uint64_t *post_composition;     /* [6][10001] */
    const uint64_t *pre_length_hist;      /* [pre_len_size] */
    const uint64_t *post_length_hist;     /* [post_len_size] */
} fq_stats_view;

typedef struct fq_ctx fq_ctx;

/* Library / build identification. */
int         fq_abi_version(void);
const char *fq_build_info(void);     /* e.g. "faqcs_b200 sm_100a nvcc 12.9" */

/* Create a context on CUDA device `device`.  Options are copied (incl. adapters).
 * Replaces: Options consumed by trim() (FaQCs.h:245-248) + PlotInfo / filter_stats
 * construction in main (FaQCs.cpp:67-69). */
fq_status fq_create(const fq_options *opt, int device, fq_ctx **out);
void      fq_destroy(fq_ctx *ctx);
const char *fq_last_error(const fq_ctx *ctx);   /* ctx may be NULL: last create error */

/* Pieces mode (off by default).  The routing loops of the reference write every surviving read back out
 * (FaQCs.cpp:296-361, 431-496, 634-659, 696-720; write_read, fastq.cpp:127-138) although almost all of them are untouched.
 * With pieces on, fq_batch_out describes each stream as a list of fq_out_piece: byte ranges of the CALLER'S input buffers
 * (runs of untouched records) and ranges of a small literal buffer (the records that changed).  A writer hands the list to
 * writev(2); nothing but the literal bytes and the list crosses the PCIe link on the way back. */
fq_status fq_set_output_pieces(fq_ctx *ctx, int enable);
/* Ask for per-read verdicts in fq_batch_out.results (off by default). */
fq_status fq_set_debug_results(fq_ctx *ctx, int enable);
/* parse_id(r1.def) == parse_id(r2.def) check of FaQCs.cpp:383-389 (on by default). */
fq_status fq_set_check_pair_ids(fq_ctx *ctx, int enable);
/* Change Options::quality (-q) between batches: the reference's drivers do this when a batch "looks like NextSeq data"
 * (m_opt.quality = DEFAULT_NEXTSEQ_QUALITY_SCORE, FaQCs.cpp:272-277, 406-411, 613-618, 675-680); fq_autodetect covers the
 * first batch, this call the re-check the reference makes on its final partial 32768-read batch. */
fq_status fq_set_quality(fq_ctx *ctx, int32_t quality);

/* Pinned host memory for the buffers handed to fq_process_host (pageable memory
 * works too, but the copies then cannot overlap and run at a fraction of PCIe speed). */
void *fq_host_alloc(size_t bytes);
void  fq_host_free(void *p);

/* Quality-offset auto-detection on the first batch (auto_detect_quality_offset,
 * trim.cpp:599-617, call sites FaQCs.cpp:261-270,393-402,609-611,669-671) and
 * NextSeq detection (auto_detect_next_seq, trim.cpp:619-626; raises -q to 20,
 * FaQCs.cpp:272-277,404-414).  r2 may be NULL (unpaired).  Only the first
 * FQ_REF_BATCH records are inspected.  Updates the context's options and
 * returns the detected values.  Runs on the device. */
fq_status fq_autodetect(fq_ctx *ctx, const uint8_t *r1, size_t n1,
                        const uint8_t *r2, size_t n2,
                        int32_t *input_quality_offset, int32_t *quality);

/* Process one batch of whole FASTQ records given as HOST buffers: copies to the
 * device, frames records, trims/filters, accumulates statistics, compacts the
 * four output streams in input order and copies them back.
 * Replaces: trim() x2 + the routing/emit loop for one batch
 * (FaQCs.cpp:279-361 / 416-496 / 621-659 / 685-720).
 * first_record_index: global index of the batch's first record in its file
 * (used for thread-count emulation and for the k-mer rarefaction's trim() call
 * numbers); is_final: last batch of the file. */
fq_status fq_process_host(fq_ctx *ctx, const uint8_t *r1, size_t n1,
                          const uint8_t *r2, size_t n2,
                          uint64_t first_record_index, int is_final,
                          fq_batch_out *out);

/* Pipelined form of fq_process_host for streaming runs.  fq_submit_host starts the host->device
 * copy of a batch on its own stream and returns a ticket; fq_run executes the kernels for that
 * ticket and starts the device->host copy of its outputs on another stream; fq_wait blocks until
 * those outputs are in host memory.  Two batches can be in flight, so the usual loop is
 *     submit(i+1); run(i); wait(i-1);
 * which overlaps upload(i+1), compute(i) and download(i-1).  Tickets must be run and waited in
 * submission order; the input buffers must stay valid until fq_run(ticket) has returned, the
 * output pointers until the ticket two submissions later is run. */
fq_status fq_submit_host(fq_ctx *ctx, const uint8_t *r1, size_t n1,
                         const uint8_t *r2, size_t n2,
                         uint64_t first_record_index, int is_final, uint64_t *ticket);
fq_status fq_run(fq_ctx *ctx, uint64_t ticket);
fq_status fq_wait(fq_ctx *ctx, uint64_t ticket, fq_batch_out *out);

/* Same, with the raw bytes already resident in device memory (d_r1/d_r2 are
 * device pointers on the context's device).  Output stays on the device unless
 * copy_out != 0; out->data then points at host copies as above.  With
 * copy_out == 0 the device-side output pointers can be fetched with
 * fq_device_outputs. */
fq_status fq_process_device(fq_ctx *ctx, const void *d_r1, size_t n1,
                            const void *d_r2, size_t n2,
                            uint64_t first_record_index, int is_final,
                            int copy_out, fq_batch_out *out);
fq_status fq_device_outputs(fq_ctx *ctx, const void *d_out[FQ_NUM_STREAM]);

/* Device time (ms, CUDA events on the context's stream) of the last fq_process_*
 * call, by segment: ms[0] all kernels, ms[1] framing, ms[2] pair-id check +
 * adapter pass, ms[3] trim/filter/statistics kernel, ms[4] route + scan + emit.
 * Fills min(n, 5) entries. */
fq_status fq_last_timing(fq_ctx *ctx, float *ms, int n);
/* Number of kernel launches issued by the context so far. */
uint64_t  fq_launch_count(const fq_ctx *ctx);
/* CUDA stream of the context as a void* (cudaStream_t), for event timing by the caller. */
void     *fq_stream(fq_ctx *ctx);

/* Statistics accumulated so far (device -> host copy; u32 batch accumulators
 * are already folded into the u64 totals).
 * Replaces: reads of filter_stats / adapter_stats / PlotInfo after the batch
 * loop (FaQCs.cpp:92-133). */
fq_status fq_stats(fq_ctx *ctx, fq_stats_view *view);

/* Multi-GPU merge (the reference's `omp critical` merge, trim.cpp:120-154, across
 * devices): the accumulators live in one flat u64 block in DEVICE memory whose
 * layout depends only on (row capacity, n_adapters).  Every rank first calls
 * fq_stats_reserve_rows with the same capacity (>= the longest read of any
 * rank), then all-reduces the block with SUM and the 4 x u32 row counters with
 * MAX (ncclAllReduce over NVLink; the only collective of the path).  fq_stats
 * afterwards returns the merged statistics on every rank. */
fq_status fq_stats_reserve_rows(fq_ctx *ctx, uint32_t rows);
fq_status fq_stats_device_buffer(fq_ctx *ctx, void **d_u64, size_t *n_u64,
                                 void **d_rows_u32x4);

/*
 * The collective itself, inside the library (SURVEY 8(b) fq_allreduce_stats, 8(e)): merges the accumulators of n contexts
 * -- all n ranks of a single-process run, or this process's one context of an n-rank job -- with ONE ncclAllReduce
 * (ncclUint64, ncclSum) over the flat statistics block, preceded by an agreement on the row capacity and followed by an
 * ncclAllReduce(ncclMax) of the four row counters.  Replaces the `omp critical` merge of trim() (trim.cpp:120-154) and the
 * matrix / vector operator+= it uses (matrix.h:111-142, trim.cpp:47-65) across devices.  Afterwards fq_stats returns the
 * merged statistics on every context.  NCCL is loaded at run time (libnccl.so.2); FQ_ERR_STATE if it is not available.
 *
 * fq_comm wraps one ncclComm_t bound to one context's device.
 *   single process, n devices:  fq_comm_init_all(ctx, n, comms);           fq_allreduce_stats(ctx, n, comms);
 *   one process per device:     rank 0: fq_comm_unique_id(id); broadcast id with the job's launcher;
 *                               fq_comm_init_rank(ctx, n_ranks, rank, id, &comm);   fq_allreduce_stats(&ctx, 1, &comm);
 */
typedef struct fq_comm fq_comm;
#define FQ_COMM_ID_BYTES 128
fq_status fq_comm_unique_id(uint8_t id[FQ_COMM_ID_BYTES]);
fq_status fq_comm_init_rank(fq_ctx *ctx, int n_ranks, int rank, const uint8_t id[FQ_COMM_ID_BYTES], fq_comm **out);
fq_status fq_comm_init_all(fq_ctx *const *ctx, int n, fq_comm **out);
void      fq_comm_destroy(fq_comm *comm);
fq_status fq_allreduce_stats(fq_ctx *const *ctx, int n, fq_comm *const *comm);
/* Contexts on the SAME device (a context holds one batch in flight; two of them driven by two host threads overlap
 * consecutive batches on the device): dst += src, src = 0 -- the merge of trim.cpp:120-154 without a communicator. */
fq_status fq_merge_stats(fq_ctx *dst, fq_ctx *src);
/* Device milliseconds of the last fq_allreduce_stats on this context (CUDA events around the three collectives). */
float     fq_last_allreduce_ms(const fq_ctx *ctx);

/*
 * k-mer rarefaction (--kmer_rarefaction; SURVEY 8(f) N4).  Replaces update_kmer (trim.cpp:887-931, called from
 * trim_read: on the raw read under --qc_only, trim.cpp:260-262, on what is left of a surviving read otherwise, trim.cpp:545-547), the sampling block at the end of trim() (trim.cpp:157-185) and the end-of-pass code of
 * process_paired / process_unpaired (FaQCs.cpp:518-537, 737-756).  The canonical k-mers of the raw reads go to a hash table
 * in device memory while the curve is being collected (one table per pass over an input, as in the reference); the points
 * of the curve are taken where the reference takes them -- at the end of the trim() call (32768 reads of one mate) whose
 * running read count crossed another multiple of split_size -- so batches must start on 32768-record boundaries and, unless
 * final, hold a multiple of 32768 records.  A batch's calls follow from its first_record_index (the global index of its
 * first record in the input): call = (first_record_index / 32768 + chunk) * n_mates + mate, so the batches of a pass may run
 * in any order and on several contexts, each batch exactly once.
 *   fq_kmer_enable        once, before the first batch: k (Options::kmer, 2..31), Options::split_size, Options::num_subsample
 *                         (already doubled where the reference doubles it, options.cpp:506-523); the same on every context
 *   fq_kmer_end_pass      after the last batch of an input (paired files, then the unpaired file), one context
 *   fq_kmer_end_pass_all  the same for a table sharded over several contexts (below)
 *   fq_kmer_results       PlotInfo::kmer_rarefaction and PlotInfo::kmer_frequency_histogram (what plot.cpp:683-733 prints);
 *                         the view's pointers belong to the context and stay valid until its next fq_kmer_* call
 *
 * Sharded table: every context counts its own batches into its own table.  At the end of the pass every k-mer has one owner
 * context (from the high half of its hash); the contexts send their entries to the owners in n - 1 rounds (in round r,
 * context i sends its group for i + r and receives the group of i - r: memory = the context's entries + one received group),
 * and each owner merges them into its cleared table (counts add, first calls take the minimum).  The owners' summaries are
 * then summed, so every context ends the pass with the same curve, histogram and state.  FQ_ERR_ARG if the contexts differ in
 * k, split_size or num_subsample, or if a trim() call below the highest one was run other than exactly once.
 */
typedef struct fq_rarefaction {
    uint64_t num_seq;          /* TOTAL_NUMBER when the point was taken */
    uint64_t distinct_kmer;
    uint64_t total_kmer;
} fq_rarefaction;
typedef struct fq_kmer_view {
    uint32_t n_rarefaction;
    const fq_rarefaction *rarefaction;
    uint64_t n_frequency;              /* pairs in `frequency` */
    const uint64_t *frequency;         /* {count, number of k-mers with that count}, ascending count */
} fq_kmer_view;
fq_status fq_kmer_enable(fq_ctx *ctx, uint32_t k, uint64_t split_size, uint32_t num_subsample);
fq_status fq_kmer_end_pass(fq_ctx *ctx);
/* End of one input's pass (FaQCs.cpp:518-537, 737-756) for a k-mer table sharded over n contexts.
 * comm == NULL: all n contexts of the run live in this process (same or different devices).
 * comm != NULL: n == 1, this process's context of an n-rank job (fq_comm_init_rank).
 * Afterwards fq_kmer_results returns the merged curve and histogram on every context. */
fq_status fq_kmer_end_pass_all(fq_ctx *const *ctx, int n, fq_comm *const *comm);
fq_status fq_kmer_results(fq_ctx *ctx, fq_kmer_view *view);

/*
 * Sequence duplication statistics (not part of FaQCs; the figure FastQC and fastp report).  A unit is a pair (records i of
 * r1 and r2) of a paired batch, a read of a single-end batch (r2 == NULL).  Every framed record counts, including reads that
 * trimming or filtering discard: the count depends on no option.  Two units are copies when the bytes of their sequence
 * lines -- up to the first '\r' or '\n', case-sensitive, before any masking, trimming or G -> N replacement -- are equal.
 * Each unit is counted as a 64-bit fingerprint of those bytes (defined in fq_dup.cuh): n distinct units give about
 * n^2 / 2^65 expected pairs of equal fingerprints (0.03 at 10^9 units).
 *   fq_dup_enable        before the first batch of a pass; afterwards every batch path counts (fq_process_host,
 *                        fq_submit_host / fq_run / fq_wait, fq_process_device, byte and pieces mode), in any order, on any
 *                        context, from any first_record_index.  Nothing is allocated and no kernel runs without it.
 *   fq_dup_end_pass_all  after the last batch of an input: merges the tables of n contexts (n == 1 and comm == NULL for one
 *                        context; otherwise as for fq_kmer_end_pass_all), publishes the pass's result on every context and
 *                        clears the tables for the next pass.
 *   fq_dup_results       the last finished pass; `levels` belongs to the context and stays valid until its next fq_dup_* call.
 * Duplicate units = units - distinct.  FQ_ERR_STATE for an end of pass or results on a context that never enabled the table;
 * FQ_ERR_ARG when the contexts of one end of pass differ in whether the table is enabled or in paired versus single-end
 * units, and for a batch whose kind differs from the earlier batches of the pass on the same context.
 */
typedef struct fq_dup_view {
    uint64_t units, distinct;
    uint64_t n_levels;                 /* pairs in `levels` */
    const uint64_t *levels;            /* {multiplicity, distinct keys with that multiplicity}, ascending multiplicity */
} fq_dup_view;
fq_status fq_dup_enable(fq_ctx *ctx);
fq_status fq_dup_end_pass_all(fq_ctx *const *ctx, int n, fq_comm *const *comm);
fq_status fq_dup_results(fq_ctx *ctx, fq_dup_view *view);

/*
 * Paired-end insert size and overlap error profile (not part of FaQCs).  For every pair of a paired batch (records i of r1
 * and r2, including pairs that trimming or filtering discard: the result depends on no option) the library looks for the
 * overlap of R1 with the reverse complement of R2, both as framed (up to the first '\r' or '\n').  A, C, G, T in either case
 * are known bases; every other byte is unknown, and a position matches only when both bases are known and equal.  A
 * candidate insert size s puts R1 on fragment positions [0, L1) and reverse-complemented R2 on [s - L2, s); candidates have
 * an overlap o(s) of at least min_overlap positions, and s is accepted when its mismatches m(s) <= min(diff_limit,
 * floor(o(s) * diff_percent / 100)).  The pair's insert size is the accepted s with the fewest mismatches, then the longest
 * overlap, then the smallest s (this selection rule is the library's own; the defaults 30 / 5 / 20 are fastp's).  Per
 * overlapped pair: insert_hist[s] += 1; r1_adapter += s < L1, r2_adapter += s < L2 (the mate reads into adapter);
 * overlap_bases += o(s), mismatch_bases += m(s); overlap position x is R1 cycle x and R2 cycle s - 1 - x (0-based), each
 * counted in r*_overlap and, where the bases disagree, in r*_mismatch.  too_short counts pairs with a mate shorter than
 * min_overlap.  Arrays end at their last non-zero entry (n_cycles: the longest of the four).
 *   fq_overlap_enable        before the first batch of a pass (FQ_ERR_STATE in the middle of one); FQ_ERR_ARG for
 *                            min_overlap == 0 or diff_percent > 100.  Afterwards every batch path counts paired batches;
 *                            single-end batches are neither counted nor refused.  Nothing is allocated and no kernel runs
 *                            without it.
 *   fq_overlap_end_pass_all  after the last batch of an input: sums the accumulators of n contexts (n == 1 and comm == NULL
 *                            for one context; one context per rank with comm), publishes the pass's result on every context
 *                            and clears the accumulators.  FQ_ERR_ARG when the contexts differ in enablement or parameters.
 *   fq_overlap_results       the last finished pass; the pointers belong to the context and stay valid until its next
 *                            fq_overlap_* call.  FQ_ERR_STATE (also for an end of pass) on a context that never enabled it.
 */
typedef struct fq_overlap_view {
    uint64_t pairs, too_short, overlapped, r1_adapter, r2_adapter, overlap_bases, mismatch_bases;
    uint32_t n_insert;   const uint64_t *insert_hist;           /* index = insert size */
    uint32_t n_cycles;   const uint64_t *r1_overlap, *r1_mismatch, *r2_overlap, *r2_mismatch;   /* index = 0-based cycle */
} fq_overlap_view;
fq_status fq_overlap_enable(fq_ctx *ctx, uint32_t min_overlap, uint32_t diff_limit, uint32_t diff_percent);
fq_status fq_overlap_end_pass_all(fq_ctx *const *ctx, int n, fq_comm *const *comm);
fq_status fq_overlap_results(fq_ctx *ctx, fq_overlap_view *view);

/*
 * Overrepresented sequences (not part of FaQCs; the list FastQC and fastp print, without FastQC's truncation of reads over
 * 75 bases to 50 and without its contaminant list).  A unit is one read: the mates of a pair count separately (mate 1, 2;
 * a single-end batch has mate 1 only), and every framed record counts, including reads that trimming or filtering discard,
 * so no option changes the result.  A read's prefix is the first min(len, prefix_len) bytes of its sequence line as framed
 * (up to the first '\r' or '\n', case-sensitive, before any masking, trimming or G -> N replacement); reads with equal
 * prefixes are one sequence, and reads of length 0 count in reads[] but are never listed.  Each prefix is counted exactly
 * as a 64-bit key (fq_overrep.cuh; n distinct prefixes of one mate give about n^2 / 2^64 expected pairs of equal keys).  A
 * sequence of mate m with count c is listed when c * 10^6 >= min_ppm * reads[m - 1] and c >= 2, i.e. c >= min_count[m - 1].
 * The bytes of every listed sequence are kept by a capture rule that needs no second pass (DESIGN.md section 7).
 *   fq_overrep_enable        before the first batch of a pass (FQ_ERR_STATE in the middle of one): prefix_len 1..256
 *                            (default 50), min_ppm 10..1000000 (default 1000 = 0.1 %); FQ_ERR_ARG otherwise.  Afterwards every
 *                            batch path counts.  Nothing is allocated and no kernel runs without it.  Memory: a count table of
 *                            16-byte slots at load <= 1/2 (about 8.6 GB for 100 M pairs of mostly distinct reads) and a capture
 *                            store of (16 + prefix_len) bytes per entry that grows by at most 2 x floor(10^6 / min_ppm)
 *                            entries per batch.
 *   fq_overrep_end_pass_all  after the last batch of an input: merges the count tables of n contexts (n == 1 and comm == NULL
 *                            for one context; otherwise as for fq_kmer_end_pass_all), gathers the captured bytes, publishes the
 *                            pass's list on every context and clears the table and store.  FQ_ERR_ARG when the contexts differ
 *                            in enablement or parameters; FQ_ERR_STATE if a listed sequence has no captured bytes (a bug).
 *   fq_overrep_results       the last finished pass; the pointers belong to the context and stay valid until its next
 *                            fq_overrep_* call.  FQ_ERR_STATE (also for an end of pass) on a context that never enabled it.
 * Order of seqs: count descending, then mate ascending, then bytes ascending (memcmp on the common length, shorter first).
 */
typedef struct fq_overrep_seq {
    uint64_t count;
    uint32_t mate;                     /* 1 or 2 */
    uint32_t len;                      /* bytes of the sequence (its prefix) */
    uint64_t offset;                   /* of its bytes in fq_overrep_view::bytes */
} fq_overrep_seq;
typedef struct fq_overrep_view {
    uint32_t prefix_len, min_ppm;
    uint64_t reads[2];                 /* reads of mate 1 and mate 2 in the pass */
    uint64_t min_count[2];             /* max(2, ceil(min_ppm * reads[m] / 10^6)) */
    uint64_t n_seqs;
    const fq_overrep_seq *seqs;
    const uint8_t *bytes;
} fq_overrep_view;
fq_status fq_overrep_enable(fq_ctx *ctx, uint32_t prefix_len, uint32_t min_ppm);
fq_status fq_overrep_end_pass_all(fq_ctx *const *ctx, int n, fq_comm *const *comm);
fq_status fq_overrep_results(fq_ctx *ctx, fq_overrep_view *view);

/*
 * Per flowcell tile sequence quality (not part of FaQCs; the per-tile plot FastQC draws, used to find bubbles, a bad swath or
 * a smeared tile).  Every framed record counts, whatever trimming, filtering or --qc_only do later; the mates of a pair count
 * separately (mate 1, 2; a single-end pass has mate 1 only).
 * A read's (lane, tile): its name is the header-line bytes after '@' up to the first ' ', '\t', '\r' or '\n', split at ':'
 * into n fields f[0..n-1].  n >= 7 (Casava 1.8 / bcl-convert, with or without a UMI field): lane = f[3], tile = f[4]; n = 5
 * or 6 (@inst:lane:tile:x:y#idx/1): lane = f[1], tile = f[2]; otherwise, or when lane or tile is not 1 to 9 ASCII digits, the
 * read is untiled.  Lane and tile compare as values (01101 and 1101 are one tile).  No parity with FastQC is claimed: it
 * splits the whole line rather than the name and ignores the lane.
 * A base's score is max(0, byte - input_quality_offset) on the quality line as framed, before terminal-N masking, with no
 * upper clamp.  A score above 41 fails the batch with FQ_ERR_QUALITY, with or without qc_only, unless the base lies in a
 * leading or trailing run of 'N' (which the masking covers); such a base counts here with its score as read.
 * Per (tile, mate): reads, bases and score sum of whole reads, and at each cycle 1..cycles the bases (the reads at least
 * that long) and their score sum; cycles = min(longest read of the pass, 1024), and bases past cycle 1024 count in
 * the whole-read totals only.  Per mate: reads and untiled reads of the pass.
 * At most 16384 distinct (lane, tile) keys per pass: when the union of the keys of all contexts is larger, overflow = 1 and
 * the pass reports reads[] and untiled[] but no table (n_tiles = 0), however the batches were dealt to the contexts.
 *   fq_tile_qual_enable        before the first batch of a pass (FQ_ERR_STATE in the middle of one).  Afterwards every batch
 *                              path counts.  Nothing is allocated and no kernel runs without it.  Memory: a 512 KiB key table,
 *                              2 bytes per read and mate of the largest batch, and 8 x mates x (3 + 2 x cycle capacity)
 *                              bytes per tile (tiles seen rounded up to a power of two, at least 64 / mates; cycle capacity:
 *                              the longest read rounded up to 32, at most 1024): 537 MB at the extreme of 16 384 tiles,
 *                              2 mates and 1024 cycles, a few MB for a real flowcell.  The end of a pass holds the summed
 *                              counts on the host and hands every context its own copy of the result.
 *   fq_tile_qual_end_pass_all  after the last batch of an input: unites the keys of n contexts (n == 1 and comm == NULL for
 *                              one context; otherwise as for fq_kmer_end_pass_all), sums their counts, publishes the pass on
 *                              every context and clears the tables.  FQ_ERR_ARG when the profile is enabled on some contexts
 *                              only, or when some counted paired batches and others single-end ones (a batch of the other
 *                              kind in a pass is refused with FQ_ERR_ARG too).  FQ_ERR_STATE when a batch of the pass
 *                              failed part-way (its error was returned by the batch call): the pass is dropped, the
 *                              contexts are cleared for the next one, and the results stay those of the last finished pass.
 *   fq_tile_qual_results       the last finished pass; the pointers belong to the context and stay valid until its next
 *                              fq_tile_qual_* call.  FQ_ERR_STATE (also for an end of pass) on a context that never enabled it.
 */
typedef struct fq_tile_qual_view {
    uint32_t n_mates;                  /* 2 paired, 1 single-end, 0 no batch in the pass */
    uint32_t overflow;                 /* 1: more than 16384 keys, no table */
    uint32_t n_tiles, cycles;
    uint64_t reads[2], untiled[2];     /* per mate */
    const uint32_t *lane, *tile;       /* [n_tiles], ascending by (lane, tile) */
    const uint64_t *tile_reads, *tile_bases, *tile_qsum;        /* [n_tiles][n_mates] */
    const uint64_t *cycle_bases, *cycle_qsum;                   /* [n_tiles][n_mates][cycles] */
} fq_tile_qual_view;
fq_status fq_tile_qual_enable(fq_ctx *ctx);
fq_status fq_tile_qual_end_pass_all(fq_ctx *const *ctx, int n, fq_comm *const *comm);
fq_status fq_tile_qual_results(fq_ctx *ctx, fq_tile_qual_view *view);

/* Zero the accumulators (new run on the same context). */
fq_status fq_reset_stats(fq_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif /* FAQCS_B200_H */
