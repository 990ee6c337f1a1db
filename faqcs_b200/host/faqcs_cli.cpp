// faqcs_cli.cpp -- command-line driver with the FaQCs v2.10 flag set, output file names and
// QC.stats.txt layout, running the trim / filter / statistics path on the GPU through the C ABI
// (include/faqcs_b200.h).  Host side only: option parsing (options.cpp:72-774), gz/plain input
// (zlib), batching at record boundaries, ordered writers, write_stats (FaQCs.cpp:759-1034) and
// the --debug data files of plot() (plot.cpp:540-733), the k-mer rarefaction files included.  The R/PDF
// report is out of scope (DESIGN.md section 7).
//
//   faqcs_b200 -1 r1.fq -2 r2.fq -d outdir [FaQCs flags]        extra: --device N | --devices 0,1,.., --batch_mb N
#include <fcntl.h>
#include <getopt.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <sys/uio.h>
#include <unistd.h>
#include <zlib.h>

#include "fork_join.hpp"
#include "pgzip.hpp"

#include <algorithm>
#include <cerrno>
#include <chrono>
#include <climits>
#include <condition_variable>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <deque>
#include <fstream>
#include <functional>
#include <iomanip>
#include <iostream>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#include "../../include/faqcs_b200.h"

using namespace std;

#define FAQCS_VERSION "2.10"
static const char *kPhiX = "__PhiX174_NC_001422__";
static const char *kPhiXComplement = "__PhiX174_NC_001422_complement__";
static const char *kPhiXSeq =
#include "phix174.inc"
    ;
static const char *kBuiltinAdapters[][2] = {              // options.cpp:576-618 (sequence data)
    {"cre-loxp-forward", "TCGTATAACTTCGTATAATGTATGCTATACGAAGTTATTACG"},
    {"cre-loxp-reverse", "AGCATATTGAAGCATATTACATACGATATGCTTCAATAATGC"},
    {"TruSeq-adapter-1", "GGGGTAGTGTGGATCCTCCTCTAGGCAGTTGGGTTATTCTAGAAGCAGATGTGTTGGCTGTTTCTGAAACTCTGGAAAA"},
    {"TruSeq-adapter-3", "CAACAGCCGGTCAAAACATCTGGAGGGTAAGCCATAAACACCTCAACAGAAAA"},
    {"PCR-primer-1", "CGATAACTTCGTATAATGTATGCTATACGAAGTTATTACG"},
    {"PCR-primer-2", "GCATAACTTCGTATAGCATACATTATACGAAGTTATACGA"},
    {"Nextera-primer-adapter-1", "GATCGGAAGAGCACACGTCTGAACTCCAGTCAC"},
    {"Nextera-primer-adapter-2", "GATCGGAAGAGCGTCGTGTAGGGAAAGAGTGT"},
    {"Nextera-junction-adapter-1", "CTGTCTCTTATACACATCTAGATGTGTATAAGAGACAG"}};

struct Cli {
    bool print_usage = false, protect_5 = false, replace_N = false, kmer_rarefaction = false, discard_output = false;
    bool qc_only = false, trim_only = false, filter_adapter = false, filter_phiX = false, debug = false;
    int mode = FQ_MODE_BWA_PLUS;
    string prefix = "QC", plots_file, stats_file, input_read1_file, input_read2_file, input_unpaired_file;
    string trimmed_read1_file, trimmed_read2_file, trimmed_unpaired_file, trimmed_discard_file, output_dir, artifact_file;
    float average_quality = 0.0f, low_complexity_cutoff_ratio = 0.85f, filterAdapterMismatchRate = 0.2f;
    char input_quality_offset = SCHAR_MIN, output_quality_offset = 33, quality = 5;
    unsigned num_thread = 0, min_read_length = 50, max_num_poly_N = 2, kmer = 31, num_subsample = 10, trim_5 = 0, trim_3 = 0;
    unsigned split_size = 1000000, replace_to_N_q = 0;
    vector<pair<string, string>> adapter;
    int device = 0;
    size_t batch_mb = 64;
    bool gz_out = false;            // trimmed reads as blocked gzip (BGZF), deflated by several threads
    bool dup_stats = false;         // sequence duplication of each input pass -> prefix.duplication.txt
    bool insert_size = false;       // insert size and overlap error profile of the paired pass -> prefix.insert_size.txt
    long long insert_min_overlap = 30, insert_diff_limit = 5, insert_diff_pct = 20;    // checked after parsing
    bool insert_bad_number = false;
    bool overrep = false;           // overrepresented sequences of each input pass -> prefix.overrepresented.txt
    long long overrep_len = 50, overrep_ppm = 1000;    // checked after parsing
    bool overrep_bad_number = false;
    vector<pair<string, string>> artifacts;            // --artifactFile entries (also in `adapter`)
    bool tile_quality = false;      // per flowcell tile quality of each input pass -> prefix.tile_quality.txt
    bool keep_unpaired = false;     // the -u pass appends to prefix.unpaired.trimmed.fastq instead of truncating it (the reference's Q11 quirk, fixed)
    vector<int> devices;            // --devices 0,1,...: consecutive batches go to consecutive GPUs, one NCCL all-reduce at the end
    bool has_paired() const { return !input_read1_file.empty(); }       // has_paired() tests read1 twice, FaQCs.h:135-138
    bool has_unpaired() const { return !input_unpaired_file.empty(); }
};

static unsigned strtou(const string &b)      // options.cpp:798-818
{
    size_t ret = 0;
    long long p = 1;
    for (auto i = b.rbegin(); i != b.rend(); ++i) {
        if (!isdigit((unsigned char)*i)) throw "options.cpp:strtou: Invalid character";
        ret += (size_t)(*i - '0') * p;
        p *= 10;
    }
    if (ret > UINT_MAX) throw "options.cpp:strtou: Overflow!";
    return (unsigned)ret;
}

static string reverse_complement(string s)   // options.cpp:894-996
{
    for (char &c : s) {
        switch (c) {
            case 'A': c = 'T'; break; case 'a': c = 't'; break; case 'T': c = 'A'; break; case 't': c = 'a'; break;
            case 'G': c = 'C'; break; case 'g': c = 'c'; break; case 'C': c = 'G'; break; case 'c': c = 'g'; break;
            case 'M': c = 'K'; break; case 'm': c = 'k'; break; case 'R': c = 'Y'; break; case 'r': c = 'y'; break;
            case 'V': c = 'B'; break; case 'v': c = 'b'; break; case 'Y': c = 'R'; break; case 'y': c = 'r'; break;
            case 'H': c = 'D'; break; case 'h': c = 'd'; break; case 'K': c = 'M'; break; case 'k': c = 'm'; break;
            case 'D': c = 'H'; break; case 'd': c = 'h'; break; case 'B': c = 'V'; break; case 'b': c = 'v'; break;
            default: break;      // S, W, N map to themselves
        }
    }
    reverse(s.begin(), s.end());
    return s;
}

static void parse_artifact_file(const string &fn, vector<pair<string, string>> &out)   // options.cpp:820-891
{
    gzFile fin = gzopen(fn.c_str(), "r");
    if (!fin) {
        cerr << "Unable to open " << fn << " for loading artifact sequences" << endl;
        throw "I/O error";
    }
    const int buffer_len = 4096;
    char buffer[buffer_len];
    string defline;
    string data;
    while (gzgets(fin, buffer, buffer_len)) {
        char *ptr = strchr(buffer, '>');
        if (ptr) {
            if (!data.empty()) out.push_back(make_pair(defline, data));
            data.clear();
            ++ptr;
            for (char *p = ptr; *p; ++p)
                if (*p == '\n' || *p == '\r') *p = '\0';
            if (strlen(ptr) == (size_t)(buffer_len - 1)) defline = buffer + string("...");
            else defline = ptr;
        } else {
            for (char *p = buffer; *p; ++p)
                if (!isspace((unsigned char)*p)) data.push_back(*p);
        }
    }
    if (!data.empty()) out.push_back(make_pair(defline, data));
    gzclose(fin);
}

static void usage()
{
    cerr << "FaQCs version " << FAQCS_VERSION << " (faqcs_b200: GPU trim/filter/statistics path)" << endl;
    cerr << "Input File(s):\n\t-u\t\t\t<File> Unpaired reads\n\t-1\t\t\t<File> First paired read file\n\t-2\t\t\t<File> Second paired read file\n";
    cerr << "Trim:\n\t--mode\t\t\t\"HARD\" or \"BWA\" or \"BWA_plus\" (default BWA_plus)\n\t-q\t\t\t<INT> Targets # as quality level (default 5) for trimming\n";
    cerr << "\t--5end\t\t\t<INT> Cut # bp from 5 end before quality trimming/filtering\n\t--3end\t\t\t<INT> Cut # bp from 3 end before quality trimming/filtering\n";
    cerr << "\t--adapter\t\t<bool> Trim reads with illumina adapter/primers (default: no)\n\t--rate\t\t\t<FLOAT> Mismatch ratio of adapters' length (default: 0.2, allow 20% mismatches)\n";
    cerr << "\t--polyA\t\t\t<bool>  Trim poly A ( > 15 )\n\t--artifactFile\t\t<File> additional artifact (adapters/primers/contaminations) reference file in fasta format\n";
    cerr << "Filters:\n\t--min_L\t\t\t<INT> Trimmed read should have to be at least this minimum length (default:50)\n\t--avg_q\t\t\t<NUM> Average quality cutoff (default:0, no filtering)\n";
    cerr << "\t-n\t\t\t<INT> Trimmed read has greater than or equal to this number of continuous base \"N\" will be discarded.\n\t--lc\t\t\t<FLOAT> Low complexity filter ratio (default: 0.85)\n\t--phiX\t\t\t<bool> Filter phiX reads (slow)\n";
    cerr << "Q_Format:\n\t--ascii\t\t\tEncoding type: 33 or 64 or autoCheck (default)\n\t--out_ascii\t\tOutput encoding. (default: 33)\n";
    cerr << "Output:\n\t--prefix\t\t<TEXT> Output file prefix. (default: QC)\n\t--stats\t\t\t<File> Statistical numbers output file (default: prefix.stats.txt)\n\t-d\t\t\t<PATH> Output directory.\n";
    cerr << "Options:\n\t-t\t\t\t<INT > # of CPUs the reference would run with (only reproduces its -t dependent adapter threshold)\n";
    cerr << "\t--split_size\t\t<INT> reads per point of the k-mer rarefaction curve (default: 1000000)\n\t--kmer_rarefaction\t<bool> count canonical 31-mers; prefix.Kmercount.txt / prefix.kmerH.txt with --debug\n\t--subset\t\t<INT> points of the curve = 2 x this (default: 10)\n\t--qc_only\t\t<bool> no Filters, no Trimming, report numbers.\n\t--discard\t\t<bool> Output discarded reads\n";
    cerr << "\t--substitute\t\t<bool> (not implemented, as in FaQCs)\n\t--trim_only\t\t<bool> No quality report. Output trimmed reads only.\n\t--replace_to_N_q\t<INT> Replace base G to N when below this quality score (default:0, off)\n";
    cerr << "\t--5trim_off\t\t<bool> Turn off trimming from 5'end.\n\t--debug\t\t\t<bool> Keep intermediate files\n\t--version\t\t<bool> Print the version and exit\n";
    cerr << "GPU:\n\t--device\t\t<INT> CUDA device (default 0)\n\t--devices\t\t<INT,INT,..> several CUDA devices: batches are dealt out in order, statistics merged with one NCCL all-reduce\n"
            "\t--batch_mb\t\t<INT> MiB of FASTQ per mate per batch (default 64)\n"
            "Output (extensions):\n\t--gz_out\t\t<bool> write the trimmed reads as blocked gzip (prefix.*.trimmed.fastq.gz), deflated in parallel\n"
            "\t--keep_unpaired\t\t<bool> with -1/-2 and -u: append the -u pass to prefix.unpaired.trimmed.fastq instead of overwriting it\n"
            "\t--dup_stats\t\t<bool> count identical reads (-u) and read pairs (-1/-2) of each input: prefix.duplication.txt\n"
            "\t--insert_size\t\t<bool> with -1/-2: insert size of each pair from the overlap of R1 with reverse-complemented R2,\n"
            "\t\t\t\tadapter read-through and mismatches per cycle in the overlap: prefix.insert_size.txt\n"
            "\t--insert_min_overlap\t<INT> shortest overlap tested (default 30, at least 1)\n"
            "\t--insert_diff_limit\t<INT> most mismatches in an accepted overlap (default 5)\n"
            "\t--insert_diff_pct\t<INT> most mismatches in an accepted overlap, in percent of its length (default 20, 0-100)\n"
            "\t--overrep\t\t<bool> list the sequences (read prefixes, each mate on its own) above a share of the reads of each\n"
            "\t\t\t\tinput, with the built-in adapter, PhiX or --artifactFile entry they match: prefix.overrepresented.txt\n"
            "\t--overrep_len\t\t<INT> bases of each read's prefix compared (default 50, 1-256)\n"
            "\t--overrep_ppm\t\t<INT> smallest listed share, in reads per million of the mate (default 1000 = 0.1 %, 10-1000000)\n"
            "\t--tile_quality\t\t<bool> mean quality per cycle of each flowcell tile (lane and tile from the read names) against\n"
            "\t\t\t\tall tiles, each mate on its own, for each input: prefix.tile_quality.txt\n";
}

static void parse_options(int argc, char *argv[], Cli &o)
{
    for (int i = 1; i < argc; ++i) {                      // deprecated -p f1 f2 (options.cpp:78-96)
        if (strncmp(argv[i], "-p", 2) == 0 && strncmp(argv[i], "-prefix", 7) != 0 && strcmp(argv[i], "-phiX") != 0 && strcmp(argv[i], "-polyA") != 0) {
            if (i + 2 >= argc) throw "options.cpp:Options: Unable to extract file names after depricated '-p' flag";
            o.input_read1_file = argv[i + 1];
            o.input_read2_file = argv[i + 2];
            cerr << "The paired read flag (-p) has been deprecated. Please specify paired read files with -1 <file> and -2 <file>" << endl;
        }
    }
    o.print_usage = (argc == 1);
    bool trim_polyA = false, version = false;
    int config_opt = 0, long_index = 0;
    const char *options = "d:t:n:1:2:p:q:u:?h";
    struct option long_opts[] = {
        {"mode", true, &config_opt, 1}, {"5end", true, &config_opt, 2}, {"3end", true, &config_opt, 3}, {"adapter", false, &config_opt, 4},
        {"rate", true, &config_opt, 5}, {"polyA", false, &config_opt, 6}, {"artifactFile", true, &config_opt, 7}, {"min_L", true, &config_opt, 8},
        {"avg_q", true, &config_opt, 9}, {"lc", true, &config_opt, 10}, {"phiX", false, &config_opt, 11}, {"ascii", true, &config_opt, 12},
        {"out_ascii", true, &config_opt, 13}, {"prefix", true, &config_opt, 14}, {"stats", true, &config_opt, 15}, {"split_size", true, &config_opt, 16},
        {"qc_only", false, &config_opt, 17}, {"kmer_rarefaction", false, &config_opt, 18}, {"subset", true, &config_opt, 19},
        {"discard", false, &config_opt, 20}, {"substitute", false, &config_opt, 21}, {"trim_only", false, &config_opt, 22},
        {"5trim_off", false, &config_opt, 23}, {"debug", false, &config_opt, 24}, {"version", false, &config_opt, 25}, {"R1", true, &config_opt, 26},
        {"R2", true, &config_opt, 27}, {"replace_to_N_q", true, &config_opt, 31}, {"device", true, &config_opt, 40}, {"batch_mb", true, &config_opt, 41}, {"devices", true, &config_opt, 42}, {"gz_out", false, &config_opt, 43}, {"keep_unpaired", false, &config_opt, 44}, {"dup_stats", false, &config_opt, 45},
        {"insert_size", false, &config_opt, 46}, {"insert_min_overlap", true, &config_opt, 47}, {"insert_diff_limit", true, &config_opt, 48},
        {"insert_diff_pct", true, &config_opt, 49}, {"overrep", false, &config_opt, 50}, {"overrep_len", true, &config_opt, 51},
        {"overrep_ppm", true, &config_opt, 52}, {"tile_quality", false, &config_opt, 53},
        {0, 0, 0, 0}};
    int opt_code;
    opterr = 0;
    while ((opt_code = getopt_long_only(argc, argv, options, long_opts, &long_index)) != EOF) {
        switch (opt_code) {
            case 0:
                switch (config_opt) {
                    case 1: {
                        string m = optarg;
                        for (char &c : m) c = (char)tolower(c);
                        o.mode = m == "hard" ? FQ_MODE_HARD : m == "bwa" ? FQ_MODE_BWA : m == "bwa_plus" ? FQ_MODE_BWA_PLUS : -1;
                        break;
                    }
                    case 2: o.trim_5 = strtou(optarg); break;
                    case 3: o.trim_3 = strtou(optarg); break;
                    case 4: o.filter_adapter = true; break;
                    case 5: o.filterAdapterMismatchRate = (float)atof(optarg); break;
                    case 6: trim_polyA = true; break;
                    case 7: o.artifact_file = optarg; o.filter_adapter = true; break;
                    case 8: o.min_read_length = strtou(optarg); break;
                    case 9: o.average_quality = (float)atof(optarg); break;
                    case 10: o.low_complexity_cutoff_ratio = (float)atof(optarg); break;
                    case 11: o.filter_phiX = true; break;
                    case 12: {
                        const int v = atoi(optarg);
                        if (v <= SCHAR_MIN || v > SCHAR_MAX) throw "options.cpp:Options::Options: ascii out of bounds!";
                        o.input_quality_offset = (char)v;
                        break;
                    }
                    case 13: {
                        const int v = atoi(optarg);
                        if (v <= SCHAR_MIN || v > SCHAR_MAX) throw "options.cpp:Options::Options: out_ascii out of bounds!";
                        o.output_quality_offset = (char)v;
                        break;
                    }
                    case 14: o.prefix = optarg; break;
                    case 15: o.stats_file = optarg; break;
                    case 16: o.split_size = strtou(optarg); break;
                    case 17: o.qc_only = true; break;
                    case 18: o.kmer_rarefaction = true; break;
                    case 19: o.num_subsample = strtou(optarg); break;
                    case 20: o.discard_output = true; break;
                    case 21: o.replace_N = true; break;
                    case 22: o.trim_only = true; break;
                    case 23: o.protect_5 = true; break;
                    case 24: o.debug = true; break;
                    case 25: version = true; break;
                    case 26: o.input_read1_file = optarg; break;
                    case 27: o.input_read2_file = optarg; break;
                    case 31: o.replace_to_N_q = strtou(optarg); break;
                    case 40: o.device = atoi(optarg); break;
                    case 41: o.batch_mb = (size_t)max(1, atoi(optarg)); break;
                    case 42: {
                        o.devices.clear();
                        for (const char *p = optarg; *p;) {
                            char *end = nullptr;
                            const long d = strtol(p, &end, 10);
                            if (end == p || d < 0) { cerr << "--devices expects a comma separated list of CUDA device indices" << endl; o.print_usage = true; break; }
                            o.devices.push_back((int)d);
                            p = *end == ',' ? end + 1 : end;
                        }
                        break;
                    }
                    case 43: o.gz_out = true; break;
                    case 44: o.keep_unpaired = true; break;
                    case 45: o.dup_stats = true; break;
                    case 46: o.insert_size = true; break;
                    case 47: case 48: case 49: {
                        char *end = nullptr;
                        errno = 0;
                        const long long v = strtoll(optarg, &end, 10);
                        if (end == optarg || *end || errno) o.insert_bad_number = true;
                        (config_opt == 47 ? o.insert_min_overlap : config_opt == 48 ? o.insert_diff_limit : o.insert_diff_pct) = v;
                        break;
                    }
                    case 50: o.overrep = true; break;
                    case 53: o.tile_quality = true; break;
                    case 51: case 52: {
                        char *end = nullptr;
                        errno = 0;
                        const long long v = strtoll(optarg, &end, 10);
                        if (end == optarg || *end || errno) o.overrep_bad_number = true;
                        (config_opt == 51 ? o.overrep_len : o.overrep_ppm) = v;
                        break;
                    }
                    default: cerr << "Unknown flag!" << endl; break;
                }
                break;
            case '1': o.input_read1_file = optarg; break;
            case '2': o.input_read2_file = optarg; break;
            case 'u': o.input_unpaired_file = optarg; break;
            case 'd': o.output_dir = optarg; break;
            case 'n': o.max_num_poly_N = strtou(optarg); break;
            case 'q': {
                const int v = atoi(optarg);
                if (v <= SCHAR_MIN || v > SCHAR_MAX) throw "options.cpp:Options::Options: q out of bounds!";
                o.quality = (char)v;
                break;
            }
            case 't': o.num_thread = strtou(optarg); break;
            case 'h': case '?': o.print_usage = true; break;
            case 'p': break;
            default: cerr << '"' << (char)opt_code << "\" is not a valid option!" << endl; break;
        }
    }
    if (o.print_usage) { usage(); return; }
    if (version) { cerr << "Version: " << FAQCS_VERSION << endl; o.print_usage = true; return; }
    if (o.input_read1_file.empty() != o.input_read2_file.empty()) {
        if (o.input_read1_file.empty()) cerr << "Please specify a read one file (-1 <file>)" << endl;
        if (o.input_read2_file.empty()) cerr << "Please specify a read one file (-2 <file>)" << endl;
        o.print_usage = true;
        return;
    }
    if (o.input_unpaired_file.empty() && o.input_read1_file.empty() && o.input_read2_file.empty()) {
        cerr << "Please specify either a pair of fastq files (-1 <file> -2 <file>)  or a single fastq file of unpaired reads (-u <file>)" << endl;
        o.print_usage = true;
        return;
    }
    if (o.low_complexity_cutoff_ratio > 1.0 || o.low_complexity_cutoff_ratio < 0.0) {
        cerr << "Please specify a low complexity cutoff ration (-lc) in the range 0 <= ratio <= 1.0" << endl;
        o.print_usage = true;
        return;
    }
    if (o.filterAdapterMismatchRate > 1.0 || o.filterAdapterMismatchRate < 0.0) {
        cerr << "Please specify an adapter mismatch rate (-adapter) in the range 0 <= rate <= 1.0" << endl;
        o.print_usage = true;
        return;
    }
    if (o.split_size == 0) {
        cerr << "Please specify a split_size (--split_size) value greater than 0" << endl;
        o.print_usage = true;
        return;
    }
    if (o.num_subsample == 0) {
        cerr << "Please specify a subset (--subset) value greater than 0" << endl;
        o.print_usage = true;
        return;
    }
    if (o.insert_size && !o.has_paired()) {
        cerr << "--insert_size needs paired reads (-1 <file> -2 <file>): the insert size is measured on the overlap of the two mates" << endl;
        o.print_usage = true;
        return;
    }
    if (o.insert_bad_number || o.insert_min_overlap < 1 || o.insert_min_overlap > UINT_MAX || o.insert_diff_limit < 0 || o.insert_diff_limit > UINT_MAX ||
        o.insert_diff_pct < 0 || o.insert_diff_pct > 100) {
        cerr << "Please specify --insert_min_overlap as an integer >= 1, --insert_diff_limit as an integer >= 0 and --insert_diff_pct as an integer "
                "in the range 0 <= percent <= 100" << endl;
        o.print_usage = true;
        return;
    }
    if (o.overrep_bad_number || o.overrep_len < 1 || o.overrep_len > 256 || o.overrep_ppm < 10 || o.overrep_ppm > 1000000) {
        cerr << "Please specify --overrep_len as an integer in the range 1 <= length <= 256 and --overrep_ppm as an integer in the range "
                "10 <= ppm <= 1000000" << endl;
        o.print_usage = true;
        return;
    }
    o.num_subsample *= 2;      // options.cpp:519-523: doubled on every command line that gets this far, paired input or not
    if (o.replace_N) cerr << "**Warning** \"-substitue\" is not currently implemented" << endl;
    if (o.filter_adapter)                                 // built-in adapters, options.cpp:576-618
        for (auto &b : kBuiltinAdapters) o.adapter.push_back(make_pair(string(b[0]), string(b[1])));
    if (trim_polyA) o.adapter.push_back(make_pair(string("polyA"), string(20, 'A')));
    if (o.filter_phiX) {
        o.adapter.push_back(make_pair(string(kPhiX), string(kPhiXSeq)));
        o.adapter.push_back(make_pair(string(kPhiXComplement), reverse_complement(kPhiXSeq)));
    }
    if (!o.artifact_file.empty()) {
        parse_artifact_file(o.artifact_file, o.artifacts);
        o.adapter.insert(o.adapter.end(), o.artifacts.begin(), o.artifacts.end());
    }
    const string base = o.output_dir + "/" + o.prefix;    // options.cpp:696-741
    if (!o.input_read1_file.empty() && !o.input_read2_file.empty()) {
        o.trimmed_read1_file = base + ".1.trimmed.fastq";
        o.trimmed_read2_file = base + ".2.trimmed.fastq";
    }
    o.trimmed_unpaired_file = base + ".unpaired.trimmed.fastq";
    o.trimmed_discard_file = o.discard_output ? base + ".discard.trimmed.fastq" : "";
    if (o.gz_out)
        for (string *f : {&o.trimmed_read1_file, &o.trimmed_read2_file, &o.trimmed_unpaired_file, &o.trimmed_discard_file})
            if (!f->empty()) *f += ".gz";
    if (o.plots_file.empty()) o.plots_file = base + "_qc_report.pdf";
    if (o.stats_file.empty()) o.stats_file = base + ".stats.txt";
    if (o.mode < 0) {
        o.mode = FQ_MODE_BWA_PLUS;
        if (!o.qc_only) cerr << "Not recognized mode. Bwa extension trimming algorithm is used." << endl;
    } else if (!o.qc_only) {
        cerr << (o.mode == FQ_MODE_HARD ? "Hard trimming is used." : o.mode == FQ_MODE_BWA ? "Bwa trimming is used." : "Bwa extension trimming is used.") << endl;
    }
}

// ---- host pipeline (SURVEY 8(f) N1/N2): reader threads -> GPU -> writer threads --------------------
// A worker thread that runs posted jobs in order; wait_idle() rethrows the first error a job raised.
class Worker {
    mutex mu;
    condition_variable cv, cv_idle;
    deque<function<void()>> jobs;
    size_t busy = 0;
    bool stop = false;
    const char *err = nullptr;
    thread th;          // last member: the thread starts only after the state it uses is constructed
    void loop()
    {
        for (;;) {
            function<void()> job;
            {
                unique_lock<mutex> lk(mu);
                cv.wait(lk, [&] { return stop || !jobs.empty(); });
                if (jobs.empty()) return;
                job = move(jobs.front());
                jobs.pop_front();
            }
            try { job(); }
            catch (const char *e) { lock_guard<mutex> lk(mu); if (!err) err = e; }
            catch (const std::exception &) { lock_guard<mutex> lk(mu); if (!err) err = "I/O worker failed (std::exception)"; }
            catch (...) { lock_guard<mutex> lk(mu); if (!err) err = "I/O worker failed"; }
            {
                lock_guard<mutex> lk(mu);
                --busy;
            }
            cv_idle.notify_all();
        }
    }
public:
    Worker() : th([this] { loop(); }) {}
    ~Worker()
    {
        { lock_guard<mutex> lk(mu); stop = true; }
        cv.notify_all();
        th.join();
    }
    void post(function<void()> f)
    {
        { lock_guard<mutex> lk(mu); jobs.push_back(move(f)); ++busy; }
        cv.notify_all();
    }
    void wait_idle()
    {
        unique_lock<mutex> lk(mu);
        cv_idle.wait(lk, [&] { return busy == 0; });
        if (err) { const char *e = err; err = nullptr; throw e; }
    }
};

constexpr int kIoThreads = 4;      // threads per plain input file (pread slices) and per output file (mapped copies)
// transfers below this size use plain read(2) / write(2); FAQCS_B200_IO_SLICE_MIN overrides it (the tests use a tiny value)
static size_t io_slice_min()
{
    static const size_t v = [] { const char *e = getenv("FAQCS_B200_IO_SLICE_MIN"); return e ? (size_t)strtoull(e, nullptr, 10) : (size_t)(8u << 20); }();
    return v;
}

static size_t count_newlines(const uint8_t *buf, size_t n)
{
    size_t c = 0;
    for (size_t i = 0; i < n; ++i) c += buf[i] == '\n';      // vectorised by the compiler
    return c;
}

// ---- input: gz or plain, whole records per batch -------------------------------------------------
// Plain files are read with pread straight into the pinned batch buffer.  Gzip input (magic 1f 8b) is inflated by several
// threads: blocked gzip (BGZF: bgzip, bcl-convert, samtools) member by member, as its members carry their compressed size in
// the header, and ordinary gzip by entering the deflate stream at block boundaries (pgzip.hpp).
static int g_input_files = 2;      // files read at the same time (two mates, or one file of unpaired reads)
static int inflate_threads()      // per input file: the cores divided among the files, 2 .. 32
{
    return (int)min(32u, max(2u, thread::hardware_concurrency() / (unsigned)max(1, g_input_files)));
}

// A BGZF member at p[0..avail): its total size, or 0 if the bytes are not a complete BGZF header (RFC 1952 member with
// FEXTRA holding the subfield 'B','C',2,BSIZE; SAM specification 4.1).
static size_t bgzf_member_size(const uint8_t *p, size_t avail)
{
    if (avail < 18 || p[0] != 0x1f || p[1] != 0x8b || p[2] != 8 || !(p[3] & 4)) return 0;
    const size_t xlen = p[10] | (size_t)p[11] << 8;
    if (avail < 12 + xlen) return 0;
    for (size_t q = 12; q + 4 <= 12 + xlen;) {
        const size_t slen = p[q + 2] | (size_t)p[q + 3] << 8;
        if (p[q] == 'B' && p[q + 1] == 'C' && slen == 2 && q + 6 <= 12 + xlen) return (size_t)(p[q + 4] | (size_t)p[q + 5] << 8) + 1;
        q += 4 + slen;
    }
    return 0;
}

// pread until all n bytes are in; an I/O error or the end of the file before that is the reader's error
static void pread_full(int fd, uint8_t *dst, size_t n, off_t at)
{
    for (size_t done = 0; done < n;) {
        const ssize_t got = pread(fd, dst + done, n - done, at + (off_t)done);
        if (got < 0 && errno == EINTR) continue;
        if (got <= 0) throw "fastq.cpp:next_read: Unable to read header";
        done += (size_t)got;
    }
}

struct Source {
    // Sliced: a regular plain file, read by kIoThreads threads into disjoint slices of the buffer (a single read(2) stream is
    //   a single-core page-cache copy).
    // Zlib: one zlib stream, as the reference reads every input (fastq.cpp:8-30): small or FAQCS_B200_PGZIP=0 gzip, and any
    //   input that is not a regular file (pipes, process substitution, /dev/stdin), whose bytes cannot be read twice to sniff
    //   the format; zlib passes plain text through.
    // Bgzf, Pgzip: blocked and ordinary gzip, inflated by several threads.
    enum class Mode { Sliced, Zlib, Bgzf, Pgzip };
    Mode mode = Mode::Sliced;
    bool bgzf = false, pgzip = false;     // open()'s choice, as reported by tests/host_io_harness.cpp (a Bgzf file may go on to Zlib)
    int fd = -1;
    bool eof = false;
    off_t pos = 0, size = 0;              // Sliced, Bgzf, Pgzip: the next byte of the file to read, the file size
    vector<uint8_t> cbuf;                 // Bgzf, Pgzip: compressed bytes of one fill / round
    gzFile gz = nullptr;                  // Zlib
    struct {                              // Pgzip
        bool in_member = false;
        size_t bit = 0;                   // first undecoded bit of the member's deflate stream, relative to byte pos
        size_t window_len = 0;            // valid bytes at the end of window (output of this member so far, at most 32 KiB)
        vector<uint8_t> window;           // the last 32 KiB of output
        deque<pgz::Bytes> pend;           // decoded pieces not yet handed out (the front one from pend_off on)
        size_t pend_off = 0;
        size_t span = 0;                  // compressed bytes looked at per round
        size_t min_piece = 256u << 10;    // a thread gets at least this much compressed data
        int solo_rounds = 0;              // rounds left in which no entry points are looked for
        uint32_t crc = 0;
        uint64_t isize = 0;
    } pz;
    bool open(const string &fn)
    {
        fd = ::open(fn.c_str(), O_RDONLY);
        if (fd < 0) return false;
        struct stat st;
        if (fstat(fd, &st) != 0 || !S_ISREG(st.st_mode)) return open_zlib();      // no sniffing: bytes read from a pipe are gone
        size = st.st_size;
        unsigned char head[64];
        const ssize_t got = pread(fd, head, sizeof(head), 0);
        if (got >= 18 && bgzf_member_size(head, (size_t)got) && !getenv("FAQCS_B200_NO_BGZF")) mode = Mode::Bgzf;
        else if (got >= 2 && head[0] == 0x1f && head[1] == 0x8b) {
            // FAQCS_B200_PGZIP=0: one zlib stream.  FAQCS_B200_PGZIP_MIN / _PIECE / _SPAN: smallest file, smallest piece,
            // bytes per round (the tests shrink them)
            const char *e = getenv("FAQCS_B200_PGZIP");
            const char *m = getenv("FAQCS_B200_PGZIP_MIN"), *pc = getenv("FAQCS_B200_PGZIP_PIECE"), *sp = getenv("FAQCS_B200_PGZIP_SPAN");
            if (size < (off_t)(m ? strtoull(m, nullptr, 10) : (4u << 20)) || (e && e[0] == '0')) return open_zlib();
            if (pc) pz.min_piece = (size_t)strtoull(pc, nullptr, 10);
            if (sp) pz.span = (size_t)strtoull(sp, nullptr, 10);
            pz.window.assign(pgz::kWin, 0);
            mode = Mode::Pgzip;
        }
        bgzf = mode == Mode::Bgzf;
        pgzip = mode == Mode::Pgzip;
        return true;
    }
    bool open_zlib()
    {
        mode = Mode::Zlib;
        gz = gzdopen(fd, "r");
        if (!gz) return false;
        gzbuffer(gz, 1 << 20);
        return true;
    }
    void close()
    {
        if (gz) gzclose(gz);
        else if (fd >= 0) ::close(fd);
        gz = nullptr;
        fd = -1;
    }
    // append to buf[have..cap); returns the bytes now in buf and the newlines in the appended part
    size_t fill(uint8_t *buf, size_t have, size_t cap, size_t *new_lines)
    {
        switch (mode) {
            case Mode::Sliced: return fill_sliced(buf, have, cap, new_lines);
            case Mode::Zlib: return fill_zlib(buf, have, cap, new_lines);
            case Mode::Bgzf: return fill_bgzf(buf, have, cap, new_lines);
            case Mode::Pgzip: return fill_pgzip(buf, have, cap, new_lines);
        }
        return have;
    }
    size_t fill_sliced(uint8_t *buf, size_t have, size_t cap, size_t *new_lines)
    {
        const size_t want = (size_t)min<off_t>((off_t)(cap - have), size - pos);
        const int nt = want >= io_slice_min() && want >= (size_t)kIoThreads ? kIoThreads : 1;
        const size_t per = (want + nt - 1) / nt;
        vector<size_t> lines(nt, 0);
        fork_join(nt, [&](int t) {
            const size_t lo = min(want, per * t), hi = min(want, per * (t + 1));
            pread_full(fd, buf + have + lo, hi - lo, pos + (off_t)lo);       // the file shrank, or an I/O error: throws
            lines[t] = count_newlines(buf + have + lo, hi - lo);
        });
        for (size_t l : lines) *new_lines += l;
        pos += (off_t)want;
        if (pos >= size) eof = true;
        return have + want;
    }
    size_t fill_zlib(uint8_t *buf, size_t have, size_t cap, size_t *new_lines)
    {
        size_t n = have;
        while (!eof && n < cap) {
            const int got = gzread(gz, buf + n, (unsigned)min<size_t>(cap - n, 1u << 30));
            if (got < 0) throw "fastq.cpp:next_read: Unable to read header";
            if (got == 0) eof = true;
            n += (size_t)got;
        }
        *new_lines += count_newlines(buf + have, n - have);
        return n;
    }
    void read_cbuf(size_t want)
    {
        cbuf.resize(want);
        pread_full(fd, cbuf.data(), want, pos);
    }
    // BGZF: members up to the buffer's capacity, inflated by inflate_threads() threads into their places.  Anything that is
    // not a BGZF member (plain gzip members appended to the file) hands the rest of the file to zlib.
    size_t fill_bgzf(uint8_t *buf, size_t have, size_t cap, size_t *new_lines)
    {
        struct Member { size_t in, in_len, out, out_len; uint32_t crc; };
        vector<Member> members;
        size_t n = have;
        const size_t want = (size_t)min<off_t>(size - pos, (off_t)(cap - have) + (1 << 16));
        read_cbuf(want);
        size_t p = 0;
        bool to_zlib = false;
        while (p < want) {
            const size_t msize = bgzf_member_size(cbuf.data() + p, want - p);
            if (msize == 0) { to_zlib = want - p >= 18 || pos + (off_t)want >= size; break; }   // not BGZF (or a cut header: next fill)
            if (p + msize > want) break;                                                        // cut member: next fill
            const uint8_t *m = cbuf.data() + p;
            const size_t hdr = 12 + (m[10] | (size_t)m[11] << 8);
            if (msize < hdr + 8) throw "corrupt BGZF member";
            const uint32_t crc = m[msize - 8] | (uint32_t)m[msize - 7] << 8 | (uint32_t)m[msize - 6] << 16 | (uint32_t)m[msize - 5] << 24;
            const size_t isize = m[msize - 4] | (size_t)m[msize - 3] << 8 | (size_t)m[msize - 2] << 16 | (size_t)m[msize - 1] << 24;
            if (n + isize > cap) break;
            members.push_back(Member{p + hdr, msize - hdr - 8, n, isize, crc});
            n += isize;
            p += msize;
        }
        const int nt = (int)max<size_t>(1, min<size_t>((size_t)inflate_threads(), members.size() / 4));
        vector<size_t> lines(nt, 0);
        fork_join(nt, [&](int t) {
            z_stream zs{};
            if (inflateInit2(&zs, -15) != Z_OK) throw "fastq.cpp:next_read: Unable to read header";
            const size_t lo = members.size() * t / nt, hi = members.size() * (t + 1) / nt;
            bool ok = true;
            for (size_t k = lo; ok && k < hi; ++k) {
                const Member &mb = members[k];
                zs.next_in = cbuf.data() + mb.in; zs.avail_in = (uInt)mb.in_len;
                zs.next_out = buf + mb.out; zs.avail_out = (uInt)mb.out_len;
                const int rc = mb.out_len || mb.in_len ? inflate(&zs, Z_FINISH) : Z_STREAM_END;
                ok = rc == Z_STREAM_END && zs.avail_out == 0 && (uint32_t)crc32(crc32(0L, Z_NULL, 0), buf + mb.out, (uInt)mb.out_len) == mb.crc;
                inflateReset(&zs);
            }
            inflateEnd(&zs);
            if (!ok) throw "fastq.cpp:next_read: Unable to read header";       // what a failed gzgets turns into
            if (hi > lo) lines[t] = count_newlines(buf + members[lo].out, members[hi - 1].out + members[hi - 1].out_len - members[lo].out);
        });
        for (size_t l : lines) *new_lines += l;
        pos += (off_t)p;
        if (pos >= size) eof = true;
        if (to_zlib) {                       // the rest of the file through zlib, from this member on
            if (lseek(fd, pos, SEEK_SET) < 0 || !open_zlib()) throw "fastq.cpp:next_read: Unable to read header";
            if (n < cap) return fill_zlib(buf, n, cap, new_lines);
        }
        return n;
    }
    // ---- ordinary gzip, inflated by several threads (pgzip.hpp) ----
    // the header of the member at pos (RFC 1952); false: no further member (end of file, or bytes that are not gzip: ignored as gzread does)
    bool pz_member_header()
    {
        const size_t want = (size_t)min<off_t>(size - pos, 1 << 16);
        if (want < 18) return false;
        read_cbuf(want);
        const uint8_t *h = cbuf.data();
        if (h[0] != 0x1f || h[1] != 0x8b) return false;
        if (h[2] != 8 || (h[3] & 0xe0)) throw "fastq.cpp:next_read: Unable to read header";
        size_t p = 10;
        if (h[3] & 4) { if (p + 2 > want) return false; p += 2 + (h[p] | (size_t)h[p + 1] << 8); }
        if (h[3] & 8) { while (p < want && h[p]) ++p; ++p; }
        if (h[3] & 16) { while (p < want && h[p]) ++p; ++p; }
        if (h[3] & 2) p += 2;
        if (p >= want) throw "fastq.cpp:next_read: Unable to read header";
        pos += (off_t)p;
        pz.bit = 0;
        pz.window_len = 0;
        pz.crc = (uint32_t)crc32(0L, Z_NULL, 0);
        pz.isize = 0;
        pz.in_member = true;
        return true;
    }
    // one round: more decoded bytes into pz.pend (or eof)
    void pz_produce()
    {
        if (!pz.in_member && (pos >= size || !pz_member_header())) { eof = true; return; }
        const int threads = inflate_threads();
        if (!pz.span) pz.span = max<size_t>((size_t)threads * (2u << 20), 8u << 20);
        for (;;) {
            const size_t want = (size_t)min<off_t>(size - pos, (off_t)pz.span);
            read_cbuf(want);
            // a stream without entry points (stored or fixed blocks, blocks larger than a piece) is left to one thread for a few
            // rounds instead of being searched again and again
            const int use = pz.solo_rounds > 0 ? 1 : threads;
            if (pz.solo_rounds > 0) --pz.solo_rounds;
            pgz::Result R = pgz::inflate_parallel(cbuf.data(), want, pz.bit, pz.window, pz.window_len, use, pz.min_piece);
            if (use > 1 && R.pieces.size() == 1 && !R.error) pz.solo_rounds = 8;
            if (R.error) throw "fastq.cpp:next_read: Unable to read header";
            size_t total = 0;
            for (const pgz::Piece &pc : R.pieces) total += pc.out.size();
            if (total == 0 && !R.stream_end) {
                // not one whole block in this span: look at more of the file -- or the file is cut short: what one zlib stream
                // still gets out of it is handed out and the input ends there, as it does for gzread / gzgets (fastq.cpp:8-30)
                if ((off_t)want >= size - pos) {
                    pgz::Bytes tail;
                    if (!pgz::inflate_truncated_tail(cbuf.data(), want, pz.bit, pz.window.data() + (pgz::kWin - pz.window_len), pz.window_len, tail))
                        throw "fastq.cpp:next_read: Unable to read header";
                    if (tail.size()) pz.pend.push_back(std::move(tail));
                    pos = size;
                    pz.in_member = false;
                    return;
                }
                pz.span *= 2;
                continue;
            }
            // CRC-32 of the pieces in parallel, combined in order (RFC 1952 trailer)
            vector<uint32_t> crcs(R.pieces.size());
            fork_join((int)R.pieces.size(), [&](int q) {
                uLong c = crc32(0L, Z_NULL, 0);
                const pgz::Bytes &o = R.pieces[q].out;
                for (size_t at = 0; at < o.size(); at += 1u << 30) c = crc32(c, o.data() + at, (uInt)min<size_t>(o.size() - at, 1u << 30));
                crcs[q] = (uint32_t)c;
            });
            for (size_t q = 0; q < R.pieces.size(); ++q) {
                pz.crc = (uint32_t)crc32_combine(pz.crc, crcs[q], (z_off_t)R.pieces[q].out.size());
                if (R.pieces[q].out.size()) pz.pend.push_back(std::move(R.pieces[q].out));
            }
            pz.isize += total;
            pz.window_len = min(pgz::kWin, pz.window_len + total);
            pos += (off_t)(R.end_bit >> 3);
            pz.bit = R.end_bit & 7;
            if (R.stream_end) {
                if (size - pos < 8) { pos = size; pz.in_member = false; return; }      // the file ends inside the trailer: cut short, as above
                uint8_t t[8];
                pread_full(fd, t, 8, pos);
                const uint32_t crc = t[0] | (uint32_t)t[1] << 8 | (uint32_t)t[2] << 16 | (uint32_t)t[3] << 24;
                const uint32_t isz = t[4] | (uint32_t)t[5] << 8 | (uint32_t)t[6] << 16 | (uint32_t)t[7] << 24;
                if (crc != pz.crc || isz != (uint32_t)pz.isize) throw "fastq.cpp:next_read: Unable to read header";
                pos += 8;
                pz.in_member = false;
            }
            return;
        }
    }
    size_t fill_pgzip(uint8_t *buf, size_t have, size_t cap, size_t *new_lines)
    {
        size_t n = have;
        while (n < cap) {
            if (pz.pend.empty()) {
                if (eof) break;
                pz_produce();           // sets eof when the file holds no further member
                continue;
            }
            const pgz::Bytes &front = pz.pend.front();
            const size_t take = min(cap - n, front.size() - pz.pend_off);
            memcpy(buf + n, front.data() + pz.pend_off, take);
            pz.pend_off += take;
            n += take;
            if (pz.pend_off == front.size()) { pz.pend.pop_front(); pz.pend_off = 0; }
        }
        *new_lines += count_newlines(buf + have, n - have);
        return n;
    }
};

// offset just past the keep-th of the `total` newlines in buf[0..n): walks back from the end
static size_t offset_after_line(const uint8_t *buf, size_t n, size_t total, size_t keep)
{
    const uint8_t *q = buf + n;
    for (size_t i = total; i >= keep; --i) {
        q = (const uint8_t *)memrchr(buf, '\n', (size_t)(q - buf));
        if (!q) return n;
        if (i == keep) break;
    }
    return (size_t)(q - buf) + 1;
}
static size_t offset_of_record(const uint8_t *buf, size_t n, size_t k)
{
    size_t lines = 0;
    const uint8_t *p = buf, *end = buf + n;
    if (k == 0) return 0;
    while (p < end) {
        const uint8_t *nl = (const uint8_t *)memchr(p, '\n', (size_t)(end - p));
        if (!nl) break;
        p = nl + 1;
        if (++lines == 4 * k) return (size_t)(p - buf);
    }
    return n;
}

struct Run {
    Cli &o;
    fq_ctx *ctx = nullptr;          // context of the first device: autodetection, statistics after the merge
    vector<fq_ctx *> ctxs;          // one per device; batch k runs on ctxs[k % n] (created after autodetection, with its result)
    fq_options fopt{};
    uint64_t records_done = 0, batches_done = 0;
    bool first_batch = true;
    bool pieces_mode = false;       // streams come back as pieces of the input buffers + literal bytes (fq_set_output_pieces)
    explicit Run(Cli &opt) : o(opt) {}
    void check(fq_status st, fq_ctx *c = nullptr) { if (st != FQ_OK) throw string(fq_last_error(c ? c : ctx)); }
    // the other devices' contexts, once the quality offset is known (A1 runs once, before sharding: SURVEY 8(e))
    void create_peers()
    {
        while (ctxs.size() < o.devices.size()) {
            fq_options f = fopt;
            f.input_quality_offset = o.input_quality_offset;
            f.quality = o.quality;
            fq_ctx *c = nullptr;
            if (fq_create(&f, o.devices[ctxs.size()], &c) != FQ_OK) throw string(fq_last_error(nullptr));
            ctxs.push_back(c);
            if (pieces_mode) check(fq_set_output_pieces(c, 1), c);
            if (o.kmer_rarefaction) check(fq_kmer_enable(c, o.kmer, o.split_size, o.num_subsample), c);   // one shard of the pass's table
            if (o.dup_stats) check(fq_dup_enable(c), c);
            if (o.insert_size) check(fq_overlap_enable(c, (uint32_t)o.insert_min_overlap, (uint32_t)o.insert_diff_limit, (uint32_t)o.insert_diff_pct), c);
            if (o.overrep) check(fq_overrep_enable(c, (uint32_t)o.overrep_len, (uint32_t)o.overrep_ppm), c);
            if (o.tile_quality) check(fq_tile_qual_enable(c), c);
        }
    }
    // end of an input's pass: the contexts' k-mer tables merge into the run's curve and histogram (FaQCs.cpp:518-537, 737-756)
    void kmer_end_pass() { check(fq_kmer_end_pass_all(ctxs.data(), (int)ctxs.size(), nullptr)); }
    // --dup_stats: the contexts' duplication tables merge into the pass's result, one block of prefix.duplication.txt
    string dup_report;
    void dup_end_pass(bool paired)
    {
        if (!o.dup_stats) return;
        check(fq_dup_end_pass_all(ctxs.data(), (int)ctxs.size(), nullptr));
        fq_dup_view v;
        check(fq_dup_results(ctx, &v));
        dup_report += string("pass\t") + (paired ? "paired" : "unpaired") + "\tunits\t" + to_string(v.units) + "\tdistinct\t" + to_string(v.distinct) +
                      "\tduplicates\t" + to_string(v.units - v.distinct) + "\n";
        for (uint64_t i = 0; i < v.n_levels; ++i) dup_report += to_string(v.levels[2 * i]) + "\t" + to_string(v.levels[2 * i + 1]) + "\n";
    }
    // --insert_size: the contexts' overlap accumulators summed after the paired pass, the text of prefix.insert_size.txt
    string insert_report;
    void overlap_end_pass()
    {
        if (!o.insert_size) return;
        check(fq_overlap_end_pass_all(ctxs.data(), (int)ctxs.size(), nullptr));
        fq_overlap_view v;
        check(fq_overlap_results(ctx, &v));
        const pair<const char *, uint64_t> totals[] = {{"pairs", v.pairs}, {"too_short", v.too_short}, {"overlapped", v.overlapped},
                                                       {"r1_adapter", v.r1_adapter}, {"r2_adapter", v.r2_adapter},
                                                       {"overlap_bases", v.overlap_bases}, {"mismatch_bases", v.mismatch_bases}};
        for (const auto &t : totals) insert_report += string(t.first) + "\t" + to_string(t.second) + "\n";
        insert_report += "#insert_size\tpairs\n";
        for (uint32_t s = 0; s < v.n_insert; ++s)
            if (v.insert_hist[s]) insert_report += to_string(s) + "\t" + to_string(v.insert_hist[s]) + "\n";
        insert_report += "#cycle\tr1_overlap\tr1_mismatch\tr2_overlap\tr2_mismatch\n";
        for (uint32_t c = 0; c < v.n_cycles; ++c)
            insert_report += to_string(c + 1) + "\t" + to_string(v.r1_overlap[c]) + "\t" + to_string(v.r1_mismatch[c]) + "\t" +
                             to_string(v.r2_overlap[c]) + "\t" + to_string(v.r2_mismatch[c]) + "\n";
    }
    // --overrep: the contexts' count tables merged after each input pass, one block of prefix.overrepresented.txt
    string overrep_report;
    void overrep_end_pass(bool paired)
    {
        if (!o.overrep) return;
        check(fq_overrep_end_pass_all(ctxs.data(), (int)ctxs.size(), nullptr));
        fq_overrep_view v;
        check(fq_overrep_results(ctx, &v));
        overrep_report += string("pass\t") + (paired ? "paired" : "unpaired") + "\tprefix_len\t" + to_string(v.prefix_len) + "\tppm\t" + to_string(v.min_ppm) + "\n";
        overrep_report += "#mate\treads\tmin_count\n";
        for (int m = 0; m < (paired ? 2 : 1); ++m) overrep_report += to_string(m + 1) + "\t" + to_string(v.reads[m]) + "\t" + to_string(v.min_count[m]) + "\n";
        overrep_report += "#mate\tcount\tpercent\tsequence\tsource\n";
        for (uint64_t i = 0; i < v.n_seqs; ++i) {
            const fq_overrep_seq &q = v.seqs[i];
            const string seq(reinterpret_cast<const char *>(v.bytes + q.offset), q.len);
            char pct[32];
            snprintf(pct, sizeof pct, "%.4f", 100.0 * (double)q.count / (double)v.reads[q.mate - 1]);
            overrep_report += to_string(q.mate) + "\t" + to_string(q.count) + "\t" + pct + "\t" + seq + "\t" + overrep_source(seq) + "\n";
        }
    }
    // --tile_quality: the contexts' tile tables united after each input pass, one block of prefix.tile_quality.txt.  Means
    // and deltas are double arithmetic on the exact sums, printed %.2f; NA where there is no base.
    string tile_report;
    static string fixed2(double x)
    {
        char b[64];
        snprintf(b, sizeof b, "%.2f", x);
        return b;
    }
    void tile_qual_end_pass(bool paired)
    {
        if (!o.tile_quality) return;
        check(fq_tile_qual_end_pass_all(ctxs.data(), (int)ctxs.size(), nullptr));
        fq_tile_qual_view v;
        check(fq_tile_qual_results(ctx, &v));
        const uint32_t M = paired ? 2 : 1, C = v.cycles, T = v.n_tiles;
        tile_report += string("pass\t") + (paired ? "paired" : "unpaired") + "\ttiles\t" + to_string(T) + "\tcycles\t" + to_string(C) +
                       "\toverflow\t" + to_string(v.overflow) + "\n";
        tile_report += "#mate\treads\ttiled\tuntiled\n";
        for (uint32_t m = 0; m < M; ++m)
            tile_report += to_string(m + 1) + "\t" + to_string(v.reads[m]) + "\t" + to_string(v.reads[m] - v.untiled[m]) + "\t" + to_string(v.untiled[m]) + "\n";
        if (v.overflow) return;
        // v.n_mates is 0 for a pass without batches: every row then has no reads
        auto at = [&](const uint64_t *a, uint32_t t, uint32_t m, uint32_t c) { return m < v.n_mates ? a[((size_t)t * v.n_mates + m) * C + c] : 0ull; };
        auto tot = [&](const uint64_t *a, uint32_t t, uint32_t m) { return m < v.n_mates ? a[(size_t)t * v.n_mates + m] : 0ull; };
        vector<double> all((size_t)M * C, 0.0);
        vector<bool> has((size_t)M * C, false);
        tile_report += "#mate\tmean_by_cycle\n";
        for (uint32_t m = 0; m < M; ++m) {
            tile_report += to_string(m + 1);
            for (uint32_t c = 0; c < C; ++c) {
                uint64_t b = 0, q = 0;
                for (uint32_t t = 0; t < T; ++t) { b += at(v.cycle_bases, t, m, c); q += at(v.cycle_qsum, t, m, c); }
                has[(size_t)m * C + c] = b != 0;
                if (b) all[(size_t)m * C + c] = (double)q / (double)b;
                tile_report += "\t" + (b ? fixed2(all[(size_t)m * C + c]) : string("NA"));
            }
            tile_report += "\n";
        }
        tile_report += "#lane\ttile\tmate\treads\tbases\tmean\tworst_cycle\tworst_delta\tdelta_by_cycle\n";
        for (uint32_t t = 0; t < T; ++t)
            for (uint32_t m = 0; m < M; ++m) {
                const uint64_t bases = tot(v.tile_bases, t, m);
                string row = to_string(v.lane[t]) + "\t" + to_string(v.tile[t]) + "\t" + to_string(m + 1) + "\t" + to_string(tot(v.tile_reads, t, m)) + "\t" +
                             to_string(bases) + "\t" + (bases ? fixed2((double)tot(v.tile_qsum, t, m) / (double)bases) : string("NA"));
                string deltas;
                uint32_t worst = C;
                double worst_d = 0.0;
                for (uint32_t c = 0; c < C; ++c) {
                    const uint64_t b = at(v.cycle_bases, t, m, c);
                    if (!b) { deltas += "\tNA"; continue; }
                    const double d = (double)at(v.cycle_qsum, t, m, c) / (double)b - all[(size_t)m * C + c];
                    if (worst == C || d < worst_d) { worst = c; worst_d = d; }
                    deltas += "\t" + fixed2(d);
                }
                row += worst < C ? "\t" + to_string(worst + 1) + "\t" + fixed2(worst_d) : string("\tNA\tNA");
                tile_report += row + deltas + "\n";
            }
    }
    // The first of the nine built-in adapters, PhiX174 and the --artifactFile entries (in that order) that holds some 20-base
    // window of the upper-cased sequence (the whole sequence if it is shorter), on either strand; "No Hit" otherwise.
    vector<pair<string, string>> sources;      // name, upper-cased entry + '\n' + its reverse complement
    unordered_map<string, size_t> source_of;   // 20-base window -> first entry holding it
    string overrep_source(string s)
    {
        const size_t W = 20;
        if (sources.empty()) {
            vector<pair<string, string>> list;
            for (auto &b : kBuiltinAdapters) list.push_back(make_pair(string(b[0]), string(b[1])));
            list.push_back(make_pair(string("PhiX174"), string(kPhiXSeq)));
            list.insert(list.end(), o.artifacts.begin(), o.artifacts.end());
            for (size_t k = 0; k < list.size(); ++k) {
                string e = list[k].second;
                for (char &c : e) c = (char)toupper((unsigned char)c);
                e += "\n" + reverse_complement(e);
                for (size_t p = 0; p + W <= e.size(); ++p) source_of.emplace(e.substr(p, W), k);
                sources.push_back(make_pair(list[k].first, e));
            }
        }
        for (char &c : s) c = (char)toupper((unsigned char)c);
        size_t best = sources.size();
        if (s.size() < W) {
            for (size_t k = 0; k < sources.size() && best == sources.size(); ++k)
                if (sources[k].second.find(s) != string::npos) best = k;
        } else {
            for (size_t p = 0; p + W <= s.size(); ++p) {
                const auto it = source_of.find(s.substr(p, W));
                if (it != source_of.end()) best = min(best, it->second);
            }
        }
        return best < sources.size() ? sources[best].first : string("No Hit");
    }
    void set_quality_everywhere(int q) { for (fq_ctx *c : ctxs) check(fq_set_quality(c, q), c); }
};

static int open_out(const string &fn, const char *what, bool append = false)
{
    const int fd = ::open(fn.c_str(), O_RDWR | O_CREAT | (append ? 0 : O_TRUNC), 0666);      // O_RDWR: shared mappings need read access
    if (fd < 0 || (append && lseek(fd, 0, SEEK_END) < 0 && errno != ESPIPE)) { cerr << "Unable to open " << fn << " for writing " << what << endl; throw "I/O error"; }
    return fd;
}
static void write_all(int fd, const uint8_t *p, size_t n)
{
    while (n) {
        const ssize_t w = ::write(fd, p, min<size_t>(n, 1u << 30));
        if (w < 0) {
            if (errno == EINTR) continue;
            throw "I/O error while writing the trimmed reads";
        }
        p += w;
        n -= (size_t)w;
    }
}
// --gz_out: one batch of a stream as BGZF members (<= 0xff00 bytes of text each, SAM specification 4.1), deflated by
// several threads into per-thread buffers and written in order.  Concatenated members are a valid gzip file; the empty
// end-of-file member is written when the stream is closed.
static void bgzf_member(vector<uint8_t> &out, z_stream &zs, const uint8_t *p, size_t n)
{
    const size_t at = out.size();
    out.resize(at + 18 + compressBound((uLong)n) + 8);
    uint8_t *h = out.data() + at;
    const uint8_t head[16] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0};
    memcpy(h, head, 16);
    deflateReset(&zs);
    zs.next_in = const_cast<uint8_t *>(p); zs.avail_in = (uInt)n;
    zs.next_out = h + 18; zs.avail_out = (uInt)(out.size() - at - 18 - 8);
    if (deflate(&zs, Z_FINISH) != Z_STREAM_END) throw "I/O error while compressing the trimmed reads";
    const size_t clen = zs.total_out, total = 18 + clen + 8;
    if (total > 0x10000) throw "I/O error while compressing the trimmed reads";       // cannot happen: 0xff00 bytes of input
    h[16] = (uint8_t)((total - 1) & 0xff); h[17] = (uint8_t)((total - 1) >> 8);
    const uint32_t crc = (uint32_t)crc32(crc32(0L, Z_NULL, 0), p, (uInt)n), isize = (uint32_t)n;
    uint8_t *t = h + 18 + clen;
    for (int i = 0; i < 4; ++i) { t[i] = (uint8_t)(crc >> (8 * i)); t[4 + i] = (uint8_t)(isize >> (8 * i)); }
    out.resize(at + total);
}
static void write_bgzf(int fd, const uint8_t *p, size_t n)
{
    constexpr size_t kBlock = 0xff00;
    const size_t blocks = (n + kBlock - 1) / kBlock;
    const int nt = (int)max<size_t>(1, min<size_t>((size_t)inflate_threads(), blocks / 8));      // deflate is the slow side: as many threads as the readers get
    vector<vector<uint8_t>> part(nt);
    fork_join(nt, [&](int t) {
        z_stream zs{};
        if (deflateInit2(&zs, 4, Z_DEFLATED, -15, 8, Z_DEFAULT_STRATEGY) != Z_OK) throw "I/O error while compressing the trimmed reads";
        const unique_ptr<z_stream, int (*)(z_streamp)> end(&zs, deflateEnd);
        for (size_t b = blocks * t / nt; b < blocks * (t + 1) / nt; ++b) bgzf_member(part[t], zs, p + b * kBlock, min(kBlock, n - b * kBlock));
    });
    for (const vector<uint8_t> &b : part) write_all(fd, b.data(), b.size());
}
static void close_bgzf(int fd)
{
    static const uint8_t eof_member[28] = {0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 'B', 'C', 2, 0, 0x1b, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0};
    write_all(fd, eof_member, sizeof(eof_member));
}

// Large appends to a regular file: reserve the range (posix_fallocate reports a full disk as an error instead of a
// SIGBUS later), map it and let kIoThreads threads copy disjoint slices -- write(2) calls on one file serialise on its
// inode lock, page faults into a shared mapping do not.  dst stays null when the file cannot be mapped (not a regular file,
// the position not at its end, no room, mmap refused); the caller then writes with write(2).
struct AppendMap {
    uint8_t *dst = nullptr;
    void *m = MAP_FAILED;
    size_t len = 0;
    off_t end = 0;
    AppendMap(int fd, size_t n)
    {
        struct stat st;
        const off_t base = lseek(fd, 0, SEEK_CUR);
        if (base < 0 || fstat(fd, &st) != 0 || !S_ISREG(st.st_mode) || st.st_size != base || posix_fallocate(fd, base, (off_t)n) != 0) return;
        const long page = sysconf(_SC_PAGESIZE);
        const off_t map_off = base / page * page;
        len = (size_t)(base - map_off) + n;
        end = base + (off_t)n;
        m = mmap(nullptr, len, PROT_READ | PROT_WRITE, MAP_SHARED, fd, map_off);
        if (m != MAP_FAILED) dst = (uint8_t *)m + (base - map_off);
        else if (ftruncate(fd, base) != 0) throw "I/O error while writing the trimmed reads";
    }
    AppendMap(const AppendMap &) = delete;
    AppendMap &operator=(const AppendMap &) = delete;
    ~AppendMap() { if (m != MAP_FAILED) munmap(m, len); }
    // all n bytes are in place: the next write goes after them
    void finish(int fd) const { if (lseek(fd, end, SEEK_SET) < 0) throw "I/O error while writing the trimmed reads"; }
};

static void write_mapped(int fd, const uint8_t *p, size_t n)
{
    if (n >= io_slice_min() && n >= (size_t)kIoThreads) {
        AppendMap a(fd, n);
        if (a.dst) {
            const size_t per = (n + kIoThreads - 1) / kIoThreads;
            fork_join(kIoThreads, [&](int t) {
                const size_t lo = min(n, per * t), hi = min(n, per * (t + 1));
                memcpy(a.dst + lo, p + lo, hi - lo);
            });
            a.finish(fd);
            return;
        }
    }
    write_all(fd, p, n);
}

// Pieces mode (fq_set_output_pieces): a stream of one batch is a list of pieces of the batch's own input buffers plus the
// literal bytes of the records that changed; only those crossed the PCIe link on the way back.  The file range is reserved and
// mapped like write_mapped's; kIoThreads threads copy disjoint runs of pieces (a first pass gives every run its offset).
static void write_pieces(int fd, const fq_out_piece *pc, size_t n_pc, const uint8_t *const src[3], size_t total)
{
    if (total == 0) return;
    if (total >= (size_t)kIoThreads) {
        AppendMap a(fd, total);
        if (a.dst) {
            const int nt = kIoThreads;
            size_t start[kIoThreads + 1] = {0};
            fork_join(nt, [&](int t) {
                size_t b = 0;
                for (size_t k = n_pc * t / nt; k < n_pc * (t + 1) / nt; ++k) b += pc[k].source < 3 ? pc[k].length : total + 1;     // unknown source: fail below
                start[t + 1] = b;
            });
            for (int t = 0; t < nt; ++t) start[t + 1] += start[t];
            if (start[nt] != total) throw "pieces of a stream do not add up to its size";
            fork_join(nt, [&](int t) {
                uint8_t *d = a.dst + start[t];
                for (size_t k = n_pc * t / nt; k < n_pc * (t + 1) / nt; ++k) { memcpy(d, src[pc[k].source] + pc[k].offset, pc[k].length); d += pc[k].length; }
            });
            a.finish(fd);
            return;
        }
    }
    vector<iovec> iov;                                // pipes, odd files: gather the pieces with writev
    iov.reserve(1024);
    auto flush = [&] {
        size_t done = 0;
        while (done < iov.size()) {
            ssize_t w = writev(fd, iov.data() + done, (int)min<size_t>(iov.size() - done, 1024));
            if (w < 0) { if (errno == EINTR) continue; throw "I/O error while writing the trimmed reads"; }
            while (w > 0 && done < iov.size()) {
                if ((size_t)w >= iov[done].iov_len) { w -= (ssize_t)iov[done].iov_len; ++done; }
                else { iov[done].iov_base = (uint8_t *)iov[done].iov_base + w; iov[done].iov_len -= (size_t)w; w = 0; }
            }
        }
        iov.clear();
    };
    for (size_t k = 0; k < n_pc; ++k) {
        if (pc[k].source > 2) throw "pieces of a stream do not add up to its size";
        iov.push_back(iovec{(void *)(src[pc[k].source] + pc[k].offset), pc[k].length});
        if (iov.size() == 1024) flush();
    }
    flush();
}

static double now_s() { return chrono::duration<double>(chrono::steady_clock::now().time_since_epoch()).count(); }

// process_paired (FaQCs.cpp:153-538) / process_unpaired (:540-757): read -> GPU -> four ordered writers.
// One reader thread per input file fills the pinned buffer of the next batch while the GPU works on the
// current one; one writer thread per output file drains the previous batch.
static void process(Run &R, bool paired)
{
    Cli &o = R.o;
    const bool timing = getenv("FAQCS_B200_TIMING") != nullptr;
    const int n_mates = paired ? 2 : 1;
    g_input_files = n_mates;
    Source src[2];
    if (paired) {
        if (!src[0].open(o.input_read1_file)) { cerr << "Unable to open " << o.input_read1_file << " for loading read one sequences" << endl; throw "I/O error"; }
        if (!src[1].open(o.input_read2_file)) { cerr << "Unable to open " << o.input_read2_file << " for loading read two sequences" << endl; throw "I/O error"; }
    } else if (!src[0].open(o.input_unpaired_file)) {
        cerr << "Unable to open " << o.input_unpaired_file << " for loading unpaired read sequences" << endl;
        throw "I/O error";
    }
    int fout[4] = {-1, -1, -1, -1};
    if (!o.qc_only) {
        if (paired) {
            fout[0] = open_out(o.trimmed_read1_file, "read one sequences");
            fout[1] = open_out(o.trimmed_read2_file, "read two sequences");
        }
        // re-opened (truncated) by the -u pass: Q11 -- unless --keep_unpaired asks for the paired pass's orphans to survive
        fout[2] = open_out(o.trimmed_unpaired_file, "unpaired sequences", !paired && o.keep_unpaired && o.has_paired());
        if (!o.trimmed_discard_file.empty()) fout[3] = open_out(o.trimmed_discard_file, "discarded sequences");
    }
    const size_t cap = o.batch_mb << 20;
    // Pieces mode: the writers copy most output bytes out of the batch's own INPUT buffers, so a buffer cycles through
    // read -> GPU -> write before it is filled again: three slots instead of two.
    const bool pieces_mode = R.pieces_mode;
    const int n_slots = pieces_mode ? 3 : 2;
    uint8_t *buf[3][2] = {{nullptr, nullptr}, {nullptr, nullptr}, {nullptr, nullptr}};      // [slot][mate], pinned
    for (int k = 0; k < n_slots; ++k)
        for (int m = 0; m < n_mates; ++m)
            if (!(buf[k][m] = (uint8_t *)fq_host_alloc(cap))) throw "unable to allocate pinned host memory";
    // Q3 and the k-mer rarefaction curve (points are taken where trim() calls end): keep batches on 32768-record boundaries
    const bool emulate = o.filter_adapter || o.filter_phiX || o.kmer_rarefaction;
    struct Filled { size_t n = 0, lines = 0; } filled[2];
    double t_read = 0, t_gpu = 0, t_write_wait = 0, t_cut = 0;
    {
        Worker readers[2], writers[4];
        auto post_fill = [&](int slot, int m, size_t have) {
            readers[m].post([&, slot, m, have] {
                size_t lines = count_newlines(buf[slot][m], have);        // the carried tail
                filled[m].n = src[m].fill(buf[slot][m], have, cap, &lines);
                filled[m].lines = lines;
            });
        };
        for (int m = 0; m < n_mates; ++m) post_fill(0, m, 0);
        uint64_t first_index = 0, pending_ticket = 0;
        fq_ctx *pending_ctx = nullptr;
        const uint8_t *pending_src[2] = {nullptr, nullptr};
        bool have_pending = false;
        auto drain = [&](fq_ctx *c, uint64_t ticket) {
            fq_batch_out out;
            R.check(fq_wait(c, ticket, &out), c);
            for (int s = 0; s < 4; ++s)
                if (fout[s] >= 0 && out.bytes[s]) {
                    const uint8_t *p = out.data[s];
                    const size_t n = out.bytes[s];
                    const int fd = fout[s];
                    const bool gz = o.gz_out;
                    if (pieces_mode) {
                        const fq_out_piece *pc = out.pieces[s];
                        const size_t n_pc = out.n_pieces[s];
                        const uint8_t *s0 = pending_src[0], *s1 = pending_src[1];
                        writers[s].post([fd, pc, n_pc, s0, s1, p, n] { const uint8_t *const src3[3] = {s0, s1, p}; write_pieces(fd, pc, n_pc, src3, n); });
                    } else writers[s].post([fd, p, n, gz] { if (gz) write_bgzf(fd, p, n); else write_mapped(fd, p, n); });
                }
        };
        for (int slot = 0;; slot = (slot + 1) % n_slots) {
            const int next = (slot + 1) % n_slots;
            double t0 = now_s();
            for (int m = 0; m < n_mates; ++m) readers[m].wait_idle();
            t_read += now_s() - t0;
            t0 = now_s();
            const size_t n1 = filled[0].n, n2 = paired ? filled[1].n : 0;
            const bool at_eof = src[0].eof && (!paired || src[1].eof);
            size_t use1 = n1, use2 = n2, nrec = filled[0].lines / 4;
            if (!at_eof) {
                const size_t r1 = filled[0].lines / 4, r2 = paired ? filled[1].lines / 4 : r1;
                nrec = min(r1, r2);
                // whole reference batches where possible: Q3 emulation needs it, and the NextSeq re-check at the end of the
                // input looks at the first read of the reference's final partial batch
                if ((emulate || (int)o.quality < 20) && nrec >= FQ_REF_BATCH) nrec -= nrec % FQ_REF_BATCH;
                if (nrec == 0) {
                    // one file ran out of whole records while the other still has data: the reference's uneven-pair error (FaQCs.cpp:370-380)
                    if (paired && ((src[0].eof && r1 == 0) || (src[1].eof && r2 == 0))) {
                        cerr << "Did not find a match to read " << (r1 == 0 ? "two" : "one") << endl;
                        throw "FaQCs.cppI/O error";
                    }
                    throw "record larger than the batch buffer: raise --batch_mb";
                }
                if (o.kmer_rarefaction && nrec % FQ_REF_BATCH) throw "--kmer_rarefaction needs batches of at least 32768 records: raise --batch_mb";
                use1 = offset_after_line(buf[slot][0], n1, filled[0].lines, 4 * nrec);
                if (paired) use2 = offset_after_line(buf[slot][1], n2, filled[1].lines, 4 * nrec);
                // the tails open the next batch; its buffers are free (their batch has been run -- and, in pieces mode, written:
                // the writers of the batch that used them read their pieces from these buffers)
                if (pieces_mode)
                    for (Worker &w : writers) w.wait_idle();
                memcpy(buf[next][0], buf[slot][0] + use1, n1 - use1);
                post_fill(next, 0, n1 - use1);
                if (paired) {
                    memcpy(buf[next][1], buf[slot][1] + use2, n2 - use2);
                    post_fill(next, 1, n2 - use2);
                }
            }
            if (R.first_batch) {
                // A1 on the first 32768 records (FaQCs.cpp:261-277, 393-414, 609-619, 669-683); an empty input throws
                const size_t a1 = offset_of_record(buf[slot][0], use1, FQ_REF_BATCH), a2 = paired ? offset_of_record(buf[slot][1], use2, FQ_REF_BATCH) : 0;
                int32_t off = 0, q = 0;
                const int q_before = o.quality;
                R.check(fq_autodetect(R.ctx, buf[slot][0], a1, paired ? buf[slot][1] : nullptr, a2, &off, &q));
                o.input_quality_offset = (char)off;
                o.quality = (char)q;
                if (q != q_before) cerr << "The input looks like NextSeq data and the quality level (-q) is adjusted to 20 for trimming." << endl;
                R.first_batch = false;
                R.create_peers();
                R.set_quality_everywhere(o.quality);
            }
            t_cut += now_s() - t0;
            // One piece per batch; the last batch may be cut in two at the start of the reference's final partial
            // 32768-read batch, whose first header the reference tests for "@NS" once more (FaQCs.cpp:272-277, 613-618).
            struct Piece { size_t o1, n1, o2, n2, nrec; bool final, recheck; };
            Piece pieces[2] = {{0, use1, 0, use2, nrec, at_eof, false}, {}};
            int n_pieces = 1;
            if (at_eof && nrec && (int)o.quality < 20) {
                const uint64_t total = first_index + nrec, rem = total % FQ_REF_BATCH;
                if (rem && total - rem >= first_index) {            // else: that batch is empty, or began in a batch already run
                    const size_t f_local = (size_t)(total - rem - first_index);
                    if (f_local == 0) pieces[0].recheck = true;
                    else {
                        const size_t c1 = offset_of_record(buf[slot][0], use1, f_local), c2 = paired ? offset_of_record(buf[slot][1], use2, f_local) : 0;
                        pieces[0] = Piece{0, c1, 0, c2, f_local, false, false};
                        pieces[1] = Piece{c1, use1 - c1, c2, use2 - c2, nrec - f_local, true, true};
                        n_pieces = 2;
                    }
                }
            }
            for (int k = 0; k < n_pieces; ++k) {
                const Piece &pc = pieces[k];
                if (!(pc.n1 || pc.n2 || pc.final)) continue;
                const uint8_t *p1 = buf[slot][0] + pc.o1, *p2 = paired ? buf[slot][1] + pc.o2 : nullptr;
                if (pc.recheck && (int)o.quality < 20 && pc.n1 >= 3 && p1[0] == '@' && p1[1] == 'N' && p1[2] == 'S') {
                    cerr << "The input looks like NextSeq data and the quality level (-q) is adjusted to 20 for trimming." << endl;
                    o.quality = 20;
                    R.set_quality_everywhere(20);
                }
                uint64_t ticket = 0;
                // this batch's outputs reuse the host slot of the batch two tickets back: its writes must be done
                t0 = now_s();
                for (Worker &w : writers) w.wait_idle();
                t_write_wait += now_s() - t0;
                t0 = now_s();
                fq_ctx *c = R.ctxs[R.batches_done++ % R.ctxs.size()];          // consecutive batches on consecutive devices
                R.check(fq_submit_host(c, p1, pc.n1, p2, pc.n2, first_index, pc.final ? 1 : 0, &ticket), c);
                R.check(fq_run(c, ticket), c);
                if (have_pending) drain(pending_ctx, pending_ticket);
                t_gpu += now_s() - t0;
                pending_ticket = ticket;
                pending_ctx = c;
                pending_src[0] = p1;
                pending_src[1] = p2;
                have_pending = true;
                first_index += pc.nrec;
            }
            if (at_eof) break;
        }
        if (have_pending) {
            for (Worker &w : writers) w.wait_idle();
            drain(pending_ctx, pending_ticket);
        }
        const double t0 = now_s();
        for (Worker &w : writers) w.wait_idle();
        t_write_wait += now_s() - t0;
    }
    if (timing)
        cerr << "[timing] waiting for readers " << t_read << " s, cut/autodetect " << t_cut << " s, submit+run+wait " << t_gpu
             << " s, waiting for writers " << t_write_wait << " s" << endl;
    for (int k = 0; k < 3; ++k)
        for (int m = 0; m < 2; ++m) fq_host_free(buf[k][m]);
    for (int s = 0; s < 4; ++s)
        if (fout[s] >= 0) {
            // a gzip stream ends with the empty member -- except the unpaired file of the paired pass when the -u pass will append to it
            if (o.gz_out && !(s == 2 && paired && o.keep_unpaired && o.has_unpaired())) close_bgzf(fout[s]);
            ::close(fout[s]);
        }
    src[0].close();
    src[1].close();
}

// write_stats (FaQCs.cpp:759-1034): same expressions, same stream state.
static void write_stats(const fq_stats_view &v, const Cli &o)
{
    ofstream fout(o.stats_file.c_str());
    if (!fout) { cerr << "Unable to open " << o.stats_file << " for writing filtering statistics" << endl; return; }
    const uint64_t *S = v.filter_stats;
    auto pct = [](uint64_t a, uint64_t b) { return (100.0 * a) / b; };
    // adapter stats are keyed by name (duplicates merge); phiX pseudo-adapters are not listed (FaQCs.cpp:92-116)
    map<string, pair<size_t, size_t>> adapters;
    for (uint32_t j = 0; j < v.n_adapters; ++j) {
        const string &name = o.adapter[j].first;
        if (name == kPhiX || name == kPhiXComplement) continue;
        if (v.adapter_reads[j] == 0 && adapters.find(name) == adapters.end()) continue;
        adapters[name].first += v.adapter_reads[j];
        adapters[name].second += v.adapter_bases[j];
    }
    auto adapter_lines = [&]() {
        deque<pair<size_t, string>> order;
        for (auto &a : adapters) order.push_back(make_pair(a.second.first, a.first));
        sort(order.begin(), order.end());
        for (auto i = order.rbegin(); i != order.rend(); ++i) {
            const auto &st = adapters[i->second];
            fout << "    " << i->second << " " << st.first << " reads (" << pct(st.first, S[FQ_TOTAL_NUMBER]) << " %) " << st.second << " bases ("
                 << pct(st.second, S[FQ_TOTAL_LENGTH]) << " %)\n";
        }
    };
    fout << fixed << setprecision(2);
    if (o.qc_only) {
        fout << "\n";
        fout << "Reads #: " << S[FQ_TOTAL_COUNT] << "\n";
        fout << "Total bases: " << S[FQ_TOTAL_LENGTH] << "\n";
        fout << "Reads Length: " << float(S[FQ_TOTAL_LENGTH]) / S[FQ_TOTAL_COUNT] << "\n";
        fout << "Processed " << S[FQ_TOTAL_NUMBER] << " reads for quality check only\n";
        fout << "  Reads length < " << o.min_read_length << " bp: " << S[FQ_READ_LENGTH] << " (" << pct(S[FQ_READ_LENGTH], S[FQ_TOTAL_NUMBER]) << " %)\n";
        fout << "  Reads have " << o.max_num_poly_N << " continuous base \"N\": " << S[FQ_READ_NN] << " (" << pct(S[FQ_READ_NN], S[FQ_TOTAL_NUMBER]) << " %)\n";
        fout << "  Low complexity Reads  (>" << o.low_complexity_cutoff_ratio * 100.0 << "% mono/di-nucleotides): " << S[FQ_READ_LOW_COMPLEXITY] << " ("
             << pct(S[FQ_READ_LOW_COMPLEXITY], S[FQ_TOTAL_NUMBER]) << " %)\n";
        fout << "  Reads < average quality " << o.average_quality << ": " << S[FQ_READ_AVG_Q] << " (" << pct(S[FQ_READ_AVG_Q], S[FQ_TOTAL_NUMBER]) << " %)\n";
        if (o.filter_phiX) fout << "  Reads hits to phiX sequence: " << S[FQ_READ_PHIX] << " (" << pct(S[FQ_READ_PHIX], S[FQ_TOTAL_NUMBER]) << " %)\n";
        if (o.filter_adapter) {
            fout << "  Reads with Adapters/Primers: " << S[FQ_READ_ADAPTER] << " (" << pct(S[FQ_READ_ADAPTER], S[FQ_TOTAL_NUMBER]) << " %)\n";
            adapter_lines();
        }
        return;
    }
    fout << "Before Trimming\n";
    fout << "Reads #: " << S[FQ_TOTAL_NUMBER] << "\n";
    fout << "Total bases: " << S[FQ_TOTAL_LENGTH] << "\n";
    fout << "Reads Length: " << float(S[FQ_TOTAL_LENGTH]) / S[FQ_TOTAL_NUMBER] << "\n";
    fout << "\nAfter Trimming\n";
    fout << "Reads #: " << S[FQ_TOTAL_TRIMMED_NUMBER] << " (" << pct(S[FQ_TOTAL_TRIMMED_NUMBER], S[FQ_TOTAL_NUMBER]) << " %)\n";
    fout << "Total bases: " << S[FQ_TOTAL_TRIMMED_LENGTH] << " (" << pct(S[FQ_TOTAL_TRIMMED_LENGTH], S[FQ_TOTAL_LENGTH]) << " %)\n";
    if (S[FQ_TOTAL_TRIMMED_NUMBER] > 0) fout << "Mean Reads Length: " << float(S[FQ_TOTAL_TRIMMED_LENGTH]) / S[FQ_TOTAL_TRIMMED_NUMBER] << "\n";
    else fout << "Mean Reads Length: 0\n";
    if (o.has_paired()) {
        fout << "  Paired Reads #: " << S[FQ_PAIRED_READ_NUMBER] << " (" << pct(S[FQ_PAIRED_READ_NUMBER], S[FQ_TOTAL_TRIMMED_NUMBER]) << " %)\n";
        fout << "  Paired total bases: " << S[FQ_PAIRED_BASE_LENGTH] << " (" << pct(S[FQ_PAIRED_BASE_LENGTH], S[FQ_TOTAL_TRIMMED_LENGTH]) << " %)\n";
        fout << "  Unpaired Reads #: " << S[FQ_TOTAL_TRIMMED_NUMBER] - S[FQ_PAIRED_READ_NUMBER] << " ("
             << pct(S[FQ_TOTAL_TRIMMED_NUMBER] - S[FQ_PAIRED_READ_NUMBER], S[FQ_TOTAL_TRIMMED_NUMBER]) << " %)\n";
        fout << "  Unpaired total bases: " << S[FQ_TOTAL_TRIMMED_LENGTH] - S[FQ_PAIRED_BASE_LENGTH] << " ("
             << pct(S[FQ_TOTAL_TRIMMED_LENGTH] - S[FQ_PAIRED_BASE_LENGTH], S[FQ_TOTAL_TRIMMED_LENGTH]) << " %)\n";
    }
    fout << "\nDiscarded reads #: " << S[FQ_TOTAL_NUMBER] - S[FQ_TOTAL_TRIMMED_NUMBER] << " (" << pct(S[FQ_TOTAL_NUMBER] - S[FQ_TOTAL_TRIMMED_NUMBER], S[FQ_TOTAL_NUMBER]) << " %)\n";
    fout << "Trimmed bases: " << S[FQ_TOTAL_LENGTH] - S[FQ_TOTAL_TRIMMED_LENGTH] << " (" << pct(S[FQ_TOTAL_LENGTH] - S[FQ_TOTAL_TRIMMED_LENGTH], S[FQ_TOTAL_LENGTH]) << " %)\n";
    fout << "  Reads Filtered by length cutoff (" << o.min_read_length << " bp): " << S[FQ_READ_LENGTH] << " (" << pct(S[FQ_READ_LENGTH], S[FQ_TOTAL_NUMBER]) << " %)\n";
    fout << "  Bases Filtered by length cutoff: " << S[FQ_BASE_LENGTH] << " (" << pct(S[FQ_BASE_LENGTH], S[FQ_TOTAL_LENGTH]) << " %)\n";
    fout << "  Reads Filtered by continuous base \"N\" (" << o.max_num_poly_N << "): " << S[FQ_READ_NN] << " (" << pct(S[FQ_READ_NN], S[FQ_TOTAL_NUMBER]) << " %)\n";
    fout << "  Bases Filtered by continuous base \"N\": " << S[FQ_BASE_NN] << " (" << pct(S[FQ_BASE_NN], S[FQ_TOTAL_LENGTH]) << " %)\n";
    fout << "  Reads Filtered by low complexity ratio (" << setprecision(1) << o.low_complexity_cutoff_ratio << setprecision(2) << "): " << S[FQ_READ_LOW_COMPLEXITY]
         << " (" << pct(S[FQ_READ_LOW_COMPLEXITY], S[FQ_TOTAL_NUMBER]) << " %)\n";
    fout << "  Bases Filtered by low complexity ratio: " << S[FQ_BASE_LOW_COMPLEXITY] << " (" << pct(S[FQ_BASE_LOW_COMPLEXITY], S[FQ_TOTAL_LENGTH]) << " %)\n";
    if (o.average_quality > 0.0) {
        fout << "  Reads Filtered by avg quality (" << o.average_quality << "): " << S[FQ_READ_AVG_Q] << " (" << pct(S[FQ_READ_AVG_Q], S[FQ_TOTAL_NUMBER]) << " %)\n";
        fout << "  Bases Filtered by avg quality: " << S[FQ_BASE_AVG_Q] << " (" << pct(S[FQ_BASE_AVG_Q], S[FQ_TOTAL_LENGTH]) << " %)\n";
    }
    if (o.filter_phiX) {
        fout << "  Reads Filtered by phiX sequence: " << S[FQ_READ_PHIX] << " (" << pct(S[FQ_READ_PHIX], S[FQ_TOTAL_NUMBER]) << " %)\n";
        fout << "  Bases Filtered by phiX sequence: " << S[FQ_BASE_PHIX] << " (" << pct(S[FQ_BASE_PHIX], S[FQ_TOTAL_LENGTH]) << " %)\n";
    }
    fout << "  Reads Trimmed by quality (" << setprecision(1) << float(o.quality) << setprecision(2) << "): " << S[FQ_READ_QUAL_TRIM] << " ("
         << pct(S[FQ_READ_QUAL_TRIM], S[FQ_TOTAL_NUMBER]) << " %)\n";
    fout << "  Bases Trimmed by quality: " << S[FQ_BASE_QUAL_TRIM] << " (" << pct(S[FQ_BASE_QUAL_TRIM], S[FQ_TOTAL_LENGTH]) << " %)\n";
    if (o.trim_5 > 0) fout << "  Reads Trimmed with " << o.trim_5 << " bp from 5' end\n";
    if (o.trim_3 > 0) fout << "  Reads Trimmed with " << o.trim_3 << " bp from 3' end\n";
    if (o.filter_adapter) {
        fout << "  Reads Trimmed with Adapters/Primers: " << S[FQ_READ_ADAPTER] << " (" << pct(S[FQ_READ_ADAPTER], S[FQ_TOTAL_NUMBER]) << " %)\n";
        fout << "  Bases Trimmed with Adapters/Primers: " << S[FQ_BASE_ADAPTER] << " (" << pct(S[FQ_BASE_ADAPTER], S[FQ_TOTAL_LENGTH]) << " %)\n";
        adapter_lines();
    }
    if (o.replace_N) fout << "\nN base random substitution: A " << S[FQ_N_TO_A] << ", T " << S[FQ_N_TO_T] << ", C " << S[FQ_N_TO_C] << ", G " << S[FQ_N_TO_G] << "\n";
}

// The ten --debug data files of plot() (plot.cpp:31-78, writers :540-681).
static void write_debug_files(const fq_stats_view &v, const Cli &o)
{
    const string dir = o.output_dir + "/";
    auto write_matrix = [&](const string &fn, const uint64_t *m, uint32_t rows, uint32_t cols) {
        if (rows == 0) return;
        ofstream f(fn.c_str());
        for (uint32_t i = 0; i < rows; ++i) {
            f << m[(size_t)i * cols];
            for (uint32_t j = 1; j < cols; ++j) f << '\t' << m[(size_t)i * cols + j];
            f << endl;
        }
    };
    auto write_qhist = [&](const string &fn, const uint64_t *r, const uint64_t *b) {
        ofstream f(fn.c_str());
        f << "Score\treadsNum\treadsBases" << endl;
        for (int i = FQ_MAX_QUALITY_SCORE; i >= 0; --i) f << i << '\t' << r[i] << '\t' << b[i] << endl;
    };
    auto write_content = [&](const string &fn, const uint64_t *c) {
        ofstream f(fn.c_str());
        f << setprecision(2) << fixed;
        static const char *label[6] = {"A", "T", "C", "G", "N", "GC"};
        for (int h = 0; h < 6; ++h)
            for (unsigned i = 0; i < FQ_NUM_COMPOSITION_BIN; ++i) {
                const uint64_t num = c[(size_t)h * FQ_NUM_COMPOSITION_BIN + i];
                if (num) f << label[h] << "\t" << i * 0.01 << '\t' << num << endl;
            }
    };
    auto write_len = [&](const string &fn, const uint64_t *h, uint32_t n) {
        ofstream f(fn.c_str());
        for (uint32_t i = 1; i < n; ++i) f << i << '\t' << h[i] << endl;
    };
    write_matrix(dir + "qa." + o.prefix + ".quality.matrix", v.pre_quality_matrix, v.pre_rows, FQ_NUM_QUAL);
    write_matrix(dir + o.prefix + ".quality.matrix", v.post_quality_matrix, v.post_rows, FQ_NUM_QUAL);
    write_matrix(dir + "qa." + o.prefix + ".base.matrix", v.pre_base_matrix, v.pre_rows, FQ_NUM_BASE);
    write_matrix(dir + o.prefix + ".base.matrix", v.post_base_matrix, v.post_rows, FQ_NUM_BASE);
    write_qhist(dir + "qa." + o.prefix + ".for_qual_histogram.txt", v.pre_read_quality_hist, v.pre_base_quality_hist);
    write_qhist(dir + o.prefix + ".for_qual_histogram.txt", v.post_read_quality_hist, v.post_base_quality_hist);
    write_content(dir + "qa." + o.prefix + ".base_content.txt", v.pre_composition);
    write_content(dir + o.prefix + ".base_content.txt", v.post_composition);
    write_len(dir + "qa." + o.prefix + ".length_count.txt", v.pre_length_hist, v.pre_len_size);
    write_len(dir + o.prefix + ".length_count.txt", v.post_length_hist, v.post_len_size);
}

static void remove_file(const string &fn)      // FaQCs.cpp:1046-1053
{
    struct stat st;
    if (!fn.empty() && stat(fn.c_str(), &st) == 0) {
        cerr << "The output " << fn << " file exists and will be overwritten." << endl;
        unlink(fn.c_str());
    }
}

// plot.cpp:81-91, writers :683-733: prefix.kmerH.txt ("count number", ascending count) and prefix.Kmercount.txt (reads since
// the previous point, distinct k-mers, k-mer instances), only when some k-mer was counted.
static void write_kmer_files(const fq_kmer_view &kv, const Cli &o)
{
    if (kv.n_frequency == 0) return;
    const string base = o.output_dir + "/" + o.prefix;
    {
        ofstream fout((base + ".kmerH.txt").c_str());
        if (!fout) cerr << "Warning: Unable to write kmer histogram file: " << base << ".kmerH.txt" << endl;
        else
            for (uint64_t i = 0; i < kv.n_frequency; ++i) fout << kv.frequency[2 * i] << ' ' << kv.frequency[2 * i + 1] << '\n';
    }
    ofstream fout((base + ".Kmercount.txt").c_str());
    if (!fout) { cerr << "Warning: Unable to write kmer rarefaction file: " << base << ".Kmercount.txt" << endl; return; }
    uint64_t last = 0;
    for (uint32_t i = 0; i < kv.n_rarefaction; ++i) {
        fout << kv.rarefaction[i].num_seq - last << '\t' << kv.rarefaction[i].distinct_kmer << '\t' << kv.rarefaction[i].total_kmer << '\n';
        last = kv.rarefaction[i].num_seq;
    }
}

int main(int argc, char *argv[])
{
    Cli o;
    fq_ctx *ctx = nullptr;
    try {
        parse_options(argc, argv, o);
        if (o.print_usage) return EXIT_FAILURE;
        struct stat st;
        if (!(stat(o.output_dir.c_str(), &st) == 0 && S_ISDIR(st.st_mode)) && mkdir(o.output_dir.c_str(), 0700) != 0) {
            cerr << "Unable to create requested output directory: \"" << o.output_dir << '"' << endl;
            return EXIT_FAILURE;
        }
        for (const string *f : {&o.plots_file, &o.stats_file, &o.trimmed_read1_file, &o.trimmed_read2_file, &o.trimmed_unpaired_file, &o.trimmed_discard_file}) remove_file(*f);

        vector<fq_adapter> adapters;
        for (auto &a : o.adapter) adapters.push_back(fq_adapter{a.first.c_str(), a.second.c_str()});
        fq_options f{};
        f.mode = o.mode; f.quality = o.quality; f.trim_5 = o.trim_5; f.trim_3 = o.trim_3; f.min_read_length = o.min_read_length;
        f.max_num_poly_N = o.max_num_poly_N; f.average_quality = o.average_quality; f.low_complexity_cutoff_ratio = o.low_complexity_cutoff_ratio;
        f.adapter_mismatch_rate = o.filterAdapterMismatchRate;
        f.input_quality_offset = o.input_quality_offset == SCHAR_MIN ? FQ_OFFSET_AUTO : (int)o.input_quality_offset;
        f.output_quality_offset = o.output_quality_offset; f.replace_to_N_q = o.replace_to_N_q; f.qc_only = o.qc_only; f.protect_5 = o.protect_5;
        f.filter_adapter = o.filter_adapter || o.filter_phiX; f.discard_output = o.discard_output;
        f.num_thread = o.num_thread ? o.num_thread : max(1u, thread::hardware_concurrency());     // -t 0 = all cores (options.cpp:124)
        f.n_adapters = (uint32_t)adapters.size(); f.adapters = adapters.data();
        const bool timing = getenv("FAQCS_B200_TIMING") != nullptr;
        const double t_start = now_s();
        if (o.devices.empty()) o.devices.push_back(o.device);
        if (fq_create(&f, o.devices[0], &ctx) != FQ_OK) throw string(fq_last_error(nullptr));
        if (o.kmer_rarefaction && fq_kmer_enable(ctx, o.kmer, o.split_size, o.num_subsample) != FQ_OK) throw string(fq_last_error(ctx));
        if (o.dup_stats && fq_dup_enable(ctx) != FQ_OK) throw string(fq_last_error(ctx));
        if (o.insert_size && fq_overlap_enable(ctx, (uint32_t)o.insert_min_overlap, (uint32_t)o.insert_diff_limit, (uint32_t)o.insert_diff_pct) != FQ_OK)
            throw string(fq_last_error(ctx));
        if (o.overrep && fq_overrep_enable(ctx, (uint32_t)o.overrep_len, (uint32_t)o.overrep_ppm) != FQ_OK) throw string(fq_last_error(ctx));
        if (o.tile_quality && fq_tile_qual_enable(ctx) != FQ_OK) throw string(fq_last_error(ctx));
        const double t_created = now_s();
        Run R(o);
        R.ctx = ctx;
        R.ctxs.push_back(ctx);
        R.fopt = f;
        // plain output files: most bytes are written straight from the input buffers (FAQCS_B200_CLI_BYTES=1: byte streams)
        R.pieces_mode = !o.gz_out && !o.qc_only && getenv("FAQCS_B200_CLI_BYTES") == nullptr;
        if (R.pieces_mode) R.check(fq_set_output_pieces(ctx, 1));
        if (o.has_paired()) {
            process(R, true);
            R.kmer_end_pass();                     // FaQCs.cpp:518-537
            R.dup_end_pass(true);
            R.overlap_end_pass();
            R.overrep_end_pass(true);
            R.tile_qual_end_pass(true);
        }
        if (o.has_unpaired()) {
            R.first_batch = true;      // offset detection only if still unknown; the NextSeq check runs per input (FaQCs.cpp:586,673-683)
            process(R, false);
            R.kmer_end_pass();                     // FaQCs.cpp:737-756
            R.dup_end_pass(false);
            R.overrep_end_pass(false);
            R.tile_qual_end_pass(false);
        }
        const double t_processed = now_s();
        if (R.ctxs.size() > 1) {
            // the path's only collective (SURVEY 8(e)): one ncclAllReduce of the integer statistics over NVLink
            // (a device listed more than once = several contexts on it, so that its batches overlap: those merge locally first)
            vector<fq_ctx *> heads;
            vector<int> head_dev;
            for (size_t k = 0; k < R.ctxs.size(); ++k) {
                size_t h = 0;
                while (h < heads.size() && head_dev[h] != o.devices[k]) ++h;
                if (h == heads.size()) { heads.push_back(R.ctxs[k]); head_dev.push_back(o.devices[k]); }
                else R.check(fq_merge_stats(heads[h], R.ctxs[k]), heads[h]);
            }
            if (heads.size() > 1) {
                vector<fq_comm *> comms(heads.size(), nullptr);
                R.check(fq_comm_init_all(heads.data(), (int)heads.size(), comms.data()));
                const fq_status st = fq_allreduce_stats(heads.data(), (int)heads.size(), comms.data());
                for (fq_comm *c : comms) fq_comm_destroy(c);
                R.check(st);
            }
        }
        fq_stats_view v;
        if (fq_stats(ctx, &v) != FQ_OK) throw string(fq_last_error(ctx));
        write_stats(v, o);
        if (o.dup_stats) {
            const string fn = o.output_dir + "/" + o.prefix + ".duplication.txt";
            ofstream fout(fn.c_str());
            fout << R.dup_report;
            fout.close();
            if (!fout) throw string("Unable to write the duplication statistics file: ") + fn;
        }
        if (o.insert_size) {
            const string fn = o.output_dir + "/" + o.prefix + ".insert_size.txt";
            ofstream fout(fn.c_str());
            fout << R.insert_report;
            fout.close();
            if (!fout) throw string("Unable to write the insert size file: ") + fn;
        }
        if (o.overrep) {
            const string fn = o.output_dir + "/" + o.prefix + ".overrepresented.txt";
            ofstream fout(fn.c_str());
            fout << R.overrep_report;
            fout.close();
            if (!fout) throw string("Unable to write the overrepresented sequences file: ") + fn;
        }
        if (o.tile_quality) {
            const string fn = o.output_dir + "/" + o.prefix + ".tile_quality.txt";
            ofstream fout(fn.c_str());
            fout << R.tile_report;
            fout.close();
            if (!fout) throw string("Unable to write the tile quality file: ") + fn;
        }
        if (!o.trim_only && o.debug) {                           // the reference deletes these unless --debug (plot.cpp:517-537)
            write_debug_files(v, o);
            fq_kmer_view kv;
            if (fq_kmer_results(ctx, &kv) != FQ_OK) throw string(fq_last_error(ctx));
            write_kmer_files(kv, o);
        }
        const double t_stats = now_s();
        // Every output file is closed by now.  Releasing gigabytes of pinned and device memory and tearing the CUDA context down
        // costs more than short runs take; the driver reclaims all of it when the process ends, so the orderly teardown is opt-in
        // (FAQCS_B200_FULL_TEARDOWN=1: leak checkers).
        const bool teardown = getenv("FAQCS_B200_FULL_TEARDOWN") != nullptr;
        if (teardown) {
            for (size_t k = 1; k < R.ctxs.size(); ++k) fq_destroy(R.ctxs[k]);
            fq_destroy(ctx);
        }
        if (timing)
            cerr << "[timing] fq_create " << t_created - t_start << " s, process " << t_processed - t_created << " s, stats files "
                 << t_stats - t_processed << " s, fq_destroy " << now_s() - t_stats << " s" << endl;
        if (!teardown) {
            cerr.flush();
            cout.flush();
            _exit(EXIT_SUCCESS);
        }
    } catch (const char *error) {
        cerr << "Caught the error " << error << endl;
        if (ctx) fq_destroy(ctx);
        return EXIT_FAILURE;
    } catch (const string &error) {
        cerr << "Caught the error " << error << endl;
        if (ctx) fq_destroy(ctx);
        return EXIT_FAILURE;
    }
    return EXIT_SUCCESS;
}
