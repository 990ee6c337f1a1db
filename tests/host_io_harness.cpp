// Test harness for the command-line driver's host-side I/O (no GPU needed): the input Source (plain / gzip / blocked gzip,
// whole batches into a caller's buffer), the writers and fork_join, driven exactly as faqcs_cli.cpp drives them.
//   host_io_harness read   IN OUT BUFFER_KIB       fill buffers of that size until EOF, append what arrives to OUT
//   host_io_harness write  IN OUT                  IN -> BGZF in two write_bgzf calls + the end-of-file member
//   host_io_harness mapped IN OUT                  IN -> OUT in two write_mapped calls
//   host_io_harness pieces R1 R2 LIT LIST OUT      the pieces of LIST (lines "source offset length"; sources R1, R2, LIT) -> OUT
//                                                  in two write_pieces calls, the first with the first half of the list
//   host_io_harness fork_join N K KIND             on a Worker: fork_join(N) whose job K throws a const char * (KIND str) or
//                                                  std::bad_alloc (KIND bad_alloc); the other jobs count themselves
#define main faqcs_cli_main
#include "../faqcs_b200/host/faqcs_cli.cpp"
#undef main

#include <atomic>

static std::vector<uint8_t> slurp(const char *fn)
{
    FILE *f = fopen(fn, "rb");
    if (!f) throw "cannot open an input of the harness";
    std::vector<uint8_t> b;
    uint8_t chunk[1 << 16];
    for (size_t got; (got = fread(chunk, 1, sizeof(chunk), f)) > 0;) b.insert(b.end(), chunk, chunk + got);
    fclose(f);
    return b;
}

int main(int argc, char **argv)
{
    if (argc < 4) return 64;
    const std::string mode = argv[1];
    try {
        if (mode == "read") {
            Source s;
            if (!s.open(argv[2])) return 2;
            const bool was_pgzip = s.pgzip, was_bgzf = s.bgzf;
            const size_t cap = (size_t)atoi(argv[4]) << 10;
            std::vector<uint8_t> buf(cap);
            FILE *f = fopen(argv[3], "wb");
            size_t fills = 0, total_lines = 0;
            while (!s.eof) {
                size_t lines = 0;
                const size_t n = s.fill(buf.data(), 0, cap, &lines);
                if (count_newlines(buf.data(), n) != lines) { fprintf(stderr, "newline count mismatch\n"); return 3; }
                if (n == 0 && !s.eof) { fprintf(stderr, "no progress\n"); return 4; }
                fwrite(buf.data(), 1, n, f);
                total_lines += lines;
                ++fills;
            }
            fclose(f);
            printf("fills %zu lines %zu mode %s\n", fills, total_lines, was_pgzip ? "pgzip" : was_bgzf ? "bgzf" : s.gz ? "zlib" : "plain");
            return 0;
        }
        if (mode == "write" || mode == "mapped") {
            const std::vector<uint8_t> b = slurp(argv[2]);
            const size_t n = b.size(), cut = n / 3;
            const int fd = open_out(argv[3], "test output");
            if (mode == "write") {
                write_bgzf(fd, b.data(), cut);
                write_bgzf(fd, b.data() + cut, n - cut);
                close_bgzf(fd);
            } else {
                write_mapped(fd, b.data(), cut);
                write_mapped(fd, b.data() + cut, n - cut);
            }
            ::close(fd);
            return 0;
        }
        if (mode == "pieces" && argc == 7) {
            const std::vector<uint8_t> r1 = slurp(argv[2]), r2 = slurp(argv[3]), lit = slurp(argv[4]);
            const uint8_t *const src[3] = {r1.data(), r2.data(), lit.data()};
            std::vector<fq_out_piece> list;
            FILE *f = fopen(argv[5], "r");
            if (!f) return 2;
            unsigned long long s, o, l;
            while (fscanf(f, "%llu %llu %llu", &s, &o, &l) == 3) list.push_back(fq_out_piece{o, (uint32_t)l, (uint32_t)s});
            fclose(f);
            const int fd = open_out(argv[6], "test output");
            const size_t half = list.size() / 2;
            for (const auto &[k0, k1] : {std::make_pair((size_t)0, half), std::make_pair(half, list.size())}) {
                size_t total = 0;
                for (size_t k = k0; k < k1; ++k) total += list[k].length;
                write_pieces(fd, list.data() + k0, k1 - k0, src, total);
            }
            ::close(fd);
            return 0;
        }
        if (mode == "fork_join" && argc == 5) {
            const int n = atoi(argv[2]), k = atoi(argv[3]);
            const bool oom = std::string(argv[4]) == "bad_alloc";
            std::atomic<int> others{0};
            Worker w;
            w.post([&] {
                fork_join(n, [&](int i) {
                    if (i == k) {
                        if (oom) throw std::bad_alloc();
                        throw "job failed";
                    }
                    std::this_thread::sleep_for(std::chrono::milliseconds(20));      // still running when job k throws
                    ++others;
                });
            });
            try {
                w.wait_idle();
            } catch (const char *e) {
                fprintf(stderr, "error: %s (other jobs finished: %d)\n", e, others.load());
                return 5;
            }
            return 0;
        }
    } catch (const char *e) {
        fprintf(stderr, "error: %s\n", e);
        return 5;
    }
    return 64;
}
