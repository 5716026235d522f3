// `trew` command line: same subcommands, positionals, option names, defaults, validation messages and
// exit codes as the reference's main (src/trew.cpp:22-477), driving the B200 scan through the C ABI.
// -t / -m / -q are accepted and validated for compatibility but do not steer the GPU path (the consumers are GPUs,
// the host side always uses every core; the rotation table and the chunk queue do not exist here).
#include <algorithm>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <filesystem>
#include <iostream>
#include <string>
#include <vector>

#include "../../include/trew_b200.h"

namespace {

const char* kVersion = "0.5.0";

void usage(const std::string& cmd) {
    if (cmd == "long") {
        std::cerr << "Usage: long [--help] [--version] [--thread THREAD] [--table_max_mer TABLE_MAX_MER] [--low_baseline LOW_BASELINE] "
                     "[--high_baseline HIGH_BASELINE] [--slice_length SLICE_LENGTH] [--queue_size QUEUE_SIZE] [--read_hits READ_HITS] "
                     "MIN_MER MAX_MER LONG_FASTQ...\n\n"
                     "Estimate TRM from long-read sequencing data.\n";
    } else if (cmd == "short") {
        std::cerr << "Usage: short [--help] [--version] [--thread THREAD] [--paired_end] [--fq1 FASTQ_FRONT...] [--fq2 FASTQ_REVERSE...] "
                     "[--table_max_mer TABLE_MAX_MER] [--low_baseline LOW_BASELINE] [--high_baseline HIGH_BASELINE] "
                     "[--queue_size QUEUE_SIZE] [--read_hits READ_HITS] MIN_MER MAX_MER SHORT_FASTQ...\n\n"
                     "Estimate TRM from short-read sequencing data.\n";
    } else {
        std::cerr << "Usage: trew [--help] [--version] {long,short}\n\nSubcommands:\n"
                     "  long          Estimate TRM from long-read sequencing data.\n"
                     "  short         Estimate TRM from short-read sequencing data.\n";
    }
}

bool parse_int(const char* s, int* out) {
    char* end = nullptr;
    long v = strtol(s, &end, 10);
    if (end == s || *end) return false;
    *out = (int)v;
    return true;
}

bool parse_double(const char* s, double* out) {
    char* end = nullptr;
    double v = strtod(s, &end);
    if (end == s || *end) return false;
    *out = v;
    return true;
}

bool has_gz_ext(const std::filesystem::path& p) {  // src/trew.cpp:407, 422-433
    std::string e = p.extension().string();
    return e == ".gz" || e == ".bgz";
}

// --read_hits: one TSV line per unit record of a file -- file, record (0-based FASTQ record / pair index), table, k, the repeat
// unit as bases (the reference's 2-bit code T=0 G=1 C=2 A=3, first base in the most significant bits) and the count
void write_read_hits(FILE* out, const std::string& file, const trew_unit_record* r, uint64_t n) {
    static const char* kTable[6] = {"F_h", "F_l", "B_h", "B_l", "O_h", "O_l"};
    std::string unit;
    for (uint64_t i = 0; i < n; i++) {
        const int k = r[i].k;
        unit.resize((size_t)k);
        for (int j = 0; j < k; j++) {
            const int sh = 2 * (k - 1 - j);
            const uint64_t code = sh >= 64 ? (r[i].seq_hi >> (sh - 64)) & 3u : (r[i].seq_lo >> sh) & 3u;
            unit[(size_t)j] = "TGCA"[code];
        }
        fprintf(out, "%s\t%llu\t%s\t%d\t%s\t%u\n", file.c_str(), (unsigned long long)r[i].unit, kTable[r[i].table % 6], k, unit.c_str(),
                r[i].count);
    }
}

}  // namespace

int main(int argc, char** argv) {
    if (argc < 2) { usage(""); return 1; }
    std::string cmd = argv[1];
    if (cmd == "--version" || cmd == "-v") { std::cout << kVersion << "\n"; return 0; }
    if (cmd == "--help" || cmd == "-h") { usage(""); return 0; }
    if (cmd != "long" && cmd != "short") { usage(""); return 1; }
    const bool is_short = cmd == "short";

    int min_mer = 0, max_mer = 0, num_thread = 2, table_max_mer = 12, slice_length = 150, queue_size = -1;
    double low = 0.5, high = 0.8;
    bool paired = false, used_fq1 = false, used_fq2 = false;
    const char* read_hits = nullptr;
    std::vector<std::string> positional, fq1, fq2;
    std::vector<std::string>* sink = &positional;
    // argparse also takes `--name=value` and a value glued to a short option (`-t4`): split those first
    std::vector<std::string> av;
    for (int i = 2; i < argc; i++) {
        std::string a = argv[i];
        size_t eq;
        if (a.size() > 2 && a[0] == '-' && a[1] == '-' && (eq = a.find('=')) != std::string::npos) {
            av.push_back(a.substr(0, eq)); av.push_back(a.substr(eq + 1));
        } else if (a.size() > 2 && a[0] == '-' && strchr("tmLHsq", a[1]) && ((a[2] >= '0' && a[2] <= '9') || a[2] == '.' || a[2] == '-')) {
            av.push_back(a.substr(0, 2)); av.push_back(a.substr(2));
        } else av.push_back(a);
    }
    const int ac = (int)av.size();
    for (int i = 0; i < ac; i++) {
        const std::string& a = av[(size_t)i];
        auto value = [&](const char** v) { if (i + 1 >= ac) return false; *v = av[(size_t)++i].c_str(); return true; };
        const char* v = nullptr;
        bool ok = true;
        if (a == "-h" || a == "--help") { usage(cmd); return 0; }
        else if (a == "-t" || a == "--thread") { ok = value(&v) && parse_int(v, &num_thread); sink = &positional; }
        else if (a == "-m" || a == "--table_max_mer") { ok = value(&v) && parse_int(v, &table_max_mer); sink = &positional; }
        else if (a == "-L" || a == "--low_baseline") { ok = value(&v) && parse_double(v, &low); sink = &positional; }
        else if (a == "-H" || a == "--high_baseline") { ok = value(&v) && parse_double(v, &high); sink = &positional; }
        else if (!is_short && (a == "-s" || a == "--slice_length")) { ok = value(&v) && parse_int(v, &slice_length); sink = &positional; }
        else if (a == "-q" || a == "--queue_size") { ok = value(&v) && parse_int(v, &queue_size); sink = &positional; }
        else if (is_short && a == "--paired_end") { paired = true; sink = &positional; }
        else if (a == "--read_hits") { ok = value(&read_hits); sink = &positional; }
        else if (is_short && a == "--fq1") { used_fq1 = true; sink = &fq1; }
        else if (is_short && a == "--fq2") { used_fq2 = true; sink = &fq2; }
        else if (a.size() > 1 && a[0] == '-' && !(a[1] >= '0' && a[1] <= '9')) ok = false;
        else sink->push_back(a);
        if (!ok) { usage(cmd); return 1; }
    }
    if (positional.size() < 2 || !parse_int(positional[0].c_str(), &min_mer) || !parse_int(positional[1].c_str(), &max_mer)) {
        usage(cmd);
        return 1;
    }
    std::vector<std::string> files(positional.begin() + 2, positional.end());
    if (!is_short && files.empty()) { usage(cmd); return 1; }

    // argument checks, same order and messages as src/trew.cpp:174-228 / 255-304
    auto bad = [&](const char* msg) { fputs(msg, stderr); usage(cmd); return 1; };
    if (min_mer > max_mer) return bad("MIN_MER must not be greater than MAX_MER.\n");
    if (min_mer < 3) return bad("MIN_MER must be greater than or equal to 3.\n");
    if (max_mer > 64) return bad("MAX_MER must be less than or equal to 64.\n");
    if (table_max_mer > 15) return bad("TABLE_MAX_MER must be less than or equal to 15.\n");
    if (!is_short && slice_length < 2 * max_mer) return bad("SLICE_LENGTH must be greater than or equal to twice of MAX_MER.\n");
    if (queue_size != -1 && queue_size < 4) return bad("QUEUE_SIZE must be -1 (unlimited) or greater than or equal to 4.\n");
    if (table_max_mer <= 0) return bad("TABLE_MAX_MER must be positive.\n");
    if (num_thread <= 0) return bad("number of threads must be positive.\n");
    if (!(0 < low && low <= 1) || !(0 < high && high <= 1)) return bad("Baseline must be in range 0 to 1.\n");
    if (low > high) return bad("Low baseline must be smaller than high baseline.\n");
    if (num_thread < 2) return bad("You must use at least two threads.\n");

    std::vector<std::filesystem::path> paths;
    if (is_short && paired) {
        if (!files.empty()) return bad("SHORT_FASTQ must not be provided when --IS_PAIRED_END is used.\n");
        if (!used_fq1 || !used_fq2) return bad("--fq1 and --fq2 are required in paired-end mode.\n");
        if (fq1.size() != fq2.size()) return bad("--fq1 and --fq2 must have the same number of files.\n");
        for (size_t i = 0; i < fq1.size(); i++) {
            if (!std::filesystem::is_regular_file(fq1[i])) { std::cerr << fq1[i] << " : file not found\n"; usage(cmd); return 1; }
            if (!std::filesystem::is_regular_file(fq2[i])) { std::cerr << fq2[i] << " : file not found\n"; usage(cmd); return 1; }
            paths.emplace_back(fq1[i]);
            paths.emplace_back(fq2[i]);
        }
    } else {
        if (is_short && files.empty()) return bad("SHORT_FASTQ is required in single-end mode.\n");
        if (is_short && (used_fq1 || used_fq2)) return bad("--fq1 and --fq2 should not be used in single-end mode.\n");
        for (auto& f : files) {
            if (!std::filesystem::is_regular_file(f)) {
                if (is_short) { std::cerr << f << " : file not found\n"; usage(cmd); }
                else fprintf(stderr, "%s : file not found\n", f.c_str());
                return 1;
            }
            paths.emplace_back(f);
        }
    }

    trew_config cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.mode = is_short ? (paired ? TREW_MODE_PAIR : TREW_MODE_SHORT) : TREW_MODE_LONG;
    cfg.min_mer = min_mer; cfg.max_mer = max_mer; cfg.slice_length = slice_length;
    cfg.low_baseline = low; cfg.high_baseline = high;
    // -t sized the reference's consumer pool; the consumers are GPUs here, and the host side (FASTQ index, packer,
    // BGZF inflate) always uses every core: a reference command line with the default -t 2 must not throttle it.
    cfg.host_threads = 0;
    // Which GPUs: TREW_DEVICES = "all", a count, or a comma list of ordinals; TREW_DEVICE = one ordinal.  By default
    // every visible GPU takes part once the input is large enough to feed more than one (512 MiB), else device 0.
    std::vector<int32_t> devices;
    {
        const char* list = getenv("TREW_DEVICES");
        const char* one = getenv("TREW_DEVICE");
        uintmax_t input_bytes = 0;
        for (auto& p : paths) { std::error_code ec; uintmax_t sz = std::filesystem::file_size(p, ec); if (!ec) input_bytes += sz; }
        if (list && *list && strcmp(list, "all") != 0) {
            if (strchr(list, ',')) { for (const char* q = list; q && *q; q = strchr(q, ',') ? strchr(q, ',') + 1 : nullptr) devices.push_back(atoi(q)); }
            else { int n = atoi(list); for (int i = 0; i < n; i++) devices.push_back(i); }
        } else if (!(list && *list)) {
            if (one && *one) devices.push_back(atoi(one));
            else if (input_bytes < ((uintmax_t)512 << 20)) devices.push_back(0);
        }   // empty list = all visible devices
    }
    // Only the chosen devices are made visible to the CUDA runtime (unless the caller set CUDA_VISIBLE_DEVICES already):
    // initialising the driver takes time per visible GPU, and a small input that runs on one GPU of an eight-GPU box
    // should not pay for the other seven.
    if (!devices.empty() && !getenv("CUDA_VISIBLE_DEVICES")) {
        std::vector<int32_t> uniq;
        for (int32_t d : devices) if (std::find(uniq.begin(), uniq.end(), d) == uniq.end()) uniq.push_back(d);
        std::string vis;
        for (size_t i = 0; i < uniq.size(); i++) vis += (i ? "," : "") + std::to_string(uniq[i]);
        setenv("CUDA_VISIBLE_DEVICES", vis.c_str(), 1);
        for (int32_t& d : devices) d = (int32_t)(std::find(uniq.begin(), uniq.end(), d) - uniq.begin());
    }
    // TREW_CLI_TIMING=1: wall-clock of the phases on stderr
    const bool timing = getenv("TREW_CLI_TIMING") != nullptr;
    auto now = [] { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    const double t_start = now();
    trew_multi* ctx = nullptr;
    int rc = trew_multi_create(&cfg, devices.empty() ? nullptr : devices.data(), (int32_t)devices.size(), &ctx);
    if (rc != TREW_OK) {
        const char* why = trew_multi_last_error(nullptr);
        fprintf(stderr, "trew: cannot create device context: %s\n", why && *why ? why : trew_status_string(rc));
        return 1;
    }
    // One input (file or pair): only rows that can reach the report leave the device (see trew_dev_set_report_filter);
    // with several inputs every entry is needed, small counts add up across files (src/trew.cpp:454-467).
    if (paths.size() == (cfg.mode == TREW_MODE_PAIR ? 2u : 1u) && !getenv("TREW_FULL_TABLES")) trew_multi_set_report_filter(ctx, 10);
    if (timing) fprintf(stderr, "[trew] contexts on %d device(s): %.1f ms\n", trew_multi_device_count(ctx), now() - t_start);
    trew_report* rep = nullptr;
    trew_report_create(min_mer, &rep);
    // --read_hits: unit records, sized from the input (a file that needs more is scanned again with what it needed)
    FILE* hits = nullptr;
    uint64_t rec_cap = 0;
    if (read_hits) {
        hits = fopen(read_hits, "w");
        if (!hits) { fprintf(stderr, "%s : cannot open for writing\n", read_hits); trew_report_destroy(rep); trew_multi_destroy(ctx); return 1; }
        uintmax_t input_bytes = 0;
        for (auto& p : paths) { std::error_code ec; uintmax_t sz = std::filesystem::file_size(p, ec); if (!ec) input_bytes += has_gz_ext(p) ? 4 * sz : sz; }
        rec_cap = std::min<uint64_t>(std::max<uint64_t>(input_bytes / 128, 1u << 12), 1u << 26);   // 2.4 per 150-base FASTQ record
        trew_multi_enable_unit_records(ctx, rec_cap);
    }

    const bool is_pair = cfg.mode == TREW_MODE_PAIR;
    size_t printed = 0;   // bytes of the report text already written to stdout
    for (size_t i = 0; i < paths.size() / (is_pair ? 2 : 1); i++) {
        std::string a, b;
        bool g1, g2 = false;
        if (is_pair) {
            a = std::filesystem::canonical(paths[2 * i]).string(); b = std::filesystem::canonical(paths[2 * i + 1]).string();
            g1 = has_gz_ext(paths[2 * i]); g2 = has_gz_ext(paths[2 * i + 1]);
        } else {
            a = std::filesystem::canonical(paths[i]).string();
            g1 = has_gz_ext(paths[i]);
        }
        const double t_file = now();
        trew_multi_reset(ctx);
        rc = trew_multi_process_file(ctx, a.c_str(), g1, is_pair ? b.c_str() : nullptr, g2);
        const trew_entry* entries = nullptr;
        uint64_t n = 0;
        const double t_scanned = now();
        if (rc == TREW_OK) rc = trew_multi_finish(ctx, &entries, &n);
        if (timing) fprintf(stderr, "[trew] %s: read + scan %.1f ms, tables %.1f ms\n", a.c_str(), t_scanned - t_file, now() - t_scanned);
        if (rc != TREW_OK) {
            fprintf(stderr, "%s\n", trew_multi_last_error(ctx));  // the reference prints and exit(EXIT_FAILURE)s
            trew_report_destroy(rep);
            trew_multi_destroy(ctx);
            return 1;
        }
        trew_report_add_file(rep, a.c_str(), entries, n);
        if (hits) {
            const trew_unit_record* recs = nullptr;
            uint64_t nr = 0;
            rc = trew_multi_unit_records(ctx, &recs, &nr);
            unsigned long long need = 0;
            const char* why = trew_multi_last_error(ctx);
            const char* at = rc == TREW_ERR_TABLE_FULL && why ? strstr(why, "a capacity of ") : nullptr;
            if (at && sscanf(at, "a capacity of %llu", &need) == 1) {   // once more, with the capacity that is enough
                rec_cap = need;
                rc = trew_multi_reset(ctx);
                if (rc == TREW_OK) rc = trew_multi_enable_unit_records(ctx, rec_cap);
                if (rc == TREW_OK) rc = trew_multi_process_file(ctx, a.c_str(), g1, is_pair ? b.c_str() : nullptr, g2);
                if (rc == TREW_OK) rc = trew_multi_unit_records(ctx, &recs, &nr);
            }
            if (rc != TREW_OK) {
                fprintf(stderr, "%s\n", trew_multi_last_error(ctx));
                fclose(hits);
                trew_report_destroy(rep);
                trew_multi_destroy(ctx);
                return 1;
            }
            write_read_hits(hits, a, recs, nr);
            fflush(hits);
        }
        // each file's sections go out as soon as they are ready, like process_output prints them (src/kmer.cpp:1615-1631):
        // a later file that fails leaves the earlier sections on stdout
        const char* part = nullptr;
        size_t part_len = 0;
        trew_report_text(rep, &part, &part_len);
        fwrite(part + printed, 1, part_len - printed, stdout);
        fflush(stdout);
        printed = part_len;
    }
    const char* text = nullptr;
    size_t len = 0;
    trew_report_finish(rep, &text, &len);
    fwrite(text + printed, 1, len - printed, stdout);
    trew_report_destroy(rep);
    if (hits) fclose(hits);
    const double t_done = now();
    trew_multi_destroy(ctx);
    if (timing) fprintf(stderr, "[trew] report %.1f ms after the last file, teardown %.1f ms, total %.1f ms\n", t_done - t_start, now() - t_done, now() - t_start);
    return 0;
}
