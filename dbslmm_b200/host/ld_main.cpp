// ld_main.cpp -- `ld` command line: the `plink --r2` table of SNP pairs within a window, computed on the GPU by
// dbslmm_b200_ld_pairs.  Users look at LD around a hit with it, and a clumping pass can read the pairs it has tested.
//
//   ld --bfile <prefix> --r2 [gz] [--ld-window N] [--ld-window-kb K] [--ld-window-r2 R] --out <prefix>
//
// PLINK 1.9's selection with its defaults (N = 10, K = 1000, R = 0.2): a pair (a, b) of .bim lines a < b of one chromosome
// is written when b - a <= N - 1, bp_b - bp_a <= 1000 K and r^2 >= R.  r is the project's (dbslmm_b200_ld_pairs): the
// Pearson r of the mean-imputed allele counts, which is the Pearson r of the allele counts when neither SNP has a missing
// call.  A variant with no called genotype or zero variance forms no pair but counts toward N.  A chromosome is a run of
// equal .bim column-1 tokens; it must be contiguous and its bp non-decreasing.
// Writes <out>.ld (or <out>.ld.gz with `gz`: concatenated gzip members, which gunzip and zlib read as one stream) with the
// header CHR_A BP_A SNP_A CHR_B BP_B SNP_B R2, single-space separated, R2 to 6 significant digits, and <out>.log.  The pairs
// arrive from the GPU in slices; each slice is formatted (and compressed) in chunks on the host worker pool and written in
// order while the GPU computes the next slice.  The .bed is mapped, never read whole.
#include <sys/mman.h>
#include <zlib.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <iostream>
#include <sstream>
#include <string>
#include <thread>
#include <vector>

#include "../csrc/hostpool.hpp"
#include "dbslmm_b200.h"
#include "plink_bed.hpp"

using namespace std;
using plink::Bim;

namespace {

[[noreturn]] void die(const string& msg, int code = 1) {
    cerr << "ERROR: " << msg << endl;
    exit(code);
}

void print_help() {
    cout << " ld --bfile <prefix> --r2 [gz] [--ld-window N] [--ld-window-kb K] [--ld-window-r2 R] --out <prefix>" << endl;
    cout << endl;
    cout << " --bfile        [prefix]  reference panel: <prefix>.bed (SNP-major), .bim, .fam." << endl;
    cout << " --r2 [gz]                write r^2 of the SNP pairs within the window (required); gz: <out>.ld.gz." << endl;
    cout << " --ld-window    [N]       pairs at most N - 1 variants apart (default 10, N >= 2)." << endl;
    cout << " --ld-window-kb [K]       pairs at most K kb apart (default 1000)." << endl;
    cout << " --ld-window-r2 [R]       pairs with r^2 >= R (default 0.2, 0 <= R <= 1)." << endl;
    cout << " --out          [prefix]  writes <out>.ld[.gz] and <out>.log." << endl;
}

double parse_num(const string& opt, const string& v) {
    char* e = nullptr;
    const double x = strtod(v.c_str(), &e);
    if (v.empty() || *e != '\0' || !std::isfinite(x)) die(opt + " needs a number, not '" + v + "'");
    return x;
}

struct Params {
    string bfile, out;
    bool r2 = false, gz = false;
    double window = 10, kb = 1000, r2_min = 0.2;
};

Params parse(int argc, char** argv) {
    Params p;
    auto value = [&](int& i, const string& a) -> string {
        if (i + 1 >= argc) die(a + " needs a value");
        return argv[++i];
    };
    for (int i = 1; i < argc; ++i) {
        const string a = argv[i];
        if (a == "--bfile") p.bfile = value(i, a);
        else if (a == "--out") p.out = value(i, a);
        else if (a == "--r2") {
            p.r2 = true;
            for (; i + 1 < argc && strncmp(argv[i + 1], "--", 2) != 0; ++i) {
                const string m = argv[i + 1];
                if (m == "gz") p.gz = true;
                else die("--r2 modifier '" + m + "' is not supported (ld writes the table of pairs, plain or gz; square, square0, "
                         "triangle, bin, bin4, dprime, with-freqs, inter-chr and the others are refused)");
            }
        } else if (a == "--ld-window") p.window = parse_num(a, value(i, a));
        else if (a == "--ld-window-kb") p.kb = parse_num(a, value(i, a));
        else if (a == "--ld-window-r2") p.r2_min = parse_num(a, value(i, a));
        else if (a == "--r") die("--r is not supported: ld writes r^2 (--r2)");
        else
            die("unsupported option '" + a + "' (ld takes --bfile, --r2 [gz], --ld-window, --ld-window-kb, --ld-window-r2 and --out; "
                "PLINK's --ld-snp, --ld-snp-list, --maf, --keep, --extract and the others are refused)");
    }
    if (p.bfile.empty()) die("--bfile is required");
    if (!p.r2) die("--r2 is required (ld writes the r^2 table only)");
    if (p.out.empty()) die("--out is required");
    if (p.window < 2 || p.window != std::floor(p.window) || p.window > 2147483647.0) die("--ld-window needs a whole number >= 2");
    if (p.kb < 0) die("--ld-window-kb needs a number >= 0");
    if (p.r2_min < 0 || p.r2_min > 1) die("--ld-window-r2 needs a number in [0, 1]");
    return p;
}

// One gzip member holding `in` (level 6, as gzip's default)
string gzip_member(const string& in) {
    z_stream z;
    memset(&z, 0, sizeof z);
    if (deflateInit2(&z, 6, Z_DEFLATED, 15 + 16, 8, Z_DEFAULT_STRATEGY) != Z_OK) die("zlib: deflateInit2 failed");
    string out(deflateBound(&z, (uLong)in.size()), '\0');
    z.next_in = (Bytef*)in.data();
    z.avail_in = (uInt)in.size();
    z.next_out = (Bytef*)&out[0];
    z.avail_out = (uInt)out.size();
    if (deflate(&z, Z_FINISH) != Z_STREAM_END) die("zlib: deflate failed");
    out.resize(z.total_out);
    deflateEnd(&z);
    return out;
}

double seconds_since(chrono::steady_clock::time_point t) { return chrono::duration<double>(chrono::steady_clock::now() - t).count(); }

struct Writer {
    const Bim* bim;
    bool gz;
    FILE* f;
    dbslmm::HostPool pool;
    double sink_s = 0, format_s = 0, gzip_s = 0;     // wall time in the sink; CPU time of the formatting and gzip tasks
    int64_t bytes = 0;
    static constexpr int64_t kChunk = 1 << 14;       // pairs per formatting task (and gzip member): a slice spreads over the pool

    int take(int64_t a0, int64_t a1, const int64_t* off, const int32_t* b, const double* r) {
        const auto t0 = chrono::steady_clock::now();
        const int64_t n = off[a1 - a0];
        const int64_t n_chunks = (n + kChunk - 1) / kChunk;
        vector<string> out((size_t)n_chunks);
        vector<double> fs((size_t)n_chunks), zs((size_t)n_chunks);
        dbslmm::TaskGroup g;
        for (int64_t c = 0; c < n_chunks; ++c) {
            pool.submit(g, [&, c]() {
                const auto tf = chrono::steady_clock::now();
                const int64_t p0 = c * kChunk, p1 = std::min(n, p0 + kChunk);
                int64_t a = a0 + (std::upper_bound(off, off + (a1 - a0) + 1, p0) - off) - 1;
                string& s = out[c];
                s.reserve((size_t)(p1 - p0) * 48);
                char buf[32];
                for (int64_t p = p0; p < p1; ++p) {
                    while (off[a + 1 - a0] <= p) ++a;
                    const int64_t bb = b[p];
                    snprintf(buf, sizeof buf, "%.6g", r[p] * r[p]);
                    s += bim->chr[a]; s += ' '; s += bim->bp_tok[a]; s += ' '; s += bim->snp[a]; s += ' ';
                    s += bim->chr[bb]; s += ' '; s += bim->bp_tok[bb]; s += ' '; s += bim->snp[bb]; s += ' ';
                    s += buf; s += '\n';
                }
                fs[c] = seconds_since(tf);
                if (gz) {
                    const auto tz = chrono::steady_clock::now();
                    s = gzip_member(s);
                    zs[c] = seconds_since(tz);
                }
            });
        }
        pool.wait(g);
        for (int64_t c = 0; c < n_chunks; ++c) {
            if (fwrite(out[c].data(), 1, out[c].size(), f) != out[c].size()) return 1;
            bytes += (int64_t)out[c].size();
            format_s += fs[c];
            gzip_s += zs[c];
        }
        sink_s += seconds_since(t0);
        return 0;
    }
};

int sink(void* user, int64_t a0, int64_t a1, const int64_t* off, const int32_t* b, const double* r) {
    return static_cast<Writer*>(user)->take(a0, a1, off, b, r);
}

}  // namespace

int main(int argc, char* argv[]) {
    if (argc <= 1 || (argc == 2 && (strcmp(argv[1], "-h") == 0 || strcmp(argv[1], "--help") == 0))) { print_help(); return EXIT_SUCCESS; }
    const auto t0 = chrono::steady_clock::now();
    const Params P = parse(argc, argv);
    ostringstream log;
    auto say = [&](const string& s) { cout << s << endl; log << s << "\n"; };
    {
        ostringstream o;
        o << "Options: --bfile " << P.bfile << " --r2" << (P.gz ? " gz" : "") << " --ld-window " << (int64_t)P.window << " --ld-window-kb "
          << P.kb << " --ld-window-r2 " << P.r2_min << " --out " << P.out;
        say(o.str());
    }

    // ---- panel
    int64_t n = 0;
    Bim bim;
    for (const string& err : {plink::count_fam(P.bfile + ".fam", n), plink::read_bim(P.bfile + ".bim", bim)})
        if (!err.empty()) die(err);
    const int64_t n_snp = (int64_t)bim.chr.size();
    if (n == 0) die(P.bfile + ".fam lists no individual");
    if (n > 409344) die(P.bfile + ".fam lists " + to_string(n) + " individuals; ld takes at most 409,344");
    if (n_snp == 0) die(P.bfile + ".bim lists no variant");
    if (n_snp > 2147483647) die(P.bfile + ".bim: too many variants");
    const string bed_path = P.bfile + ".bed";
    BedFile bedf;
    {
        const string err = open_bed(bed_path, n, n_snp, bedf);
        if (!err.empty()) die(err);
    }
    vector<int32_t> chr_off;
    vector<string> chr_name;
    {
        const string err = plink::bim_chromosomes(bim, P.bfile + ".bim", &bim.bp, "bp", chr_off, chr_name);
        if (!err.empty()) die(err);
    }
    say(to_string(n) + " individuals and " + to_string(n_snp) + " variants on " + to_string(chr_name.size()) + " chromosome(s) in " +
        P.bfile + ".bed/.bim/.fam");
    const string path = P.out + (P.gz ? ".ld.gz" : ".ld");
    Writer w;
    w.bim = &bim;
    w.gz = P.gz;
    w.f = fopen(path.c_str(), "wb");
    if (!w.f) die("cannot write " + path);
    // One thread per core, next to the library's own pool: the two overlap only while the library gathers the next segment's
    // .bed rows (memcpy of about 64 MB), a short share of a slice's formatting and gzip, which is what this pool is for.
    w.pool.start((int)std::max(1u, std::thread::hardware_concurrency()));
    const string head = "CHR_A BP_A SNP_A CHR_B BP_B SNP_B R2\n";
    const string head_out = P.gz ? gzip_member(head) : head;
    if (fwrite(head_out.data(), 1, head_out.size(), w.f) != head_out.size()) die("cannot write " + path);

    // ---- GPU
    void* map = mmap(nullptr, (size_t)bedf.size, PROT_READ, MAP_SHARED, bedf.fd, 0);
    if (map == MAP_FAILED) die("cannot map " + bed_path);
    close(bedf.fd);
    const uint8_t* payload = (const uint8_t*)map + 3;
    vector<int32_t> rows((size_t)n_snp);
    for (int64_t i = 0; i < n_snp; ++i) rows[i] = (int32_t)i;
    vector<uint8_t> usable((size_t)n_snp);
    int64_t n_pairs = 0, n_miss = 0;
    float ms = 0.0f;
    dbslmm_b200_handle* h = nullptr;
    if (dbslmm_b200_create(0, &h) != DBSLMM_B200_OK) die("cannot initialise the GPU (there is no CPU fallback)", 2);
    const auto tg = chrono::steady_clock::now();
    const int rc = dbslmm_b200_ld_pairs(h, payload, n_snp, (int32_t)n, rows.data(), n_snp, chr_off.data(), (int32_t)chr_name.size(),
                                        bim.bp.data(), (int32_t)P.window, 1000.0 * P.kb, P.r2_min, 0, sink, &w, usable.data(),
                                        &n_pairs, &n_miss, &ms);
    if (rc == DBSLMM_B200_ERR_SINK) die("cannot write " + path);
    if (rc != DBSLMM_B200_OK) die(string("ld: ") + dbslmm_b200_last_error(h), 2);
    const double call_s = seconds_since(tg);
    dbslmm_b200_destroy(h);
    munmap(map, (size_t)bedf.size);
    if (fclose(w.f) != 0) die("cannot write " + path);

    int64_t unusable = 0;
    for (uint8_t u : usable) unusable += u ? 0 : 1;
    {
        ostringstream o;
        o << n_pairs << " pairs written to " << path << "; " << unusable
          << " variant(s) with no called genotype or zero variance (no pair); " << n_miss << " pair(s) with a SNP with missing calls";
        say(o.str());
        ostringstream t;
        t << "GPU kernel time " << ms << " ms; ld_pairs call " << call_s << " s, of which sink " << w.sink_s << " s (formatting "
          << w.format_s << " s and gzip " << w.gzip_s << " s of CPU time on " << w.pool.size() << " threads), " << w.bytes
          << " bytes written; wall time " << seconds_since(t0) << " s";
        say(t.str());
    }
    ofstream lf((P.out + ".log").c_str());
    lf << log.str();
    return EXIT_SUCCESS;
}
