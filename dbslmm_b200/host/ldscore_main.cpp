// ldscore_main.cpp -- `ldscore` command line: the `ldsc.py --bfile <panel> --l2` step that makes the LD Scores LDSC needs
// for the heritability (-h) and SNP count (-nsnp) DBSLMM's driver reads from an LDSC log (DBSLMM_script.sh:63-64).
//
//   ldscore --bfile <prefix> --l2 (--ld-wind-cm X | --ld-wind-kb X | --ld-wind-snps N) [--maf X] [--print-snps FILE]
//           [--annot FILE [--thin-annot]] [--yes-really] --out <prefix>
//
// Semantics restated from ldsc 1.0.1 (ldscore.py / ldsc.py), computed by dbslmm_b200_ldscore: SNPs with MAF <= --maf (default
// 0) or without a homozygous call are dropped; r^2 is bias-corrected, r^2 - (1 - r^2) / (n - 2), and summed over a symmetric
// window of cM (.bim column 3), kb (column 4) or SNPs.  One deliberate difference: windows never cross a chromosome (ldsc
// would pair SNPs of different chromosomes by raw coordinates).  A chromosome is a run of equal .bim column-1 tokens; it must
// be contiguous and its window coordinates non-decreasing.  As ldsc does, a chromosome whose last kept SNP's window reaches
// its first kept SNP is refused without --yes-really: the kept SNPs decide it, so the statistics pass runs first on its own
// and the LD pass only if no chromosome is refused.
// Writes <out>.l2.ldscore.gz (CHR SNP BP L2, tab-separated, L2 as %.3f), <out>.l2.M, <out>.l2.M_5_50 and <out>.log -- the
// file set `ldsc.py --ref-ld <out> --w-ld <out>` reads.  The .bed is mapped, never read whole.
// --annot FILE (plain or gzip; ldsc's .annot[.gz]) gives partitioned LD Scores, one column per annotation, computed by
// dbslmm_b200_ldscore_annot: a header CHR BP SNP CM <names...> (--thin-annot: the names only) and one row per .bim line,
// whose SNP column must equal the .bim's.  The .ldscore.gz then holds <name>L2 per annotation (plain L2 for a single one)
// and .l2.M / .l2.M_5_50 the sum of each annotation over the kept SNPs (with MAF > 0.05), tab-separated.
#include <sys/mman.h>
#include <zlib.h>

#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <iostream>
#include <sstream>
#include <string>
#include <unordered_map>
#include <unordered_set>
#include <vector>

#include "dbslmm_b200.h"
#include "plink_bed.hpp"

using namespace std;
using plink::Bim;
using plink::bim_chromosomes;
using plink::count_fam;
using plink::read_bim;
using plink::split_ws;

namespace {

[[noreturn]] void die(const string& msg, int code = 1) {
    cerr << "ERROR: " << msg << endl;
    exit(code);
}

void print_header() {
    cout << endl;
    cout << "*************************************************************" << endl;
    cout << "  LD Scores of a PLINK fileset (ldscore), B200 build" << endl;
    cout << "  Type ./ldscore -h for detailed help" << endl;
    cout << "*************************************************************" << endl;
    cout << endl;
}

void print_help() {
    cout << " ldscore --bfile <prefix> --l2 (--ld-wind-cm X | --ld-wind-kb X | --ld-wind-snps N) [--maf X]" << endl;
    cout << "         [--print-snps FILE] [--annot FILE [--thin-annot]] [--yes-really] --out <prefix>" << endl;
    cout << endl;
    cout << " --bfile        [prefix]  reference panel: <prefix>.bed (SNP-major), .bim, .fam." << endl;
    cout << " --l2                     compute LD Scores (required)." << endl;
    cout << " --ld-wind-cm   [X]       window of X cM (.bim column 3); exactly one window option is required." << endl;
    cout << " --ld-wind-kb   [X]       window of X kb (.bim column 4)." << endl;
    cout << " --ld-wind-snps [N]       window of N kept SNPs on each side." << endl;
    cout << " --maf          [X]       drop SNPs with MAF <= X (default 0)." << endl;
    cout << " --print-snps   [FILE]    write only the SNPs listed in the first column of FILE (the counts cover all)." << endl;
    cout << " --annot        [FILE]    partitioned LD Scores: ldsc's .annot file (plain or gzip), one row per .bim line," << endl;
    cout << "                          header CHR BP SNP CM <names...>; one LD Score column per annotation." << endl;
    cout << " --thin-annot             the --annot file has no CHR BP SNP CM columns: its header holds the names only." << endl;
    cout << " --yes-really             allow a window that spans a whole chromosome." << endl;
    cout << " --out          [prefix]  writes <out>.l2.ldscore.gz, <out>.l2.M, <out>.l2.M_5_50 and <out>.log." << endl;
}

double parse_num(const string& opt, const string& v) {
    char* e = nullptr;
    const double x = strtod(v.c_str(), &e);
    if (v.empty() || *e != '\0' || !std::isfinite(x) || x < 0) die(opt + " needs a number >= 0, not '" + v + "'");
    return x;
}

struct Params {
    string bfile, out, print_snps, annot;
    bool l2 = false, yes_really = false, thin_annot = false;
    int n_wind = 0;
    int kind = 0;                 // 0 cM, 1 kb, 2 SNPs
    double wind = 0.0, maf = 0.0;
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
        else if (a == "--l2") p.l2 = true;
        else if (a == "--yes-really") p.yes_really = true;
        else if (a == "--print-snps") p.print_snps = value(i, a);
        else if (a == "--annot") p.annot = value(i, a);
        else if (a == "--thin-annot") p.thin_annot = true;
        else if (a == "--maf") {
            p.maf = parse_num(a, value(i, a));
            if (p.maf >= 0.5) die("--maf must be below 0.5");
        } else if (a == "--ld-wind-cm" || a == "--ld-wind-kb" || a == "--ld-wind-snps") {
            ++p.n_wind;
            p.kind = a == "--ld-wind-cm" ? 0 : a == "--ld-wind-kb" ? 1 : 2;
            p.wind = parse_num(a, value(i, a));
            if (p.kind == 2 && (p.wind != std::floor(p.wind) || p.wind > 2147483647.0)) die("--ld-wind-snps needs a whole number");
        } else {
            die("unsupported option '" + a + "' (ldscore takes --bfile, --l2, --ld-wind-cm/--ld-wind-kb/--ld-wind-snps, --maf, "
                "--print-snps, --annot, --thin-annot, --yes-really and --out; ldsc's --cts-bin, --keep, --extract, --per-allele, "
                "--pq-exp, --chunk-size and the others are refused)");
        }
    }
    if (p.bfile.empty()) die("--bfile is required");
    if (!p.l2) die("--l2 is required (ldscore computes LD Scores only)");
    if (p.n_wind != 1) die("exactly one of --ld-wind-cm, --ld-wind-kb and --ld-wind-snps is required");
    if (p.out.empty()) die("--out is required");
    if (p.thin_annot && p.annot.empty()) die("--thin-annot needs --annot");
    return p;
}

// ldsc's .annot[.gz]: names and a row-major [n_snp][C] matrix; the SNP column (full format) must match the .bim's
struct Annot { vector<string> names; vector<double> a; };

Annot read_annot(const string& path, bool thin, const vector<string>& bim_snp) {
    gzFile f = gzopen(path.c_str(), "rb");                 // reads plain files as they are
    if (!f) die("'--annot' file " + path + " does not exist or cannot be read");
    auto line = [&](string& out) {
        out.clear();
        char buf[1 << 16];
        while (gzgets(f, buf, sizeof buf)) {
            out += buf;
            if (!out.empty() && out.back() == '\n') return true;
        }
        int err = 0;
        gzerror(f, &err);
        if (err != Z_OK && err != Z_STREAM_END) die("cannot read the '--annot' file " + path);
        return !out.empty();
    };
    Annot A;
    string ln;
    size_t no = 0;
    vector<string> t;
    while (line(ln)) { ++no; t = split_ws(ln); if (!t.empty()) break; }
    const size_t skip = thin ? 0 : 4;
    if (t.size() <= skip)
        die(path + ": no annotation columns (the header " + string(thin ? "lists no name" : "needs CHR BP SNP CM and one name or more") + ")");
    A.names.assign(t.begin() + skip, t.end());
    const size_t C = A.names.size();
    if (C > (size_t)DBSLMM_B200_LD_MAX_ANNOT)
        die(path + ": " + to_string(C) + " annotations; ldscore takes at most " + to_string(DBSLMM_B200_LD_MAX_ANNOT));
    A.a.reserve(bim_snp.size() * C);
    size_t row = 0;
    while (line(ln)) {
        ++no;
        t = split_ws(ln);
        if (t.empty()) continue;
        if (t.size() != skip + C)
            die(path + " line " + to_string(no) + ": " + to_string(t.size()) + " columns, the header has " + to_string(skip + C));
        if (row >= bim_snp.size()) die(path + " has more rows than the .bim has variants (" + to_string(bim_snp.size()) + ")");
        if (!thin && t[2] != bim_snp[row])
            die(path + " line " + to_string(no) + ": SNP " + t[2] + " is not " + bim_snp[row] + ", line " + to_string(row + 1) +
                " of the .bim (the rows must list the .bim's SNPs in its order)");
        for (size_t c = 0; c < C; ++c) {
            const string& v = t[skip + c];
            char* e = nullptr;
            const double x = strtod(v.c_str(), &e);
            if (v.empty() || *e != '\0' || !std::isfinite(x))
                die(path + " line " + to_string(no) + ": '" + v + "' (annotation " + A.names[c] + ") is not a finite number");
            A.a.push_back(x);
        }
        ++row;
    }
    gzclose(f);
    if (row != bim_snp.size())
        die(path + " has " + to_string(row) + " rows; the .bim has " + to_string(bim_snp.size()) + " variants");
    return A;
}

// a value of .l2.M / .l2.M_5_50: whole numbers as integers (ldsc's 0/1 annotations), others with every digit
string format_m(double x) {
    char b[64];
    if (x == std::floor(x) && std::fabs(x) < 9.0e15) snprintf(b, sizeof b, "%lld", (long long)x);
    else snprintf(b, sizeof b, "%.17g", x);
    return b;
}

}  // namespace

int main(int argc, char* argv[]) {
    if (argc <= 1) { print_header(); return EXIT_SUCCESS; }
    if (argc == 2 && (strcmp(argv[1], "-h") == 0 || strcmp(argv[1], "--help") == 0)) { print_help(); return EXIT_SUCCESS; }
    const auto t0 = chrono::steady_clock::now();
    const Params P = parse(argc, argv);
    ostringstream log;
    auto say = [&](const string& s) { cout << s << endl; log << s << "\n"; };
    static const char* kWind[3] = {"--ld-wind-cm", "--ld-wind-kb", "--ld-wind-snps"};
    {
        ostringstream o;
        o << "Options: --bfile " << P.bfile << " --l2 " << kWind[P.kind] << " " << P.wind << " --maf " << P.maf;
        if (!P.print_snps.empty()) o << " --print-snps " << P.print_snps;
        if (!P.annot.empty()) o << " --annot " << P.annot << (P.thin_annot ? " --thin-annot" : "");
        if (P.yes_really) o << " --yes-really";
        o << " --out " << P.out;
        say(o.str());
    }

    // ---- panel
    int64_t n = 0;
    Bim bim;
    for (const string& err : {count_fam(P.bfile + ".fam", n), read_bim(P.bfile + ".bim", bim)})
        if (!err.empty()) die(err);
    const int64_t n_snp = (int64_t)bim.chr.size();
    if (n == 0) die(P.bfile + ".fam lists no individual");
    if (n > 409344) die(P.bfile + ".fam lists " + to_string(n) + " individuals; ldscore takes at most 409,344");
    if (n_snp == 0) die(P.bfile + ".bim lists no variant");
    if (n_snp > 2147483647) die(P.bfile + ".bim: too many variants");
    const string bed_path = P.bfile + ".bed";
    BedFile bedf;
    {
        const string err = open_bed(bed_path, n, n_snp, bedf);
        if (!err.empty()) die(err);
    }
    say(to_string(n) + " individuals and " + to_string(n_snp) + " variants in " + P.bfile + ".bed/.bim/.fam");

    // ---- chromosomes: contiguous runs, coordinates of the window's kind non-decreasing
    vector<int32_t> chr_off;
    vector<string> chr_name;
    const vector<double>* cx = P.kind == 0 ? &bim.cm : P.kind == 1 ? &bim.bp : nullptr;
    {
        const string err = bim_chromosomes(bim, P.bfile + ".bim", cx, P.kind == 0 ? "cM" : "bp", chr_off, chr_name);
        if (!err.empty()) die(err);
    }
    unordered_set<string> print_ids;
    if (!P.print_snps.empty()) {
        ifstream f(P.print_snps.c_str());
        if (!f) die(P.print_snps + " does not exist");
        string line;
        while (getline(f, line)) {
            const vector<string> t = split_ws(line);
            if (!t.empty()) print_ids.insert(t[0]);
        }
        bool any = false;
        for (const string& v : bim.snp) any = any || print_ids.count(v);
        if (!any) die("no SNP of " + P.print_snps + " is in " + P.bfile + ".bim");
    }

    Annot annot;
    if (!P.annot.empty()) {
        annot = read_annot(P.annot, P.thin_annot, bim.snp);
        say("read " + to_string(annot.names.size()) + " annotation(s) for " + to_string(n_snp) + " SNPs from " + P.annot);
    }
    const int64_t C = annot.names.empty() ? 1 : (int64_t)annot.names.size();

    // ---- GPU
    void* map = mmap(nullptr, (size_t)bedf.size, PROT_READ, MAP_SHARED, bedf.fd, 0);
    if (map == MAP_FAILED) die("cannot map " + bed_path);
    close(bedf.fd);
    const uint8_t* payload = (const uint8_t*)map + 3;
    vector<int32_t> rows((size_t)n_snp);
    for (int64_t i = 0; i < n_snp; ++i) rows[i] = (int32_t)i;
    vector<double> coord;
    if (cx) coord = *cx;
    const double max_dist = P.kind == 1 ? 1000.0 * P.wind : P.wind;
    const int32_t n_chr = (int32_t)chr_name.size();
    vector<uint8_t> kept((size_t)n_snp);
    vector<double> maf((size_t)n_snp), l2((size_t)(n_snp * C));
    vector<int32_t> guard((size_t)n_chr);
    float ms = 0.0f;
    dbslmm_b200_handle* h = nullptr;
    if (dbslmm_b200_create(0, &h) != DBSLMM_B200_OK) die("cannot initialise the GPU (there is no CPU fallback)", 2);
    // without --yes-really, the statistics pass alone first (l2 NULL): the kept SNPs decide the guard, and a refused
    // chromosome must not cost the LD pass (nor fail it for want of device memory)
    for (int full = P.yes_really ? 1 : 0; full < 2; ++full) {
        const int32_t wk = cx ? DBSLMM_B200_LD_WIND_COORD : DBSLMM_B200_LD_WIND_SNPS;
        const int rc = annot.names.empty()
            ? dbslmm_b200_ldscore(h, payload, n_snp, (int32_t)n, rows.data(), n_snp, chr_off.data(), n_chr, wk, cx ? coord.data() : nullptr,
                                  max_dist, P.maf, 0, kept.data(), maf.data(), full ? l2.data() : nullptr, guard.data(), &ms)
            : dbslmm_b200_ldscore_annot(h, payload, n_snp, (int32_t)n, rows.data(), n_snp, chr_off.data(), n_chr, wk,
                                        cx ? coord.data() : nullptr, max_dist, P.maf, 0, annot.a.data(), (int32_t)C, kept.data(),
                                        maf.data(), full ? l2.data() : nullptr, guard.data(), &ms);
        if (rc != DBSLMM_B200_OK) die(string("ldscore: ") + dbslmm_b200_last_error(h), 2);
        for (int32_t c = 0; c < n_chr && !P.yes_really; ++c)
            if (guard[c])
                die("the window of the last kept SNP of chromosome " + chr_name[c] + " reaches its first kept SNP: do you really want "
                    "whole-chromosome LD Scores? (--yes-really)");
    }
    dbslmm_b200_destroy(h);
    munmap(map, (size_t)bedf.size);

    // ---- <out>.l2.ldscore.gz, <out>.l2.M, <out>.l2.M_5_50
    int64_t m_all = 0, m_5_50 = 0, printed = 0;
    for (int64_t i = 0; i < n_snp; ++i)
        if (kept[i]) {
            ++m_all;
            if (maf[i] > 0.05) ++m_5_50;
            if (print_ids.empty() || print_ids.count(bim.snp[i])) ++printed;
        }
    if (m_all == 0) die("no SNP is kept (--maf " + to_string(P.maf) + ")");
    if (printed == 0) die("none of the SNPs of " + P.print_snps + " is kept");
    const string gz = P.out + ".l2.ldscore.gz";
    gzFile f = gzopen(gz.c_str(), "wb");
    if (!f) die("cannot write " + gz);
    if (annot.names.empty()) {
        gzputs(f, "CHR\tSNP\tBP\tL2\n");
        for (int64_t i = 0; i < n_snp; ++i) {
            if (!kept[i] || (!print_ids.empty() && !print_ids.count(bim.snp[i]))) continue;
            if (gzprintf(f, "%s\t%s\t%s\t%.3f\n", bim.chr[i].c_str(), bim.snp[i].c_str(), bim.bp_tok[i].c_str(), l2[i]) <= 0) die("cannot write " + gz);
        }
        if (gzclose(f) != Z_OK) die("cannot write " + gz);
        for (const auto& mf : {make_pair(P.out + ".l2.M", m_all), make_pair(P.out + ".l2.M_5_50", m_5_50)}) {
            FILE* o = fopen(mf.first.c_str(), "w");
            if (!o || fprintf(o, "%lld\n", (long long)mf.second) < 0 || fclose(o) != 0) die("cannot write " + mf.first);
        }
    } else {
        string head = "CHR\tSNP\tBP";
        for (const string& v : annot.names) head += "\t" + (C == 1 ? string() : v) + "L2";
        gzputs(f, (head + "\n").c_str());
        string row;
        char b[64];
        for (int64_t i = 0; i < n_snp; ++i) {
            if (!kept[i] || (!print_ids.empty() && !print_ids.count(bim.snp[i]))) continue;
            row = bim.chr[i] + "\t" + bim.snp[i] + "\t" + bim.bp_tok[i];
            for (int64_t c = 0; c < C; ++c) { snprintf(b, sizeof b, "\t%.3f", l2[i * C + c]); row += b; }
            row += "\n";
            if (gzwrite(f, row.data(), (unsigned)row.size()) != (int)row.size()) die("cannot write " + gz);
        }
        if (gzclose(f) != Z_OK) die("cannot write " + gz);
        // sum of each annotation over the kept SNPs (and those with MAF > 0.05), in .bim order
        vector<double> s_all((size_t)C, 0.0), s_550((size_t)C, 0.0);
        for (int64_t i = 0; i < n_snp; ++i)
            for (int64_t c = 0; kept[i] && c < C; ++c) {
                s_all[c] += annot.a[i * C + c];
                if (maf[i] > 0.05) s_550[c] += annot.a[i * C + c];
            }
        for (const auto& mf : {make_pair(P.out + ".l2.M", &s_all), make_pair(P.out + ".l2.M_5_50", &s_550)}) {
            string txt;
            for (int64_t c = 0; c < C; ++c) txt += (c ? "\t" : "") + format_m((*mf.second)[c]);
            FILE* o = fopen(mf.first.c_str(), "w");
            if (!o || fprintf(o, "%s\n", txt.c_str()) < 0 || fclose(o) != 0) die("cannot write " + mf.first);
        }
    }
    {
        ostringstream o;
        o << m_all << " SNPs kept (" << m_5_50 << " with MAF > 0.05) on " << n_chr << " chromosome(s); " << printed
          << " written to " << gz;
        say(o.str());
        ostringstream t;
        t << "GPU kernel time " << ms << " ms; wall time " << chrono::duration<double>(chrono::steady_clock::now() - t0).count() << " s";
        say(t.str());
    }
    ofstream lf((P.out + ".log").c_str());
    lf << log.str();
    return EXIT_SUCCESS;
}
