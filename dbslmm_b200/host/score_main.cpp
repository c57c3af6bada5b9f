// score_main.cpp -- `score` command line: the `plink --bfile <target> --score <eff>.txt 1 2 4 sum` step that DBSLMM's driver
// runs after the fit (DBSLMM_script.sh:87), for one or several score files in ONE pass over the target panel.
//
//   score --bfile <prefix> --score <file>[,<file>...] [varcol allelecol scorecol] [header] sum [--out <prefix>]
//
// Semantics restated from PLINK 1.9's documentation of --score (sum mode, mean imputation of missing calls):
//   SCORESUM_i = sum_j beta_j * dosage_ij, dosage = copies of the score file's allele (A1 copies, or A2 copies when the
//   allele is the .bim A2), a missing call replaced by the variant's mean dosage over the called genotypes;
//   CNT_i = 2 x the called genotypes of i over the loaded variants, CNT2_i = copies of the scored allele among them.
// Score-file IDs without a .bim match, alleles that are neither A1 nor A2, and non-finite scores are skipped and counted.
// Refused, by choice: PLINK's other --score modifiers (their semantics are not restated here), an ID repeated in a score
// file, an ID naming several .bim rows, a scored variant outside chromosomes 1-22 (ploidy rules), a .fam with parents
// (founder-only imputation frequencies), and individual-major .bed files.  Every check runs before the GPU is touched.
// The .bed is mapped, never read whole; the library gathers the scored rows chunk by chunk (dbslmm_b200_score_stream).
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>

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
#include <vector>

#include "dbslmm_b200.h"
#include "plink_bed.hpp"

using namespace std;

namespace {

[[noreturn]] void die(const string& msg, int code = 1) {
    cerr << "ERROR: " << msg << endl;
    exit(code);
}

void print_header() {
    cout << endl;
    cout << "*************************************************************" << endl;
    cout << "  Polygenic scores of a PLINK fileset (score), B200 build" << endl;
    cout << "  Type ./score -h for detailed help" << endl;
    cout << "*************************************************************" << endl;
    cout << endl;
}

void print_help() {
    cout << " score --bfile <prefix> --score <file>[,<file>...] [varcol allelecol scorecol] [header] sum [--out <prefix>]" << endl;
    cout << endl;
    cout << " --bfile   [prefix]    " << " target fileset: <prefix>.bed (SNP-major), .bim, .fam." << endl;
    cout << " --score   [file,...]  " << " score file(s); columns are 1-based, default 1 2 4 (DBSLMM's <eff>.txt:" << endl;
    cout << "                       " << " snp a1 beta beta/sqrt(2maf(1-maf)) flag).  `header` skips the first line." << endl;
    cout << "                       " << " `sum` is required: PLINK's sum mode with mean imputation of missing calls." << endl;
    cout << "                       " << " Several files (same variants and alleles in the same order, e.g. the" << endl;
    cout << "                       " << " <eff>_f<k>.txt of one dbslmm --h2-folds run) are scored in one pass." << endl;
    cout << " --out     [prefix]    " << " output prefix (default plink): <out>.profile, or <out>_f<k>.profile for" << endl;
    cout << "                       " << " several files; <out>.log." << endl;
}

vector<string> split_ws(const string& line) {
    vector<string> t;
    istringstream ss(line);
    string x;
    while (ss >> x) t.push_back(x);
    return t;
}

bool is_uint(const string& s) {
    if (s.empty()) return false;
    for (char c : s) if (c < '0' || c > '9') return false;
    return true;
}

// chromosome code 1..22 (optionally "chr"-prefixed), else 0
int autosome(const string& c) {
    string s = c;
    if (s.size() > 3 && (s.compare(0, 3, "chr") == 0 || s.compare(0, 3, "CHR") == 0)) s = s.substr(3);
    if (!is_uint(s) || s.size() > 2) return 0;
    const int v = atoi(s.c_str());
    return (v >= 1 && v <= 22) ? v : 0;
}

struct Params {
    string bfile, out = "plink";
    vector<string> score_files;
    int varcol = 1, allelecol = 2, scorecol = 4;
    bool header = false, sum = false;
};

Params parse(int argc, char** argv) {
    Params p;
    bool have_score = false;
    for (int i = 1; i < argc; ++i) {
        const string a = argv[i];
        if (a == "--bfile") {
            if (i + 1 >= argc) die("--bfile needs a prefix");
            p.bfile = argv[++i];
        } else if (a == "--out") {
            if (i + 1 >= argc) die("--out needs a prefix");
            p.out = argv[++i];
        } else if (a == "--score") {
            if (i + 1 >= argc) die("--score needs a file name");
            have_score = true;
            string list = argv[++i];
            size_t s0 = 0;
            for (;;) {
                const size_t c = list.find(',', s0);
                const string f = list.substr(s0, c == string::npos ? string::npos : c - s0);
                if (f.empty()) die("--score: empty file name in '" + list + "'");
                p.score_files.push_back(f);
                if (c == string::npos) break;
                s0 = c + 1;
            }
            // modifiers up to the next --option: three column numbers, `header`, `sum`; anything else is refused
            vector<string> nums;
            while (i + 1 < argc && strncmp(argv[i + 1], "--", 2) != 0) {
                const string m = argv[++i];
                if (is_uint(m)) nums.push_back(m);
                else if (m == "header") p.header = true;
                else if (m == "sum") p.sum = true;
                else die("--score modifier '" + m + "' is not supported (only varcol allelecol scorecol, header and sum; "
                         "PLINK's average mode, no-mean-imputation, center, double-dosage and the others are refused)");
            }
            if (!nums.empty()) {
                if (nums.size() != 3) die("--score takes exactly three column numbers (varcol allelecol scorecol)");
                p.varcol = atoi(nums[0].c_str()); p.allelecol = atoi(nums[1].c_str()); p.scorecol = atoi(nums[2].c_str());
                if (p.varcol < 1 || p.allelecol < 1 || p.scorecol < 1) die("--score column numbers are 1-based");
                if (p.varcol == p.allelecol || p.varcol == p.scorecol || p.allelecol == p.scorecol) die("--score column numbers must differ");
            }
        } else {
            die("unsupported option '" + a + "' (score takes --bfile, --score and --out; --read-freq and the other PLINK options are refused)");
        }
    }
    if (p.bfile.empty()) die("--bfile is required");
    if (!have_score) die("--score is required");
    if (!p.sum) die("--score needs the `sum` modifier (PLINK's default average mode is not supported)");
    return p;
}

struct ScoreFile {
    vector<string> id, allele;
    vector<double> score;
};

ScoreFile read_score(const string& path, const Params& p) {
    ifstream f(path.c_str());
    if (!f) die(path + " does not exist");
    ScoreFile s;
    unordered_map<string, size_t> seen;
    string line;
    size_t ln = 0;
    const int need = max(p.varcol, max(p.allelecol, p.scorecol));
    while (getline(f, line)) {
        ++ln;
        if (ln == 1 && p.header) continue;
        const vector<string> t = split_ws(line);
        if (t.empty()) continue;
        if ((int)t.size() < need) die(path + " line " + to_string(ln) + ": " + to_string(t.size()) + " columns, needs " + to_string(need));
        const string& id = t[p.varcol - 1];
        if (!seen.emplace(id, s.id.size()).second) die(path + ": variant ID '" + id + "' is repeated (line " + to_string(ln) + ")");
        s.id.push_back(id);
        s.allele.push_back(t[p.allelecol - 1]);
        const char* v = t[p.scorecol - 1].c_str();
        char* e = nullptr;
        const double x = strtod(v, &e);
        s.score.push_back((e != v && *e == '\0') ? x : NAN);      // unparsable -> not finite -> skipped and counted
    }
    return s;
}

struct Fam { vector<string> fid, iid, pheno; };

Fam read_fam(const string& path) {
    ifstream f(path.c_str());
    if (!f) die(path + " does not exist");
    Fam fam;
    string line;
    size_t ln = 0;
    while (getline(f, line)) {
        ++ln;
        const vector<string> t = split_ws(line);
        if (t.empty()) continue;
        if (t.size() < 6) die(path + " line " + to_string(ln) + ": a .fam line has 6 columns");
        if (t[2] != "0" || t[3] != "0")
            die(path + " line " + to_string(ln) + " lists parents: PLINK imputes from founders only, which score does not restate; "
                "set columns 3 and 4 to 0");
        fam.fid.push_back(t[0]); fam.iid.push_back(t[1]); fam.pheno.push_back(t[5]);
    }
    return fam;
}

struct Bim { vector<string> chr, a1, a2; unordered_map<string, int64_t> row; unordered_map<string, int> dup; };

Bim read_bim(const string& path) {
    ifstream f(path.c_str());
    if (!f) die(path + " does not exist");
    Bim b;
    string line;
    int64_t n = 0;
    size_t ln = 0;
    while (getline(f, line)) {
        ++ln;
        const vector<string> t = split_ws(line);
        if (t.empty()) continue;
        if (t.size() < 6) die(path + " line " + to_string(ln) + ": a .bim line has 6 columns");
        b.chr.push_back(t[0]); b.a1.push_back(t[4]); b.a2.push_back(t[5]);
        if (!b.row.emplace(t[1], n).second) b.dup[t[1]]++;
        ++n;
    }
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
    {
        ostringstream o;
        o << "Options: --bfile " << P.bfile << " --score ";
        for (size_t k = 0; k < P.score_files.size(); ++k) o << (k ? "," : "") << P.score_files[k];
        o << " " << P.varcol << " " << P.allelecol << " " << P.scorecol << (P.header ? " header" : "") << " sum --out " << P.out;
        say(o.str());
    }

    // ---- target fileset
    const Fam fam = read_fam(P.bfile + ".fam");
    const Bim bim = read_bim(P.bfile + ".bim");
    const int64_t n = (int64_t)fam.iid.size(), n_snp = (int64_t)bim.chr.size();
    if (n == 0) die(P.bfile + ".fam lists no individual");
    if (n > INT32_MAX) die(P.bfile + ".fam: too many individuals");
    const int64_t pitch = (n + 3) / 4;
    const string bed_path = P.bfile + ".bed";
    BedFile bedf;
    {
        const string err = open_bed(bed_path, n, n_snp, bedf);
        if (!err.empty()) die(err);
    }
    say(to_string(n) + " individuals and " + to_string(n_snp) + " variants in " + P.bfile + ".bed/.bim/.fam");

    // ---- score files: the same variants and alleles in the same order in every file
    vector<ScoreFile> files;
    for (const string& f : P.score_files) files.push_back(read_score(f, P));
    for (size_t k = 1; k < files.size(); ++k) {
        if (files[k].id.size() != files[0].id.size()) die(P.score_files[k] + " has " + to_string(files[k].id.size()) + " variants, " + P.score_files[0] + " has " + to_string(files[0].id.size()));
        for (size_t j = 0; j < files[0].id.size(); ++j)
            if (files[k].id[j] != files[0].id[j] || files[k].allele[j] != files[0].allele[j])
                die(P.score_files[k] + " line " + to_string(j + 1) + " names " + files[k].id[j] + " " + files[k].allele[j] + ", " +
                    P.score_files[0] + " names " + files[0].id[j] + " " + files[0].allele[j] + ": several score files must list the same variants and alleles in the same order");
    }
    const size_t n_var = files[0].id.size();
    // matching (shared by every file): .bim row and flip, or a skip reason
    vector<int64_t> row(n_var, -1);
    vector<uint8_t> flipv(n_var, 0);
    int64_t n_unmatched = 0, n_allele = 0;
    for (size_t j = 0; j < n_var; ++j) {
        auto it = bim.row.find(files[0].id[j]);
        if (it == bim.row.end()) { ++n_unmatched; continue; }
        if (bim.dup.count(files[0].id[j])) die("variant ID '" + files[0].id[j] + "' names several rows of " + P.bfile + ".bim");
        const int64_t r = it->second;
        const string& al = files[0].allele[j];
        if (al == bim.a1[r]) flipv[j] = 0;
        else if (al == bim.a2[r]) flipv[j] = 1;
        else { ++n_allele; continue; }
        if (!autosome(bim.chr[r]))
            die("variant " + files[0].id[j] + " is on chromosome " + bim.chr[r] + ": score handles chromosomes 1-22 only (PLINK applies ploidy rules elsewhere)");
        row[j] = r;
    }
    // a non-finite score skips its variant in that file; files with the same skip pattern share one streaming pass
    vector<vector<char>> use(files.size(), vector<char>(n_var, 0));
    vector<int64_t> n_nonfinite(files.size(), 0), n_loaded(files.size(), 0);
    for (size_t k = 0; k < files.size(); ++k)
        for (size_t j = 0; j < n_var; ++j) {
            if (row[j] < 0) continue;
            if (!std::isfinite(files[k].score[j])) { ++n_nonfinite[k]; continue; }
            use[k][j] = 1;
            ++n_loaded[k];
        }
    for (size_t k = 0; k < files.size(); ++k) {
        ostringstream o;
        o << P.score_files[k] << ": " << n_var << " variants, " << n_loaded[k] << " loaded; skipped: " << n_unmatched
          << " with no ID match in the .bim, " << n_allele << " with an allele that is neither A1 nor A2, " << n_nonfinite[k]
          << " with a non-finite score";
        say(o.str());
    }

    // ---- GPU
    void* map = mmap(nullptr, (size_t)bedf.size, PROT_READ, MAP_SHARED, bedf.fd, 0);
    if (map == MAP_FAILED) die("cannot map " + bed_path);
    close(bedf.fd);
    const uint8_t* payload = (const uint8_t*)map + 3;
    dbslmm_b200_handle* h = nullptr;
    if (dbslmm_b200_create(0, &h) != DBSLMM_B200_OK) die("cannot initialise the GPU (there is no CPU fallback)", 2);
    const size_t nf = files.size();
    vector<vector<double>> scores(nf, vector<double>((size_t)n, 0.0));
    vector<vector<int32_t>> cnt(nf), cnt2(nf);
    vector<int32_t> n_empty(nf, 0);
    vector<char> done(nf, 0);
    double gpu_ms = 0.0, bytes_streamed = 0.0;
    int passes = 0;
    for (size_t k0 = 0; k0 < nf; ++k0) {
        if (done[k0]) continue;
        vector<size_t> group;
        for (size_t k = k0; k < nf; ++k) if (!done[k] && use[k] == use[k0]) { group.push_back(k); done[k] = 1; }
        vector<int32_t> pos;
        vector<uint8_t> fl;
        for (size_t j = 0; j < n_var; ++j) if (use[k0][j]) { pos.push_back((int32_t)row[j]); fl.push_back(flipv[j]); }
        const int64_t m = (int64_t)pos.size();
        vector<double> beta(group.size() * (size_t)m);
        for (size_t g = 0; g < group.size(); ++g) {
            int64_t q = 0;
            for (size_t j = 0; j < n_var; ++j) if (use[k0][j]) beta[g * (size_t)m + (size_t)q++] = files[group[g]].score[j];
        }
        vector<double> sc(group.size() * (size_t)n);
        vector<int32_t> c1((size_t)n), c2((size_t)n);
        int32_t empty = 0;
        float ms = 0.0f;
        const int rc = dbslmm_b200_score_stream(h, payload, n_snp, (int32_t)n, pos.data(), fl.data(), m, beta.data(), (int32_t)group.size(),
                                                0, sc.data(), c1.data(), c2.data(), &empty, &ms);
        if (rc != DBSLMM_B200_OK) die(string("score_stream: ") + dbslmm_b200_last_error(h), 2);
        gpu_ms += ms;
        bytes_streamed += (double)m * (double)pitch;
        ++passes;
        for (size_t g = 0; g < group.size(); ++g) {
            scores[group[g]].assign(sc.begin() + (ptrdiff_t)(g * (size_t)n), sc.begin() + (ptrdiff_t)((g + 1) * (size_t)n));
            cnt[group[g]] = c1;
            cnt2[group[g]] = c2;
            n_empty[group[g]] = empty;
        }
    }
    dbslmm_b200_destroy(h);
    munmap(map, (size_t)bedf.size);

    // ---- <out>.profile / <out>_f<k>.profile: FID IID PHENO CNT CNT2 SCORESUM, one row per .fam line in .fam order
    for (size_t k = 0; k < nf; ++k) {
        string name = P.out + ".profile";
        if (nf > 1) name = P.out + "_f" + to_string(k) + ".profile";
        FILE* f = fopen(name.c_str(), "w");
        if (!f) die("cannot write " + name);
        fprintf(f, "%10s %10s %6s %6s %6s %12s\n", "FID", "IID", "PHENO", "CNT", "CNT2", "SCORESUM");
        for (int64_t i = 0; i < n; ++i)
            fprintf(f, "%10s %10s %6s %6d %6d %12.6g\n", fam.fid[i].c_str(), fam.iid[i].c_str(), fam.pheno[i].c_str(), cnt[k][i],
                    cnt2[k][i], scores[k][i]);
        if (fclose(f) != 0) die("cannot write " + name);
        say("Results written to " + name + " (" + to_string(n_empty[k]) + " loaded variant(s) with no called genotype)");
    }
    {
        ostringstream o;
        o << "Streamed " << bytes_streamed << " bytes of genotypes in " << passes << " pass(es); GPU kernel time " << gpu_ms
          << " ms; wall time " << chrono::duration<double>(chrono::steady_clock::now() - t0).count() << " s";
        say(o.str());
    }
    ofstream lf((P.out + ".log").c_str());
    lf << log.str();
    return EXIT_SUCCESS;
}
