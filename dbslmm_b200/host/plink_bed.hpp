// plink_bed.hpp -- opening and checking a SNP-major PLINK .bed (shared by the `score`, `ldscore` and `ld` command lines), and
// reading a .fam, a .bim and its chromosomes (`ldscore` and `ld`).
#pragma once
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <cmath>
#include <cstdint>
#include <cstdlib>
#include <fstream>
#include <sstream>
#include <string>
#include <unordered_set>
#include <vector>

struct BedFile {
    int fd = -1;
    uint64_t size = 0;
};

// Opens <bed_path> and checks the magic bytes, SNP-major mode and a size of exactly 3 + n_snp x ceil(n / 4) bytes.  Returns ""
// (f holds the open descriptor and the size) or the message to stop with.
inline std::string open_bed(const std::string& bed_path, int64_t n, int64_t n_snp, BedFile& f) {
    const int fd = open(bed_path.c_str(), O_RDONLY);
    if (fd < 0) return bed_path + " does not exist";
    struct stat sb;
    if (fstat(fd, &sb) != 0) return "cannot stat " + bed_path;
    unsigned char magic[3] = {0, 0, 0};
    if (sb.st_size < 3 || pread(fd, magic, 3, 0) != 3 || magic[0] != 0x6c || magic[1] != 0x1b)
        return bed_path + " is not a PLINK .bed file (magic bytes 6c 1b expected)";
    if (magic[2] != 0x01) return bed_path + " is individual-major; only SNP-major .bed files (third byte 01) are supported";
    const uint64_t pitch = (uint64_t)(n + 3) / 4;
    const uint64_t want = 3 + (uint64_t)n_snp * pitch;
    if ((uint64_t)sb.st_size != want) {
        std::ostringstream o;
        o << bed_path << " has " << sb.st_size << " bytes; " << n_snp << " variants x " << n << " individuals need " << want
          << " (3 + n_snp x ceil(n/4))";
        return o.str();
    }
    f.fd = fd;
    f.size = (uint64_t)sb.st_size;
    return "";
}

// (in a namespace: score_main.cpp has .bim helpers of its own)
namespace plink {

inline std::vector<std::string> split_ws(const std::string& line) {
    std::vector<std::string> t;
    std::istringstream ss(line);
    std::string x;
    while (ss >> x) t.push_back(x);
    return t;
}

// Non-empty lines of a .fam -> n.  Returns "" or the message to stop with.
inline std::string count_fam(const std::string& path, int64_t& n) {
    std::ifstream f(path.c_str());
    if (!f) return path + " does not exist";
    std::string line;
    n = 0;
    while (std::getline(f, line)) if (!split_ws(line).empty()) ++n;
    return "";
}

struct Bim { std::vector<std::string> chr, snp, bp_tok; std::vector<double> cm, bp; };

// A .bim: six columns, cM and bp numbers.  Returns "" or the message to stop with.
inline std::string read_bim(const std::string& path, Bim& b) {
    std::ifstream f(path.c_str());
    if (!f) return path + " does not exist";
    std::string line;
    size_t ln = 0;
    while (std::getline(f, line)) {
        ++ln;
        const std::vector<std::string> t = split_ws(line);
        if (t.empty()) continue;
        if (t.size() < 6) return path + " line " + std::to_string(ln) + ": a .bim line has 6 columns";
        char* e1 = nullptr;
        char* e2 = nullptr;
        const double cm = std::strtod(t[2].c_str(), &e1), bp = std::strtod(t[3].c_str(), &e2);
        if (*e1 != '\0' || *e2 != '\0' || !std::isfinite(cm) || !std::isfinite(bp))
            return path + " line " + std::to_string(ln) + ": columns 3 and 4 (cM, bp) must be numbers";
        b.chr.push_back(t[0]); b.snp.push_back(t[1]); b.bp_tok.push_back(t[3]); b.cm.push_back(cm); b.bp.push_back(bp);
    }
    return "";
}

// The chromosomes of a .bim: runs of equal column-1 tokens, each contiguous, with coordinates x (cM or bp, `unit`; NULL: not
// checked) non-decreasing within each.  chr_off gets n_chr + 1 offsets, chr_name the names.  Returns "" or the message.
inline std::string bim_chromosomes(const Bim& b, const std::string& bim_path, const std::vector<double>* x, const char* unit,
                                   std::vector<int32_t>& chr_off, std::vector<std::string>& chr_name) {
    chr_off.assign(1, 0);
    chr_name.clear();
    std::unordered_set<std::string> seen;
    const int64_t n_snp = (int64_t)b.chr.size();
    for (int64_t i = 0; i < n_snp; ++i) {
        if (i == 0 || b.chr[i] != b.chr[i - 1]) {
            if (!seen.insert(b.chr[i]).second)
                return "chromosome " + b.chr[i] + " is not contiguous in " + bim_path + " (it appears again at line " + std::to_string(i + 1) +
                       "): sort the fileset by chromosome";
            if (i > 0) chr_off.push_back((int32_t)i);
            chr_name.push_back(b.chr[i]);
        } else if (x && (*x)[i] < (*x)[i - 1]) {
            return bim_path + " line " + std::to_string(i + 1) + ": the " + unit + " coordinates of chromosome " + b.chr[i] + " are not sorted";
        }
    }
    chr_off.push_back((int32_t)n_snp);
    return "";
}

}  // namespace plink
