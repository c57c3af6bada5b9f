// plink_bed.hpp -- opening and checking a SNP-major PLINK .bed, shared by the `score` and `ldscore` command lines.
#pragma once
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <cstdint>
#include <sstream>
#include <string>

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
