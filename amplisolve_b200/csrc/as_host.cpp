// Host side of the two drop-in programs: text formats in and out, the libstdc++ hash-order emulation the
// reference's outputs depend on, per-call annotations (Fisher strand bias, 10-mers, homopolymer, flags)
// and the argv-compatible mains.  All arithmetic of the hot path (noise model, Poisson tests, call
// decision) happens on the GPU through the C ABI in as_capi.cu; nothing here evaluates it on the CPU.
//
//   EE = source_codes/AmpliSolveErrorEstimation.cpp, VC = source_codes/AmpliSolveVariantCalling.cpp
#include <sys/stat.h>
#include <sys/types.h>
#include <dirent.h>
#include <fcntl.h>
#include <sys/mman.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <clocale>
#include <cerrno>
#include <cmath>
#include <condition_variable>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <ctime>
#include <fstream>
#include <functional>
#include <iomanip>
#include <iostream>
#include <map>
#include <mutex>
#include <sstream>
#include <string>
#include <thread>
#include <unordered_map>
#include <vector>

#if defined(__x86_64__) && defined(__GNUC__)
#include <immintrin.h>
#endif

#include "../../include/amplisolve_b200.h"
#include "as_bam.h"
#include "as_factorials.h"
#include "as_wire.h"

namespace {

const char* GREEN = "\x1b[32m";
const char* RED = "\x1b[31m";
const char* YELLOW = "\x1b[33m";
const char* RESET = "\x1b[0m";
const char* STARS =
    "************************************************************************************************************************************";

// ---------------------------------------------------------------------------------------------------
// panel: the slots of the BED enumeration (EE) or of the noise table (VC), with twin links
// ---------------------------------------------------------------------------------------------------
struct Panel {
    std::vector<std::string> chroms;
    std::unordered_map<std::string, int32_t> chrom_idx;
    std::vector<int32_t> slot_chrom, slot_pos;
    std::vector<std::string> pos_text;  // VC prints the position text of the ASEQ row; kept for the noise-table route
    std::vector<std::string> ref;       // reference text per slot
    std::vector<uint8_t> dup;           // position enumerated at least twice (EE:664) / flagged YES (VC:514)
    std::vector<int32_t> twin_next, twin_head;
    // (chrom, pos) -> first and last slot of the position so far: one flat table with linear probing (a node-based
    // unordered_map pair cost 0.2 us per slot, a fifth of the caller program's run on a 200,000-slot panel)
    struct PosEntry { uint64_t key; int32_t first, last; };
    std::vector<PosEntry> table;
    uint64_t table_mask = 0;
    int64_t n_positions = 0;  // distinct (chrom, pos)
    bool has_twins = false;

    int32_t chrom_id(const std::string& c) {
        auto it = chrom_idx.find(c);
        if (it != chrom_idx.end()) return it->second;
        const int32_t id = (int32_t)chroms.size();
        chroms.push_back(c);
        chrom_idx.emplace(c, id);
        return id;
    }
    int32_t find_chrom(const char* c, size_t n) const {
        auto it = chrom_idx.find(std::string(c, n));
        return it == chrom_idx.end() ? -1 : it->second;
    }
    static uint64_t key(int32_t chrom, int32_t pos) { return ((uint64_t)(uint32_t)chrom << 32) | (uint32_t)pos; }
    static uint64_t mix(uint64_t k) {  // consecutive positions must not land in consecutive cells of one long run
        k *= 0x9E3779B97F4A7C15ull;
        return k ^ (k >> 29);
    }
    int64_t size() const { return (int64_t)slot_pos.size(); }
    void add_slot(int32_t chrom, int32_t pos) {
        slot_chrom.push_back(chrom);
        slot_pos.push_back(pos);
    }
    // twin links: slots of the same position chained in panel order
    void link() {
        const int64_t P = size();
        twin_next.assign(P, -1);
        twin_head.resize(P);
        uint64_t cap = 16;
        while (cap < (uint64_t)P * 2 + 2) cap <<= 1;
        table.assign(cap, PosEntry{0, -1, -1});
        table_mask = cap - 1;
        n_positions = 0;
        for (int64_t i = 0; i < P; ++i) {
            const uint64_t k = key(slot_chrom[i], slot_pos[i]);
            uint64_t h = mix(k) & table_mask;
            while (table[h].first >= 0 && table[h].key != k) h = (h + 1) & table_mask;
            PosEntry& en = table[h];
            if (en.first < 0) {
                en.key = k;
                en.first = en.last = (int32_t)i;
                twin_head[i] = (int32_t)i;
                ++n_positions;
            } else {
                twin_next[en.last] = (int32_t)i;
                twin_head[i] = en.first;
                en.last = (int32_t)i;
                has_twins = true;
            }
        }
    }
    int32_t lookup(int32_t chrom, int32_t pos) const {
        if (table.empty()) return -1;
        const uint64_t k = key(chrom, pos);
        uint64_t h = mix(k) & table_mask;
        while (table[h].first >= 0 && table[h].key != k) h = (h + 1) & table_mask;
        return table[h].first;
    }
};

bool read_file(const std::string& path, std::string& out) {
    FILE* f = fopen(path.c_str(), "rb");
    if (!f) return false;
    fseek(f, 0, SEEK_END);
    const long n = ftell(f);
    fseek(f, 0, SEEK_SET);
    out.resize(n > 0 ? (size_t)n : 0);
    const size_t got = n > 0 ? fread(&out[0], 1, (size_t)n, f) : 0;
    fclose(f);
    out.resize(got);
    return true;
}

inline const char* skip_ws(const char* p, const char* e) {
    while (p < e && (*p == ' ' || *p == '\t' || *p == '\r')) ++p;
    return p;
}
inline const char* token_end(const char* p, const char* e) {
    while (p < e && *p != ' ' && *p != '\t' && *p != '\r' && *p != '\n') ++p;
    return p;
}

// BED: chrom start end [...], whitespace separated, both ends inclusive (EE:633-637, EE:2595-2606)
bool load_bed(const std::string& path, Panel& panel, int& n_amplicons) {
    std::string text;
    if (!read_file(path, text)) return false;
    n_amplicons = 0;
    const char* p = text.data();
    const char* e = p + text.size();
    while (p < e) {
        const char* eol = (const char*)memchr(p, '\n', e - p);
        if (!eol) eol = e;
        const char* q = skip_ws(p, eol);
        const char* t = token_end(q, eol);
        if (t > q) {
            std::string chrom(q, t);
            char* endp = nullptr;
            const long s = strtol(t, &endp, 10);
            const long en = strtol(endp, &endp, 10);
            if (endp > t) {
                ++n_amplicons;
                const int32_t c = panel.chrom_id(chrom);
                for (long idx = s; idx <= en; ++idx) panel.add_slot(c, (int32_t)idx);
            }
        }
        p = eol + 1;
    }
    return true;
}

// Reference bases straight from the .fai-indexed FASTA: the base samtools faidx <fa> chr:p-p prints (EE:644),
// without one fork per position.
struct FaiEntry { long long len, off, linebases, linewidth; };
bool annotate_reference(const std::string& fasta, Panel& panel, std::string& err) {
    std::string fai;
    if (!read_file(fasta + ".fai", fai)) { err = "cannot open " + fasta + ".fai (index the FASTA with samtools faidx)"; return false; }
    std::unordered_map<std::string, FaiEntry> idx;
    {
        const char* p = fai.data();
        const char* e = p + fai.size();
        while (p < e) {
            const char* eol = (const char*)memchr(p, '\n', e - p);
            if (!eol) eol = e;
            const char* t = (const char*)memchr(p, '\t', eol - p);
            if (t) {
                FaiEntry en;
                if (sscanf(t + 1, "%lld\t%lld\t%lld\t%lld", &en.len, &en.off, &en.linebases, &en.linewidth) == 4 && en.linebases > 0)
                    idx.emplace(std::string(p, t), en);
            }
            p = eol + 1;
        }
    }
    // the FASTA is mapped, not read: only the pages that hold panel positions are ever touched (one page fault per
    // ~4 kb of panel instead of one pread -- or, in the reference, one samtools fork -- per position)
    const int fd = open(fasta.c_str(), O_RDONLY);
    if (fd < 0) { err = "cannot open " + fasta; return false; }
    struct stat sb;
    if (fstat(fd, &sb) != 0) { close(fd); err = "cannot stat " + fasta; return false; }
    const size_t fsize = (size_t)sb.st_size;
    const char* base = fsize ? (const char*)mmap(nullptr, fsize, PROT_READ, MAP_PRIVATE, fd, 0) : nullptr;
    close(fd);
    if (fsize && base == (const char*)MAP_FAILED) { err = "cannot map " + fasta; return false; }
    const int64_t P = panel.size();
    panel.ref.resize(P);
    bool ok = true;
    int32_t last_chrom = -1;
    const FaiEntry* en = nullptr;
    for (int64_t i = 0; i < P && ok; ++i) {
        if (panel.slot_chrom[i] != last_chrom) {  // one index lookup per run of slots on the same contig
            last_chrom = panel.slot_chrom[i];
            auto it = idx.find(panel.chroms[last_chrom]);
            en = it == idx.end() ? nullptr : &it->second;
        }
        const long long pos = panel.slot_pos[i];
        if (!en || pos < 1 || pos > en->len) {
            err = "region " + panel.chroms[panel.slot_chrom[i]] + ":" + std::to_string(pos) + " is not in " + fasta;
            ok = false;
            break;
        }
        const long long off = en->off + (pos - 1) / en->linebases * en->linewidth + (pos - 1) % en->linebases;
        if (off < 0 || (size_t)off >= fsize) { err = "short read in " + fasta; ok = false; break; }
        panel.ref[i] = std::string(1, base[off]);
    }
    if (base) munmap((void*)base, fsize);
    return ok;
}

// ---------------------------------------------------------------------------------------------------
// file lists in the reference's order: `ls <dir>/*.ASEQ` (EE:556, VC:391) inserted into an unordered_map
// keyed by the listed path (EE:832), then iterated (EE:1081, VC:672)
// ---------------------------------------------------------------------------------------------------
struct CountFile { std::string path, sample; };

inline bool ends_with(const std::string& n, const char* tail) {
    const size_t k = strlen(tail);
    return n.size() >= k && n.compare(n.size() - k, k, tail) == 0;
}

// A count directory is read as BAM input when it holds *.bam files and no *.ASEQ file (names starting with '.' do not
// count, as for `ls <dir>/*.ASEQ`); a directory with an ASEQ file is read as ASEQ text whatever else it holds.
bool bam_input_dir(const std::string& dir) {
    DIR* d = opendir(dir.c_str());
    if (!d) return false;
    bool aseq = false, bam = false;
    while (dirent* en = readdir(d)) {
        const std::string n = en->d_name;
        if (n[0] == '.') continue;
        aseq = aseq || ends_with(n, ".ASEQ");
        bam = bam || ends_with(n, ".bam");
    }
    closedir(d);
    return bam && !aseq;
}

// *bam_mode (when not NULL): the directory holds BAM input (bam_input_dir).  A BAM file <name>.bam takes the place its computeCounts output
// <name>.PILEUP.ASEQ would take: the same sort and the same hash keys give the same sample order and names, only the path
// (and the list file) names the BAM.
bool list_count_files(const std::string& dir, std::vector<CountFile>& files, std::vector<std::string>& listed, bool* bam_mode = nullptr) {
    DIR* d = opendir(dir.c_str());
    if (!d) return false;
    std::vector<std::string> names, bams;
    while (dirent* en = readdir(d)) {
        const std::string n = en->d_name;
        if (n.size() >= 5 && n.compare(n.size() - 5, 5, ".ASEQ") == 0 && n[0] != '.') names.push_back(n);
        if (ends_with(n, ".bam") && n[0] != '.') bams.push_back(n);
    }
    closedir(d);
    const bool bam = bam_mode && names.empty() && !bams.empty();
    if (bam_mode) *bam_mode = bam;
    std::map<std::string, std::string> bam_of;  // "<dir>/<name>.PILEUP.ASEQ" -> "<dir>/<name>.bam"
    if (bam) {
        for (const std::string& b : bams) {
            names.push_back(b.substr(0, b.size() - 4) + ".PILEUP.ASEQ");
            bam_of[dir + "/" + names.back()] = dir + "/" + b;
        }
    }
    setlocale(LC_COLLATE, "");
    std::sort(names.begin(), names.end(), [](const std::string& a, const std::string& b) {
        const int c = strcoll(a.c_str(), b.c_str());
        return c != 0 ? c < 0 : a < b;
    });
    std::unordered_map<std::string, std::string> hash;  // exactly the container of EE:832 / VC:615
    for (const std::string& n : names) {
        const std::string path = dir + "/" + n;
        listed.push_back(bam ? bam_of[path] : path);
        // sample name = listed path minus "<dir>/" and the 12 characters of ".PILEUP.ASEQ" (EE:831)
        std::string sample = n.size() > 12 ? n.substr(0, n.size() - 12) : std::string();
        hash.insert(std::make_pair(path, sample));
    }
    for (auto it = hash.begin(); it != hash.end(); ++it) files.push_back(CountFile{bam ? bam_of[it->first] : it->first, it->second});
    return true;
}

// ---------------------------------------------------------------------------------------------------
// .PILEUP.ASEQ -> dense counts of one sample (EE:1114-1176, VC:723-770)
//
// Text ingestion is what bounds a real run once the kernels are at the HBM roof (SURVEY.md 8 f2), so the row loop is
// built for speed: the file is mmap'ed (no copy), a row in the usual shape -- one tab between fields, digits only -- is
// parsed by a branch-light scanner without bounds checks (anything else, and the last 256 bytes of the file, go through
// the general whitespace-tolerant parser, which accepts everything sscanf("%s %s %s %s %s %s %d ...") of the reference
// does), and the slot of a row is found by a CURSOR: ASEQ files follow the panel enumeration, so the next row almost
// always belongs to the next slot (or a few slots further when rows are missing); the hash lookup is the fallback.
// ---------------------------------------------------------------------------------------------------
struct AseqStats {
    int64_t rows = 0, outside = 0, extra = 0, bad_rd = 0;
    bool ok = true;
    bool in_order = true;                 // every row landed on a later slot than the row before it (row order == slot order)
    std::vector<int32_t> slot_of_row;     // filled only for files that are NOT in order (second parse): row -> slot or -1
    std::vector<as_wide_record> wide;     // records of this file that do not fit the wire format
    // Rows the dense tensor has no place for, kept so that the programs count them like the reference does:
    struct ExtraRow {   // a row beyond the number of panel slots of its position (the reference inserts every row, EE:1241-1245)
        int32_t row, slot, k;        // row of the file, first slot of the position, 0-based rank among the position's extra rows
        uint32_t fw[4], bw[4];
        long long rd;
    };
    struct RdFix { int32_t slot; long long rd; };  // a row whose RD column is not A+C+G+T (the reference divides by the column)
    std::vector<ExtraRow> extras;
    std::vector<RdFix> rd_fix;
};

// Host layouts of a count tensor (include/amplisolve_b200.h).  FMT = bytes per count in the two plain layouts (4: the
// canonical uint32, 2: the 16-bit wire format), 1 = the packed wire format (one uint32 per (sample, strand, slot)).
template <int FMT> struct Wire;
template <> struct Wire<4> { typedef uint32_t E; enum { PER = 4 }; };
template <> struct Wire<2> { typedef uint16_t E; enum { PER = 4 }; };
template <> struct Wire<1> { typedef uint32_t E; enum { PER = 1 }; };

inline bool parse_int(const char*& p, const char* e, long long& v) {
    p = skip_ws(p, e);
    bool neg = false;
    if (p < e && (*p == '-' || *p == '+')) { neg = *p == '-'; ++p; }
    if (p >= e || *p < '0' || *p > '9') return false;
    long long x = 0;
    while (p < e && *p >= '0' && *p <= '9') { x = x * 10 + (*p - '0'); ++p; }
    v = neg ? -x : x;
    return true;
}

// std::stof of the text [b, end) of a threshold (VC:889-890), 0 for an empty one.  The cells a noise table holds -- "%f" of a
// float ("0.001234"), "-2", "0.01" -- are [-]digits[.digits] with at most 8 digits in all: the digits are an integer n < 10^8
// and the value is n / 10^s, s <= 8.  double(n) / 10^s is the correctly rounded double of the decimal, and narrowing it gives
// the correctly rounded FLOAT as strtof does: a float rounding boundary m / 2^k (m < 2^25) near n / 10^s differs from it by
// at least 1 / (10^s * 2^k) -- relative 1 / (n * 2^k) ~ 1 / (m * 10^s) > 2^-52 -- or not at all, so the first rounding never
// lands on a boundary it was not on (checked against strtof for every n < 10^7 at s = 6: scripts/parse_bench.cpp).
// Anything else (exponents, nan, more digits) goes to strtof.
inline float threshold_text_to_float(const char* b, const char* end) {
    if (b >= end) return 0.f;
    static const double pow10[9] = {1., 10., 100., 1e3, 1e4, 1e5, 1e6, 1e7, 1e8};
    const char* q = b;
    const bool neg = *q == '-';
    q += neg ? 1 : 0;
    uint32_t n = 0;
    int digits = 0, frac = 0;
    while (q < end && (unsigned)(*q - '0') <= 9u) { n = n * 10u + (uint32_t)(*q - '0'); ++q; ++digits; }
    if (q < end && *q == '.') {
        ++q;
        while (q < end && (unsigned)(*q - '0') <= 9u) { n = n * 10u + (uint32_t)(*q - '0'); ++q; ++digits; ++frac; }
    }
    if (q != end || digits == 0 || digits > 8) return strtof(b, nullptr);
    const float v = (float)((double)n / pow10[frac]);
    return neg ? -v : v;
}

// "%f" of a float threshold (EE:1787), appended to o.  For 0 <= v < 2^20 the value v * 10^6 is EXACT in a double (a 24-bit
// significand times 10^6 < 2^20), so rint() under the default rounding mode is the round-half-even of the exact decimal that
// printf performs (compared with snprintf for every float in [0, 0.0625] and a sample above); anything else (negative,
// -0, huge, nan, inf) goes to snprintf.
inline void append_percent_f(std::string& o, float v) {
    if (!(v >= 0.f && v < 1048576.f) || std::signbit(v)) {  // -0 prints its sign
        char cell[64];
        snprintf(cell, sizeof cell, "%f", (double)v);
        o += cell;
        return;
    }
    const uint64_t n = (uint64_t)__builtin_rint((double)v * 1e6);
    uint64_t ip = n / 1000000u;
    uint32_t fp = (uint32_t)(n % 1000000u);
    char buf[32];
    char* e = buf + sizeof buf;
    char* q = e;
    for (int k = 0; k < 6; ++k) { *--q = (char)('0' + fp % 10u); fp /= 10u; }
    *--q = '.';
    do { *--q = (char)('0' + ip % 10u); ip /= 10u; } while (ip);
    o.append(q, (size_t)(e - q));
}

// "%g" of a float Germ_Max value (the reference's ostream << double, EE:2815) for 1e-4 <= v < 1: six significant digits in
// fixed notation, trailing zeros removed.  Exact: v = m * 2^-s with m < 2^24, and m * 10^D < 2^54 for the D <= 9 decimals
// needed, so the round-half-even of v * 10^D is integer arithmetic (equal to snprintf on every float of [1e-4, 1):
// scripts/parse_bench.cpp --percent-g).  Returns false -- nothing appended -- for any other value: the caller uses snprintf.
inline bool append_percent_g(std::string& o, float v) {
    if (!(v >= 1e-4f && v < 1.0f)) return false;
    uint32_t bits;
    memcpy(&bits, &v, 4);
    const uint64_t m = (bits & 0x7FFFFFu) | 0x800000u;  // a normal number
    const int s = 150 - (int)(bits >> 23);               // v = m * 2^-s, 24 <= s <= 37
    static const uint64_t p10[10] = {1ull, 10ull, 100ull, 1000ull, 10000ull, 100000ull, 1000000ull, 10000000ull, 100000000ull, 1000000000ull};
    int D = v >= 0.1f ? 6 : v >= 0.01f ? 7 : v >= 0.001f ? 8 : 9;  // decimals of six significant digits
    uint64_t n;
    for (;;) {
        const uint64_t N = m * p10[D];
        const uint64_t half = 1ull << (s - 1), rem = N & ((half << 1) - 1);
        n = N >> s;
        n += (rem > half || (rem == half && (n & 1))) ? 1 : 0;
        if (n < 100000ull && D < 9) { ++D; continue; }  // the float constant sat on the other side of the decimal boundary
        break;
    }
    if (n < 100000ull) return false;
    if (n >= 1000000ull) {  // rounded up into the next decade: 1.00000 x 10^(X+1)
        n = 100000ull;
        if (--D < 6) return false;
    }
    char buf[16];
    int len = 0;
    buf[len++] = '0';
    buf[len++] = '.';
    for (int z = 6; z < D; ++z) buf[len++] = '0';
    char dig[6];
    for (int k = 5; k >= 0; --k) { dig[k] = (char)('0' + n % 10); n /= 10; }
    int last = 5;
    while (last > 0 && dig[last] == '0') --last;
    for (int k = 0; k <= last; ++k) buf[len++] = dig[k];
    o.append(buf, (size_t)len);
    return true;
}

struct MappedFile {  // read-only view of a whole file
    const char* p = nullptr;
    size_t n = 0;
    bool ok = false;
    explicit MappedFile(const std::string& path) {
        const int fd = open(path.c_str(), O_RDONLY);
        if (fd < 0) return;
        struct stat sb;
        if (fstat(fd, &sb) != 0) { close(fd); return; }
        n = (size_t)sb.st_size;
        ok = true;
        if (n > 0) {
            void* m = mmap(nullptr, n, PROT_READ, MAP_PRIVATE, fd, 0);
            if (m == MAP_FAILED) { ok = false; n = 0; }
            else { p = (const char*)m; madvise(m, n, MADV_SEQUENTIAL); }
        }
        close(fd);
    }
    ~MappedFile() { if (p) munmap((void*)p, n); }
    MappedFile(const MappedFile&) = delete;
    MappedFile& operator=(const MappedFile&) = delete;
};

struct AseqRow {
    const char* chrom;
    size_t chrom_len;
    long long pos, v[9];  // A C G T RD Ars Crs Grs Trs
};

// The usual row, "chr\tpos\tx\tx\tx\tx\tA\tC\tG\tT\tRD\tArs\tCrs\tGrs\tTrs\n" with unsigned decimal numbers: no bounds checks
// (the caller guarantees 256 readable bytes), returns false -- p untouched -- at the first byte that does not fit.
inline bool parse_row_fast(const char*& p, AseqRow& r) {
    const char* q = p;
    r.chrom = q;
    while ((unsigned char)*q > ' ') ++q;
    r.chrom_len = (size_t)(q - p);
    if (*q != '\t' || r.chrom_len == 0) return false;
    ++q;
    unsigned d = (unsigned)(*q - '0');
    if (d > 9) return false;
    uint64_t x = 0;
    do { x = x * 10 + d; d = (unsigned)(*++q - '0'); } while (d <= 9);
    r.pos = (long long)x;
    uint64_t dots;
    memcpy(&dots, q, 8);
    if (dots == 0x2E092E092E092E09ull) {  // "\t.\t.\t.\t." -- dbsnp MAF ref alt as the pileup step writes them
        q += 8;
    } else {
        for (int k = 0; k < 4; ++k) {
            if (*q != '\t') return false;
            ++q;
            if ((unsigned char)*q <= ' ') return false;
            while ((unsigned char)*q > ' ') ++q;
        }
    }
    for (int k = 0; k < 9; ++k) {
        if (*q != '\t') return false;
        d = (unsigned)(*++q - '0');
        if (d > 9) return false;
        uint32_t y = 0;
        int digits = 0;
        do { y = y * 10 + d; d = (unsigned)(*++q - '0'); ++digits; } while (d <= 9);
        if (digits > 9) return false;  // beyond 32 bits: the general parser decides
        r.v[k] = y;
    }
    if (*q == '\r') ++q;
    if (*q != '\n') return false;
    p = q + 1;
    return true;
}

#if defined(__x86_64__) && defined(__GNUC__)
#define AS_ROW_AVX2 1
__attribute__((target("avx2,bmi,bmi2"))) static inline uint64_t mask64(__m256i lo, __m256i hi) {
    return (uint64_t)(uint32_t)_mm256_movemask_epi8(lo) | ((uint64_t)(uint32_t)_mm256_movemask_epi8(hi) << 32);
}
// four numbers of up to eight digits: lane k holds the eight bytes that END where number k ends, keep = the mask of its own
// digits (the leading bytes belong to the field before).  Digit values -> pairs -> fours -> the number, in 64-bit lanes.
__attribute__((target("avx2,bmi,bmi2"))) static inline __m256i digits8x4(__m256i text, __m256i keep) {
    const __m256i d = _mm256_and_si256(_mm256_sub_epi8(text, _mm256_set1_epi8('0')), keep);
    const __m256i pairs = _mm256_maddubs_epi16(d, _mm256_set1_epi16(0x010A));           // byte0 * 10 + byte1
    const __m256i fours = _mm256_madd_epi16(pairs, _mm256_set1_epi32(0x00010064));     // pair0 * 100 + pair1
    return _mm256_add_epi64(_mm256_mul_epu32(fours, _mm256_set1_epi64x(10000)), _mm256_srli_epi64(fours, 32));
}
__attribute__((target("avx2,bmi,bmi2"))) static inline __m256i load8x4(const char* a, const char* b, const char* c, const char* d) {
    long long w0, w1, w2, w3;
    memcpy(&w0, a - 8, 8); memcpy(&w1, b - 8, 8); memcpy(&w2, c - 8, 8); memcpy(&w3, d - 8, 8);
    return _mm256_set_epi64x(w3, w2, w1, w0);
}

// The rows parse_row_fast takes, without a branch per byte: one 64-byte window gives the bit masks of tabs, the newline,
// digits and white space; the 14 tabs delimit the fields, the masks prove the shape (no empty field, digits where numbers
// are, nothing else below '!'), and the ten numbers are converted four at a time in vector lanes.  Returns false -- p
// untouched -- for anything it is not sure about (a row of more than 63 bytes, a count of more than 8 digits, a position of
// more than 16): the scalar scanner and then the general parser decide.  Needs 16 readable bytes before p and 64 from p on.
__attribute__((target("avx2,bmi,bmi2"), noinline)) bool parse_row_avx2(const char*& p, AseqRow& r) {
    const __m256i a = _mm256_loadu_si256((const __m256i*)p), b = _mm256_loadu_si256((const __m256i*)(p + 32));
    const __m256i nl = _mm256_set1_epi8('\n'), tab = _mm256_set1_epi8('\t'), zero = _mm256_set1_epi8('0');
    const __m256i nine = _mm256_set1_epi8(9), space = _mm256_set1_epi8(' ');
    const uint64_t nlm = mask64(_mm256_cmpeq_epi8(a, nl), _mm256_cmpeq_epi8(b, nl));
    if (nlm == 0) return false;
    const unsigned n = (unsigned)__builtin_ctzll(nlm);  // the row is bytes [0, n)
    const uint64_t row = _bzhi_u64(~0ull, n);
    const uint64_t tm = mask64(_mm256_cmpeq_epi8(a, tab), _mm256_cmpeq_epi8(b, tab)) & row;
    const __m256i da = _mm256_sub_epi8(a, zero), db = _mm256_sub_epi8(b, zero);
    const uint64_t dm = mask64(_mm256_cmpeq_epi8(_mm256_min_epu8(da, nine), da), _mm256_cmpeq_epi8(_mm256_min_epu8(db, nine), db));
    const uint64_t wm = mask64(_mm256_cmpeq_epi8(_mm256_min_epu8(a, space), a), _mm256_cmpeq_epi8(_mm256_min_epu8(b, space), b)) & row;
    unsigned end = n;
    if (wm != tm) {  // the only other byte <= ' ' a row may hold is a '\r' before the newline
        if (n == 0 || p[n - 1] != '\r' || wm != (tm | (1ull << (n - 1)))) return false;
        end = n - 1;
    }
    if (__builtin_popcountll(tm) != 14 || (tm & (tm >> 1)) != 0 || (tm & 1) != 0) return false;
    alignas(32) uint32_t t[16];
    uint64_t x = tm;
#pragma GCC unroll 14
    for (int k = 0; k < 14; ++k) { t[k] = (unsigned)__builtin_ctzll(x); x = _blsr_u64(x); }
    t[14] = end;
    t[15] = end;
    if (t[13] + 1 >= end) return false;
    // digits: the position field and everything from the sixth tab to the end, tabs aside
    const uint64_t counts_at = _bzhi_u64(~0ull, end) & ~_bzhi_u64(~0ull, t[5]) & ~tm;
    const uint64_t numbers = counts_at | (_bzhi_u64(~0ull, t[1]) & ~_bzhi_u64(~0ull, t[0] + 1));
    if ((numbers & ~dm) != 0) return false;
    uint64_t run = counts_at;  // a count of nine digits or more: a run of nine set bits
    run &= run >> 1;
    run &= run >> 2;
    run &= run >> 4;
    run &= run >> 1;
    const unsigned lp = t[1] - t[0] - 1;
    if (run != 0 || lp > 16) return false;
    // lengths of the count fields 6..13 -> the masks of their digits inside the 8-byte windows
    const __m256i len8 = _mm256_sub_epi32(_mm256_sub_epi32(_mm256_loadu_si256((const __m256i*)(t + 6)), _mm256_loadu_si256((const __m256i*)(t + 5))),
                                          _mm256_set1_epi32(1));
    const __m256i ones = _mm256_set1_epi64x(-1), c64 = _mm256_set1_epi64x(64);
    const __m256i sh_a = _mm256_sub_epi64(c64, _mm256_slli_epi64(_mm256_cvtepu32_epi64(_mm256_castsi256_si128(len8)), 3));
    const __m256i sh_b = _mm256_sub_epi64(c64, _mm256_slli_epi64(_mm256_cvtepu32_epi64(_mm256_extracti128_si256(len8, 1)), 3));
    const unsigned lp_lo = lp < 8 ? lp : 8, lp_hi = lp - lp_lo;
    const __m256i sh_c = _mm256_sub_epi64(c64, _mm256_slli_epi64(_mm256_set_epi64x(0, lp_hi, lp_lo, end - t[13] - 1), 3));
    const __m256i va = digits8x4(load8x4(p + t[6], p + t[7], p + t[8], p + t[9]), _mm256_sllv_epi64(ones, sh_a));
    const __m256i vb = digits8x4(load8x4(p + t[10], p + t[11], p + t[12], p + t[13]), _mm256_sllv_epi64(ones, sh_b));
    const __m256i vc = digits8x4(load8x4(p + end, p + t[1], p + t[1] - 8, p + t[1]), _mm256_sllv_epi64(ones, sh_c));
    _mm256_storeu_si256((__m256i*)(r.v), va);
    _mm256_storeu_si256((__m256i*)(r.v + 4), vb);
    alignas(32) long long last[4];
    _mm256_store_si256((__m256i*)last, vc);
    r.v[8] = last[0];
    r.pos = last[2] * 100000000ll + last[1];
    r.chrom = p;
    r.chrom_len = t[0];
    p += n + 1;
    return true;
}
#endif

// Any row the reference's sscanf accepts (whitespace-separated, signs allowed).  Returns 0 = blank line, 1 = parsed,
// -1 = a first token but not 15 fields.  p moves past the line either way.
inline int parse_row_general(const char*& p, const char* e, AseqRow& r) {
    const char* eol = (const char*)memchr(p, '\n', (size_t)(e - p));
    if (!eol) eol = e;
    const char* q = skip_ws(p, eol);
    const char* t = token_end(q, eol);
    p = eol < e ? eol + 1 : e;
    if (t == q) return 0;
    r.chrom = q;
    r.chrom_len = (size_t)(t - q);
    const char* c = t;
    bool ok = parse_int(c, eol, r.pos);
    for (int k = 0; k < 4 && ok; ++k) { c = skip_ws(c, eol); c = token_end(c, eol); }
    for (int k = 0; k < 9 && ok; ++k) ok = parse_int(c, eol, r.v[k]);
    return ok ? 1 : -1;
}

// counts: this sample's plane pair, [2][P][PER], preset to "absent".  In the wire formats a record that does not fit (a
// count of 65534 or more in the 16-bit one; a major count beyond 16 bits or another count beyond 4 bits in the packed
// one) is escaped and goes to stats.wide.  record_rows: also fill stats.slot_of_row (files that are not in panel order).
// rd_rows_aside (the caller program): a row whose RD column is not A+C+G+T stays out of the tensor and is kept in
// stats.extras with k = -1 -- the reference's forward-strand test and Fisher table use RD - reverse reads (VC:895, VC:902),
// so such a row is tested separately with that depth.
template <int FMT>
void parse_aseq(const MappedFile& file, const Panel& panel, typename Wire<FMT>::E* counts, int32_t sample, bool record_rows,
                bool rd_rows_aside, AseqStats& st) {
    typedef typename Wire<FMT>::E E;
    const int PER = Wire<FMT>::PER;
    const E absent = (E)~(E)0;
    const int64_t P = panel.size();
    const int32_t* slot_pos = panel.slot_pos.data();
    const int32_t* slot_chrom = panel.slot_chrom.data();
    const char* p = file.p;
    const char* e = p + file.n;
    const char* eol = p ? (const char*)memchr(p, '\n', file.n) : nullptr;  // first line is the header (EE:1113)
    p = eol ? eol + 1 : e;
    const char* fast_end = file.n > 256 ? e - 256 : file.p;
    int32_t last_chrom = -2;
    const char* last_name = nullptr;
    size_t last_len = 0;
    int64_t cursor = 0, last_slot = -1;
    AseqRow r;
    auto taken = [&](int64_t c) {  // free in the tensor, but owned by a row that was set aside
        for (const AseqStats::ExtraRow& x : st.extras)
            if (x.k < 0 && x.slot == (int32_t)c) return true;
        return false;
    };
#ifdef AS_ROW_AVX2
    static const bool avx2 = __builtin_cpu_supports("avx2") && __builtin_cpu_supports("bmi") && __builtin_cpu_supports("bmi2") &&
                             !(getenv("AS_ROW_SCAN") && strcmp(getenv("AS_ROW_SCAN"), "scalar") == 0);  // the tests run both scanners
    const char* const simd_begin = file.p + 16;
#endif
    while (p < e) {
#ifdef AS_ROW_AVX2
        if (avx2 && p < fast_end && p >= simd_begin && parse_row_avx2(p, r)) {
            ++st.rows;
        } else
#endif
        if (!(p < fast_end && parse_row_fast(p, r))) {
            const int got = parse_row_general(p, e, r);
            if (got == 0) continue;
            ++st.rows;
            if (got < 0) { if (record_rows) st.slot_of_row.push_back(-1); continue; }
        } else {
            ++st.rows;
        }
        if (last_name == nullptr || last_len != r.chrom_len || memcmp(last_name, r.chrom, r.chrom_len) != 0) {
            last_name = r.chrom;
            last_len = r.chrom_len;
            last_chrom = panel.find_chrom(r.chrom, r.chrom_len);
        }
        // ---- the slot of this row: the k-th row of a position in a file takes the position's k-th slot (EE:1241-1245
        // keys records by position; the slots only matter for the order of the output rows)
        int64_t slot = -1;
        const int32_t pos = (int32_t)r.pos;
        if (last_chrom >= 0 && r.pos == (long long)pos) {
            for (int64_t c = cursor, ce = std::min(P, cursor + 32); c < ce; ++c)
                if (slot_pos[c] == pos && slot_chrom[c] == last_chrom && counts[c * PER] == absent && (st.extras.empty() || !taken(c))) { slot = c; break; }
            if (slot < 0) {  // not where the panel order says: hash lookup, then the first free slot of the position
                slot = panel.lookup(last_chrom, pos);
                if (slot < 0) {
                    ++st.outside;
                } else {
                    const int64_t first = slot;
                    while (slot >= 0 && (counts[slot * PER] != absent || (!st.extras.empty() && taken(slot)))) slot = panel.has_twins ? panel.twin_next[slot] : -1;
                    if (slot < 0) {  // more rows than panel slots for this position
                        ++st.extra;
                        st.in_order = false;  // the writer orders this file by rows
                        AseqStats::ExtraRow x;
                        x.row = (int32_t)(st.rows - 1);
                        x.slot = (int32_t)first;
                        x.k = 0;
                        for (const AseqStats::ExtraRow& y : st.extras) x.k += (y.k >= 0 && y.slot == x.slot) ? 1 : 0;
                        for (int b = 0; b < 4; ++b) { x.fw[b] = (uint32_t)(r.v[b] - r.v[5 + b]); x.bw[b] = (uint32_t)r.v[5 + b]; }
                        x.rd = r.v[4];
                        st.extras.push_back(x);
                    }
                }
            }
        } else {
            ++st.outside;
        }
        if (record_rows) st.slot_of_row.push_back((int32_t)slot);
        if (slot < 0) continue;
        if (slot < last_slot) st.in_order = false;
        last_slot = slot;
        cursor = slot + 1;
        // A C G T RD Ars Crs Grs Trs -> fw[b] = X - X_rs, bw[b] = X_rs (EE:1155-1176)
        const long long* v = r.v;
        if (v[0] + v[1] + v[2] + v[3] != v[4]) {
            ++st.bad_rd;
            if (rd_rows_aside) {
                st.in_order = false;  // the writer orders this file by rows
                AseqStats::ExtraRow x;
                x.row = (int32_t)(st.rows - 1);
                x.slot = (int32_t)slot;
                x.k = -1;
                for (int b = 0; b < 4; ++b) { x.fw[b] = (uint32_t)(v[b] - v[5 + b]); x.bw[b] = (uint32_t)v[5 + b]; }
                x.rd = v[4];
                st.extras.push_back(x);
                continue;
            }
            st.rd_fix.push_back(AseqStats::RdFix{(int32_t)slot, v[4]});
        }
        E* fw = counts + slot * PER;
        E* bw = counts + (P + slot) * PER;
        bool escape = false;
        if (FMT == 1) {
            uint32_t f4[4], r4[4], wf = 0, wb = 0;
            for (int b = 0; b < 4; ++b) {
                const long long f = v[b] - v[5 + b], r2 = v[5 + b];
                if (f < 0 || r2 < 0 || f > 0xFFFF || r2 > 0xFFFF) escape = true;
                f4[b] = (uint32_t)f;
                r4[b] = (uint32_t)r2;
            }
            if (!escape) escape = !(as_pack_word(f4, &wf) && as_pack_word(r4, &wb));
            fw[0] = (E)wf;
            bw[0] = (E)wb;
        } else {
            for (int b = 0; b < 4; ++b) {
                const long long f = v[b] - v[5 + b], r2 = v[5 + b];
                if (FMT == 2 && (f >= AS_WIRE_ESCAPE || r2 >= AS_WIRE_ESCAPE || f < 0 || r2 < 0)) escape = true;
                fw[b] = (E)f;
                bw[b] = (E)r2;
            }
        }
        if (escape) {
            as_wide_record w;
            w.sample = sample;
            w.slot = (int32_t)slot;
            for (int b = 0; b < 4; ++b) {
                w.fw[b] = (uint32_t)(v[b] - v[5 + b]);
                w.bw[b] = (uint32_t)v[5 + b];
                if (b < PER) fw[b] = bw[b] = (E)(absent - 1);  // AS_WIRE_ESCAPE / AS_PACKED_ESCAPE
            }
            st.wide.push_back(w);
        }
    }
}

template <int FMT>
AseqStats load_aseq(const std::string& path, const Panel& panel, typename Wire<FMT>::E* counts, int32_t sample, bool rd_rows_aside) {
    typedef typename Wire<FMT>::E E;
    AseqStats st;
    MappedFile file(path);
    if (!file.ok) { st.ok = false; return st; }
    const size_t words = (size_t)panel.size() * 2 * Wire<FMT>::PER;
    memset(counts, 0xFF, words * sizeof(E));
    parse_aseq<FMT>(file, panel, counts, sample, false, rd_rows_aside, st);
    if (!st.in_order) {  // rare: rows not in panel order.  Parse again, recording the slot of every row (the writer needs it)
        st = AseqStats();
        memset(counts, 0xFF, words * sizeof(E));
        parse_aseq<FMT>(file, panel, counts, sample, true, rd_rows_aside, st);
        st.in_order = false;
    }
    return st;
}

// ---------------------------------------------------------------------------------------------------
// Host threads that stay.  Every parallel phase of the programs (parsing files, the noise table in and out, the call
// writers) used to start hardware_concurrency threads of its own and join them: about a millisecond per phase on a
// 32-thread host, eight phases in a 70 ms job.  The pool's workers are created once (by the first phase; the resident
// service keeps them between programs) and sleep on a condition variable in between.  One phase runs at a time; a phase
// that finds the pool busy (the GPU worker thread of the caller program beside the main thread's parser) starts threads
// of its own as before.  The work functions share their items through atomics of their own, so it does not matter which
// or how many threads arrive.
// ---------------------------------------------------------------------------------------------------
class HostPool {
  public:
    static HostPool& get() {
        static HostPool* pool = new HostPool();  // never destroyed: the programs leave through _exit, the service stays
        return *pool;
    }
    // work() on up to n_threads threads, the caller's included; false (nothing done) when another phase holds the pool.
    // Only as many workers as the phase wants are woken; a worker that arrives after the caller has finished its own share
    // finds the phase closed, so the caller never waits for a thread that has not started.
    bool run(unsigned n_threads, const std::function<void()>& work) {
        std::unique_lock<std::mutex> phase(phase_m_, std::try_to_lock);
        if (!phase.owns_lock()) return false;
        unsigned wanted;
        {
            std::lock_guard<std::mutex> g(m_);
            job_ = &work;
            wanted = wanted_ = std::min<unsigned>(n_threads - 1, (unsigned)th_.size());
            taken_ = 0;
            ++gen_;
        }
        if (wanted >= th_.size()) cv_.notify_all();
        else for (unsigned k = 0; k < wanted; ++k) cv_.notify_one();
        work();
        std::unique_lock<std::mutex> g(m_);
        wanted_ = taken_;  // closed: no worker starts from here on
        done_cv_.wait(g, [this]() { return running_ == 0; });
        job_ = nullptr;
        return true;
    }

  private:
    HostPool() {
        const unsigned hw = std::min(256u, std::max(1u, std::thread::hardware_concurrency()));
        for (unsigned t = 1; t < hw; ++t) th_.emplace_back([this]() { loop(); });
        for (auto& t : th_) t.detach();
    }
    void loop() {
        unsigned seen = 0;
        for (;;) {
            const std::function<void()>* f = nullptr;
            {
                std::unique_lock<std::mutex> g(m_);
                cv_.wait(g, [&]() { return gen_ != seen; });
                seen = gen_;
                if (taken_ < wanted_) { ++taken_; ++running_; f = job_; }
            }
            if (!f) continue;
            (*f)();
            {
                std::lock_guard<std::mutex> g(m_);
                if (--running_ == 0) done_cv_.notify_one();
            }
        }
    }
    std::mutex phase_m_, m_;
    std::condition_variable cv_, done_cv_;
    std::vector<std::thread> th_;
    const std::function<void()>* job_ = nullptr;
    unsigned wanted_ = 0, taken_ = 0, running_ = 0, gen_ = 0;
};

void run_on_threads(unsigned n_threads, const std::function<void()>& work) {
    if (n_threads <= 1) { work(); return; }
    if (HostPool::get().run(n_threads, work)) return;
    std::vector<std::thread> th;
    for (unsigned t = 1; t < n_threads; ++t) th.emplace_back(work);
    work();
    for (auto& t : th) t.join();
}

// samples [first, first + n) of `files` into one tensor [n][2][P][PER]; sample ids in the wide records are 0..n-1
template <int FMT>
bool load_all(const std::vector<CountFile>& files, size_t first, size_t n, const Panel& panel, typename Wire<FMT>::E* counts,
              std::vector<AseqStats>& stats, bool rd_rows_aside = false) {
    typedef typename Wire<FMT>::E E;
    const int PER = Wire<FMT>::PER;
    const int64_t P = panel.size();
    stats.assign(n, AseqStats());
    std::atomic<size_t> next(0);
    auto work = [&]() {
        for (size_t i = next.fetch_add(1); i < n; i = next.fetch_add(1))
            stats[i] = load_aseq<FMT>(files[first + i].path, panel, counts + (int64_t)i * 2 * P * PER, (int32_t)i, rd_rows_aside);
    };
    run_on_threads(std::max(1u, std::min(std::thread::hardware_concurrency(), (unsigned)std::max<size_t>(1, n))), work);
    for (const AseqStats& s : stats)
        if (!s.ok) return false;
    return true;
}

template <class F>
void parallel_for(size_t n, F body) {
    if (n == 0) return;
    std::atomic<size_t> next(0);
    const size_t grain = 256;
    auto work = [&]() {
        for (size_t b = next.fetch_add(grain); b < n; b = next.fetch_add(grain))
            for (size_t i = b; i < std::min(n, b + grain); ++i) body(i);
    };
    run_on_threads((unsigned)std::max<size_t>(1, std::min<size_t>(std::thread::hardware_concurrency(), (n + grain - 1) / grain)), work);
}

// The count tensor of a group of samples in a wire format (a quarter / half of the pinned memory and PCIe traffic of
// uint32), in pinned memory owned by this object and reused from group to group.  The loader writes the packed format
// (8 bytes per record); when more than 1 record in 16 would have to be escaped (ultra-deep or very noisy data) the group is
// parsed again into the 16-bit format, and later groups go straight there.  Escaped records are in `wide`, sorted by
// (slot, sample).  AS_WIRE=16 / AS_WIRE=packed in the environment forces one of the two.
// Pinned buffers of finished programs, kept by the resident service for the next one (pinning memory costs about a
// millisecond per 4 MB: more than the GPU step of a configs[1] job).  At most four buffers and 4 GB stay parked.
struct PinnedPool {
    std::mutex m;
    std::vector<std::pair<void*, size_t>> free_list;
    void* take(size_t n, size_t& got) {  // the smallest parked buffer of at least n bytes
        std::lock_guard<std::mutex> g(m);
        size_t best = free_list.size();
        for (size_t i = 0; i < free_list.size(); ++i)
            if (free_list[i].second >= n && (best == free_list.size() || free_list[i].second < free_list[best].second)) best = i;
        if (best == free_list.size()) return nullptr;
        void* p = free_list[best].first;
        got = free_list[best].second;
        free_list.erase(free_list.begin() + (long)best);
        return p;
    }
    void give(void* p, size_t n) {
        void* drop = nullptr;
        {
            std::lock_guard<std::mutex> g(m);
            size_t total = n;
            for (const auto& f : free_list) total += f.second;
            if (n > (size_t)4 << 30) {
                drop = p;
            } else {
                free_list.emplace_back(p, n);
                while (free_list.size() > 4 || total > (size_t)4 << 30) {  // the oldest goes
                    total -= free_list.front().second;
                    if (drop) as_host_free(drop);
                    drop = free_list.front().first;
                    free_list.erase(free_list.begin());
                }
            }
        }
        if (drop) as_host_free(drop);
    }
};
PinnedPool g_pinned_pool;

struct HostCounts {
    void* p = nullptr;
    size_t bytes = 0;
    int fmt = 1;  // 1 packed, 2 uint16
    std::vector<as_wide_record> wide;
    void release() {
        if (p) {
            if (as_process_is_resident()) g_pinned_pool.give(p, bytes);
            else as_host_free(p);
        }
        p = nullptr;
        bytes = 0;
    }
    ~HostCounts() { release(); }
    bool reserve(size_t n) {
        if (n <= bytes) return true;
        release();
        n = std::max<size_t>(16, n);
        if (as_process_is_resident()) {
            size_t got = 0;
            if (void* q = g_pinned_pool.take(n, got)) { p = q; bytes = got; return true; }
        }
        if (as_host_alloc(&p, n) != AS_OK) { p = nullptr; return false; }
        bytes = n;
        return true;
    }
    // the eight counts of (sample, slot) of the group; P = slots of the panel
    void record(int64_t sample, int64_t slot, int64_t P, uint32_t (&fw)[4], uint32_t (&bw)[4]) const {
        const int64_t wf = (sample * 2) * P + slot, wb = wf + P;
        bool escaped;
        if (fmt == 2) {
            const uint16_t* f = (const uint16_t*)p + wf * 4;
            const uint16_t* b = (const uint16_t*)p + wb * 4;
            escaped = f[0] == AS_WIRE_ESCAPE;
            for (int i = 0; i < 4; ++i) { fw[i] = f[i]; bw[i] = b[i]; }
        } else {
            const uint32_t* w = (const uint32_t*)p;
            escaped = w[wf] == AS_PACKED_ESCAPE;
            as_unpack_word(w[wf], fw);
            as_unpack_word(w[wb], bw);
        }
        if (escaped) {
            as_wide_record key;
            key.slot = (int32_t)slot;
            key.sample = (int32_t)sample;
            auto it = std::lower_bound(wide.begin(), wide.end(), key, [](const as_wide_record& x, const as_wide_record& y) {
                return x.slot != y.slot ? x.slot < y.slot : x.sample < y.sample;
            });
            if (it != wide.end() && it->slot == slot && it->sample == sample) {
                for (int i = 0; i < 4; ++i) { fw[i] = it->fw[i]; bw[i] = it->bw[i]; }
            }
        }
    }
};
// samples [first, first + n) of `files`.  returns 0 ok, 1 pinned allocation failed, 2 a file could not be opened
int load_counts(const std::vector<CountFile>& files, size_t first, size_t n, const Panel& panel, HostCounts& hc,
                std::vector<AseqStats>& stats, bool rd_rows_aside = false) {
    const size_t strand_words = n * 2 * (size_t)panel.size();
    const char* force = getenv("AS_WIRE");
    if (force && !strcmp(force, "16")) hc.fmt = 2;
    hc.wide.clear();
    for (int fmt = hc.fmt; fmt <= 2; ++fmt) {
        if (!hc.reserve(std::max<size_t>(16, strand_words * 4 * (size_t)fmt))) return 1;
        hc.fmt = fmt;
        const bool ok = fmt == 1 ? load_all<1>(files, first, n, panel, (uint32_t*)hc.p, stats, rd_rows_aside)
                                 : load_all<2>(files, first, n, panel, (uint16_t*)hc.p, stats, rd_rows_aside);
        if (!ok) return 2;
        int64_t rows = 0, escaped = 0;
        for (const AseqStats& s : stats) { rows += s.rows; escaped += (int64_t)s.wide.size(); }
        if (fmt == 1 && escaped * 16 > rows && !(force && !strcmp(force, "packed"))) continue;  // too many: the 16-bit format is denser
        break;
    }
    for (AseqStats& s : stats) {
        hc.wide.insert(hc.wide.end(), s.wide.begin(), s.wide.end());
        s.wide.clear();
        s.wide.shrink_to_fit();
    }
    std::sort(hc.wide.begin(), hc.wide.end(), [](const as_wide_record& x, const as_wide_record& y) {
        return x.slot != y.slot ? x.slot < y.slot : x.sample < y.sample;
    });
    return 0;
}

// Rows beyond the number of panel slots of their position (a file that lists a position more often than the BED enumerates
// it).  The reference keys records by position and inserts every row (EE:1241-1245), so such rows count like all others:
// sums, N of the 0.338*N rule, Germ_Max, in file order.  The dense tensor gets SPILL SLOTS for them -- virtual slots
// appended after the panel's P slots and chained to the end of their position's twin group (chain order = row order within
// a file), absent in every sample that has no such row -- and the library reduces them like any duplicated position.
// Returns the new number of slots (P when there is nothing to do); twin_next / twin_head are the extended links.
int64_t add_spill_slots(const Panel& panel, HostCounts& hc, const std::vector<AseqStats>& stats, std::vector<int32_t>& twin_next,
                        std::vector<int32_t>& twin_head) {
    const int64_t P = panel.size();
    const size_t S = stats.size();
    std::map<int32_t, int32_t> need;  // first slot of a position -> spill slots it needs
    for (const AseqStats& st : stats)
        for (const AseqStats::ExtraRow& x : st.extras)
            if (x.k >= 0) need[x.slot] = std::max(need[x.slot], x.k + 1);
    twin_next = panel.twin_next;
    twin_head = panel.twin_head;
    if (need.empty()) return P;
    std::map<int32_t, int32_t> base;  // first slot -> id of its first spill slot
    int64_t P2 = P;
    for (const auto& kv : need) {
        base[kv.first] = (int32_t)P2;
        int32_t last = kv.first;
        while (twin_next[(size_t)last] >= 0) last = twin_next[(size_t)last];
        for (int32_t k = 0; k < kv.second; ++k) {
            twin_next[(size_t)last] = (int32_t)P2;
            twin_next.push_back(-1);
            twin_head.push_back(twin_head[(size_t)kv.first]);
            last = (int32_t)P2++;
        }
    }
    const size_t w = hc.fmt == 2 ? 8 : 4;  // bytes per (sample, strand, slot)
    void* mem = nullptr;
    if (as_host_alloc(&mem, std::max<size_t>(16, S * 2 * (size_t)P2 * w)) != AS_OK) return -1;
    memset(mem, 0xFF, S * 2 * (size_t)P2 * w);
    for (size_t pl = 0; pl < S * 2; ++pl) memcpy((char*)mem + pl * (size_t)P2 * w, (const char*)hc.p + pl * (size_t)P * w, (size_t)P * w);
    for (size_t smp = 0; smp < S; ++smp) {
        for (const AseqStats::ExtraRow& x : stats[smp].extras) {
            if (x.k < 0) continue;
            const int64_t id = base[x.slot] + x.k;
            bool escape = false;
            if (hc.fmt == 2) {
                uint16_t* f = (uint16_t*)mem + ((smp * 2) * (size_t)P2 + (size_t)id) * 4;
                uint16_t* b = (uint16_t*)mem + ((smp * 2 + 1) * (size_t)P2 + (size_t)id) * 4;
                for (int i = 0; i < 4; ++i) escape = escape || x.fw[i] >= AS_WIRE_ESCAPE || x.bw[i] >= AS_WIRE_ESCAPE;
                for (int i = 0; i < 4; ++i) { f[i] = escape ? AS_WIRE_ESCAPE : (uint16_t)x.fw[i]; b[i] = escape ? AS_WIRE_ESCAPE : (uint16_t)x.bw[i]; }
            } else {
                uint32_t wf = 0, wb = 0;
                escape = !(as_pack_word(x.fw, &wf) && as_pack_word(x.bw, &wb));
                ((uint32_t*)mem)[(smp * 2) * (size_t)P2 + (size_t)id] = escape ? AS_PACKED_ESCAPE : wf;
                ((uint32_t*)mem)[(smp * 2 + 1) * (size_t)P2 + (size_t)id] = escape ? AS_PACKED_ESCAPE : wb;
            }
            if (escape) {
                as_wide_record r;
                r.sample = (int32_t)smp;
                r.slot = (int32_t)id;
                memcpy(r.fw, x.fw, 16);
                memcpy(r.bw, x.bw, 16);
                hc.wide.push_back(r);
            }
        }
    }
    std::sort(hc.wide.begin(), hc.wide.end(), [](const as_wide_record& x, const as_wide_record& y) {
        return x.slot != y.slot ? x.slot < y.slot : x.sample < y.sample;
    });
    as_host_free(hc.p);
    hc.p = mem;
    hc.bytes = S * 2 * (size_t)P2 * w;
    return P2;
}

// ---------------------------------------------------------------------------------------------------
// BAM input: a count directory of *.bam files is piled up on the GPU (as_bam.h reads the files, as_pileup.cu counts) and
// every sample ends straight in the wire tensor (as_pileup_end_wire), with what computeCounts mbq= mrq= mdc= for a position
// file listing the panel's slots in order, followed by the ASEQ loader, would have given.
// ---------------------------------------------------------------------------------------------------
int env_int(const char* name, int fallback) {
    const char* v = getenv(name);
    return v && *v ? atoi(v) : fallback;
}

struct BamInput {
    int mbq = env_int("AS_BAM_MBQ", 20), mrq = env_int("AS_BAM_MRQ", 20), mdc = env_int("AS_BAM_MDC", 20);  // computeCounts' defaults
    std::map<std::string, int32_t> contig_id;  // panel chromosome -> pileup contig (= panel chromosome id)
    std::vector<int64_t> contig_first;         // the pileup's positions: sorted, unique, 0-based per contig
    std::vector<int32_t> upos;
    std::vector<int32_t> slot_unique;          // panel slot -> its position in upos (0 for the slots below)
    std::vector<int32_t> no_position;          // slots at a position below 1: computeCounts skips such lines, they stay absent
    asbam::Reader reader;

    void setup(const Panel& panel) {
        const int64_t P = panel.size();
        const int32_t n_contig = (int32_t)panel.chroms.size();
        std::vector<std::vector<int32_t>> per((size_t)n_contig);
        for (int64_t s = 0; s < P; ++s)
            if (panel.slot_chrom[s] >= 0 && panel.slot_pos[s] >= 1) per[(size_t)panel.slot_chrom[s]].push_back(panel.slot_pos[s] - 1);
        contig_first.assign((size_t)n_contig + 1, 0);
        for (int32_t c = 0; c < n_contig; ++c) {
            contig_id[panel.chroms[(size_t)c]] = c;
            auto& v = per[(size_t)c];
            std::sort(v.begin(), v.end());
            v.erase(std::unique(v.begin(), v.end()), v.end());
            contig_first[(size_t)c + 1] = contig_first[(size_t)c] + (int64_t)v.size();
            upos.insert(upos.end(), v.begin(), v.end());
        }
        slot_unique.assign((size_t)P, 0);
        for (int64_t s = 0; s < P; ++s) {
            const int32_t c = panel.slot_chrom[s];
            if (c < 0 || panel.slot_pos[s] < 1) { no_position.push_back((int32_t)s); continue; }
            const auto b = upos.begin() + contig_first[(size_t)c], e = upos.begin() + contig_first[(size_t)c + 1];
            slot_unique[(size_t)s] = (int32_t)(std::lower_bound(b, e, panel.slot_pos[s] - 1) - upos.begin());
        }
    }
};

// A packed group -> the 16-bit format, on the host and losslessly (the pileups are not run again): a record escaped in the
// packed form may fit the 16-bit one (a second count above 15) and a record that fits the packed form may not (a count of
// 65534 or 65535).  hc.wide must be sorted by (slot, sample).
bool transcode_to_16(HostCounts& hc, size_t n, int64_t P) {
    HostCounts out;
    out.fmt = 2;
    if (!out.reserve(std::max<size_t>(16, n * 2 * (size_t)P * 8))) return false;
    std::vector<as_wide_record> wide;
    std::mutex m;
    const uint32_t* w = (const uint32_t*)hc.p;
    uint16_t* o = (uint16_t*)out.p;
    parallel_for(n * (size_t)P, [&](size_t i) {
        const int64_t smp = (int64_t)i / P, s = (int64_t)i % P;
        uint16_t* f = o + ((smp * 2) * P + s) * 4;
        uint16_t* b = f + P * 4;
        if (w[(smp * 2) * P + s] == AS_PACKED_ABSENT) {
            for (int k = 0; k < 4; ++k) f[k] = b[k] = AS_WIRE_ABSENT;
            return;
        }
        as_wide_record r;
        hc.record(smp, s, P, r.fw, r.bw);
        const bool fits = as_wire16_fits(r.fw) && as_wire16_fits(r.bw);
        for (int k = 0; k < 4; ++k) {
            f[k] = fits ? (uint16_t)r.fw[k] : (uint16_t)AS_WIRE_ESCAPE;
            b[k] = fits ? (uint16_t)r.bw[k] : (uint16_t)AS_WIRE_ESCAPE;
        }
        if (!fits) {
            r.sample = (int32_t)smp;
            r.slot = (int32_t)s;
            std::lock_guard<std::mutex> g(m);
            wide.push_back(r);
        }
    });
    std::sort(wide.begin(), wide.end(), [](const as_wide_record& x, const as_wide_record& y) {
        return x.slot != y.slot ? x.slot < y.slot : x.sample < y.sample;
    });
    hc.release();
    std::swap(hc.p, out.p);
    std::swap(hc.bytes, out.bytes);
    hc.fmt = 2;
    hc.wide = std::move(wide);
    return true;
}

// samples [first, first + n) of `files` (BAM files) with the contract of load_counts: the same HostCounts, one AseqStats per
// file (rows = present slots, in panel order).  The wire-format policy is load_counts' too: packed, and the 16-bit format for
// the group when more than 1 record in 16 escapes (AS_WIRE=16 / packed forces one).  Returns 0 ok, 1 pinned allocation
// failed, 3 a BAM could not be read or piled up (computeCounts' message printed).  pctx runs the pileups: no other thread
// may use it meanwhile.
int load_bam_counts(const std::vector<CountFile>& files, size_t first, size_t n, const Panel& panel, BamInput& bi, as_ctx* pctx,
                    HostCounts& hc, std::vector<AseqStats>& stats) {
    const int64_t P = panel.size();
    const char* force = getenv("AS_WIRE");
    if (force && !strcmp(force, "16")) hc.fmt = 2;
    const int fmt = hc.fmt;
    const size_t per_sample = 2 * (size_t)P * 4 * (size_t)fmt;  // bytes of one sample's slice
    if (!hc.reserve(std::max<size_t>(16, n * per_sample))) return 1;
    hc.wide.clear();
    stats.assign(n, AseqStats());
    if (bi.upos.empty()) {
        printf("Error from computeCounts: no positions in the panel\n");
        return 3;
    }
    const int threads = (int)std::max(1u, std::thread::hardware_concurrency());
    std::vector<as_wide_record> w((size_t)P);
    int64_t rows_all = 0;
    for (size_t i = 0; i < n; ++i) {
        const int rc = bi.reader.pileup(files[first + i].path, bi.contig_id, threads, bi.mbq, bi.mrq, [&]() -> as_ctx* {
            if (as_pileup_begin(pctx, bi.contig_first.data(), (int32_t)(bi.contig_first.size() - 1), bi.upos.data(), (int64_t)bi.upos.size()) != AS_OK) {
                printf("Error from computeCounts: %s\n", as_last_error());
                return nullptr;
            }
            return pctx;
        }, nullptr);
        if (rc != 0) return 3;
        char* slice = (char*)hc.p + i * per_sample;
        int64_t n_wide = 0, rows = 0;
        if (as_pileup_end_wire(pctx, bi.slot_unique.data(), P, bi.mdc, fmt, (int32_t)i, slice, w.data(), P, &n_wide, &rows, nullptr) != AS_OK) {
            printf("Error from computeCounts: %s\n", as_last_error());
            return 3;
        }
        for (int32_t s : bi.no_position) {  // no line of the position file: absent whatever mdc is
            const bool present = fmt == 1 ? ((uint32_t*)slice)[s] != AS_PACKED_ABSENT : ((uint16_t*)slice)[(size_t)s * 4] != AS_WIRE_ABSENT;
            rows -= present ? 1 : 0;
            if (fmt == 1) ((uint32_t*)slice)[s] = ((uint32_t*)slice)[P + s] = AS_PACKED_ABSENT;
            else memset(slice + (size_t)s * 8, 0xFF, 8), memset(slice + (size_t)(P + s) * 8, 0xFF, 8);
        }
        for (int64_t k = 0; k < n_wide; ++k) {
            const as_wide_record& r = w[(size_t)k];
            if (bi.no_position.empty() || !std::binary_search(bi.no_position.begin(), bi.no_position.end(), r.slot)) hc.wide.push_back(r);
        }
        stats[i].rows = rows;
        rows_all += rows;
    }
    std::sort(hc.wide.begin(), hc.wide.end(), [](const as_wide_record& x, const as_wide_record& y) {
        return x.slot != y.slot ? x.slot < y.slot : x.sample < y.sample;
    });
    if (fmt == 1 && (int64_t)hc.wide.size() * 16 > rows_all && !(force && !strcmp(force, "packed")))  // the 16-bit format is denser
        if (!transcode_to_16(hc, n, P)) return 1;
    return 0;
}

// The GPUs of a run, chosen BEFORE the first CUDA call from the size of the ASEQ directory (bytes / 45 ~ records):
//   AS_DEVICES ("0,2,3") names them; otherwise a job below 2^28 records (2 GB in the packed format, ~40 ms of GPU time) runs
//   on one GPU -- several would only add start-up time -- and a larger one on every visible GPU (as_create_multi).
// When the process's device list is not fixed from outside, CUDA_VISIBLE_DEVICES is narrowed to the chosen devices first, so
// that the driver initialises those only (start-up grows with the number of visible GPUs).  The context is created on a
// thread at program entry: CUDA start-up takes 0.2-4 s on the test boxes, the panel / noise table is read meanwhile.
// A directory of BAM input (bam_input_dir) is sized from its BAM bytes: an amplicon BAM holds some thousands of compressed
// bytes per panel position (150-base reads at a few thousand x), so bytes / 4096 ~ records errs towards one GPU.
double aseq_dir_records(const std::string& dir) {
    double bytes = 0, bam_bytes = 0;
    if (DIR* d = opendir(dir.c_str())) {
        while (dirent* en = readdir(d)) {
            const std::string n = en->d_name;
            struct stat sb;
            if (n.size() >= 5 && n.compare(n.size() - 5, 5, ".ASEQ") == 0 && stat((dir + "/" + n).c_str(), &sb) == 0) bytes += (double)sb.st_size;
            if (ends_with(n, ".bam") && n[0] != '.' && stat((dir + "/" + n).c_str(), &sb) == 0) bam_bytes += (double)sb.st_size;
        }
        closedir(d);
    }
    return bam_input_dir(dir) ? bam_bytes / 4096.0 : bytes / 45.0;
}

// In the resident service (as_serve.cpp: one request at a time) the context object of a finished program is parked, not
// destroyed: the next program that asks for the same devices takes it over with its streams, events and grow-only device
// and pinned buffers (re-allocating them cost 8 ms of a 0.2 s configs[1] job and 45 ms of a 0.5 s configs[2] slice).
struct ParkedContext {
    std::mutex m;
    as_ctx* ctx = nullptr;
    std::vector<int> devs;
};
ParkedContext g_parked;

struct GpuContext {
    std::vector<int> made_for;  // device list the context was created for (empty: every visible GPU)
    as_ctx* ctx = nullptr;
    int rc = AS_OK;
    std::string error;
    std::thread starter;
    void start(double estimated_records) {
        // the device list and the environment are settled here, on the calling thread (setenv must not race with getenv)
        std::vector<int> devs;
        if (const char* env = getenv("AS_DEVICES")) {
            for (const char* q = env; *q;) {
                char* endp = nullptr;
                const long d = strtol(q, &endp, 10);
                if (endp == q) break;
                devs.push_back((int)d);
                q = *endp == ',' ? endp + 1 : endp;
            }
        }
        double threshold = 268435456.0;
        if (const char* env = getenv("AS_WIDEN_RECORDS")) threshold = atof(env);  // tests
        if (devs.empty() && estimated_records < threshold) devs.push_back(0);
        if (!devs.empty() && getenv("CUDA_VISIBLE_DEVICES") == nullptr && !as_process_is_resident()) {  // initialise only what is used; ordinals become 0..n-1 (the resident service is initialised already)
            std::string list;
            for (size_t i = 0; i < devs.size(); ++i) list += (i ? "," : "") + std::to_string(devs[i]);
            setenv("CUDA_VISIBLE_DEVICES", list.c_str(), 1);
            for (size_t i = 0; i < devs.size(); ++i) devs[i] = (int)i;
        }
        made_for = devs;
        if (as_process_is_resident() && getenv("AS_DEFER_CHUNKS") == nullptr) {  // (that knob is read when a context is created)
            std::lock_guard<std::mutex> g(g_parked.m);
            if (g_parked.ctx && g_parked.devs == devs) {
                ctx = g_parked.ctx;
                g_parked.ctx = nullptr;
                return;
            }
        }
        starter = std::thread([this, devs]() mutable {
            if (devs.empty()) {  // a large job: every visible GPU
                int n = 0;
                if (as_device_count(&n) != AS_OK || n == 0) n = 1;  // as_create(0) below fails with the "no CUDA device" message
                for (int i = 0; i < n; ++i) devs.push_back(i);
            }
            rc = devs.size() == 1 ? as_create(devs[0], &ctx) : as_create_multi(devs.data(), (int)devs.size(), &ctx);
            if (rc != AS_OK) error = as_last_error();
        });
    }
    bool wait() {
        if (starter.joinable()) starter.join();
        return rc == AS_OK && ctx != nullptr;
    }
    // The programs end right after their last output file: the context is NOT torn down piece by piece (frees, stream and
    // event destruction, a device synchronisation: tenths of a second to seconds on a busy box); the thin mains leave
    // through _exit and the driver reclaims everything at once.  An error path that returns early still joins the thread.
    ~GpuContext() {
        if (starter.joinable()) starter.join();
        if (ctx && as_process_is_resident()) {  // the service lives on: keep one context for the next program, free any other
            as_ctx* old = nullptr;
            {
                std::lock_guard<std::mutex> g(g_parked.m);
                old = g_parked.ctx;
                g_parked.ctx = ctx;
                g_parked.devs = made_for;
            }
            if (old) as_destroy(old);
        }
    }
};

bool make_dir(const std::string& path) {  // mkdir -p (EE:3079)
    std::string cur;
    for (size_t i = 0; i <= path.size(); ++i) {
        if (i == path.size() || path[i] == '/') {
            if (!cur.empty() && cur != "." && cur != "..") mkdir(cur.c_str(), 0777);
        }
        if (i < path.size()) cur.push_back(path[i]);
    }
    struct stat sb;
    return stat(path.c_str(), &sb) == 0 && S_ISDIR(sb.st_mode);
}

std::string arg_value(const char* arg, const char* key) {  // sscanf(arg, "key=%s", out) of EE:300-326
    const size_t n = strlen(key);
    if (strncmp(arg, key, n) != 0) return std::string();
    const char* p = arg + n;
    while (*p == ' ' || *p == '\t' || *p == '\n') ++p;
    const char* q = p;
    while (*q && *q != ' ' && *q != '\t' && *q != '\n') ++q;
    return std::string(p, q);
}

// AS_TIMING=1 in the environment prints one "AS_TIMING <phase> <seconds>" line per phase on stderr
// (stdout stays what the reference prints)
struct PhaseTimer {
    bool on;
    double t0;
    static double now() {
        timespec ts;
        clock_gettime(CLOCK_MONOTONIC, &ts);
        return ts.tv_sec + 1e-9 * ts.tv_nsec;
    }
    PhaseTimer() : on(getenv("AS_TIMING") != nullptr), t0(now()) {}
    void lap(const char* phase, double units = 0, const char* unit = "") {
        const double t1 = now();
        if (on) {
            fprintf(stderr, "AS_TIMING %s %.6f", phase, t1 - t0);
            if (units > 0) fprintf(stderr, " (%.3g %s/s)", units / (t1 - t0), unit);
            fprintf(stderr, "\n");
        }
        t0 = t1;
    }
};


// ---------------------------------------------------------------------------------------------------
// per-call annotations (host only: these run for called variants, a vanishing fraction of the records)
// ---------------------------------------------------------------------------------------------------
// two-sided Fisher exact test as VC:3797-3814.  Boost.Math 1.61 is not part of the reference tree
// (.MISSING_LARGE_BLOBS); the pdf is C(r,k) C(N-r,n-k) / C(N,n) through lgamma, like the oracle's stand-in.
// This scalar form backs as_fisher_test (the checker the Boost pin runs against); the programs evaluate all calls at once
// on the device (as_fisher_tests_host, as_fisher.cu) from the same lgamma values.
inline double lg1(double x) {  // lgamma(x + 1)
    int sign = 0;
    return lgamma_r(x + 1.0, &sign);
}
// log C(n, k) with the operands in a canonical order (the smaller of k, n - k first): C(n, k) and C(n, n - k) are then
// bitwise equal, so two terms of the hypergeometric distribution that are tied mathematically (symmetric tables: r = N - r,
// n = N - n) are tied in floating point too, and `pdf(k) <= cutoff` (VC:3811) keeps or drops them together
double log_choose(double n, double k) {
    const double lo = std::min(k, n - k), hi = std::max(k, n - k);
    return (lg1(n) - lg1(lo)) - lg1(hi);
}
// Boost.Math's hypergeometric pdf for N <= 170 (hypergeometric_pdf_factorial_imp: n! r! (N-n)! (N-r)! over
// N! k! (n-k)! (r-k)! (N-n-r+k)! from a table of factorials, multiplying while the running value is <= 1 and dividing while
// it is >= 1, clamped to 1).  Restated operation for operation: bit-identical to the pdf SciPy's compiled-in Boost returns on
// 1.4 million (N, r, n, k) points, which matters because the terms of a symmetric table are NOT bitwise equal under it and
// the two-sided sum keeps or drops the mirror term accordingly (tests/golden/fisher_boost.npz, tie tables).
double hyper_pdf_factorial(unsigned r, unsigned n, unsigned N, unsigned k) {
    double result = AS_FACTORIAL[n];
    const double num[3] = {AS_FACTORIAL[r], AS_FACTORIAL[N - n], AS_FACTORIAL[N - r]};
    const double den[5] = {AS_FACTORIAL[N], AS_FACTORIAL[k], AS_FACTORIAL[n - k], AS_FACTORIAL[r - k], AS_FACTORIAL[N - n - r + k]};
    int i = 0, j = 0;
    while (i < 3 || j < 5) {
        while (j < 5 && (result >= 1 || i >= 3)) result /= den[j++];
        while (i < 3 && (result <= 1 || j >= 5)) result *= num[i++];
    }
    return result > 1 ? 1.0 : result;
}
double hyper_pdf(unsigned r, unsigned n, unsigned N, unsigned k) {
    if (N <= 170) return hyper_pdf_factorial(r, n, N, k);
    return exp(log_choose(r, k) + log_choose((double)N - r, (double)n - k) - log_choose(N, n));
}
double fisher_test(int a, int b, int c, int d) {
    const unsigned N = a + b + c + d, r = a + c, n = c + d;
    const unsigned hi = std::min(r, n);
    const int lo_i = (int)(r + n - N);
    const unsigned lo = lo_i > 0 ? (unsigned)lo_i : 0u;
    const double cutoff = hyper_pdf(r, n, N, (unsigned)c);
    double acc = 0.0;
    for (int k = (int)lo; k < (int)hi + 1; ++k) {
        const double p = hyper_pdf(r, n, N, (unsigned)k);
        if (p <= cutoff) acc += p;
    }
    return acc;
}

// 10-mers from the noise table's reference column (VC:3307-3611): a missing neighbour contributes "-|",
// except at offsets -6, -3, -1 and +10 where it contributes "-".
std::string kmer(const Panel& panel, int32_t chrom, int32_t pos, bool down) {
    std::string out;
    for (int i = 0; i < 10; ++i) {
        const int off = down ? -(10 - i) : (i + 1);
        const int32_t s = panel.lookup(chrom, pos + off);
        if (s >= 0) {
            out += panel.ref[s];
        } else {
            const bool bare = down ? (off == -6 || off == -3 || off == -1) : (off == 10);
            out += bare ? "-" : "-|";
        }
    }
    return out;
}

int homopolymer_test(const std::string& down, const std::string& up, char sub) {  // VC:3615-3718
    int n[4] = {0, 0, 0, 0};
    const char* L = "ACGT";
    for (int b = 0; b < 4; ++b)
        if (sub == L[b]) n[b] = 1;
    for (const std::string* s : {&down, &up})
        for (char ch : *s)
            for (int b = 0; b < 4; ++b)
                if (ch == L[b]) ++n[b];
    for (int i = 0; i < 4; ++i)
        for (int j = i + 1; j < 4; ++j)
            if (n[i] + n[j] > 18) return 1;
    return 0;
}

// the long double Q of VC:3868-3882 from the double p the device produced
long double q_from_p(double p) {
    long double pvalue = p;
    long double p_limit = 0.0000000001;
    if (pvalue < p_limit) return -10 * log10l(p_limit);
    if (pvalue == 1) return 0;
    return -10 * log10l(pvalue);
}

int report_gpu_error(const char* what) {
    std::cout << RED << "Error: " << what << ": " << as_last_error() << RESET << std::endl;
    return 1;
}

void usage_bam() {
    std::cout << "\tA count directory that holds *.bam files and no *.ASEQ file is read as BAM input: every BAM is piled up on the GPU\n"
                 "\tas computeCounts would (sample name = file name minus .bam), with AS_BAM_MBQ / AS_BAM_MRQ / AS_BAM_MDC in the\n"
                 "\tenvironment for its mbq / mrq / mdc (default 20 / 20 / 20)."
              << std::endl;
}

void usage_ee() {
    std::cout << "Please type the following: " << std::endl;
    std::cout << "\n./AmpliSolveErrorEstimation" << GREEN << " panel_design=" << RESET << "/your/panel/design/file/in/bed/format" << GREEN
              << " reference_genome=" << RESET << "/your/reference/genome/in/fasta/format/indexed" << GREEN << " germline_dir=" << RESET
              << "/dir/with/normal/count/files/or/BAM/files" << GREEN << " C_value=" << RESET << "/C/value/of/the/error/model" << GREEN
              << " coverage_cutoff=" << RESET << "/coverage/per/strand" << GREEN << " default_error=" << RESET
              << "/platform/specific/error/used/without/normals" << GREEN << " output_dir=" << RESET << "/dir/to/store/all/outputs"
              << std::endl;
    std::cout << "\nExecution example:" << std::endl;
    std::cout << "./AmpliSolveErrorEstimation panel_design=panel.bed reference_genome=hg19.fasta germline_dir=NORMAL_ASEQ_DIR "
                 "C_value=0.002 coverage_cutoff=100 default_error=0.01 output_dir=ErrorEstimation_Testing"
              << std::endl;
    std::cout << "\n\tIt is important to give the arguments in this order. Otherwise the program will crach !" << std::endl;
    usage_bam();
    std::cout << STARS << std::endl;
}

void usage_vc() {
    std::cout << "Please type the following: " << std::endl;
    std::cout << "\n./AmpliSolveVariantCalling" << GREEN << " errorFile=" << RESET << "/the/file/produced/by/AmpliSolveErrorEstimation" << GREEN
              << " tumour_dir=" << RESET << "/your/dir/with/tumour/read/count/files/or/BAM/files " << GREEN << "output_dir=" << RESET
              << "/dir/to/store/all/outputs" << GREEN << " coverage_cutoff=" << RESET << "/coverage/per/strand/required/to/do/predictions"
              << GREEN << " p_value=" << RESET << "/Fisher's/exact/test/p/value/for/strand/bias" << std::endl;
    std::cout << "\nExecution example:" << std::endl;
    std::cout << "./AmpliSolveVariantCalling errorFile=positionSpecificNoise_0.0020.txt tumour_dir=TUMOUR_ASEQ_DIR "
                 "output_dir=VariantCalling_Testing coverage_cutoff=100 p_value=0.05"
              << std::endl;
    std::cout << "\n\tIt is important to give the arguments in this order. Otherwise the program will crach !" << std::endl;
    usage_bam();
    std::cout << "\tAn optional sixth argument " << GREEN << "sites=" << RESET << "/listed/SNVs.vcf writes <output_dir>/Site_Report.txt: the\n"
                 "\tstrand tests of every listed SNV in every tumour, called or not.  The file is VCF-like: '#' lines are skipped,\n"
                 "\tcolumns are CHROM POS ID REF ALT..., tab-separated; ALT may list several bases (A,T); records whose REF or ALT is\n"
                 "\tnot one base are skipped.  A site is tested at the first panel slot of its position.  Status: CALLED,\n"
                 "\tNOT_CALLED, LOW_COVERAGE, NO_DATA, NOT_TESTABLE, NOT_IN_PANEL or REF_MISMATCH."
              << std::endl;
    std::cout << STARS << std::endl;
}

void write_list_file(const std::string& path, const std::vector<std::string>& listed) {
    std::ofstream f(path.c_str());
    for (const std::string& s : listed) f << s << "\n";
}

void report_load(const std::vector<CountFile>& files, size_t first, const std::vector<AseqStats>& stats, bool noise_model) {
    for (size_t i = 0; i < stats.size(); ++i) {
        const AseqStats& s = stats[i];
        for (int64_t k = 0; k < s.bad_rd; ++k) std::cout << "malakia paizei edo" << std::endl;  // EE:1178-1181, VC:762-765
        if (s.bad_rd && noise_model)
            std::cout << "Warning: " << files[first + i].path << " has " << s.bad_rd << " row(s) whose RD column is not A+C+G+T; "
                      << "Germ_Max of their positions uses the sum of the counts, the reference the column" << std::endl;
    }
}

}  // namespace

extern "C" {

// fisherTest(FW, BW, alt_fw, alt_bw) of VC:3797-3814 as the variant-calling program evaluates it for every call
// (VC:902).  Host arithmetic only; pinned against Boost.Math's hypergeometric pdf in tests/test_oracle_golden.py.
double as_fisher_test(int32_t fw, int32_t bw, int32_t alt_fw, int32_t alt_bw) {
    if (fw < 0 || bw < 0 || alt_fw < 0 || alt_bw < 0) return -1.0;
    return fisher_test(fw, bw, alt_fw, alt_bw);
}

// The reference walks std::unordered_map<std::string,std::string> containers (EE:1081 normals, VC:672
// tumours, VC:1046 FILTER flags) and that order is visible in its outputs.  The only faithful model of
// libstdc++'s order is libstdc++: insert the same keys in the same sequence, read the order back.
int as_hash_iteration_order(const char* const* keys, int32_t n, int32_t* order_out) {
    if (!keys || !order_out || n < 0) return AS_EINVAL;
    std::unordered_map<std::string, std::string> m;
    std::unordered_map<std::string, int32_t> first;
    for (int32_t i = 0; i < n; ++i) {
        m.insert(std::make_pair(std::string(keys[i]), std::string()));
        first.insert(std::make_pair(std::string(keys[i]), i));
    }
    int32_t j = 0;
    for (auto it = m.begin(); it != m.end(); ++it) order_out[j++] = first[it->first];
    return j;
}

// ===================================================================================================
// AmpliSolveErrorEstimation (EE:241-520)
// ===================================================================================================
int as_error_estimation_main(int argc, char** argv) {
    if (argc != 8) {
        std::cout << STARS << std::endl;
        std::cout << RED << "                                        Your input arguments are not correct !" << RESET << std::endl;
        std::cout << "                         amplisolve_b200 (B200-native AmpliSolveErrorEstimation, argv-compatible)\n" << std::endl;
        usage_ee();
        return 0;
    }
    const std::string panel_design = arg_value(argv[1], "panel_design=");
    const std::string reference_genome = arg_value(argv[2], "reference_genome=");
    const std::string germline_dir = arg_value(argv[3], "germline_dir=");
    const std::string C_value = arg_value(argv[4], "C_value=");
    const std::string coverage_cutoff = arg_value(argv[5], "coverage_cutoff=");
    const std::string default_error = arg_value(argv[6], "default_error=");
    const std::string output_dir = arg_value(argv[7], "output_dir=");
    float C_value_float = (float)atof(C_value.c_str());  // EE:329
    // C_value=a,b,c: a noise-floor sweep, one table per value from one parse of the normals.  Every element is converted
    // like a single value (atof, <= 0 -> 0.002); a value without a comma takes the single-value path unchanged.
    const bool sweep = C_value.find(',') != std::string::npos;
    std::vector<std::string> c_texts;
    std::vector<float> c_values;
    if (sweep) {
        for (size_t b = 0;;) {
            const size_t e = C_value.find(',', b);
            c_texts.push_back(C_value.substr(b, e == std::string::npos ? std::string::npos : e - b));
            if (e == std::string::npos) break;
            b = e + 1;
        }
        std::vector<std::string> names;
        for (const std::string& t : c_texts) {
            if (t.empty()) {
                std::cout << "Error: C_value=" << C_value << " has an empty value" << std::endl;
                return 0;
            }
            float v = (float)atof(t.c_str());
            if (v <= 0) v = 0.002f;
            char name[64];
            snprintf(name, sizeof name, "%.4f", v);
            if (std::find(names.begin(), names.end(), name) != names.end()) {
                std::cout << "Error: C_value=" << C_value << ": " << t << " gives positionSpecificNoise_" << name
                          << ".txt a second time" << std::endl;
                return 0;
            }
            names.push_back(name);
            c_values.push_back(v);
        }
    }
    int cut = atoi(coverage_cutoff.c_str());
    const bool with_germlines = germline_dir != "not_available";  // EE:349
    float default_error_float = 0.01f;

    std::cout << STARS << "\n" << std::endl;
    std::cout << "                                Error estimation required for AmpliSolveVariantCalling program \n" << std::endl;
    std::cout << "                        amplisolve_b200: B200-native implementation (" << as_version() << ")\n" << std::endl;
    std::cout << "Execution started under the following parameters:" << std::endl;
    std::cout << "\t1. Panel design                                   : " << GREEN << panel_design << RESET << std::endl;
    std::cout << "\t2. Reference genome                               : " << GREEN << reference_genome << RESET << std::endl;
    if (!with_germlines) {
        default_error_float = (float)atof(default_error.c_str());
        if (default_error_float > 0) {
            std::cout << "\t3. Germline count dir                             : " << RED << "NO germline count files available" << RESET
                      << ". Estimation of error is based on platform-specific error level given by user equal to "
                      << default_error_float << std::endl;
        } else {
            default_error_float = 0.01f;  // EE:359-362
            std::cout << "\t3. Germline count dir                             : " << RED << "NO germline count files available" << RESET
                      << ". User gave wrong platform-specific error level and the estimation will be based on Error="
                      << default_error_float << std::endl;
        }
    } else {
        std::cout << "\t3. Germline count dir                             : " << GREEN << germline_dir << RESET << std::endl;
    }
    if (sweep) {
        std::cout << "\t4. C values                                       : " << GREEN;
        for (size_t i = 0; i < c_values.size(); ++i) {
            if (i) std::cout << ",";
            std::cout << c_values[i];
        }
        std::cout << RESET;
        for (size_t i = 0; i < c_values.size(); ++i)
            if ((float)atof(c_texts[i].c_str()) <= 0) std::cout << ". User gave: " << c_texts[i] << ", converted to 0.002";
        std::cout << std::endl;
    } else if (C_value_float <= 0) {
        C_value_float = 0.002f;  // EE:372-376
        std::cout << "\t4. C value                                         : " << RED << "User gave: " << C_value << RESET
                  << ". The value is converted to 0.002" << std::endl;
    } else {
        std::cout << "\t4. C value                                        : " << GREEN << C_value_float << RESET << std::endl;
    }
    if (cut <= 0) {
        cut = 100;  // EE:383-387
        std::cout << "\t5. Coverage cutoff                                  : " << RED << "User gave: " << coverage_cutoff << RESET
                  << ". The value is converted 100" << std::endl;
    } else {
        std::cout << "\t5. Coverage cutoff                                : " << GREEN << cut << RESET << std::endl;
    }
    std::cout << "\t6. Output dir                                     : " << GREEN << output_dir << RESET << std::endl;
    const bool bam_input = with_germlines && bam_input_dir(germline_dir);
    BamInput bam;
    if (bam_input)
        std::cout << "\t7. BAM pileup (AS_BAM_MBQ / AS_BAM_MRQ / AS_BAM_MDC) : " << GREEN << bam.mbq << " / " << bam.mrq << " / " << bam.mdc
                  << RESET << std::endl;

    const std::string interm = output_dir + "/AmpliSolveErrorEstimation_interm_files";
    if (!make_dir(interm)) {
        std::cout << "Error: cannot create " << interm << std::endl;
        return 0;
    }
    GpuContext gpu;  // CUDA start-up runs beside the panel / reference-base work below (no CPU fallback: see as_create)
    if (with_germlines) gpu.start(aseq_dir_records(germline_dir));
    srand((unsigned)time(nullptr));
    const int seed = rand() % 1000;  // EE:581-584
    const std::string stem = interm + "/" + std::to_string(seed);

    // panel enumeration, reference bases, duplicated positions (replaces generateReferenceBases, EE:578-670)
    PhaseTimer timer;
    std::cout << "\nRunning function generateReferenceBases: ";
    Panel panel;
    int n_amplicons = 0;
    if (!load_bed(panel_design, panel, n_amplicons)) {
        printf("Error from generateReferenceBases: Cannot open file: %s\n", panel_design.c_str());
        return 0;
    }
    panel.link();
    std::string err;
    if (!annotate_reference(reference_genome, panel, err)) {
        std::cout << "Error from generateReferenceBases: " << err << std::endl;
        return 0;
    }
    const int64_t P = panel.size();
    panel.dup.assign(P, 0);
    for (int64_t i = 0; i < P; ++i)
        if (panel.twin_next[i] >= 0 || panel.twin_head[i] != (int32_t)i) panel.dup[i] = 1;
    {
        // the two intermediate lists, formatted into one string each (an ostream insertion per field was a third of this phase)
        std::string text;
        text.reserve((size_t)P * 24);
        char num[16];
        for (int64_t i = 0; i < P; ++i) {
            text += panel.chroms[panel.slot_chrom[i]];
            text += '\t';
            text.append(num, (size_t)snprintf(num, sizeof num, "%d", panel.slot_pos[i]));
            text += '\t';
            text += panel.ref[i];
            text += '\n';
        }
        std::ofstream refs((stem + "_panelReferenceBases.txt").c_str());
        refs.write(text.data(), (std::streamsize)text.size());
        text.clear();
        for (int64_t i = 0; i < P; ++i)
            if (panel.dup[i] && panel.twin_head[i] == (int32_t)i) {
                text += panel.chroms[panel.slot_chrom[i]];
                text += '\t';
                text.append(num, (size_t)snprintf(num, sizeof num, "%d", panel.slot_pos[i]));
                text += '\n';
            }
        std::ofstream dups((stem + "_ampliconDuplicatedPositions.txt").c_str());
        dups.write(text.data(), (std::streamsize)text.size());
    }
    std::cout << "Reference bases and amplicon duplicated positions have generated" << "\n\t\t --> Parsed in total " << n_amplicons
              << " amplicons and annotated " << P << " positions." << std::endl;
    std::cout << "Running function storeReference: panel reference bases stored with success " << GREEN << panel.n_positions
              << RESET << std::endl;

    timer.lap("panel_and_reference_bases", (double)P, "positions");
    const char* header =
        "chrom\tposition\treference\tduplicate\tThres_A\tThres_C\tThres_G\tThres_T\tGerm_Max_A\tGerm_Max_C\tGerm_Max_G\tGerm_Max_T";
    if (!with_germlines) {
        // generateFinalOutput_default (EE:2948-3043)
        const std::string out_name = output_dir + "/positionSpecificNoise_default.txt";
        std::ofstream output(out_name.c_str());
        output << header << "\n";
        char value[64];
        snprintf(value, sizeof value, "%.4f_%.4f", default_error_float, default_error_float);
        for (int64_t i = 0; i < P; ++i) {
            output << panel.chroms[panel.slot_chrom[i]] << "\t" << panel.slot_pos[i] << "\t" << panel.ref[i];
            output << "\t" << (panel.dup[i] ? "YES" : "NO");
            output << "\t" << value << "\t" << value << "\t" << value << "\t" << value << "\t-\t-\t-\t-" << "\n";
        }
        std::cout << "\nAmpliSolveErrorEstimation execution was successful. Results can be found at: " << YELLOW << out_name << RESET
                  << std::endl;
        std::cout << "\n" << STARS << std::endl;
        return 0;
    }

    // normals in the reference's file order
    std::vector<CountFile> files;
    std::vector<std::string> listed;
    bool bam_files = false;
    if (!list_count_files(germline_dir, files, listed, &bam_files)) {
        std::cout << "Error: cannot list " << germline_dir << "/*.ASEQ" << std::endl;
        return 0;
    }
    write_list_file(stem + "_germline_count_list_original.txt", listed);
    std::cout << "\nRunning function storeList: " << GREEN << stem << "_germline_count_list_original.txt" << RESET
              << " stored with success. It contains " << GREEN << files.size() << RESET << " samples" << std::endl;
    const int S = (int)files.size();
    if (!gpu.wait()) {  // without a B200 there is nothing this program can do (no CPU fallback)
        std::cout << RED << "Error: as_create: " << gpu.error << RESET << std::endl;
        return 1;
    }
    as_ctx* ctx = gpu.ctx;
    timer.lap("cuda_context_wait");
    std::cout << "Running function storeGermlineStatistics:" << std::endl;
    HostCounts counts;
    std::vector<AseqStats> stats;
    if (bam_files) bam.setup(panel);  // the pileups run on this program's context: nothing else uses it meanwhile
    const int lrc = bam_files ? load_bam_counts(files, 0, files.size(), panel, bam, ctx, counts, stats)
                              : load_counts(files, 0, files.size(), panel, counts, stats);
    if (lrc == 1) return report_gpu_error("pinned host allocation");
    if (lrc == 3) return 0;  // a BAM that cannot be read: reported like an ASEQ file that cannot be opened
    if (lrc == 2) {
        for (int i = 0; i < S; ++i)
            if (!stats[i].ok) printf("Error: Cannot open %s\n", files[i].path.c_str());
        return 0;
    }
    report_load(files, 0, stats, true);
    {
        double rows = 0;
        for (const AseqStats& st : stats) rows += (double)st.rows;
        timer.lap(bam_files ? "pileup_normals" : "parse_normals", rows, "rows");
    }

    std::cout << "Running function estimateThresholds: ";
    std::vector<int32_t> links_next, links_head;
    const int64_t PS = add_spill_slots(panel, counts, stats, links_next, links_head);  // P + spill slots for rows beyond the panel's slots
    if (PS < 0) return report_gpu_error("pinned host allocation");
    if (!sweep) c_values.assign(1, C_value_float);
    const size_t n_tables = c_values.size();
    std::vector<float> thr(n_tables * (size_t)PS * 8), germ_val((size_t)PS * 4);
    std::vector<uint8_t> germ_state((size_t)PS * 4);
    std::vector<uint32_t> count((size_t)PS * 4), nrec((size_t)PS);
    const bool linked = panel.has_twins || PS > P;
    const int32_t* tn = linked ? links_next.data() : nullptr;
    const int32_t* th = linked ? links_head.data() : nullptr;
    for (size_t c0 = 0; c0 < n_tables; c0 += 8) {  // at most 8 values of C per pass over the normals
        const int32_t nc = (int32_t)std::min<size_t>(8, n_tables - c0);
        float* thr_c = thr.data() + c0 * (size_t)PS * 8;
        const int rc = counts.fmt == 2
                           ? as_noise_estimate_sweep_host16(ctx, (const uint16_t*)counts.p, counts.wide.data(), (int64_t)counts.wide.size(),
                                                            S, PS, tn, th, &c_values[c0], nc, cut, thr_c, germ_val.data(),
                                                            germ_state.data(), count.data(), nrec.data(), nullptr)
                           : as_noise_estimate_sweep_host_packed(ctx, (const uint32_t*)counts.p, counts.wide.data(),
                                                                 (int64_t)counts.wide.size(), S, PS, tn, th, &c_values[c0], nc, cut,
                                                                 thr_c, germ_val.data(), germ_state.data(), count.data(), nrec.data(),
                                                                 nullptr);
        if (rc != AS_OK) return report_gpu_error("as_noise_estimate_host");
    }
    timer.lap("noise_model_gpu", (double)P * (double)n_tables, "positions");
    std::cout << "thresholds for " << panel.n_positions << " positions estimated on the GPU" << std::endl;

    // generateFinalOutput (EE:2546-2944), one table per value of C
    char out_name[4096];
    for (size_t ti = 0; ti < n_tables; ++ti) {
        snprintf(out_name, sizeof out_name, "%s/positionSpecificNoise_%.4f.txt", output_dir.c_str(), c_values[ti]);
        const float* thr_t = thr.data() + ti * (size_t)PS * 8;
        // rows are formatted in chunks on all host threads (2 M rows took 2.7 s on one: "%f" eight times a row) and written
        // in order; the bytes are what the reference's streams produce: "%f" (EE:1787), operator<<(double) = "%g" (EE:2815)
        std::ofstream output(out_name);
        output << header << "\n";
        // chunk size: every thread gets a few chunks also on a small panel
        const int64_t CH = std::max<int64_t>(512, std::min<int64_t>(16384, P / (4 * (int64_t)std::max(1u, std::thread::hardware_concurrency()))));
        const size_t n_chunks = (size_t)((P + CH - 1) / CH);
        const size_t WAVE = 256;  // chunks formatted before they are written: bounds the text held in memory
        std::vector<std::string> text(std::min(n_chunks, WAVE));
        for (size_t w0 = 0; w0 < n_chunks; w0 += WAVE) {
            const size_t wn = std::min(WAVE, n_chunks - w0);
            std::atomic<size_t> next(0);
            auto work = [&]() {
                const char* L = "ACGT";
                char cell[160];
                for (size_t k = next.fetch_add(1); k < wn; k = next.fetch_add(1)) {
                    std::string& o = text[k];
                    o.clear();
                    const int64_t i0 = (int64_t)(w0 + k) * CH, i1 = std::min(P, i0 + CH);
                    for (int64_t i = i0; i < i1; ++i) {
                        o += panel.chroms[panel.slot_chrom[i]];
                        o += '\t';
                        o += std::to_string(panel.slot_pos[i]);
                        o += '\t';
                        o += panel.ref[i];
                        o += panel.dup[i] ? "\tYES" : "\tNO";
                        for (int b = 0; b < 4; ++b) {
                            const float tf = thr_t[(size_t)i * 8 + b * 2], tb = thr_t[(size_t)i * 8 + b * 2 + 1];
                            if (panel.ref[i].size() == 1 && panel.ref[i][0] == L[b]) {
                                o += "\t-2_-2";  // EE:2668-2673
                            } else if (std::isnan(tf) || std::isnan(tb)) {
                                o += "\t0.01_0.01";  // "-1_-1" -> EE:2680-2684
                            } else {
                                o += '\t';  // "%f_%f", EE:1787
                                append_percent_f(o, tf);
                                o += '_';
                                append_percent_f(o, tb);
                            }
                        }
                        for (int b = 0; b < 4; ++b) {
                            if (germ_state[(size_t)i * 4 + b] == 0) {
                                o += "\t-";  // EE:2807-2849
                            } else {  // ostream << double
                                o += '\t';
                                const float g = germ_val[(size_t)i * 4 + b];
                                if (g == 0.f && !std::signbit(g)) {
                                    o += '0';
                                } else if (!append_percent_g(o, g)) {
                                    snprintf(cell, sizeof cell, "%g", (double)g);
                                    o += cell;
                                }
                            }
                        }
                        o += '\n';
                    }
                }
            };
            run_on_threads((unsigned)std::max<size_t>(1, std::min<size_t>(std::thread::hardware_concurrency(), wn)), work);
            for (size_t k = 0; k < wn; ++k) output.write(text[k].data(), (std::streamsize)text[k].size());
        }
    }
    timer.lap("write_noise_table", (double)P * (double)n_tables, "rows");
    char msg_name[4096];
    if (sweep) {
        std::cout << "\nAmpliSolveErrorEstimation execution was successful. Results can be found at:";
        for (const float v : c_values) {
            snprintf(msg_name, sizeof msg_name, "%s/positionSpecificNoise_%.4f.txt", output_dir.c_str(), v);
            std::cout << " " << YELLOW << msg_name << RESET;
        }
        std::cout << std::endl;
    } else {
        snprintf(msg_name, sizeof msg_name, "%s/positionSpecific_%.4f.txt", output_dir.c_str(), C_value_float);  // sic, EE:458
        std::cout << "\nAmpliSolveErrorEstimation execution was successful. Results can be found at: " << YELLOW << msg_name << RESET
                  << std::endl;
    }
    std::cout << "\n" << STARS << std::endl;
    return 0;
}

namespace {
// ---------------------------------------------------------------------------------------------------
// The noise table of the error-estimation program (storeInputFile, VC:430-576): one panel slot per row -- chrom, position,
// reference, duplicated flag, four threshold cells "<fw>_<bw>", four Germ_Max cells.  Fills the panel's slot arrays,
// thr_view [P][4][2] (std::stof of the cells, VC:889-890), germ_text [P][4] and the text of dummyVCF_1.vcf (VC:564) in
// pieces to be written one after the other.  force_pieces > 0 fixes the number of pieces (tests).
// ---------------------------------------------------------------------------------------------------
void parse_noise_table(const std::string& text, int force_pieces, Panel& panel, std::vector<float>& thr_view,
                       std::vector<std::string>& germ_text, std::vector<std::string>& dummy_pieces) {
    // The table is cut into pieces at line ends and parsed on all host threads (a 2,000,000-row table is 170 MB of text:
    // one thread needs 1.4 s for it, most of it in strtof).  Pass 1 counts the rows of every piece and collects its
    // chromosome names in order of appearance; the names are registered piece by piece, so ids follow the first
    // appearance in the file as a sequential parse gives them; pass 2 writes every row at its final index.
    const char* p = text.data();
    const char* e = p + text.size();
    const char* eol = (const char*)memchr(p, '\n', e - p);  // header
    p = eol ? eol + 1 : e;
    const size_t body = (size_t)(e - p);
    const unsigned n_piece = force_pieces > 0 ? (unsigned)force_pieces
                                              : (unsigned)std::max<size_t>(1, std::min<size_t>(std::max(1u, std::thread::hardware_concurrency()), body / (256 << 10)));
    std::vector<const char*> cut_at(n_piece + 1, e);
    cut_at[0] = p;
    for (unsigned k = 1; k < n_piece; ++k) {
        const char* c = p + body * k / n_piece;
        c = std::max(c, cut_at[k - 1]);
        const char* nl = c < e ? (const char*)memchr(c, '\n', (size_t)(e - c)) : nullptr;
        cut_at[k] = nl ? nl + 1 : e;
    }
    struct Piece {
        size_t rows = 0;
        std::vector<std::string> names;  // distinct chromosome names in order of appearance
        std::string dummy;               // this piece of dummyVCF_1.vcf (VC:564)
    };
    std::vector<Piece> pieces(n_piece);
    auto run_pieces = [&](const std::function<void(unsigned)>& f) {
        std::atomic<unsigned> next(0);
        run_on_threads(n_piece, [&]() {
            for (unsigned k = next.fetch_add(1); k < n_piece; k = next.fetch_add(1)) f(k);
        });
    };
    run_pieces([&](unsigned k) {
        Piece& pc = pieces[k];
        const char* last_b = nullptr;
        size_t last_n = 0;
        for (const char* c = cut_at[k]; c < cut_at[k + 1];) {
            const char* le = (const char*)memchr(c, '\n', (size_t)(cut_at[k + 1] - c));
            if (!le) le = cut_at[k + 1];
            const char* q = skip_ws(c, le);
            const char* t = token_end(q, le);
            if (t > q) {
                ++pc.rows;
                const size_t cn = (size_t)(t - q);
                if (!last_b || cn != last_n || memcmp(last_b, q, cn) != 0) {
                    last_b = q;
                    last_n = cn;
                    std::string name(q, t);
                    if (std::find(pc.names.begin(), pc.names.end(), name) == pc.names.end()) pc.names.push_back(name);
                }
            }
            c = le + 1;
        }
    });
    size_t rows = 0;
    std::vector<size_t> first_row(n_piece + 1, 0);
    for (unsigned k = 0; k < n_piece; ++k) {
        for (const std::string& name : pieces[k].names) panel.chrom_id(name);
        first_row[k] = rows;
        rows += pieces[k].rows;
    }
    first_row[n_piece] = rows;
    panel.slot_chrom.resize(rows); panel.slot_pos.resize(rows); panel.pos_text.resize(rows); panel.ref.resize(rows);
    panel.dup.resize(rows); thr_view.resize(rows * 8); germ_text.resize(rows * 4);
    const Panel& names = panel;  // pass 2 only reads the name table
    run_pieces([&](unsigned k) {
        Piece& pc = pieces[k];
        pc.dummy.reserve((size_t)(cut_at[k + 1] - cut_at[k]) / 3);
        size_t row = first_row[k];
        const char* last_chrom_b = nullptr;
        size_t last_chrom_n = 0;
        int32_t last_chrom_id = -1;
        for (const char* c = cut_at[k]; c < cut_at[k + 1];) {
            const char* le = (const char*)memchr(c, '\n', (size_t)(cut_at[k + 1] - c));
            if (!le) le = cut_at[k + 1];
            const char* fb[12];
            const char* fe[12];
            const char* q = c;
            int nf = 0;
            for (; nf < 12; ++nf) {
                q = skip_ws(q, le);
                const char* t = token_end(q, le);
                if (t == q) break;
                fb[nf] = q;
                fe[nf] = t;
                q = t;
            }
            for (int f = nf; f < 12; ++f) fb[f] = fe[f] = le;  // missing fields read as empty strings
            if (nf >= 1) {
                const size_t cn = (size_t)(fe[0] - fb[0]);
                if (last_chrom_id < 0 || cn != last_chrom_n || memcmp(last_chrom_b, fb[0], cn) != 0) {
                    last_chrom_id = names.find_chrom(fb[0], cn);
                    last_chrom_b = fb[0];
                    last_chrom_n = cn;
                }
                panel.slot_chrom[row] = last_chrom_id;
                panel.slot_pos[row] = (int32_t)strtol(fb[1], nullptr, 10);  // fields end at a blank, a tab or the line end: strtol stops there
                panel.pos_text[row].assign(fb[1], fe[1]);
                panel.ref[row].assign(fb[2], fe[2]);
                panel.dup[row] = (fe[3] - fb[3] == 3 && memcmp(fb[3], "YES", 3) == 0) ? 1 : 0;
                for (int b = 0; b < 4; ++b) {
                    // a threshold cell "<fw>_<bw>" as sscanf("%[^_]_%[^_]") + std::stof read it (VC:888-890); no copies
                    const char* cb = fb[4 + b];
                    const char* ce = fe[4 + b];
                    const char* us = (const char*)memchr(cb, '_', (size_t)(ce - cb));
                    float a = 0.f, bwv = 0.f;
                    if (us) {
                        const char* us2 = (const char*)memchr(us + 1, '_', (size_t)(ce - us - 1));  // %[^_] stops at a second '_'
                        a = threshold_text_to_float(cb, us);
                        bwv = threshold_text_to_float(us + 1, us2 ? us2 : ce);
                    }
                    thr_view[row * 8 + (size_t)b * 2] = a;
                    thr_view[row * 8 + (size_t)b * 2 + 1] = bwv;
                    germ_text[row * 4 + (size_t)b].assign(fb[8 + b], fe[8 + b]);
                }
                pc.dummy.append(fb[0], fe[0]).push_back('\t');
                pc.dummy.append(fb[1], fe[1]).append("\t.\t.\t.\t.\t.\t.\n");
                ++row;
            }
            c = le + 1;
        }
    });
    dummy_pieces.clear();
    for (Piece& pc : pieces) dummy_pieces.push_back(std::move(pc.dummy));
}

// ---------------------------------------------------------------------------------------------------
// sites=<file> of the variant-calling program: listed SNVs whose strand tests are reported for every tumour, called or not
// (Site_Report.txt).  VCF-like text: '#' lines are skipped, columns are CHROM POS ID REF ALT..., tab-separated, so a
// program's own <sample>.vcf or a hotspot list is read as is; an ALT list "A,T" gives one site per base.
// ---------------------------------------------------------------------------------------------------
enum { SITE_NOT_IN_PANEL = 6, SITE_REF_MISMATCH = 7 };  // statuses set on the host, after the AS_SITE_* of the device
const char* site_status_text(int32_t st) {
    switch (st) {
        case AS_SITE_CALLED: return "CALLED";
        case AS_SITE_NOT_CALLED: return "NOT_CALLED";
        case AS_SITE_LOW_COVERAGE: return "LOW_COVERAGE";
        case AS_SITE_NO_DATA: return "NO_DATA";
        case AS_SITE_NOT_TESTABLE: return "NOT_TESTABLE";
        case SITE_NOT_IN_PANEL: return "NOT_IN_PANEL";
        default: return "REF_MISMATCH";
    }
}

struct SiteList {
    std::vector<std::string> chrom, pos_text;  // as the file writes them
    std::vector<long> pos;
    std::vector<char> ref, alt;
    // resolve_sites: the first panel slot of the site's position, the status set on the host (0: tested on the device) and
    // the site's index among the tested ones
    std::vector<int32_t> slot, host_status, dev;
    std::vector<int32_t> dev_slot, dev_alt;  // the tested sites
};

// 0 ok, 1 the file cannot be opened, 2 a malformed line (reported)
int load_sites(const std::string& path, SiteList& sl) {
    std::string text;
    if (!read_file(path, text)) return 1;
    auto split = [](const std::string& s, char sep, size_t max_parts) {
        std::vector<std::string> v;
        for (size_t a = 0;;) {
            const size_t b = v.size() + 1 == max_parts ? std::string::npos : s.find(sep, a);
            v.push_back(s.substr(a, b == std::string::npos ? std::string::npos : b - a));
            if (b == std::string::npos) return v;
            a = b + 1;
        }
    };
    auto base = [](const std::string& b) { return b.size() == 1 && strchr("ACGT", b[0]) != nullptr; };
    size_t line = 0;
    for (size_t p = 0; p < text.size();) {
        size_t e = text.find('\n', p);
        if (e == std::string::npos) e = text.size();
        std::string ln = text.substr(p, e - p);
        p = e + 1;
        ++line;
        if (!ln.empty() && ln.back() == '\r') ln.pop_back();
        if (ln.empty() || ln[0] == '#') continue;
        const std::vector<std::string> col = split(ln, '\t', 6);
        if (col.size() < 5) {
            printf("Error: %s line %zu has fewer than five tab-separated columns (CHROM POS ID REF ALT)\n", path.c_str(), line);
            return 2;
        }
        char* end = nullptr;
        errno = 0;
        const long pos = strtol(col[1].c_str(), &end, 10);
        if (col[1].empty() || *end != '\0' || errno != 0) {
            printf("Error: %s line %zu: POS \"%s\" is not an integer\n", path.c_str(), line, col[1].c_str());
            return 2;
        }
        const std::vector<std::string> alt = split(col[4], ',', 0);
        bool snv = base(col[3]);
        for (const std::string& x : alt) snv = snv && base(x);
        if (!snv) {
            std::cout << "Warning: " << path << " line " << line << ": REF or ALT is not a single base (A, C, G, T); record skipped"
                      << std::endl;
            continue;
        }
        for (const std::string& x : alt) {
            sl.chrom.push_back(col[0]);
            sl.pos_text.push_back(col[1]);
            sl.pos.push_back(pos);
            sl.ref.push_back(col[3][0]);
            sl.alt.push_back(x[0]);
        }
    }
    return 0;
}

// Sites -> panel slots: CHROM is matched as text against the noise table's names; a site is tested at the FIRST slot of its
// position (rows beyond a position's slots are not reported) and its REF must be the panel's reference text.
void resolve_sites(const Panel& panel, SiteList& sl) {
    const size_t n = sl.chrom.size();
    sl.slot.assign(n, -1);
    sl.host_status.assign(n, 0);
    sl.dev.assign(n, -1);
    for (size_t i = 0; i < n; ++i) {
        const int32_t c = panel.find_chrom(sl.chrom[i].data(), sl.chrom[i].size());
        const int32_t s = (c < 0 || sl.pos[i] != (long)(int32_t)sl.pos[i]) ? -1 : panel.lookup(c, (int32_t)sl.pos[i]);
        if (s < 0) { sl.host_status[i] = SITE_NOT_IN_PANEL; continue; }
        sl.slot[i] = s;
        if (panel.ref[(size_t)s] != std::string(1, sl.ref[i])) { sl.host_status[i] = SITE_REF_MISMATCH; continue; }
        sl.dev[i] = (int32_t)sl.dev_slot.size();
        sl.dev_slot.push_back(s);
        sl.dev_alt.push_back((int32_t)(strchr("ACGT", sl.alt[i]) - "ACGT"));
    }
}

// A row whose RD column is not A+C+G+T: the reference's forward-strand test takes (alt_fw, RD - reverse reads) (VC:895),
// so the row goes to the device with the reference base's forward count absorbing the difference (alt counts untouched).
// False when the column is too small for that (rb = the slot's reference base, 0..3).
bool rd_column_forward(const AseqStats::ExtraRow& x, uint8_t rb, uint32_t& ref_fw) {
    long long FW = 0, BW = 0;
    for (int b = 0; b < 4; ++b) { FW += x.fw[b]; BW += x.bw[b]; }
    const long long v = (long long)x.fw[rb] + (x.rd - (FW + BW));
    if (v < 0 || x.rd - BW < 1) return false;
    ref_fw = (uint32_t)v;
    return true;
}

}  // namespace

// ===================================================================================================
// AmpliSolveVariantCalling (VC:199-360, VC:430-576, VC:633-3304)
// ===================================================================================================
int as_variant_calling_main(int argc, char** argv) {
    if ((argc != 6 && argc != 7) || (argc == 7 && strncmp(argv[6], "sites=", 6) != 0)) {
        std::cout << STARS << std::endl;
        std::cout << RED << "                                        Your input arguments are not correct !" << RESET << std::endl;
        std::cout << "                         amplisolve_b200 (B200-native AmpliSolveVariantCalling, argv-compatible)\n" << std::endl;
        usage_vc();
        return 0;
    }
    const std::string error_file = arg_value(argv[1], "errorFile=");
    const std::string tumour_dir = arg_value(argv[2], "tumour_dir=");
    const std::string output_dir = arg_value(argv[3], "output_dir=");
    const std::string coverage_cutoff = arg_value(argv[4], "coverage_cutoff=");
    const std::string p_value = arg_value(argv[5], "p_value=");
    const std::string sites_file = argc == 7 ? arg_value(argv[6], "sites=") : std::string();
    float p_value_float = (float)atof(p_value.c_str());  // VC:263
    int cut = atoi(coverage_cutoff.c_str());

    std::cout << STARS << "\n" << std::endl;
    std::cout << "                          AmpliSolve variant calling for batch execution of multiple samples\n" << std::endl;
    std::cout << "                        amplisolve_b200: B200-native implementation (" << as_version() << ")\n" << std::endl;
    std::cout << "Execution started under the following parameters:" << std::endl;
    std::cout << "\t1. Error estimation                               : " << GREEN << error_file << RESET << std::endl;
    std::cout << "\t2. Tumour count dir                               : " << GREEN << tumour_dir << RESET << std::endl;
    std::cout << "\t3. Output dir                                     : " << GREEN << output_dir << RESET << std::endl;
    if (cut <= 0) {
        cut = 100;  // VC:277-281
        std::cout << "\t4. Coverage cutoff                                  : " << RED << "User gave: " << coverage_cutoff << RESET
                  << ". The value is converted to default 100" << std::endl;
    } else {
        std::cout << "\t4. Coverage cutoff                                : " << GREEN << cut << RESET << std::endl;
    }
    if (p_value_float <= 0 || p_value_float > 1) {
        p_value_float = 0.05f;  // VC:289-293
        std::cout << "\t5. p-value                                         : " << RED << "User gave: " << p_value << RESET
                  << ". The value is converted to default 0.05" << std::endl;
    } else {
        std::cout << "\t5. p-value                                        : " << GREEN << p_value_float << RESET << std::endl;
    }
    BamInput bam;
    if (bam_input_dir(tumour_dir))
        std::cout << "\t6. BAM pileup (AS_BAM_MBQ / AS_BAM_MRQ / AS_BAM_MDC) : " << GREEN << bam.mbq << " / " << bam.mrq << " / " << bam.mdc
                  << RESET << std::endl;
    if (argc == 7)
        std::cout << "\t" << (bam_input_dir(tumour_dir) ? 7 : 6) << ". Sites (Site_Report.txt)                        : " << GREEN << sites_file
                  << RESET << std::endl;
    std::cout << std::endl;
    // sites=<file>: read before anything is written, so that a malformed file leaves no output behind
    SiteList sites;
    if (argc == 7) {
        const int src = load_sites(sites_file, sites);
        if (src == 1) printf("Error from the sites file: Cannot open %s\n", sites_file.c_str());
        if (src != 0) return 0;
    }

    // errorFile=<directory>: a noise-floor sweep over every positionSpecificNoise_*.txt in it, in name order.  Table X.txt
    // writes to <output_dir>/X/ what errorFile=<directory>/X.txt output_dir=<output_dir>/X writes alone; the tumours are
    // parsed (or piled up) once and go through the caller once per pass of up to 8 tables.
    std::vector<std::string> table_paths, out_dirs;
    struct stat est;
    const bool sweep = stat(error_file.c_str(), &est) == 0 && S_ISDIR(est.st_mode);
    if (sweep) {
        std::vector<std::string> names;
        if (DIR* d = opendir(error_file.c_str())) {
            const std::string pre = "positionSpecificNoise_";
            while (dirent* de = readdir(d)) {
                const std::string n = de->d_name;
                if (n.size() > pre.size() + 4 && n.compare(0, pre.size(), pre) == 0 && ends_with(n, ".txt")) names.push_back(n);
            }
            closedir(d);
        }
        std::sort(names.begin(), names.end());
        if (names.empty()) {
            printf("Error from storeInputFile function: Cannot open %s\n", error_file.c_str());
            return 0;
        }
        for (const std::string& n : names) {
            table_paths.push_back(error_file + "/" + n);
            out_dirs.push_back(output_dir + "/" + n.substr(0, n.size() - 4));
        }
    } else {
        table_paths.push_back(error_file);
        out_dirs.push_back(output_dir);
    }
    const size_t NT = table_paths.size();
    const std::string interm_name = "/AmpliSolveVariantCalling_interm_files";
    if (!sweep && !make_dir(output_dir + interm_name)) {  // a sweep creates its directories once the tables agree
        std::cout << "Error: cannot create " << output_dir + interm_name << std::endl;
        return 0;
    }

    GpuContext gpu;  // CUDA start-up runs beside the parse of the noise table (no CPU fallback: see as_create)
    gpu.start(aseq_dir_records(tumour_dir));
    PhaseTimer timer;
    // ---- noise table (storeInputFile, VC:430-576): one slot per row; also re-emits the dummy VCF (VC:564)
    Panel panel;
    std::vector<float> thr_view;                         // [NT][P][4][2] through std::stof (VC:889-890)
    std::vector<std::vector<std::string>> germ_texts(NT);  // [NT][P][4]
    std::vector<std::vector<std::string>> dummy_pieces(NT);  // dummyVCF_1.vcf (VC:564) of every table
    for (size_t k = 0; k < NT; ++k) {
        std::string text;
        if (!read_file(table_paths[k], text)) {
            printf("Error from storeInputFile function: Cannot open %s\n", table_paths[k].c_str());
            return 0;
        }
        if (k == 0) {
            parse_noise_table(text, 0, panel, thr_view, germ_texts[0], dummy_pieces[0]);
            continue;
        }
        // the tables of a sweep must describe the same panel; their thresholds and Germ_Max cells may differ
        Panel pk;
        std::vector<float> tv;
        parse_noise_table(text, 0, pk, tv, germ_texts[k], dummy_pieces[k]);
        const size_t rows = panel.slot_pos.size(), rows_k = pk.slot_pos.size();
        size_t bad = std::min(rows, rows_k);
        for (size_t r = 0; r < std::min(rows, rows_k); ++r)
            if (panel.chroms[(size_t)panel.slot_chrom[r]] != pk.chroms[(size_t)pk.slot_chrom[r]] || panel.pos_text[r] != pk.pos_text[r] ||
                panel.ref[r] != pk.ref[r] || panel.dup[r] != pk.dup[r]) {
                bad = r;
                break;
            }
        if (bad < std::max(rows, rows_k)) {
            printf("Error from storeInputFile function: %s line %zu does not describe the panel of %s\n", table_paths[k].c_str(),
                   bad + 2, table_paths[0].c_str());
            return 0;
        }
        thr_view.insert(thr_view.end(), tv.begin(), tv.end());
    }
    for (size_t k = 0; k < NT; ++k) {
        const std::string interm = out_dirs[k] + interm_name;
        if (sweep && !make_dir(interm)) {
            std::cout << "Error: cannot create " << interm << std::endl;
            return 0;
        }
        std::ofstream dummy((interm + "/dummyVCF_1.vcf").c_str());
        for (const std::string& d : dummy_pieces[k]) dummy.write(d.data(), (std::streamsize)d.size());
    }
    dummy_pieces.clear();
    panel.link();
    const int64_t P = panel.size();
    // rows of a duplicated position: the hashes keep the FIRST row's reference, thresholds, Germ_Max (insert does
    // not overwrite, VC:505-560) and flag it if ANY row says YES
    for (int64_t i = 0; i < P; ++i) {
        const int32_t h = panel.twin_head[i];
        if (h != (int32_t)i) {
            if (panel.dup[i]) panel.dup[h] = 1;
        }
    }
    for (int64_t i = 0; i < P; ++i) {
        const int32_t h = panel.twin_head[i];
        if (h != (int32_t)i) {
            panel.dup[i] = panel.dup[h];
            panel.ref[i] = panel.ref[h];
            for (size_t t = 0; t < NT; ++t) {
                float* tv = thr_view.data() + t * (size_t)P * 8;
                std::vector<std::string>& gt = germ_texts[t];
                for (int k = 0; k < 8; ++k) tv[(size_t)i * 8 + k] = tv[(size_t)h * 8 + k];
                for (int k = 0; k < 4; ++k) gt[(size_t)i * 4 + k] = gt[(size_t)h * 4 + k];
            }
        }
    }
    std::cout << "Running function storeInputFile: the error levels have stored with success " << P << RESET << std::endl;
    resolve_sites(panel, sites);
    const int64_t HS = (int64_t)sites.dev_slot.size();  // sites tested on the device
    // Site_Report.txt of every table, rows appended group by group (tumours in the summary's order, sites in file order)
    std::vector<std::ofstream> site_reports;
    if (argc == 7)
        for (size_t k = 0; k < NT; ++k) {
            site_reports.emplace_back((out_dirs[k] + "/Site_Report.txt").c_str());
            site_reports.back() << "Filename\tChrom\tPosition\tRef\tAlt\tRD_fw\tRD_bw\tReads_fw\tReads_bw\tAF\tNoise_fw\tNoise_bw\tQscore_fw\t"
                                   "Qscore_bw\tStatus\n";
        }
    std::vector<uint8_t> ref_code((size_t)P, 255);
    for (int64_t i = 0; i < P; ++i) {
        const std::string& r = panel.ref[i];
        if (r == "A") ref_code[i] = 0;
        else if (r == "C") ref_code[i] = 1;
        else if (r == "G") ref_code[i] = 2;
        else if (r == "T") ref_code[i] = 3;
    }

    timer.lap("parse_noise_table", (double)P, "rows");
    // ---- tumour files in the reference's order
    srand((unsigned)time(nullptr));
    const int seed = rand() % 1000;  // VC:328-331
    std::vector<CountFile> files;
    std::vector<std::string> listed;
    bool bam_files = false;
    if (!list_count_files(tumour_dir, files, listed, &bam_files)) {
        std::cout << "Error: cannot list " << tumour_dir << "/*.ASEQ" << std::endl;
        return 0;
    }
    const std::string list_tail = interm_name + "/" + std::to_string(seed) + "_tumour_count_list_original.txt";
    for (size_t k = 0; k < NT; ++k) write_list_file(out_dirs[k] + list_tail, listed);
    const std::string list_name = out_dirs[0] + list_tail;
    std::cout << "\nRunning function storeList: " << GREEN << list_name << RESET << " stored with success. It contains " << GREEN
              << files.size() << RESET << " samples" << std::endl;
    const int T = (int)files.size();
    if (!gpu.wait()) {  // without a B200 there is nothing this program can do (no CPU fallback)
        std::cout << RED << "Error: as_create: " << gpu.error << RESET << std::endl;
        return 1;
    }
    as_ctx* ctx = gpu.ctx;
    // BAM input: the pileups of group g + 1 run on the main thread while the caller of group g runs on the worker thread
    // below, so they get a context of their own (as_ctx is not thread-safe) on the run's first device
    struct PileupContext {
        as_ctx* c = nullptr;
        ~PileupContext() { if (c && as_process_is_resident()) as_destroy(c); }  // the service lives on; a program leaves through _exit
    } pile;
    if (bam_files) {
        int dev = 0;
        as_context_devices(ctx, &dev, 1);
        if (as_create(dev, &pile.c) != AS_OK) return report_gpu_error("as_create (pileup)");
        bam.setup(panel);
    }
    timer.lap("cuda_context_wait");
    std::cout << "\nRunning function callVariants...." << std::endl;

    // ---- the hot path on the GPU, in groups of samples: while the GPUs work on one group (upload, caller, sorted
    // download) the host threads parse the next one into the other pinned buffer, so pinned memory is two groups, not
    // the whole run, and the text parse hides behind the GPU step (or the other way round)
    struct CallCounts { uint32_t fw[4], bw[4]; };  // the record of a call, kept for the Fisher test and the writers
    struct TableCalls {  // the calls of one noise table
        std::vector<as_call> calls;
        std::vector<CallCounts> call_counts;
        std::vector<int32_t> call_row;   // file row of a call that came from a row beyond its position's slots (-1: see slot_of_row)
        std::vector<long long> call_rd;  // RD column of the call's row where it is not A+C+G+T (-1: the sum); VC:814-817 divide by the column
    };
    std::vector<TableCalls> per_table(NT);
    std::vector<AseqStats> file_stats((size_t)T);  // order information of every file (slot_of_row only when out of order)
    double total_rows = 0, parse_s = 0, gpu_s = 0;
    if (T > 0 && P > 0) {
        int64_t budget_mb = 512;
        if (const char* env = getenv("AS_GROUP_MB")) budget_mb = std::max<long long>(1, atoll(env));
        int64_t G = std::max<int64_t>(1, std::min<int64_t>(T, (budget_mb << 20) / std::max<int64_t>(1, 16 * P)));
        if (const char* env = getenv("AS_GROUP_SAMPLES")) G = std::max<long long>(1, std::min<long long>(T, atoll(env)));  // tests
        HostCounts buf[2];
        std::vector<AseqStats> stats[2];
        auto load_group = [&](int64_t first, int which) -> int {
            const double t0 = PhaseTimer::now();
            const size_t n = (size_t)std::min<int64_t>(G, T - first);
            buf[which].fmt = std::max(buf[which].fmt, buf[which ^ 1].fmt);  // once the 16-bit format was needed it stays
            const int lrc = bam_files ? load_bam_counts(files, (size_t)first, n, panel, bam, pile.c, buf[which], stats[which])
                                      : load_counts(files, (size_t)first, n, panel, buf[which], stats[which], true);
            if (lrc == 2)
                for (size_t i = 0; i < n; ++i)
                    if (!stats[which][i].ok) printf("\tError from callVariants:  Cannot open %s\n", files[(size_t)first + i].path.c_str());
            parse_s += PhaseTimer::now() - t0;
            return lrc;
        };
        std::unordered_map<int32_t, std::vector<int32_t>> sites_at;  // slot -> the tested sites there
        for (int64_t h = 0; h < HS; ++h) sites_at[sites.dev_slot[(size_t)h]].push_back((int32_t)h);
        int lrc = load_group(0, 0);
        if (lrc == 1) return report_gpu_error("pinned host allocation");
        if (lrc >= 2) return 0;  // 3: a BAM that cannot be read, reported like an ASEQ file that cannot be opened
        for (int64_t first = 0, g = 0; first < T; first += G, ++g) {
            const int which = (int)(g & 1);
            const int32_t Tg = (int32_t)std::min<int64_t>(G, T - first);
            report_load(files, (size_t)first, stats[which], false);
            for (int i = 0; i < Tg; ++i) {
                for (int64_t k = 0; k < stats[which][(size_t)i].outside; ++k) std::cout << "mistake..." << std::endl;  // VC:847-852
                total_rows += (double)stats[which][(size_t)i].rows;
                file_stats[(size_t)(first + i)] = std::move(stats[which][(size_t)i]);
            }
            // GPU step of this group on a worker thread (passes of up to 8 tables) ...
            std::vector<std::vector<as_call>> parts(NT);
            std::vector<as_site_test> site_part;  // [NT][Tg][HS]
            int rc = AS_OK;
            std::string gpu_error;
            const char* gpu_what = "as_call_variants_host";
            const HostCounts& hc = buf[which];
            std::thread worker([&]() {
                const double t0 = PhaseTimer::now();
                std::vector<as_call> list;
                int64_t n_part[8];
                for (size_t c0 = 0; c0 < NT && rc == AS_OK; c0 += 8) {
                    const int32_t nc = (int32_t)std::min<size_t>(8, NT - c0);
                    const float* tv = thr_view.data() + c0 * (size_t)P * 8;
                    int64_t cap = std::max<int64_t>(1 << 16, (int64_t)Tg * P / 256);
                    for (;;) {
                        list.resize((size_t)cap * (size_t)nc);
                        rc = hc.fmt == 2
                                 ? as_call_variants_sweep_host16(ctx, (const uint16_t*)hc.p, hc.wide.data(), (int64_t)hc.wide.size(), Tg,
                                                                 P, ref_code.data(), tv, nc, cut, list.data(), cap, n_part)
                                 : as_call_variants_sweep_host_packed(ctx, (const uint32_t*)hc.p, hc.wide.data(), (int64_t)hc.wide.size(),
                                                                      Tg, P, ref_code.data(), tv, nc, cut, list.data(), cap, n_part);
                        if (rc != AS_EOVERFLOW) break;
                        cap = *std::max_element(n_part, n_part + nc);  // the largest true count: run the group again with room for all
                    }
                    if (rc == AS_OK)
                        for (int32_t i = 0; i < nc; ++i)
                            parts[c0 + (size_t)i].assign(list.begin() + (long)(i * cap), list.begin() + (long)(i * cap + n_part[i]));
                }
                // the listed sites of this group, while its buffer is valid: all tables in one kernel pass per 8
                if (rc == AS_OK && HS > 0) {
                    site_part.resize(NT * (size_t)Tg * (size_t)HS);
                    for (size_t c0 = 0; c0 < NT && rc == AS_OK; c0 += 8) {
                        const int32_t nc = (int32_t)std::min<size_t>(8, NT - c0);
                        const float* tv = thr_view.data() + c0 * (size_t)P * 8;
                        as_site_test* o = site_part.data() + c0 * (size_t)Tg * (size_t)HS;
                        rc = hc.fmt == 2 ? as_site_tests_host16(ctx, (const uint16_t*)hc.p, hc.wide.data(), (int64_t)hc.wide.size(), Tg, P,
                                                                ref_code.data(), tv, nc, sites.dev_slot.data(), sites.dev_alt.data(), HS, cut, o)
                                         : as_site_tests_host_packed(ctx, (const uint32_t*)hc.p, hc.wide.data(), (int64_t)hc.wide.size(), Tg,
                                                                     P, ref_code.data(), tv, nc, sites.dev_slot.data(), sites.dev_alt.data(),
                                                                     HS, cut, o);
                    }
                    if (rc != AS_OK) gpu_what = "as_site_tests_host";
                }
                if (rc != AS_OK) gpu_error = as_last_error();
                gpu_s += PhaseTimer::now() - t0;
            });
            // ... while the next group is parsed
            int next_rc = 0;
            if (first + G < T) next_rc = load_group(first + G, which ^ 1);
            worker.join();
            if (rc != AS_OK) {
                std::cout << RED << "Error: " << gpu_what << ": " << gpu_error << RESET << std::endl;
                return 1;
            }
            if (next_rc == 1) return report_gpu_error("pinned host allocation");
            if (next_rc >= 2) return 0;
            // ---- rows the tensor has no slot for (a file listing a position more often than the panel enumerates it): the
            // reference tests every row (VC:869-3288), so they go through the caller as well, in one small pass of their own
            // (one "sample", one "slot" per row, thresholds and reference base of the row's position)
            std::vector<std::pair<int32_t, const AseqStats::ExtraRow*>> xr;
            bool fixes = false;
            for (int i = 0; i < Tg; ++i) {
                for (const AseqStats::ExtraRow& x : file_stats[(size_t)(first + i)].extras) xr.emplace_back((int32_t)(first + i), &x);
                fixes = fixes || !file_stats[(size_t)(first + i)].rd_fix.empty();
            }
            std::vector<std::pair<int32_t, const AseqStats::ExtraRow*>> use;
            std::vector<std::vector<as_call>> xcalls(NT);
            if (!xr.empty()) {
                // The reference's strand tests take (alt_fw, RD - reverse reads) and (alt_bw, reverse reads), RD being the COLUMN
                // (VC:895-896); the coverage gate takes the sums (VC:898).  So the gate is applied here and the row goes to the
                // caller with its forward depth set to RD - reverse reads (the reference base's count absorbs the difference;
                // alt counts are untouched) and a cutoff of 1.
                std::vector<uint32_t> fwadj;
                for (const auto& pr : xr) {
                    const AseqStats::ExtraRow& x = *pr.second;
                    long long FW = 0, BW = 0;
                    for (int b = 0; b < 4; ++b) { FW += x.fw[b]; BW += x.bw[b]; }
                    const uint8_t rb = ref_code[(size_t)x.slot];
                    if (FW < cut || BW < cut || rb > 3) continue;  // VC:898 / VC:3290: never a call
                    uint32_t ref_fw = 0;
                    if (!rd_column_forward(x, rb, ref_fw)) {
                        std::cout << "Warning: " << files[(size_t)pr.first].path << " row " << x.row + 2
                                  << ": RD column smaller than the alt reads; row skipped" << std::endl;
                        continue;
                    }
                    use.push_back(pr);
                    fwadj.push_back(ref_fw);
                }
                const int64_t M = (int64_t)use.size();
                std::vector<uint32_t> xc((size_t)M * 8 + 4);
                uint32_t* xcp = (uint32_t*)(((uintptr_t)xc.data() + 15) & ~(uintptr_t)15);
                std::vector<uint8_t> xref((size_t)M);
                std::vector<float> xthr(NT * (size_t)M * 8);  // [NT][M][4][2]
                for (int64_t m = 0; m < M; ++m) {
                    const AseqStats::ExtraRow& x = *use[(size_t)m].second;
                    memcpy(xcp + m * 4, x.fw, 16);
                    memcpy(xcp + (M + m) * 4, x.bw, 16);
                    xref[(size_t)m] = ref_code[(size_t)x.slot];
                    xcp[m * 4 + xref[(size_t)m]] = fwadj[(size_t)m];
                    for (size_t k = 0; k < NT; ++k)
                        memcpy(&xthr[(k * (size_t)M + (size_t)m) * 8], &thr_view[(k * (size_t)P + (size_t)x.slot) * 8], 32);
                }
                const int64_t xcap = M * 3 + 1;  // at most three calls per row: never an overflow
                std::vector<as_call> xlist;
                int64_t nx[8];
                for (size_t c0 = 0; M > 0 && c0 < NT; c0 += 8) {
                    const int32_t nc = (int32_t)std::min<size_t>(8, NT - c0);
                    xlist.resize((size_t)xcap * (size_t)nc);
                    if (as_call_variants_sweep_host(ctx, xcp, 1, M, xref.data(), xthr.data() + c0 * (size_t)M * 8, nc, 1, xlist.data(), xcap,
                                                    nx) != AS_OK)
                        return report_gpu_error("as_call_variants_host");
                    for (int32_t i = 0; i < nc; ++i)
                        xcalls[c0 + (size_t)i].assign(xlist.begin() + (long)(i * xcap), xlist.begin() + (long)(i * xcap + nx[i]));
                }
            }
            for (size_t tk = 0; tk < NT; ++tk) {
                std::vector<as_call>& calls = per_table[tk].calls;
                std::vector<CallCounts>& call_counts = per_table[tk].call_counts;
                std::vector<int32_t>& call_row = per_table[tk].call_row;
                std::vector<long long>& call_rd = per_table[tk].call_rd;
                const std::vector<as_call>& part = parts[tk];
                const size_t base = calls.size();
                calls.resize(base + part.size());
                call_counts.resize(base + part.size());
                call_row.resize(base + part.size(), -1);
                call_rd.resize(base + part.size(), -1);
                parallel_for(part.size(), [&](size_t i) {
                    as_call c = part[i];
                    hc.record(c.sample, c.slot, P, call_counts[base + i].fw, call_counts[base + i].bw);
                    c.sample += (int32_t)first;
                    calls[base + i] = c;
                });
                if (!xr.empty()) {
                    const std::vector<as_call>& xc = xcalls[tk];
                    for (size_t i = 0; i < xc.size(); ++i) {
                        const AseqStats::ExtraRow& x = *use[(size_t)xc[i].slot].second;
                        as_call c = xc[i];
                        c.sample = use[(size_t)xc[i].slot].first;
                        c.slot = x.slot;
                        CallCounts k;
                        memcpy(k.fw, x.fw, 16);
                        memcpy(k.bw, x.bw, 16);
                        long long sum = 0;
                        for (int b = 0; b < 4; ++b) sum += (long long)x.fw[b] + x.bw[b];
                        calls.push_back(c);
                        call_counts.push_back(k);
                        call_row.push_back(x.row);
                        call_rd.push_back(x.rd != sum ? x.rd : -1);
                    }
                }
                if (fixes) {  // RD column of rows where it is not the sum of the counts
                    for (size_t i = base; i < base + part.size(); ++i) {
                        for (const AseqStats::RdFix& f : file_stats[(size_t)calls[i].sample].rd_fix)
                            if (f.slot == calls[i].slot) call_rd[i] = f.rd;
                    }
                }
                if (!xr.empty()) {  // back into sample order (the calls of the extra rows were appended behind the group's)
                    std::vector<size_t> order(calls.size() - base);
                    for (size_t i = 0; i < order.size(); ++i) order[i] = base + i;
                    std::stable_sort(order.begin(), order.end(), [&](size_t a, size_t b) { return calls[a].sample < calls[b].sample; });
                    std::vector<as_call> c2(order.size());
                    std::vector<CallCounts> k2(order.size());
                    std::vector<int32_t> r2(order.size());
                    std::vector<long long> d2(order.size());
                    for (size_t i = 0; i < order.size(); ++i) { c2[i] = calls[order[i]]; k2[i] = call_counts[order[i]]; r2[i] = call_row[order[i]]; d2[i] = call_rd[order[i]]; }
                    std::copy(c2.begin(), c2.end(), calls.begin() + (long)base);
                    std::copy(k2.begin(), k2.end(), call_counts.begin() + (long)base);
                    std::copy(r2.begin(), r2.end(), call_row.begin() + (long)base);
                    std::copy(d2.begin(), d2.end(), call_rd.begin() + (long)base);
                }
            }
            if (!site_reports.empty()) {
                // a site whose row was set aside because its RD column is not A+C+G+T (extras with k = -1: the tensor holds
                // no record there) is tested as the extra-row pass tests that row: forward depth RD - reverse reads
                // (rd_column_forward), cutoff 1 on the device, the coverage gate on the sums (VC:898) here
                struct SetAside { int32_t i; const AseqStats::ExtraRow* x; bool ok; };
                std::vector<SetAside> aside;
                std::vector<int32_t> a_slot, a_alt, a_entry;  // per tested entry: mini-tensor slot, alt, index into aside
                for (int i = 0; i < Tg && !sites_at.empty(); ++i)
                    for (const AseqStats::ExtraRow& x : file_stats[(size_t)(first + i)].extras) {
                        auto it = sites_at.find(x.slot);
                        if (x.k >= 0 || it == sites_at.end()) continue;
                        const int32_t m = (int32_t)aside.size();
                        uint32_t ref_fw = 0;
                        const uint8_t rb = ref_code[(size_t)x.slot];
                        aside.push_back(SetAside{i, &x, rb > 3 || rd_column_forward(x, rb, ref_fw)});
                        for (int32_t h : it->second) { a_slot.push_back(m); a_alt.push_back(h); }
                    }
                const int64_t M = (int64_t)aside.size(), NA = (int64_t)a_slot.size();
                if (M > 0) {
                    std::vector<uint32_t> xc((size_t)M * 8 + 4);
                    uint32_t* xcp = (uint32_t*)(((uintptr_t)xc.data() + 15) & ~(uintptr_t)15);
                    std::vector<uint8_t> xref((size_t)M);
                    std::vector<float> xthr(NT * (size_t)M * 8);  // [NT][M][4][2]
                    for (int64_t m = 0; m < M; ++m) {
                        const AseqStats::ExtraRow& x = *aside[(size_t)m].x;
                        memcpy(xcp + m * 4, x.fw, 16);
                        memcpy(xcp + (M + m) * 4, x.bw, 16);
                        xref[(size_t)m] = ref_code[(size_t)x.slot];
                        uint32_t ref_fw = 0;
                        if (xref[(size_t)m] <= 3 && rd_column_forward(x, xref[(size_t)m], ref_fw)) xcp[m * 4 + xref[(size_t)m]] = ref_fw;
                        for (size_t k = 0; k < NT; ++k)
                            memcpy(&xthr[(k * (size_t)M + (size_t)m) * 8], &thr_view[(k * (size_t)P + (size_t)x.slot) * 8], 32);
                    }
                    std::vector<int32_t> alt_of((size_t)NA);
                    for (int64_t j = 0; j < NA; ++j) alt_of[(size_t)j] = sites.dev_alt[(size_t)a_alt[(size_t)j]];
                    std::vector<as_site_test> xo(NT * (size_t)NA);
                    for (size_t c0 = 0; c0 < NT; c0 += 8) {
                        const int32_t nc = (int32_t)std::min<size_t>(8, NT - c0);
                        if (as_site_tests_host(ctx, xcp, 1, M, xref.data(), xthr.data() + c0 * (size_t)M * 8, nc, a_slot.data(), alt_of.data(),
                                               NA, 1, xo.data() + c0 * (size_t)NA) != AS_OK)
                            return report_gpu_error("as_site_tests_host");
                    }
                    for (size_t k = 0; k < NT; ++k)
                        for (int64_t j = 0; j < NA; ++j) {
                            const SetAside& a = aside[(size_t)a_slot[(size_t)j]];
                            as_site_test r = xo[k * (size_t)NA + (size_t)j];
                            long long FW = 0, BW = 0;
                            for (int b = 0; b < 4; ++b) { FW += a.x->fw[b]; BW += a.x->bw[b]; }
                            if (!a.ok) {  // the RD column is smaller than the alt reads: the caller skips the row (warning above)
                                r.status = AS_SITE_NOT_TESTABLE;
                                r.p_fw = r.p_bw = std::nan("");
                            } else if (r.status != AS_SITE_NOT_TESTABLE && (FW < cut || BW < cut)) {
                                r.status = AS_SITE_LOW_COVERAGE;
                            }
                            site_part[(k * (size_t)Tg + (size_t)a.i) * (size_t)HS + (size_t)a_alt[(size_t)j]] = r;
                        }
                }
                // rows of this group: tumours in order, sites in file order
                for (size_t k = 0; k < NT; ++k) {
                    std::ostringstream os;
                    os << std::setprecision(4);
                    const float* tv = thr_view.data() + k * (size_t)P * 8;
                    char nf[64], nb[64];
                    for (int i = 0; i < Tg; ++i)
                        for (size_t j = 0; j < sites.chrom.size(); ++j) {
                            os << files[(size_t)(first + i)].sample << "\t" << sites.chrom[j] << "\t" << sites.pos_text[j] << "\t" << sites.ref[j]
                               << "\t" << sites.alt[j] << "\t";
                            int32_t st = sites.host_status[j];
                            const as_site_test* r = st ? nullptr : &site_part[(k * (size_t)Tg + (size_t)i) * (size_t)HS + (size_t)sites.dev[j]];
                            if (r) st = r->status;
                            if (!r || st == AS_SITE_NO_DATA) {
                                os << "-\t-\t-\t-\t-\t-\t-\t-\t-\t";
                            } else {
                                const uint32_t depth = r->depth_fw + r->depth_bw, reads = r->alt_fw + r->alt_bw;
                                const float* e = tv + (size_t)sites.slot[j] * 8 + (size_t)sites.dev_alt[(size_t)sites.dev[j]] * 2;
                                snprintf(nf, sizeof nf, "%f", (double)e[0]);
                                snprintf(nb, sizeof nb, "%f", (double)e[1]);
                                os << r->depth_fw << "\t" << r->depth_bw << "\t" << r->alt_fw << "\t" << r->alt_bw << "\t"
                                   << (depth == 0 ? 0.f : float(reads) / float(depth)) << "\t" << nf << "\t" << nb << "\t";
                                for (double pv : {r->p_fw, r->p_bw}) {  // Q as the summary prints it (VC:895-896, VC:1066)
                                    if (std::isnan(pv)) os << "-\t";
                                    else os << std::setprecision(4) << q_from_p(pv) << "\t";
                                }
                            }
                            os << site_status_text(st) << "\n";
                        }
                    site_reports[k] << os.str();
                }
            }
        }
        // The device returns (sample, slot, alt) order = the reference's file-row order (VC:869-3288: rows, then alts
        // A,C,G,T) for every file whose rows follow the panel enumeration.  A file that does not is re-ordered by its rows.
        for (TableCalls& tc : per_table) {
            std::vector<as_call>& calls = tc.calls;
            std::vector<CallCounts>& call_counts = tc.call_counts;
            std::vector<int32_t>& call_row = tc.call_row;
            std::vector<long long>& call_rd = tc.call_rd;
            std::vector<size_t> run_begin((size_t)T + 1, calls.size());
            for (size_t i = calls.size(); i-- > 0;) run_begin[(size_t)calls[i].sample] = i;
            for (int t = T - 1; t >= 0; --t) run_begin[(size_t)t] = std::min(run_begin[(size_t)t], run_begin[(size_t)t + 1]);
            for (int t = 0; t < T; ++t) {
                if (file_stats[(size_t)t].in_order) continue;
                std::vector<int32_t> row_of((size_t)P, -1);
                const std::vector<int32_t>& sor = file_stats[(size_t)t].slot_of_row;
                for (size_t r = 0; r < sor.size(); ++r)
                    if (sor[r] >= 0) row_of[(size_t)sor[r]] = (int32_t)r;
                const size_t lo = run_begin[(size_t)t], hi = run_begin[(size_t)t + 1];
                std::vector<size_t> order(hi - lo);
                for (size_t i = 0; i < order.size(); ++i) order[i] = lo + i;
                std::stable_sort(order.begin(), order.end(), [&](size_t x, size_t y) {
                    const int32_t rx = call_row[x] >= 0 ? call_row[x] : row_of[(size_t)calls[x].slot];
                    const int32_t ry = call_row[y] >= 0 ? call_row[y] : row_of[(size_t)calls[y].slot];
                    return rx != ry ? rx < ry : calls[x].alt < calls[y].alt;
                });
                std::vector<as_call> c2(order.size());
                std::vector<CallCounts> k2(order.size());
                std::vector<int32_t> r2(order.size());
                std::vector<long long> d2(order.size());
                for (size_t i = 0; i < order.size(); ++i) { c2[i] = calls[order[i]]; k2[i] = call_counts[order[i]]; r2[i] = call_row[order[i]]; d2[i] = call_rd[order[i]]; }
                std::copy(c2.begin(), c2.end(), calls.begin() + (long)lo);
                std::copy(k2.begin(), k2.end(), call_counts.begin() + (long)lo);
                std::copy(r2.begin(), r2.end(), call_row.begin() + (long)lo);
                std::copy(d2.begin(), d2.end(), call_rd.begin() + (long)lo);
            }
        }
    }
    if (timer.on) fprintf(stderr, "AS_TIMING %s %.6f (%.3g rows/s)\nAS_TIMING caller_gpu_busy %.6f\n",
                          bam_files ? "pileup_tumours_busy" : "parse_tumours_busy", parse_s, total_rows / std::max(parse_s, 1e-9), gpu_s);
    timer.lap("parse_and_call", 6.0 * (double)T * (double)P, "tests");

    std::string summary_name;
    for (size_t tk = 0; tk < NT; ++tk) {  // every table's outputs in its own directory
        const std::vector<as_call>& calls = per_table[tk].calls;
        const std::vector<CallCounts>& call_counts = per_table[tk].call_counts;
        const std::vector<long long>& call_rd = per_table[tk].call_rd;
        const std::vector<std::string>& germ_text = germ_texts[tk];
        const std::string& output_dir = out_dirs[tk];
        // Fisher strand-bias p of every call (VC:902) on the device: one warp per call's 2x2 table
        std::vector<double> fisher_p(calls.size());
        {
            std::vector<int32_t> tables(calls.size() * 4);
            parallel_for(calls.size(), [&](size_t i) {
                const CallCounts& k = call_counts[i];
                const int32_t FWs = (int32_t)(k.fw[0] + k.fw[1] + k.fw[2] + k.fw[3]), BWs = (int32_t)(k.bw[0] + k.bw[1] + k.bw[2] + k.bw[3]);
                tables[i * 4 + 0] = call_rd[i] >= 0 ? (int32_t)(call_rd[i] - BWs) : FWs;  // fisherTest(RD - RD_reverse, RD_reverse, alt_fw, alt_bw), VC:902
                tables[i * 4 + 1] = BWs;
                tables[i * 4 + 2] = (int32_t)k.fw[calls[i].alt];
                tables[i * 4 + 3] = (int32_t)k.bw[calls[i].alt];
            });
            const int frc = as_fisher_tests_host(ctx, tables.data(), (int64_t)calls.size(), fisher_p.data());
            if (frc != AS_OK) return report_gpu_error("as_fisher_tests_host");
        }
        timer.lap("fisher_tests", (double)calls.size(), "calls");  // once per table in a sweep

        // ---- writers (VC:662-688, VC:1040-1066)
        summary_name = output_dir + "/Summary_Variant_Info.txt";
        std::ofstream output(summary_name.c_str());
        output << "Filename\tChrom\tPosition\tSubtitution\tRD\tRD_fw\tRD_bw\tAF\tReads_fw\tReads_bw\tAF_fw\tAF_bw\tAmpliconEdge_"
                  "StrandBias\tFisherPvalue\tQscore_fw\tQscore_bw\tReadTier\tGermlineInfo\tMaxGermlineAF\t10merDownstream\t10merUpstream\tHo"
                  "mopolymerFlag"
               << "\n";
        const char* L = "ACGT";
        // One tumour = one VCF and one run of summary rows: the tumours are formatted on all host threads (ostream formatting of
        // ~20 numbers per call was the largest phase of a configs[1] run), every thread writes its own VCFs, and the summary
        // runs are written in tumour order afterwards.
        std::vector<size_t> call_begin((size_t)T + 1, calls.size());
        for (size_t i = calls.size(); i-- > 0;) call_begin[(size_t)calls[i].sample] = i;
        for (int t = T - 1; t >= 0; --t) call_begin[(size_t)t] = std::min(call_begin[(size_t)t], call_begin[(size_t)t + 1]);
        std::vector<std::string> summary_rows((size_t)T);
        auto write_tumour = [&](int t) {
            std::ostringstream output;
            // setprecision(4) is sticky on the reference's summary stream (VC:1066): only the first row of the run prints its
            // leading columns with the default precision
            if (call_begin[(size_t)t] > 0) output << std::setprecision(4);
            const std::string vcf_name = output_dir + "/" + files[t].sample + ".vcf";
            std::ofstream vcf(vcf_name.c_str());
            time_t now = time(nullptr);
            char dt_buf[64];
            const char* dt = ctime_r(&now, dt_buf);
            vcf << "##fileformat=VCF-like\n##fileDate=" << dt
                << "##source=AmpliSolveVariantCalling\n##reference=Not_Specified_here\n##phasing=Not_Specified_here\n##FILTER=<ID="
                   "XXXXXXXXX,Description='XXXXXXXXX'>\n##FILTER=<ID=XXXXXXXXX,Description='XXXXXXXXX'>\n##FILTER=<ID=XXXXXXXXX,"
                   "Description='XXXXXXXXX'>\n##FILTER=<ID=XXXXXXXXX,Description='XXXXXXXXX'>\n##INFO=<ID=RD,Number=1,Type=Integer,"
                   "Description='Total Read Depth'>\n##SAMPLE=<ID=Not_Specified_here,SampleName="
                << files[t].sample
                << ">\n##INFO=<ID=AF,Number=.,Type=Float,Description='Allele Frequency'>\n##INFO=<ID=SR,Number=1,Type=String,"
                   "Description='Supporting Reads'>\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO"
                << "\n";
            for (size_t ci = call_begin[(size_t)t]; ci < call_begin[(size_t)t + 1]; ++ci) {
                const as_call& c = calls[ci];
                const int64_t s = c.slot;
                const uint32_t* fw = call_counts[ci].fw;
                const uint32_t* bw = call_counts[ci].bw;
                const int FW = (int)(fw[0] + fw[1] + fw[2] + fw[3]), BW = (int)(bw[0] + bw[1] + bw[2] + bw[3]);
                const int RD = call_rd[ci] >= 0 ? (int)call_rd[ci] : FW + BW;  // the RD column (VC:752), normally the sum
                const int a = c.alt;
                const int k_fw = (int)fw[a], k_bw = (int)bw[a];
                const float AF = float(k_fw + k_bw) / float(RD);                    // VC:814-817
                const float AF_fw = FW == 0 ? 0.f : float(k_fw) / float(FW);        // VC:776-795
                const float AF_bw = BW == 0 ? 0.f : float(k_bw) / float(BW);        // VC:797-812
                const long double Q_fw = q_from_p(c.p_fw), Q_bw = q_from_p(c.p_bw);  // VC:895-896
                const double p = fisher_p[ci];                                      // VC:902
                const char* flag_fisher = (p <= p_value_float) ? "YES" : "NO";      // VC:903-910
                const char* flag_dup = panel.dup[s] ? "YES" : "NO";
                const bool high = !(k_fw < 5 || k_bw < 5);                          // VC:912-919
                const char* tier = high ? "HighQual" : "LowQual";
                const std::string& max_germ_text = germ_text[(size_t)s * 4 + a];    // VC:943-954
                const double max_germ = atof(max_germ_text.c_str());                // VC:972
                const std::string chrom = panel.chroms[panel.slot_chrom[s]];
                const std::string down = kmer(panel, panel.slot_chrom[s], panel.slot_pos[s], true);   // VC:964
                const std::string up = kmer(panel, panel.slot_chrom[s], panel.slot_pos[s], false);    // VC:965
                const int homo = homopolymer_test(down, up, L[a]);
                const double Q = double(Q_fw + Q_bw) / 2.000;                       // VC:967
                const std::string cat = std::string(flag_dup) + "_" + flag_fisher;
                // FILTER: keys of an unordered_map in ITS iteration order (VC:993-1059)
                std::unordered_map<std::string, std::string> flags;
                int not_pass = 0;
                if (cat == "YES_NO") { flags.insert(std::make_pair(std::string("AmpliconEdge"), std::string("AmpliconEdge"))); not_pass = 1; }
                if (cat == "YES_YES") { flags.insert(std::make_pair(std::string("AmpliconEdge;StrandBias"), std::string("AmpliconEdge;StrandBias"))); not_pass = 1; }
                if (cat == "NO_YES") { flags.insert(std::make_pair(std::string("StrandBias"), std::string("StrandBias"))); not_pass = 1; }
                if (AF < max_germ && cat == "NO_NO" && !high) { flags.insert(std::make_pair(std::string("PositionWithHighNoise"), std::string("PositionWithHighNoise"))); not_pass = 1; }
                if (homo == 1) { flags.insert(std::make_pair(std::string("HomoPolymerRegion"), std::string("HomoPolymerRegion"))); not_pass = 1; }
                if (Q_fw < 20 || Q_bw < 20) { flags.insert(std::make_pair(std::string("LowQ"), std::string("LowQ"))); not_pass = 1; }
                if (!high) { flags.insert(std::make_pair(std::string("LowSupportingReads"), std::string("LowSupportingReads"))); not_pass = 1; }
                const std::string& pos_text = panel.pos_text[s];
                const char* id = ".";
                std::string filter = "PASS";
                if (not_pass) {
                    filter.clear();
                    int first = 0;
                    for (auto it = flags.begin(); it != flags.end(); ++it) {
                        filter = first == 0 ? it->first : filter + ";" + it->first;
                        ++first;
                    }
                    if (c.ref == 1 && a == 2) id = "-";  // the reference writes ID "-" for non-PASS C->G rows (VC:1856)
                }
                vcf << chrom << "\t" << pos_text << "\t" << id << "\t" << L[c.ref] << "\t" << L[a] << "\t" << Q << "\t" << filter << "\t"
                    << AF << ";" << RD << ";" << k_fw + k_bw << "\n";
                // summary row; setprecision(4) is sticky on this stream exactly as in VC:1066
                output << files[t].sample << "\t" << chrom << "\t" << pos_text << "\t" << L[c.ref] << "->" << L[a] << "\t" << RD << "\t"
                       << FW << "\t" << BW << "\t" << AF << "\t" << k_fw << "\t" << k_bw << "\t" << AF_fw << "\t" << AF_bw << "\t"
                       << flag_dup << "_" << flag_fisher << "\t" << p << "\t" << std::setprecision(4) << Q_fw << "\t"
                       << std::setprecision(4) << Q_bw << "\t" << tier << "\t" << "-" << "\t" << max_germ_text << "\t" << down << "\t"
                       << up << "\t" << homo << "\n";
            }
            summary_rows[(size_t)t] = output.str();
        };
        {
            std::atomic<int> next(0);
            auto work = [&]() {
                for (int t = next.fetch_add(1); t < T; t = next.fetch_add(1)) write_tumour(t);
            };
            run_on_threads(std::max(1u, std::min(std::thread::hardware_concurrency(), (unsigned)std::max(1, T))), work);
        }
        for (int t = 0; t < T; ++t) {
            if ((t + 1) % 50 == 0)
                std::cout << "\tParsed successfully " << GREEN << (t + 1) << "/" << T << RESET << "  samples" << std::endl;
            output.write(summary_rows[(size_t)t].data(), (std::streamsize)summary_rows[(size_t)t].size());
        }
        output.close();
        timer.lap("write_outputs", (double)calls.size(), "calls");
    }
    std::cout << "\nAmpliSolveVariantCalling execution was successful. The results can be found at : " << YELLOW << summary_name
              << RESET << std::endl;
    std::cout << "\n" << STARS << std::endl;
    return 0;
}

}  // extern "C"
