// computeCounts / ASEQ PILEUP mode: BAM -> <name>.PILEUP.ASEQ (SURVEY.md §8 f4; Execution_examples.md:16-54).
//
//   ./computeCounts [vcf=dummyVCF.txt] [bam=myBAM.bam] [threads=int] [mbq=int] [mrq=int] [mdc=int] [out=Out_DIR]
//
// The reference ships this step as a Mach-O binary without source (Pre-compiled_binaries/computeCounts), so nothing here
// restates reference code; the output format is the one both reference programs parse (EE:1114-1149, VC:723-752: a header
// line, then chr pos dbsnp MAF ref alt A C G T RD Ars Crs Grs Trs) and the counting conventions are those of a
// samtools-style pileup (as_pileup.cu).  Host side: the BGZF container is walked block by block, the blocks of a piece
// are inflated on `threads` host threads (zlib, CRC checked), the record boundaries are indexed, and the records go to
// the GPU (as_pileup_add_host), which walks the CIGARs and counts.  Rows are written in the order of the position file,
// one row per line of it (a position listed twice -- overlapping amplicons -- gets two identical rows, which is what the
// noise model's twin slots expect), and a position with fewer than mdc counted bases is left out.  The reader (asbam::Reader,
// as_bam.h) is shared with the two programs, which pile up a directory of BAM files themselves (as_host.cpp).
#include <fcntl.h>
#include <sys/mman.h>
#include <sys/stat.h>
#include <unistd.h>
#include <zlib.h>

#include <algorithm>
#include <atomic>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <condition_variable>
#include <cstring>
#include <functional>
#include <map>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "amplisolve_b200.h"
#include "as_bam.h"

namespace {

struct Mapped {
    const uint8_t* p = nullptr;
    size_t n = 0;
    int fd = -1;
    bool open(const std::string& path) {
        fd = ::open(path.c_str(), O_RDONLY);
        if (fd < 0) return false;
        struct stat sb;
        if (fstat(fd, &sb) != 0) return false;
        n = (size_t)sb.st_size;
        if (n == 0) return true;
        void* m = mmap(nullptr, n, PROT_READ, MAP_PRIVATE, fd, 0);
        if (m == MAP_FAILED) return false;
        p = (const uint8_t*)m;
        madvise(m, n, MADV_SEQUENTIAL);
        return true;
    }
    ~Mapped() {
        if (p) munmap((void*)p, n);
        if (fd >= 0) close(fd);
    }
};

uint32_t le32(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8) | ((uint32_t)p[2] << 16) | ((uint32_t)p[3] << 24); }
uint32_t le16(const uint8_t* p) { return (uint32_t)p[0] | ((uint32_t)p[1] << 8); }

struct Block {
    size_t data_off, data_len;  // deflate stream inside the file
    size_t out_off;             // where it inflates to, inside the piece
    uint32_t isize, crc;
};

// header of the BGZF block at `off`: total block length, or 0 when it is not one
size_t bgzf_block(const uint8_t* f, size_t n, size_t off, Block& b) {
    if (off + 18 > n) return 0;
    const uint8_t* h = f + off;
    if (h[0] != 31 || h[1] != 139 || h[2] != 8 || !(h[3] & 4)) return 0;
    const size_t xlen = le16(h + 10);
    if (off + 12 + xlen > n) return 0;
    size_t bsize = 0;
    for (size_t x = 0; x + 4 <= xlen;) {  // extra subfields: SI1 SI2 SLEN data
        const uint8_t* e = h + 12 + x;
        const size_t slen = le16(e + 2);
        if (e[0] == 'B' && e[1] == 'C' && slen == 2 && x + 6 <= xlen) bsize = (size_t)le16(e + 4) + 1;
        x += 4 + slen;
    }
    if (bsize < 12 + xlen + 8 || off + bsize > n) return 0;
    b.data_off = off + 12 + xlen;
    b.data_len = bsize - 12 - xlen - 8;
    b.crc = le32(f + off + bsize - 8);
    b.isize = le32(f + off + bsize - 4);
    return bsize;
}

bool inflate_block(const uint8_t* f, const Block& b, uint8_t* out) {
    if (b.isize == 0) return true;
    z_stream zs;
    memset(&zs, 0, sizeof zs);
    if (inflateInit2(&zs, -15) != Z_OK) return false;
    zs.next_in = const_cast<Bytef*>(f + b.data_off);
    zs.avail_in = (uInt)b.data_len;
    zs.next_out = out;
    zs.avail_out = b.isize;
    const int rc = inflate(&zs, Z_FINISH);
    const bool ok = rc == Z_STREAM_END && zs.total_out == b.isize;
    inflateEnd(&zs);
    return ok && (uint32_t)crc32(crc32(0L, Z_NULL, 0), out, b.isize) == b.crc;
}

std::string arg_of(const char* a, const char* key) {
    const size_t n = strlen(key);
    return strncmp(a, key, n) == 0 ? std::string(a + n) : std::string();
}

void usage() {
    printf("\nUsage: computeCounts [vcf=positions.txt] [bam=myBAM.bam] [threads=int] [mbq=int] [mrq=int] [mdc=int] [out=Out_DIR]\n"
           "  vcf      VCF-like list of ALL positions of the panel: chr <tab> pos <tab> id <tab> ref <tab> alt ...\n"
           "  bam      coordinate-sorted or unsorted BAM file (no index needed); several files: bam=a.bam,b.bam\n"
           "  threads  host threads that inflate the BGZF blocks (default: all)\n"
           "  mbq      minimum base quality (default 20)\n"
           "  mrq      minimum read (mapping) quality (default 20)\n"
           "  mdc      minimum depth of coverage of a reported position (default 20)\n"
           "  out      directory of <bam name>.PILEUP.ASEQ (default .)\n\n");
}

// byte buffer that grows without zero-filling (std::vector::resize would memset every piece)
struct RawBuf {
    uint8_t* p = nullptr;
    size_t cap = 0;
    ~RawBuf() { free(p); }
    uint8_t* data() { return p; }
    bool ensure(size_t keep, size_t n) {  // room for n bytes, the first `keep` bytes preserved
        if (n <= cap) return true;
        const size_t want = n + n / 8 + 4096;
        uint8_t* q = (uint8_t*)malloc(want);
        if (!q) return false;
        if (keep) memcpy(q, p, keep);
        free(p);
        p = q;
        cap = want;
        return true;
    }
};

// One helper thread that runs the GPU side of a piece while the main thread inflates the next one (a thread that stays: the
// first CUDA call of a NEW thread costs tens of milliseconds, which a thread per piece would pay every time).
class Worker {
  public:
    Worker() : th_([this]() { loop(); }) {}
    ~Worker() {
        { std::lock_guard<std::mutex> g(m_); stop_ = true; }
        cv_.notify_all();
        th_.join();
    }
    void submit(std::function<int()> f) {  // at most one job at a time: wait() first
        { std::lock_guard<std::mutex> g(m_); job_ = std::move(f); busy_ = true; }
        cv_.notify_all();
    }
    int wait() {  // result of the last job (0 when there was none)
        std::unique_lock<std::mutex> g(m_);
        cv_.wait(g, [this]() { return !busy_; });
        const int rc = rc_;
        rc_ = 0;
        return rc;
    }

  private:
    void loop() {
        for (;;) {
            std::function<int()> f;
            {
                std::unique_lock<std::mutex> g(m_);
                cv_.wait(g, [this]() { return stop_ || (busy_ && job_); });
                if (stop_ && !(busy_ && job_)) return;
                f = std::move(job_);
                job_ = nullptr;
            }
            const int rc = f();
            { std::lock_guard<std::mutex> g(m_); rc_ = rc; busy_ = false; }
            cv_.notify_all();
        }
    }
    std::mutex m_;
    std::condition_variable cv_;
    std::function<int()> job_;
    bool busy_ = false, stop_ = false;
    int rc_ = 0;
    std::thread th_;
};


double now_s() {
    timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec + 1e-9 * ts.tv_nsec;
}

}  // namespace

namespace asbam {

struct Reader::Impl {
    RawBuf bufs[2];  // carried bytes of the previous piece + the inflated blocks of this one (reused by every BAM)
    std::vector<int64_t> offs[2];
    Worker gpu;  // runs as_pileup_add_host of a piece while the next piece inflates
};

Reader::Reader() : impl_(new Impl()) {}
Reader::~Reader() = default;

int Reader::pileup(const std::string& bam, const std::map<std::string, int32_t>& contig_id, int threads, int mbq, int mrq,
                   const std::function<as_ctx*()>& begin, uint64_t* n_records_out) {
    RawBuf* bufs = impl_->bufs;
    std::vector<int64_t>* offs = impl_->offs;
    Worker& gpu = impl_->gpu;
    const bool timing = getenv("AS_TIMING") != nullptr;
    // ---- BAM container
    Mapped f;
    if (!f.open(bam)) { printf("Error from computeCounts: Cannot open file: %s\n", bam.c_str()); return 1; }
    Block probe;
    if (f.n < 28 || bgzf_block(f.p, f.n, 0, probe) == 0) { printf("Error from computeCounts: %s is not a BGZF (BAM) file\n", bam.c_str()); return 1; }

    // Two piece buffers: while the GPU takes the records of one piece (upload + kernel, on a helper thread), the host
    // threads inflate the next piece into the other buffer.
    const size_t piece_budget = (size_t)(getenv("AS_BAM_PIECE_MB") ? atol(getenv("AS_BAM_PIECE_MB")) : 64) << 20;
    std::string job_err;
    int cur = 0;
    std::vector<int32_t> ref_contig;
    size_t file_off = 0, carried = 0;
    bool header_done = false;
    as_ctx* ctx = nullptr;  // set by begin(): the pileup has started
    uint64_t n_records = 0, bytes_inflated = 0;
    double t_inflate = 0, t_gpu = 0;
    int32_t n_ref = 0;
    // declared last, destroyed first: no job outlives what it reads on an early return
    struct Drain { Worker& w; ~Drain() { w.wait(); } } drain{gpu};

    while (file_off < f.n || carried > 0) {
        // blocks of this piece
        std::vector<Block> blocks;
        size_t out_bytes = 0;
        while (file_off < f.n && (blocks.empty() || out_bytes < piece_budget)) {
            Block b;
            const size_t len = bgzf_block(f.p, f.n, file_off, b);
            if (len == 0) { printf("Error from computeCounts: corrupt BGZF block at byte %zu of %s\n", file_off, bam.c_str()); return 1; }
            b.out_off = out_bytes;
            out_bytes += b.isize;
            blocks.push_back(b);
            file_off += len;
        }
        if (blocks.empty() && carried > 0) { printf("Error from computeCounts: %s ends inside a record\n", bam.c_str()); return 1; }
        RawBuf& buf = bufs[cur];  // no job reads it: the one that did was waited for before the carry-over
        std::vector<int64_t>& rec_off = offs[cur];
        if (!buf.ensure(carried, carried + out_bytes + 8)) { printf("Error from computeCounts: out of memory\n"); return 1; }
        const double ti = now_s();
        {
            std::atomic<size_t> next{0};
            std::atomic<bool> bad{false};
            const int nt = (int)std::min<size_t>((size_t)threads, std::max<size_t>(1, blocks.size()));
            std::vector<std::thread> th;
            for (int t = 0; t < nt; ++t)
                th.emplace_back([&]() {
                    for (size_t i; (i = next.fetch_add(1)) < blocks.size();)
                        if (!inflate_block(f.p, blocks[i], buf.data() + carried + blocks[i].out_off)) bad = true;
                });
            for (auto& t : th) t.join();
            if (bad) { printf("Error from computeCounts: a BGZF block of %s does not inflate (or fails its CRC)\n", bam.c_str()); return 1; }
        }
        t_inflate += now_s() - ti;
        bytes_inflated += out_bytes;
        const size_t have = carried + out_bytes;
        size_t off = 0;
        if (!header_done) {
            // magic, l_text, text, n_ref, (l_name, name, l_ref) * n_ref
            bool complete = false;
            do {
                if (have < 12) break;
                if (memcmp(buf.data(), "BAM\1", 4) != 0) { printf("Error from computeCounts: %s is not a BAM file\n", bam.c_str()); return 1; }
                size_t o = 8 + (size_t)le32(buf.data() + 4);
                if (o + 4 > have) break;
                n_ref = (int32_t)le32(buf.data() + o);
                o += 4;
                std::vector<int32_t> map;
                bool ok = true;
                for (int32_t r = 0; r < n_ref; ++r) {
                    if (o + 4 > have) { ok = false; break; }
                    const size_t l_name = le32(buf.data() + o);
                    if (o + 4 + l_name + 4 > have) { ok = false; break; }
                    std::string name((const char*)buf.data() + o + 4, l_name ? l_name - 1 : 0);
                    auto it = contig_id.find(name);
                    map.push_back(it == contig_id.end() ? -1 : it->second);
                    o += 4 + l_name + 4;
                }
                if (!ok) break;
                ref_contig = std::move(map);
                off = o;
                complete = true;
            } while (false);
            if (!complete) {
                if (file_off >= f.n) { printf("Error from computeCounts: %s ends inside its header\n", bam.c_str()); return 1; }
                carried = have;  // keep everything and read more blocks
                continue;
            }
            header_done = true;
            if (n_ref < 1) ref_contig.assign(1, -1), n_ref = 1;
        }
        // records of this piece
        rec_off.clear();
        const size_t first = off;
        while (off + 4 <= have) {
            const size_t bs = le32(buf.data() + off);
            if (off + 4 + bs > have) break;
            if (bs >= 32) rec_off.push_back((int64_t)(off - first));
            off += 4 + bs;
        }
        n_records += rec_off.size();
        if (!ctx && !(ctx = begin())) return 1;
        // the other buffer's job (the previous piece) ran while this piece inflated; it must be over before the
        // carried bytes are copied into that buffer
        const double tg = now_s();
        if (gpu.wait() != AS_OK) { printf("Error from computeCounts: %s\n", job_err.c_str()); return 1; }
        t_gpu += now_s() - tg;
        carried = have - off;
        if (file_off >= f.n && carried > 0) { printf("Error from computeCounts: %s ends inside a record\n", bam.c_str()); return 1; }
        if (carried > 0) {
            if (!bufs[cur ^ 1].ensure(0, carried)) { printf("Error from computeCounts: out of memory\n"); return 1; }
            memcpy(bufs[cur ^ 1].data(), buf.data() + off, carried);
        }
        if (!rec_off.empty()) {
            const uint8_t* rec = buf.data() + first;
            const int64_t n_bytes = (int64_t)(off - first), n_rec = (int64_t)rec_off.size();
            const int64_t* ro = rec_off.data();
            gpu.submit([&, rec, n_bytes, ro, n_rec]() {
                const int rc = as_pileup_add_host(ctx, rec, n_bytes, ro, n_rec, ref_contig.data(), n_ref, mbq, mrq, 0x704u);
                if (rc != AS_OK) job_err = as_last_error();
                return rc;
            });
        }
        cur ^= 1;
    }
    {
        const double tg = now_s();
        if (gpu.wait() != AS_OK) { printf("Error from computeCounts: %s\n", job_err.c_str()); return 1; }
        t_gpu += now_s() - tg;
    }
    if (!header_done) { printf("Error from computeCounts: %s holds no BAM header\n", bam.c_str()); return 1; }
    // a BAM without records: every count is zero, nothing to report -- still needs no CPU path: the GPU zeroes
    if (!ctx && !(ctx = begin())) return 1;
    if (timing) {
        fprintf(stderr, "AS_TIMING inflate_busy %.6f (%.3g B/s)\n", t_inflate, t_inflate > 0 ? bytes_inflated / t_inflate : 0.0);
        fprintf(stderr, "AS_TIMING pileup_gpu_wait %.6f\n", t_gpu);
    }
    if (n_records_out) *n_records_out = n_records;
    return 0;
}

}  // namespace asbam

extern "C" int as_compute_counts_main(int argc, char** argv) {
    std::string vcf, bam, out = ".";
    int threads = (int)std::max(1u, std::thread::hardware_concurrency()), mbq = 20, mrq = 20, mdc = 20;
    for (int i = 1; i < argc; ++i) {
        std::string v;
        if (!(v = arg_of(argv[i], "vcf=")).empty()) vcf = v;
        else if (!(v = arg_of(argv[i], "bam=")).empty()) bam = v;
        else if (!(v = arg_of(argv[i], "out=")).empty()) out = v;
        else if (!(v = arg_of(argv[i], "threads=")).empty()) threads = std::max(1, atoi(v.c_str()));
        else if (!(v = arg_of(argv[i], "mbq=")).empty()) mbq = atoi(v.c_str());
        else if (!(v = arg_of(argv[i], "mrq=")).empty()) mrq = atoi(v.c_str());
        else if (!(v = arg_of(argv[i], "mdc=")).empty()) mdc = atoi(v.c_str());
        else { printf("Unknown argument: %s\n", argv[i]); usage(); return 0; }
    }
    if (vcf.empty() || bam.empty()) { usage(); return 0; }
    const bool timing = getenv("AS_TIMING") != nullptr;
    double t0 = now_s();
    auto lap = [&](const char* what) {
        const double t1 = now_s();
        if (timing) fprintf(stderr, "AS_TIMING %s %.6f\n", what, t1 - t0);
        t0 = t1;
    };

    // the GPU context starts while the files are opened and the first blocks inflate
    as_ctx* ctx = nullptr;
    int ctx_rc = AS_OK;
    std::string ctx_err;
    // in the resident service the context goes back when the program returns (declared before the joiner: destroyed after it)
    struct CtxGuard { as_ctx*& c; ~CtxGuard() { if (c && as_process_is_resident()) as_destroy(c); } } ctx_guard{ctx};
    std::thread starter([&]() {
        ctx_rc = as_create(0, &ctx);
        if (ctx_rc != AS_OK) ctx_err = as_last_error();
    });
    struct Joiner { std::thread& t; ~Joiner() { if (t.joinable()) t.join(); } } joiner{starter};

    // ---- positions
    struct Line { int32_t contig; int32_t pos0; std::string chr, id, ref, alt; };
    std::vector<Line> lines;
    std::vector<std::string> contig_names;
    std::map<std::string, int32_t> contig_id;
    {
        Mapped m;
        if (!m.open(vcf)) { printf("Error from computeCounts: Cannot open file: %s\n", vcf.c_str()); return 1; }
        const char* p = (const char*)m.p;
        const char* end = p + m.n;
        while (p < end) {
            const char* eol = (const char*)memchr(p, '\n', (size_t)(end - p));
            if (!eol) eol = end;
            if (eol > p && *p != '#') {
                std::vector<std::string> col;
                const char* q = p;
                while (q <= eol && col.size() < 5) {
                    const char* t = q;
                    while (t < eol && *t != '\t' && *t != ' ' && *t != '\r') ++t;
                    if (t > q) col.emplace_back(q, t);
                    if (t >= eol) break;
                    q = t + 1;
                }
                if (col.size() >= 2) {
                    Line l;
                    l.chr = col[0];
                    l.pos0 = (int32_t)atol(col[1].c_str()) - 1;
                    l.id = col.size() > 2 ? col[2] : ".";
                    l.ref = col.size() > 3 ? col[3] : ".";
                    l.alt = col.size() > 4 ? col[4] : ".";
                    auto it = contig_id.find(l.chr);
                    if (it == contig_id.end()) {
                        it = contig_id.emplace(l.chr, (int32_t)contig_names.size()).first;
                        contig_names.push_back(l.chr);
                    }
                    l.contig = it->second;
                    if (l.pos0 >= 0) lines.push_back(std::move(l));
                }
            }
            p = eol + 1;
        }
    }
    if (lines.empty()) { printf("Error from computeCounts: no positions in %s\n", vcf.c_str()); return 1; }
    const int32_t n_contig = (int32_t)contig_names.size();
    std::vector<std::vector<int32_t>> per((size_t)n_contig);
    for (const Line& l : lines) per[(size_t)l.contig].push_back(l.pos0);
    std::vector<int64_t> contig_first((size_t)n_contig + 1, 0);
    std::vector<int32_t> slot_pos;
    for (int32_t c = 0; c < n_contig; ++c) {
        auto& v = per[(size_t)c];
        std::sort(v.begin(), v.end());
        v.erase(std::unique(v.begin(), v.end()), v.end());
        contig_first[(size_t)c + 1] = contig_first[(size_t)c] + (int64_t)v.size();
        slot_pos.insert(slot_pos.end(), v.begin(), v.end());
    }
    const int64_t P = (int64_t)slot_pos.size();
    lap("positions");

    const std::string bam_list = bam;
    asbam::Reader reader;
    auto one_bam = [&](const std::string& bam) -> int {
        uint64_t n_records = 0;
        const int rrc = reader.pileup(bam, contig_id, threads, mbq, mrq, [&]() -> as_ctx* {
            if (starter.joinable()) starter.join();
            if (ctx_rc != AS_OK || !ctx) { printf("Error from computeCounts: %s\n", ctx_err.c_str()); return nullptr; }
            lap("cuda_context_wait");
            if (as_pileup_begin(ctx, contig_first.data(), n_contig, slot_pos.data(), P) != AS_OK) {
                printf("Error from computeCounts: %s\n", as_last_error());
                return nullptr;
            }
            return ctx;
        }, &n_records);
        if (rrc != 0) return rrc;
        std::vector<uint32_t> counts((size_t)P * 8);
        uint64_t stats[2] = {0, 0};
        if (as_pileup_end_host(ctx, counts.data(), stats) != AS_OK) { printf("Error from computeCounts: %s\n", as_last_error()); return 1; }
        lap("inflate_and_pileup");

        // ---- <out>/<name>.PILEUP.ASEQ
        {
            std::string cur;
            for (size_t i = 0; i <= out.size(); ++i) {
                if ((i == out.size() || out[i] == '/') && !cur.empty() && cur != "." && cur != "..") mkdir(cur.c_str(), 0777);
                if (i < out.size()) cur.push_back(out[i]);
            }
        }
        std::string name = bam.substr(bam.find_last_of('/') == std::string::npos ? 0 : bam.find_last_of('/') + 1);
        if (name.size() > 4 && name.compare(name.size() - 4, 4, ".bam") == 0) name.resize(name.size() - 4);
        const std::string path = out + "/" + name + ".PILEUP.ASEQ";
        FILE* o = fopen(path.c_str(), "w");
        if (!o) { printf("Error from computeCounts: Cannot write file: %s\n", path.c_str()); return 1; }
        std::vector<char> obuf(1 << 20);
        setvbuf(o, obuf.data(), _IOFBF, obuf.size());
        fputs("chr\tpos\tdbsnp\tMAF\tref\talt\tA\tC\tG\tT\tRD\tArs\tCrs\tGrs\tTrs\n", o);
        uint64_t rows = 0;
        for (const Line& l : lines) {
            const int64_t c0 = contig_first[(size_t)l.contig], c1 = contig_first[(size_t)l.contig + 1];
            const int64_t j = std::lower_bound(slot_pos.begin() + c0, slot_pos.begin() + c1, l.pos0) - slot_pos.begin();
            const uint32_t* fw = counts.data() + (size_t)j * 4;
            const uint32_t* bw = counts.data() + ((size_t)P + (size_t)j) * 4;
            const uint64_t A = (uint64_t)fw[0] + bw[0], C = (uint64_t)fw[1] + bw[1], G = (uint64_t)fw[2] + bw[2], T = (uint64_t)fw[3] + bw[3];
            const uint64_t rd = A + C + G + T;
            if (rd < (uint64_t)std::max(0, mdc)) continue;
            fprintf(o, "%s\t%d\t%s\t.\t%s\t%s\t%llu\t%llu\t%llu\t%llu\t%llu\t%u\t%u\t%u\t%u\n", l.chr.c_str(), l.pos0 + 1, l.id.c_str(), l.ref.c_str(),
                    l.alt.c_str(), (unsigned long long)A, (unsigned long long)C, (unsigned long long)G, (unsigned long long)T,
                    (unsigned long long)rd, bw[0], bw[1], bw[2], bw[3]);
            rows += 1;
        }
        fclose(o);
        lap("write_aseq");
        printf("computeCounts: %llu records of %s, %llu reads and %llu bases counted on %lld positions, %llu rows (RD >= %d) written to %s\n",
               (unsigned long long)n_records, bam.c_str(), (unsigned long long)stats[0], (unsigned long long)stats[1], (long long)P,
               (unsigned long long)rows, mdc, path.c_str());
    return 0;
    };
    // bam= may name several files (comma-separated, an extension over the reference's one file per run): the position
    // file and the GPU context are set up once and every BAM gets its own <name>.PILEUP.ASEQ
    int rc_all = 0;
    for (size_t a = 0; a <= bam_list.size();) {
        size_t b = bam_list.find(',', a);
        if (b == std::string::npos) b = bam_list.size();
        if (b > a) {
            const int rc = one_bam(bam_list.substr(a, b - a));
            if (rc != 0) rc_all = rc;
        }
        a = b + 1;
    }
    return rc_all;
}
