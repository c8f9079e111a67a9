// urmb_host.cpp -- host side of the drop-in: URMAP's command line, FASTQ/FASTA readers, SAM writer and the
// byte-identical CPU -make_ufi, all above the C-ABI of include/urmb.h.  The per-read search itself only ever
// runs in the CUDA kernels behind urmb_submit/urmb_wait; there is no CPU mapping path in this file.
//
//   urmap_b200 -make_ufi ref.fa -output ref.ufi [-wordlength 24] [-maxix 32] [-slots N] [-load_factor 0.6] [-veryfast] [-gpu_build]
//   urmap_b200 -map reads.fq[.gz] -ufi ref.ufi -samout out.sam [-threads N] [-veryfast] [-gpus G] [-batch N]
//   urmap_b200 -map2 R1.fq -reverse R2.fq -ufi ref.ufi -samout out.sam [-tabbedout out.tab] [-threads N] [-veryfast] [-minq 10]
//   urmap_b200 -map / -map2 ... -ref ref.fa[.gz] [-wordlength 24] [-maxix 32] [-slots N] [-load_factor 0.6] (index built on the
//              GPU(s) at start-up, the table -make_ufi writes for the same options; no UFI file)
//   urmap_b200 -ufi_info ref.ufi
//   urmap_b200 -ufi_validate ref.ufi          (also: -make_ufi ... -validate)
//
// Reference behaviour restated here (file:line under /root/reference/src):
//   option spellings / errors   cmdline.cpp:148-269, myopts.h, getcmd.cpp:6-26, myutils.cpp:915-960
//   FASTQ records               fastqseqsource.cpp:9-116, linereader.cpp:54-99
//   FASTA -> SeqData            fastaseqsource.cpp:26-112, ufindex.cpp:462-510 (upper-case, 32 x '-' pads)
//   index construction          ufindex.cpp:83-408, 945-1000; ufindexio.cpp:15-49,117-179; prime.cpp:11
//   SAM text                    setsam.cpp:12-207, output1.cpp:8-30, output2.cpp:18-132, state1.cpp:129-145,736-752
//   CIGAR                       cigar.cpp:4-41,141-199, state1.cpp:717-734
//   end-of-run summary          state1.cpp:593-632
#include <ctype.h>
#include <errno.h>
#include <fcntl.h>
#include <omp.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <sys/mman.h>
#include <sys/resource.h>
#include <sys/stat.h>
#include <unistd.h>
#include <zlib.h>
#if defined(__SSE2__)
#include <emmintrin.h>
#endif

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <functional>
#include <memory>
#include <mutex>
#include <string>
#include <thread>
#include <vector>

#include "../../include/urmb.h"

extern "C" int urmb_build_index_device(const void *d_seq, uint64_t seq_data_size, uint64_t slot_count,
                                       uint32_t word_length, uint32_t max_ix, void *d_blob, uint64_t *stats);
extern "C" const char *urmb_build_last_error();

#define URMB_VERSION "0.1"

static std::vector<std::string> g_argv;
static bool g_quiet = false;
static FILE *g_log = nullptr;

[[noreturn]] static void Die(const char *fmt, ...) {  // myutils.cpp:915-960
    char msg[4096];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(msg, sizeof msg, fmt, ap);
    va_end(ap);
    for (FILE *f : {stderr, g_log}) {
        if (!f) continue;
        fprintf(f, "\n");
        for (auto &a : g_argv) fprintf(f, "%s ", a.c_str());
        fprintf(f, "\n\n---Fatal error---\n%s\n", msg);
        fflush(f);
    }
    exit(1);
}

static void Progress(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    if (!g_quiet) {
        va_list ap2;
        va_copy(ap2, ap);
        vfprintf(stderr, fmt, ap2);
        va_end(ap2);
    }
    if (g_log) vfprintf(g_log, fmt, ap);
    va_end(ap);
}

static double now_s() {
    return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// ------------------------------------------------------------------------------------------------
// options
// ------------------------------------------------------------------------------------------------
struct Opts {
    std::string make_ufi, map, map2, reverse, ufi, ref, samout, output, log, slots, ufi_info, ufi_validate, fastq_dump, sam_bench, tabbedout;
    unsigned threads = 0, wordlength = 24, maxix = 32, minq = 10, gpus = 1, batch = 262144;
    double load_factor = 0.6;
    bool veryfast = false, quiet = false, gpu_build = false, version = false, validate = false;
    bool set_maxix = false, set_wordlength = false, set_threads = false;
    std::vector<std::string> given;   // every option name on the command line (CheckUsedOpts, cmdline.cpp:13-26)
};

static Opts ParseCmdLine(int argc, char **argv) {
    Opts o;
    auto bad = [&](const std::string &why) {
        fprintf(stderr, "\nInvalid command line\n%s\n\n", why.c_str());  // cmdline.cpp:28-38
        exit(1);
    };
    // "file: args.txt" anywhere on the command line is replaced by the white-space separated fields of that file, '#' starts
    // a comment (cmdline.cpp:40-56,162-179)
    std::vector<std::string> args;
    for (int i = 0; i < argc;) {
        if (std::string(argv[i]) == "file:" && i + 1 < argc) {
            FILE *f = fopen(argv[i + 1], "rb");
            if (!f) Die("Cannot open %s", argv[i + 1]);
            std::string line;
            int c;
            auto flush = [&]() {
                const size_t h = line.find('#');
                if (h != std::string::npos) line.resize(h);
                size_t k = 0;
                while (k < line.size()) {
                    while (k < line.size() && isspace((unsigned char)line[k])) ++k;
                    size_t e = k;
                    while (e < line.size() && !isspace((unsigned char)line[e])) ++e;
                    if (e > k) args.push_back(line.substr(k, e - k));
                    k = e;
                }
                line.clear();
            };
            while ((c = fgetc(f)) != EOF) {
                if (c == '\n') flush();
                else if (c != '\r') line.push_back((char)c);
            }
            flush();
            fclose(f);
            i += 2;
        } else {
            args.push_back(argv[i]);
            i += 1;
        }
    }
    g_argv = args;
    argc = (int)args.size();
    std::vector<char *> argp;
    for (auto &a : args) argp.push_back(const_cast<char *>(a.c_str()));
    argv = argp.data();
    for (int i = 1; i < argc; ++i) {
        std::string a = argv[i];
        if (a.size() < 2 || a[0] != '-') bad("Expected -option_name, got '" + a + "'");
        std::string name = a.substr(a[1] == '-' ? 2 : 1);
        o.given.push_back(name);
        auto val = [&]() -> std::string {
            if (i + 1 >= argc) bad("Missing value for option -" + name);
            return std::string(argv[++i]);
        };
        if (name == "make_ufi") o.make_ufi = val();
        else if (name == "map") o.map = val();
        else if (name == "map2") o.map2 = val();
        else if (name == "reverse") o.reverse = val();
        else if (name == "ufi_info") o.ufi_info = val();
        else if (name == "ufi_validate") o.ufi_validate = val();
        else if (name == "validate") o.validate = true;
        else if (name == "fastq_dump") o.fastq_dump = val();
        else if (name == "sam_bench") o.sam_bench = val();
        else if (name == "ufi") o.ufi = val();
        else if (name == "ref") o.ref = val();
        else if (name == "samout") o.samout = val();
        else if (name == "tabbedout") o.tabbedout = val();
        else if (name == "output") o.output = val();
        else if (name == "log") o.log = val();
        else if (name == "slots") o.slots = val();
        else if (name == "threads") { o.threads = (unsigned)strtoul(val().c_str(), nullptr, 10); o.set_threads = true; }
        else if (name == "wordlength") { o.wordlength = (unsigned)strtoul(val().c_str(), nullptr, 10); o.set_wordlength = true; }
        else if (name == "maxix") { o.maxix = (unsigned)strtoul(val().c_str(), nullptr, 10); o.set_maxix = true; }
        else if (name == "minq") o.minq = (unsigned)strtoul(val().c_str(), nullptr, 10);
        else if (name == "load_factor") o.load_factor = atof(val().c_str());
        else if (name == "gpus") o.gpus = (unsigned)strtoul(val().c_str(), nullptr, 10);
        else if (name == "batch") o.batch = (unsigned)strtoul(val().c_str(), nullptr, 10);
        else if (name == "veryfast") o.veryfast = true;
        else if (name == "quiet") o.quiet = true;
        else if (name == "gpu_build") o.gpu_build = true;
        else if (name == "version") o.version = true;
        else bad("Unknown option " + name);
    }
    int ncmd = (!o.make_ufi.empty()) + (!o.map.empty()) + (!o.map2.empty()) + (o.version ? 1 : 0) + (!o.ufi_info.empty()) +
               (!o.ufi_validate.empty()) + (!o.fastq_dump.empty()) + (!o.sam_bench.empty());
    if (ncmd == 0) bad("No command specified");       // getcmd.cpp:6-11
    if (ncmd > 1) bad("Two commands specified");
    return o;
}

// ------------------------------------------------------------------------------------------------
// line reader (plain or .gz), linereader.cpp:54-99: CR dropped, last line may lack LF
// ------------------------------------------------------------------------------------------------
class LineReader {
   public:
    explicit LineReader(const std::string &path) : path_(path) {
        gz_ = gzopen(path.c_str(), "rb");  // transparently reads uncompressed files too
        if (!gz_) Die("Cannot open %s", path.c_str());
        gzbuffer(gz_, 1 << 20);
        buf_.resize(32u << 20);
    }
    ~LineReader() { if (gz_) gzclose(gz_); }
    // returns false at EOF with nothing read; line excludes the terminator
    bool ReadLine(const char *&p, size_t &n) {
        line_.clear();
        bool any = false;
        for (;;) {
            if (off_ >= len_) {
                if (eof_) break;
                int r = gzread(gz_, buf_.data(), (unsigned)buf_.size());
                if (r < 0) Die("Read error in %s", path_.c_str());
                len_ = (size_t)r;
                off_ = 0;
                if (r == 0) { eof_ = true; break; }
            }
            const char *b = buf_.data() + off_;
            const char *e = (const char *)memchr(b, '\n', len_ - off_);
            size_t m = e ? (size_t)(e - b) : len_ - off_;
            if (line_.empty() && e) {  // fast path: whole line inside the buffer
                ++line_nr_;
                off_ += m + 1;
                if (memchr(b, '\r', m) == nullptr) { p = b; n = m; return true; }
                append_nocr(b, m);
                p = line_.data(); n = line_.size();
                return true;
            }
            append_nocr(b, m);
            any = true;
            off_ += m + (e ? 1 : 0);
            if (e) { ++line_nr_; p = line_.data(); n = line_.size(); return true; }
        }
        if (!any && line_.empty()) return false;
        ++line_nr_;
        p = line_.data(); n = line_.size();
        return n > 0;
    }
    unsigned line_nr() const { return line_nr_; }
    const std::string &path() const { return path_; }

   private:
    void append_nocr(const char *b, size_t m) {
        for (size_t i = 0; i < m; ++i) if (b[i] != '\r') line_.push_back(b[i]);
    }
    std::string path_;
    gzFile gz_ = nullptr;
    std::vector<char> buf_;
    size_t off_ = 0, len_ = 0;
    bool eof_ = false;
    std::string line_;
    unsigned line_nr_ = 0;
};

// ------------------------------------------------------------------------------------------------
// worker pool: Run(fn) executes fn(t, n) on n persistent threads (t = 0 runs on the caller)
// ------------------------------------------------------------------------------------------------
class Pool {
   public:
    explicit Pool(int n) : n_(std::max(1, n)) {
        for (int t = 1; t < n_; ++t) th_.emplace_back([this, t]() { Loop(t); });
    }
    ~Pool() {
        {
            std::lock_guard<std::mutex> lk(mu_);
            stop_ = true;
        }
        cv_.notify_all();
        for (auto &t : th_) t.join();
    }
    int size() const { return n_; }
    template <class F>
    void Run(F &&fn) {
        std::function<void(int, int)> f = std::forward<F>(fn);
        {
            std::lock_guard<std::mutex> lk(mu_);
            fn_ = &f;
            left_ = n_ - 1;
            ++gen_;
        }
        cv_.notify_all();
        f(0, n_);
        std::unique_lock<std::mutex> lk(mu_);
        done_.wait(lk, [this]() { return left_ == 0; });
        fn_ = nullptr;
    }

   private:
    void Loop(int t) {
        uint64_t seen = 0;
        for (;;) {
            const std::function<void(int, int)> *f;
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [&]() { return stop_ || gen_ != seen; });
                if (stop_) return;
                seen = gen_;
                f = fn_;
            }
            (*f)(t, n_);
            std::lock_guard<std::mutex> lk(mu_);
            if (--left_ == 0) done_.notify_one();
        }
    }
    int n_;
    std::vector<std::thread> th_;
    std::mutex mu_;
    std::condition_variable cv_, done_;
    const std::function<void(int, int)> *fn_ = nullptr;
    uint64_t gen_ = 0;
    int left_ = 0;
    bool stop_ = false;
};

// ------------------------------------------------------------------------------------------------
// FASTQ batches.  The reference parses a byte at a time under a global lock (seqsource.cpp:37-49,
// linereader.cpp:54-99); here a batch is carved out of a large window of the (decompressed) file: newline positions are
// found by all threads in parallel, records are validated and their bases copied into one contiguous buffer (what the
// C ABI takes) in parallel, labels and qualities stay where they are (the window) and are read again by the SAM writer.
// ------------------------------------------------------------------------------------------------
struct RawBuf {   // recycled byte buffer (no zero-fill, no shrink)
    char *p = nullptr;
    size_t cap = 0;
    ~RawBuf() { free(p); }
    void need(size_t n, size_t keep = 0) {
        if (n <= cap) return;
        size_t ncap = std::max(n, cap + cap / 2);
        char *q = (char *)malloc(ncap);
        if (!q) Die("Out of memory (%zu bytes)", ncap);
        if (keep) memcpy(q, p, keep);
        free(p);
        p = q;
        cap = ncap;
    }
};

struct PinnedBuf {   // bases of a batch in page-locked memory: urmb_submit then copies them to the device without staging
    char *p = nullptr;
    size_t cap = 0;
    bool pinned = false;
    ~PinnedBuf() { release(); }
    void release() {
        if (pinned) urmb_host_free(p); else free(p);
        p = nullptr;
        cap = 0;
    }
    void need(size_t n) {   // contents are not kept
        if (n <= cap) return;
        release();
        const size_t ncap = ((n + n / 8) | ((1u << 20) - 1)) + 1;
        void *q = nullptr;
        static bool can_pin = true;   // false once the driver said no (host-only diagnostics without a GPU)
        if (can_pin && urmb_host_alloc(ncap, &q) == 0) pinned = true;
        else {
            can_pin = false;
            pinned = false;
            q = malloc(ncap);
            if (!q) Die("Out of memory (%zu bytes)", ncap);
        }
        p = (char *)q;
        cap = ncap;
    }
};

struct HostBatch {
    uint32_t n = 0;
    PinnedBuf seqs;                    // bases of all reads, concatenated
    std::vector<uint32_t> offs;        // n + 1 offsets into seqs
    std::vector<uint32_t> lab, lablen, qual;   // per read: label / quality offsets into text
    const char *text = nullptr;        // the window the offsets refer to: own.p or a view into the mapped file
    RawBuf own;                        // window bytes when they had to be materialised (gz input, CR stripping)
    const uint8_t *Seq(uint32_t i) const { return (const uint8_t *)seqs.p + offs[i]; }
    unsigned Len(uint32_t i) const { return offs[i + 1] - offs[i]; }
    const uint8_t *Label(uint32_t i) const { return (const uint8_t *)text + lab[i]; }
    const uint8_t *Qual(uint32_t i) const { return (const uint8_t *)text + qual[i]; }
};

class FastqReader {  // FASTQSeqSource::GetNextLo, fastqseqsource.cpp:9-116
   public:
    FastqReader(const std::string &path, Pool &pool) : path_(path), pool_(pool) {
        FILE *f = fopen(path.c_str(), "rb");
        if (!f) Die("Cannot open %s", path.c_str());
        unsigned char magic[2] = {0, 0};
        size_t got = fread(magic, 1, 2, f);
        struct stat sb;
        const bool regular = fstat(fileno(f), &sb) == 0 && S_ISREG(sb.st_mode);
        fclose(f);
        if (regular && !(got == 2 && magic[0] == 0x1f && magic[1] == 0x8b) && sb.st_size > 0) {
            int fd = open(path.c_str(), O_RDONLY);
            if (fd < 0) Die("Cannot open %s", path.c_str());
            void *m = mmap(nullptr, (size_t)sb.st_size, PROT_READ, MAP_PRIVATE, fd, 0);
            close(fd);
            if (m != MAP_FAILED) {
                madvise(m, (size_t)sb.st_size, MADV_SEQUENTIAL);
                map_ = (const char *)m;
                map_len_ = (size_t)sb.st_size;
            }
        }
        if (!map_) {   // compressed, a pipe, or empty: stream through zlib (reads plain data transparently too)
            gz_ = gzopen(path.c_str(), "rb");
            if (!gz_) Die("Cannot open %s", path.c_str());
            gzbuffer(gz_, 1 << 20);
        }
    }
    ~FastqReader() {
        if (gz_) gzclose(gz_);
        if (map_) munmap((void *)map_, map_len_);
    }

    // Fills b with up to max_reads records; returns the number read (0 at end of file).
    uint32_t Fill(HostBatch &b, uint32_t max_reads) {
        b.n = 0;
        b.offs.assign(1, 0);
        if (finished_ || max_reads == 0) return 0;
        size_t want = std::max<size_t>((size_t)(max_reads * est_rec_ * 1.05) + 4096, 1 << 16);
        const char *w = nullptr;
        size_t wn = 0;
        bool eof = false, stripped = false;
        for (;;) {   // grow the window until it holds 4 * max_reads lines or the rest of the file
            Window(b, want, w, wn, eof, stripped);
            if (ScanLines(w, wn, eof) /* saw '\r' */ && !stripped) {
                // CR bytes are dropped wherever they are (linereader.cpp:75): rare, so strip them from a private copy
                stripped = true;
                continue;
            }
            if (nl_.size() >= 4 * (size_t)max_reads || eof) break;
            want = want + want / 2 + (1 << 20);
        }
        size_t lines = nl_.size();
        if (eof) {   // empty lines are allowed at the end of the file only ...
            const size_t all = lines;
            while (lines > 0 && LineLen(lines - 1) == 0) --lines;
            // ... but the empty sequence / quality lines of a last record ("@r", "", "+", "") belong to it
            if (lines % 4 != 0 && lines + (4 - lines % 4) <= all) lines += 4 - lines % 4;
        }
        uint32_t nrec = (uint32_t)std::min<size_t>(lines / 4, max_reads);
        // an empty line where a record should start: fine if nothing but empty lines follows, fatal otherwise
        const uint32_t cand = (uint32_t)std::min<size_t>((lines + 3) / 4, max_reads);
        const uint32_t first_empty = FirstEmptyLabel(cand);
        if (first_empty < cand) {
            const unsigned ln = line_base_ + 4 * first_empty + 1;
            if (!RestIsEmpty(w, wn, LineStart(4 * (size_t)first_empty), eof))
                Die("Empty line nr %u in FASTQ file '%s'", ln, path_.c_str());
            nrec = first_empty;
            finished_ = true;
        } else if (eof && lines % 4 != 0 && lines / 4 < max_reads) {
            // a truncated last record: the reference dies when it runs out of lines inside a record
            CheckLabelLines(w, (uint32_t)(lines / 4) + 1, lines);
            Die("Unexpected end-of-file in FASTQ file %s", path_.c_str());
        }
        Parse(b, w, nrec);
        const size_t used = nrec ? (size_t)nl_[4 * (size_t)nrec - 1] + 1 : 0;
        Consume(b, w, std::min(used, wn), wn);
        line_base_ += 4 * nrec;
        if (nrec) est_rec_ = std::max(16.0, (double)used / nrec);
        if (nrec < max_reads && (eof || finished_)) finished_ = true;
        return nrec;
    }

   private:
    // ---- window management: [w, w + wn) are the next unread bytes of the decompressed file
    void Window(HostBatch &b, size_t want, const char *&w, size_t &wn, bool &eof, bool strip_cr) {
        if (map_ && !strip_cr && !seen_cr_) {
            w = map_ + map_pos_;
            wn = std::min(want, map_len_ - map_pos_);
            eof = map_pos_ + wn == map_len_;
            b.text = w;
            return;
        }
        // materialised window in b.own: carry-over of the previous batch first, then fresh bytes
        RawBuf &o = b.own;
        if (carry_n_) {
            o.need(std::max(want, carry_n_));
            memcpy(o.p, carry_.p, carry_n_);
            own_n_ = carry_n_;
            carry_n_ = 0;
        }
        o.need(want + 1, own_n_);
        while (own_n_ < want && !src_eof_) {
            size_t got;
            if (map_) {   // CR stripping of a mapped file
                got = std::min(want - own_n_, map_len_ - map_pos_);
                memcpy(o.p + own_n_, map_ + map_pos_, got);
                map_pos_ += got;
                if (map_pos_ == map_len_) src_eof_ = true;
            } else {
                int r = gzread(gz_, o.p + own_n_, (unsigned)std::min<size_t>(want - own_n_, 1u << 30));
                if (r < 0) Die("Read error in %s", path_.c_str());
                got = (size_t)r;
                if (r == 0) src_eof_ = true;
            }
            if (strip_cr || seen_cr_) {
                char *e = std::remove(o.p + own_n_, o.p + own_n_ + got, '\r');
                got = (size_t)(e - (o.p + own_n_));
            }
            own_n_ += got;
        }
        if (strip_cr && !seen_cr_) {   // first CR seen: also clean what was already in the window
            seen_cr_ = true;
            own_n_ = (size_t)(std::remove(o.p, o.p + own_n_, '\r') - o.p);
        }
        w = o.p;
        wn = own_n_;
        eof = src_eof_;
        b.text = w;
    }
    void Consume(HostBatch &b, const char *w, size_t used, size_t wn) {
        if (map_ && !seen_cr_) { map_pos_ += used; return; }
        carry_n_ = wn - used;   // unread tail of the materialised window goes to the next batch
        if (carry_n_) {
            carry_.need(carry_n_);
            memcpy(carry_.p, w + used, carry_n_);
        }
        own_n_ = 0;
    }

    // newline offsets of w[lo, hi) appended to v, 64 bytes per step (SSE2 compares, one bit per byte); true if a CR was seen
    static bool ScanRange(const char *w, size_t lo, size_t hi, std::vector<uint32_t> &v) {
        size_t i = lo;
        bool cr = false;
#if defined(__SSE2__)
        const __m128i nl = _mm_set1_epi8('\n'), crv = _mm_set1_epi8('\r');
        v.reserve(v.size() + (hi - lo) / 48 + 16);
        for (; i + 64 <= hi; i += 64) {
            const __m128i a = _mm_loadu_si128((const __m128i *)(w + i)), b = _mm_loadu_si128((const __m128i *)(w + i + 16));
            const __m128i c = _mm_loadu_si128((const __m128i *)(w + i + 32)), d = _mm_loadu_si128((const __m128i *)(w + i + 48));
            uint64_t m = (uint64_t)(uint32_t)_mm_movemask_epi8(_mm_cmpeq_epi8(a, nl)) |
                         ((uint64_t)(uint32_t)_mm_movemask_epi8(_mm_cmpeq_epi8(b, nl)) << 16) |
                         ((uint64_t)(uint32_t)_mm_movemask_epi8(_mm_cmpeq_epi8(c, nl)) << 32) |
                         ((uint64_t)(uint32_t)_mm_movemask_epi8(_mm_cmpeq_epi8(d, nl)) << 48);
            const __m128i anycr = _mm_or_si128(_mm_or_si128(_mm_cmpeq_epi8(a, crv), _mm_cmpeq_epi8(b, crv)),
                                               _mm_or_si128(_mm_cmpeq_epi8(c, crv), _mm_cmpeq_epi8(d, crv)));
            if (_mm_movemask_epi8(anycr)) cr = true;
            while (m) {
                v.push_back((uint32_t)(i + (size_t)__builtin_ctzll(m)));
                m &= m - 1;
            }
        }
#endif
        for (; i < hi; ++i) {
            if (w[i] == '\n') v.push_back((uint32_t)i);
            else if (w[i] == '\r') cr = true;
        }
        return cr;
    }

    // every byte a letter (fastqseqsource.cpp:60-70 rejects anything else)
    static bool AllAlpha(const char *p, size_t n) {
        size_t i = 0;
        unsigned bad = 0;
#if defined(__SSE2__)
        const __m128i lower = _mm_set1_epi8(0x20), a = _mm_set1_epi8('a'), lim = _mm_set1_epi8(25);
        __m128i acc = _mm_setzero_si128();
        for (; i + 16 <= n; i += 16) {
            const __m128i x = _mm_sub_epi8(_mm_or_si128(_mm_loadu_si128((const __m128i *)(p + i)), lower), a);
            acc = _mm_or_si128(acc, _mm_subs_epu8(x, lim));   // non-zero where x > 25 (unsigned)
        }
        bad = (unsigned)_mm_movemask_epi8(_mm_cmpeq_epi8(acc, _mm_setzero_si128())) ^ 0xFFFFu;
#endif
        for (; i < n; ++i) bad |= (unsigned)(((unsigned char)(((unsigned char)p[i] | 0x20) - 'a')) > 25);
        return bad == 0;
    }

    // ---- newline index of the window; returns true when a CR byte was seen
    bool ScanLines(const char *w, size_t wn, bool eof) {
        const int T = pool_.size();
        if ((int)parts_.size() < T) parts_.resize(T);
        std::vector<char> cr(T, 0);
        pool_.Run([&](int t, int nt) {
            std::vector<uint32_t> v;   // local header: the threads' vector objects would share cache lines
            v.swap(parts_[t]);
            v.clear();
            const size_t lo = wn * t / nt, hi = wn * (t + 1) / nt;
            if (ScanRange(w, lo, hi, v)) cr[t] = 1;
            v.swap(parts_[t]);
        });
        for (int t = 0; t < T; ++t) if (cr[t]) return true;
        size_t total = 0;
        std::vector<size_t> base(T + 1, 0);
        for (int t = 0; t < T; ++t) { base[t] = total; total += parts_[t].size(); }
        const bool virt = eof && wn > 0 && w[wn - 1] != '\n';   // last line of the file may lack its LF
        nl_.resize(total + (virt ? 1 : 0));
        pool_.Run([&](int t, int) {
            if (!parts_[t].empty()) memcpy(nl_.data() + base[t], parts_[t].data(), parts_[t].size() * sizeof(uint32_t));
        });
        if (virt) nl_[total] = (uint32_t)wn;
        return false;
    }
    size_t LineStart(size_t line) const { return line ? (size_t)nl_[line - 1] + 1 : 0; }
    size_t LineLen(size_t line) const { return (size_t)nl_[line] - LineStart(line); }
    uint32_t FirstEmptyLabel(uint32_t nrec) {
        std::vector<uint32_t> first(pool_.size(), nrec);
        pool_.Run([&](int t, int nt) {
            const uint32_t lo = (uint32_t)((uint64_t)nrec * t / nt), hi = (uint32_t)((uint64_t)nrec * (t + 1) / nt);
            for (uint32_t r = lo; r < hi; ++r)
                if (LineLen(4 * (size_t)r) == 0) { first[t] = r; break; }
        });
        return *std::min_element(first.begin(), first.end());
    }
    bool RestIsEmpty(const char *w, size_t wn, size_t from, bool eof) {
        for (size_t i = from; i < wn; ++i) if (w[i] != '\n' && w[i] != '\r') return false;
        if (eof) return true;
        if (map_) {   // bytes of the file behind the window
            const size_t start = (w >= map_ && w < map_ + map_len_) ? (size_t)(w - map_) + wn : map_pos_;
            for (size_t i = start; i < map_len_; ++i) if (map_[i] != '\n' && map_[i] != '\r') return false;
            return true;
        }
        std::vector<char> tmp(1 << 20);
        for (;;) {
            int r = gzread(gz_, tmp.data(), (unsigned)tmp.size());
            if (r < 0) Die("Read error in %s", path_.c_str());
            if (r == 0) return true;
            for (int i = 0; i < r; ++i) if (tmp[i] != '\n' && tmp[i] != '\r') return false;
        }
    }
    void CheckLabelLines(const char *w, uint32_t nrec, size_t lines) {
        for (uint32_t r = 0; r < nrec && 4 * (size_t)r < lines; ++r)
            if (LineLen(4 * (size_t)r) && w[LineStart(4 * (size_t)r)] != '@')
                Die("Bad line %u in FASTQ file '%s': expected '@'", line_base_ + 4 * r + 1, path_.c_str());
    }

    // ---- records [0, nrec) of the window -> b
    void Parse(HostBatch &b, const char *w, uint32_t nrec) {
        b.n = nrec;
        b.offs.resize((size_t)nrec + 1);
        b.lab.resize(nrec);
        b.lablen.resize(nrec);
        b.qual.resize(nrec);
        const int T = pool_.size();
        std::vector<uint64_t> sum(T + 1, 0);
        struct Bad { uint32_t rec = UINT32_MAX; int kind = 0; unsigned a = 0, b = 0; };
        std::vector<Bad> bad(T);
        // pass 1: line geometry (no byte of the records is touched but the '@')
        pool_.Run([&](int t, int nt) {
            const uint32_t lo = (uint32_t)((uint64_t)nrec * t / nt), hi = (uint32_t)((uint64_t)nrec * (t + 1) / nt);
            uint64_t s = 0;
            for (uint32_t r = lo; r < hi; ++r) {
                const size_t l0 = 4 * (size_t)r;
                const size_t s0 = LineStart(l0), n0 = (size_t)nl_[l0] - s0;
                const size_t s1 = (size_t)nl_[l0] + 1, n1 = (size_t)nl_[l0 + 1] - s1;
                const size_t s3 = (size_t)nl_[l0 + 2] + 1, n3 = (size_t)nl_[l0 + 3] - s3;
                if (w[s0] != '@') { if (bad[t].rec == UINT32_MAX) bad[t] = Bad{r, 1, 0, 0}; }
                else if (n3 != n1) { if (bad[t].rec == UINT32_MAX) bad[t] = Bad{r, 2, (unsigned)n1, (unsigned)n3}; }
                b.lab[r] = (uint32_t)(s0 + 1);
                b.lablen[r] = (uint32_t)(n0 - 1);
                b.qual[r] = (uint32_t)s3;
                b.offs[r + 1] = (uint32_t)n1;   // length for now
                s += n1;
            }
            sum[t + 1] = s;
        });
        for (int t = 0; t < T; ++t) sum[t + 1] += sum[t];
        if (sum[T] >= 0xFFFFFFF0ull) Die("FASTQ batch larger than 4 GB of bases; use a smaller -batch");
        b.seqs.need(sum[T] + 64);
        // pass 2: offsets, base validation and copy
        pool_.Run([&](int t, int nt) {
            const uint32_t lo = (uint32_t)((uint64_t)nrec * t / nt), hi = (uint32_t)((uint64_t)nrec * (t + 1) / nt);
            uint32_t off = (uint32_t)sum[t];
            for (uint32_t r = lo; r < hi; ++r) {
                const uint32_t L = b.offs[r + 1];
                const char *src = w + (size_t)nl_[4 * (size_t)r] + 1;
                char *dst = b.seqs.p + off;
                memcpy(dst, src, L);
                const bool badc = !AllAlpha(src, L);
                if (badc && bad[t].rec == UINT32_MAX) bad[t] = Bad{r, 3, 0, 0};
                off += L;
                b.offs[r + 1] = off;
            }
        });
        b.offs[0] = 0;
        Bad first;
        for (int t = 0; t < T; ++t) if (bad[t].rec < first.rec) first = bad[t];
        if (first.rec != UINT32_MAX) {
            const unsigned ln = line_base_ + 4 * first.rec;
            if (first.kind == 1) Die("Bad line %u in FASTQ file '%s': expected '@'", ln + 1, path_.c_str());
            if (first.kind == 2)
                Die("Bad FASTQ record: %u bases, %u quals line %u file %s label %.*s", first.a, first.b, ln + 4, path_.c_str(),
                    (int)b.lablen[first.rec], (const char *)b.Label(first.rec));
            const uint8_t *s = b.Seq(first.rec);
            for (unsigned i = 0; i < b.Len(first.rec); ++i)
                if (!isalpha(s[i])) {
                    if (isprint(s[i])) Die("Invalid sequence letter '%c' in FASTQ, line %u file %s", s[i], ln + 2, path_.c_str());
                    Die("Non-printing byte 0x%02x in FASTQ sequence line %u file %s", s[i], ln + 2, path_.c_str());
                }
        }
    }

    std::string path_;
    Pool &pool_;
    gzFile gz_ = nullptr;
    const char *map_ = nullptr;
    size_t map_len_ = 0, map_pos_ = 0;
    RawBuf carry_;
    size_t carry_n_ = 0, own_n_ = 0;
    bool src_eof_ = false, seen_cr_ = false, finished_ = false;
    std::vector<std::vector<uint32_t>> parts_;
    std::vector<uint32_t> nl_;
    double est_rec_ = 400.0;
    unsigned line_base_ = 0;
};

// ------------------------------------------------------------------------------------------------
// alphabet helpers (alpha.cpp:1309, 3005, 3525)
// ------------------------------------------------------------------------------------------------
static uint8_t g_Letter[256], g_CompLetter[256], g_CompChar[256];
static void InitAlpha() {
    memset(g_Letter, 0xFF, 256);
    memset(g_CompLetter, 0xFF, 256);
    memset(g_CompChar, '?', 256);
    const char *s = "ACGTU";
    const uint8_t v[5] = {0, 1, 2, 3, 3};
    for (int i = 0; i < 5; ++i) {
        g_Letter[(uint8_t)s[i]] = v[i];
        g_Letter[(uint8_t)(s[i] | 0x20)] = v[i];
        g_CompLetter[(uint8_t)s[i]] = 3 - v[i];
        if (s[i] != 'U') g_CompLetter[(uint8_t)(s[i] | 0x20)] = 3 - v[i];
    }
    const char *from = "ABCDGHKMNRSTUVWXY", *to = "TVGHCDMKNYSAABWXR";
    for (int i = 0; from[i]; ++i) {
        g_CompChar[(uint8_t)from[i]] = (uint8_t)to[i];
        if (from[i] != 'U') g_CompChar[(uint8_t)(from[i] | 0x20)] = (uint8_t)(to[i] | 0x20);
    }
}

// ------------------------------------------------------------------------------------------------
// SAM
// ------------------------------------------------------------------------------------------------
struct Contigs {
    std::vector<std::string> labels;
    std::vector<uint32_t> lengths, offsets;
    // UFIndex::PosToCoordL, ufindex.cpp:729-755
    uint32_t PosToCoordL(uint32_t Pos, int &idx, uint32_t &L) const {
        int64_t Lo = 0, Hi = (int64_t)labels.size() - 1;
        while (Lo <= Hi) {
            int64_t k = (Lo + Hi) / 2;
            uint32_t Off = offsets[k], Len = lengths[k];
            if (Pos >= Off && Pos < Off + Len) { idx = (int)k; L = Len; return Pos - Off; }
            if (Pos > Off) Lo = k + 1; else Hi = k - 1;
        }
        idx = -1;
        L = 0;
        return UINT32_MAX;
    }
};

// Append-only text buffer of one formatter thread (capacity is kept from batch to batch).
struct alignas(128) OutBuf {   // one per formatter thread: own cache lines, the counters are written per byte
    char *p = nullptr;
    size_t n = 0, cap = 0;
    ~OutBuf() { free(p); }
    void clear() { n = 0; }
    size_t size() const { return n; }
    const char *data() const { return p; }
    void reserve(size_t want) {   // one allocation up front: growing a large block under many threads is what costs
        if (want <= cap) return;
        char *q = (char *)malloc(want);
        if (!q) Die("Out of memory (%zu bytes of SAM text)", want);
        if (n) memcpy(q, p, n);
        free(p);
        p = q;
        cap = want;
    }
    inline char *room(size_t k) {   // pointer to k writable bytes at the end (not yet counted)
        if (n + k > cap) {
            cap = std::max(n + k, cap + cap / 2 + 4096);
            p = (char *)realloc(p, cap);
            if (!p) Die("Out of memory (%zu bytes of SAM text)", cap);
        }
        return p + n;
    }
    inline void push_back(char c) { *room(1) = c; ++n; }
    inline void append(const char *s, size_t k) { memcpy(room(k), s, k); n += k; }
    inline OutBuf &operator+=(const std::string &s) { append(s.data(), s.size()); return *this; }
    inline OutBuf &operator+=(const char *s) { append(s, strlen(s)); return *this; }
};

static inline void put_u(OutBuf &o, uint32_t v) {
    char t[12];
    int k = 12;
    do { t[--k] = (char)('0' + v % 10); v /= 10; } while (v);
    o.append(t + k, 12 - k);
}
static inline void put_i(OutBuf &o, int v) {
    if (v < 0) { o.push_back('-'); put_u(o, (uint32_t)(-(int64_t)v)); }
    else put_u(o, (uint32_t)v);
}

// PathToCIGAR (cigar.cpp:4-41, D<->I swapped) + CIGAROpsFixDanglingMs (cigar.cpp:141-199).  The reference's
// second fix-up block cannot fire once the first has (it would need a length that is both <= 2 and > 4).
static void RunsToCigar(const uint16_t *runs, unsigned nruns, unsigned QL, OutBuf &o) {
    if (nruns == 0) { put_u(o, QL); o.push_back('M'); return; }
    char ops[512];
    unsigned lens[512];
    unsigned N = 0;
    for (unsigned i = 0; i < nruns && N < 512; ++i) {
        unsigned op = runs[i] & 3, len = runs[i] >> 2;
        char c = op == 0 ? 'M' : (op == 1 ? 'I' : 'D');
        if (N && ops[N - 1] == c) lens[N - 1] += len;
        else { ops[N] = c; lens[N] = len; ++N; }
    }
    unsigned first = 0, last = N;
    if (N >= 3) {
        if (ops[0] == 'M' && lens[0] <= 2 && lens[1] > 4 && ops[2] == 'M') { lens[2] += lens[0]; first = 1; }
        else if (ops[N - 1] == 'M' && lens[N - 1] <= 2 && lens[N - 2] > 4 && ops[N - 3] == 'M') { lens[N - 3] += lens[N - 1]; last = N - 1; }
    }
    for (unsigned i = first; i < last; ++i) { put_u(o, lens[i]); o.push_back(ops[i]); }
}

static void AppendQName(OutBuf &o, const uint8_t *Label, unsigned n) {  // setsam.cpp:32-44
    if (n > 2 && Label[n - 2] == '/' && (Label[n - 1] == '1' || Label[n - 1] == '2')) n -= 2;
    char *d = o.room(n);
    unsigned k = 0;
    for (; k < n; ++k) {
        char c = (char)Label[k];
        if (c == ' ' || c == '\t') break;
        d[k] = c;
    }
    o.n += k;
}

struct Mapped { int idx; uint32_t coord; };

static Mapped SetMappedPos(const Contigs &C, const urmb_result &r, unsigned QL) {  // state1.cpp:129-145
    Mapped m{-1, UINT32_MAX};
    if (!(r.flags & 2)) return m;
    uint32_t TL;
    int idx;
    uint32_t c = C.PosToCoordL(r.db_pos, idx, TL);
    if (c + QL > TL) return m;
    m.idx = idx;
    m.coord = c;
    return m;
}

static void SamUnmapped(OutBuf &o, uint32_t aFlags, const uint8_t *Label, unsigned LabelLen, const uint8_t *Seq,
                        const uint8_t *Qual, unsigned QL) {  // setsam.cpp:12-73
    uint32_t Flags = 0x04;
    if (aFlags & 0x01) Flags |= 0x01;
    if (aFlags & 0x40) Flags |= 0x40; else if (aFlags & 0x80) Flags |= 0x80;
    if (aFlags & 0x08) Flags |= 0x08; else if (aFlags & 0x20) Flags |= 0x20;
    AppendQName(o, Label, LabelLen);
    o.push_back('\t');
    put_u(o, Flags);
    o += "\t*\t0\t0\t*\t*\t0\t0\t";
    o.append((const char *)Seq, QL);
    o.push_back('\t');
    o.append((const char *)Qual, QL);
    o.push_back('\n');
}

static void SamRecord(const Contigs &C, OutBuf &o, uint32_t Flags, const Mapped &self, const urmb_result &r,
                      const uint16_t *runs, int MateIdx, uint32_t MatePos, int TLEN, const uint8_t *Label,
                      unsigned LabelLen, const uint8_t *Seq, const uint8_t *Qual, unsigned QL) {  // setsam.cpp:75-207
    if (self.idx < 0) { SamUnmapped(o, Flags, Label, LabelLen, Seq, Qual, QL); return; }
    const bool Plus = (r.flags & 1) != 0;
    AppendQName(o, Label, LabelLen);
    o.push_back('\t');
    put_u(o, Flags);
    o.push_back('\t');
    o += C.labels[self.idx];
    o.push_back('\t');
    put_u(o, self.coord + 1);
    o.push_back('\t');
    put_u(o, r.mapq);
    o.push_back('\t');
    RunsToCigar(runs + r.path_off, r.path_runs, QL, o);
    o.push_back('\t');
    if (MateIdx < 0 || C.labels[MateIdx].empty() || C.labels[MateIdx] == "*") o.push_back('*');
    else if (C.labels[MateIdx] == C.labels[self.idx]) o.push_back('=');
    else o += C.labels[MateIdx];
    o.push_back('\t');
    if (MatePos == 0 || MatePos == UINT32_MAX) o.push_back('0'); else put_u(o, MatePos + 1);
    o.push_back('\t');
    put_i(o, TLEN);
    o.push_back('\t');
    if (Plus) o.append((const char *)Seq, QL);
    else {
        char *d = o.room(QL);
        for (unsigned i = 0; i < QL; ++i) d[i] = (char)g_CompChar[Seq[QL - 1 - i]];
        o.n += QL;
    }
    o.push_back('\t');
    if (Plus) o.append((const char *)Qual, QL);
    else {
        char *d = o.room(QL);
        for (unsigned i = 0; i < QL; ++i) d[i] = (char)Qual[QL - 1 - i];
        o.n += QL;
    }
    o.push_back('\n');
}

static uint32_t GetPairedFlags(bool First, bool RevComp, bool MateRevComp, bool MateUnmapped) {  // output2.cpp:18-36
    uint32_t Flags = First ? 0x41 : 0x81;
    if (RevComp) Flags |= 0x10;
    if (MateUnmapped) Flags |= 0x08; else if (MateRevComp) Flags |= 0x20;
    return Flags;
}

struct alignas(128) HitCounters { uint64_t query = 0, accept = 0, reject = 0, nohit = 0; };

static inline void UpdateHitStats(HitCounters &hc, bool has_top, unsigned mapq, unsigned minq) {  // output1.cpp:20-30
    ++hc.query;
    if (!has_top) ++hc.nohit;
    else if (mapq >= minq) ++hc.accept;
    else ++hc.reject;
}

// upper estimate of the SAM text of reads [lo,hi): both copies of bases and qualities, the label, and the fixed columns
static size_t SamTextEstimate(const HostBatch &b, uint32_t lo, uint32_t hi) {
    if (hi <= lo) return 0;
    const size_t bases = b.offs[hi] - b.offs[lo];
    const size_t labels = (size_t)(b.lab[hi - 1] + b.lablen[hi - 1]) - b.lab[lo];   // spans the records' whole text: generous
    return 2 * bases + std::min(labels, (size_t)(hi - lo) * 256) + (size_t)(hi - lo) * 96;
}

// formats reads [lo,hi) of a finished batch
static void FormatSE(const Contigs &C, const HostBatch &b, const urmb_result *res, const uint16_t *runs, uint32_t lo,
                     uint32_t hi, unsigned minq, OutBuf &o, HitCounters &hc) {
    for (uint32_t i = lo; i < hi; ++i) {  // State1::Output1: SetSAM(0, "*", UINT32_MAX, 0)
        const unsigned QL = b.Len(i);
        Mapped m = SetMappedPos(C, res[i], QL);
        SamRecord(C, o, 0, m, res[i], runs, -1, UINT32_MAX, 0, b.Label(i), b.lablen[i], b.Seq(i), b.Qual(i), QL);
        UpdateHitStats(hc, m.idx >= 0, m.idx >= 0 ? res[i].mapq : 0, minq);
    }
}

// sam_active: -samout was given.  State2::Output2 (output2.cpp:10-16) runs OutputSAM2 -> OutputTab2 -> UpdateHitStats, and only
// OutputSAM2 (when a SAM file is open) calls SetMappedPos, which clears m_TopHit of a mate that overhangs its contig
// (SetSAM_Unmapped then zeroes m_Mapq): the tabbed line and the hit statistics see that cleared state.  Without -samout they
// see the raw search result.
static void FormatPE(const Contigs &C, const HostBatch &b1, const HostBatch &b2, const urmb_result *r1,
                     const urmb_result *r2, const uint16_t *runs, uint32_t lo, uint32_t hi, unsigned minq, OutBuf &o,
                     HitCounters &hc, bool sam_active) {
    if (!sam_active) {
        for (uint32_t i = lo; i < hi; ++i) {
            UpdateHitStats(hc, (r1[i].flags & 2) != 0, r1[i].mapq, minq);
            UpdateHitStats(hc, (r2[i].flags & 2) != 0, r2[i].mapq, minq);
        }
        return;
    }
    for (uint32_t i = lo; i < hi; ++i) {  // State2::SetSAM2, output2.cpp:71-132
        const unsigned L1 = b1.Len(i), L2 = b2.Len(i);
        Mapped m1 = SetMappedPos(C, r1[i], L1), m2 = SetMappedPos(C, r2[i], L2);
        const bool Mapped1 = m1.idx >= 0, Mapped2 = m2.idx >= 0;
        const bool Plus1 = Mapped1 && (r1[i].flags & 1), Plus2 = Mapped2 && (r2[i].flags & 1);
        const bool StrandsConsistent = Mapped1 && Mapped2 && (Plus1 != Plus2);
        int TLEN1 = 0, TLEN2 = 0;
        bool CorrectlyPaired = false;
        if (Mapped1 && Mapped2) {
            if (m1.coord <= m2.coord) {
                TLEN1 = int(m2.coord + L2) - int(m1.coord);
                if (TLEN1 > 0 && TLEN1 < 1000 && StrandsConsistent) CorrectlyPaired = true;
                if (TLEN1 > 1000) TLEN1 = 0;
                TLEN2 = -TLEN1;
            } else {
                TLEN2 = int(m1.coord + L1) - int(m2.coord);
                if (TLEN2 > 0 && TLEN2 < 1000 && StrandsConsistent) CorrectlyPaired = true;
                if (TLEN2 > 1000) TLEN2 = 0;
                TLEN1 = -TLEN2;
            }
        }
        const bool RevComp1 = Mapped1 && !(r1[i].flags & 1), RevComp2 = Mapped2 && !(r2[i].flags & 1);
        uint32_t Flags1 = GetPairedFlags(true, RevComp1, RevComp2, !Mapped2);
        uint32_t Flags2 = GetPairedFlags(false, RevComp2, RevComp1, !Mapped1);
        if (CorrectlyPaired) { Flags1 |= 0x02; Flags2 |= 0x02; }
        SamRecord(C, o, Flags1, m1, r1[i], runs, m2.idx, m2.coord, TLEN1, b1.Label(i), b1.lablen[i], b1.Seq(i),
                  b1.Qual(i), L1);
        SamRecord(C, o, Flags2, m2, r2[i], runs, m1.idx, m1.coord, TLEN2, b2.Label(i), b2.lablen[i], b2.Seq(i),
                  b2.Qual(i), L2);
        UpdateHitStats(hc, Mapped1, Mapped1 ? r1[i].mapq : 0, minq);
        UpdateHitStats(hc, Mapped2, Mapped2 ? r2[i].mapq : 0, minq);
    }
}

// State2::OutputTab2 (outputtab2.cpp:6-119): pair label, top pair, MAPQs, second pair, TL/score info.  A "hit" here is
// (has, DBStartPos, Plus, Score); positions go through UFIndex::PosToCoord (ufindex.cpp:701-727): a position in the
// padding between contigs leaves the label empty and prints coordinate 0 (UINT32_MAX + 1).
struct TabHit { bool has; uint32_t pos; bool plus; int score; };

static void TabChrPos(const Contigs &C, const TabHit &h, const char *&lab, size_t &lablen, uint32_t &coord) {
    int idx;
    uint32_t L;
    coord = C.PosToCoordL(h.pos, idx, L);
    if (idx >= 0) { lab = C.labels[idx].data(); lablen = C.labels[idx].size(); }
    else { lab = ""; lablen = 0; }
}

static void TabPairPos1(const Contigs &C, OutBuf &o, const TabHit &h, bool Fwd) {  // GetPairPosStr1
    const char *lab; size_t n; uint32_t coord;
    TabChrPos(C, h, lab, n, coord);
    o.append(lab, n);
    o.push_back(':');
    put_u(o, coord + 1);
    o.push_back('(');
    o.push_back(h.plus ? '+' : '-');
    o += ")/";
    o.push_back(Fwd ? '1' : '2');
}

static void TabPairPos(const Contigs &C, OutBuf &o, const TabHit &h1, const TabHit &h2) {  // GetPairPosStr
    if (!h1.has && !h2.has) { o.push_back('*'); return; }
    if (h1.has && !h2.has) { TabPairPos1(C, o, h1, true); return; }
    if (!h1.has && h2.has) { TabPairPos1(C, o, h2, false); return; }
    const char *l1, *l2; size_t n1, n2; uint32_t c1, c2;
    TabChrPos(C, h1, l1, n1, c1);
    TabChrPos(C, h2, l2, n2, c2);
    if (n1 == n2 && memcmp(l1, l2, n1) == 0 && h1.plus != h2.plus) {
        o.append(l1, n1);
        o.push_back(':');
        put_u(o, c1 + 1);
        o.push_back('-');
        put_u(o, c2 + 1);
        return;
    }
    TabPairPos1(C, o, h1, true);
    o.push_back(',');
    TabPairPos1(C, o, h2, false);
}

static unsigned TabTemplateLength(const TabHit &h1, const TabHit &h2, unsigned L1, unsigned L2) {  // output2.cpp:49-69
    int iTL = h1.pos <= h2.pos ? int(h2.pos + L2) - int(h1.pos) : int(h1.pos + L1) - int(h2.pos);
    if (iTL < 0 || iTL > 1000) iTL = 0;
    return (unsigned)iTL;
}

static void FormatTab2(const Contigs &C, const HostBatch &b1, const HostBatch &b2, const urmb_result *r1, const urmb_result *r2,
                       const urmb_second *s1, const urmb_second *s2, uint32_t lo, uint32_t hi, OutBuf &o, bool sam_active) {
    for (uint32_t i = lo; i < hi; ++i) {
        // after OutputSAM2 a mate whose top hit overhangs its contig has no top hit and MAPQ 0 (see FormatPE)
        const bool has1 = sam_active ? SetMappedPos(C, r1[i], b1.Len(i)).idx >= 0 : (r1[i].flags & 2) != 0;
        const bool has2 = sam_active ? SetMappedPos(C, r2[i], b2.Len(i)).idx >= 0 : (r2[i].flags & 2) != 0;
        const unsigned mq1 = (sam_active && !has1) ? 0u : r1[i].mapq, mq2 = (sam_active && !has2) ? 0u : r2[i].mapq;
        const TabHit t1{has1, r1[i].db_pos, (r1[i].flags & 1) != 0, r1[i].score};
        const TabHit t2{has2, r2[i].db_pos, (r2[i].flags & 1) != 0, r2[i].score};
        const TabHit u1{(s1[i].flags & 2) != 0, s1[i].db_pos, (s1[i].flags & 1) != 0, s1[i].score};
        const TabHit u2{(s2[i].flags & 2) != 0, s2[i].db_pos, (s2[i].flags & 1) != 0, s2[i].score};
        AppendQName(o, b1.Label(i), b1.lablen[i]);   // State1::GetPairLabel, state1.cpp:762-778
        o.push_back('\t');
        TabPairPos(C, o, t1, t2);
        o.push_back('\t');
        put_u(o, mq1);
        o.push_back(',');
        put_u(o, mq2);
        o.push_back('\t');
        if (u1.has) TabPairPos(C, o, u1, u2); else o.push_back('*');
        if (t1.has && t2.has && u1.has && u2.has) {   // State2::GetInfoStr
            o.push_back('\t');
            const unsigned L1 = b1.Len(i), L2 = b2.Len(i);
            const unsigned TopTL = TabTemplateLength(t1, t2, L1, L2), SecondTL = TabTemplateLength(u1, u2, L1, L2);
            if (TopTL == SecondTL) { o += "TL="; put_u(o, TopTL); }
            else { o += "TL/"; put_u(o, TopTL); o.push_back(','); put_u(o, SecondTL); }
            o.push_back(';');
            const int TopScore = t1.score + t2.score, SecondScore = u1.score + u2.score;
            if (TopScore == SecondScore) { o += "Score="; put_i(o, TopScore); }
            else { o += "Score/"; put_i(o, TopScore); o.push_back(','); put_i(o, SecondScore); }
            o.push_back(';');
        }
        o.push_back('\n');
    }
}

// ------------------------------------------------------------------------------------------------
// -map / -map2
// ------------------------------------------------------------------------------------------------
static std::string Commas(uint64_t v) {
    std::string s = std::to_string(v), o;
    for (size_t i = 0; i < s.size(); ++i) {
        o.push_back(s[i]);
        size_t rem = s.size() - 1 - i;
        if (rem && rem % 3 == 0) o.push_back(',');
    }
    return o;
}

struct InFlight {
    std::unique_ptr<HostBatch> b1, b2;
    int gpu = 0, slot = 0;
};

static void WriteAll(int fd, const char *p, size_t n, const std::string &path) {
    while (n) {
        ssize_t w = write(fd, p, n);
        if (w < 0) { if (errno == EINTR) continue; Die("Write error on %s: %s", path.c_str(), strerror(errno)); }
        p += w;
        n -= (size_t)w;
    }
}

// Bounded hand-over between two pipeline stages; Close() ends the consumer's loop once the queue has drained.
template <class T>
class Channel {
   public:
    explicit Channel(size_t cap) : cap_(cap) {}
    void Push(T v) {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [&]() { return q_.size() < cap_; });
        q_.push_back(std::move(v));
        cv_.notify_all();
    }
    bool Pop(T &v) {
        std::unique_lock<std::mutex> lk(mu_);
        cv_.wait(lk, [&]() { return !q_.empty() || closed_; });
        if (q_.empty()) return false;
        v = std::move(q_.front());
        q_.pop_front();
        cv_.notify_all();
        return true;
    }
    void Close() {
        std::lock_guard<std::mutex> lk(mu_);
        closed_ = true;
        cv_.notify_all();
    }

   private:
    size_t cap_;
    std::mutex mu_;
    std::condition_variable cv_;
    std::deque<T> q_;
    bool closed_ = false;
};

// Results of one finished batch, copied out of the slot's pinned buffers so that the slot can take the next batch
// while this one is being formatted.
struct FormatJob {
    std::unique_ptr<HostBatch> b1, b2;
    std::vector<urmb_result> res;   // mate 1 results, then mate 2
    std::vector<uint16_t> runs;
    std::vector<urmb_second> second;   // -tabbedout: second pair of mate 1, then mate 2
};
struct TextSet {   // SAM text of one batch, one piece per formatter thread, in record order (+ the -tabbedout text)
    std::vector<OutBuf> parts, tab;
};

// SAM output.  A regular file is extended and filled through a shared mapping by several threads (write(2) serialises
// on the inode and was the slowest stage of the pipeline); anything else (pipe, device) gets plain sequential writes.
class SamSink {
   public:
    SamSink(const std::string &path, int nthreads)
        : path_(path), pool_(getenv("URMB_WRITE_THREADS") ? std::max(1, atoi(getenv("URMB_WRITE_THREADS"))) : std::max(1, std::min(nthreads, 8))) {
        if (path.empty()) return;
        fd_ = open(path.c_str(), O_WRONLY | O_CREAT | O_TRUNC, 0666);
        if (fd_ < 0) Die("Cannot create %s", path.c_str());
        struct stat sb;
        map_ = fstat(fd_, &sb) == 0 && S_ISREG(sb.st_mode) && !getenv("URMB_NO_MMAP_OUT");
        page_ = (size_t)sysconf(_SC_PAGESIZE);
    }
    ~SamSink() { Close(); }
    bool active() const { return fd_ >= 0; }
    void Header(const std::string &h) {
        if (fd_ < 0) return;
        WriteAll(fd_, h.data(), h.size(), path_);
        off_ += (off_t)h.size();
    }
    void Append(const std::vector<OutBuf> &parts) {   // the parts in order
        if (fd_ < 0) return;
        const size_t np = parts.size();
        woff_.assign(np + 1, 0);
        for (size_t i = 0; i < np; ++i) woff_[i + 1] = woff_[i] + parts[i].size();
        const size_t len = woff_[np], lead = (size_t)off_ % page_;
        char *m = nullptr;
        if (map_ && len) {
            if (ftruncate(fd_, off_ + (off_t)len) == 0) {
                void *q = mmap(nullptr, len + lead, PROT_READ | PROT_WRITE, MAP_SHARED, fd_, off_ - (off_t)lead);
                if (q != MAP_FAILED) m = (char *)q;
            }
            if (!m) {   // not mappable after all: position the descriptor and stay with write(2)
                map_ = false;
                if (ftruncate(fd_, off_) != 0 || lseek(fd_, off_, SEEK_SET) < 0) Die("Write error on %s: %s", path_.c_str(), strerror(errno));
            }
        }
        if (m) {
            pool_.Run([&](int t, int nt) {
                for (size_t i = (size_t)t; i < np; i += (size_t)nt) memcpy(m + lead + woff_[i], parts[i].data(), parts[i].size());
            });
            munmap(m, len + lead);
        } else {
            for (auto &part : parts) WriteAll(fd_, part.data(), part.size(), path_);
        }
        off_ += (off_t)len;
    }
    void Close() {
        if (fd_ >= 0 && close(fd_) != 0) Die("Write error on %s: %s", path_.c_str(), strerror(errno));
        fd_ = -1;
    }

   private:
    std::string path_;
    Pool pool_;
    int fd_ = -1;
    off_t off_ = 0;
    bool map_ = false;
    size_t page_ = 4096;
    std::vector<size_t> woff_;
};

// The host pipeline (SURVEY.md §8f rank 1), one thread per stage, every stage internally parallel or cheap:
//   reader (block FASTQ parse, rpool) -> main (urmb_submit / urmb_wait: the only thread that talks to the C ABI)
//   -> formatter (SAM text, fpool) -> writer (write(2) in record order)
static std::string MemBytesToStr(double Bytes);
// CheckUsedOpts (cmdline.cpp:13-26, urmap_main.cpp:37): after a command that ends normally every option that was given but
// never looked at gets "WARNING: Option -x not used", in the order of myopts.h.  Which options a command looks at was taken
// from the reference binary itself, one extra option at a time; the output files, -log and -quiet count as used everywhere
// (main opens them), and so do this program's own options (-gpus, -batch, -gpu_build, -ref; -threads with -ufi_validate).
// With -ref the index options (-slots, -wordlength, -maxix, -load_factor) are used as -make_ufi uses them.
static void WarnUnusedOpts(const Opts &o, const char *cmd) {
    static const char *order[] = {"slots", "ufi", "reverse", "threads", "wordlength", "minq", "maxix", "load_factor", "validate", "veryfast"};
    const std::string c = cmd;
    auto used = [&](const std::string &n) {
        if ((c == "map" || c == "map2") && !o.ref.empty() && (n == "slots" || n == "wordlength" || n == "maxix" || n == "load_factor"))
            return true;
        if (c == "make_ufi") return n == "slots" || n == "wordlength" || n == "maxix" || n == "load_factor" || n == "validate" || n == "veryfast";
        if (c == "map") return n == "ufi" || n == "threads" || n == "veryfast";
        if (c == "map2") return n == "ufi" || n == "reverse" || n == "threads" || n == "minq" || n == "veryfast";
        if (c == "ufi_validate") return n == "threads";
        return false;   // ufi_info
    };
    for (const char *n : order)
        if (std::find(o.given.begin(), o.given.end(), n) != o.given.end() && !used(n)) {
            fprintf(stderr, "\nWARNING: Option -%s not used\n\n", n);   // Warning_, myutils.cpp:965-982
            if (g_log) fprintf(g_log, "\nWARNING: Option -%s not used\n", n);
        }
}

static time_t g_started = 0;
// What urmap_main.cpp:36-39 does after a command that ended normally: unused-option warnings, then elapsed time and memory
// into the log file.
static void FinishRun(const Opts &o, const char *cmd) {
    WarnUnusedOpts(o, cmd);
    if (g_log) {   // LogElapsedTimeAndRAM, myutils.cpp
        const time_t t_done = time(nullptr);
        const long secs = (long)(t_done - g_started);
        struct rusage ru;
        getrusage(RUSAGE_SELF, &ru);
        fprintf(g_log, "\nFinished %sElapsed time %02ld:%02ld\nMax memory %s\n", ctime(&t_done), secs / 60, secs % 60,
                MemBytesToStr((double)ru.ru_maxrss * 1024.0).c_str());
        fflush(g_log);
    }
}

// The table the index options select for a FASTA file (cmd_make_ufi, ufindexio.cpp:117-179): -make_ufi and -ref both take it
// from here, so that `-ref g.fa <opts>` maps with the table of `-make_ufi g.fa <opts>`.
struct IndexShape {
    uint32_t W = 24, MaxIx = 32;
    uint64_t SlotCount = 0;
    int64_t GenomeSize = 0;   // bytes of the file on disk (compressed, for a .gz file)
};
static IndexShape IndexShapeFor(const Opts &o, const std::string &fasta);

// Whole FASTA file in memory for -ref: plain files are mapped, gzip files (magic 1f 8b, as gzopen tells them apart) are
// inflated on the host into one buffer.
struct RawFile {
    const uint8_t *p = nullptr;
    size_t n = 0;
    void *map = nullptr;
    std::vector<uint8_t> buf;
    explicit RawFile(const std::string &path) {
        const int fd = open(path.c_str(), O_RDONLY);
        if (fd < 0) Die("Cannot open %s", path.c_str());
        struct stat sb;
        if (fstat(fd, &sb) != 0) Die("Cannot stat %s", path.c_str());
        uint8_t magic[2] = {0, 0};
        const bool gz = pread(fd, magic, 2, 0) == 2 && magic[0] == 0x1f && magic[1] == 0x8b;
        if (!gz) {
            n = (size_t)sb.st_size;
            if (n) {
                map = mmap(nullptr, n, PROT_READ, MAP_PRIVATE | MAP_POPULATE, fd, 0);
                if (map == MAP_FAILED) Die("Cannot map %s", path.c_str());
                p = (const uint8_t *)map;
            }
            close(fd);
            return;
        }
        gzFile g = gzdopen(fd, "rb");
        if (!g) Die("Cannot open %s", path.c_str());
        gzbuffer(g, 1 << 20);
        size_t cap = std::max<size_t>((size_t)sb.st_size * 4, 1 << 20);
        for (;;) {
            buf.resize(cap);
            while (n < cap) {
                const unsigned want = (unsigned)std::min<size_t>(cap - n, 1u << 30);
                const int r = gzread(g, buf.data() + n, want);
                if (r < 0) Die("Read error in %s", path.c_str());
                if (r == 0) break;
                n += (size_t)r;
            }
            if (n < cap) break;
            cap *= 2;
        }
        gzclose(g);
        buf.resize(n);
        p = buf.data();
    }
    ~RawFile() { if (map) munmap(map, n); }
};

static int CmdMap(const Opts &o, bool paired) {
    if (o.ufi.empty() && o.ref.empty()) Die("-ufi required (or -ref)");
    if (!o.ufi.empty() && !o.ref.empty()) Die("-ufi and -ref are mutually exclusive");
    if (paired && o.reverse.empty()) Die("-reverse required");  // map2.cpp:42
    const double t_start = now_s();
    urmb_index_host *hix = nullptr;
    IndexShape X;
    if (!o.ref.empty()) X = IndexShapeFor(o, o.ref);
    else if (urmb_index_load_host(o.ufi.c_str(), &hix) != 0) Die("%s", urmb_last_error(nullptr));
    urmb_index_desc d;
    uint32_t ncontig = 0;
    Contigs C;
    auto read_contigs = [&]() {   // the contig table of a UFI file or of the index built from -ref
        urmb_index_info(hix, &d, &ncontig);
        for (uint32_t i = 0; i < ncontig; ++i) {
            urmb_contig c;
            urmb_index_contig(hix, i, &c);
            C.labels.push_back(c.label);
            C.lengths.push_back(c.length);
            C.offsets.push_back(c.offset);
        }
    };
    if (hix) read_contigs();
    const uint32_t word_length = hix ? d.word_length : X.W, max_ix = hix ? d.max_ix : X.MaxIx;
    if (o.veryfast && max_ix > 3) fprintf(stderr, "\nWARNING: index not optimal for -veryfast\n\n");  // map.cpp:49
    urmb_params p{};
    p.method = (!paired && o.veryfast) ? 7 : 6;       // map.cpp:34-37; map2 always uses method 6 (map2.cpp:15)
    p.pe_method = (paired && o.veryfast) ? 5 : 4;     // map2.cpp:46-48
    p.band_radius = -1;
    p.minq = (int)o.minq;
    const bool want_tab = paired && !o.tabbedout.empty();   // outputtab2.cpp: only State2 writes it
    p.want_second = want_tab ? 1 : 0;
    const int ngpu = (int)std::max(1u, o.gpus);
    std::vector<urmb_ctx *> ctxs(ngpu, nullptr);
    for (int g = 0; g < ngpu; ++g)
        if (urmb_ctx_create(g, &p, &ctxs[g]) != 0) Die("GPU %d: %s", g, urmb_last_error(nullptr));
    // page-locked batch buffers are slow to allocate (~0.4 s for the ones in circulation): get them while the index loads
    std::mutex mu;   // guards the spare lists
    std::vector<std::unique_ptr<HostBatch>> spare;
    std::thread prealloc([&]() {
        for (int g = 0; g < ngpu; ++g)   // slot buffers for reads of up to 160 bases; longer reads grow them later
            if (urmb_reserve(ctxs[g], o.batch, 160, paired ? 1 : 0, word_length) != 0) Die("GPU %d: %s", g, urmb_last_error(ctxs[g]));
        const int want = (paired ? 2 : 1) * (6 + ngpu * URMB_SLOTS);
        for (int i = 0; i < want; ++i) {
            std::unique_ptr<HostBatch> b(new HostBatch);
            b->seqs.need((size_t)o.batch * 152 + 64);
            std::lock_guard<std::mutex> lk(mu);
            spare.push_back(std::move(b));
        }
    });
    if (hix) {
        if (urmb_index_broadcast(ctxs.data(), ngpu, hix) != 0) Die("index upload: %s", urmb_last_error(ctxs[0]));
    } else {
        std::unique_ptr<RawFile> fa(new RawFile(o.ref));
        const double t_read = now_s();
        const int rc = urmb_index_from_fasta(ctxs.data(), ngpu, fa->p, fa->n, X.W, X.MaxIx, X.SlotCount, &hix);
        if (rc == URMB_E_IO) Die("Bad FASTA file %s, %s", o.ref.c_str(), urmb_last_error(ctxs[0]));
        if (rc == URMB_E_OVERFLOW || rc == URMB_E_UNSUPPORTED)
            Die("GPU index build of %s: %s; build the index with -make_ufi (it builds every table on the host) and map with -ufi",
                o.ref.c_str(), urmb_last_error(ctxs[0]));
        if (rc != 0) Die("index from %s: %s", o.ref.c_str(), urmb_last_error(ctxs[0]));
        fa.reset();
        const char *lab;
        for (uint32_t i = 0; urmb_index_dropped(hix, i, &lab) == 0; ++i)
            fprintf(stderr, "\nWARNING: Empty sequence in FASTA file %s, label >%s\n\n", o.ref.c_str(), lab);   // as -make_ufi
        double t[5];
        urmb_index_fasta_times(hix, t);
        read_contigs();
        Progress("Index of %s built on %d GPU(s): read %.1f s, upload %.1f s, parse %.2f s (kernels %.4f s), build %.2f s, "
                 "total %.1f s\n", o.ref.c_str(), ngpu, t_read - t_start, t[0], t[1], t[4], t[2], now_s() - t_start);
    }
    prealloc.join();
    const double t_loaded = now_s();
    if (o.ref.empty()) Progress("Index %s loaded into %d GPU(s) in %.1f s\n", o.ufi.c_str(), ngpu, t_loaded - t_start);

    int nthreads = o.set_threads ? (int)o.threads : std::min((int)std::thread::hardware_concurrency(), 32);
    if (nthreads < 1) nthreads = 1;
    SamSink tabsink(paired ? o.tabbedout : std::string(), nthreads);
    if (!paired && !o.tabbedout.empty()) { FILE *f = fopen(o.tabbedout.c_str(), "w"); if (f) fclose(f); }   // created, stays empty
    SamSink sink(o.samout, nthreads);
    if (sink.active()) {
        std::string h;
        for (uint32_t i = 0; i < ncontig; ++i) h += "@SQ\tSN:" + C.labels[i] + "\tLN:" + std::to_string(C.lengths[i]) + "\n";
        h += "@PG\tID:urmap\tPN:urmap\tVN:" URMB_VERSION "-b200\tCL:";  // state1.cpp:736-752
        for (auto &a : g_argv) h += a + " ";
        h += "\n";
        sink.Header(h);
    }
    Pool rpool(nthreads), fpool(nthreads);

    FastqReader rd1(paired ? o.map2 : o.map, rpool);
    std::unique_ptr<FastqReader> rd2;
    if (paired) rd2.reset(new FastqReader(o.reverse, rpool));

    typedef std::pair<std::unique_ptr<HostBatch>, std::unique_ptr<HostBatch>> Item;
    Channel<Item> parsed(3);
    Channel<std::unique_ptr<FormatJob>> to_format(2);
    Channel<std::unique_ptr<TextSet>> to_write(2);
    std::vector<std::unique_ptr<FormatJob>> spare_jobs;
    std::vector<std::unique_ptr<TextSet>> spare_text;
    double t_read = 0, t_qwait = 0, t_submit = 0, t_gpuwait = 0, t_copy = 0, t_format = 0, t_write = 0;
    auto fresh = [&]() {
        std::lock_guard<std::mutex> lk(mu);
        if (spare.empty()) return std::unique_ptr<HostBatch>(new HostBatch);
        std::unique_ptr<HostBatch> b = std::move(spare.back());
        spare.pop_back();
        return b;
    };
    std::thread reader([&]() {
        for (;;) {
            std::unique_ptr<HostBatch> a = fresh(), b;
            const double t0 = now_s();
            uint32_t n1 = rd1.Fill(*a, o.batch), n2 = 0;
            if (paired) {
                b = fresh();
                n2 = rd2->Fill(*b, o.batch);
                if (n1 != n2) Die("Premature end of file in FASTQ%c", n1 > n2 ? '2' : '1');  // map2.cpp:31
            }
            t_read += now_s() - t0;
            if (n1 == 0) { parsed.Close(); return; }
            parsed.Push(Item(std::move(a), std::move(b)));
        }
    });

    HitCounters total;
    std::thread formatter([&]() {
        std::vector<HitCounters> hcs(nthreads);
        std::unique_ptr<FormatJob> job;
        while (to_format.Pop(job)) {
            std::unique_ptr<TextSet> ts;
            {
                std::lock_guard<std::mutex> lk(mu);
                if (!spare_text.empty()) { ts = std::move(spare_text.back()); spare_text.pop_back(); }
            }
            if (!ts) { ts.reset(new TextSet); ts->parts.resize(nthreads); ts->tab.resize(want_tab ? nthreads : 0); }
            const double t0 = now_s();
            const uint32_t n = job->b1->n;
            const urmb_result *r1 = job->res.data(), *r2 = r1 + n;
            const uint16_t *runs = job->runs.data();
            fpool.Run([&](int t, int nt) {
                OutBuf &out = ts->parts[t];
                out.clear();
                hcs[t] = HitCounters();
                uint32_t lo = (uint32_t)((uint64_t)n * t / nt), hi = (uint32_t)((uint64_t)n * (t + 1) / nt);
                out.reserve(SamTextEstimate(*job->b1, lo, hi) + (paired ? SamTextEstimate(*job->b2, lo, hi) : 0));
                if (paired) FormatPE(C, *job->b1, *job->b2, r1, r2, runs, lo, hi, o.minq, out, hcs[t], sink.active());
                else FormatSE(C, *job->b1, r1, runs, lo, hi, o.minq, out, hcs[t]);
                if (want_tab) {
                    ts->tab[t].clear();
                    FormatTab2(C, *job->b1, *job->b2, r1, r2, job->second.data(), job->second.data() + n, lo, hi, ts->tab[t], sink.active());
                }
            });
            for (int t = 0; t < nthreads; ++t) {
                total.query += hcs[t].query; total.accept += hcs[t].accept; total.reject += hcs[t].reject; total.nohit += hcs[t].nohit;
            }
            t_format += now_s() - t0;
            {
                std::lock_guard<std::mutex> lk(mu);
                spare.push_back(std::move(job->b1));
                if (job->b2) spare.push_back(std::move(job->b2));
                spare_jobs.push_back(std::move(job));
            }
            to_write.Push(std::move(ts));
        }
        to_write.Close();
    });
    std::thread writer([&]() {
        std::unique_ptr<TextSet> ts;
        while (to_write.Pop(ts)) {
            const double t0 = now_s();
            sink.Append(ts->parts);
            if (want_tab) tabsink.Append(ts->tab);
            t_write += now_s() - t0;
            std::lock_guard<std::mutex> lk(mu);
            spare_text.push_back(std::move(ts));
        }
    });

    std::deque<InFlight> fly;
    auto retire = [&](InFlight &f) {
        const urmb_result *r1, *r2;
        const uint16_t *runs;
        uint32_t used;
        double t0 = now_s();
        if (urmb_wait(ctxs[f.gpu], f.slot, &r1, &r2, &runs, &used) != 0) Die("GPU %d: %s", f.gpu, urmb_last_error(ctxs[f.gpu]));
        double t1 = now_s();
        t_gpuwait += t1 - t0;
        std::unique_ptr<FormatJob> job;
        {
            std::lock_guard<std::mutex> lk(mu);
            if (!spare_jobs.empty()) { job = std::move(spare_jobs.back()); spare_jobs.pop_back(); }
        }
        if (!job) job.reset(new FormatJob);
        const uint32_t n = f.b1->n;
        job->res.resize((size_t)n * (paired ? 2 : 1));
        memcpy(job->res.data(), r1, (size_t)n * sizeof(urmb_result));
        if (paired) memcpy(job->res.data() + n, r2, (size_t)n * sizeof(urmb_result));
        job->runs.resize(used);
        if (used) memcpy(job->runs.data(), runs, (size_t)used * sizeof(uint16_t));
        if (want_tab) {
            const urmb_second *s1, *s2;
            if (urmb_second_hits(ctxs[f.gpu], f.slot, &s1, &s2) != 0) Die("GPU %d: %s", f.gpu, urmb_last_error(ctxs[f.gpu]));
            job->second.resize((size_t)n * 2);
            memcpy(job->second.data(), s1, (size_t)n * sizeof(urmb_second));
            memcpy(job->second.data() + n, s2, (size_t)n * sizeof(urmb_second));
        }
        job->b1 = std::move(f.b1);
        job->b2 = std::move(f.b2);
        t_copy += now_s() - t1;
        to_format.Push(std::move(job));
    };
    uint64_t k = 0;
    const size_t max_fly = (size_t)ngpu * URMB_SLOTS;
    for (;;) {
        Item item;
        const double tq = now_s();
        const bool more = parsed.Pop(item);
        t_qwait += now_s() - tq;
        if (!more) break;
        if (fly.size() == max_fly) { retire(fly.front()); fly.pop_front(); }
        InFlight f;
        f.gpu = (int)(k % ngpu);
        f.slot = (int)((k / ngpu) % URMB_SLOTS);
        f.b1 = std::move(item.first);
        f.b2 = std::move(item.second);
        urmb_batch u1{f.b1->n, (const uint8_t *)f.b1->seqs.p, f.b1->offs.data()}, u2{0, nullptr, nullptr};
        if (paired) u2 = urmb_batch{f.b2->n, (const uint8_t *)f.b2->seqs.p, f.b2->offs.data()};
        const double t0 = now_s();
        if (urmb_submit(ctxs[f.gpu], f.slot, &u1, paired ? &u2 : nullptr) != 0) Die("GPU %d: %s", f.gpu, urmb_last_error(ctxs[f.gpu]));
        t_submit += now_s() - t0;
        fly.push_back(std::move(f));
        ++k;
    }
    while (!fly.empty()) { retire(fly.front()); fly.pop_front(); }
    to_format.Close();
    reader.join();
    formatter.join();
    writer.join();
    sink.Close();
    tabsink.Close();
    const double t_end = now_s();
    const double secs = t_end - t_loaded;
    const bool profile = getenv("URMB_PROFILE") != nullptr;
    if (profile)
        fprintf(stderr, "[urmb host] %llu batches; load %.3fs; stage busy times: reader %.3fs, main (queue wait %.3fs, submit "
                "%.3fs, gpu wait %.3fs, result copy %.3fs), formatter %.3fs, writer %.3fs; mapper total %.3fs\n",
                (unsigned long long)k, t_loaded - t_start, t_read, t_qwait, t_submit, t_gpuwait, t_copy, t_format, t_write, secs);
    auto pct = [&](uint64_t x) { return total.query ? 100.0 * x / total.query : 0.0; };
    if (g_log) fprintf(g_log, "@rps=%.1f\n", secs > 0 ? total.query / secs : 0.0);   // state1.cpp:608
    Progress("\n%16.1f  Seconds to load index\n%16.1f  Seconds in mapper\n", t_loaded - t_start, secs);  // state1.cpp:593-632
    Progress("%16s  Reads (%llu)\n", Commas(total.query).c_str(), (unsigned long long)total.query);
    Progress("%16.0f  Reads/sec. (%d GPUs, %d host threads)\n", secs > 0 ? total.query / secs : 0.0, ngpu, nthreads);
    Progress("%16s  Mapped Q>=%u (%.1f%%)\n", Commas(total.accept).c_str(), o.minq, pct(total.accept));
    Progress("%16s  Mapped Q< %u (%.1f%%)\n", Commas(total.reject).c_str(), o.minq, pct(total.reject));
    Progress("%16s  Unmapped (%.1f%%)\n\n", Commas(total.nohit).c_str(), pct(total.nohit));
    uint64_t overflowed = 0;
    for (auto c : ctxs) {
        uint64_t t = 0;
        urmb_overflow_count(c, 0, nullptr, &t);
        overflowed += t;
    }
    uint64_t too_long = 0;
    for (auto c : ctxs) {
        uint64_t t = 0;
        urmb_unsupported_count(c, 0, nullptr, &t);
        too_long += t;
    }
    if (too_long)
        Progress("\nWARNING: %llu read(s) longer than %d bases (or mates of such reads) were not searched and are reported "
                 "unmapped\n\n", (unsigned long long)too_long, URMB_MAX_READ_LEN);
    if (overflowed)
        Progress("\nWARNING: %llu read(s) exceeded a per-read capacity of the GPU search (hit / HSP / path lists); their records "
                 "are reported but may differ from urmap's\n\n", (unsigned long long)overflowed);
    FinishRun(o, paired ? "map2" : "map");
    if (g_log) { fclose(g_log); g_log = nullptr; }
    fflush(nullptr);
    if (!getenv("URMB_TEARDOWN")) _exit(0);   // the output is complete: leave the 70 GB of mappings and device memory to the OS
    for (auto c : ctxs) urmb_ctx_destroy(c);
    urmb_index_free_host(hix);
    if (profile) fprintf(stderr, "[urmb host] teardown %.3fs\n", now_s() - t_end);
    return 0;
}

// ------------------------------------------------------------------------------------------------
// -make_ufi (CPU, byte-identical to the reference)
// ------------------------------------------------------------------------------------------------
static bool IsPrime64(uint64_t n) {
    if (n < 2) return false;
    if (n % 2 == 0) return n == 2;
    for (uint64_t dd = 3; dd * dd <= n; dd += 2) if (n % dd == 0) return false;
    return true;
}
static uint64_t GetPrime(uint64_t n) {  // prime.cpp:11; primes.h = first prime >= x, x = 100, x <- x*100/95
    uint64_t x = 100;
    for (int i = 0; i < 410; ++i) {
        uint64_t p = x;
        while (!IsPrime64(p)) ++p;
        if (p >= n) return p;
        x = x * 100 / 95;
    }
    Die("GetPrime(%.3g) overflow", (double)n);
}

static inline uint64_t murmur64(uint64_t h) {
    h ^= (h >> 33); h *= 0xff51afd7ed558ccdULL; h ^= (h >> 33); h *= 0xc4ceb9fe1a85ec53ULL; h ^= (h >> 33);
    return h;
}

struct UfiBuilder {
    static const uint8_t T_FREE = 0, T_END = 127, T_MY = 128, T_PLUS1 = 254, T_BOTH1 = 255, T_LONG_MINE = 253, T_LONG_OTHER = 125;
    uint32_t W = 24, MaxIx = 32;
    uint64_t SlotCount = 0, ShiftMask = 0;
    std::vector<uint8_t> Blob, Seq, CntP, CntM;
    std::vector<std::string> Labels;
    std::vector<uint32_t> Lengths, Offsets;
    uint32_t Truncated = 0;

    uint8_t Tally(uint64_t s) const { return Blob[5 * s]; }
    uint32_t Pos(uint64_t s) const { uint32_t v; memcpy(&v, &Blob[5 * s + 1], 4); return v; }
    void SetTally(uint64_t s, uint8_t t) { Blob[5 * s] = t; }
    void SetPos(uint64_t s, uint32_t p) { memcpy(&Blob[5 * s + 1], &p, 4); }
    void SetNext(uint64_t s, uint8_t nx) { SetTally(s, (uint8_t)((Tally(s) & T_MY) | nx)); }
    uint64_t Slot(uint64_t word) const { return murmur64(word & ShiftMask) % SlotCount; }

    void ReadFasta(const std::string &path) {  // fastaseqsource.cpp:26-112 (trunclabels on, gaps stripped) + ufindex.cpp:462-510
        LineReader lr(path);
        const char *p;
        size_t n;
        std::vector<std::vector<uint8_t>> seqs;
        std::vector<std::string> labs;
        bool have = false;
        while (lr.ReadLine(p, n)) {
            if (n > 0 && p[0] == '>') {
                std::string lab;
                for (size_t i = 1; i < n && !isspace((unsigned char)p[i]); ++i) lab.push_back(p[i]);
                labs.push_back(lab);
                seqs.emplace_back();
                have = true;
                continue;
            }
            if (!have) {
                if (n == 0) continue;
                Die("Bad FASTA file %s, expected '>' in line %u", path.c_str(), lr.line_nr());
            }
            auto &s = seqs.back();
            for (size_t i = 0; i < n; ++i) {
                unsigned char c = (unsigned char)p[i];
                if (isspace(c) || c == '-' || c == '.') continue;
                if (!isalpha(c)) continue;  // BadByte: counted and skipped
                s.push_back((uint8_t)toupper(c));
            }
        }
        uint64_t size = 0;
        std::vector<size_t> keep;
        for (size_t i = 0; i < seqs.size(); ++i)
            if (!seqs[i].empty()) keep.push_back(i);
            else fprintf(stderr, "\nWARNING: Empty sequence in FASTA file %s, label >%s\n\n", path.c_str(), labs[i].c_str());
        for (size_t k = 0; k < keep.size(); ++k) {
            size_t i = keep[k];
            Labels.push_back(labs[i]);
            Lengths.push_back((uint32_t)seqs[i].size());
            Offsets.push_back((uint32_t)size);
            size += seqs[i].size();
            if (k + 1 != keep.size()) size += 32;  // PADGAP
        }
        Seq.resize(size);
        uint64_t off = 0;
        for (size_t k = 0; k < keep.size(); ++k) {
            auto &s = seqs[keep[k]];
            memcpy(&Seq[off], s.data(), s.size());
            off += s.size();
            if (k + 1 != keep.size()) { memset(&Seq[off], '-', 32); off += 32; }
            std::vector<uint8_t>().swap(s);
        }
    }

    template <class F> void ForEachPlusWord(F f) const {  // rolling word of ufindex.cpp:105-146
        uint64_t Word = 0;
        uint32_t K = 0;
        for (uint64_t p = 0; p < Seq.size(); ++p) {
            uint8_t L = g_Letter[Seq[p]];
            if (L == 0xFF) { K = 0; Word = 0; continue; }
            if (K < W) ++K;
            Word = (Word << 2) | L;
            if (K == W) f(Slot(Word), (uint32_t)(p - (W - 1)));
        }
    }

    uint64_t FindEndOfList(uint64_t s) const {  // ufindex.cpp:945-985
        uint64_t s2 = s;
        for (;;) {
            uint8_t T = Tally(s2);
            uint32_t P = Pos(s2);
            if (T == T_PLUS1 || T == T_BOTH1 || T == T_END) return s2;
            if (T == T_LONG_MINE || T == T_LONG_OTHER) {
                uint64_t a = (s2 + (P & 0xffff)) % SlotCount;
                s2 = (a + (P >> 16)) % SlotCount;
            } else
                s2 = (s2 + (T & 127)) % SlotCount;
        }
    }
    unsigned FindFreeSlot(uint64_t s) const {  // ufindex.cpp:987-1000
        for (unsigned i = 1; i < 0xffff; ++i) {
            uint64_t s2 = (s + i) % SlotCount;
            uint8_t n = CntP[s2];
            if (n > 0 && n <= MaxIx) continue;
            if (Tally(s2) == T_FREE) return i;
        }
        return UINT32_MAX;
    }
    void TruncateSlot(uint64_t s) {  // ufindex.cpp:153-192
        ++Truncated;
        uint64_t s2 = s;
        for (;;) {
            uint8_t T = Tally(s2);
            uint32_t P = Pos(s2);
            SetTally(s2, T_FREE);
            SetPos(s2, UINT32_MAX);
            if (T == T_PLUS1 || T == T_BOTH1 || T == T_END) return;
            if (T == T_LONG_MINE || T == T_LONG_OTHER) {
                uint64_t a = (s2 + (P & 0xffff)) % SlotCount;
                s2 = (a + (P >> 16)) % SlotCount;
            } else
                s2 = (s2 + (T & 127)) % SlotCount;
        }
    }
    void UpdateSlot(uint64_t s, uint32_t pos) {  // ufindex.cpp:194-322
        uint8_t n = CntP[s], m = CntM[s];
        if (n > MaxIx || m > MaxIx) return;
        if (Tally(s) == T_FREE) {
            SetPos(s, pos);
            SetTally(s, (n == 1 && m == 0) ? T_BOTH1 : T_PLUS1);
            return;
        }
        uint64_t eol = FindEndOfList(s);
        unsigned step = FindFreeSlot(eol);
        if (step == UINT32_MAX) { TruncateSlot(s); return; }
        uint64_t fs = (eol + step) % SlotCount;
        if (step > 124) {
            unsigned step2 = FindFreeSlot(fs);
            if (step2 == UINT32_MAX) { TruncateSlot(s); return; }
            uint32_t eolpos = Pos(eol);
            uint64_t fs2 = (fs + step2) % SlotCount;
            SetNext(eol, eol == s ? (uint8_t)(T_LONG_MINE & 127) : T_LONG_OTHER);
            SetPos(eol, step | (step2 << 16));
            SetTally(fs, T_LONG_OTHER);
            SetPos(fs, eolpos);
            SetTally(fs2, T_END);
            SetPos(fs2, pos);
            return;
        }
        SetNext(eol, (uint8_t)step);
        SetTally(fs, T_END);
        SetPos(fs, pos);
    }

    void MakeIndex() {  // ufindex.cpp:83-151
        Blob.resize(5 * SlotCount);
        for (uint64_t s = 0; s < SlotCount; ++s) { SetTally(s, T_FREE); SetPos(s, UINT32_MAX); }
        CntP.assign(SlotCount, 0);
        CntM.assign(SlotCount, 0);
        ForEachPlusWord([&](uint64_t s, uint32_t) { if (CntP[s] < 255) ++CntP[s]; });
        {  // CountSlots_Minus, ufindex.cpp:373-408: walk backwards through the complement letters
            uint64_t Word = 0;
            uint32_t K = 0;
            for (uint64_t p = Seq.size(); p-- > 0;) {
                uint8_t L = g_CompLetter[Seq[p]];
                if (L == 0xFF) { K = 0; Word = 0; continue; }
                if (K < W) ++K;
                Word = (Word << 2) | L;
                if (K == W) { uint64_t s = Slot(Word); if (CntM[s] < 255) ++CntM[s]; }
            }
        }
        ForEachPlusWord([&](uint64_t s, uint32_t pos) { UpdateSlot(s, pos); });
    }

    void ToFile(const std::string &path) const {  // ufindexio.cpp:15-49
        FILE *f = fopen(path.c_str(), "wb");
        if (!f) Die("Cannot create %s", path.c_str());
        auto w32 = [&](uint32_t v) { fwrite(&v, 4, 1, f); };
        w32(0x55464931u); w32(W); w32(MaxIx); w32((uint32_t)Seq.size());
        fwrite(&SlotCount, 8, 1, f);
        w32((uint32_t)Labels.size());
        for (size_t i = 0; i < Labels.size(); ++i) {
            w32(Lengths[i]); w32(Offsets[i]); w32((uint32_t)Labels[i].size());
            fwrite(Labels[i].data(), 1, Labels[i].size(), f);
        }
        w32(0x55464932u);
        fwrite(Blob.data(), 1, Blob.size(), f);
        w32(0x55464933u);
        fwrite(Seq.data(), 1, Seq.size(), f);
        w32(0x55464935u);
        if (fclose(f) != 0) Die("Write error %s", path.c_str());
    }
};

static IndexShape IndexShapeFor(const Opts &o, const std::string &fasta) {
    IndexShape x;
    x.W = o.set_wordlength ? o.wordlength : 24;
    x.MaxIx = o.veryfast ? 3 : 32;
    if (o.set_maxix) x.MaxIx = o.maxix;
    FILE *f = fopen(fasta.c_str(), "rb");
    if (!f) Die("Cannot open %s", fasta.c_str());
    fseeko(f, 0, SEEK_END);
    x.GenomeSize = ftello(f);
    fclose(f);
    if (!o.slots.empty()) x.SlotCount = strtoull(o.slots.c_str(), nullptr, 10);
    else x.SlotCount = GetPrime((uint64_t)(int64_t)(x.GenomeSize / o.load_factor));
    if (x.GenomeSize > (int64_t)UINT32_MAX - 100000) Die("Genome too big (%lld)", (long long)x.GenomeSize);
    return x;
}

extern "C" int urmb_host_gpu_build(const uint8_t *seq, uint64_t n, uint64_t slots, uint32_t W, uint32_t maxix, uint8_t *blob);
static std::string ValidateTable(const uint8_t *Blob, const uint8_t *Seq, uint64_t SlotCount, uint32_t SeqDataSize, uint32_t W,
                                 uint32_t MaxIx, int nthreads);

static int CmdMakeUfi(const Opts &o) {  // cmd_make_ufi, ufindexio.cpp:117-179
    UfiBuilder B;
    const IndexShape X = IndexShapeFor(o, o.make_ufi);
    const int64_t GenomeSize = X.GenomeSize;
    B.W = X.W;
    B.MaxIx = X.MaxIx;
    B.SlotCount = X.SlotCount;
    B.ShiftMask = B.W >= 32 ? ~0ull : ((1ull << (2 * B.W)) - 1);
    Progress("\n  Genome size  %lld\n        Slots  %llu\n  Load factor  %.2f\n  Word length  %u\n   Max abund.  %u\n\n",
             (long long)GenomeSize, (unsigned long long)B.SlotCount, GenomeSize / (double)B.SlotCount, B.W, B.MaxIx);
    double t0 = now_s();
    B.ReadFasta(o.make_ufi);
    Progress("Read %zu sequences, %zu bases (%.1f s)\n", B.Labels.size(), B.Seq.size(), now_s() - t0);
    t0 = now_s();
    if (o.gpu_build) {
        B.Blob.resize(5 * B.SlotCount);
        const int rc = urmb_host_gpu_build(B.Seq.data(), B.Seq.size(), B.SlotCount, B.W, B.MaxIx, B.Blob.data());
        if (rc == URMB_E_OVERFLOW || rc == URMB_E_UNSUPPORTED) {   // a list would have to be truncated (TruncateSlot), -maxix above 254: exact on the host only
            Progress("GPU index build: %s; building on the host instead\n", urmb_build_last_error());
            std::vector<uint8_t>().swap(B.Blob);
            B.MakeIndex();
            Progress("Index built in %.1f s\n%u slots truncated\n", now_s() - t0, B.Truncated);
        } else if (rc != 0) {
            Die("GPU index build failed: %s", urmb_build_last_error());
        } else {
            Progress("Index built on the GPU (byte-identical to the sequential builder) in %.1f s\n", now_s() - t0);
        }
    } else {
        B.MakeIndex();
        Progress("Index built in %.1f s\n%u slots truncated\n", now_s() - t0, B.Truncated);
    }
    if (o.validate) {   // ufindexio.cpp:171-172
        Progress("Validate\n");
        const int nthreads = o.set_threads ? (int)std::max(1u, o.threads) : std::max(1, std::min((int)std::thread::hardware_concurrency(), 32));
        const std::string err = ValidateTable(B.Blob.data(), B.Seq.data(), B.SlotCount, (uint32_t)B.Seq.size(), B.W, B.MaxIx, nthreads);
        if (!err.empty()) Die("%s", err.c_str());
    }
    B.ToFile(o.output);
    return 0;
}

// UFIndex::Validate / ValidateSlot / GetRow_Validate (ufindex.cpp:611-658, 834-882): every position stored in the list of every
// owned slot must hash back to that slot.  The reference walks the table on one thread and dies at the first failure with
// "WordToSlot != Slot" (its asserts on the list structure die with their own text); here the slot range is split over the
// host threads and the failure at the lowest slot is reported -- the same one.  Returns "" when the table is consistent.
static std::string ValidateTable(const uint8_t *Blob, const uint8_t *Seq, uint64_t SlotCount, uint32_t SeqDataSize, uint32_t W,
                                 uint32_t MaxIx, int nthreads) {
    auto tally = [&](uint64_t s) { return Blob[5 * s]; };
    auto pos = [&](uint64_t s) { uint32_t v; memcpy(&v, Blob + 5 * s + 1, 4); return v; };
    uint64_t bad_slot = UINT64_MAX;
    std::string bad_msg;
    std::mutex mu;
    auto fail = [&](uint64_t s, const char *msg) {
        std::lock_guard<std::mutex> lk(mu);
        if (s < bad_slot) { bad_slot = s; bad_msg = msg; }
    };
    const uint64_t piece = (SlotCount + (uint64_t)nthreads * 64 - 1) / ((uint64_t)nthreads * 64);
#pragma omp parallel for num_threads(nthreads) schedule(dynamic, 1)
    for (int64_t chunk = 0; chunk < (int64_t)nthreads * 64; ++chunk) {
        std::vector<uint32_t> PosVec(MaxIx);
        const uint64_t lo = (uint64_t)chunk * piece, hi = std::min(SlotCount, lo + piece);
        for (uint64_t Slot = lo; Slot < hi; ++Slot) {
            if (Slot > bad_slot) break;   // a failure at a lower slot is already known
            uint8_t T = tally(Slot);
            if ((T & 128) == 0) continue;   // TallyOther: not the head of a list
            uint64_t Slot2 = Slot;
            uint32_t K = 0;
            const char *err = nullptr;
            for (;;) {   // GetRow_Validate
                T = tally(Slot2);
                const uint32_t P = pos(Slot2);
                PosVec[K++] = P;
                if (T == 254 || T == 255) break;        // PLUS1 / BOTH1: a single entry
                if (K == MaxIx) break;
                if ((Slot2 == Slot) != ((T & 128) != 0)) { err = "list element with the wrong owner bit"; break; }   // asserta(TallyMine / TallyOther)
                if (T == 127) break;                    // END
                if (T == 253 || T == 125) {             // long link: the position is parked in slot + StepA
                    const uint64_t SlotA = (Slot2 + (P & 0xffffu)) % SlotCount;
                    Slot2 = (SlotA + (P >> 16)) % SlotCount;
                    PosVec[K - 1] = pos(SlotA);
                    if (tally(SlotA) != 125) { err = "long link without its parking slot"; break; }   // asserta(TA == TALLY_NEXT_LONG_OTHER)
                } else {
                    const uint32_t Next = T & 127u;
                    if (Next == 0 || Next > 124) { err = "bad link step"; break; }
                    Slot2 = (Slot2 + Next) % SlotCount;
                }
            }
            if (err) { fail(Slot, err); break; }
            for (uint32_t k = 0; k < K && !err; ++k) {   // ValidateSlot
                const uint32_t P = PosVec[k];
                if (P >= SeqDataSize || (uint64_t)P + W > SeqDataSize) { err = "position beyond the sequence data"; break; }
                uint64_t Word = 0;
                bool valid = true;
                for (uint32_t i = 0; i < W; ++i) {   // GetWord, ufindex.cpp:68-81
                    const uint8_t c = Seq[P + i] & 0xDF;
                    const uint32_t l = c == 'A' ? 0 : c == 'C' ? 1 : c == 'G' ? 2 : (c == 'T' || c == 'U') ? 3 : 4;
                    if (l > 3) { valid = false; break; }
                    Word = (Word << 2) | l;
                }
                if (!valid) Word = UINT64_MAX;
                uint64_t h = Word;   // WordToSlot, ufindex.h:50-65
                h ^= h >> 33; h *= 0xff51afd7ed558ccdULL; h ^= h >> 33; h *= 0xc4ceb9fe1a85ec53ULL; h ^= h >> 33;
                if (h % SlotCount != Slot) err = "WordToSlot != Slot";
            }
            if (err) { fail(Slot, err); break; }
        }
    }
    if (bad_slot == UINT64_MAX) return std::string();
    char t[160];
    snprintf(t, sizeof t, "%s (slot 0x%llx)", bad_msg.c_str(), (unsigned long long)bad_slot);
    return bad_msg == "WordToSlot != Slot" ? bad_msg : std::string(t);
}

// cmd_ufi_validate, ufistats.cpp:141-146
static int CmdUfiValidate(const Opts &o) {
    urmb_index_host *h = nullptr;
    Progress("Reading index %s\n", o.ufi_validate.c_str());
    if (urmb_index_load_host(o.ufi_validate.c_str(), &h) != 0) Die("%s", urmb_last_error(nullptr));
    urmb_index_desc d;
    uint32_t nc = 0;
    if (urmb_index_info(h, &d, &nc) != 0) Die("%s", urmb_last_error(nullptr));
    const int nthreads = o.set_threads ? (int)std::max(1u, o.threads) : std::max(1, std::min((int)std::thread::hardware_concurrency(), 32));
    Progress("Validate\n");
    const std::string err = ValidateTable((const uint8_t *)d.d_blob, (const uint8_t *)d.d_seq, d.slot_count, d.seq_data_size,
                                          d.word_length, d.max_ix, nthreads);
    urmb_index_free_host(h);
    if (!err.empty()) Die("%s", err.c_str());
    return 0;
}

// cmd_ufi_info, ufistats.cpp:148-172: the four header fields, same text
static std::string MemBytesToStr(double Bytes) {  // myutils.cpp:1220-1235
    char t[64];
    if (Bytes < 1e4) snprintf(t, sizeof t, "%.1fb", Bytes);
    else if (Bytes < 1e6) snprintf(t, sizeof t, "%.1fkb", Bytes / 1e3);
    else if (Bytes < 10e6) snprintf(t, sizeof t, "%.1fMb", Bytes / 1e6);
    else if (Bytes < 1e9) snprintf(t, sizeof t, "%.0fMb", Bytes / 1e6);
    else if (Bytes < 100e9) snprintf(t, sizeof t, "%.1fGb", Bytes / 1e9);
    else snprintf(t, sizeof t, "%.0fGb", Bytes / 1e9);
    return t;
}

static int CmdUfiInfo(const Opts &o) {
    FILE *f = fopen(o.ufi_info.c_str(), "rb");
    if (!f) Die("Cannot open %s", o.ufi_info.c_str());
    uint32_t h[4];
    uint64_t SlotCount;
    if (fread(h, 4, 4, f) != 4 || fread(&SlotCount, 8, 1, f) != 1) Die("Error reading %s", o.ufi_info.c_str());
    fclose(f);
    if (h[0] != ((uint32_t)'U' << 24 | (uint32_t)'F' << 16 | (uint32_t)'I' << 8 | (uint32_t)'1')) Die("%s is not a UFI file (bad magic)", o.ufi_info.c_str());  // UFI_MAGIC1, ufindex.h
    Progress(" Word length  %u\n", h[1]);
    Progress("       MaxIx  %u\n", h[2]);
    Progress("     SeqData  %u (%s)\n", h[3], MemBytesToStr((double)h[3]).c_str());
    Progress("       Slots  %llu (%s)\n", (unsigned long long)SlotCount, MemBytesToStr((double)SlotCount).c_str());
    return 0;
}

// Diagnostic (no reference counterpart): the records the block FASTQ reader hands to the mapper, one per line as
// label <TAB> bases <TAB> qualities; with -reverse the mates alternate.  Lets the CPU tests pin the reader.
static int CmdFastqDump(const Opts &o) {
    if (o.output.empty()) Die("-output required");
    int nthreads = o.set_threads ? (int)std::max(1u, o.threads) : 4;
    Pool pool(nthreads);
    FastqReader rd1(o.fastq_dump, pool);
    std::unique_ptr<FastqReader> rd2;
    if (!o.reverse.empty()) rd2.reset(new FastqReader(o.reverse, pool));
    FILE *f = fopen(o.output.c_str(), "wb");
    if (!f) Die("Cannot create %s", o.output.c_str());
    HostBatch a, b;
    double t_fill = 0;
    uint64_t nrec = 0;
    const bool discard = o.output == "/dev/null";
    for (;;) {
        const double t0 = now_s();
        uint32_t n1 = rd1.Fill(a, o.batch), n2 = rd2 ? rd2->Fill(b, o.batch) : 0;
        t_fill += now_s() - t0;
        nrec += n1 + n2;
        if (discard && n1) continue;
        if (rd2 && n1 != n2) Die("Premature end of file in FASTQ%c", n1 > n2 ? '2' : '1');
        if (n1 == 0) break;
        for (uint32_t i = 0; i < n1; ++i)
            for (const HostBatch *h : {(const HostBatch *)&a, rd2 ? (const HostBatch *)&b : (const HostBatch *)nullptr}) {
                if (!h) continue;
                fwrite(h->Label(i), 1, h->lablen[i], f);
                fputc('\t', f);
                fwrite(h->Seq(i), 1, h->Len(i), f);
                fputc('\t', f);
                fwrite(h->Qual(i), 1, h->Len(i), f);
                fputc('\n', f);
            }
    }
    fclose(f);
    if (getenv("URMB_PROFILE")) fprintf(stderr, "[urmb host] %llu records parsed in %.3f s (%d threads)\n", (unsigned long long)nrec, t_fill, nthreads);
    return 0;
}

// Diagnostic (no reference counterpart): host-only timing of the FASTQ reader and the SAM formatter over made-up
// results (every read mapped gapless, alternating strands), to size the host stages without a GPU.
static int CmdSamBench(const Opts &o) {
    int nthreads = o.set_threads ? (int)std::max(1u, o.threads) : (int)std::thread::hardware_concurrency();
    Pool pool(nthreads);
    FastqReader rd1(o.sam_bench, pool);
    std::unique_ptr<FastqReader> rd2;
    if (!o.reverse.empty()) rd2.reset(new FastqReader(o.reverse, pool));
    Contigs C;
    C.labels = {"chr1", "chr2"};
    C.lengths = {2000000000u, 1000000000u};
    C.offsets = {0u, 2000000032u};
    std::vector<OutBuf> outs(nthreads);
    std::vector<HitCounters> hcs(nthreads);
    std::vector<urmb_result> res;
    HostBatch a, b;
    double t_fill = 0, t_fmt = 0, t_wr = 0;
    uint64_t nrec = 0, bytes = 0;
    const int reps = getenv("URMB_BENCH_REPS") ? atoi(getenv("URMB_BENCH_REPS")) : 1;
    SamSink sink(o.output, nthreads);
    for (;;) {
        double t0 = now_s();
        uint32_t n1 = rd1.Fill(a, o.batch), n2 = rd2 ? rd2->Fill(b, o.batch) : 0;
        double t1 = now_s();
        t_fill += t1 - t0;
        if (n1 == 0) break;
        res.resize((size_t)n1 * 2);
        for (uint32_t i = 0; i < 2 * n1; ++i) {
            urmb_result r;
            memset(&r, 0, sizeof r);
            r.db_pos = (uint32_t)((nrec + i) * 977 % 1900000000u) + (i >= n1 ? 300 : 0);
            r.flags = (uint8_t)(2 | ((i ^ (i >= n1)) & 1));
            r.mapq = 40;
            res[i] = r;
        }
        t1 = now_s();
        for (int rep = 1; rep < reps; ++rep) {
            const double r0 = now_s();
            pool.Run([&](int t, int nt) {
                outs[t].clear();
                uint32_t lo = (uint32_t)((uint64_t)n1 * t / nt), hi = (uint32_t)((uint64_t)n1 * (t + 1) / nt);
                outs[t].reserve(SamTextEstimate(a, lo, hi) + (rd2 ? SamTextEstimate(b, lo, hi) : 0));
                if (rd2) FormatPE(C, a, b, res.data(), res.data() + n1, nullptr, lo, hi, 10, outs[t], hcs[t], true);
                else FormatSE(C, a, res.data(), nullptr, lo, hi, 10, outs[t], hcs[t]);
            });
            fprintf(stderr, "  rep %d: %.3fs\n", rep, now_s() - r0);
        }
        t1 = now_s();
        pool.Run([&](int t, int nt) {
            outs[t].clear();
            uint32_t lo = (uint32_t)((uint64_t)n1 * t / nt), hi = (uint32_t)((uint64_t)n1 * (t + 1) / nt);
            outs[t].reserve(SamTextEstimate(a, lo, hi) + (rd2 ? SamTextEstimate(b, lo, hi) : 0));
            if (rd2) FormatPE(C, a, b, res.data(), res.data() + n1, nullptr, lo, hi, 10, outs[t], hcs[t], true);
            else FormatSE(C, a, res.data(), nullptr, lo, hi, 10, outs[t], hcs[t]);
        });
        double t2 = now_s();
        t_fmt += t2 - t1;
        for (auto &x : outs) bytes += x.size();
        sink.Append(outs);
        t_wr += now_s() - t2;
        nrec += n1 + n2;
        (void)n2;
    }
    sink.Close();
    fprintf(stderr, "[urmb host] %llu records, %d threads: read %.3fs, format %.3fs (%.1f MB of SAM), write %.3fs\n",
            (unsigned long long)nrec, nthreads, t_fill, t_fmt, bytes / 1e6, t_wr);
    return 0;
}

int main(int argc, char **argv) {
    InitAlpha();
    Opts o = ParseCmdLine(argc, argv);
    g_quiet = o.quiet;
    if (!o.log.empty()) g_log = fopen(o.log.c_str(), "w");
    g_started = time(nullptr);
    const time_t t_started = g_started;
    if (g_log) {   // LogProgramInfoAndCmdLine, myutils.cpp: program, command line, start time
        fprintf(g_log, "\nurmap_b200 v%s\n", URMB_VERSION);
        for (auto &a : g_argv) fprintf(g_log, "%s ", a.c_str());
        fprintf(g_log, "\nStarted %s", ctime(&t_started));
        fflush(g_log);
    }
    if (o.version) { printf("urmap_b200 v%s (B200-native drop-in for urmap -map/-map2)\n", URMB_VERSION); return 0; }
    int rc;
    const char *cmd = nullptr;
    if (!o.make_ufi.empty()) { rc = CmdMakeUfi(o); cmd = "make_ufi"; }
    else if (!o.ufi_info.empty()) { rc = CmdUfiInfo(o); cmd = "ufi_info"; }
    else if (!o.ufi_validate.empty()) { rc = CmdUfiValidate(o); cmd = "ufi_validate"; }
    else if (!o.fastq_dump.empty()) rc = CmdFastqDump(o);
    else if (!o.sam_bench.empty()) rc = CmdSamBench(o);
    else if (!o.map.empty()) { rc = CmdMap(o, false); cmd = "map"; }
    else { rc = CmdMap(o, true); cmd = "map2"; }
    if (rc == 0 && cmd && std::string(cmd) != "map" && std::string(cmd) != "map2") FinishRun(o, cmd);   // CmdMap finishes its own run
    return rc;
}
