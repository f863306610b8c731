// vcfx_host.cpp — streaming chunk reader + output writer over the libvcfx_cuda C ABI.
#include "vcfx_host.h"

#include <algorithm>
#include <cctype>
#include <cerrno>
#include <cstdlib>
#include <cstring>
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>
#include <zlib.h>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <mutex>
#include <thread>

namespace vcfxh {

// ---------------------------------------------------------------------------------- Source
Source::~Source() {
    if (zs_) { inflateEnd(static_cast<z_stream *>(zs_)); delete static_cast<z_stream *>(zs_); }
}

long Source::raw_read(char *dst, size_t cap) {
    if (peek_pos_ < peek_.size()) {
        size_t k = std::min(cap, peek_.size() - peek_pos_);
        memcpy(dst, peek_.data() + peek_pos_, k);
        peek_pos_ += k;
        return (long)k;
    }
    for (;;) {
        ssize_t r = ::read(fd_, dst, cap);
        if (r < 0 && errno == EINTR) continue;
        if (r < 0) failed_ = true;
        return (long)r;
    }
}

bool Source::at_eof_initially() {
    if (!peek_.empty()) return false;
    char c;
    long r = raw_read(&c, 1);
    if (r <= 0) return true;
    peek_.assign(1, c); peek_pos_ = 0;
    return false;
}

bool Source::sniff_gzip() {
    while (peek_.size() < 2) {
        char c;
        ssize_t r = ::read(fd_, &c, 1);
        if (r < 0 && errno == EINTR) continue;
        if (r <= 0) break;
        peek_.push_back(c);
    }
    peek_pos_ = 0;
    return peek_.size() >= 2 && (unsigned char)peek_[0] == 0x1f && (unsigned char)peek_[1] == 0x8b;
}

void Source::enable_gzip() {
    z_stream *z = new z_stream();
    memset(z, 0, sizeof *z);
    if (inflateInit2(z, 15 + 32) != Z_OK) { delete z; failed_ = true; return; }
    zs_ = z; gz_ = true; zin_.resize(1 << 16);
}

// A regular file is read with several threads, each pread()ing its own slice of the destination
// (the pinned input slot): one thread copies out of the page cache at 6-7 GB/s, which is far
// below what the PCIe link takes (SURVEY §8f rank 1).  Pipes, gzip streams and small reads keep
// the single read(2).
long Source::parallel_read(char *dst, size_t cap) {
    if (!io_init_) {
        io_init_ = true;
        struct stat st;
        file_size_ = -1;                                    // "not a regular file"
        if (fstat(fd_, &st) == 0 && S_ISREG(st.st_mode) && lseek(fd_, 0, SEEK_CUR) >= 0) file_size_ = st.st_size;
        const char *e = getenv("VCFX_IO_THREADS");
        unsigned hw = std::thread::hardware_concurrency();
        io_threads_ = e ? std::max(1, atoi(e)) : (int)std::min(8u, std::max(1u, hw));
    }
    if (file_size_ < 0 || io_threads_ <= 1) return -2;
    // the descriptor's own offset is the one source of truth: small reads in between go through read(2) and move it
    const off_t cur = lseek(fd_, 0, SEEK_CUR);
    if (cur < 0) return -2;
    file_off_ = cur;
    const long long left = file_size_ - file_off_;
    if (left <= 0) return 0;
    const size_t n = (size_t)std::min<long long>((long long)cap, left);
    const size_t min_slice = (size_t)4 << 20;
    if (n < 2 * min_slice) return -2;
    const int parts = (int)std::min<size_t>((size_t)io_threads_, n / min_slice);
    const size_t slice = (((n + parts - 1) / parts) + 4095) & ~(size_t)4095;   // parts * slice >= n
    std::vector<size_t> got(parts, 0);
    std::vector<std::thread> th;
    auto work = [&](int i) {
        const size_t b = std::min(n, (size_t)i * slice), e2 = std::min(n, b + slice);
        size_t done = b;
        while (done < e2) {
            ssize_t r = ::pread(fd_, dst + done, e2 - done, (off_t)(file_off_ + (long long)done));
            if (r < 0 && errno == EINTR) continue;
            if (r <= 0) break;                              // error or the file shrank
            done += (size_t)r;
        }
        got[i] = done - b;
    };
    for (int i = 1; i < parts; ++i) th.emplace_back(work, i);
    work(0);
    for (auto &t : th) t.join();
    size_t total = 0;                                       // the contiguous prefix that was read
    for (int i = 0; i < parts; ++i) {
        const size_t b = std::min(n, (size_t)i * slice), e2 = std::min(n, b + slice);
        total += got[i];
        if (got[i] < e2 - b) break;
    }
    file_off_ += (long long)total;
    lseek(fd_, (off_t)file_off_, SEEK_SET);
    return (long)total;
}

long Source::read(char *dst, size_t cap) {
    if (!gz_) {
        if (peek_pos_ >= peek_.size() && cap >= ((size_t)8 << 20)) {
            const long r = parallel_read(dst, cap);
            if (r != -2) return r;
        }
        return raw_read(dst, cap);
    }
    if (gz_done_ || cap == 0) return 0;
    z_stream *z = static_cast<z_stream *>(zs_);
    z->next_out = reinterpret_cast<Bytef *>(dst);
    z->avail_out = (uInt)std::min<size_t>(cap, 1u << 30);
    while (z->avail_out == (uInt)std::min<size_t>(cap, 1u << 30)) {
        if (zin_pos_ == zin_len_) {
            long r = raw_read(zin_.data(), zin_.size());
            if (r < 0) return -1;
            if (r == 0) { gz_done_ = true; break; }
            zin_len_ = (size_t)r; zin_pos_ = 0;
        }
        z->next_in = reinterpret_cast<Bytef *>(zin_.data() + zin_pos_);
        z->avail_in = (uInt)(zin_len_ - zin_pos_);
        int ret = inflate(z, Z_NO_FLUSH);
        zin_pos_ = zin_len_ - z->avail_in;
        if (ret == Z_STREAM_END) {
            // like the reference loop (variant_counter.cpp:239-275) the first member ends the stream
            gz_done_ = true; break;
        }
        if (ret != Z_OK && ret != Z_BUF_ERROR) { failed_ = true; return -1; }
    }
    return (long)(std::min<size_t>(cap, 1u << 30) - z->avail_out);
}

// ---------------------------------------------------------------------------------- helpers
// Large outputs (missing_detector ~ input size, allele_counter ~ 9x) to a regular file that is not
// in append mode are written by several threads with pwrite() at their final offsets.
static bool write_parallel(int fd, const char *p, size_t n) {
    static int threads = -1;
    if (threads < 0) {
        const char *e = getenv("VCFX_IO_THREADS");
        unsigned hw = std::thread::hardware_concurrency();
        threads = e ? std::max(1, atoi(e)) : (int)std::min(8u, std::max(1u, hw));
    }
    const size_t min_slice = (size_t)4 << 20;
    if (threads <= 1 || n < 2 * min_slice) return false;
    struct stat st;
    if (fstat(fd, &st) != 0 || !S_ISREG(st.st_mode)) return false;
    const int fl = fcntl(fd, F_GETFL);
    if (fl < 0 || (fl & O_APPEND)) return false;
    const off_t base = lseek(fd, 0, SEEK_CUR);
    if (base < 0) return false;
    const int parts = (int)std::min<size_t>((size_t)threads, n / min_slice);
    const size_t slice = (((n + parts - 1) / parts) + 4095) & ~(size_t)4095;   // parts * slice >= n
    std::vector<char> ok(parts, 0);
    std::vector<std::thread> th;
    auto work = [&](int i) {
        size_t b = std::min(n, (size_t)i * slice);
        const size_t e2 = std::min(n, b + slice);
        while (b < e2) {
            ssize_t w = ::pwrite(fd, p + b, e2 - b, base + (off_t)b);
            if (w < 0 && errno == EINTR) continue;
            if (w <= 0) return;
            b += (size_t)w;
        }
        ok[i] = 1;
    };
    for (int i = 1; i < parts; ++i) th.emplace_back(work, i);
    work(0);
    for (auto &t : th) t.join();
    for (int i = 0; i < parts; ++i) if (!ok[i]) return false;   // the caller falls back to write(2) from `base`
    lseek(fd, base + (off_t)n, SEEK_SET);
    return true;
}

bool write_all(int fd, const char *p, size_t n) {
    if (write_parallel(fd, p, n)) return true;
    while (n) {
        ssize_t w = ::write(fd, p, n);
        if (w < 0 && errno == EINTR) continue;
        if (w <= 0) return false;
        p += w; n -= (size_t)w;
    }
    return true;
}

void finish(int rc) {
    fflush(stdout); fflush(stderr);
    _exit(rc);
}

bool read_sample_header(Source &src, std::string &head, std::vector<std::string> &names, const char *format) {
    std::string chrom;
    bool found_chrom = false;
    {
        std::string buf(1 << 16, '\0');
        size_t scan = 0;
        bool eof = false;
        for (;;) {
            size_t nl;
            while ((nl = head.find('\n', scan)) == std::string::npos && !eof) {
                long r = src.read(&buf[0], buf.size());
                if (r < 0) { fputs("Error: read error\n", stderr); return false; }
                if (r == 0) { eof = true; break; }
                head.append(buf.data(), (size_t)r);
            }
            if (scan >= head.size()) break;
            size_t end = (nl == std::string::npos) ? head.size() : nl;
            if (end > scan && head[end - 1] == '\r') --end;
            if (end > scan) {
                if (head[scan] != '#') {
                    if (!found_chrom) { fputs("Error: VCF header (#CHROM) not found before variant records.\n", stderr); return false; }
                    break;
                }
                if (!found_chrom && end - scan >= 6 && head.compare(scan, 6, "#CHROM") == 0) {
                    found_chrom = true;
                    chrom = head.substr(scan, end - scan);
                }
            }
            if (nl == std::string::npos) break;
            scan = nl + 1;
        }
    }
    if (!found_chrom) { fputs("Error: no #CHROM header line in the input.\n", stderr); return false; }
    {
        size_t p = 0;
        for (int col = 0;; ++col) {
            const size_t t = chrom.find('\t', p);
            const size_t e = t == std::string::npos ? chrom.size() : t;
            if (col >= 9) names.push_back(chrom.substr(p, e - p));
            if (t == std::string::npos) break;
            p = t + 1;
        }
        if (!names.empty() && names.back().empty()) names.pop_back();      // an empty column behind a final tab
    }
    for (size_t i = 0; i < names.size(); ++i) {
        bool bad = names[i].empty();
        for (unsigned char ch : names[i]) bad |= isspace(ch) != 0;
        if (bad) {
            fprintf(stderr, "Error: sample %zu ('%s') is empty or contains a blank; %s is whitespace-delimited.\n", i + 1, names[i].c_str(), format);
            return false;
        }
    }
    return true;
}

bool AsideFiles::open_all() {
    fd.assign(ext.size(), -1);
    tmp.assign(ext.size(), std::string());
    for (size_t i = 0; i < ext.size(); ++i) {
        tmp[i] = prefix + ext[i] + "." + std::to_string((long)getpid()) + ".part";
        fd[i] = open(tmp[i].c_str(), O_WRONLY | O_CREAT | O_TRUNC | O_EXCL, 0666);
        if (fd[i] < 0) { fprintf(stderr, "Error: cannot create '%s%s'\n", prefix.c_str(), ext[i].c_str()); return false; }
    }
    return true;
}

void AsideFiles::discard() {
    for (size_t i = 0; i < fd.size(); ++i) {
        if (fd[i] >= 0) { close(fd[i]); fd[i] = -1; }
        if (!tmp[i].empty()) unlink(tmp[i].c_str());
    }
}

bool AsideFiles::commit() {
    for (size_t i = 0; i < fd.size(); ++i) {
        const int rc = close(fd[i]);
        fd[i] = -1;
        if (rc != 0) { fprintf(stderr, "Error: cannot write '%s%s'\n", prefix.c_str(), ext[i].c_str()); return false; }
    }
    for (size_t i = 0; i < fd.size(); ++i)
        if (rename(tmp[i].c_str(), (prefix + ext[i]).c_str()) != 0) {
            fprintf(stderr, "Error: cannot create '%s%s'\n", prefix.c_str(), ext[i].c_str());
            for (size_t j = 0; j < i; ++j) unlink((prefix + ext[j]).c_str());
            return false;
        }
    return true;
}

int env_device() {
    const char *e = getenv("VCFX_CUDA_DEVICE");
    return e ? atoi(e) : 0;
}

// VCFX_CUDA_DEVICES=0,1,2,3 (or "all"): one context per GPU in this one process, chunks dealt round-robin and drained
// in submission order — the text leaves in file order, exactly as with one GPU (the reference's own decomposition at
// thread level: allele_counter.cpp:870-947 cuts the data into newline-aligned ranges and writes the results in order).
std::vector<int> env_devices() {
    std::vector<int> d;
    const char *e = getenv("VCFX_CUDA_DEVICES");
    if (e && *e) {
        if (strcmp(e, "all") == 0) {
            int n = 0;
            vcfx_cuda_device_count(&n);
            for (int i = 0; i < n; ++i) d.push_back(i);
        } else {
            const char *p = e;
            while (*p) {
                char *end = nullptr;
                long v = strtol(p, &end, 10);
                if (end == p) break;
                if (v >= 0) d.push_back((int)v);
                p = (*end == ',') ? end + 1 : end;
                if (*end && *end != ',') break;
            }
        }
    }
    if (d.empty()) d.push_back(env_device());
    return d;
}

namespace {

// Finished text goes to the output descriptor on a thread of its own, in order: while chunk k is being written
// (a pipe or a file can be slow) the main thread reads and submits the next chunk and the library copies chunk
// k+1 back from the device.  A slot's pinned output buffer is handed to a new chunk only after its text was written
// (wait_done before the slot is acquired again).
class Writer {
  public:
    Writer(int fd) : fd_(fd), th_([this] { loop(); }) {}
    ~Writer() { { std::lock_guard<std::mutex> g(m_); stop_ = true; } cv_.notify_all(); th_.join(); }
    void push(const char *p, size_t n) { { std::lock_guard<std::mutex> g(m_); q_.push_back({p, n}); ++pushed_; } cv_.notify_all(); }
    // block until the first k pieces are written (pieces are pushed one per drained chunk, in order)
    void wait_done_at_least(long k) { std::unique_lock<std::mutex> g(m_); cv_.wait(g, [&] { return done_ >= std::min(k, pushed_); }); }
    bool failed() { std::lock_guard<std::mutex> g(m_); return failed_; }

  private:
    void loop() {
        for (;;) {
            std::pair<const char *, size_t> it;
            {
                std::unique_lock<std::mutex> g(m_);
                cv_.wait(g, [&] { return stop_ || !q_.empty(); });
                if (q_.empty()) return;
                it = q_.front(); q_.pop_front();
            }
            bool ok = true;
            { std::lock_guard<std::mutex> g(m_); ok = !failed_; }
            if (ok && !write_all(fd_, it.first, it.second)) { std::lock_guard<std::mutex> g(m_); failed_ = true; }   // like the reference, a closed pipe is not an error
            { std::lock_guard<std::mutex> g(m_); ++done_; }
            cv_.notify_all();
        }
    }
    int fd_;
    std::mutex m_; std::condition_variable cv_;
    std::deque<std::pair<const char *, size_t>> q_;
    long pushed_ = 0, done_ = 0;
    bool stop_ = false, failed_ = false;
    std::thread th_;
};

struct Drain {
    std::vector<vcfx_ctx *> ctxs; const RunOptions &opt; Totals &tot; Writer *writer = nullptr; uint64_t line_base = 0;
    long drained = 0, final_index = -1;
    struct Input { const char *buf; size_t nbytes; uint64_t file_offset; size_t tail_out; bool has_data; };
    std::deque<Input> inputs;               // the pinned input of every chunk in flight (intact until its slot is acquired again)
    std::string held;                       // hold_trailing_hash: '#' lines waiting for a data line
    int one(std::string &err) {
        const char *text = nullptr; size_t n = 0; vcfx_chunk_stats st;
        vcfx_ctx *ctx = ctxs[(size_t)drained % ctxs.size()];        // chunks were dealt round-robin: the oldest one is this context's
        int rc = vcfx_cuda_next_output(ctx, &text, &n, &st);
        if (rc != VCFX_OK) { err = std::string(vcfx_cuda_strerror(rc)) + ": " + vcfx_cuda_last_error(ctx); return rc; }
        if (opt.on_output && !inputs.empty()) {
            const Input &in = inputs.front();
            if (!opt.on_output(in.buf, in.nbytes, in.file_offset, &text, &n)) { err = "output hook failed"; return VCFX_E_INVALID; }
        }
        if (opt.hold_trailing_hash && !inputs.empty()) {
            const Input &in = inputs.front();
            const size_t tail = std::min(in.tail_out, n);
            if (in.has_data) {
                if (!held.empty()) { write_all(opt.out_fd, held.data(), held.size()); held.clear(); }
                write_all(opt.out_fd, text, n - tail);
                held.assign(text + (n - tail), tail);
            } else held.append(text, n);
        }
        else if (opt.capture) { if (n) opt.capture->append(text, n); }
        else if (opt.capture_final && drained == final_index) { if (n) opt.capture_final->append(text, n); }
        else if (opt.sink) { if (n && !opt.sink(text, n)) { err = "output sink failed"; return VCFX_E_INVALID; } }
        else if (writer) writer->push(text, n);        // (empty pieces too: the writer's count follows the chunks)
        tot.bytes_in += st.bytes_in; tot.bytes_out += st.bytes_out; tot.data_lines += st.data_lines;
        tot.rows += st.rows; tot.flagged += st.flagged; tot.pre_header += st.pre_header;
        tot.short_lines += st.short_lines; tot.dots_terminated += st.dots_terminated;
        tot.last_unterminated_flagged = st.last_unterminated_flagged;
        tot.kernel_ms += st.kernel_ms;
        if (st.first_short_line && !tot.first_short_line) tot.first_short_line = line_base + st.first_short_line;
        if (opt.want_short_lines && st.n_events) {
            std::vector<uint64_t> ev((size_t)std::min<uint64_t>(st.n_events, 1u << 20));
            size_t got = 0;
            vcfx_cuda_short_lines(ctx, ev.data(), ev.size(), &got);
            for (size_t i = 0; i < got; ++i) tot.short_line_numbers.push_back(line_base + ev[i]);
        }
        if (opt.on_events && st.n_events && !inputs.empty()) {
            std::vector<uint64_t> ev((size_t)st.n_events);
            size_t got = 0;
            vcfx_cuda_short_lines(ctx, ev.data(), ev.size(), &got);
            opt.on_events(inputs.front().buf, inputs.front().nbytes, ev.data(), got);
        }
        if (!inputs.empty()) inputs.pop_front();
        tot.lines += st.lines;
        line_base += st.lines;
        ++drained;
        return VCFX_OK;
    }
};

}  // namespace

// ---------------------------------------------------------------------------------- run_stream
int run_stream(Source &src, const RunOptions &opt, Totals &tot, std::string &err) {
    vcfx_cfg cfg;
    memset(&cfg, 0, sizeof cfg);
    cfg.device = env_device(); cfg.op = opt.op; cfg.mode = opt.mode; cfg.flags = opt.flags;
    size_t chunk = opt.chunk_bytes;
    if (!chunk) { const char *e = getenv("VCFX_CHUNK_BYTES"); chunk = e ? (size_t)strtoull(e, nullptr, 10) : (size_t)64 << 20; }
    cfg.chunk_bytes = chunk; cfg.n_slots = 3;
    std::string names_blob; std::vector<uint32_t> name_off;
    if (!opt.query.empty()) { cfg.n_sel = (uint32_t)opt.query.size(); cfg.sel_names = opt.query.data(); }
    else if (opt.n_sel) cfg.n_sel = opt.n_sel;
    else if (!opt.sel_col.empty()) {
        name_off.push_back(0);
        for (const auto &s : opt.sel_names) { names_blob += s; names_blob.push_back('\t'); name_off.push_back((uint32_t)names_blob.size()); }
        cfg.n_sel = (uint32_t)opt.sel_col.size(); cfg.sel_col = opt.sel_col.data();
        cfg.sel_names = names_blob.data(); cfg.sel_name_off = name_off.data();
    }
    const bool timing = getenv("VCFX_TIMING") != nullptr;
    auto now = [] { return std::chrono::duration<double>(std::chrono::steady_clock::now().time_since_epoch()).count(); };
    double t_start = now(), t_read = 0, t_submit = 0, t_drain = 0, t_acquire = 0;
    std::vector<int> devices = env_devices();
    if (opt.single_device && devices.size() > 1) devices.resize(1);
    // One GPU: hide the others from the CUDA runtime before it initialises (it would set up every visible GPU — on an
    // 8-GPU box that is most of a tool's wall time).  VCFX_CUDA_DEVICE counts within CUDA_VISIBLE_DEVICES when that is set.
    if (devices.size() == 1 && !getenv("VCFX_KEEP_VISIBLE")) {
        const char *vis = getenv("CUDA_VISIBLE_DEVICES");
        std::string pick;
        if (!vis || !*vis) pick = std::to_string(devices[0]);
        else {
            std::string v(vis);
            size_t pos = 0; int k = 0;
            while (pos <= v.size()) {
                size_t c = v.find(',', pos);
                if (c == std::string::npos) c = v.size();
                if (k == devices[0]) { pick = v.substr(pos, c - pos); break; }
                pos = c + 1; ++k;
            }
        }
        if (!pick.empty()) { setenv("CUDA_VISIBLE_DEVICES", pick.c_str(), 1); devices[0] = 0; }
    }
    std::vector<vcfx_ctx *> ctxs;
    int rc = VCFX_OK;
    auto destroy_all = [&ctxs] { for (vcfx_ctx *c : ctxs) vcfx_cuda_destroy(c); ctxs.clear(); };
    {
        // one context per GPU, created side by side (a CUDA context costs about a second, most of a tool's wall time)
        std::vector<vcfx_ctx *> made(devices.size(), nullptr);
        std::vector<int> rcs(devices.size(), VCFX_OK);
        std::vector<std::thread> th;
        auto make = [&](size_t i) { vcfx_cfg c = cfg; c.device = devices[i]; rcs[i] = vcfx_cuda_create(&c, &made[i]); };
        for (size_t i = 1; i < devices.size(); ++i) th.emplace_back(make, i);
        make(0);
        for (auto &t : th) t.join();
        for (size_t i = 0; i < devices.size(); ++i) if (made[i]) ctxs.push_back(made[i]);
        for (size_t i = 0; i < devices.size(); ++i)
            if (rcs[i] != VCFX_OK) { rc = rcs[i]; err = vcfx_cuda_strerror(rc); destroy_all(); return rc; }
    }
    const size_t G = ctxs.size();
    if (opt.first_device) *opt.first_device = devices[0];
    double t_create = now() - t_start;
    auto in_flight_total = [&ctxs] { long k = 0; for (vcfx_ctx *c : ctxs) k += vcfx_cuda_in_flight(c); return k; };

    const bool direct = !opt.capture && !opt.sink && !opt.hold_trailing_hash;
    Writer *writer = direct ? new Writer(opt.out_fd) : nullptr;
    struct WriterGuard { Writer *w; ~WriterGuard() { delete w; } } writer_guard{writer};     // joins after the last piece is out
    Drain drain{ctxs, opt, tot, writer};
    const long n_slots = (long)cfg.n_slots * (long)G;     // pinned output buffers in rotation over all the contexts
    std::string carry = opt.preface;
    bool eof = false, chrom_seen = false, in_hash_block = true, index_saw_hash = false, format_seen = false, final_submitted = false;
    uint64_t file_pos = 0;                         // offset of the next chunk in the whole input
    long submitted = 0;
    while (!eof) {
        char *buf = nullptr; size_t cap = 0;
        vcfx_ctx *ctx = ctxs[(size_t)submitted % G];                 // this chunk's GPU
        double t0 = now();
        rc = vcfx_cuda_acquire_input(ctx, &buf, &cap);
        t_acquire += now() - t0;
        while (rc == VCFX_E_BUSY) {
            t0 = now();
            if ((rc = drain.one(err)) != VCFX_OK) { destroy_all(); return rc; }
            t_drain += now() - t0;
            t0 = now();
            rc = vcfx_cuda_acquire_input(ctx, &buf, &cap);
            t_acquire += now() - t0;
        }
        t0 = now();
        if (rc != VCFX_OK) { err = std::string(vcfx_cuda_strerror(rc)) + ": " + vcfx_cuda_last_error(ctx); destroy_all(); return rc; }
        // the slot just acquired held the chunk n_slots back (drained by now): its text must have left the pinned
        // output buffer before this chunk's text can land there
        if (writer) writer->wait_done_at_least(submitted - n_slots + 1);
        // bytes already in hand (the tail of the previous chunk, or what the caller consumed while
        // looking at the header) go first; the source is only read once they fit
        size_t have = std::min(carry.size(), cap);
        memcpy(buf, carry.data(), have);
        carry.erase(0, have);
        if (opt.preface_only && carry.empty()) eof = true;
        while (have < cap && carry.empty() && !opt.preface_only) {
            long r = src.read(buf + have, cap - have);
            if (r < 0) { err = "read error"; destroy_all(); return VCFX_E_INVALID; }
            if (r == 0) { eof = true; break; }
            have += (size_t)r;
        }
        t_read += now() - t0;
        size_t nbytes = have;
        if (!eof) {
            const char *nl = static_cast<const char *>(memrchr(buf, '\n', have));
            if (!nl) { err = "a line is longer than the chunk size (set VCFX_CHUNK_BYTES)"; destroy_all(); return VCFX_E_INVALID; }
            nbytes = (size_t)(nl - buf) + 1;
            carry.insert(0, buf + nbytes, have - nbytes);
        } else if (opt.last_unterminated_line && nbytes && buf[nbytes - 1] != '\n') {
            const char *nl = static_cast<const char *>(memrchr(buf, '\n', nbytes));
            const char *s = nl ? nl + 1 : buf;
            opt.last_unterminated_line->assign(s, (size_t)(buf + nbytes - s));
        }
        if (nbytes == 0 && !(opt.always_submit_final && !final_submitted)) break;
        if (eof) final_submitted = true;
        vcfx_chunk_info info; memset(&info, 0, sizeof info);
        info.is_final = eof ? 1 : 0;
        info.file_offset = file_pos;
        file_pos += nbytes;
        if (opt.rule == HeaderRule::ChromHeader) {
            // data lines before the first line that starts with "#CHROM" are skipped with a warning
            // (allele_freq_calc.cpp:372-386): a prefix fact, found once, here
            if (chrom_seen) info.data_valid_from = 0;
            else {
                size_t off = nbytes;
                if (nbytes >= 6 && memcmp(buf, "#CHROM", 6) == 0) off = 0;
                else if (const void *m = memmem(buf, nbytes, "\n#CHROM", 7)) off = (size_t)(static_cast<const char *>(m) - buf) + 1;
                if (off < nbytes) chrom_seen = true;
                info.data_valid_from = off;
            }
            if (opt.op == VCFX_OP_PHASE_CHECK && opt.mode == VCFX_MODE_FILE && !format_seen) {
                // VCFX_phase_checker's file mode keeps the last FORMAT string with its GT index and starts with ("", 0): an empty
                // FORMAT column means "GT first" for the lines in front of the first one with a non-empty FORMAT (:486-488, :313-316)
                size_t pos = (size_t)info.data_valid_from, bound = nbytes;
                while (pos < nbytes) {
                    const char *nl = static_cast<const char *>(memchr(buf + pos, '\n', nbytes - pos));
                    const size_t le = nl ? (size_t)(nl - buf) : nbytes;
                    size_t e2 = le;
                    if (e2 > pos && buf[e2 - 1] == '\r') --e2;
                    if (e2 > pos && buf[pos] != '#') {
                        size_t p = pos; int tabs = 0;
                        while (p < e2 && tabs < 8) { if (buf[p] == '\t') ++tabs; ++p; }
                        if (tabs == 8 && p < e2 && buf[p] != '\t') { bound = pos; format_seen = true; break; }
                    }
                    pos = le + 1;
                }
                info.format_cache_from = bound;
            }
        } else if (opt.rule == HeaderRule::IndexChrom) {
            // VCFX_indexer: rows start behind the first "#CHROM" line — file mode: blanks / tabs, then "#CHROM" (:108-122);
            // stdin mode: white space, then a first field that is exactly "#CHROM" with a second one behind it (:349-356).
            // A data line in front of every '#' line makes the tool complain once (:313-316 / :362-366).
            if (chrom_seen) info.data_valid_from = 0;
            else {
                size_t pos = 0, off = nbytes;
                while (pos < nbytes) {
                    const char *nl = static_cast<const char *>(memchr(buf + pos, '\n', nbytes - pos));
                    const size_t le = nl ? (size_t)(nl - buf) : nbytes;
                    size_t e2 = le;
                    if (e2 > pos && buf[e2 - 1] == '\r') --e2;
                    if (e2 > pos) {
                        size_t p = pos;
                        if (opt.mode == VCFX_MODE_FILE) while (p < e2 && (buf[p] == ' ' || buf[p] == '\t')) ++p;
                        else while (p < e2 && (buf[p] == ' ' || (buf[p] >= 9 && buf[p] <= 13))) ++p;
                        if (p < e2 && buf[p] == '#') {
                            index_saw_hash = true;
                            bool hit;
                            if (opt.mode == VCFX_MODE_FILE) hit = e2 - pos >= 6 && e2 - p >= 6 && memcmp(buf + p, "#CHROM", 6) == 0;
                            else hit = e2 - p >= 7 && memcmp(buf + p, "#CHROM\t", 7) == 0;
                            if (hit) { off = pos; break; }
                        } else if (!index_saw_hash) tot.index_warned = true;
                    }
                    pos = le + 1;
                }
                if (off < nbytes) {
                    chrom_seen = true; tot.index_header_found = true;
                    if (!opt.header_row.empty()) {
                        if (opt.capture) opt.capture->append(opt.header_row);
                        else if (opt.sink) opt.sink(opt.header_row.data(), opt.header_row.size());
                        else write_all(opt.out_fd, opt.header_row.data(), opt.header_row.size());
                    }
                }
                info.data_valid_from = off;
            }
        } else if (opt.rule == HeaderRule::LeadingHashBlock) {
            // end of the leading block of '#' lines (missing_detector.cpp:378-383)
            size_t pos = 0;
            while (in_hash_block && pos < nbytes) {
                if (buf[pos] != '#') { in_hash_block = false; break; }
                const char *nl = static_cast<const char *>(memchr(buf + pos, '\n', nbytes - pos));
                pos = nl ? (size_t)(nl - buf) + 1 : nbytes;
            }
            info.data_valid_from = pos;
        }
        if (eof) drain.final_index = submitted;
        t0 = now();
        rc = vcfx_cuda_submit(ctx, nbytes, &info);
        t_submit += now() - t0;
        {
            Drain::Input in{buf, nbytes, info.file_offset, 0, true};
            if (opt.hold_trailing_hash) {
                // the run of '#' and empty lines at the end of the chunk: what it puts out ('#' line + '\n' each), and whether
                // any data line stands in front of it
                size_t end = nbytes;
                in.has_data = false;
                while (end > 0) {
                    const size_t le = (buf[end - 1] == '\n') ? end - 1 : end;          // line end (the last line may lack its '\n')
                    const void *pnl = le ? memrchr(buf, '\n', le) : nullptr;
                    const size_t ls = pnl ? (size_t)(static_cast<const char *>(pnl) - buf) + 1 : 0;
                    if (le > ls) {
                        if (buf[ls] != '#') { in.has_data = true; break; }
                        in.tail_out += le - ls + 1;
                    }
                    end = ls;
                }
            }
            drain.inputs.push_back(in);
        }
        ++submitted;
        if (rc != VCFX_OK) { err = std::string(vcfx_cuda_strerror(rc)) + ": " + vcfx_cuda_last_error(ctx); destroy_all(); return rc; }
        if (opt.stop_at_first_short && in_flight_total() >= 2) {
            // --strict only needs the first short line: check as chunks complete, stop early
            if ((rc = drain.one(err)) != VCFX_OK) { destroy_all(); return rc; }
            if (tot.short_lines) break;
        }
    }
    double t0 = now();
    while (in_flight_total() > 0)
        if ((rc = drain.one(err)) != VCFX_OK) { destroy_all(); return rc; }
    if (writer) writer->wait_done_at_least(submitted);
    t_drain += now() - t0;
    t0 = now();
    if (!opt.skip_destroy) destroy_all();
    if (timing)
        fprintf(stderr, "[vcfx timing] create %.3f acquire %.3f read %.3f submit %.3f drain %.3f destroy %.3f total %.3f s, kernels %.3f ms, %ld chunks, %zu GPU(s)\n",
                t_create, t_acquire, t_read, t_submit, t_drain, now() - t0, now() - t_start, tot.kernel_ms, submitted, G);
    return VCFX_OK;
}

}  // namespace vcfxh
