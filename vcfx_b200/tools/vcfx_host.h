// vcfx_host.h — host side shared by the five drop-in tools: the streaming chunk reader that
// replaces the per-line loops of the reference (include/vcfx_io.h:14-24 getline + split_tabs,
// and each tool's private MappedFile / findNewlineSIMD loop), feeding libvcfx_cuda through its
// C ABI.  Nothing here parses records: it moves bytes, keeps chunks newline-aligned, tracks the
// two header facts that are prefix state (first "#CHROM" line, end of the leading '#' block),
// and writes the returned text to stdout in order.
#pragma once
#include <cstdint>
#include <cstdio>
#include <functional>
#include <string>
#include <vector>

#include "vcfx_cuda.h"

namespace vcfxh {

// A byte source: a plain fd, or a gzip stream on an fd (variant_counter's stdin, the only place
// the reference inflates on this path: VCFX_variant_counter.cpp:223-290).
class Source {
  public:
    explicit Source(int fd) : fd_(fd) {}
    ~Source();
    // true when the first two bytes are the gzip magic (consumes nothing)
    bool sniff_gzip();
    bool at_eof_initially();              // like std::cin.peek() == EOF
    void enable_gzip();
    // read up to cap bytes; 0 = end of input; < 0 = error
    long read(char *dst, size_t cap);
    bool failed() const { return failed_; }

  private:
    long raw_read(char *dst, size_t cap);
    long parallel_read(char *dst, size_t cap);   // -2: not applicable (pipe, small read, one thread)
    int fd_;
    long long file_size_ = -1, file_off_ = 0;    // regular files only (-1: not a regular file)
    bool io_init_ = false;
    int io_threads_ = 1;
    std::string peek_;                    // bytes read ahead by sniff/peek
    size_t peek_pos_ = 0;
    bool gz_ = false, gz_done_ = false, failed_ = false;
    void *zs_ = nullptr;                  // z_stream*
    std::vector<char> zin_;
    size_t zin_len_ = 0, zin_pos_ = 0;
};

struct Totals {
    uint64_t bytes_in = 0, bytes_out = 0, lines = 0, data_lines = 0, rows = 0, flagged = 0;
    uint64_t pre_header = 0, short_lines = 0, first_short_line = 0, dots_terminated = 0;
    uint64_t last_unterminated_flagged = 0;
    std::vector<uint64_t> short_line_numbers;   // 1-based, whole input
    double kernel_ms = 0;
    bool index_header_found = false;            // IndexChrom: a "#CHROM" line was seen (the header row was written)
    bool index_warned = false;                  // IndexChrom: a data line came before any '#' line
};

enum class HeaderRule { None, ChromHeader, LeadingHashBlock, IndexChrom };

struct RunOptions {
    int op = 0, mode = 0;
    unsigned flags = 0;
    HeaderRule rule = HeaderRule::None;
    bool want_short_lines = false;        // collect line numbers of short lines (variant_counter)
    bool stop_at_first_short = false;     // --strict: stop reading once a short line was seen
    int out_fd = 1;
    size_t chunk_bytes = 0;               // 0 = VCFX_CHUNK_BYTES env or 64 MiB
    // allele_counter selection
    std::vector<uint32_t> sel_col;
    std::vector<std::string> sel_names;
    // when set, the text is appended here instead of being written to out_fd
    std::string *capture = nullptr;
    // IndexChrom: written once, in stream order, when the "#CHROM" line is found (VCFX_indexer prints its header row then)
    std::string header_row;
    // when set, every piece of text is handed to this function instead (in order; false = stop with an error)
    std::function<bool(const char *, size_t)> sink;
    // when set, called once per chunk that has events, in stream order, with the chunk's input bytes and its sorted event
    // list (VCFX_OP_PHASE_CHECK: offset of a dropped line in the chunk << 2 | reason)
    std::function<void(const char *chunk, size_t nbytes, const uint64_t *events, size_t n)> on_events;
    // when set, called once per drained chunk, in stream order, with the chunk's input bytes, its offset in the whole input
    // and its output piece, before the piece goes out; it may narrow the piece to what is written (false = stop with an error)
    std::function<bool(const char *chunk, size_t nbytes, uint64_t file_offset, const char **out, size_t *n)> on_output;
    // cfg.n_sel for an op that takes a plain count (dosage_calculator's matrix / .bed width W)
    uint32_t n_sel = 0;
    // genotype_query: the -g argument (cfg.sel_names = its bytes, cfg.n_sel = its length)
    std::string query;
    // nothing is read from the source: the input is `preface` alone
    bool preface_only = false;
    // VCFX_genotype_query's stdin mode prints '#' lines only once a data line follows them: the text of the '#' lines at the
    // end of a chunk is held back until a later chunk has a data line, and dropped at the end of the input
    bool hold_trailing_hash = false;
    // a chunk marked final is always submitted, an empty one if need be (an op whose text only comes with the final chunk)
    bool always_submit_final = false;
    // chunks go to one GPU only, in order (an op that carries state from chunk to chunk)
    bool single_device = false;
    // when set, only the text of the FINAL chunk is held back here (everything before is written)
    std::string *capture_final = nullptr;
    // keeps a copy of the last line of the input when it has no '\n' (missing_detector's quirk)
    std::string *last_unterminated_line = nullptr;
    // bytes that were already consumed from the source and belong in front of it
    std::string preface;
    // a tool that exits right after the run does not tear the CUDA context down (the OS does, faster)
    bool skip_destroy = true;
};

// Streams `src` through libvcfx_cuda. Returns 0, or a negative vcfx_err; err_text gets a message.
int run_stream(Source &src, const RunOptions &opt, Totals &tot, std::string &err_text);

int env_device();
std::vector<int> env_devices();       // VCFX_CUDA_DEVICES=0,1,.. | all (else the one device of VCFX_CUDA_DEVICE)
// flush stdio and leave without running the CUDA runtime's exit handlers (they cost up to a second)
[[noreturn]] void finish(int rc);
bool write_all(int fd, const char *p, size_t n);

}  // namespace vcfxh
