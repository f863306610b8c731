// vcfx_kernels.cuh — sm_100a kernels of the VCFX hot path.
//
// K1  vcfx_scan_kernel<OP>   one fused pass over the bytes: line scan, field location,
//                            genotype parse, per-variant reduction, row records
// K2a tile_scan_kernel       exclusive scan of the per-tile output sizes / line counts
// K2b format_rows_kernel<OP> a warp per 32 rows: verbatim CHROM..ALT prefix + number text built in shared
//                            memory, written row by row at the final, file-ordered offset
// K2c md_copy_kernel         missing_detector: the input with insertions (warp per item, 128-bit copies)
//
// Decomposition (DESIGN.md §3): the chunk is cut into byte tiles of `tile_bytes`; one WARP
// owns every line that STARTS inside its tile — the reference's own thread-chunking rule
// (allele_counter.cpp:890-903, missing_detector.cpp:404-422) applied at warp granularity, so
// a line is always parsed from its first byte by one owner and no parser state is stitched
// across tiles.  A warp streams its lines in 512-byte windows (16 B per lane, coalesced
// 128-bit loads, later windows already in flight, L2 prefetch further ahead):
//   stage 1  '\n' and '\t' found with exact SWAR byte compares + __ballot_sync / __popc
//   stage 2  tabs 1..9 of the record ranked by a warp prefix sum; FORMAT -> GT index
//   stage 3  genotypes, three tiers, each exact on what it accepts:
//            tier 1  the whole line is the period-4 lattice "a<sep>b\t", a, b in {0,1}: rounds of two
//                    windows, four funnel shifts per lane and window, one vote per round, alleles
//                    summed as packed words (no per-word XOR, HWE via a sum of squares)
//            tier 2  per-lane lattice (any digit, either separator, per-lane phase)
//            tier 3  every sample from its leading tab: the quick shapes of all tabs of a word at
//                    once (byte-class markers shifted by 1..4 bytes), scalar parsers for the rest
//   stage 4  warp REDUX of the tallies -> one 32-byte row record; K2 turns records into text.
// Tensor cores are not involved: this is byte scanning and integer reduction, HBM-bound.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include "vcfx_numfmt.cuh"

namespace vcfx {

constexpr unsigned FULL = 0xFFFFFFFFu;
constexpr int WARPS_PER_CTA = 8;
constexpr uint32_t WINDOW = 512;

enum : int { OP_VC = 0, OP_AF = 1, OP_HWE = 2, OP_MD = 3, OP_AC = 4, OP_NR = 5, OP_IX = 6, OP_PC = 7, OP_IB = 8, OP_GQ = 9, OP_DS = 10 };
constexpr uint32_t NR_PLAIN = 0xFFFFFFFFu;     // Rec::b of a nonref_filter record: the line is written as its content + '\n' (or not at all)
enum : int { MODE_FILE = 0, MODE_STDIN = 1 };
enum : int { AC_TEXT_MT = 0, AC_TEXT_FWD = 1, AC_AGG = 2, AC_BIN = 3 };
constexpr uint32_t AC_STAGE = 2048;     // per-warp staging bytes for allele_counter rows

struct Rec {                 // one output row (32 B)
    uint32_t tile;           // owning tile
    uint32_t ls_rel;         // line start - tile start
    uint32_t prefix_len;     // bytes of "CHROM\tPOS\tID\tREF\tALT\t" taken verbatim from the line
    uint32_t off_in_tile;    // output offset of this row inside its tile's output
    uint32_t a, b, c, d;     // op-specific integers (AF: alt,total; HWE: homRef,het,homAlt)
};

// inbreeding_calculator: what a sample contributes at a site, by its genotype code (0, 1, 2, IB_NONE); rows in file order
struct IbEntry {
    double x;                     // expected heterozygosity 2 f (1 - f) to add (+0.0 when the sample adds nothing here)
    uint32_t inc;                 // bit 0: the site counts as used for the sample; bit 16: an observed heterozygote
    uint32_t flag;                // (entry IB_NONE only) 1: some sample column of the row is IB_ABSENT
};
struct IbMeta { IbEntry e[4]; };  // 64 B per row; the panels hold 16 * code, the byte offset of a sample's entry
struct IbState {
    unsigned long long seq;       // chunks accumulated so far
    unsigned long long variants;  // used sites of the stream so far
    double *sum;                  // [S] expected heterozygotes, summed in file order
    unsigned long long *het;      // [S] observed heterozygotes
    unsigned int *used;           // [S] sites counted
    uint8_t *last;                // [S] code of the last line that had the column (the reference reuses its code buffer)
};
constexpr uint32_t IB_NONE = 3, IB_ABSENT = 4;
constexpr uint32_t IB_F_GLOBAL = 1, IB_F_SKIP_BOUNDARY = 2, IB_F_COUNT_BOUNDARY = 4;      // = VCFX_F_IB_* of the header

constexpr unsigned int REC_BLOCK = 32;          // row-record slots a warp reserves at a time
constexpr uint32_t RESUME_DONE = 0xFFFFFFFFu;
constexpr uint32_t REC_INVALID = 0xFFFFFFFFu;   // Rec::tile of a reserved slot that was never filled

struct DevStats {
    unsigned long long lines, data_lines, rows, flagged, pre_header, short_lines;
    unsigned long long first_short_key;   // (tile << 32 | line index in tile), min
    unsigned long long n_events;
    unsigned long long dots_terminated;
    unsigned long long last_unterminated_flagged;
    unsigned long long bytes_out;
    unsigned long long overflow;          // OV_* bits: why the launch has to run again (vcfx_api.cu grows what they name)
    unsigned long long first_short_line;  // filled by tile_scan_kernel
    unsigned long long n_recs;            // row-record slots reserved (may exceed rec_cap: then overflow)
    unsigned long long n_unfinished;      // tiles the lattice kernel left to the general kernel
};

// DevStats::overflow.  A launch that sets any of them wrote nothing that can be used; the host grows what the bit names
// and runs the chunk again (its input is still on the device)
enum : unsigned long long {
    OV_RECS = 1,          // more rows than row records (n_recs > rec_cap)
    OV_OUTPUT = 2,        // more output bytes than out_cap (inbreeding_calculator: than text_cap)
    OV_AC_SPEC = 4,       // allele_counter's speculative row sizes were wrong (a count of two digits): size rows by parsing
    OV_IB_ORDER = 8,      // inbreeding_calculator: an earlier chunk is being run again, so this one has to be too
    OV_IB_PANELS = 16,    // inbreeding_calculator: more rows x samples than the panels hold
};

// shared-memory event counters of K1: slot = index of the 64-bit field in DevStats
enum : int { C_LINES = 0, C_DATA = 1, C_ROWS = 2, C_FLAG = 3, C_PRE = 4, C_SHORT = 5, C_DOTS = 8, CNT_SLOTS = 9 };
static_assert(offsetof(DevStats, lines) == 8 * C_LINES && offsetof(DevStats, data_lines) == 8 * C_DATA && offsetof(DevStats, rows) == 8 * C_ROWS &&
              offsetof(DevStats, flagged) == 8 * C_FLAG && offsetof(DevStats, pre_header) == 8 * C_PRE && offsetof(DevStats, short_lines) == 8 * C_SHORT &&
              offsetof(DevStats, dots_terminated) == 8 * C_DOTS, "counter slots follow DevStats");

struct KParams {
    const uint8_t *in;       // chunk bytes; readable and '\n'-filled for >= 64 B past n
    uint64_t n;              // valid bytes
    uint32_t tile_bytes;
    uint32_t n_tiles;
    int32_t mode;
    uint32_t flags;
    uint64_t valid_from;
    uint64_t file_offset;            // offset of the chunk in the whole input (indexer)
    int32_t is_final;
    uint8_t *out;
    uint64_t out_cap;
    uint32_t *tile_lines;            // [n_tiles] lines started in each tile
    unsigned long long *tile_out;    // [n_tiles] output bytes produced by each tile
    unsigned long long *tile_base;   // [n_tiles] exclusive scan of tile_out (K2a)
    unsigned long long *line_base;   // [n_tiles] exclusive scan of tile_lines (K2a)
    uint32_t *tail_start;            // MISSING_DETECT [n_tiles]: verbatim tail of the tile (offset from tile start)
    uint32_t *tail_len;              //   its length; bit 31 = append a '\n' (stdin mode, unterminated last line)
    uint32_t *tail_off;              //   its offset inside the tile's output
    // ALLELE_COUNT
    int32_t ac_fmt;                  // AC_TEXT_MT / AC_TEXT_FWD / AC_AGG / AC_BIN
    int32_t ac_pass;                 // 0 = size the rows, 1 = write them
    int32_t ac_ident;                // the selection is columns 0 .. n_sel-1 in order (-a then needs no per-column scratch)
    int32_t ac_spec;                 // TEXT_MT: size the rows without parsing genotypes (every count one digit); pass 1 verifies
    uint32_t n_sel;                  // selected samples, in output order
    const uint32_t *sel_col;         // [n_sel] sample column (running maximum in the forward modes)
    const uint32_t *name_off;        // [n_sel + 1] offsets into names
    const uint8_t *names;            // selected names, each followed by a tab
    const uint4 *names16;            // [n_sel] the same, one 16-byte zero-padded slot per sample, when all are name_len bytes long
    int32_t ac_bulk;                 // flush the staged rows with cp.async.bulk (shared -> global) instead of 128-bit stores
    uint32_t name_len;               // bytes of every selected name + its tab (<= 12), 0 when they differ: the fast row writer is off
    uint32_t max_col;                // 1 + largest selected column
    uint2 *col_scratch;              // [resident warps][max_col] (ref, alt) of the current line
    unsigned int *ticket;            // dynamic tile counter (zeroed before launch)
    unsigned int *ticket2;           // the same for the general kernel (allele_freq_calc / hwe_tester)
    uint32_t *tile_resume;           // [n_tiles] allele_freq_calc / hwe_tester: where the lattice kernel stopped in the tile (RESUME_DONE: it did not)
    Rec *recs;
    uint8_t *rec_prefix;             // [rec_cap][32] copy of the row prefix when it is <= 32 bytes (AF / HWE)
    uint64_t rec_cap;
    DevStats *stats;
    unsigned long long *events;      // short-line events (tile << 32 | index in tile)
    uint32_t ev_cap;
    unsigned long long fmt0_until;   // phase_checker, file mode: an empty FORMAT column of a line starting below this offset means GT index 0
    int32_t c4_bulk;                 // the skip-ahead loop (FORMAT with several keys) is fed by cp.async.bulk through a ring in shared memory
    // GENOTYPE_QUERY
    uint8_t gq_query[64];            // the -g argument (gq_len bytes)
    uint32_t gq_len;
    int32_t gq_a, gq_b;              // its two alleles, sorted (whatever parseDiploidAlleles left in them; -1 = nothing)
    int32_t gq_strict;               // --strict: the GT must equal the query byte for byte
    // INBREEDING (sample-axis reduction): the scan leaves one code per sample column, a second pass walks the rows in file order
    uint8_t *ib_codes;               // [n + pad] code of sample column j of the line starting at byte L: ib_codes[L + j] (0, 1, 2, IB_NONE, IB_ABSENT)
    IbMeta *ib_rows;                 // [rec_cap] the chunk's rows in file order (ib_rows_kernel)
    uint8_t *ib_panels;              // codes again, in file order and in panels of 32 samples: [panel][row][32] (what a warp of the second pass streams)
    uint64_t ib_panel_cap;           // bytes
    IbState *ib;                     // what lives from chunk to chunk: per-sample sums, the last code of every column, the order guard
    unsigned long long ib_seq;       // number of this chunk in its context (chunks are accumulated strictly in this order)
    int32_t ib_first;                // first chunk of a stream: the per-sample state starts from zero
    uint64_t text_cap;               // bytes the final text may take in out (out_cap is not compared with the row count)
    int32_t ev_raw;                  // 1: events are final values (phase_checker: line offset << 2 | kind), not (tile, index) keys
    // DOSAGE matrix and .bed modes (VCFX_F_DS_MATRIX, VCFX_F_DS_BED): a row is one unit of tile output (tile_base +
    // off_in_tile = its rank), n_sel = W
    int32_t ds_matrix;
    uint64_t unit_bytes;             // output bytes per unit of tile output: 1, or 16 + W (matrix) / 16 + ceil(W / 4) (.bed) (tile_scan_kernel's bytes_out)
};

// ---------------------------------------------------------------------------------------
// byte-parallel compares on a 32-bit word; result has 0x80 in every matching byte (exact)
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t zero_bytes(uint32_t x) {
    return ~(((x & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | x) & 0x80808080u;
}
__device__ __forceinline__ uint32_t eq_bytes(uint32_t w, uint32_t c4) { return zero_bytes(w ^ c4); }

constexpr uint32_t C_TAB = 0x09090909u, C_NL = 0x0A0A0A0Au, C_DOT = 0x2E2E2E2Eu;

// 0x80 in the bytes of a word starting at position `base` that satisfy lo <= pos < hi
__device__ __forceinline__ uint32_t range_mask(uint32_t base, uint32_t lo, uint32_t hi) {
    uint32_t m = 0x80808080u;
    if (lo > base) { uint32_t s = lo - base; m = (s >= 4) ? 0u : (m << (8 * s)); }
    if (hi < base + 4) { m = (hi <= base) ? 0u : (m & (0x80808080u >> (8 * (base + 4 - hi)))); }
    return m;
}

// The same for the four words of a lane at once (bytes pb .. pb+15): one 16-bit keep mask, then each
// nibble is spread to the 0x80 bit of its byte.  Cheaper than four range_mask calls.
__device__ __forceinline__ uint32_t lane_keep16(uint32_t pb, uint32_t lo, uint32_t hi) {
    const uint32_t a = lo > pb ? min(lo - pb, 16u) : 0u;
    const uint32_t b = hi > pb ? min(hi - pb, 16u) : 0u;
    return b > a ? (((1u << b) - 1u) & ~((1u << a) - 1u)) : 0u;
}
__device__ __forceinline__ uint32_t nib80(uint32_t keep16, int j) {
    return ((((keep16 >> (4 * j)) & 0xFu) * 0x00204081u) & 0x01010101u) << 7;
}
__device__ __forceinline__ void clip4(uint32_t &m0, uint32_t &m1, uint32_t &m2, uint32_t &m3, uint32_t pb, uint32_t lo, uint32_t hi) {
    const uint32_t k = lane_keep16(pb, lo, hi);
    m0 &= nib80(k, 0); m1 &= nib80(k, 1); m2 &= nib80(k, 2); m3 &= nib80(k, 3);
}

__device__ __forceinline__ uint4 ld16(const uint8_t *p) { return __ldg(reinterpret_cast<const uint4 *>(p)); }
__device__ __forceinline__ uint32_t ldb(const uint8_t *p) { return (uint32_t)__ldg(p); }
__device__ __forceinline__ uint32_t ldw(const uint8_t *p) { return __ldg(reinterpret_cast<const uint32_t *>(p)); }
// VCFX_EMU: the test-only warp emulator build of this file (tests/emu/); PTX has no meaning there
#ifdef VCFX_EMU
#define VCFX_GRID_CONSTANT
__device__ __forceinline__ void prefetch_l2(const void *) {}
__device__ __forceinline__ void prefetch_l1(const void *) {}
__device__ __forceinline__ int lane_id() { return (int)(threadIdx.x & 31u); }
#else
#define VCFX_GRID_CONSTANT __grid_constant__      // the parameter block may be passed on by reference without a local copy
__device__ __forceinline__ void prefetch_l2(const void *p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
__device__ __forceinline__ void prefetch_l1(const void *p) { asm volatile("prefetch.global.L1 [%0];" ::"l"(p)); }
// %laneid: one S2R when the compiler rematerialises it (it does, a dozen times per line)
__device__ __forceinline__ int lane_id() { int l; asm("mov.u32 %0, %%laneid;" : "=r"(l)); return l; }
#endif

__device__ __forceinline__ bool is_dig(uint32_t b) { return (b - 48u) <= 9u; }
__device__ __forceinline__ bool is_sep(uint32_t b) { return b == '/' || b == '|'; }

// ---------------------------------------------------------------------------------------
// exact scalar parsers (rare path; the bytes were just streamed by this warp, so L1/L2 hits)
// ---------------------------------------------------------------------------------------

// allele_freq_calc.cpp:321-337 + 262-293 for the sample column starting at p.  The column ends
// at the next tab or at the line end; with strip_cr a '\r' directly before the '\n' is not
// content (:363-364).  The chunk is '\n'-padded past its last byte, so the scan always stops.
__device__ __noinline__ uint2 af_sample_slow(const uint8_t *p, bool strip_cr, int gt_index) {
    uint32_t alt = 0, total = 0;
    const uint8_t *se = p;
    uint32_t c = ldb(se);
    while (c != '\t' && c != '\n') { ++se; c = ldb(se); }
    if (strip_cr && c == '\n' && se > p && ldb(se - 1) == '\r') --se;
    for (int i = 0; i < gt_index && p < se; ++i) {
        while (p < se && ldb(p) != ':') ++p;
        if (p < se) ++p;
    }
    if (p >= se) return make_uint2(0u, 0u);
    const uint8_t *ge = p;
    while (ge < se && ldb(ge) != ':') ++ge;
    while (p < ge) {
        while (p < ge && is_sep(ldb(p))) ++p;
        if (p >= ge) break;
        const uint8_t *q = p; bool numeric = true, zero = true; const uint32_t first = ldb(p);
        while (q < ge) {
            uint32_t d = ldb(q);
            if (is_sep(d)) break;
            if (numeric) { if (!is_dig(d)) numeric = false; else if (d != '0') zero = false; }
            ++q;
        }
        if (first != '.' && numeric) { ++total; if (!zero) ++alt; }
        p = q;
    }
    return make_uint2(alt, total);
}

// hwe_tester.cpp:339-378 for the sample column starting at p: first ':' piece only.  A '\r'
// before the '\n' never changes the class (neither digit nor separator), so the piece simply
// ends at ':' / tab / '\n'.
__device__ __noinline__ int hwe_sample_slow(const uint8_t *p) {
    const uint8_t *e = p;
    for (;;) { uint32_t c = ldb(e); if (c == '\t' || c == ':' || c == '\n') break; ++e; }
    while (p < e) { uint32_t c = ldb(p); if (c == ' ' || c == '\r') ++p; else break; }
    if (p >= e) return -1;
    if (!is_dig(ldb(p))) return -1;
    int a1 = 0, a2 = 0;
    while (p < e && is_dig(ldb(p))) { a1 = (a1 > 1) ? 2 : a1 * 10 + (int)(ldb(p) - 48u); ++p; }
    if (p >= e || !is_sep(ldb(p))) return -1;
    ++p;
    if (p >= e || !is_dig(ldb(p))) return -1;
    while (p < e && is_dig(ldb(p))) { a2 = (a2 > 1) ? 2 : a2 * 10 + (int)(ldb(p) - 48u); ++p; }
    if (a1 > 1 || a2 > 1) return -1;       // saturating at 2 keeps ">1" without int overflow
    if (a1 == 0 && a2 == 0) return 0;
    if (a1 == 1 && a2 == 1) return 2;
    return 1;
}

// allele_freq_calc.cpp:298-316 on the FORMAT field [p, e)
__device__ __noinline__ int gt_index_of(const uint8_t *p, const uint8_t *e) {
    int idx = 0;
    while (p < e) {
        const uint8_t *q = p;
        while (q < e && ldb(q) != ':') ++q;
        if (q - p == 2 && ldb(p) == 'G' && ldb(p + 1) == 'T') return idx;
        ++idx;
        p = (q < e) ? q + 1 : q;
    }
    return -1;
}

// VCFX_nonref_filter.cpp for the sample column starting at p: is its GT "definitely" homozygous reference?
//   file mode  (:248-309 allSamplesHomRefDirect): the column ends at a tab or at the line end ('\r' before '\n' is not
//              content); at the line end there is no column (the reference's loop is over: true, "nothing against it");
//              an empty column keeps the line; GT = the piece before the first ':' (gt_index 0) or the gt_index-th piece
//              (empty when there are fewer: keeps the line); three bytes must be 0/0 or 0|0, any other non-empty GT
//              may hold nothing but '0' '/' '|'
//   stdin mode (:553-631 filterNonRef + :419-449 isDefinitelyHomRef): the column ends at a tab or '\n' ('\r' is content);
//              pieces as std::getline yields them (none for an empty column, no empty piece after a final ':'):
//              gt_index beyond them keeps the line; the GT may hold nothing but '0' '/' '|' and must not be empty
__device__ __noinline__ bool nr_sample_homref(const uint8_t *p, bool file_mode, int gt_index) {
    const uint8_t *se = p;
    uint32_t c = ldb(se);
    while (c != '\t' && c != '\n') { ++se; c = ldb(se); }
    if (file_mode && c == '\n' && ldb(se - 1) == '\r') { if (se - 1 >= p) --se; else return true; }   // ("\t\r\n": the line ended before p)
    if (se == p) return (c == '\n') ? file_mode : false;
    const uint8_t *gs = p, *ge = se;
    if (file_mode && gt_index == 0) { ge = p; while (ge < se && ldb(ge) != ':') ++ge; }
    else {
        int idx = 0; const uint8_t *fs = p; bool got = false;
        for (const uint8_t *q = p; q <= se; ++q) {
            if (q == se || ldb(q) == ':') {
                if (idx == gt_index) { gs = fs; ge = q; got = true; break; }
                ++idx; fs = q + 1;
            }
        }
        if (!got) return false;
        if (!file_mode && ge == se && gs == se && ldb(se - 1) == ':') return false;     // std::getline yields no empty piece after a final ':'
    }
    const uint32_t n = (uint32_t)(ge - gs);
    if (n == 0) return false;
    if (file_mode && n == 3) return ldb(gs) == '0' && is_sep(ldb(gs + 1)) && ldb(gs + 2) == '0';
    for (const uint8_t *q = gs; q < ge; ++q) { const uint32_t b = ldb(q); if (b != '0' && !is_sep(b)) return false; }
    return true;
}

// VCFX_phase_checker.cpp:218-268 isFullyPhasedFast on the GT of the sample column starting at p.  The column ends at a tab
// or at the line end (file mode: a '\r' before the '\n' is not content; stdin mode: it is).  At the line end there is no
// column in file mode (the reference's loop is over: true) and an empty one in stdin mode (false); an empty column in the
// middle is never phased.  GT = the piece before the first ':' (gt_index 0) or the gt_index-th piece (:194-213, empty when
// there are fewer).  Three bytes: x|y with x, y not '.'; one byte: no; otherwise every '|'-separated allele must be
// non-empty and not ".", no '/', at least one '|'.
__device__ __noinline__ bool pc_sample_phased(const uint8_t *p, bool file_mode, int gt_index) {
    const uint8_t *se = p;
    uint32_t c = ldb(se);
    while (c != '\t' && c != '\n') { ++se; c = ldb(se); }
    if (file_mode && c == '\n' && ldb(se - 1) == '\r') { if (se - 1 >= p) --se; else return true; }
    if (se == p) return (c == '\n') ? file_mode : false;
    const uint8_t *gs = p, *ge = se;
    if (gt_index == 0) { ge = p; while (ge < se && ldb(ge) != ':') ++ge; }
    else {
        int idx = 0; const uint8_t *fs = p; bool got = false;
        for (const uint8_t *q = p; q <= se; ++q) {
            if (q == se || ldb(q) == ':') {
                if (idx == gt_index) { gs = fs; ge = q; got = true; break; }
                ++idx; fs = q + 1;
            }
        }
        if (!got) return false;
    }
    const uint32_t n = (uint32_t)(ge - gs);
    if (n == 0 || n == 1) return false;
    if (n == 3) return ldb(gs + 1) == '|' && ldb(gs) != '.' && ldb(gs + 2) != '.';
    if (ldb(gs) == '.' && is_sep(ldb(gs + 1)) && ldb(gs + 2) == '.') return false;
    bool pipe = false; const uint8_t *as = gs;
    for (const uint8_t *q = gs; q < ge; ++q) {
        const uint32_t b = ldb(q);
        if (b == '|') {
            const uint32_t al = (uint32_t)(q - as);
            if (al == 0 || (al == 1 && ldb(as) == '.')) return false;
            pipe = true; as = q + 1;
        } else if (b == '/') return false;
    }
    const uint32_t al = (uint32_t)(ge - as);
    if (al == 0 || (al == 1 && ldb(as) == '.')) return false;
    return pipe;
}

// VCFX_genotype_query.cpp:322-344 / 275-317: does the GT of the sample column starting at p equal the query?  The column ends at
// a tab or the line end (a '\r' is content); GT = the gt_index-th ':' piece, an empty one never matches.  --strict: byte for
// byte.  Otherwise both sides are digits, '/' or '|', digits, and the allele pairs are compared without their order.
struct GqQuery { const uint8_t *q; uint32_t len; int a, b; bool strict; };
// the same for a GT of exactly three bytes (the low three bytes of u)
__device__ __forceinline__ bool gq_match3(uint32_t u, const GqQuery &Q) {
    if (Q.strict) return Q.len == 3u && ((u ^ ((uint32_t)Q.q[0] | ((uint32_t)Q.q[1] << 8) | ((uint32_t)Q.q[2] << 16))) & 0x00FFFFFFu) == 0u;
    const uint32_t b1 = (u >> 8) & 0xFFu, d0 = (u & 0xFFu) - '0', d2 = ((u >> 16) & 0xFFu) - '0';
    if ((b1 != '/' && b1 != '|') || d0 > 9u || d2 > 9u) return false;
    return (int)min(d0, d2) == Q.a && (int)max(d0, d2) == Q.b;
}
__device__ __noinline__ bool gq_sample_match(const uint8_t *p, int gt_index, const GqQuery Q) {
    const uint8_t *se = p;
    uint32_t c = ldb(se);
    while (c != '\t' && c != '\n') { ++se; c = ldb(se); }
    const uint8_t *gs = p, *ge = se;
    {
        int idx = 0; const uint8_t *fs = p; bool got = false;
        for (const uint8_t *q = p; q <= se; ++q) {
            if (q == se || ldb(q) == ':') {
                if (idx == gt_index) { gs = fs; ge = q; got = true; break; }
                ++idx; fs = q + 1;
            }
        }
        if (!got) return false;
    }
    const uint32_t n = (uint32_t)(ge - gs);
    if (n == 0) return false;
    if (Q.strict) {
        if (n != Q.len) return false;
        for (uint32_t i = 0; i < n; ++i) if (ldb(gs + i) != Q.q[i]) return false;
        return true;
    }
    uint32_t sp = 0;
    while (sp < n && ldb(gs + sp) != '|' && ldb(gs + sp) != '/') ++sp;
    if (sp == n || sp == 0 || sp == n - 1) return false;
    uint32_t a1 = 0, a2 = 0;
    for (uint32_t i = 0; i < sp; ++i) { const uint32_t d = ldb(gs + i) - '0'; if (d > 9u) return false; a1 = a1 * 10u + d; }
    for (uint32_t i = sp + 1; i < n; ++i) { const uint32_t d = ldb(gs + i) - '0'; if (d > 9u) return false; a2 = a2 * 10u + d; }
    int x = (int)a1, y = (int)a2;
    if (x > y) { const int t = x; x = y; y = t; }
    return x == Q.a && y == Q.b;
}

// VCFX_inbreeding_calculator.cpp:296-339 parseGenotypeCode on the sample column starting at p: blanks and '\r' in front are
// skipped, then digits, '/' or '|', digits — nothing behind them is looked at (a ':' only ends the genotype, and everything
// that ends it is neither a digit nor a separator) — both alleles 0 or 1: 0, 1, 2; anything else IB_NONE.  A column that
// starts at the line end (after a '\r' in front of the '\n' was cut) does not exist: IB_ABSENT.
__device__ __noinline__ uint32_t ib_sample_code(const uint8_t *p) {
    uint32_t c = ldb(p);
    if (c == '\n' || (c == '\r' && ldb(p + 1) == '\n')) return IB_ABSENT;
    while (c == ' ' || c == '\r') { ++p; c = ldb(p); }
    if (c - '0' > 9u) return IB_NONE;
    uint32_t a1 = 0, a2 = 0;
    while (c - '0' <= 9u) { a1 = a1 * 10u + (c - '0'); ++p; c = ldb(p); }
    if (c != '/' && c != '|') return IB_NONE;
    ++p; c = ldb(p);
    if (c - '0' > 9u) return IB_NONE;
    while (c - '0' <= 9u) { a2 = a2 * 10u + (c - '0'); ++p; c = ldb(p); }
    if (a1 > 1u || a2 > 1u) return IB_NONE;
    return a1 + a2;
}

// VCFX_dosage_calculator.cpp:111-154 parseDosageInline on the GT (:182-204 extractGTFromSample: the gt_index-th ':' piece, none when it
// is empty or missing) of the sample column starting at p: separators are skipped, every allele is a run of digits, a '.' or
// any other byte spoils it, exactly two alleles: the number of alleles > 0; else IB_NONE ("NA").  The column ends at a tab or the
// line end (file mode: a '\r' in front of the '\n' is cut first); a column that starts at the line end does not exist: IB_ABSENT.
__device__ __noinline__ uint32_t ds_sample_code(const uint8_t *p, bool file_mode, int gt_index) {
    const uint8_t *se = p;
    uint32_t c = ldb(se);
    while (c != '\t' && c != '\n') { ++se; c = ldb(se); }
    if (file_mode && c == '\n' && se > p && ldb(se - 1) == '\r') --se;
    if (se == p && c == '\n') return IB_ABSENT;
    const uint8_t *gs = p, *ge = se;
    {
        int idx = 0; const uint8_t *fs = p; bool got = false;
        for (const uint8_t *q = p; q <= se; ++q) {
            if (q == se || ldb(q) == ':') {
                if (idx == gt_index) { gs = fs; ge = q; got = true; break; }
                ++idx; fs = q + 1;
            }
        }
        if (!got || ge == gs) return IB_NONE;
    }
    uint32_t dosage = 0, alleles = 0;
    const uint8_t *q = gs;
    while (q < ge) {
        while (q < ge && is_sep(ldb(q))) ++q;
        if (q >= ge) break;
        uint32_t allele = 0; bool digit = false;
        while (q < ge && ldb(q) - '0' <= 9u) { allele = allele * 10u + (ldb(q) - '0'); digit = true; ++q; }
        if (!digit) return IB_NONE;                                  // a '.' or any other byte
        if ((int)allele > 0) ++dosage;
        if (++alleles > 2) return IB_NONE;
    }
    return alleles == 2 ? dosage : IB_NONE;
}

// VCFX_indexer on one data line [s, e) (a '\r' before the '\n' already cut off): where CHROM is and what POS reads as.
//   file mode  (VCFX_indexer.cpp:74-105 extractChromPos): blanks and tabs in front are skipped, CHROM runs to the first
//              tab (not empty, the tab must exist), POS is the digit run behind it in wrapping 64-bit arithmetic and
//              must come out > 0
//   stdin mode (:373-397): fields as splitTabs cuts the line (CHROM = everything in front of the first tab, possibly
//              empty or led by blanks; a second field must exist), POS as std::stoll reads it (white space, a sign,
//              at least one digit, anything behind ignored, out of range = no row)
// A line whose first non-blank byte is '#' is a header line: no row.
__device__ __noinline__ bool ix_parse_line(const uint8_t *s, const uint8_t *e, bool file_mode, uint32_t &c_off, uint32_t &c_len, long long &pos) {
    auto space = [](uint32_t c) { return c == ' ' || (c >= 9u && c <= 13u); };
    const uint8_t *p = s;
    if (file_mode) {
        while (p < e && (ldb(p) == ' ' || ldb(p) == '\t')) ++p;
        if (p >= e || ldb(p) == '#') return false;
        const uint8_t *cs = p;
        while (p < e && ldb(p) != '\t') ++p;
        if (p == cs || p >= e) return false;
        c_off = (uint32_t)(cs - s); c_len = (uint32_t)(p - cs);
        ++p;
        unsigned long long v = 0;
        while (p < e && is_dig(ldb(p))) { v = v * 10ULL + (ldb(p) - 48u); ++p; }
        pos = (long long)v;
        return pos > 0;
    }
    while (p < e && space(ldb(p))) ++p;
    if (p < e && ldb(p) == '#') return false;
    const uint8_t *tab = s;
    while (tab < e && ldb(tab) != '\t') ++tab;
    if (tab >= e) return false;
    c_off = 0; c_len = (uint32_t)(tab - s);
    const uint8_t *q = tab + 1, *pe = q;
    while (pe < e && ldb(pe) != '\t') ++pe;
    while (q < pe && space(ldb(q))) ++q;
    bool neg = false;
    if (q < pe && (ldb(q) == '+' || ldb(q) == '-')) { neg = ldb(q) == '-'; ++q; }
    if (q >= pe || !is_dig(ldb(q))) return false;
    const unsigned long long lim = neg ? 9223372036854775808ULL : 9223372036854775807ULL;
    unsigned long long v = 0;
    while (q < pe && is_dig(ldb(q))) {
        const unsigned long long d = ldb(q) - 48u;
        if (v > (lim - d) / 10ULL) return false;
        v = v * 10ULL + d; ++q;
    }
    pos = neg ? (long long)(0ULL - v) : (long long)v;
    return true;
}
__device__ __forceinline__ uint32_t dec_len64(long long v) {
    unsigned long long u = v < 0 ? 0ULL - (unsigned long long)v : (unsigned long long)v;
    uint32_t n = v < 0 ? 1u : 0u;
    do { ++n; u /= 10ULL; } while (u);
    return n;
}
__device__ __forceinline__ uint8_t *put_dec64(uint8_t *d, long long v) {
    unsigned long long u = v < 0 ? 0ULL - (unsigned long long)v : (unsigned long long)v;
    if (v < 0) *d++ = '-';
    char t[24]; int n = 0;
    do { t[n++] = (char)('0' + (int)(u % 10ULL)); u /= 10ULL; } while (u);
    while (n) *d++ = (uint8_t)t[--n];
    return d;
}

// byte index (0..15) of the first set 0x80-bit over the lane's four mask words, with selects instead of
// branches (the lanes of a warp hold their first tab in different words)
__device__ __forceinline__ int first_byte(uint32_t m0, uint32_t m1, uint32_t m2, uint32_t m3) {
    const uint32_t m = m0 ? m0 : (m1 ? m1 : (m2 ? m2 : m3));
    const int base = m0 ? 0 : (m1 ? 4 : (m2 ? 8 : 12));
    return base + ((__ffs(m) - 1) >> 3);
}

__device__ __forceinline__ int warp_incl_scan(int v, int lane) {
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { int t = __shfl_up_sync(FULL, v, o); if (lane >= o) v += t; }
    return v;
}

// ---------------------------------------------------------------------------------------
// per-lane sample parsing from registers
// ---------------------------------------------------------------------------------------
struct Tally { uint32_t a, b, c; };   // AF: alt,total   HWE: homRef,het,homAlt

// Quick shapes of a sample column, decided from the bytes behind its leading tab WITHOUT branches, so
// the lanes of a warp do not diverge on mixed data:
//   A  <end>                 empty column / empty GT
//   B  t <end>               haploid          t = digit or '.', <end> = tab, ':' or '\n'
//   C  t sep t <end>         diploid, single-character alleles
// Everything else (multi-digit alleles, more alleles, '\r', other bytes, GT not first) goes to the
// exact scalar parsers.
// Byte classes of one word as 0x80 markers (exact)
struct WClass { uint32_t D, Z, P, S, E, O; };   // digit, '0', '.', '/' or '|', tab / ':' / '\n', '1' (HWE only)
template <int OP>
__device__ __forceinline__ WClass classify_word(uint32_t x) {
    // ge(c): 0x80 in every byte whose low seven bits are >= c (a 7-bit add cannot carry into the next
    // byte); a class is a difference of two of them, for bytes without the eighth bit
    const uint32_t x7 = x & 0x7F7F7F7Fu, ok = ~x & 0x80808080u;
#define VCFX_GE(c) (x7 + (0x80808080u - 0x01010101u * (uint32_t)(c)))
    const uint32_t g2e = VCFX_GE(0x2E), g2f = VCFX_GE(0x2F), g30 = VCFX_GE(0x30), g31 = VCFX_GE(0x31);
    const uint32_t g3a = VCFX_GE(0x3A), g3b = VCFX_GE(0x3B), g7c = VCFX_GE(0x7C), g7d = VCFX_GE(0x7D);
    const uint32_t g09 = VCFX_GE(0x09), g0b = VCFX_GE(0x0B);
    WClass c;
    c.P = g2e & ~g2f & ok;                                  // '.'
    c.Z = g30 & ~g31 & ok;                                  // '0'
    c.D = g30 & ~g3a & ok;                                  // '0'..'9'
    c.S = ((g2f & ~g30) | (g7c & ~g7d)) & ok;               // '/' '|'
    c.E = ((g09 & ~g0b) | (g3a & ~g3b)) & ok;               // '\t' '\n' ':'
    c.O = (OP == OP_HWE) ? (g31 & ~VCFX_GE(0x32) & ok) : 0u;   // '1'
#undef VCFX_GE
    return c;
}
// markers of the pair (lo, hi) moved down by k bytes: marker at byte i of the result = marker at byte i + k
__device__ __forceinline__ uint32_t down(uint32_t lo, uint32_t hi, int k) { return __funnelshift_rc(lo, hi, 8u * (uint32_t)k); }

// generic: one sample per owned tab (tab masks m0..m3 over the lane's words w0..w3, la = next 4 B).
// All the tabs of a word are judged at once: the classes of the bytes behind a tab are the class
// markers moved down by 1..4 bytes, so the quick shapes A / B / C above become a few AND/POPC per word; only tabs whose sample is none of them go to the scalar
// parsers, one by one.  Kept out of line: it must not cost the lattice path registers.
template <int OP>
__device__ __noinline__ uint4 lane_samples_generic(uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3, uint32_t la,
                                                   uint32_t m0, uint32_t m1, uint32_t m2, uint32_t m3,
                                                   const uint8_t *lane_ptr, bool strip_cr, int gt_index) {
    const uint32_t ws[5] = {w0, w1, w2, w3, la};
    const uint32_t ms[4] = {m0, m1, m2, m3};
    uint32_t ta = 0, tb = 0, tc = 0, irregular = 0;          // irregular: some sample is not "digit sep digit"
    WClass lo = classify_word<OP>(ws[0]);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const WClass hi = classify_word<OP>(ws[j + 1]);
        const uint32_t m = ms[j];
        uint32_t rest = m;
        if (m) {
            const uint32_t d1 = down(lo.D, hi.D, 1), d3 = down(lo.D, hi.D, 3), s2 = down(lo.S, hi.S, 2);
            if (OP == OP_AF) {
                if (gt_index == 0) {
                    const uint32_t tokl = lo.D | lo.P, tokh = hi.D | hi.P;
                    const uint32_t t1 = down(tokl, tokh, 1), t3 = down(tokl, tokh, 3);
                    const uint32_t e1 = down(lo.E, hi.E, 1), e2 = down(lo.E, hi.E, 2), e4 = hi.E;
                    const uint32_t z1 = down(lo.Z, hi.Z, 1), z3 = down(lo.Z, hi.Z, 3);
                    const uint32_t A = m & e1, B = m & t1 & e2, C = m & t1 & s2 & t3 & e4, any = B | C;
                    tb += __popc(any & d1) + __popc(C & d3);                          // total
                    ta += __popc(any & d1 & ~z1) + __popc(C & d3 & ~z3);              // alt
                    rest = m & ~(A | any);
                    irregular |= m & ~(C & d1 & d3);
                } else irregular = 1;
            } else {
                const uint32_t d2 = down(lo.D, hi.D, 2), d4 = hi.D, p1 = down(lo.P, hi.P, 1);
                const uint32_t o1 = down(lo.O, hi.O, 1), o3 = down(lo.O, hi.O, 3);
                const uint32_t l1 = o1 | down(lo.Z, hi.Z, 1), l3 = o3 | down(lo.Z, hi.Z, 3);   // allele <= 1
                const uint32_t full = m & d1 & s2 & d3 & ~d4;
                const uint32_t rej = m & ((~d1 & p1) | (d1 & ~s2 & ~d2) | (d1 & s2 & ~d3));
                const uint32_t ok = full & l1 & l3;
                ta += __popc(ok & ~o1 & ~o3); tb += __popc(ok & (o1 ^ o3)); tc += __popc(ok & o1 & o3);
                rest = m & ~(full | rej);
                irregular |= m & ~full;
            }
        }
        while (rest) {
            const int k = (__ffs(rest) - 1) >> 3;
            rest &= rest - 1;
            const uint8_t *p = lane_ptr + 4 * j + k + 1;
            if (OP == OP_AF) { const uint2 r = af_sample_slow(p, strip_cr, gt_index); ta += r.x; tb += r.y; }
            else { const int c = hwe_sample_slow(p); ta += (c == 0); tb += (c == 1); tc += (c == 2); }
        }
        lo = hi;
    }
    return make_uint4(ta, tb, tc, irregular);
}

// Lattice check of one lane, branch-free.  tau = byte of the first tab in word 0; the 16 bytes
// after it must be four times [digit, '/' or '|', digit, '\t'].  When that holds the lane's tabs
// are exactly tau+4j, it owns exactly those four diploid single-digit samples, and bytes
// tau+1..tau+16 hold no line end (bytes 0..tau-1 are vouched for by the previous lane's check or
// by the caller's word-0 newline mask).  A word-0 without tab, or with a second tab, cannot
// satisfy the pattern, so no separate test is needed.  Tallies come back packed:
// AF : count of non-'0' digits (the allele total is 8)
// HWE: n01 | het << 8 | homAlt << 16   (n01 = samples whose two digits are both 0/1)
template <int OP>
__device__ __forceinline__ bool lane_lattice(uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3, uint32_t la,
                                             uint32_t &packed, uint32_t &sh) {
    const uint32_t t0 = eq_bytes(w0, C_TAB);
    sh = (uint32_t)__ffs(t0);                               // 8,16,24,32 = 8 * (tau + 1); 0 when no tab
    const uint32_t xs[4] = {__funnelshift_rc(w0, w1, sh), __funnelshift_rc(w1, w2, sh),
                            __funnelshift_rc(w2, w3, sh), __funnelshift_rc(w3, la, sh)};
    uint32_t bad = 0, acc = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const uint32_t y = xs[j] ^ 0x09300030u;              // [d0-'0', sep, d1-'0', 0] when well formed
        // tab byte zero, both digit bytes <= 9 (adding 6 must not reach bit 4)
        bad |= ((y + 0x00060006u) | y) & 0xFFF000F0u;
        const uint32_t sp = y & 0x0000FF00u;
        bad |= (uint32_t)((sp != 0x00007C00u) & (sp != 0x00002F00u));
        if (OP == OP_AF) {
            acc += (y + 0x000F000Fu) & 0x00100010u;          // bit 4 / bit 20 set for digits 1..9
        } else {
            const uint32_t a = y & 0xFFu, b = (y >> 16) & 0xFFu;
            const uint32_t ok = (uint32_t)((a | b) <= 1u);
            acc += ok + ((ok & (a ^ b)) << 8) + ((ok & a & b) << 16);
        }
    }
    packed = (OP == OP_AF) ? (((acc >> 4) & 0xFFu) + (acc >> 20)) : acc;
    return bad == 0;
}

// missing_detector.cpp:290-336 for the '.' bytes of one lane (masks d0..d3 over its 16 bytes at p).
// A '.' marks a missing genotype when it lies in the first ':' piece of its sample and touches the
// piece boundary or a '/' '|' separator on either side.  Neighbour bytes are read back from L1.
__device__ __noinline__ bool md_lane_dots(const uint8_t *p, uint32_t d0, uint32_t d1, uint32_t d2, uint32_t d3, bool strip_cr) {
    uint32_t ds[4] = {d0, d1, d2, d3};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        uint32_t m = ds[j];
        while (m) {
            const int k = (__ffs(m) - 1) >> 3;
            m &= m - 1;
            const uint8_t *q = p + 4 * j + k;
            const uint32_t prev = ldb(q - 1), next = ldb(q + 1);
            const bool a = (prev == '\t') || is_sep(prev);
            const bool b = is_sep(next) || next == ':' || next == '\t' || next == '\n' ||
                           (strip_cr && next == '\r' && ldb(q + 2) == '\n');
            if (!(a || b)) continue;
            if (prev == '\t') return true;
            const uint8_t *r = q - 1;                      // in the first piece <=> a tab comes before any ':'
            for (;;) { const uint32_t c = ldb(r); if (c == '\t') return true; if (c == ':') break; --r; }
        }
    }
    return false;
}

// allele_counter.cpp:267-294 on the first ':' piece of the sample column starting at p: separators
// are skipped, '.' consumes one byte, a digit run is one allele (all zeros = ref, else alt).  The
// reference never advances on any other byte (it hangs); here such a byte is skipped — inputs
// outside [0-9./|] are outside the parity domain (SURVEY.md Appendix B).
__device__ __noinline__ uint2 ac_sample_slow(const uint8_t *p) {
    uint32_t ref = 0, alt = 0;
    for (;;) {
        uint32_t c = ldb(p);
        if (c == ':' || c == '\t' || c == '\n') break;
        if (is_dig(c)) {
            bool nz = false;
            do { nz |= (c != '0'); ++p; c = ldb(p); } while (is_dig(c));
            if (nz) ++alt; else ++ref;
        } else ++p;
    }
    return make_uint2(ref, alt);
}
__device__ __forceinline__ uint32_t dec_len(int v) {       // characters of the decimal form, sign included
    if ((uint32_t)v < 10u) return 1u;                      // allele counts of one sample: almost always
    uint32_t n = (v < 0) ? 1u : 0u;
    uint32_t u = (v < 0) ? (uint32_t)(-v) : (uint32_t)v;
    do { ++n; u /= 10u; } while (u);
    return n;
}
__device__ __forceinline__ uint8_t *put_dec(uint8_t *d, int v) {
    if ((uint32_t)v < 10u) { *d = (uint8_t)('0' + v); return d + 1; }
    if (v < 0) { *d++ = '-'; v = -v; }
    char t[12]; int n = 0; uint32_t u = (uint32_t)v;
    do { t[n++] = (char)('0' + u % 10u); u /= 10u; } while (u);
    while (n) *d++ = (uint8_t)t[--n];
    return d;
}
// flush n staged bytes (shared memory) to dst.  The bytes were staged at the same offset modulo 16 as
// dst (st - (dst & 15) is 16-byte aligned), so the middle goes out as aligned 128-bit loads / stores.
__device__ __forceinline__ void warp_flush_smem(uint8_t *dst, const uint8_t *st, uint32_t n, int lane) {
    const uint32_t head = min(n, (uint32_t)((16 - ((uintptr_t)dst & 15)) & 15));
    if (lane < (int)head) dst[lane] = st[lane];
    const uint32_t nq = (n - head) >> 4;
    uint4 *d16 = reinterpret_cast<uint4 *>(dst + head);
    const uint4 *s16 = reinterpret_cast<const uint4 *>(st + head);
    for (uint32_t i = lane; i < nq; i += 32) d16[i] = s16[i];
    const uint32_t done = head + (nq << 4);
    if (lane < (int)(n - done)) dst[done + lane] = st[done + lane];
}

// The same flush with the 16-byte aligned middle handed to the bulk-copy engine: ONE cp.async.bulk (shared -> global,
// the 1-D TMA path: UBLKCP in SASS) issued by lane 0 instead of a loop of 128-bit stores by all lanes.  The staged bytes
// were written through the generic proxy, so a proxy fence comes first; wait_group.read returns when the engine has read
// the shared memory (the global writes may still be in flight), i.e. when the buffer may be reused.
__device__ __forceinline__ void warp_flush_smem_bulk(uint8_t *dst, const uint8_t *st, uint32_t n, int lane) {
#ifdef VCFX_EMU
    warp_flush_smem(dst, st, n, lane);
#else
    const uint32_t head = min(n, (uint32_t)((16 - ((uintptr_t)dst & 15)) & 15));
    if (lane < (int)head) dst[lane] = st[lane];
    const uint32_t nq = (n - head) >> 4;
    if (lane == 0 && nq) {
        const uint32_t saddr = (uint32_t)__cvta_generic_to_shared(st + head);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" :: "l"(dst + head), "r"(saddr), "r"(nq << 4) : "memory");
        asm volatile("cp.async.bulk.commit_group;" ::: "memory");
        asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
    }
    const uint32_t done = head + (nq << 4);
    if (lane < (int)(n - done)) dst[done + lane] = st[done + lane];
#endif
}

// Tier-1 check of one window (warp-uniform phase and separator): every lane's four rotated words
// must be [0|1, sep, 0|1, tab].  y = x ^ pat is then [a, 0, b, 0] with a, b the allele values.
// Returns false (and changes nothing) when any lane disagrees.
template <int OP>
__device__ __forceinline__ bool t1_eval(uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3, uint32_t la,
                                        uint32_t sh_u, uint32_t pat, uint32_t &accp, uint32_t &hetp, uint32_t &hap) {
    const uint32_t y0 = __funnelshift_rc(w0, w1, sh_u) ^ pat;
    const uint32_t y1 = __funnelshift_rc(w1, w2, sh_u) ^ pat;
    const uint32_t y2 = __funnelshift_rc(w2, w3, sh_u) ^ pat;
    const uint32_t y3 = __funnelshift_rc(w3, la, sh_u) ^ pat;
    const uint32_t bad = (y0 | y1 | y2 | y3) & 0xFFFEFFFEu;
    if (__any_sync(FULL, bad != 0)) return false;
    if (OP == OP_AF) accp += y0 + y1 + y2 + y3;
    else {
        const uint32_t pk = y0 + 2u * y1 + 4u * y2 + 8u * y3;   // a-bits in 0..3, b-bits in 16..19
        const uint32_t ab = pk & 0xFu, bb = (pk >> 16) & 0xFu;
        hetp += __popc(ab ^ bb); hap += __popc(ab & bb);
    }
    return true;
}

template <int OP> struct OutCount { typedef uint32_t type; };
template <> struct OutCount<OP_AC> { typedef unsigned long long type; };

// Tally four verified (or zeroed) y words: y = [a, 0, b, 0], a and b the allele bits of one sample.
template <int OP>
__device__ __forceinline__ void t1_tally(uint32_t y0, uint32_t y1, uint32_t y2, uint32_t y3, uint32_t &accp, uint32_t &hetp, uint32_t &hap) {
    if (OP == OP_AF) accp += y0 + y1 + y2 + y3;
    else {
        const uint32_t pk = y0 + 2u * y1 + 4u * y2 + 8u * y3;   // a-bits in 0..3, b-bits in 16..19
        const uint32_t ab = pk & 0xFu, bb = (pk >> 16) & 0xFu;
        hetp += __popc(ab ^ bb); hap += __popc(ab & bb);
    }
}

// ---------------------------------------------------------------------------------------
// Digit path: the rest of a line whose FORMAT is exactly "GT" once it is off the tier-1 lattice (missing calls,
// haploid calls, mixed separators — the default shape of multi-sample VCFs).  Nothing is assumed about where a
// sample starts; every byte is classified by range with SWAR adds (bit 7 of x + (0x80 - c) is set iff the byte
// is >= c, for bytes < 0x80; the bounds of a word are monotone, so a union of ranges is the XOR of its bounds):
//   allele_freq_calc   B = tab '\n' '/' '|'.  While no two non-B bytes touch (every token is ONE character)
//                      and there is no ':' (everything is in the first piece), parseGenotypeAndCount
//                      (allele_freq_calc.cpp:262-293) counts exactly the digit bytes: total = #[0-9], alt = #[1-9]
//                      ('.' and any other single byte are tokens that count nothing).
//   allele_counter -a  parseGenotypeRaw (allele_counter.cpp:267-294) counts digit RUNS of the first piece: while no
//                      two digits touch and there is no ':', ref = #'0', alt = #[1-9].
// A digit at byte k is counted by the lane that holds byte k + 1 (the byte that proves the token ends there), so a
// token is never split between two windows' verdicts.  Anything else (a multi-character token, a ':', a byte
// >= 0x80, "\r\n" in stdin mode) makes the function return false with nothing kept: the caller then runs its exact
// per-sample path over the same bytes, as if this function had not been called.
// Returns true when the line's '\n' was reached: e = its position, a / b / tabs = this lane's partial counts.
// ---------------------------------------------------------------------------------------
#ifdef VCFX_EMU
__device__ __forceinline__ uint32_t dp4a_u(uint32_t a, uint32_t b, uint32_t c) {
    return c + (a & 0xFFu) * (b & 0xFFu) + ((a >> 8) & 0xFFu) * ((b >> 8) & 0xFFu) + ((a >> 16) & 0xFFu) * ((b >> 16) & 0xFFu) + (a >> 24) * (b >> 24);
}
#else
__device__ __forceinline__ uint32_t dp4a_u(uint32_t a, uint32_t b, uint32_t c) { return __dp4a(a, b, c); }
#endif
constexpr uint32_t M80 = 0x80808080u;
#define VCFX_GE(x, c) ((x) + (0x80808080u - 0x01010101u * (uint32_t)(c)))
// markers moved up by one byte: byte i of the result = byte i - 1 of (prev : w)
__device__ __forceinline__ uint32_t up1(uint32_t prev, uint32_t w) { return __funnelshift_l(prev, w, 8); }

template <int OP> struct DigitClass { uint32_t adjc, D, NZ, SP, TB; };   // adjc: the class whose neighbours must not touch (AF: B, AC: digit)
template <int OP>
__device__ __forceinline__ DigitClass<OP> digit_classes(uint32_t x) {
    DigitClass<OP> c;
    const uint32_t g30 = VCFX_GE(x, 0x30), g31 = VCFX_GE(x, 0x31), g3a = VCFX_GE(x, 0x3A), g3b = VCFX_GE(x, 0x3B);
    const uint32_t g09 = VCFX_GE(x, 0x09), g0a = VCFX_GE(x, 0x0A), g0b = VCFX_GE(x, 0x0B);
    c.D = (g30 ^ g3a) & M80;
    c.NZ = (g31 ^ g3a) & M80;
    c.SP = (g0a ^ g0b ^ g3a ^ g3b) & M80;                       // '\n' ':'
    if (OP == OP_AF) {
        const uint32_t g2f = VCFX_GE(x, 0x2F), g7c = VCFX_GE(x, 0x7C), g7d = VCFX_GE(x, 0x7D);
        c.adjc = (g09 ^ g0b ^ g2f ^ g30 ^ g7c ^ g7d) & M80;     // tab '\n' '/' '|'
        c.TB = 0;
    } else {
        c.adjc = c.D;
        c.TB = (g09 ^ g0a) & M80;
    }
    return c;
}

// bytes of the lane (positions pb .. pb+15) outside [lo, hi) replaced by the filler byte
__device__ __forceinline__ void patch_outside(uint4 &v, uint32_t pb, uint32_t lo, uint32_t hi, uint32_t filler4) {
    const uint32_t keep = lane_keep16(pb, lo, hi);
    const uint32_t k0 = (nib80(keep, 0) >> 7) * 0xFFu, k1 = (nib80(keep, 1) >> 7) * 0xFFu;
    const uint32_t k2 = (nib80(keep, 2) >> 7) * 0xFFu, k3 = (nib80(keep, 3) >> 7) * 0xFFu;
    v.x = (v.x & k0) | (filler4 & ~k0); v.y = (v.y & k1) | (filler4 & ~k1);
    v.z = (v.z & k2) | (filler4 & ~k2); v.w = (v.w & k3) | (filler4 & ~k3);
}

// One window of the digit path: the lane's counts (128 x: the markers are 0x80 per byte) of digits / non-zero digits /
// tabs among bytes pb-1 .. pb+14 (the byte before the lane comes from its left neighbour, lane 0's from `carry_in`),
// and `odd` != 0 when the window holds anything the path does not decide (two touching bytes of the class that must
// stand alone, a '\n', a ':', a byte >= 0x80).  next_carry (valid in lane 0) = the class bits of the window's last byte.
template <int OP>
__device__ __forceinline__ void digits_window(const uint4 cur, const uint32_t carry_in, const int lane,
                                              uint32_t &tB, uint32_t &tA, uint32_t &tT, uint32_t &odd, uint32_t &next_carry) {
    uint32_t pk, adj_first;
    tT = 0;
    {
        const DigitClass<OP> c3 = digit_classes<OP>(cur.w);
        // this lane's last byte, for the lane to its right: bit 31 adjacency class, bit 30 digit, bit 29 non-zero digit
        pk = (c3.adjc & 0x80000000u) | ((c3.D >> 1) & 0x40000000u) | ((c3.NZ >> 2) & 0x20000000u);
        const DigitClass<OP> c2 = digit_classes<OP>(cur.z);
        const uint32_t a3 = up1(c2.adjc, c3.adjc);
        odd = ((OP == OP_AF) ? (~(c3.adjc | a3) & M80) : (c3.adjc & a3)) | c3.SP | c2.SP;
        tB = dp4a_u(c3.D, 0x00010101u, dp4a_u(c2.D, 0x01010101u, 0u));
        tA = dp4a_u(c3.NZ, 0x00010101u, dp4a_u(c2.NZ, 0x01010101u, 0u));
        if (OP == OP_AC) tT = dp4a_u(c3.TB, 0x01010101u, dp4a_u(c2.TB, 0x01010101u, 0u));
        const DigitClass<OP> c1 = digit_classes<OP>(cur.y);
        const uint32_t a2 = up1(c1.adjc, c2.adjc);
        odd |= ((OP == OP_AF) ? (~(c2.adjc | a2) & M80) : (c2.adjc & a2)) | c1.SP;
        tB = dp4a_u(c1.D, 0x01010101u, tB); tA = dp4a_u(c1.NZ, 0x01010101u, tA);
        if (OP == OP_AC) tT = dp4a_u(c1.TB, 0x01010101u, tT);
        const DigitClass<OP> c0 = digit_classes<OP>(cur.x);
        const uint32_t a1 = up1(c0.adjc, c1.adjc);
        odd |= ((OP == OP_AF) ? (~(c1.adjc | a1) & M80) : (c1.adjc & a1)) | c0.SP;
        tB = dp4a_u(c0.D, 0x01010101u, tB); tA = dp4a_u(c0.NZ, 0x01010101u, tA);
        if (OP == OP_AC) tT = dp4a_u(c0.TB, 0x01010101u, tT);
        adj_first = c0.adjc;
    }
    uint32_t pv = __shfl_sync(FULL, pk, (lane + 31) & 31);
    next_carry = pv;
    if (lane == 0) pv = carry_in;
    const uint32_t a0 = up1(pv, adj_first);
    odd |= ((OP == OP_AF) ? (~(adj_first | a0) & M80) : (adj_first & a0)) | ((cur.x | cur.y | cur.z | cur.w) & M80);
    tB += (pv >> 23) & 0x80u;
    tA += (pv >> 22) & 0x80u;
}

template <int OP>
__device__ __forceinline__ bool line_digits(const uint8_t *__restrict__ tin, uint32_t wb, const uint32_t lo, const uint32_t nrel,
                                           const bool strip_cr, uint32_t &out_a, uint32_t &out_b, uint32_t &out_tabs, uint32_t &out_e) {
    const int lane = lane_id();
    // bytes outside the sample region are overwritten with a byte that counts nothing and touches nothing before they
    // are classified: a tab for allele_freq_calc, a blank for allele_counter (whose tabs are counted)
    constexpr uint32_t FILL = (OP == OP_AF) ? 0x09090909u : 0x20202020u;
    uint32_t accA = 0, accB = 0, accT = 0;               // 128 x count
    uint32_t carry = (OP == OP_AF) ? 0x80000000u : 0u;    // lane 0: class bits of the last byte of the window before
    uint4 cur = ld16(tin + wb + 16 * lane);
    uint4 nxt = ld16(tin + wb + WINDOW + 16 * lane);
    uint4 nx2 = ld16(tin + wb + 2 * WINDOW + 16 * lane);
    patch_outside(cur, wb + 16 * lane, lo, ~0u, FILL);    // the first window: nothing before `lo` is a sample
    bool first = true;                                    // (the caller has counted the tabs of this window)
    for (;;) {
        uint32_t tB, tA, tT, odd, nc;
        digits_window<OP>(cur, carry, lane, tB, tA, tT, odd, nc);
        if (__any_sync(FULL, odd != 0)) {
            // the window with the '\n' (or something the path does not decide)
            const uint32_t n0 = eq_bytes(cur.x, C_NL), n1 = eq_bytes(cur.y, C_NL), n2 = eq_bytes(cur.z, C_NL), n3 = eq_bytes(cur.w, C_NL);
            const unsigned ebal = __ballot_sync(FULL, (n0 | n1 | n2 | n3) != 0);
            if (!ebal) return false;
            const int src = __ffs(ebal) - 1;
            int k = first_byte(n0, n1, n2, n3);
            k = __shfl_sync(FULL, k, src);
            const uint32_t e = wb + 16 * src + k;
            uint32_t ee = e;                              // end of the content (a stripped '\r' is not content)
            if (OP == OP_AF && strip_cr && e > lo && ldb(tin + e - 1) == '\r') ee = e - 1;
            patch_outside(cur, wb + 16 * lane, 0u, ee, FILL);
            digits_window<OP>(cur, carry, lane, tB, tA, tT, odd, nc);
            if (__any_sync(FULL, odd != 0)) return false;
            accB += tB; accA += tA; if (OP == OP_AC && !first) accT += tT;
            out_a = accA >> 7; out_b = accB >> 7; out_tabs = accT >> 7; out_e = e;
            return true;
        }
        accB += tB; accA += tA; if (OP == OP_AC && !first) accT += tT;
        if (lane == 0) carry = nc;
        first = false;
        wb += WINDOW; cur = nxt; nxt = nx2; nx2 = ld16(tin + wb + 2 * WINDOW + 16 * lane);
        if (((wb >> 9) & 7u) == 0) {                      // every 8th window: L2 prefetch of the 4 KB that follow
            const uint32_t pf = wb + 10 * WINDOW + 128 * lane;
            if (pf < nrel) prefetch_l2(tin + pf);
        }
    }
}

// Row-record slots are reserved REC_BLOCK at a time: one atomic on the single global counter per 32 rows
// (one per row is the kernel's bottleneck: same-address atomics serialise in L2).  The block's state lives in
// shared memory, only lane 0 touches it; the slots a warp leaves unused are marked invalid when it exits.
__device__ __forceinline__ unsigned long long alloc_slot(unsigned long long *rec_base, unsigned int *rec_used, DevStats *stats) {   // lane 0 only
    unsigned int used = *rec_used;
    if (used == REC_BLOCK) { *rec_base = atomicAdd(&stats->n_recs, (unsigned long long)REC_BLOCK); used = 0; }
    *rec_used = used + 1;
    return *rec_base + used;
}

// what a warp keeps in shared memory (pointers to this warp's entries)
struct WarpShared {
    volatile uint32_t *tp;                 // positions of tabs 1..9 of the current line
    uint8_t *stage0;                       // allele_counter row staging
    uint32_t *u;                           // allele_counter: the bytes all rows of the current line share (see the fast row writer)
    unsigned int *cnt;                     // event counters (CNT_SLOTS)
    unsigned long long *rec_base; unsigned int *rec_used;
    volatile unsigned int *odd, *reg, *tag;   // [WARPS_PER_CTA] arrays (indexed by the warp)
    uint8_t *ring;                         // general kernel: C4_RING bytes of input staged by the bulk-copy engine
    unsigned long long *bars;              //   its C4_STAGES mbarriers
    uint32_t *ring_par;                    //   and their parities (bit s: what stage s is waited on next)
};
// what a warp carries from line to line inside a tile
template <int OP> struct TileState {
    uint32_t ls, nlines;
    typename OutCount<OP>::type out_bytes;  // only allele_counter's per-sample rows can exceed 32 bits (input offsets cannot)
    uint32_t md_prev_end, md_last_end;      // MISSING_DETECT: end of the last rewritten line / of the last line
    bool md_add_nl;
    uint32_t offlattice_lines;              // VAR 1: lines whose first sample window was not on the tier-1 lattice
};

// One window of a line whose FORMAT has several keys (GT first), for the lane that holds its 16 bytes at p: the sample
// that starts in the lane — if one does — decided from its first four bytes.  Returns true when the window holds
// anything this does not decide (then nothing may be added for the window).
//   allele_freq_calc (allele_freq_calc.cpp:262-293): "d sep d" closed by ':' or a tab is two alleles, ". sep ." is none
//   hwe_tester (hwe_tester.cpp:339-378): "d sep d" and no third digit is a call (both alleles <= 1 count), ". sep ." is none
// ---- the ring the bulk-copy engine fills for the skip-ahead loop (north_star stage 3: "TMA bulk loads where record spans are
// long enough to pay off"): C4_STAGES pieces of C4_PIECE bytes per warp; piece k of a run that starts at global offset g0 sits
// at ring offset (k * C4_PIECE) mod C4_RING, so a byte at g0 + x sits at x mod C4_RING; ONE cp.async.bulk (global -> shared,
// UBLKCP) per piece, completion on the piece's mbarrier
// MEASURED (profiles/README.md, round 2): the stand-alone scan gains 27-31 % from this feed, the product's loop nothing (C4 hwe_tester
// 1.928 -> 1.938 ms, allele_freq_calc 1.916 -> 1.887 ms), and the 32 KiB of shared memory per CTA cost the loop's L1 hits 4-5 % even
// with the ring unused — so the ring is compiled in only with -DVCFX_C4_RING=1 (the warp emulator's build does, to keep it tested).
#ifndef VCFX_C4_RING
#define VCFX_C4_RING 0
#endif
constexpr uint32_t C4_PIECE = 1024, C4_STAGES = 4, C4_RING = C4_PIECE * C4_STAGES;
__device__ __forceinline__ void ring_init(unsigned long long *bars, int lane) {
#ifndef VCFX_EMU
    if (lane == 0) {
        const uint32_t b = (uint32_t)__cvta_generic_to_shared(bars);
        for (uint32_t i = 0; i < C4_STAGES; ++i) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"(b + 8u * i));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncwarp();
#endif
}
__device__ __forceinline__ void ring_issue(uint8_t *ring, unsigned long long *bars, const uint8_t *g0, uint32_t k) {   // lane 0 only
    const uint32_t st = k % C4_STAGES;
#ifdef VCFX_EMU
    for (uint32_t i = 0; i < C4_PIECE; ++i) ring[st * C4_PIECE + i] = g0[(size_t)k * C4_PIECE + i];
#else
    const uint32_t bar = (uint32_t)__cvta_generic_to_shared(bars + st), dst = (uint32_t)__cvta_generic_to_shared(ring + st * C4_PIECE);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(bar), "r"(C4_PIECE) : "memory");
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 :: "r"(dst), "l"(g0 + (size_t)k * C4_PIECE), "r"(C4_PIECE), "r"(bar) : "memory");
#endif
}
__device__ __forceinline__ void ring_wait(unsigned long long *bars, uint32_t st, uint32_t parity) {
#ifndef VCFX_EMU
    const uint32_t bar = (uint32_t)__cvta_generic_to_shared(bars + st);
    uint32_t done = 0;
    while (!done)
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }" : "=r"(done) : "r"(bar), "r"(parity) : "memory");
#endif
}

// RING: the four bytes behind the tab come from the ring (x = offset of p from the start of the run) instead of global memory
template <int OP, bool RING = false>
__device__ __forceinline__ bool multikey_window(const uint4 v, const uint8_t *__restrict__ p, uint32_t &da, uint32_t &db, uint32_t &dc,
                                                const uint8_t *ring = nullptr, uint32_t x = 0) {
    // tab and '\n' markers by range: 3 adds and 2 LOP3 per word
    const uint32_t a0 = VCFX_GE(v.x, 0x09), b0 = VCFX_GE(v.x, 0x0A), c0 = VCFX_GE(v.x, 0x0B);
    const uint32_t a1 = VCFX_GE(v.y, 0x09), b1 = VCFX_GE(v.y, 0x0A), c1 = VCFX_GE(v.y, 0x0B);
    const uint32_t a2 = VCFX_GE(v.z, 0x09), b2 = VCFX_GE(v.z, 0x0A), c2 = VCFX_GE(v.z, 0x0B);
    const uint32_t a3 = VCFX_GE(v.w, 0x09), b3 = VCFX_GE(v.w, 0x0A), c3 = VCFX_GE(v.w, 0x0B);
    const uint32_t tm0 = (a0 ^ b0) & M80, tm1 = (a1 ^ b1) & M80, tm2 = (a2 ^ b2) & M80, tm3 = (a3 ^ b3) & M80;
    bool odd = (((b0 ^ c0) | (b1 ^ c1) | (b2 ^ c2) | (b3 ^ c3) | v.x | v.y | v.z | v.w) & M80) != 0;     // '\n' or a high byte
    da = 0; db = 0; dc = 0;
    if (tm0 | tm1 | tm2 | tm3) {
        // one bit per byte of the lane (see the header phase), then the first tab's byte index
        const uint32_t m16 = ((tm0 * 0x00204081u) >> 28) | (((tm1 * 0x00204081u) >> 24) & 0xF0u) |
                             (((tm2 * 0x00204081u) >> 20) & 0xF00u) | (((tm3 * 0x00204081u) >> 16) & 0xF000u);
        if (m16 & (m16 - 1u)) odd = true;            // two sample starts in 16 bytes
        // the four bytes behind the tab: two aligned loads (L1: the bytes were streamed by this warp a moment ago)
        uint32_t q;
        if (RING) {
            const uint32_t xs = x + (uint32_t)__ffs(m16);
            const uint32_t w0 = *reinterpret_cast<const uint32_t *>(ring + ((xs & ~3u) & (C4_RING - 1u)));
            const uint32_t w1 = *reinterpret_cast<const uint32_t *>(ring + (((xs & ~3u) + 4u) & (C4_RING - 1u)));
            q = __funnelshift_r(w0, w1, 8u * (xs & 3u));
        } else {
            const uint8_t *s = p + __ffs(m16);
            const uint32_t *s4 = reinterpret_cast<const uint32_t *>((uintptr_t)s & ~(uintptr_t)3);
            q = __funnelshift_r(__ldg(s4), __ldg(s4 + 1), 8u * (uint32_t)((uintptr_t)s & 3));
        }
        const uint32_t q1 = (q >> 8) & 0xFFu, q3 = q >> 24;
        const bool sep = (q1 == '/') | (q1 == '|');
        const uint32_t dg = q & 0x00FF00FFu;         // bytes 0 and 2
        const bool two_digits = ((dg & 0x00F000F0u) == 0x00300030u) & ((((dg & 0x000F000Fu) + 0x00060006u) & 0x00100010u) == 0u);
        if (OP == OP_AF) {
            const bool end = (q3 == ':') | (q3 == '\t');
            if (sep & end & two_digits) { db = 2; da = (uint32_t)((dg & 0x0000000Fu) != 0u) + (uint32_t)((dg & 0x000F0000u) != 0u); }
            else if (!(sep & end & (dg == 0x002E002Eu))) odd = true;
        } else {
            const bool more = (q3 - 48u) <= 9u;
            if (sep & two_digits & !more) {
                const uint32_t al = dg & 0x000F000Fu;   // the two allele values
                if ((al & 0x000E000Eu) == 0u) { const uint32_t c = (al & 1u) + (al >> 16); da = (c == 0); db = (c == 1); dc = (c == 2); }
            } else if (!(sep & (dg == 0x002E002Eu))) odd = true;
        }
    }
    return odd;
}

// Every line that starts in the tile, from st.ls on.  Two variants of the same text for allele_freq_calc and hwe_tester
// (both inlined into the kernel, so that neither pays for the other's registers):
//   VAR 0  the lattice variant: tier 1 + the exact path.  It stops — returning false with st.ls at the line, nothing
//          of it consumed — at the first line whose first sample window is not tier-1 material
//   VAR 1  the general variant: the same plus the digit path and the skip-ahead loop for FORMATs with several keys;
//          it runs to the end of the tile
// The other operations have one variant (VAR 0, never stops early).
template <int OP, int VAR>
__device__ __forceinline__ bool tile_lines(const KParams &P, const WarpShared ws, const int lane, const bool strip_cr,
                                           const uint32_t tile, const uint64_t a, const uint64_t a0, const uint8_t *__restrict__ tin,
                                           const uint32_t rb, const uint32_t nrel, const uint64_t n, TileState<OP> &st) {
    constexpr bool HAS_VAR = (OP == OP_AF || OP == OP_HWE);
    constexpr int NEED_TABS = (OP == OP_VC) ? 7 : (OP == OP_IX) ? 1 : 9;        // the header phase ends once this many tabs are ranked
    volatile uint32_t *tp = ws.tp;
    const int wid = threadIdx.x >> 5;
    volatile unsigned int *s_odd = ws.odd, *s_reg = ws.reg, *s_tag = ws.tag;
    uint32_t ls = st.ls, nlines = st.nlines;
    typename OutCount<OP>::type out_bytes = st.out_bytes;
    uint32_t md_prev_end = st.md_prev_end, md_last_end = st.md_last_end;
    bool md_add_nl = st.md_add_nl;
#define VCFX_COUNT(slot, v) do { if (lane == 0) atomicAdd(&ws.cnt[slot], (unsigned int)(v)); } while (0)
#define VCFX_SAVE_STATE() do { st.ls = ls; st.nlines = nlines; st.out_bytes = out_bytes; st.md_prev_end = md_prev_end; st.md_last_end = md_last_end; st.md_add_nl = md_add_nl; } while (0)
        // ---- every line that starts in the tile
        while (ls < rb) {
            uint32_t wb = ls & ~15u;
            uint4 cur = ld16(tin + wb + 16 * lane);
            uint4 nxt = ld16(tin + wb + WINDOW + 16 * lane);
            uint4 nx2 = ld16(tin + wb + 2 * WINDOW + 16 * lane);   // two windows ahead: the look-ahead word of
                                                                    // lane 31 comes from nxt, which must have landed
            const uint32_t first = ldb(tin + ls);
            const bool hash = (first == '#');
            int tabs = 0;                      // tabs ranked so far (uniform)
            bool found = false;                // '\n' seen
            uint32_t e = 0;                    // position of the '\n'
            uint32_t ta = 0, tb = 0, tc = 0;   // per-lane tallies (AF: alt,total; HWE: homRef,het,homAlt)
            int gt_index = -1;
            bool do_samples = false;

            // ================= header phase: rank tabs until NEED_TABS are known or the line ends
            uint32_t t0, t1, t2, t3;           // tab masks of the current window (this lane)
            int rank0 = 0;                     // rank inside the line of this lane's first tab
            for (;;) {
                const uint32_t pb = wb + 16 * lane;
                t0 = eq_bytes(cur.x, C_TAB); t1 = eq_bytes(cur.y, C_TAB);
                t2 = eq_bytes(cur.z, C_TAB); t3 = eq_bytes(cur.w, C_TAB);
                uint32_t n0 = eq_bytes(cur.x, C_NL), n1 = eq_bytes(cur.y, C_NL);
                uint32_t n2 = eq_bytes(cur.z, C_NL), n3 = eq_bytes(cur.w, C_NL);
                if (wb < ls) {                 // bytes before the line start (first window only)
                    const uint32_t k = lane_keep16(pb, ls, ~0u);
                    const uint32_t k0 = nib80(k, 0), k1 = nib80(k, 1), k2 = nib80(k, 2), k3 = nib80(k, 3);
                    t0 &= k0; t1 &= k1; t2 &= k2; t3 &= k3; n0 &= k0; n1 &= k1; n2 &= k2; n3 &= k3;
                }
                unsigned ebal = __ballot_sync(FULL, (n0 | n1 | n2 | n3) != 0);
                if (ebal) {
                    int src = __ffs(ebal) - 1;
                    int k = first_byte(n0, n1, n2, n3);
                    k = __shfl_sync(FULL, k, src);
                    e = wb + 16 * src + k; found = true;
                    clip4(t0, t1, t2, t3, pb, 0, e);
                }
                int total = 0;
                if (!hash) {
                    if (OP == OP_VC) {
                        const int cnt = __popc(t0) + __popc(t1) + __popc(t2) + __popc(t3);
                        total = (int)__reduce_add_sync(FULL, (unsigned)cnt);
                    } else {
                        // one bit per byte of the lane: the 0x80 markers of a word gathered into its top nibble
                        // by a multiply (bits 7/15/23/31 times 2^21/2^14/2^7/2^0 land on 28..31, nothing collides)
                        uint32_t m16 = ((t0 * 0x00204081u) >> 28) | (((t1 * 0x00204081u) >> 24) & 0xF0u) |
                                       (((t2 * 0x00204081u) >> 20) & 0xF00u) | (((t3 * 0x00204081u) >> 16) & 0xF000u);
                        const int cnt = __popc(m16);
                        int incl = warp_incl_scan(cnt, lane);
                        total = __shfl_sync(FULL, incl, 31);
                        rank0 = tabs + incl - cnt;
                        // publish the positions of tabs 0..8
                        int rank = rank0;
                        while (m16 && rank < 9) {
                            tp[rank++] = pb + (uint32_t)(__ffs(m16) - 1);
                            m16 &= m16 - 1;
                        }
                    }
                }
                tabs += total;
                if (found || tabs >= NEED_TABS) break;
                wb += WINDOW; cur = nxt; nxt = nx2; nx2 = ld16(tin + wb + 2 * WINDOW + 16 * lane);
            }
            __syncwarp();

            // ================= decisions that need only the header
            if ((OP == OP_AF || OP == OP_HWE) && !hash && tabs >= 9) {
                const uint32_t fs = tp[7] + 1, fe = tp[8];
                if (OP == OP_AF) {
                    if (fe - fs == 2 && ldb(tin + fs) == 'G' && ldb(tin + fs + 1) == 'T') gt_index = 0;
                    else gt_index = gt_index_of(tin + fs, tin + fe);
                    do_samples = gt_index >= 0 && (a0 + ls >= P.valid_from);
                } else {
                    do_samples = (fe - fs >= 2) && ldb(tin + fs) == 'G' && ldb(tin + fs + 1) == 'T';
                    gt_index = 0;
                }
            }

            // ================= sample phase
            if ((OP == OP_AF || OP == OP_HWE) && do_samples) {
                bool first_win = true;             // `cur` is the window in which tab 9 was ranked
                bool digits_tried = false;
                bool prev_ok = false;              // the previous window ended on a verified lattice lane
                // Tier 1 speculation for the whole line: every sample is "a<sep>b" with a, b in {0,1} and the
                // separator of the first sample, hence a tab every 4 bytes at a phase (tau) that is the same
                // in every lane and window.  A window that breaks the pattern anywhere is handed to the exact
                // path below, so the speculation costs nothing in correctness.
                const uint32_t tab8 = tp[8];
                const uint32_t sep0 = ldb(tin + tab8 + 2);
                const bool lat_possible = (gt_index == 0) && (tp[8] - tp[7] == 3);      // FORMAT is exactly "GT"
                const bool t1_on = lat_possible && (sep0 == '|' || sep0 == '/');
                const uint32_t tau = tab8 & 3u;
                const uint32_t sh_u = 8u * (tau + 1u);
                const uint32_t pat = 0x09300030u | (sep0 << 8);
                uint32_t accp = 0;                 // packed sums: bits 0..15 first alleles, 16..31 second alleles
                uint32_t hetp = 0, hap = 0;        // HWE tier-1 tallies
                uint32_t n_real = 0;               // samples tallied by tier 1 (uniform)
                // ---- the window with tab 9, the cheap way.  A rotated word f_k of a lane covers the four bytes
                // after byte 4k + tau of that lane, i.e. one sample behind its leading tab when the lattice holds.
                // Tab 9 itself sits on the lattice (tau = its position mod 4), so in its lane the words from its own
                // on are samples and the earlier ones (and all earlier lanes) are header: whole words are skipped,
                // no byte masks.  If anything else is in this window the exact path below takes it from scratch.
                if (t1_on && !found) {
                    const uint32_t la_ = ldw(tin + wb + 16 * lane + 16);
                    uint32_t y0 = __funnelshift_rc(cur.x, cur.y, sh_u) ^ pat, y1 = __funnelshift_rc(cur.y, cur.z, sh_u) ^ pat;
                    uint32_t y2 = __funnelshift_rc(cur.z, cur.w, sh_u) ^ pat, y3 = __funnelshift_rc(cur.w, la_, sh_u) ^ pat;
                    const uint32_t rel = tab8 - wb, Lb = rel >> 4, kb = (rel >> 2) & 3u;
                    const uint32_t kmin = (uint32_t)lane > Lb ? 0u : ((uint32_t)lane == Lb ? kb : 4u);
                    if (kmin > 0) y0 = 0;
                    if (kmin > 1) y1 = 0;
                    if (kmin > 2) y2 = 0;
                    if (kmin > 3) y3 = 0;
                    if (!__any_sync(FULL, ((y0 | y1 | y2 | y3) & 0xFFFEFFFEu) != 0)) {
                        t1_tally<OP>(y0, y1, y2, y3, accp, hetp, hap);
                        n_real += ((wb + WINDOW - 1 - tab8) >> 2) + 1;           // lattice tabs in [tab 9, end of window)
                        first_win = false; prev_ok = true;
                        wb += WINDOW; cur = nxt; nxt = nx2; nx2 = ld16(tin + wb + 2 * WINDOW + 16 * lane);
                    }
                }
                // ---- not tier-1 material from the first sample window on: the lattice variant hands the line (and the
                // rest of the tile) to the general variant; nothing of the line has been counted yet
                if (HAS_VAR && !found && first_win) {
                    if (VAR == 0) { VCFX_SAVE_STATE(); return false; }
                }
                for (;;) {
                    // ---- steady state for a FORMAT with several keys (GT first): samples are tens of bytes long, so a
                    // lane holds at most one sample start and almost all bytes only have to be searched for tabs
                    // (multikey_window above).  Two windows per vote, two register pairs that alternate: each pair is loaded
                    // again (four windows ahead) right after its own vote by load instructions of its own, so that a wait
                    // for one window is not a wait for the newest load.  The window with the '\n', a lane with two tabs, a
                    // byte >= 0x80 and every genotype that needs more than four bytes leave the loop with nothing added, for
                    // the exact path below.
                    if (VCFX_C4_RING && VAR == 1 && !first_win && !lat_possible && gt_index == 0 && P.c4_bulk) {
                        // the same loop fed by the bulk-copy engine: pieces of two windows, four of them in the ring (the one being
                        // looked at, the next — a sample's four bytes may reach into it — and two on their way)
                        const uint8_t *g0 = tin + wb;
                        uint8_t *ring = ws.ring; unsigned long long *bars = ws.bars;
                        uint32_t par = *ws.ring_par;                  // bit s: the parity stage s completes with next
                        if (lane == 0) for (uint32_t q = 0; q < C4_STAGES; ++q) ring_issue(ring, bars, g0, q);
                        uint32_t k = 0;
                        ring_wait(bars, 0, (par >> 0) & 1u); par ^= 1u;
                        for (;;) {
                            const uint32_t st = k % C4_STAGES, st1 = (k + 1) % C4_STAGES;
                            ring_wait(bars, st1, (par >> st1) & 1u); par ^= 1u << st1;       // the piece behind this one is in as well
                            const uint8_t *rp = ring + st * C4_PIECE + 16 * lane;
                            const uint4 v0 = *reinterpret_cast<const uint4 *>(rp), v1 = *reinterpret_cast<const uint4 *>(rp + WINDOW);
                            uint32_t da0, db0, dc0, da1, db1, dc1;
                            const uint32_t x0 = k * C4_PIECE + 16u * (uint32_t)lane;
                            const bool o0 = multikey_window<OP, true>(v0, nullptr, da0, db0, dc0, ring, x0);
                            const bool o1 = multikey_window<OP, true>(v1, nullptr, da1, db1, dc1, ring, x0 + WINDOW);
                            if (__any_sync(FULL, o0 | o1)) break;
                            ta += da0 + da1; tb += db0 + db1; tc += dc0 + dc1;
                            __syncwarp();                                             // every lane is done with piece k
                            if (lane == 0) {
#ifndef VCFX_EMU
                                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
#endif
                                ring_issue(ring, bars, g0, k + C4_STAGES);
                            }
                            ++k;
                        }
                        // pieces k+2, k+3 are still on their way (k+1 has been waited for): they must have landed before the ring is used again
                        { const uint32_t s2 = (k + 2) % C4_STAGES, s3 = (k + 3) % C4_STAGES;
                          ring_wait(bars, s2, (par >> s2) & 1u); par ^= 1u << s2;
                          ring_wait(bars, s3, (par >> s3) & 1u); par ^= 1u << s3; }
                        // piece k itself was waited for at the top of round k-1 (or before the loop); its flip is already in par
                        *ws.ring_par = par;
                        // back to the three windows the rest of the line loop works with: cur = the first window not added
                        wb += k * C4_PIECE;
                        cur = ld16(tin + wb + 16 * lane); nxt = ld16(tin + wb + WINDOW + 16 * lane); nx2 = ld16(tin + wb + 2 * WINDOW + 16 * lane);
                    }
                    else if (VAR == 1 && !first_win && !lat_possible && gt_index == 0) {
                        uint4 nx3 = ld16(tin + wb + 3 * WINDOW + 16 * lane);
                        int state = 0;                           // which pair met something odd: 1 = (cur, nxt), 2 = (nx2, nx3)
                        const uint8_t *lp = tin + wb + 16 * lane;
                        uint32_t it = 0;
                        for (;;) {
                            {
                                uint32_t da0, db0, dc0, da1, db1, dc1;
                                const bool o0 = multikey_window<OP>(cur, lp, da0, db0, dc0);
                                const bool o1 = multikey_window<OP>(nxt, lp + WINDOW, da1, db1, dc1);
                                if (__any_sync(FULL, o0 | o1)) { state = 1; break; }
                                ta += da0 + da1; tb += db0 + db1; tc += dc0 + dc1;
                                cur = ld16(lp + 4 * WINDOW); nxt = ld16(lp + 5 * WINDOW);
                            }
                            {
                                uint32_t da0, db0, dc0, da1, db1, dc1;
                                const bool o0 = multikey_window<OP>(nx2, lp + 2 * WINDOW, da0, db0, dc0);
                                const bool o1 = multikey_window<OP>(nx3, lp + 3 * WINDOW, da1, db1, dc1);
                                if (__any_sync(FULL, o0 | o1)) { state = 2; break; }
                                ta += da0 + da1; tb += db0 + db1; tc += dc0 + dc1;
                                nx2 = ld16(lp + 6 * WINDOW); nx3 = ld16(lp + 7 * WINDOW);
                            }
                            if ((++it & 1u) == 0) {              // every second iteration (4 KiB): L2 prefetch of the 4 KiB that follow the loads
                                const uint8_t *pf = lp - 16 * lane + 16 * WINDOW + 128 * lane;
                                if ((uint32_t)(pf - tin) < nrel) prefetch_l2(pf);
                            }
                            lp += 4 * WINDOW;
                        }
                        // back to the three windows the rest of the line loop works with: cur = the first window not added
                        wb = (uint32_t)(lp - tin) - 16u * (uint32_t)lane;
                        if (state == 2) { const uint4 t_ = cur; wb += 2 * WINDOW; cur = nx2; nxt = nx3; nx2 = t_; }
                        // (the first window of the pair may be a regular one: the exact path below takes it all the same)
                    }
                    // ---- steady state: rounds of two raw tier-1 windows, one vote per round, two register sets.
                    // A lane reads its 16 bytes plus the word after them (20 contiguous bytes: no shuffles, no
                    // dependence on the neighbour's registers).  Set A is reloaded right after its vote and is not
                    // touched again until set B's round is over, so every load has a full round to land, and a
                    // failed vote leaves the failing windows in registers.  Nothing is XORed per word: every
                    // rotated word f is pat + y (y = the two allele bits), so the wrapping sum of the f's is
                    // N * pat + sum(y) and, for HWE, the wrapping sum of f * f yields sum(a & b) (see the flush).
                    if (t1_on && prev_ok) {
                        const uint32_t ITMAX = 64u;    // iterations (of 2 KiB) per flush: the packed sums stay exact up to 2000 (HWE) / 4000 (AF)
                        uint32_t la_c = 0, la_n = 0;                             // look-ahead words of cur / nxt once the rounds are over
                        for (;;) {
                            const uint8_t *lp = tin + wb + 16 * lane;
                            uint4 nx3 = ld16(lp + 3 * WINDOW);
                            uint32_t la0 = ldw(lp + 16), la1 = ldw(lp + WINDOW + 16);
                            uint32_t la2 = ldw(lp + 2 * WINDOW + 16), la3 = ldw(lp + 3 * WINDOW + 16);
                            const uint32_t pf_need = wb + 12 * WINDOW;
                            const uint32_t pf_iters = nrel > pf_need ? (nrel - pf_need) / (4 * WINDOW) : 0u;
                            uint32_t it = 0, accf = 0, acc2 = 0;
                            int state = 0;                                       // 1: set A's round failed, 2: set B's
#define VCFX_T1_ROUND(X, LX, Y, LY)                                                                              \
                                uint32_t bad, sum, sq = 0;                                                       \
                                {                                                                                \
                                    const uint32_t f0 = __funnelshift_rc(X.x, X.y, sh_u), f1 = __funnelshift_rc(X.y, X.z, sh_u); \
                                    const uint32_t f2 = __funnelshift_rc(X.z, X.w, sh_u), f3 = __funnelshift_rc(X.w, LX, sh_u);  \
                                    const uint32_t g0 = __funnelshift_rc(Y.x, Y.y, sh_u), g1 = __funnelshift_rc(Y.y, Y.z, sh_u); \
                                    const uint32_t g2 = __funnelshift_rc(Y.z, Y.w, sh_u), g3 = __funnelshift_rc(Y.w, LY, sh_u);  \
                                    bad = (f0 ^ pat) | (f1 ^ pat); bad |= f2 ^ pat; bad |= f3 ^ pat;             \
                                    bad |= g0 ^ pat; bad |= g1 ^ pat; bad |= g2 ^ pat; bad |= g3 ^ pat;          \
                                    sum = (f0 + f1 + f2) + (f3 + g0 + g1) + (g2 + g3);                           \
                                    if (OP == OP_HWE) sq = f0 * f0 + f1 * f1 + f2 * f2 + f3 * f3 + g0 * g0 + g1 * g1 + g2 * g2 + g3 * g3; \
                                }
                            for (; it < ITMAX; ++it) {
                                {
                                    VCFX_T1_ROUND(cur, la0, nxt, la1)
                                    if (__any_sync(FULL, (bad & 0xFFFEFFFEu) != 0)) { state = 1; break; }
                                    accf += sum; if (OP == OP_HWE) acc2 += sq;
                                    cur = ld16(lp + 4 * WINDOW); la0 = ldw(lp + 4 * WINDOW + 16);
                                    nxt = ld16(lp + 5 * WINDOW); la1 = ldw(lp + 5 * WINDOW + 16);
                                }
                                {
                                    VCFX_T1_ROUND(nx2, la2, nx3, la3)
                                    if (__any_sync(FULL, (bad & 0xFFFEFFFEu) != 0)) { state = 2; break; }
                                    accf += sum; if (OP == OP_HWE) acc2 += sq;
                                    nx2 = ld16(lp + 6 * WINDOW); la2 = ldw(lp + 6 * WINDOW + 16);
                                    nx3 = ld16(lp + 7 * WINDOW); la3 = ldw(lp + 7 * WINDOW + 16);
                                }
                                if (it < pf_iters) {          // L2 prefetch 6 KB ahead, 2 KB per iteration
                                    prefetch_l2(lp + 12 * WINDOW); prefetch_l2(lp + 13 * WINDOW);
                                    prefetch_l2(lp + 14 * WINDOW); prefetch_l2(lp + 15 * WINDOW);
#ifdef VCFX_PF1
                                    prefetch_l1(lp + 8 * WINDOW); prefetch_l1(lp + 9 * WINDOW);
                                    prefetch_l1(lp + 10 * WINDOW); prefetch_l1(lp + 11 * WINDOW);
#endif
                                }
                                lp += 4 * WINDOW;
                            }
#undef VCFX_T1_ROUND
                            // flush: N rotated words went into the sums
                            const uint32_t rounds = 2u * it + (state == 2 ? 1u : 0u);
                            const uint32_t N = 8u * rounds;
                            const uint32_t ys = accf - N * pat;                   // sum(a) in bits 0..15, sum(b) in 16..31
                            const uint32_t sa = ys & 0xFFFFu, sb = ys >> 16;
                            if (OP == OP_AF) ta += sa + sb;
                            else {
                                // f * f = pat^2 + 2 pat y + y^2 and y^2 = a + 2^17 (a & b)   (all mod 2^32)
                                const uint32_t y2 = acc2 - N * (pat * pat) - 2u * pat * ys;
                                const uint32_t sab = (y2 - sa) >> 17;
                                hetp += sa + sb - 2u * sab; hap += sab;
                            }
                            n_real += 256u * rounds; wb += 2 * WINDOW * rounds;
                            if (state == 2) { const uint4 t_ = cur; cur = nx2; nxt = nx3; nx2 = t_; la_c = la2; la_n = la3; }   // B failed: A already holds the windows after it
                            else { la_c = la0; la_n = la1; }
                            if (state != 0) break;                               // state 0: only the flush limit was reached
                        }
                        // ---- the round that failed usually holds the line's '\n'.  Its windows again, one by one, with
                        // the y words: the first word that is off, in the first lane that has one, must be a sample
                        // closed by '\n' instead of a tab (y = [a, 0, b, '\n' ^ '\t']); everything before it is tallied
                        // and the line is finished.  Anything else goes to the exact path below.
                        bool finished = false;
#pragma unroll 1
                        for (int k = 0; k < 2; ++k) {
                            uint32_t y0 = __funnelshift_rc(cur.x, cur.y, sh_u) ^ pat, y1 = __funnelshift_rc(cur.y, cur.z, sh_u) ^ pat;
                            uint32_t y2 = __funnelshift_rc(cur.z, cur.w, sh_u) ^ pat, y3 = __funnelshift_rc(cur.w, la_c, sh_u) ^ pat;
                            const uint32_t b0 = y0 & 0xFFFEFFFEu, b1 = y1 & 0xFFFEFFFEu, b2 = y2 & 0xFFFEFFFEu, b3 = y3 & 0xFFFEFFFEu;
                            const unsigned fb = __ballot_sync(FULL, (b0 | b1 | b2 | b3) != 0);
                            if (fb == 0) {
                                t1_tally<OP>(y0, y1, y2, y3, accp, hetp, hap);
                                n_real += 128; wb += WINDOW;
                                cur = nxt; nxt = nx2; nx2 = ld16(tin + wb + 2 * WINDOW + 16 * lane); la_c = la_n;
                                continue;
                            }
                            const int Lf = __ffs(fb) - 1;
                            const uint32_t kf_l = b0 ? 0u : b1 ? 1u : b2 ? 2u : 3u;
                            const uint32_t yf_l = b0 ? y0 : b1 ? y1 : b2 ? y2 : y3;
                            const uint32_t kf = __shfl_sync(FULL, kf_l, Lf), yf = __shfl_sync(FULL, yf_l, Lf);
                            if (((yf ^ 0x03000000u) & 0xFFFEFFFEu) == 0) {
                                const uint32_t keep = lane < Lf ? 4u : (lane == Lf ? kf + 1u : 0u);   // words of this lane that count
                                y0 = keep > 0 ? (y0 & 0x00010001u) : 0u;
                                y1 = keep > 1 ? (y1 & 0x00010001u) : 0u;
                                y2 = keep > 2 ? (y2 & 0x00010001u) : 0u;
                                y3 = keep > 3 ? (y3 & 0x00010001u) : 0u;
                                t1_tally<OP>(y0, y1, y2, y3, accp, hetp, hap);
                                e = wb + 16u * (uint32_t)Lf + 4u * kf + tau + 4u; found = true; finished = true;
                                n_real += (e - wb - tau) >> 2;                  // lattice tabs in [wb, e)
                            }
                            break;
                        }
                        if (OP == OP_AF) { ta += (accp & 0xFFFFu) + (accp >> 16); accp = 0; }
                        if (finished) break;
                    }
                    // ---- off the lattice.  FORMAT "GT": the digit path takes the rest of the line (once per line; when it
                    // declines, nothing of it is kept and the exact path below starts at this very window).  It may only
                    // start where the bytes before are accounted for: at tab 9, or behind windows verified on the line's
                    // lattice, whose last sample ends with the tab at wb + tau.
                    if (VAR == 1 && OP == OP_AF && lat_possible && !digits_tried && !found && (first_win || prev_ok)) {
                        digits_tried = true;
                        uint32_t da = 0, db = 0, dt = 0, de = 0;
                        if (line_digits<OP_AF>(tin, wb, first_win ? tab8 + 1u : wb + tau + 1u, nrel, strip_cr, da, db, dt, de)) {
                            ta += da; tb += db; e = de; found = true;
                            break;
                        }
                        // (declined: the windows are loaded again rather than kept in registers across the call)
                        cur = ld16(tin + wb + 16 * lane); nxt = ld16(tin + wb + WINDOW + 16 * lane); nx2 = ld16(tin + wb + 2 * WINDOW + 16 * lane);
                    }
                    // ---- this window needs a closer look
                    const uint32_t pb = wb + 16 * lane;
                    uint32_t la = __shfl_down_sync(FULL, cur.x, 1);
                    const uint32_t nx0 = __shfl_sync(FULL, nxt.x, 0);
                    if (lane == 31) la = nx0;
                    bool done = false, nl_done = false;
                    if (!done && t1_on && (first_win || prev_ok)) {
                        // Perhaps only the two ends of the sample region are in the way: the header up to tab 9
                        // (first window) and everything from the '\n' on (last window).  Overwrite those bytes
                        // with filler and try again; the filler samples are not counted.  (Past the first window
                        // this needs prev_ok: lane 0's bytes before its first tab are vouched for by the window before.)
                        if (!first_win) {
                            const uint32_t n0 = eq_bytes(cur.x, C_NL), n1 = eq_bytes(cur.y, C_NL);
                            const uint32_t n2 = eq_bytes(cur.z, C_NL), n3 = eq_bytes(cur.w, C_NL);
                            const unsigned ebal = __ballot_sync(FULL, (n0 | n1 | n2 | n3) != 0);
                            nl_done = true;
                            if (ebal) {
                                const int src = __ffs(ebal) - 1;
                                int k = first_byte(n0, n1, n2, n3);
                                k = __shfl_sync(FULL, k, src);
                                e = wb + 16 * src + k; found = true;
                            }
                        }
                        // the '\n' must sit where the lattice expects a tab, or the filler would complete a
                        // truncated last sample ("1\n" would read "1|0")
                        if ((first_win || found) && (!found || ((e - tau) & 3u) == 0)) {
                            const uint32_t lo = first_win ? tab8 : 0u, hi = found ? e : ~0u;
                            const uint32_t kk = lane_keep16(pb, lo, hi);
                            const uint32_t k0 = (nib80(kk, 0) >> 7) * 0xFFu, k1 = (nib80(kk, 1) >> 7) * 0xFFu;
                            const uint32_t k2 = (nib80(kk, 2) >> 7) * 0xFFu, k3 = (nib80(kk, 3) >> 7) * 0xFFu;
                            const uint32_t k4 = (range_mask(pb + 16, lo, hi) >> 7) * 0xFFu;
                            // filler: the bytes "\t0<sep>0" rotated so the tab sits on byte tau of every word — a
                            // well-formed 0/0 sample that adds nothing to the alt / het / homAlt sums
                            const uint32_t fill0 = 0x30003009u | (sep0 << 16);
                            const uint32_t fill = __funnelshift_l(fill0, fill0, 8u * tau);
                            done = t1_eval<OP>((cur.x & k0) | (fill & ~k0), (cur.y & k1) | (fill & ~k1),
                                               (cur.z & k2) | (fill & ~k2), (cur.w & k3) | (fill & ~k3),
                                               (la & k4) | (fill & ~k4), sh_u, pat, accp, hetp, hap);
                            if (done) {
                                // real samples of this window: leading tabs at positions = tau (mod 4) in [A, B)
                                const int A = (int)max(lo, wb), B = (int)min(hi, wb + WINDOW);
                                const int t = (int)tau;
                                n_real += (uint32_t)(max(0, (B + 3 - t) >> 2) - max(0, (A + 3 - t) >> 2));
                            }
                        }
                    }
                    unsigned gbal = FULL;                       // lanes that passed a lattice check
                    if (!done) {
                        // exact path for this window
                        uint32_t packed = 0;
                        // samples of a FORMAT with more keys carry ':' pieces: no lattice there, do not look for one
                        uint32_t sh_lane = 0;
                        // A line that keeps leaving the lattice (missing / haploid calls every few samples: two
                        // windows in a row came here) stops trying: every sample is parsed from its leading tab,
                        // until eight windows in a row held nothing but "digit sep digit".
                        // (the two counters live in shared memory — registers are short — and belong to the line
                        // whose start is in s_tag: lines that never come here never touch them)
                        if (s_tag[wid] != ls + 1u) { s_tag[wid] = ls + 1u; s_odd[wid] = 0; s_reg[wid] = 0; }
                        const bool qm = lat_possible && !first_win && s_odd[wid] >= 2;
                        uint32_t irr = 0;
                        const bool lat = lat_possible && !qm && lane_lattice<OP>(cur.x, cur.y, cur.z, cur.w, la, packed, sh_lane);
                        // Tier 1 never looks at a lane's bytes up to its first lattice tab: they must have been
                        // verified by the lane before it AT THE SAME PHASE.  After a haploid or missing call the
                        // phase of the samples shifts, so the last lane only vouches for the next window when its
                        // own phase is the line's tier-1 phase.
                        gbal = lat_possible ? __ballot_sync(FULL, lat && sh_lane == sh_u) : 0u;
                        uint32_t m0, m1, m2, m3;
                        const uint32_t n0 = eq_bytes(cur.x, C_NL);
                        m0 = eq_bytes(cur.x, C_TAB); m1 = eq_bytes(cur.y, C_TAB);
                        m2 = eq_bytes(cur.z, C_TAB); m3 = eq_bytes(cur.w, C_TAB);
                        // (the header phase's masks are not kept alive for this: registers are short)
                        if (first_win) clip4(m0, m1, m2, m3, pb, tab8, found ? e : ~0u);   // sample tabs only: tab 9 .. '\n'
                        else {
                            if (!nl_done) {
                                const uint32_t n1 = eq_bytes(cur.y, C_NL), n2 = eq_bytes(cur.z, C_NL), n3 = eq_bytes(cur.w, C_NL);
                                const unsigned ebal = __ballot_sync(FULL, (n0 | n1 | n2 | n3) != 0);
                                if (ebal) {
                                    const int src = __ffs(ebal) - 1;
                                    int k = first_byte(n0, n1, n2, n3);
                                    k = __shfl_sync(FULL, k, src);
                                    e = wb + 16 * src + k; found = true;
                                }
                            }
                            if (found) {
                                clip4(m0, m1, m2, m3, pb, 0, e);
                            }
                        }
                        // a lattice lane may be used when its bytes before the first tab are vouched for
                        // (previous lane lattice, or no '\n' in word 0) and all its tabs are sample tabs
                        bool pg = false;
                        if (lat_possible) { pg = __shfl_up_sync(FULL, (int)lat, 1) != 0; if (lane == 0) pg = prev_ok; }
                        const bool use_lat = lat && (pg || n0 == 0) && !(first_win && tp[7] >= pb);   // no header tab in the lane
                        if (use_lat) {
                            if (!found || pb < e) {          // a vouched lattice lane holds no '\n'
                                if (OP == OP_AF) { ta += packed; tb += 8; }
                                else {
                                    const uint32_t het = (packed >> 8) & 0xFF, ha = packed >> 16;
                                    ta += (packed & 0xFF) - het - ha; tb += het; tc += ha;
                                }
                            }
                        } else {
                            if (m0 | m1 | m2 | m3) {
                                bool handled = false;
                                if (__popc(m0) + __popc(m1) + __popc(m2) + __popc(m3) == 1 && gt_index == 0) {
                                    // one sample starts in this lane (the usual case when FORMAT has several
                                    // keys): classify its first four bytes right here
                                    const int B = first_byte(m0, m1, m2, m3);
                                    const uint32_t lo_ = B < 4 ? cur.x : B < 8 ? cur.y : B < 12 ? cur.z : cur.w;
                                    const uint32_t hi_ = B < 4 ? cur.y : B < 8 ? cur.z : B < 12 ? cur.w : la;
                                    const uint32_t q = __funnelshift_rc(lo_, hi_, 8u * (uint32_t)((B & 3) + 1));
                                    const uint32_t b0 = q & 0xFF, b1 = (q >> 8) & 0xFF, b2 = (q >> 16) & 0xFF, b3 = q >> 24;
                                    if (OP == OP_AF) {
                                        const bool t3 = (b3 == '\t' || b3 == ':' || b3 == '\n');
                                        if (is_dig(b0) && is_sep(b1) && is_dig(b2) && t3) {
                                            tb += 2; ta += (uint32_t)(b0 != '0') + (uint32_t)(b2 != '0'); handled = true;
                                        } else if (b0 == '.' && is_sep(b1) && b2 == '.' && t3) { handled = true; irr = 1; }
                                    } else {
                                        if (is_dig(b0) && is_sep(b1) && is_dig(b2) && !is_dig(b3)) {
                                            if (b0 <= '1' && b2 <= '1') { const uint32_t c = (b0 - '0') + (b2 - '0'); ta += (c == 0); tb += (c == 1); tc += (c == 2); }
                                            handled = true;
                                        } else if (b0 == '.') { handled = true; irr = 1; }
                                    }
                                }
                                if (!handled) {
                                    const uint4 r = lane_samples_generic<OP>(cur.x, cur.y, cur.z, cur.w, la, m0, m1, m2, m3,
                                                                             tin + pb, strip_cr, gt_index);
                                    ta += r.x; tb += r.y; tc += r.z; irr = r.w;
                                }
                            }
                        }
                        if (qm) {
                            const unsigned reg = __any_sync(FULL, irr != 0) ? 0u : s_reg[wid] + 1u;
                            s_reg[wid] = reg;
                            if (reg >= 8) { s_reg[wid] = 0; s_odd[wid] = 0; done = true; }   // (done only resets the run below)
                        }
                    }
                    if (found) break;
                    s_odd[wid] = done ? 0u : s_odd[wid] + 1u;
                    prev_ok = (gbal >> 31) != 0;
                    first_win = false;
                    wb += WINDOW; cur = nxt; nxt = nx2; nx2 = ld16(tin + wb + 2 * WINDOW + 16 * lane);
                }
                // fold the tier-1 tallies in (n_real is uniform: lane 0 carries it)
                if (OP == OP_AF) { ta += (accp & 0xFFFFu) + (accp >> 16); if (lane == 0) tb += 2u * n_real; }
                else { ta -= hetp + hap; if (lane == 0) ta += n_real; tb += hetp; tc += hap; }
            }
            // ================= ALLELE_COUNT: (ref, alt) of every sample column into the warp's scratch
            const bool ac_sizing_only = (OP == OP_AC) && P.ac_spec && P.ac_pass == 0;   // no genotype is looked at
            if (OP == OP_AC && !hash && tabs >= 9 && !ac_sizing_only) {
                uint2 *scr = P.col_scratch + (size_t)(blockIdx.x * WARPS_PER_CTA + wid) * P.max_col;
                bool firstw = true;
                // -a over all the samples, FORMAT "GT": the digit path sums the whole line (every sample column must be
                // a selected one; when it declines, the loop below does the line)
                bool summed = false;
                if (P.ac_fmt == AC_AGG && P.ac_ident && !found && tp[8] - tp[7] == 3 && ldb(tin + tp[7] + 1) == 'G' && ldb(tin + tp[7] + 2) == 'T') {
                    uint32_t da = 0, db = 0, dt = 0, de = 0;
                    if (line_digits<OP_AC>(tin, wb, tp[8] + 1u, nrel, false, da, db, dt, de) &&
                        (uint32_t)__reduce_add_sync(FULL, dt) + (uint32_t)tabs <= 8u + P.n_sel) {
                        ta = db - da; tb = da; tabs += (int)__reduce_add_sync(FULL, dt); e = de; found = true; summed = true;
                    }
                }
                if (!summed)
                for (;;) {
                    const uint32_t pb = wb + 16 * lane;
                    uint32_t m0, m1, m2, m3;
                    int r0;                                  // rank in the line of this lane's first tab
                    if (firstw) { m0 = t0; m1 = t1; m2 = t2; m3 = t3; r0 = rank0; }
                    else {
                        m0 = eq_bytes(cur.x, C_TAB); m1 = eq_bytes(cur.y, C_TAB);
                        m2 = eq_bytes(cur.z, C_TAB); m3 = eq_bytes(cur.w, C_TAB);
                        const uint32_t n0 = eq_bytes(cur.x, C_NL), n1 = eq_bytes(cur.y, C_NL);
                        const uint32_t n2 = eq_bytes(cur.z, C_NL), n3 = eq_bytes(cur.w, C_NL);
                        const unsigned ebal = __ballot_sync(FULL, (n0 | n1 | n2 | n3) != 0);
                        if (ebal) {
                            const int src = __ffs(ebal) - 1;
                            int k = first_byte(n0, n1, n2, n3);
                            k = __shfl_sync(FULL, k, src);
                            e = wb + 16 * src + k; found = true;
                            clip4(m0, m1, m2, m3, pb, 0, e);
                        }
                        const int cnt = __popc(m0) + __popc(m1) + __popc(m2) + __popc(m3);
                        const int incl = warp_incl_scan(cnt, lane);
                        r0 = tabs + incl - cnt;
                        tabs += __shfl_sync(FULL, incl, 31);
                    }
                    uint32_t la = __shfl_down_sync(FULL, cur.x, 1);
                    const uint32_t nx0 = __shfl_sync(FULL, nxt.x, 0);
                    if (lane == 31) la = nx0;
                    {
                        const uint32_t ws[5] = {cur.x, cur.y, cur.z, cur.w, la};
                        const uint32_t ms[4] = {m0, m1, m2, m3};
                        int r = r0;
                        // the quick shapes of all the tabs of a word at once (see lane_samples_generic); a tab
                        // then only picks its bits
                        WClass lo = classify_word<OP_AC>(ws[0]);
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            const WClass hi = classify_word<OP_AC>(ws[j + 1]);
                            uint32_t m = ms[j];
                            if (m) {
                                const bool agg_fast = (P.ac_fmt == AC_AGG) && P.ac_ident;   // totals only: ta = ref, tb = alt
                                const uint32_t tokl = lo.D | lo.P, tokh = hi.D | hi.P;
                                const uint32_t t1 = down(tokl, tokh, 1), t3 = down(tokl, tokh, 3), s2 = down(lo.S, hi.S, 2);
                                const uint32_t e1 = down(lo.E, hi.E, 1), e2 = down(lo.E, hi.E, 2), e4 = hi.E;
                                const uint32_t d1 = down(lo.D, hi.D, 1), d3 = down(lo.D, hi.D, 3);
                                const uint32_t z1 = down(lo.Z, hi.Z, 1), z3 = down(lo.Z, hi.Z, 3);
                                const uint32_t C = m & t1 & s2 & t3 & e4, any = (m & t1 & e2) | C, quick = (m & e1) | any;
                                const uint32_t R1 = any & z1, R3 = C & z3, A1 = any & d1 & ~z1, A3 = C & d3 & ~z3;
                                const int nm = __popc(m);
                                if (agg_fast && r >= 8 && (uint32_t)(r + nm) <= 8u + P.n_sel) {
                                    // every tab of this word leads a selected column: add the quick ones by count
                                    ta += __popc(R1) + __popc(R3); tb += __popc(A1) + __popc(A3);
                                    uint32_t rest = m & ~quick;
                                    while (rest) {
                                        const int k = (__ffs(rest) - 1) >> 3;
                                        rest &= rest - 1;
                                        const uint2 v = ac_sample_slow(tin + pb + 4 * j + k + 1);
                                        ta += v.x; tb += v.y;
                                    }
                                    r += nm; m = 0;
                                }
                                while (m) {
                                    const uint32_t bit = m & (0u - m);
                                    const int k = (__ffs(m) - 1) >> 3;
                                    m &= m - 1;
                                    if (r >= 8 && (uint32_t)(r - 8) < P.max_col) {
                                        uint2 v;
                                        if (quick & bit) v = make_uint2(((R1 & bit) ? 1u : 0u) + ((R3 & bit) ? 1u : 0u),
                                                                        ((A1 & bit) ? 1u : 0u) + ((A3 & bit) ? 1u : 0u));
                                        else v = ac_sample_slow(tin + pb + 4 * j + k + 1);
                                        if (agg_fast) { if ((uint32_t)(r - 8) < P.n_sel) { ta += v.x; tb += v.y; } }
                                        else scr[r - 8] = v;
                                    }
                                    ++r;
                                }
                            }
                            lo = hi;
                        }
                    }
                    if (found) break;
                    firstw = false;
                    wb += WINDOW; cur = nxt; nxt = nx2; nx2 = ld16(tin + wb + 2 * WINDOW + 16 * lane);
                }
                __syncwarp();
            }
            // ================= INBREEDING: the genotype code of every sample column, one byte each, next to the line's own offset
            uint32_t ib_alt = 0, ib_good = 0; bool ib_line = false;
            if (OP == OP_IB && !hash && tabs >= 9 && (a0 + ls >= P.valid_from)) {
                // ALT without a comma (:549-553 / :724); the file mode wants it non-empty too
                int ok = 0;
                if (lane == 0) {
                    const uint32_t as = tp[3] + 1, ae = tp[4];
                    ok = (P.mode == MODE_FILE) ? (ae > as) : 1;
                    for (uint32_t q = as; q < ae && ok; ++q) if (ldb(tin + q) == ',') ok = 0;
                }
                ib_line = __shfl_sync(FULL, ok, 0) != 0;
            }
            int ds_gi = -1;                    // dosage_calculator: index of the GT key, found once per line
            if (OP == OP_DS && !hash && tabs >= 9) {
                ds_gi = gt_index_of(tin + tp[7] + 1, tin + tp[8]);       // :316 / :526 findGTIndexRaw on FORMAT
                ib_line = ds_gi >= 0;
            }
            if ((OP == OP_IB || OP == OP_DS) && ib_line) {
                // (the codes of a line start within three bytes of the line's own offset, such that a lane's four codes of a
                // lattice window — see below — land on a 32-bit boundary; the record says where)
                const uint32_t first = tp[8] + 1u, tq = tp[8] & 3u;          // tq: where in a 32-bit word the tabs of a lattice line sit
                uint8_t *codes = P.ib_codes + (((a0 + ls) & ~3ULL) + ((((first + 3u) >> 2) - 1u) & 3u));
                bool firstw = true, lat = true;
                for (;;) {
                    const uint32_t pb = wb + 16 * lane;
                    uint32_t la = __shfl_down_sync(FULL, cur.x, 1);
                    const uint32_t nx0 = __shfl_sync(FULL, nxt.x, 0);
                    if (lane == 31) la = nx0;
                    // ---- lattice window: no line end in sight and every sample so far (and here) is three bytes and a tab, at the
                    // line's phase: a 32-bit word per sample, four codes per lane in one store, no ranking of tabs
                    if (!firstw && lat && (OP == OP_IB || ds_gi == 0)) {
                        const uint32_t nl_any = eq_bytes(cur.x, C_NL) | eq_bytes(cur.y, C_NL) | eq_bytes(cur.z, C_NL) | eq_bytes(cur.w, C_NL);
                        if (!__any_sync(FULL, nl_any != 0)) {
                            // like the tab-by-tab path, a window owns the samples whose leading tab lies in it: bytes tq of every word
                            const uint32_t sh8 = 8u * (tq + 1u);
                            const uint32_t u0 = __funnelshift_rc(cur.x, cur.y, sh8), u1 = __funnelshift_rc(cur.y, cur.z, sh8);
                            const uint32_t u2 = __funnelshift_rc(cur.z, cur.w, sh8), u3 = __funnelshift_rc(cur.w, la, sh8);
                            const uint32_t uu[4] = {u0, u1, u2, u3};
                            uint32_t bad = 0, pk = 0;
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const uint32_t u = uu[j];
                                bad |= (eq_bytes(u, C_TAB) ^ 0x80000000u) | eq_bytes(u, C_NL);
                                const uint32_t b1 = (u >> 8) & 0xFFu;
                                if (OP == OP_IB) {
                                    const bool quick = ((u & 0x00FE00FEu) == 0x00300030u) && (b1 == '/' || b1 == '|');
                                    pk |= (quick ? ((u & 1u) + ((u >> 16) & 1u)) : IB_NONE) << (8 * j);
                                } else {
                                    // dosage: digit, separator, digit is the only three-byte GT with two alleles (a ':' in it cuts GT short)
                                    const uint32_t d0 = (u & 0xFFu) - '0', d2 = ((u >> 16) & 0xFFu) - '0';
                                    const bool quick = d0 <= 9u && d2 <= 9u && (b1 == '/' || b1 == '|');
                                    pk |= (quick ? ((d0 ? 1u : 0u) + (d2 ? 1u : 0u)) : IB_NONE) << (8 * j);
                                }
                            }
                            // the sample behind the window's first tab is number j0 of the line: by the tabs counted so far and by position
                            const int j0 = tabs - 8;
                            bool okl = bad == 0 && j0 == (int)((wb + tq + 1u - first) >> 2) && (OP == OP_DS || (uint32_t)(j0 + 4 * lane + 4) <= P.n_sel);
                            if (lane == 0) okl = okl && ((eq_bytes(cur.x, C_TAB) & (0xFFFFFFFFu >> (24u - 8u * tq))) == (0x80u << (8u * tq)));
                            if (__all_sync(FULL, okl)) {
                                *reinterpret_cast<uint32_t *>(codes + j0 + 4 * lane) = pk;
                                const uint32_t nn = (uint32_t)__popc(eq_bytes(pk, IB_NONE * 0x01010101u));
                                if (OP == OP_IB) { ib_good += 4u - nn; ib_alt += dp4a_u(pk, 0x01010101u, 0u) - 3u * nn; }
                                else ib_alt += nn;                   // dosage_calculator: the number of "NA"s
                                tabs += 128;
                                wb += WINDOW; cur = nxt; nxt = nx2; nx2 = ld16(tin + wb + 2 * WINDOW + 16 * lane);
                                if (((wb >> 9) & 7u) == 0) {
                                    const uint32_t pf = wb + 8 * WINDOW + 128 * lane;
                                    if (pf < nrel) prefetch_l2(tin + pf);
                                }
                                continue;
                            }
                            lat = false;
                        }
                    }
                    uint32_t m0, m1, m2, m3;
                    int r0;                                  // rank in the line of this lane's first tab
                    if (firstw) { m0 = t0; m1 = t1; m2 = t2; m3 = t3; r0 = rank0; }
                    else {
                        m0 = eq_bytes(cur.x, C_TAB); m1 = eq_bytes(cur.y, C_TAB);
                        m2 = eq_bytes(cur.z, C_TAB); m3 = eq_bytes(cur.w, C_TAB);
                        const uint32_t n0 = eq_bytes(cur.x, C_NL), n1 = eq_bytes(cur.y, C_NL);
                        const uint32_t n2 = eq_bytes(cur.z, C_NL), n3 = eq_bytes(cur.w, C_NL);
                        const unsigned ebal = __ballot_sync(FULL, (n0 | n1 | n2 | n3) != 0);
                        if (ebal) {
                            const int src = __ffs(ebal) - 1;
                            int k = first_byte(n0, n1, n2, n3);
                            k = __shfl_sync(FULL, k, src);
                            e = wb + 16 * src + k; found = true;
                            clip4(m0, m1, m2, m3, pb, 0, e);
                        }
                        const int cnt = __popc(m0) + __popc(m1) + __popc(m2) + __popc(m3);
                        const int incl = warp_incl_scan(cnt, lane);
                        r0 = tabs + incl - cnt;
                        tabs += __shfl_sync(FULL, incl, 31);
                    }
                    {
                        const uint32_t wsd[5] = {cur.x, cur.y, cur.z, cur.w, la};
                        const uint32_t ms[4] = {m0, m1, m2, m3};
                        int r = r0;
#pragma unroll
                        for (int j = 0; j < 4; ++j) {
                            uint32_t m = ms[j];
                            while (m) {
                                const int k = (__ffs(m) - 1) >> 3;
                                m &= m - 1;
                                if (r >= 8 && (OP == OP_DS || (uint32_t)(r - 8) < P.n_sel)) {
                                    const uint32_t q = __funnelshift_rc(wsd[j], wsd[j + 1], 8u * (uint32_t)(k + 1));
                                    const uint32_t b1 = (q >> 8) & 0xFFu, b3 = q >> 24;
                                    uint32_t code;
                                    if (OP == OP_IB) {
                                        // the four bytes behind the tab: [01] [/|] [01] and no further digit is the whole story
                                        if ((q & 0x00FE00FEu) == 0x00300030u && (b1 == '/' || b1 == '|') && (b3 - '0') > 9u) code = (q & 1u) + ((q >> 16) & 1u);
                                        else code = ib_sample_code(tin + pb + 4 * j + k + 1);
                                        if (code < IB_NONE) { ib_alt += code; ++ib_good; }
                                    } else {
                                        // digit, separator, digit and the end of the GT (GT the first key)
                                        const uint32_t d0 = (q & 0xFFu) - '0', d2 = ((q >> 16) & 0xFFu) - '0';
                                        if (ds_gi == 0 && d0 <= 9u && d2 <= 9u && (b1 == '/' || b1 == '|') && (b3 == '\t' || b3 == ':' || b3 == '\n'))
                                            code = (d0 ? 1u : 0u) + (d2 ? 1u : 0u);
                                        else code = ds_sample_code(tin + pb + 4 * j + k + 1, P.mode == MODE_FILE, ds_gi);
                                        if (code == IB_NONE) ++ib_alt;
                                    }
                                    codes[r - 8] = (uint8_t)code;
                                }
                                ++r;
                            }
                        }
                    }
                    if (found) break;
                    firstw = false;
                    wb += WINDOW; cur = nxt; nxt = nx2; nx2 = ld16(tin + wb + 2 * WINDOW + 16 * lane);
                    if (((wb >> 9) & 7u) == 0) {          // every 8th window: L2 prefetch of the 4 KB that follow
                        const uint32_t pf = wb + 8 * WINDOW + 128 * lane;
                        if (pf < nrel) prefetch_l2(tin + pf);
                    }
                }
            }
            // ================= MISSING_DETECT: look for a missing genotype in the sample columns
            bool md_flag = false, md_any = false;
            if (OP == OP_MD && !hash && tabs >= 9) {
                const uint32_t lo = tp[8] + 1;
                bool firstw = true;
                for (;;) {
                    const uint32_t pb = wb + 16 * lane;
                    if (!firstw) {
                        const uint32_t n0 = eq_bytes(cur.x, C_NL), n1 = eq_bytes(cur.y, C_NL);
                        const uint32_t n2 = eq_bytes(cur.z, C_NL), n3 = eq_bytes(cur.w, C_NL);
                        const unsigned ebal = __ballot_sync(FULL, (n0 | n1 | n2 | n3) != 0);
                        if (ebal) {
                            const int src = __ffs(ebal) - 1;
                            int k = first_byte(n0, n1, n2, n3);
                            k = __shfl_sync(FULL, k, src);
                            e = wb + 16 * src + k; found = true;
                        }
                    }
                    if (!md_flag) {                          // the reference stops at the first hit too (:323-325)
                        uint32_t d0 = eq_bytes(cur.x, C_DOT), d1 = eq_bytes(cur.y, C_DOT);
                        uint32_t d2 = eq_bytes(cur.z, C_DOT), d3 = eq_bytes(cur.w, C_DOT);
                        if (firstw || found) {
                            const uint32_t l = firstw ? lo : 0u, h = found ? e : ~0u;
                            clip4(d0, d1, d2, d3, pb, l, h);
                        }
                        const bool any = (d0 | d1 | d2 | d3) != 0;
                        if (__any_sync(FULL, any)) {
                            md_any = true;
                            const bool hit = any && md_lane_dots(tin + pb, d0, d1, d2, d3, strip_cr);
                            md_flag = __any_sync(FULL, hit);
                        }
                    }
                    if (found) break;
                    firstw = false;
                    wb += WINDOW; cur = nxt; nxt = nx2; nx2 = ld16(tin + wb + 2 * WINDOW + 16 * lane);
                    if (((wb >> 9) & 7u) == 0) {          // every 8th window: L2 prefetch of the 4 KB that follow
                        const uint32_t pf = wb + 8 * WINDOW + 128 * lane;
                        if (pf < nrel) prefetch_l2(tin + pf);
                    }
                }
            }
            // ================= NONREF_FILTER: is every sample homozygous reference?
            bool nr_all = false;               // the line can be dropped and no sample so far speaks against it
            if ((OP == OP_NR || OP == OP_PC || OP == OP_GQ) && !hash && tabs >= 9 && (a0 + ls >= P.valid_from)) {
                const int gi_ = gt_index_of(tin + tp[7] + 1, tin + tp[8]);        // findGTIndex on FORMAT (nonref_filter :317-335, phase_checker :171-189)
                // phase_checker's file mode starts with the FORMAT cache ("", 0): an empty FORMAT column is "GT first" until a non-empty one was seen
                const int gi = (OP == OP_PC && gi_ < 0 && P.mode == MODE_FILE && tp[8] == tp[7] + 1 && (a0 + ls) < P.fmt0_until) ? 0 : gi_;
                GqQuery gq; gq.q = P.gq_query; gq.len = P.gq_len; gq.a = P.gq_a; gq.b = P.gq_b; gq.strict = P.gq_strict != 0;
                if (gi >= 0) {
                    nr_all = true;
                    const uint32_t lo = tp[8];                                    // the tab in front of the first sample
                    const bool file_mode = P.mode == MODE_FILE;
                    bool firstw = true;
                    for (;;) {
                        const uint32_t pb = wb + 16 * lane;
                        if (!firstw) {
                            const uint32_t n0 = eq_bytes(cur.x, C_NL), n1 = eq_bytes(cur.y, C_NL);
                            const uint32_t n2 = eq_bytes(cur.z, C_NL), n3 = eq_bytes(cur.w, C_NL);
                            const unsigned ebal = __ballot_sync(FULL, (n0 | n1 | n2 | n3) != 0);
                            if (ebal) {
                                const int src = __ffs(ebal) - 1;
                                int k = first_byte(n0, n1, n2, n3);
                                k = __shfl_sync(FULL, k, src);
                                e = wb + 16 * src + k; found = true;
                            }
                        }
                        // ---- lattice window: no line end in it, GT the first key, and behind every tab three bytes and the next tab, at
                        // the phase of the line's first sample — a 32-bit word per sample decides the whole window without a look at
                        // single tabs (nonref_filter: 0/0 or 0|0; phase_checker: x|y, neither a '.' nor the ':' that would end GT early)
                        bool lat_pass = false;
                        if (nr_all && !firstw && !found && gi == 0) {
                            const uint32_t tq = lo & 3u, sh8 = 8u * (tq + 1u);
                            uint32_t la = __shfl_down_sync(FULL, cur.x, 1);
                            const uint32_t nx0 = __shfl_sync(FULL, nxt.x, 0);
                            if (lane == 31) la = nx0;
                            const uint32_t uu[4] = {__funnelshift_rc(cur.x, cur.y, sh8), __funnelshift_rc(cur.y, cur.z, sh8),
                                                    __funnelshift_rc(cur.z, cur.w, sh8), __funnelshift_rc(cur.w, la, sh8)};
                            uint32_t badw = 0;
#pragma unroll
                            for (int j = 0; j < 4; ++j) {
                                const uint32_t u = uu[j];
                                if (OP == OP_NR) badw |= (u != 0x09302F30u && u != 0x09307C30u) ? 1u : 0u;
                                else if (OP == OP_GQ) {
                                    // a three-byte GT that is not the query (nr_all: "no sample has matched so far")
                                    badw |= (eq_bytes(u, C_TAB) ^ 0x80000000u) | eq_bytes(u, C_NL) | (eq_bytes(u, 0x3A3A3A3Au) & 0x00808080u);
                                    badw |= gq_match3(u, gq) ? 1u : 0u;
                                }
                                else {
                                    badw |= (eq_bytes(u, C_TAB) ^ 0x80000000u) | eq_bytes(u, C_NL);
                                    badw |= ((eq_bytes(u, C_DOT) | eq_bytes(u, 0x3A3A3A3Au)) & 0x00800080u) | ((u ^ 0x00007C00u) & 0x0000FF00u);
                                }
                            }
                            // (the bytes in front of the window's first tab belong to a sample the window before has answered for)
                            if (lane == 0) badw |= (eq_bytes(cur.x, C_TAB) & (0xFFFFFFFFu >> (24u - 8u * tq))) ^ (0x80u << (8u * tq));
                            lat_pass = __all_sync(FULL, badw == 0);
                        }
                        if (nr_all && !lat_pass) {                // the reference stops at the first sample that is not hom-ref too
                            uint32_t m0 = eq_bytes(cur.x, C_TAB), m1 = eq_bytes(cur.y, C_TAB);
                            uint32_t m2 = eq_bytes(cur.z, C_TAB), m3 = eq_bytes(cur.w, C_TAB);
                            if (firstw || found) clip4(m0, m1, m2, m3, pb, firstw ? lo : 0u, found ? e : ~0u);
                            uint32_t m16 = ((m0 * 0x00204081u) >> 28) | (((m1 * 0x00204081u) >> 24) & 0xF0u) |
                                           (((m2 * 0x00204081u) >> 20) & 0xF00u) | (((m3 * 0x00204081u) >> 16) & 0xF000u);
                            bool bad = false;
                            while (m16) {
                                const uint8_t *sp = tin + pb + __ffs(m16);          // first byte of the sample behind this tab
                                m16 &= m16 - 1u;
                                // "0/0" or "0|0" closed by a tab (by ':' as well when GT is the first key) needs no second look
                                const uint32_t *s4 = reinterpret_cast<const uint32_t *>((uintptr_t)sp & ~(uintptr_t)3);
                                const uint32_t q = __funnelshift_r(__ldg(s4), __ldg(s4 + 1), 8u * (uint32_t)((uintptr_t)sp & 3));
                                const uint32_t g3 = q & 0x00FFFFFFu, b3 = q >> 24;
                                if (OP == OP_NR) {
                                    // (only when GT is the first key: with GT further back a three-byte column has no GT at all)
                                    const bool quick = gi == 0 && (g3 == 0x00302F30u || g3 == 0x00307C30u) && (b3 == '\t' || b3 == ':');
                                    if (!quick && !nr_sample_homref(sp, file_mode, gi)) bad = true;
                                } else if (OP == OP_GQ) {
                                    // GT = exactly the three bytes behind the tab: decided from the word; anything else by the scalar matcher
                                    const uint32_t ends = eq_bytes(q, C_TAB) | eq_bytes(q, C_NL) | eq_bytes(q, 0x3A3A3A3Au);
                                    if (gi == 0 && (ends & 0x00808080u) == 0 && (ends & 0x80000000u)) { if (gq_match3(q, gq)) bad = true; }
                                    else if (gq_sample_match(sp, gi, gq)) bad = true;
                                } else {
                                    // phase_checker: "x|y" of exactly three bytes, x and y anything but '.' (and not an end of the GT)
                                    const uint32_t b0 = q & 0xFFu, b2 = (q >> 16) & 0xFFu;
                                    const bool e0 = b0 == '.' || b0 == '\t' || b0 == '\n' || b0 == ':' || b0 == '\r';
                                    const bool e2 = b2 == '.' || b2 == '\t' || b2 == '\n' || b2 == ':' || b2 == '\r';
                                    const bool quick = gi == 0 && ((q >> 8) & 0xFFu) == '|' && !e0 && !e2 && (b3 == '\t' || b3 == ':');
                                    if (!quick && !pc_sample_phased(sp, file_mode, gi)) bad = true;
                                }
                            }
                            if (__any_sync(FULL, bad)) nr_all = false;
                        }
                        if (found) break;
                        firstw = false;
                        wb += WINDOW; cur = nxt; nxt = nx2; nx2 = ld16(tin + wb + 2 * WINDOW + 16 * lane);
                        if (((wb >> 9) & 7u) == 0) {          // every 8th window: L2 prefetch of the 4 KB that follow
                            const uint32_t pf = wb + 8 * WINDOW + 128 * lane;
                            if (pf < nrel) prefetch_l2(tin + pf);
                        }
                    }
                }
            }
            // ================= no (more) per-sample work: just find the '\n'
            uint32_t wcount = 0;               // windows since the search began: prefetching on a line-relative beat
                                               // measured 7 % faster than on absolute 4 KB boundaries (variant_counter)
            while (!found) {
                wb += WINDOW; cur = nxt; nxt = nx2; nx2 = ld16(tin + wb + 2 * WINDOW + 16 * lane);
                if ((++wcount & 7u) == 0) {
                    const uint32_t pf = wb + 8 * WINDOW + 128 * lane;
                    if (pf < nrel) prefetch_l2(tin + pf);
                }
                uint32_t n0 = eq_bytes(cur.x, C_NL), n1 = eq_bytes(cur.y, C_NL);
                uint32_t n2 = eq_bytes(cur.z, C_NL), n3 = eq_bytes(cur.w, C_NL);
                unsigned ebal = __ballot_sync(FULL, (n0 | n1 | n2 | n3) != 0);
                if (ebal) {
                    int src = __ffs(ebal) - 1;
                    int k = first_byte(n0, n1, n2, n3);
                    k = __shfl_sync(FULL, k, src);
                    e = wb + 16 * src + k; found = true;
                }
            }

            // ================= end of line: [ls, ee) content, '\n' at e
            ++nlines;
            uint32_t ee = e;
            if (strip_cr && e > ls && ldb(tin + e - 1) == '\r') ee = e - 1;
            if (OP == OP_VC) {
                // variant_counter.cpp:364-380: raw-empty and '#' lines are skipped, >= 7 tabs counts
                if (e != ls && !hash) {
                    if (tabs >= 7) VCFX_COUNT(C_ROWS, 1);
                    else {
                        VCFX_COUNT(C_SHORT, 1);
                        if (lane == 0) {
                            unsigned long long key = ((unsigned long long)tile << 32) | (nlines - 1);
                            atomicMin(&P.stats->first_short_key, key);
                            unsigned long long slot = atomicAdd(&P.stats->n_events, 1ULL);
                            if (slot < P.ev_cap) P.events[slot] = key;
                        }
                    }
                }
            } else if ((OP == OP_AF || OP == OP_HWE) && ee != ls && !hash) {
                uint32_t ra_ = 0, rb_ = 0, rc_ = 0;
                if (do_samples) {
                    ra_ = __reduce_add_sync(FULL, ta); rb_ = __reduce_add_sync(FULL, tb);
                    if (OP == OP_HWE) rc_ = __reduce_add_sync(FULL, tc);
                }
                bool row = false;
                if (OP == OP_AF) {
                    if (a0 + ls < P.valid_from) VCFX_COUNT(C_PRE, 1);                 // allele_freq_calc.cpp:382-386 / 499-502
                    else if (P.mode == MODE_FILE) {
                        VCFX_COUNT(C_DATA, 1);
                        // FORMAT must exist and be non-empty (:396-401) and hold a GT key (:413)
                        if (tabs >= 9) row = gt_index >= 0;
                        else if (tabs == 8 && tp[7] + 1 < ee) row = gt_index_of(tin + tp[7] + 1, tin + ee) >= 0;
                    } else {
                        // stdin: fields = tabs + 1, minus a dropped empty tail (:509-518); < 9 warns (:520-523)
                        int nf = tabs + ((ldb(tin + ee - 1) == '\t') ? 0 : 1);
                        if (nf < 9) VCFX_COUNT(C_SHORT, 1);
                        else {
                            VCFX_COUNT(C_DATA, 1);
                            if (tabs >= 9) row = gt_index >= 0;
                            else row = gt_index_of(tin + tp[7] + 1, tin + ee) >= 0;
                        }
                    }
                } else {
                    VCFX_COUNT(C_DATA, 1);
                    if (tabs >= 9 && do_samples) {
                        bool comma = false;                              // hwe_tester.cpp:503 / :586
                        for (uint32_t q = tp[3] + 1; q < tp[4]; ++q) comma |= (ldb(tin + q) == ',');
                        row = !comma;
                        if (P.mode == MODE_FILE)                         // :497 and :516-520
                            row = row && (tp[0] > ls) && (tp[1] > tp[0] + 1) && (tp[4] > tp[3] + 1) && (tp[8] + 1 < ee);
                    }
                }
                if (row) {
                    const uint32_t prefix_len = tp[4] + 1 - ls;
                    const uint32_t row_len = prefix_len + ((OP == OP_AF) ? 7u : 9u);
                    unsigned long long slot = 0;
                    if (lane == 0) slot = alloc_slot(ws.rec_base, ws.rec_used, P.stats);
                    slot = __shfl_sync(FULL, slot, 0);
                    if (slot < P.rec_cap) {
                        if (lane == 0) {
                            Rec r; r.tile = tile; r.ls_rel = (uint32_t)(a0 + ls - a); r.prefix_len = prefix_len;
                            r.off_in_tile = (uint32_t)out_bytes; r.a = ra_; r.b = rb_; r.c = rc_; r.d = 0;
                            P.recs[slot] = r;
                        }
                        // the line's first bytes are still close (L2): keep a copy of the prefix next to the
                        // record so that the format kernel does not have to gather it from the input
                        if (prefix_len <= 32 && (uint32_t)lane < prefix_len) P.rec_prefix[slot * 32 + lane] = (uint8_t)ldb(tin + ls + lane);
                    }
                    out_bytes += row_len; VCFX_COUNT(C_ROWS, 1);
                }
            }
            else if (OP == OP_AC) {
                // allele_counter.cpp:571 / :1373: empty and '#' lines are skipped; no '\r' handling
                if (e != ls && !hash) {
                    if (P.ac_pass == 0) VCFX_COUNT(C_DATA, 1);
                    const uint2 *scr = P.col_scratch + (size_t)(blockIdx.x * WARPS_PER_CTA + wid) * P.max_col;
                    const uint32_t ns_parsed = tabs >= 9 ? (uint32_t)(tabs - 8) : 0u;
                    uint32_t n_rows = P.n_sel;
                    if (P.ac_fmt != AC_TEXT_MT) {
                        // forward walk: a column exists while its first byte lies before the line end
                        // (:1222-1229, :1416-1423); rows stop at the first selected column that does not
                        uint32_t ns_f = 0;
                        if (tabs >= 9 && tp[8] + 1 < e) ns_f = ns_parsed - ((ldb(tin + e - 1) == '\t') ? 1u : 0u);
                        uint32_t lo_ = 0, hi_ = P.n_sel;           // first i with sel_col[i] >= ns_f (non-decreasing)
                        while (lo_ < hi_) { const uint32_t mid = (lo_ + hi_) >> 1; if (P.sel_col[mid] < ns_f) lo_ = mid + 1; else hi_ = mid; }
                        n_rows = lo_;
                    }
                    const uint32_t extra_tabs = tabs >= 5 ? 0u : (uint32_t)(5 - tabs);   // absent fields are empty (:578-601)
                    const uint32_t prefix_src = tabs >= 5 ? tp[4] + 1 - ls : e - ls;
                    const uint32_t prefix_len = prefix_src + extra_tabs;
                    if (P.ac_fmt == AC_AGG) {
                        uint32_t sr = ta, sa = tb;                  // identity selection: the lanes summed while parsing
                        if (!P.ac_ident) {
                            sr = 0; sa = 0;
                            for (uint32_t i = lane; i < n_rows; i += 32) {
                                const uint32_t c = P.sel_col[i];
                                if (c < ns_parsed) { const uint2 v = scr[c]; sr += v.x; sa += v.y; }
                            }
                        }
                        sr = __reduce_add_sync(FULL, sr); sa = __reduce_add_sync(FULL, sa);
                        const uint32_t row_len = prefix_len + dec_len((int)sr) + 1 + dec_len((int)sa) + 1 + dec_len((int)n_rows) + 1;
                        if (lane == 0) {
                            unsigned long long slot = alloc_slot(ws.rec_base, ws.rec_used, P.stats);
                            if (slot < P.rec_cap) {
                                Rec r; r.tile = tile; r.ls_rel = (uint32_t)(a0 + ls - a); r.prefix_len = prefix_src;
                                r.off_in_tile = (uint32_t)out_bytes; r.a = sr; r.b = sa; r.c = n_rows; r.d = extra_tabs;
                                P.recs[slot] = r;
                            }
                        }
                        out_bytes += row_len; VCFX_COUNT(C_ROWS, 1);
                    } else {
                        uint8_t *stage0 = ws.stage0;
                        uint32_t n_rows_done = 0;
                        unsigned long long opos = (P.ac_pass ? P.tile_base[tile] : 0ULL) + out_bytes;
                        const bool text = (P.ac_fmt != AC_BIN);
                        if (ac_sizing_only) {
                            // every row is prefix + name + '\t' + one digit + '\t' + one digit + '\n'
                            out_bytes += (unsigned long long)n_rows * (prefix_len + 4u) + (P.name_off[n_rows] - P.name_off[0]);
                            n_rows_done = n_rows; n_rows = 0;
                        }
                        // ---- the fast row writer (write pass, text rows, every selected name of the same length NL <= 12 with its
                        // tab, counts of one digit): all rows of a line then have the same length L = prefix + NL + 4 and differ in
                        // 16 bytes.  Lane i assembles the ALIGNED WORDS its row covers in the staging buffer from registers: the bytes
                        // every row shares (U, built once per line: the prefix, and around it what the neighbours put there — the
                        // last 3 bytes of the row before, "\t a \n", and the first 3 of the row after, again the prefix), its own
                        // name and digits shifted into place, all of it rotated by the row's misalignment.  Neighbouring lanes write
                        // the words they share with identical contents, so no byte stores and no ordering are needed.
                        const unsigned long long out_limit = P.ac_pass ? min((unsigned long long)P.out_cap, P.tile_base[tile] + P.tile_out[tile]) : 0ULL;
                        const uint32_t NL = P.name_len;
                        const bool fast_line = P.ac_pass && text && NL != 0u && extra_tabs == 0u && prefix_src <= 40u && prefix_src >= 1u;
                        const uint32_t L = prefix_src + NL + 4u;
                        if (fast_line) {
                            __syncwarp();
                            if (lane < 20) {
                                uint32_t w = 0;
#pragma unroll
                                for (uint32_t bb = 0; bb < 4; ++bb) {
                                    const uint32_t pp = 4u * (uint32_t)lane + bb;                 // position in the lane's view of its row
                                    uint32_t byte = 0;
                                    if (pp >= 3u && pp < 3u + prefix_src) byte = ldb(tin + ls + pp - 3u);
                                    else if (pp >= 3u + L && pp < 6u + L) byte = ldb(tin + ls + pp - 3u - L);
                                    w |= byte << (8u * bb);
                                }
                                ws.u[lane] = w;
                            }
                            __syncwarp();
                        }
                        for (uint32_t i0 = 0; i0 < n_rows; i0 += 32) {
                            const uint32_t i = i0 + lane;
                            int vr = 0, va = 0; uint32_t len = 0, noff = 0, nlen = 0;
                            if (i < n_rows) {
                                const uint32_t c = P.ac_ident ? i : P.sel_col[i];      // (all samples in order: one dependent load less)
                                if (c < ns_parsed) { const uint2 v = scr[c]; vr = (int)v.x; va = (int)v.y; }
                                if (P.ac_fmt != AC_TEXT_FWD) { vr = (int)(int8_t)vr; va = (int)(int8_t)va; }   // int8 storage (:621-622, :1446-1447)
                            }
                            // rows of one length (the fast row writer's case) need no scan: row i starts at i * L
                            const bool fast = fast_line && __all_sync(FULL, i >= n_rows || ((uint32_t)vr <= 9u && (uint32_t)va <= 9u));
                            uint32_t off, btot;
                            if (fast) { off = (uint32_t)lane * L; btot = min(32u, n_rows - i0) * L; }
                            else {
                                if (i < n_rows) {
                                    if (text) {
                                        noff = P.name_off[i]; nlen = P.name_off[i + 1] - noff;     // name + '\t'
                                        len = prefix_len + nlen + dec_len(vr) + 1 + dec_len(va) + 1;
                                    } else len = 2;
                                }
                                const int incl = warp_incl_scan((int)len, lane);
                                off = (uint32_t)incl - len;
                                btot = (uint32_t)__shfl_sync(FULL, incl, 31);
                            }
                            // the write pass never stores past the bytes the size pass gave this tile (speculative sizes can be
                            // too small: a count of two digits) nor past the output buffer; the chunk is then run again, exact
                            if (P.ac_pass && opos + btot > out_limit) {
                                if (lane == 0) atomicOr(&P.stats->overflow, (unsigned long long)OV_AC_SPEC);
                            } else
                            if (fast) {
                                uint32_t *sw = reinterpret_cast<uint32_t *>(stage0);
                                const uint32_t o = (uint32_t)((uintptr_t)(P.out + opos) & 15) + (uint32_t)lane * L;   // the row's place in the staging buffer
                                const uint32_t sh = 8u * (3u - (o & 3u));
                                const uint32_t a_prev = __shfl_up_sync(FULL, (uint32_t)va, 1);
                                if (i < n_rows) {
                                    const uint32_t tl = 0x000A0009u | ((48u + a_prev) << 8);              // "\t a \n" of the row before
                                    // the row's own 16 bytes: name and tab (zero padded), then r '\t' a '\n' at byte NL
                                    const uint4 nm = __ldg(P.names16 + i);
                                    const uint32_t T = (48u + (uint32_t)vr) | (0x09u << 8) | ((48u + (uint32_t)va) << 16) | (0x0Au << 24);
                                    const uint32_t ti = NL >> 2, ts = 8u * (NL & 3u);
                                    const uint32_t Tlo = T << ts, Thi = ts ? (T >> (32u - ts)) : 0u;
                                    const uint32_t v0 = nm.x | (ti == 0 ? Tlo : 0u);
                                    const uint32_t v1 = nm.y | (ti == 1 ? Tlo : 0u) | (ti == 0 ? Thi : 0u);
                                    const uint32_t v2 = nm.z | (ti == 2 ? Tlo : 0u) | (ti == 1 ? Thi : 0u);
                                    const uint32_t v3 = nm.w | (ti == 3 ? Tlo : 0u) | (ti == 2 ? Thi : 0u);
                                    // ... moved up to byte (3 + prefix) & 3 of word q = (3 + prefix) >> 2 of the lane's view
                                    const uint32_t q = (3u + prefix_src) >> 2, sv = 8u * ((3u + prefix_src) & 3u);
                                    const uint32_t s0 = __funnelshift_l(0u, v0, sv), s1 = __funnelshift_l(v0, v1, sv), s2 = __funnelshift_l(v1, v2, sv);
                                    const uint32_t s3 = __funnelshift_l(v2, v3, sv), s4 = __funnelshift_l(v3, 0u, sv);
                                    const uint32_t nw = ((o & 3u) + L + 3u) >> 2;                          // aligned words the row touches
                                    uint32_t *dw = sw + (o >> 2);
                                    // words that hold shared bytes only
                                    for (uint32_t k = 0; k + 1u < q; ++k) {
                                        const uint32_t lo_ = ws.u[k] | (k == 0u ? tl : 0u), hi_ = ws.u[k + 1];
                                        dw[k] = __funnelshift_r(lo_, hi_, sh);
                                    }
                                    // the six words around the row's own bytes
                                    const uint32_t c_1 = ws.u[q - 1] | (q == 1u ? tl : 0u);
                                    const uint32_t c0 = ws.u[q] | s0, c1 = ws.u[q + 1] | s1, c2 = ws.u[q + 2] | s2, c3 = ws.u[q + 3] | s3, c4 = ws.u[q + 4] | s4, c5 = ws.u[q + 5];
                                    if (q - 1u < nw) dw[q - 1] = __funnelshift_r(c_1, c0, sh);
                                    if (q < nw) dw[q] = __funnelshift_r(c0, c1, sh);
                                    if (q + 1u < nw) dw[q + 1] = __funnelshift_r(c1, c2, sh);
                                    if (q + 2u < nw) dw[q + 2] = __funnelshift_r(c2, c3, sh);
                                    if (q + 3u < nw) dw[q + 3] = __funnelshift_r(c3, c4, sh);
                                    if (q + 4u < nw) dw[q + 4] = __funnelshift_r(c4, c5, sh);
                                }
                                __syncwarp();
                                if (P.ac_bulk) warp_flush_smem_bulk(P.out + opos, stage0 + (uint32_t)((uintptr_t)(P.out + opos) & 15), btot, lane);
                                else warp_flush_smem(P.out + opos, stage0 + (uint32_t)((uintptr_t)(P.out + opos) & 15), btot, lane);
                                __syncwarp();
                            } else
                            if (P.ac_pass) {
                                const bool staged = btot <= AC_STAGE;
                                // staged at the destination's offset modulo 16: the flush is aligned 128-bit copies
                                uint8_t *stage = stage0 + (uint32_t)((uintptr_t)(P.out + opos) & 15);
                                uint8_t *d = staged ? stage + off : P.out + opos + off;
                                if (i < n_rows) {
                                    if (text) {
                                        const uint8_t *src = tin + ls;
                                        for (uint32_t k = 0; k < prefix_src; ++k) d[k] = (uint8_t)ldb(src + k);
                                        d += prefix_src;
                                        for (uint32_t k = 0; k < extra_tabs; ++k) *d++ = '\t';
                                        const uint8_t *nm = P.names + noff;
                                        for (uint32_t k = 0; k < nlen; ++k) d[k] = (uint8_t)ldb(nm + k);
                                        d += nlen;
                                        d = put_dec(d, vr); *d++ = '\t'; d = put_dec(d, va); *d++ = '\n';
                                    } else { d[0] = (uint8_t)vr; d[1] = (uint8_t)va; }
                                }
                                if (staged) { __syncwarp(); warp_flush_smem(P.out + opos, stage, btot, lane); __syncwarp(); }
                            }
                            opos += btot; out_bytes += btot;
                        }
                        if (P.ac_pass == 0) VCFX_COUNT(C_ROWS, ac_sizing_only ? n_rows_done : n_rows);
                    }
                }
            }
            else if (OP == OP_IX) {
                // VCFX_indexer: a row (CHROM, POS, byte offset of the line) for every data line behind the "#CHROM" line
                // that parses; both modes cut a '\r' in front of the '\n' and skip empty lines
                if (ee != ls && (a0 + ls >= P.valid_from)) {
                    uint32_t c_off = 0, c_len = 0; long long pos = 0; bool ok = false;
                    if (lane == 0) ok = ix_parse_line(tin + ls, tin + ee, P.mode == MODE_FILE, c_off, c_len, pos);
                    ok = __shfl_sync(FULL, (int)ok, 0) != 0;
                    if (ok) {
                        uint32_t row_len = 0;
                        if (lane == 0) {
                            row_len = c_len + 1u + dec_len64(pos) + 1u + dec_len64((long long)(P.file_offset + a0 + ls)) + 1u;
                            unsigned long long slot = alloc_slot(ws.rec_base, ws.rec_used, P.stats);
                            if (slot < P.rec_cap) {
                                Rec r; r.tile = tile; r.ls_rel = (uint32_t)(a0 + ls - a); r.prefix_len = c_len;
                                r.off_in_tile = (uint32_t)out_bytes; r.a = c_off; r.b = 0;
                                r.c = (uint32_t)((unsigned long long)pos & 0xFFFFFFFFULL); r.d = (uint32_t)((unsigned long long)pos >> 32);
                                P.recs[slot] = r;
                            }
                        }
                        out_bytes += __shfl_sync(FULL, row_len, 0); VCFX_COUNT(C_ROWS, 1);
                    }
                }
            }
            else if (OP == OP_IB) {
                // VCFX_inbreeding_calculator.cpp:531-600 / :718-757: a row (alt alleles, genotyped samples, columns) for every line
                // whose genotypes were looked at; the file mode also wants a byte behind the ninth tab
                if (ib_line) {
                    const uint32_t alt = __reduce_add_sync(FULL, ib_alt), good = __reduce_add_sync(FULL, ib_good);
                    if (P.mode != MODE_FILE || tp[8] + 1 < ee) {
                        VCFX_COUNT(C_DATA, 1);
                        if (good >= 2) VCFX_COUNT(C_ROWS, 1);
                        if (lane == 0) {
                            const unsigned long long slot = alloc_slot(ws.rec_base, ws.rec_used, P.stats);
                            if (slot < P.rec_cap) {
                                Rec r; r.tile = tile; r.ls_rel = (uint32_t)(a0 + ls - a); r.prefix_len = 0;
                                r.off_in_tile = (uint32_t)out_bytes; r.a = alt; r.b = good;
                                r.c = min((uint32_t)(tabs - 8), P.n_sel); r.d = (((tp[8] + 4u) >> 2) - 1u) & 3u;
                                P.recs[slot] = r;
                            }
                        }
                        out_bytes += 1;                                  // (rows, not bytes: the scan turns them into the row's rank)
                    }
                }
            }
            else if (OP == OP_PC) {
                // VCFX_phase_checker.cpp:493-558 / 576-650: '#' lines and empty lines pass; a data line passes when it lies behind
                // the "#CHROM" line, has its ten columns and a GT key, and every sample is fully phased; each dropped line leaves
                // an event (its offset and why) for the message the tool prints on stderr.
                const bool term = (a0 + e) < n;
                const uint32_t raw_end = term ? e + 1 : e;
                const bool file_mode = P.mode == MODE_FILE;
                const uint32_t cend = file_mode ? ee : e;                // stdin mode: getline keeps a '\r'
                const bool data = (cend != ls) && !hash;
                bool drop = false; uint32_t why = 0;                     // 0 unphased (or no GT key, file mode), 1 before the header, 2 fewer than ten columns, 3 no GT key (stdin mode)
                if (data) {
                    VCFX_COUNT(C_DATA, 1);
                    if (a0 + ls < P.valid_from) { drop = true; why = 1; VCFX_COUNT(C_PRE, 1); }
                    else if (file_mode) {
                        // :296-359: eight tabs and a byte behind them, a GT key, a tab behind FORMAT, then the samples
                        if (tabs < 8 || tp[7] + 1 >= cend) { drop = true; why = 2; }
                        else if (tabs == 8) { drop = true; why = gt_index_of(tin + tp[7] + 1, tin + cend) < 0 ? 0u : 2u; }
                        else if (!nr_all) drop = true;                   // (no GT key, or a sample that is not phased)
                    } else {
                        if (tabs < 9) { drop = true; why = 2; }
                        else if (gt_index_of(tin + tp[7] + 1, tin + tp[8]) < 0) { drop = true; why = 3; }
                        else if (!nr_all) drop = true;
                    }
                }
                if (data && !drop) VCFX_COUNT(C_ROWS, 1);
                if (drop) {
                    VCFX_COUNT(C_FLAG, 1);
                    if (lane == 0) {
                        const unsigned long long slot = atomicAdd(&P.stats->n_events, 1ULL);
                        if (slot < P.ev_cap) P.events[slot] = ((unsigned long long)(a0 + ls) << 2) | why;
                    }
                }
                if (drop || cend != e || !term) {
                    const uint32_t content_len = drop ? 0u : cend - ls, mod_len = drop ? 0u : content_len + 1u;
                    if (lane == 0) {
                        unsigned long long slot = alloc_slot(ws.rec_base, ws.rec_used, P.stats);
                        if (slot < P.rec_cap) {
                            Rec r; r.tile = tile; r.ls_rel = (uint32_t)(a0 + ls - a); r.prefix_len = (uint32_t)(a0 + md_prev_end - a);
                            r.off_in_tile = (uint32_t)out_bytes; r.a = 0; r.b = NR_PLAIN; r.c = content_len; r.d = mod_len;
                            P.recs[slot] = r;
                        }
                    }
                    out_bytes += (ls - md_prev_end) + mod_len;
                    md_prev_end = raw_end;
                }
                md_add_nl = false;
                md_last_end = raw_end;
            }
            else if (OP == OP_DS) {
                // VCFX_dosage_calculator.cpp:421-591 / :228-356: a row (CHROM .. ALT, then the dosages) for every data line with ten
                // columns; "NA" alone without a GT key; a column that would start at the line end is not there
                if (ee != ls && !hash) {
                    VCFX_COUNT(C_DATA, 1);
                    if (tabs < 9) {
                        VCFX_COUNT(C_SHORT, 1);                          // "Skipping VCF line with fewer than 10 fields."
                    } else {
                        const uint32_t nna = __reduce_add_sync(FULL, ib_alt);
                        const uint32_t prefix_len = tp[4] + 1 - ls;
                        uint32_t ncols = (uint32_t)(tabs - 8);
                        if (ldb(tin + ee - 1) == '\t') --ncols;
                        const uint32_t dlen = ds_gi < 0 ? 2u : (ncols ? 2u * ncols - 1u + nna : 0u);
                        if (lane == 0) {
                            const unsigned long long slot = alloc_slot(ws.rec_base, ws.rec_used, P.stats);
                            if (slot < P.rec_cap) {
                                Rec r; r.tile = tile; r.ls_rel = (uint32_t)(a0 + ls - a); r.prefix_len = prefix_len;
                                r.off_in_tile = (uint32_t)out_bytes; r.a = ncols; r.b = dlen; r.c = ds_gi < 0 ? 1u : 0u;
                                r.d = (((tp[8] + 4u) >> 2) - 1u) & 3u;
                                P.recs[slot] = r;
                            }
                        }
                        if (P.ds_matrix) {
                            out_bytes += 1u;                             // matrix mode: the row's rank, not its text
                            if (ncols > P.n_sel) VCFX_COUNT(C_FLAG, 1);  // columns beyond W are dropped
                        } else out_bytes += prefix_len + dlen + 1u;
                        VCFX_COUNT(C_ROWS, 1);
                    }
                }
            }
            else if (OP == OP_GQ) {
                // VCFX_genotype_query.cpp:446-516 / 546-606: '#' lines pass, empty lines vanish, a data line passes when it has a
                // FORMAT column with a GT key and a sample whose GT is the query; no '\r' is cut.  (The caller feeds nothing
                // behind a data line that comes before the "#CHROM" line, and holds back stdin mode's trailing '#' lines.)
                const bool term = (a0 + e) < n;
                const uint32_t raw_end = term ? e + 1 : e;
                const bool data = (e != ls) && !hash;
                bool drop = (e == ls);
                if (data) {
                    VCFX_COUNT(C_DATA, 1);
                    if (tabs < 8) {
                        // skipToField(.., 8): NULL when a tab is missing and the line goes on; a line that ends with its last tab
                        // gets an empty FORMAT instead, and no message
                        drop = true;
                        if (ldb(tin + e - 1) != '\t') {
                            VCFX_COUNT(C_SHORT, 1);
                            if (lane == 0) {
                                const unsigned long long slot = atomicAdd(&P.stats->n_events, 1ULL);
                                if (slot < P.ev_cap) P.events[slot] = ((unsigned long long)(a0 + ls) << 2) | 2ULL;
                            }
                        }
                    }
                    else if (gt_index_of(tin + tp[7] + 1, tin + (tabs >= 9 ? tp[8] : e)) < 0) drop = true;
                    else drop = (tabs < 9) || nr_all;                    // nr_all: no sample matched
                }
                if (data && !drop) VCFX_COUNT(C_ROWS, 1);
                if (drop || !term) {
                    const uint32_t content_len = drop ? 0u : e - ls, mod_len = drop ? 0u : content_len + 1u;
                    if (lane == 0) {
                        unsigned long long slot = alloc_slot(ws.rec_base, ws.rec_used, P.stats);
                        if (slot < P.rec_cap) {
                            Rec r; r.tile = tile; r.ls_rel = (uint32_t)(a0 + ls - a); r.prefix_len = (uint32_t)(a0 + md_prev_end - a);
                            r.off_in_tile = (uint32_t)out_bytes; r.a = 0; r.b = NR_PLAIN; r.c = content_len; r.d = mod_len;
                            P.recs[slot] = r;
                        }
                    }
                    out_bytes += (ls - md_prev_end) + mod_len;
                    md_prev_end = raw_end;
                }
                md_add_nl = false;
                md_last_end = raw_end;
            }
            else if (OP == OP_NR) {
                // VCFX_nonref_filter.cpp:478-544 / 553-631: every line is written as its content + '\n' (file mode: without a
                // '\r' before the '\n'), except data lines behind the "#CHROM" line whose samples are all hom-ref.  Lines that
                // come out exactly as they went in stay part of the verbatim spans; the others get a record.
                const bool term = (a0 + e) < n;                          // a real '\n', not the pad behind the chunk
                const uint32_t raw_end = term ? e + 1 : e;
                const bool data = (ee != ls) && !hash;
                if (data) {
                    VCFX_COUNT(C_DATA, 1);
                    if (a0 + ls < P.valid_from) VCFX_COUNT(C_PRE, 1);    // "data line encountered before #CHROM": passed, with a warning
                }
                const bool drop = data && nr_all;
                if (data && !drop) VCFX_COUNT(C_ROWS, 1);
                if (drop || ee != e || !term) {
                    const uint32_t content_len = drop ? 0u : ee - ls, mod_len = drop ? 0u : content_len + 1u;
                    if (lane == 0) {
                        unsigned long long slot = alloc_slot(ws.rec_base, ws.rec_used, P.stats);
                        if (slot < P.rec_cap) {
                            Rec r; r.tile = tile; r.ls_rel = (uint32_t)(a0 + ls - a); r.prefix_len = (uint32_t)(a0 + md_prev_end - a);
                            r.off_in_tile = (uint32_t)out_bytes; r.a = 0; r.b = NR_PLAIN; r.c = content_len; r.d = mod_len;
                            P.recs[slot] = r;
                        }
                    }
                    out_bytes += (ls - md_prev_end) + mod_len;
                    md_prev_end = raw_end;
                    if (drop) VCFX_COUNT(C_FLAG, 1);
                }
                md_add_nl = false;
                md_last_end = raw_end;
            }
            else if (OP == OP_MD) {
                const bool term = (a0 + e) < n;                          // a real '\n', not the pad behind the chunk
                const uint32_t raw_end = term ? e + 1 : e;
                const bool data = (ee != ls) && !hash;                   // missing_detector.cpp:511 / :865-873
                if (data) VCFX_COUNT(C_DATA, 1);
                const bool has_samples = data && tabs >= 9;
                // the reference's pre-scan looks at every terminated line after the leading '#' block (:347-369)
                if (term && has_samples && md_any && tp[8] + 1 < e && (a0 + ls >= P.valid_from)) VCFX_COUNT(C_DOTS, 1);
                md_add_nl = false;
                if (has_samples && md_flag && tp[8] + 1 < ee) {          // :520-527, :530
                    const uint32_t info_off = tp[6] + 1 - ls, info_len = tp[7] - tp[6] - 1, content_len = ee - ls;
                    uint32_t mod_len;                                    // :559-574 / :900-909
                    if (info_len == 0 || (info_len == 1 && ldb(tin + tp[6] + 1) == '.')) mod_len = content_len - info_len + 19;
                    else mod_len = content_len + 19 + ((ldb(tin + tp[7] - 1) != ';') ? 1u : 0u);
                    mod_len += 1;                                        // the rewritten line always ends with '\n'
                    if (lane == 0) {
                        unsigned long long slot = alloc_slot(ws.rec_base, ws.rec_used, P.stats);
                        if (slot < P.rec_cap) {
                            Rec r; r.tile = tile; r.ls_rel = (uint32_t)(a0 + ls - a); r.prefix_len = (uint32_t)(a0 + md_prev_end - a);
                            r.off_in_tile = (uint32_t)out_bytes; r.a = info_off; r.b = info_len; r.c = content_len; r.d = mod_len;
                            P.recs[slot] = r;
                        }
                        if (!term) P.stats->last_unterminated_flagged = mod_len;
                    }
                    out_bytes += (ls - md_prev_end) + mod_len;
                    md_prev_end = raw_end;
                    VCFX_COUNT(C_FLAG, 1);
                } else if (!term && P.mode == MODE_STDIN) md_add_nl = true;   // getline + "\n" (:866-889)
                md_last_end = raw_end;
            }
            __syncwarp();
            ls = e + 1;
        }
    VCFX_SAVE_STATE();
    return true;
#undef VCFX_COUNT
#undef VCFX_SAVE_STATE
}

// variant_counter is light enough to run at 48 registers (5 CTAs per SM: +4.5 %); the parsing
// instantiations need 64 to keep the steady loops free of spills (measured both ways, profiles/README.md)
#ifndef VCFX_PARSE_CTAS
#define VCFX_PARSE_CTAS 4
#endif
#ifndef VCFX_AC_CTAS
#define VCFX_AC_CTAS 4               // allele_counter
#endif
#ifndef VCFX_GENERAL_CTAS
#define VCFX_GENERAL_CTAS 3          // resident CTAs per SM of the general kernel: 80 registers, no spills (C3 allele_freq_calc 1.85 ms at 4 CTAs / 64 registers, 1.90 at 5 / 48, 1.72 at 3 / 80)
#endif
// resident CTAs per SM of vcfx_scan_kernel<OP, VAR>: its __launch_bounds__, and the grids vcfx_api.cu launches it with
__host__ __device__ constexpr int scan_ctas(int op, int var) {
    return (op == OP_VC) ? 5 : (var == 1 ? VCFX_GENERAL_CTAS : (op == OP_AC ? VCFX_AC_CTAS : VCFX_PARSE_CTAS));
}
// Two kernels for allele_freq_calc and hwe_tester, launched one after the other over the same tiles, so that each is
// compiled (registers, schedule) on its own:
//   VAR 0  the lattice kernel: tier 1 + the exact path.  In a tile it stops at the first line whose first sample
//          window is not tier-1 material, leaves the tile's state (next line, lines and output bytes so far) behind
//          and goes on to the next tile
//   VAR 1  the general kernel: picks up exactly those tiles where they were left and finishes them (digit path,
//          skip-ahead loop for multi-key FORMATs, tier 1 and the exact path); it exits at once when none was left
// The other operations have one kernel (VAR 0, never stops early).
template <int OP, int VAR>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32, scan_ctas(OP, VAR))
vcfx_scan_kernel(const VCFX_GRID_CONSTANT KParams P) {
    __shared__ uint32_t s_tp[WARPS_PER_CTA][12];
    __shared__ __align__(128) uint8_t s_ring[(VCFX_C4_RING && VAR == 1) ? WARPS_PER_CTA * C4_RING : 16];
    __shared__ __align__(8) unsigned long long s_bars[(VCFX_C4_RING && VAR == 1) ? WARPS_PER_CTA * C4_STAGES : 1];
    __shared__ uint32_t s_ring_par[WARPS_PER_CTA];
    __shared__ __align__(16) uint8_t s_stage[(OP == OP_AC) ? WARPS_PER_CTA * (AC_STAGE + 32) : 16];
    __shared__ uint32_t s_u[(OP == OP_AC) ? WARPS_PER_CTA : 1][20];
    const int lane = lane_id();
    const int wid = threadIdx.x >> 5;
    const uint64_t n = P.n;
    const bool strip_cr = (OP == OP_HWE) || (P.mode == MODE_FILE && (OP == OP_AF || OP == OP_VC || OP == OP_MD || OP == OP_NR || OP == OP_PC)) || OP == OP_IX || OP == OP_IB || (OP == OP_DS && P.mode == MODE_FILE);
    if (OP == OP_AC && P.ac_pass && P.stats->overflow) return;
    if (VAR == 1 && P.stats->n_unfinished == 0) return;

    // per-warp event counters live in shared memory (fire-and-forget adds from lane 0) and are folded into
    // DevStats after every tile; the slot index is the field's index in DevStats
    __shared__ unsigned int s_cnt[WARPS_PER_CTA][CNT_SLOTS];
    if (lane < CNT_SLOTS) s_cnt[wid][lane] = 0;
    __syncwarp();
#define VCFX_COUNT(slot, v) do { if (lane == 0) atomicAdd(&s_cnt[wid][slot], (unsigned int)(v)); } while (0)
    __shared__ unsigned long long s_rec_base[WARPS_PER_CTA];
    __shared__ unsigned int s_rec_used[WARPS_PER_CTA];
    __shared__ volatile unsigned int s_odd[WARPS_PER_CTA], s_reg[WARPS_PER_CTA], s_tag[WARPS_PER_CTA];
    if (lane == 0) s_tag[wid] = 0;
    if (lane == 0) { s_rec_base[wid] = 0; s_rec_used[wid] = REC_BLOCK; }
    __syncwarp();
    WarpShared ws;
    ws.tp = s_tp[wid]; ws.stage0 = s_stage + ((OP == OP_AC) ? wid * (AC_STAGE + 32) : 0); ws.cnt = s_cnt[wid]; ws.u = s_u[(OP == OP_AC) ? wid : 0];
    ws.ring = s_ring + ((VCFX_C4_RING && VAR == 1) ? wid * C4_RING : 0); ws.bars = s_bars + ((VCFX_C4_RING && VAR == 1) ? wid * C4_STAGES : 0); ws.ring_par = &s_ring_par[wid];
    if (VCFX_C4_RING && VAR == 1) { if ((threadIdx.x & 31) == 0) s_ring_par[wid] = 0; ring_init(ws.bars, threadIdx.x & 31); }
    ws.rec_base = &s_rec_base[wid]; ws.rec_used = &s_rec_used[wid]; ws.odd = s_odd; ws.reg = s_reg; ws.tag = s_tag;

    for (;;) {
        uint32_t tile = 0;
        if (lane == 0) tile = atomicAdd(VAR == 1 ? P.ticket2 : P.ticket, 1u);
        tile = __shfl_sync(FULL, tile, 0);
        if (tile >= P.n_tiles) break;
        uint32_t resume = RESUME_DONE;
        if (VAR == 1) { resume = P.tile_resume[tile]; if (resume == RESUME_DONE) continue; }

        const uint64_t a = (uint64_t)tile * P.tile_bytes;
        const uint64_t b = min(a + (uint64_t)P.tile_bytes, n);
        // every position inside the tile's work is a 32-bit offset from a0 (16-aligned, <= a-1)
        const uint64_t a0 = a - (tile ? 16u : 0u);             // tile_bytes is a multiple of 512, so a is 16-aligned
        const uint8_t *__restrict__ tin = P.in + a0;
        const uint32_t ra = (uint32_t)(a - a0), rb = (uint32_t)(b - a0);
        const uint32_t nrel = (uint32_t)min(n - a0, (uint64_t)0xFFFFFFFFu);   // chunk end as an offset from a0 (clamped)

        // ---- first line start in [a, b): byte 0 of the chunk, or one past a '\n' at >= a-1
        uint32_t ls = rb;                                   // "none"
        if (VAR == 1) ls = resume;
        else if (a == 0) ls = 0;
        else {
            const uint32_t from = ra - 1, to = rb - 1;      // '\n' positions that give a start < b
            uint32_t wb = from & ~15u;
            while (wb < to) {
                const uint32_t pb = wb + 16 * lane;
                uint4 v = ld16(tin + pb);
                uint32_t m0 = eq_bytes(v.x, C_NL), m1 = eq_bytes(v.y, C_NL), m2 = eq_bytes(v.z, C_NL), m3 = eq_bytes(v.w, C_NL);
                clip4(m0, m1, m2, m3, pb, from, to);
                unsigned bal = __ballot_sync(FULL, (m0 | m1 | m2 | m3) != 0);
                if (bal) {
                    int src = __ffs(bal) - 1;
                    int k = first_byte(m0, m1, m2, m3);
                    k = __shfl_sync(FULL, k, src);
                    ls = wb + 16 * src + k + 1;
                    break;
                }
                wb += WINDOW;
            }
        }

        s_tag[wid] = 0;                                     // no line of this tile has used the exact-path counters yet
        TileState<OP> st;
        st.ls = ls; st.nlines = 0; st.out_bytes = 0; st.md_prev_end = ls; st.md_last_end = ls; st.md_add_nl = false; st.offlattice_lines = 0;
        if (VAR == 1) { st.nlines = P.tile_lines[tile]; st.out_bytes = (typename OutCount<OP>::type)P.tile_out[tile]; }
        const uint32_t lines_before = st.nlines;
        const bool finished = tile_lines<OP, VAR>(P, ws, lane, strip_cr, tile, a, a0, tin, rb, nrel, n, st);
        if (!finished) {
            // (VAR 0 of allele_freq_calc / hwe_tester only) the rest of the tile is the general kernel's
            if (lane == 0) { P.tile_lines[tile] = st.nlines; P.tile_out[tile] = st.out_bytes; P.tile_resume[tile] = st.ls; atomicAdd(&P.stats->n_unfinished, 1ULL); }
            VCFX_COUNT(C_LINES, st.nlines);
            __syncwarp();
            if (lane < CNT_SLOTS) {
                const unsigned int v = s_cnt[wid][lane];
                if (v) { s_cnt[wid][lane] = 0; atomicAdd(reinterpret_cast<unsigned long long *>(P.stats) + lane, (unsigned long long)v); }
            }
            __syncwarp();
            continue;
        }
        const uint32_t nlines = st.nlines;
        typename OutCount<OP>::type out_bytes = st.out_bytes;
        const uint32_t md_prev_end = st.md_prev_end, md_last_end = st.md_last_end;
        const bool md_add_nl = st.md_add_nl;

        if (!(OP == OP_AC && P.ac_pass)) VCFX_COUNT(C_LINES, VAR == 1 ? nlines - lines_before : nlines);
        if (OP == OP_MD || OP == OP_NR || OP == OP_PC || OP == OP_GQ) {
            const uint32_t tail = md_last_end - md_prev_end;
            if (lane == 0) {
                P.tail_start[tile] = (uint32_t)(a0 + md_prev_end - a);
                P.tail_len[tile] = tail | (md_add_nl ? 0x80000000u : 0u);
                P.tail_off[tile] = (uint32_t)out_bytes;
            }
            out_bytes += tail + (md_add_nl ? 1u : 0u);
        }
        if (lane == 0 && !(OP == OP_AC && P.ac_pass)) { P.tile_lines[tile] = nlines; P.tile_out[tile] = out_bytes; }
        // the write pass of a speculatively sized launch checks the sizes it was given
        if (OP == OP_AC && P.ac_pass && P.ac_spec && lane == 0 && (unsigned long long)out_bytes != P.tile_out[tile]) atomicOr(&P.stats->overflow, (unsigned long long)OV_AC_SPEC);
        __syncwarp();
        if (lane < CNT_SLOTS) {
            const unsigned int v = s_cnt[wid][lane];
            if (v) { s_cnt[wid][lane] = 0; atomicAdd(reinterpret_cast<unsigned long long *>(P.stats) + lane, (unsigned long long)v); }
        }
        __syncwarp();
    }
#undef VCFX_COUNT
    __syncwarp();
    {
        const unsigned int used = s_rec_used[wid];
        const unsigned long long slot = s_rec_base[wid] + lane;
        if ((unsigned int)lane >= used && (unsigned int)lane < REC_BLOCK && slot < P.rec_cap) P.recs[slot].tile = REC_INVALID;
    }
}

// ---------------------------------------------------------------------------------------
// K2a: exclusive scans over the tiles (output offsets, line numbers), one CTA.
// Also turns short-line keys (tile, index in tile) into 1-based line numbers.
// ---------------------------------------------------------------------------------------
constexpr uint32_t SCAN_BATCH = 8192;                            // tiles per pass: 8 per thread
constexpr uint32_t SCAN_SMEM_WORDS = SCAN_BATCH + SCAN_BATCH / 8;  // one pad word per 8 keeps thread-strided reads conflict-free
constexpr size_t SCAN_SMEM_BYTES = 2 * SCAN_SMEM_WORDS * sizeof(unsigned long long);
__device__ __forceinline__ uint32_t scan_pad(uint32_t i) { return i + (i >> 3); }

__global__ void __launch_bounds__(1024)
tile_scan_kernel(const KParams P) {
#ifdef VCFX_EMU
    unsigned long long *scan_smem = static_cast<unsigned long long *>(emu::dyn_smem());
#else
    extern __shared__ unsigned long long scan_smem[];
#endif
    unsigned long long *so = scan_smem, *sl = scan_smem + SCAN_SMEM_WORDS;
    __shared__ unsigned long long ws_o[32], ws_l[32];
    __shared__ unsigned long long carry_o, carry_l;
    const uint32_t tid = threadIdx.x, lane = tid & 31, w = tid >> 5, n_tiles = P.n_tiles;
    if (tid == 0) { carry_o = 0; carry_l = 0; }
    // A pass stages SCAN_BATCH tiles in shared memory with coalesced loads (all of them in flight
    // together), each thread scans its 8 consecutive tiles there, and the prefixes go back coalesced.
    for (uint32_t base = 0; base < n_tiles; base += SCAN_BATCH) {
        const uint32_t cnt = min(SCAN_BATCH, n_tiles - base);
#pragma unroll
        for (uint32_t j = 0; j < SCAN_BATCH / 1024; ++j) {
            const uint32_t i = j * 1024 + tid;
            so[scan_pad(i)] = i < cnt ? P.tile_out[base + i] : 0ULL;
            sl[scan_pad(i)] = i < cnt ? (unsigned long long)P.tile_lines[base + i] : 0ULL;
        }
        __syncthreads();
        unsigned long long vo = 0, vl = 0;
#pragma unroll
        for (uint32_t j = 0; j < 8; ++j) { vo += so[scan_pad(tid * 8 + j)]; vl += sl[scan_pad(tid * 8 + j)]; }
        unsigned long long io = vo, il = vl;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long to = __shfl_up_sync(FULL, io, o), tl2 = __shfl_up_sync(FULL, il, o);
            if ((int)lane >= o) { io += to; il += tl2; }
        }
        if (lane == 31) { ws_o[w] = io; ws_l[w] = il; }
        const unsigned long long c_o = carry_o, c_l = carry_l;
        __syncthreads();
        if (w == 0) {
            unsigned long long s_o = ws_o[lane], s_l = ws_l[lane];
            const unsigned long long so0 = s_o, sl0 = s_l;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long to = __shfl_up_sync(FULL, s_o, o), tl2 = __shfl_up_sync(FULL, s_l, o);
                if ((int)lane >= o) { s_o += to; s_l += tl2; }
            }
            ws_o[lane] = s_o - so0; ws_l[lane] = s_l - sl0;        // exclusive over warps
            if (lane == 31) { carry_o = c_o + s_o; carry_l = c_l + s_l; }
        }
        __syncthreads();
        unsigned long long ro = c_o + ws_o[w] + (io - vo), rl = c_l + ws_l[w] + (il - vl);
#pragma unroll
        for (uint32_t j = 0; j < 8; ++j) {
            const uint32_t k = scan_pad(tid * 8 + j);
            const unsigned long long a = so[k], b = sl[k];
            so[k] = ro; sl[k] = rl;
            ro += a; rl += b;
        }
        __syncthreads();
#pragma unroll
        for (uint32_t j = 0; j < SCAN_BATCH / 1024; ++j) {
            const uint32_t i = j * 1024 + tid;
            if (i < cnt) { P.tile_base[base + i] = so[scan_pad(i)]; P.line_base[base + i] = sl[scan_pad(i)]; }
        }
        __syncthreads();
    }
    __syncthreads();
    if (tid == 0) P.stats->bytes_out = carry_o * P.unit_bytes;
    __syncthreads();
    unsigned long long nev = P.stats->n_events;
    if (nev > P.ev_cap) nev = P.ev_cap;
    for (unsigned long long i = tid; i < nev && !P.ev_raw; i += 1024) {
        unsigned long long k = P.events[i];
        P.events[i] = P.line_base[k >> 32] + (k & 0xFFFFFFFFULL) + 1ULL;
    }
    if (tid == 0) {
        unsigned long long k = P.stats->first_short_key;
        P.stats->first_short_line = (k == ~0ULL) ? 0ULL : P.line_base[k >> 32] + (k & 0xFFFFFFFFULL) + 1ULL;
        unsigned long long ov = 0;
        if (P.stats->n_recs > P.rec_cap) ov |= OV_RECS;
        if (P.stats->bytes_out > P.out_cap) ov |= OV_OUTPUT;
        P.stats->overflow = ov;
    }
}

// ---------------------------------------------------------------------------------------
// K2b: rows -> text.  One thread per row record.
// ---------------------------------------------------------------------------------------
// AF / HWE: a warp takes 32 records; every lane builds the text of its row in a 64-byte slot of
// shared memory (prefix copy + number), then the warp writes the rows out one after the other with
// lane = byte, so a store instruction covers one row's contiguous bytes (1-2 sectors) instead of
// one byte in each of 32 rows.  Rows whose prefix did not fit the 32-byte side copy gather it from
// the input.  ALLELE_COUNT -a rows (long prefixes, few rows) keep one thread per row.
template <int OP>
__global__ void __launch_bounds__(256)
format_rows_kernel(const KParams P) {
    if (P.stats->overflow) return;
    const unsigned long long nrec = P.stats->n_recs;
    if (OP == OP_IX) {                                           // VCFX_indexer.cpp:291-303 / :397: CHROM \t POS \t FILE_OFFSET \n
        for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < nrec;
             i += (unsigned long long)gridDim.x * blockDim.x) {
            const Rec r = P.recs[i];
            if (r.tile == REC_INVALID) continue;
            uint8_t *o = P.out + P.tile_base[r.tile] + r.off_in_tile;
            const uint64_t line_off = (uint64_t)r.tile * P.tile_bytes + r.ls_rel;
            const uint8_t *src = P.in + line_off + r.a;
            for (uint32_t k = 0; k < r.prefix_len; ++k) o[k] = __ldg(src + k);
            o += r.prefix_len;
            *o++ = '\t'; o = put_dec64(o, (long long)(((unsigned long long)r.d << 32) | r.c));
            *o++ = '\t'; o = put_dec64(o, (long long)(P.file_offset + line_off)); *o = '\n';
        }
        return;
    }
    if (OP == OP_AC) {                                           // allele_counter.cpp:1454-1461
        for (unsigned long long i = blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x; i < nrec;
             i += (unsigned long long)gridDim.x * blockDim.x) {
            const Rec r = P.recs[i];
            if (r.tile == REC_INVALID) continue;
            uint8_t *o = P.out + P.tile_base[r.tile] + r.off_in_tile;
            const uint8_t *src = P.in + (uint64_t)r.tile * P.tile_bytes + r.ls_rel;
            for (uint32_t k = 0; k < r.prefix_len; ++k) o[k] = __ldg(src + k);
            o += r.prefix_len;
            for (uint32_t k = 0; k < r.d; ++k) *o++ = '\t';
            o = put_dec(o, (int)r.a); *o++ = '\t'; o = put_dec(o, (int)r.b); *o++ = '\t'; o = put_dec(o, (int)r.c); *o = '\n';
        }
        return;
    }
    __shared__ __align__(16) uint8_t rows_sm[8][32][64];
    const int lane = threadIdx.x & 31, wi = threadIdx.x >> 5;
    const unsigned long long warp0 = (blockIdx.x * (unsigned long long)blockDim.x + threadIdx.x) >> 5;
    const unsigned long long nwarps = ((unsigned long long)gridDim.x * blockDim.x) >> 5;
    for (unsigned long long base = warp0 * 32; base < nrec; base += nwarps * 32) {
        const unsigned long long i = base + lane;
        uint8_t *dst = nullptr; const uint8_t *src = nullptr;
        uint32_t plen = 0, tlen = 0;                             // prefix bytes, bytes of the row staged in shared memory
        bool gather = false;
        Rec r; r.tile = REC_INVALID;
        if (i < nrec) r = P.recs[i];
        if (r.tile != REC_INVALID) {
            dst = P.out + P.tile_base[r.tile] + r.off_in_tile;
            plen = r.prefix_len;
            uint8_t *slot = rows_sm[wi][lane];
            uint32_t at = 0;
            if (plen <= 32) {
                *reinterpret_cast<uint4 *>(slot) = *reinterpret_cast<const uint4 *>(P.rec_prefix + i * 32);
                *reinterpret_cast<uint4 *>(slot + 16) = *reinterpret_cast<const uint4 *>(P.rec_prefix + i * 32 + 16);
                at = plen;
            } else {
                gather = true;
                src = P.in + (uint64_t)r.tile * P.tile_bytes + r.ls_rel;
            }
            char num[24]; int nl;
            if (OP == OP_AF) {
                double v = af_value(r.a, r.b);
                nl = (P.mode == MODE_FILE) ? fmt_af_file(v, num) : fmt_af_stdin(v, num);
            } else {
                double pv = hwe_pvalue((int)r.a, (int)r.b, (int)r.c);
                nl = (P.mode == MODE_FILE) ? fmt_p_file(pv, num) : fmt_p_stdin(pv, num);
            }
            for (int k = 0; k < nl; ++k) slot[at + k] = (uint8_t)num[k];
            slot[at + nl] = '\n';
            tlen = at + nl + 1;
        }
        __syncwarp();
        const unsigned gm = __ballot_sync(FULL, gather);
#pragma unroll 4
        for (int j = 0; j < 32; ++j) {
            uint8_t *d = reinterpret_cast<uint8_t *>(__shfl_sync(FULL, (unsigned long long)dst, j));
            const uint32_t tl = __shfl_sync(FULL, tlen, j);
            if ((gm >> j) & 1u) {
                const uint8_t *sj = reinterpret_cast<const uint8_t *>(__shfl_sync(FULL, (unsigned long long)src, j));
                const uint32_t pl = __shfl_sync(FULL, plen, j);
                for (uint32_t k = lane; k < pl; k += 32) d[k] = __ldg(sj + k);
                d += pl;
            }
            if ((uint32_t)lane < tl) d[lane] = rows_sm[wi][j][lane];
            if ((uint32_t)lane + 32 < tl) d[lane + 32] = rows_sm[wi][j][lane + 32];
        }
        __syncwarp();
    }
}

// ---------------------------------------------------------------------------------------
// K2c (MISSING_DETECT): assemble the output.  One warp per work item; an item is either a
// rewritten line together with the verbatim bytes between it and the previous rewritten line
// of its tile, or the verbatim tail of a tile.
// ---------------------------------------------------------------------------------------
// warp-cooperative copy of n bytes, any alignment.  Large copies run on 128-bit stores to the
// 16-byte aligned middle of dst, each built from the two aligned 16-byte source blocks that straddle
// it (funnel shifts by the constant byte misalignment); the rest goes 32 bits / 1 byte at a time.
__device__ __forceinline__ void warp_copy_words(uint8_t *dst, const uint8_t *src, uint32_t n, int lane) {
    if (n == 0) return;
    const uint32_t head = min(n, (uint32_t)((4 - ((uintptr_t)dst & 3)) & 3));
    if (lane < (int)head) dst[lane] = __ldg(src + lane);
    dst += head; src += head; n -= head;
    const uint32_t nw = n >> 2;
    const uint32_t sh = 8u * (uint32_t)((uintptr_t)src & 3);
    const uint32_t *s4 = reinterpret_cast<const uint32_t *>(src - (sh >> 3));
    uint32_t *d4 = reinterpret_cast<uint32_t *>(dst);
    if (sh == 0) { for (uint32_t i = lane; i < nw; i += 32) d4[i] = __ldg(s4 + i); }
    else { for (uint32_t i = lane; i < nw; i += 32) d4[i] = __funnelshift_r(__ldg(s4 + i), __ldg(s4 + i + 1), sh); }
    const uint32_t done = nw << 2, rem = n - done;
    if (lane < (int)rem) dst[done + lane] = __ldg(src + done + lane);
}

template <int WS>   // WS = whole 32-bit words of misalignment between src and the 16-byte grid of dst
__device__ __forceinline__ uint4 realign16(const uint4 A, const uint4 B, uint32_t bs) {
    const uint32_t w[8] = {A.x, A.y, A.z, A.w, B.x, B.y, B.z, B.w};
    uint4 o;
    o.x = __funnelshift_r(w[WS], w[WS + 1], bs); o.y = __funnelshift_r(w[WS + 1], w[WS + 2], bs);
    o.z = __funnelshift_r(w[WS + 2], w[WS + 3], bs); o.w = __funnelshift_r(w[WS + 3], w[WS + 4], bs);
    return o;
}
// Four 512-byte rows per iteration: all the loads of an iteration are issued before its first store (the copy is bound by
// the latency of the loads, not by their number), and a 16-byte source block that two stores need is loaded once.
template <int WS>
__device__ __forceinline__ void copy16_loop(uint4 *__restrict__ d16, const uint4 *__restrict__ s16, uint32_t nq, uint32_t bs, int lane) {
    uint32_t i = lane;
    for (; i + 96 < nq; i += 128) {
        const uint4 A0 = __ldg(s16 + i), B0 = __ldg(s16 + i + 1), A1 = __ldg(s16 + i + 32), B1 = __ldg(s16 + i + 33);
        const uint4 A2 = __ldg(s16 + i + 64), B2 = __ldg(s16 + i + 65), A3 = __ldg(s16 + i + 96), B3 = __ldg(s16 + i + 97);
        d16[i] = realign16<WS>(A0, B0, bs); d16[i + 32] = realign16<WS>(A1, B1, bs);
        d16[i + 64] = realign16<WS>(A2, B2, bs); d16[i + 96] = realign16<WS>(A3, B3, bs);
    }
    for (; i < nq; i += 32) d16[i] = realign16<WS>(__ldg(s16 + i), __ldg(s16 + i + 1), bs);
}

__device__ __forceinline__ void warp_copy(uint8_t *dst, const uint8_t *src, uint32_t n, int lane) {
    if (n < 256) { warp_copy_words(dst, src, n, lane); return; }
    const uint32_t head = (uint32_t)((16 - ((uintptr_t)dst & 15)) & 15);
    warp_copy_words(dst, src, head, lane);
    dst += head; src += head; n -= head;
    const uint32_t nq = n >> 4;                                   // 16-byte stores
    const uint32_t mis = (uint32_t)((uintptr_t)src & 15);
    const uint4 *__restrict__ s16 = reinterpret_cast<const uint4 *>(src - mis);
    uint4 *__restrict__ d16 = reinterpret_cast<uint4 *>(dst);
    const uint32_t bs = 8u * (mis & 3u);
    if (mis == 0) {
        uint32_t i = lane;
        for (; i + 96 < nq; i += 128) {
            const uint4 a = __ldg(s16 + i), b = __ldg(s16 + i + 32), c = __ldg(s16 + i + 64), d = __ldg(s16 + i + 96);
            d16[i] = a; d16[i + 32] = b; d16[i + 64] = c; d16[i + 96] = d;
        }
        for (; i < nq; i += 32) d16[i] = __ldg(s16 + i);
    }
    else switch (mis >> 2) {                                      // the last block read ends < 32 B past src + n (pad)
        case 0: copy16_loop<0>(d16, s16, nq, bs, lane); break;
        case 1: copy16_loop<1>(d16, s16, nq, bs, lane); break;
        case 2: copy16_loop<2>(d16, s16, nq, bs, lane); break;
        default: copy16_loop<3>(d16, s16, nq, bs, lane); break;
    }
    warp_copy_words(dst + (nq << 4), src + (nq << 4), n - (nq << 4), lane);
}

__global__ void __launch_bounds__(256)
md_copy_kernel(const KParams P) {
    if (P.stats->overflow) return;
    const int lane = threadIdx.x & 31;
    const unsigned long long nrec = P.stats->n_recs, items = nrec + P.n_tiles;
    const unsigned long long nwarps = (unsigned long long)gridDim.x * (blockDim.x >> 5);
    for (unsigned long long it = (unsigned long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); it < items; it += nwarps) {
        if (it < nrec) {
            const Rec r = P.recs[it];
            if (r.tile == REC_INVALID) continue;
            const uint8_t *base = P.in + (uint64_t)r.tile * P.tile_bytes;
            uint8_t *o = P.out + P.tile_base[r.tile] + r.off_in_tile;
            const uint32_t gap = r.ls_rel - r.prefix_len;                // verbatim bytes before the line
            warp_copy(o, base + r.prefix_len, gap, lane);
            o += gap;
            const uint8_t *ln = base + r.ls_rel;
            if (r.b == NR_PLAIN) {                                       // nonref_filter: the line's content and a '\n', or nothing
                warp_copy(o, ln, r.c, lane);
                if (r.d > r.c && lane == 0) o[r.c] = '\n';
                continue;
            }
            warp_copy(o, ln, r.a, lane);                                 // up to INFO
            o += r.a;
            const uint8_t *info = ln + r.a;
            const bool replace = (r.b == 0) || (r.b == 1 && __ldg(info) == '.');
            uint32_t w = 0;
            if (!replace) {
                warp_copy(o, info, r.b, lane);
                w = r.b;
                if (__ldg(info + r.b - 1) != ';') { if (lane == 0) o[w] = ';'; ++w; }
            }
            if (lane < 19) o[w + lane] = (uint8_t)"MISSING_GENOTYPES=1"[lane];
            w += 19;
            o += w;
            const uint32_t rest = r.c - r.a - r.b;                       // from the tab after INFO to the content end
            warp_copy(o, info + r.b, rest, lane);
            if (lane == 0) o[rest] = '\n';
        } else {
            const uint32_t t = (uint32_t)(it - nrec);
            const uint32_t len = P.tail_len[t] & 0x7FFFFFFFu;
            uint8_t *o = P.out + P.tile_base[t] + P.tail_off[t];
            warp_copy(o, P.in + (uint64_t)t * P.tile_bytes + P.tail_start[t], len, lane);
            if ((P.tail_len[t] >> 31) && lane == 0) o[len] = '\n';
        }
    }
}

// ---------------------------------------------------------------------------------------
// inbreeding_calculator, second half: the sample-axis reduction
// ---------------------------------------------------------------------------------------
// K3a: row records -> rows in file order.  A warp per row: what a sample of each code contributes at this site
// (VCFX_inbreeding_calculator.cpp:596-625: global p, or p without the sample itself; boundary frequencies), and the row's
// codes copied next to those of the rows before and behind it, 32 samples to a panel.  A column the line does not have
// (and an empty last one) is IB_ABSENT in file mode — the sample then keeps the code of the last line that had it, the
// reference reuses its buffer (:574-588) — and has no genotype in stdin mode (:735-737).
__global__ void __launch_bounds__(256)
ib_rows_kernel(const KParams P) {
    if (P.stats->overflow) return;
    const unsigned long long R = P.stats->bytes_out;                 // rows of the chunk (tile_scan_kernel's total)
    const uint32_t npan = (P.n_sel + 31u) >> 5;
    if (R * 32ULL * npan > P.ib_panel_cap) {                         // (every thread sees the same: nobody writes)
        if (blockIdx.x == 0 && threadIdx.x == 0) atomicOr(&P.stats->overflow, (unsigned long long)OV_IB_PANELS);
        return;
    }
    const int lane = threadIdx.x & 31;
    const bool file_mode = P.mode == MODE_FILE;
    const unsigned long long nrec = P.stats->n_recs;
    const unsigned long long nwarps = (unsigned long long)gridDim.x * (blockDim.x >> 5);
    for (unsigned long long i = (unsigned long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < nrec; i += nwarps) {
        const Rec r = P.recs[i];
        if (r.tile == REC_INVALID) continue;
        const unsigned long long rank = P.tile_base[r.tile] + r.off_in_tile;
        // 16 codes per lane and step: aligned 32-bit loads around the (unaligned) source, one 16-byte store into the panel;
        // what is stored is 16 * code, the offset of the sample's entry in the row's table
        const uint8_t *src = P.ib_codes + ((((unsigned long long)r.tile * P.tile_bytes + r.ls_rel) & ~3ULL) + r.d);
        const uint32_t mis = (uint32_t)((uintptr_t)src & 3u), sh = 8u * mis;
        const uint32_t *s4 = reinterpret_cast<const uint32_t *>(src - mis);
        const uint32_t fill = file_mode ? IB_ABSENT : IB_NONE;
        uint32_t absent = (file_mode && r.c < P.n_sel) ? 1u : 0u;
        for (uint32_t s0 = 16u * (uint32_t)lane; s0 < (npan << 5); s0 += 512u) {
            uint32_t w[4];
            if (s0 + 16u <= r.c) {
                const uint32_t *q = s4 + (s0 >> 2);
                const uint32_t a0 = q[0], a1 = q[1], a2 = q[2], a3 = q[3], a4 = mis ? q[4] : 0u;      // (q[4] may lie behind the codes, never behind the arena's pad)
                w[0] = __funnelshift_r(a0, a1, sh); w[1] = __funnelshift_r(a1, a2, sh); w[2] = __funnelshift_r(a2, a3, sh); w[3] = __funnelshift_r(a3, a4, sh);
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    uint32_t v = 0;
#pragma unroll
                    for (int b = 0; b < 4; ++b) {
                        const uint32_t sidx = s0 + 4u * j + b;
                        const uint32_t c = sidx < r.c ? (uint32_t)src[sidx] : (sidx < P.n_sel ? fill : IB_NONE);
                        v |= c << (8 * b);
                    }
                    w[j] = v;
                }
            }
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t ab = eq_bytes(w[j], IB_ABSENT * 0x01010101u) >> 7;    // 0x01 in the bytes that are IB_ABSENT (an empty last column)
                if (file_mode) absent |= ab; else w[j] -= ab;        // ... which has no genotype in stdin mode
                w[j] <<= 4;
            }
            *reinterpret_cast<uint4 *>(P.ib_panels + ((unsigned long long)(s0 >> 5) * R + rank) * 32ULL + (s0 & 31u)) = make_uint4(w[0], w[1], w[2], w[3]);
        }
        const bool any_absent = __any_sync(FULL, absent != 0);
        if (lane == 0) {
            IbMeta m;
            for (int c = 0; c < 4; ++c) { m.e[c].x = 0.0; m.e[c].inc = 0; m.e[c].flag = 0; }
            m.e[IB_NONE].flag = any_absent ? 1u : 0u;
            const int alt_sum = (int)r.a, n_good = (int)r.b;
            if (n_good >= 2) {
                const double global_p = ddiv((double)alt_sum, dmul(2.0, (double)n_good));
                for (int c = 0; c < 3; ++c) {
                    const double freq = (P.flags & IB_F_GLOBAL) ? global_p : ddiv((double)(alt_sum - c), dmul(2.0, (double)(n_good - 1)));
                    if ((P.flags & IB_F_SKIP_BOUNDARY) && (freq <= 0.0 || freq >= 1.0)) { if (P.flags & IB_F_COUNT_BOUNDARY) m.e[c].inc = 1u; }
                    else { m.e[c].inc = (c == 1) ? 0x10001u : 1u; m.e[c].x = dmul(dmul(2.0, freq), dsub(1.0, freq)); }
                }
            }
            P.ib_rows[rank] = m;
        }
    }
}

// dosage_calculator, K2b: a warp per row record writes "CHROM \t POS \t ID \t REF \t ALT \t" and the dosages d,d,NA,.. of the line's
// sample columns from the codes the scan left (sample s: a ',' at 2s - 1 + (NAs before it) when it is not the first, its text behind)
__global__ void __launch_bounds__(256)
ds_rows_kernel(const KParams P) {
    __shared__ __align__(16) uint8_t s_stage[8][AC_STAGE + 32];      // the text is put together here and leaves in aligned 128-bit stores
    if (P.stats->overflow) return;
    const int lane = threadIdx.x & 31;
    uint8_t *stage = s_stage[threadIdx.x >> 5];
    const unsigned long long nrec = P.stats->n_recs;
    const unsigned long long nwarps = (unsigned long long)gridDim.x * (blockDim.x >> 5);
    for (unsigned long long i = (unsigned long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < nrec; i += nwarps) {
        const Rec r = P.recs[i];
        if (r.tile == REC_INVALID) continue;
        const unsigned long long line = (unsigned long long)r.tile * P.tile_bytes + r.ls_rel;
        uint8_t *o = P.out + P.tile_base[r.tile] + r.off_in_tile;
        if (P.tile_base[r.tile] + r.off_in_tile + r.prefix_len + r.b + 1u > P.out_cap) continue;        // (the scan has reported it)
        warp_copy(o, P.in + line, r.prefix_len, lane);
        o += r.prefix_len;
        if (r.c) { if (lane == 0) { o[0] = 'N'; o[1] = 'A'; o[2] = '\n'; } continue; }
        const uint8_t *codes = P.ib_codes + ((line & ~3ULL) + r.d);
        uint32_t na_before = 0, flushed = 0;
        uint32_t base = (uint32_t)((uintptr_t)o & 15u);              // the staged bytes sit at the destination's offset modulo 16
        for (uint32_t sb = 0; sb < r.a; sb += 128) {
          uint32_t c4[4];                                            // four steps' codes are under way before the first is used
#pragma unroll
          for (int u = 0; u < 4; ++u) { const uint32_t sx = sb + 32u * u + (uint32_t)lane; c4[u] = sx < r.a ? (uint32_t)codes[sx] : 0u; }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const uint32_t s0 = sb + 32u * u;
            if (s0 >= r.a) break;
            const uint32_t s = s0 + (uint32_t)lane;
            const bool in = s < r.a;
            const uint32_t c = c4[u];
            const bool na = in && c >= IB_NONE;
            const unsigned nb = __ballot_sync(FULL, na);
            if (in) {
                uint8_t *w = stage + base + (2u * s + na_before + (uint32_t)__popc(nb & ((1u << lane) - 1u)) - flushed);
                if (s) w[-1] = ',';
                if (na) { w[0] = 'N'; w[1] = 'A'; } else w[0] = (uint8_t)('0' + c);
            }
            na_before += (uint32_t)__popc(nb);
            const uint32_t s_end = min(s0 + 32u, r.a);
            const uint32_t written = 2u * s_end - 1u + na_before;    // text bytes up to (not including) the next sample's comma
            if (written - flushed + 96u + 16u > AC_STAGE) {
                __syncwarp();
                warp_flush_smem(o + flushed, stage + base, written - flushed, lane);
                __syncwarp();
                flushed = written; base = (uint32_t)((uintptr_t)(o + flushed) & 15u);
            }
          }
        }
        if (lane == 0) stage[base + (r.b - flushed)] = '\n';
        __syncwarp();
        warp_flush_smem(o + flushed, stage + base, r.b + 1u - flushed, lane);
        __syncwarp();
    }
}

// dosage_calculator matrix mode (VCFX_F_DS_MATRIX) and .bed mode (VCFX_F_DS_BED), K2b: a warp per row record.  The output
// is rows x 16 B of metadata {uint64 line offset, uint32 columns, uint32 flags} followed by rows of R bytes, row `rank` at
// 16 rows + rank R.  Matrix (R = W): int8 codes, 0 / 1 / 2 the dosage, -1 "NA" (IB_NONE, IB_ABSENT, every column of a line
// without a GT key), -2 no such column.  .bed (R = ceil(W / 4)): PLINK 1's two bits per sample, sample s at bits 2 (s & 3)
// of byte s >> 2: 00 dosage 2, 10 dosage 1, 11 dosage 0, 01 missing (the matrix's -1 and -2), 00 padding from W on.
// A row is put together in shared memory at the destination's offset modulo 16, DSM_STEP bytes at a time, and leaves in
// aligned 128-bit stores.  Every lane reads 16 samples' codes with five aligned 32-bit loads, funnel-shifted to the row's
// phase, so that a warp's loads cover consecutive words: they give 16 staged bytes of the matrix, or 4 of the .bed.
constexpr uint32_t DSM_STAGE = 2048, DSM_STEP = DSM_STAGE - 16;     // DSM_STEP is a multiple of 16: every step has the same phase
__device__ __forceinline__ uint32_t ds_matrix_word(uint32_t q, int s0, uint32_t ncols, bool no_gt) {
    const uint32_t na = ((q >> 2) | (q & (q >> 1))) & 0x01010101u;    // bytes holding IB_NONE (3) or IB_ABSENT (4)
    const uint32_t v = q | (na * 0xFFu);
    uint32_t w = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
        const int s = s0 + j;
        const uint32_t b = (s >= (int)ncols) ? 0xFEu : (no_gt ? 0xFFu : ((v >> (8 * j)) & 0xFFu));
        w |= b << (8 * j);
    }
    return w;
}
// 16 int8 codes, samples s0 .. s0 + 15
__device__ __forceinline__ uint4 ds_matrix_lane(const uint8_t *codes, int s0, int sh, uint32_t ncols, bool no_gt) {
    const int t0 = s0 - sh;                                                // sample of the aligned word that holds s0
    uint32_t w[5];
#pragma unroll
    for (int j = 0; j < 5; ++j) {
        const int t = t0 + 4 * j;
        w[j] = (!no_gt && t + 3 >= 0 && t < (int)ncols) ? ldw(codes + t) : 0u;
    }
    uint4 o;
    o.x = ds_matrix_word(__funnelshift_r(w[0], w[1], 8u * sh), s0, ncols, no_gt);
    o.y = ds_matrix_word(__funnelshift_r(w[1], w[2], 8u * sh), s0 + 4, ncols, no_gt);
    o.z = ds_matrix_word(__funnelshift_r(w[2], w[3], 8u * sh), s0 + 8, ncols, no_gt);
    o.w = ds_matrix_word(__funnelshift_r(w[3], w[4], 8u * sh), s0 + 12, ncols, no_gt);
    return o;
}
__device__ __forceinline__ uint32_t byte_mask(int n) {                // the low min(max(n, 0), 4) bytes
    return n >= 4 ? 0xFFFFFFFFu : (n <= 0 ? 0u : (1u << (8 * n)) - 1u);
}
// four codes (one byte each, samples s .. s + 3) -> one .bed byte.  Code 0 -> 11, 1 -> 10, 2 -> 00, 3 / 4 -> 01: per byte
// the low bit is b2 | !(b0 ^ b1) and the high bit !(b1 | b2) (codes are 0 .. 4).  Samples from ncols on are 01, from W on
// 00 (EDGE = false: all four are below ncols).  One multiply gathers the four 2-bit fields: the field of byte j lands at
// bits 24 + 2j, and the other partial products stay below bit 24 without overlapping.
template <bool EDGE>
__device__ __forceinline__ uint32_t ds_bed_byte(uint32_t q, int s, uint32_t ncols, uint32_t W) {
    uint32_t m = (((q >> 2) | ~(q ^ (q >> 1))) & 0x01010101u) | ((~((q >> 1) | (q >> 2)) & 0x01010101u) << 1);
    if (EDGE) {
        const uint32_t keep_c = byte_mask((int)ncols - s), keep_w = byte_mask((int)W - s);
        m = ((m & keep_c) | (0x01010101u & ~keep_c)) & keep_w;
    }
    return (m * 0x01041040u) >> 24;
}
// 4 .bed bytes, samples s0 .. s0 + 15 (s0 a multiple of 4)
template <bool EDGE>
__device__ __forceinline__ uint32_t ds_bed_lane(const uint8_t *codes, int s0, int sh, uint32_t ncols, uint32_t W) {
    const int t0 = s0 - sh;
    uint32_t w[5];
#pragma unroll
    for (int j = 0; j < 5; ++j) {
        const int t = t0 + 4 * j;
        w[j] = (!EDGE || (t + 3 >= 0 && t < (int)ncols)) ? ldw(codes + t) : 0u;
    }
    uint32_t o = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j)
        o |= ds_bed_byte<EDGE>(__funnelshift_r(w[j], w[j + 1], 8u * sh), s0 + 4 * j, ncols, W) << (8 * j);
    return o;
}
// One kernel for both layouts: the record walk, the metadata, the staging and the flush are the same, only the per-lane
// builder, its number of staged bytes and the row length differ (a compile-time choice: the matrix kernel's code is
// what it was).
template <bool BED>
__global__ void __launch_bounds__(256)
ds_matrix_kernel(const KParams P) {
    __shared__ __align__(16) uint8_t s_stage[8][DSM_STAGE];
    if (P.stats->overflow) return;
    const int lane = threadIdx.x & 31;
    uint8_t *stage = s_stage[threadIdx.x >> 5];
    const uint32_t W = P.n_sel;
    const uint32_t R = BED ? (W >> 2) + ((W & 3u) != 0u) : W;              // bytes of a row
    constexpr uint32_t LB = BED ? 4u : 16u;                                 // staged bytes a lane builds at a time
    const unsigned long long rows = P.stats->rows;
    uint8_t *const mat = P.out + 16ULL * rows;
    const unsigned long long nrec = P.stats->n_recs;
    const unsigned long long nwarps = (unsigned long long)gridDim.x * (blockDim.x >> 5);
    for (unsigned long long i = (unsigned long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); i < nrec; i += nwarps) {
        const Rec r = P.recs[i];
        if (r.tile == REC_INVALID) continue;
        const unsigned long long line = (unsigned long long)r.tile * P.tile_bytes + r.ls_rel;
        const unsigned long long rank = P.tile_base[r.tile] + r.off_in_tile;
        if (lane == 0) {
            const unsigned long long off = P.file_offset + line;
            *reinterpret_cast<uint4 *>(P.out + 16ULL * rank) = make_uint4((uint32_t)off, (uint32_t)(off >> 32), r.a, r.c);
        }
        if (R == 0) continue;
        uint8_t *const dst = mat + rank * (unsigned long long)R;              // past 2^32 for realistic shapes
        const uint8_t *const codes = P.ib_codes + ((line & ~3ULL) + r.d);
        const bool no_gt = r.c != 0;
        const uint32_t ncols = (BED && no_gt) ? 0u : min(r.a, W);           // .bed: a line without a GT key is all missing
        const int base = (int)((uintptr_t)dst & 15u);
        // staged byte k of a step holds row byte f + k - base: sample f + k - base (matrix) or 4 (f + k - base) (.bed)
        const int sh = BED ? (int)((uintptr_t)codes & 3u) : (int)(((uintptr_t)codes - (uintptr_t)base) & 3u);
        for (uint32_t f = 0; f < R; f += DSM_STEP) {
            const uint32_t n = min(R - f, DSM_STEP);
            for (uint32_t k = LB * (uint32_t)lane; k < (uint32_t)base + n; k += 32u * LB) {
                const int b0 = (int)(f + k) - base;
                if constexpr (BED) {
                    const int s0 = 4 * b0;
                    *reinterpret_cast<uint32_t *>(stage + k) = (s0 >= 0 && s0 + 16 <= (int)ncols) ? ds_bed_lane<false>(codes, s0, sh, ncols, W)
                                                                                                  : ds_bed_lane<true>(codes, s0, sh, ncols, W);
                } else {
                    *reinterpret_cast<uint4 *>(stage + k) = ds_matrix_lane(codes, b0, sh, ncols, no_gt);
                }
            }
            __syncwarp();
            warp_flush_smem(dst + f, stage + base, n, lane);
            __syncwarp();
        }
    }
}

// 16 bytes global -> shared without a register in between (LDGSTS); groups complete in order
__device__ __forceinline__ void cp_async16(void *smem, const void *gmem) {
#ifdef VCFX_EMU
    *reinterpret_cast<uint4 *>(smem) = *reinterpret_cast<const uint4 *>(gmem);
#else
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" :: "r"((uint32_t)__cvta_generic_to_shared(smem)), "l"(gmem) : "memory");
#endif
}
__device__ __forceinline__ void cp_async_commit() {
#ifndef VCFX_EMU
    asm volatile("cp.async.commit_group;" ::: "memory");
#endif
}
template <int N> __device__ __forceinline__ void cp_async_wait() {
#ifndef VCFX_EMU
    asm volatile("cp.async.wait_group %0;" :: "n"(N) : "memory");
#endif
}

// K3b: the sample-axis pass.  One thread per sample, one warp per panel of 32 samples: the warp streams its panel's codes and
// the rows' contribution tables through shared memory (IB_STAGES tiles of IB_TILE rows under way, cp.async) and every thread
// walks the chunk's sites IN FILE ORDER — the reference adds a sample's expectations in that order, in double, and any other
// order rounds differently.  Per site and sample: one table look-up and one add (a sample that adds nothing adds +0.0).
// Chunks are applied strictly in order: a chunk whose predecessor has not been applied yet (it is being run again) is left
// alone and reported by ib_finish_kernel.
constexpr int IB_TILE = 128, IB_STAGES = 3;
static_assert((IB_TILE - 16) % 16 == 0, "the row loop of ib_accumulate_kernel takes 8 + 16 n + 8 rows");
__global__ void __launch_bounds__(32)
ib_accumulate_kernel(const KParams P) {
    __shared__ __align__(16) uint8_t sm_codes[IB_STAGES][IB_TILE * 32];
    __shared__ __align__(16) IbMeta sm_meta[IB_STAGES][IB_TILE];
    if (P.stats->overflow) return;
    IbState &S = *P.ib;
    if (S.seq != P.ib_seq) return;                                   // applied already (a re-run), or not this chunk's turn yet
    const uint32_t lane = threadIdx.x, s = blockIdx.x * 32u + lane;
    const bool live = s < P.n_sel;
    const unsigned long long R = P.stats->bytes_out;
    const bool fresh = P.ib_first != 0;
    double sum = (fresh || !live) ? 0.0 : S.sum[s];
    unsigned long long het = (fresh || !live) ? 0ULL : S.het[s];
    unsigned int used = (fresh || !live) ? 0u : S.used[s];
    uint32_t last = (fresh || !live) ? 0u : 16u * (uint32_t)S.last[s];            // (as an entry offset, like the panel bytes)
    const uint8_t *pan = P.ib_panels + (unsigned long long)blockIdx.x * R * 32ULL;
    const unsigned long long ntiles = (R + IB_TILE - 1) / IB_TILE;
    auto issue = [&](unsigned long long t) {
        if (t < ntiles) {
            const int st = (int)(t % IB_STAGES);
            const uint32_t nrows = (uint32_t)min((unsigned long long)IB_TILE, R - t * IB_TILE);
            const uint8_t *gc = pan + t * (IB_TILE * 32ULL);
            const uint8_t *gm = reinterpret_cast<const uint8_t *>(P.ib_rows) + t * (IB_TILE * (unsigned long long)sizeof(IbMeta));
            for (uint32_t q = lane; q < nrows * 2u; q += 32) cp_async16(&sm_codes[st][q * 16u], gc + q * 16u);
            for (uint32_t q = lane; q < nrows * 4u; q += 32) cp_async16(reinterpret_cast<uint8_t *>(&sm_meta[st][0]) + q * 16u, gm + q * 16u);
        }
        cp_async_commit();                                           // (an empty group keeps the count of groups in step)
    };
    // one row: the sample's entry offset, its entry (one 16-byte load), one add to the chain, one to the counters
    struct Ent { double x; uint32_t inc; };
    auto entry = [](const uint8_t *row, uint32_t off) {
        union { uint4 v; IbEntry e; } u;
        u.v = *reinterpret_cast<const uint4 *>(row + off);
        Ent e; e.x = u.e.x; e.inc = u.e.inc; return e;
    };
    for (int j = 0; j < IB_STAGES - 1; ++j) issue((unsigned long long)j);
    for (unsigned long long t = 0; t < ntiles; ++t) {
        issue(t + IB_STAGES - 1);
        cp_async_wait<IB_STAGES - 1>();
        __syncwarp();
        const int st = (int)(t % IB_STAGES);
        const uint32_t nrows = (uint32_t)min((unsigned long long)IB_TILE, R - t * IB_TILE);
        const uint8_t *cs = &sm_codes[st][lane];
        const uint8_t *ms = reinterpret_cast<const uint8_t *>(&sm_meta[st][0]);
        // does any row of the tile lack a column?  (file mode only; the sample then keeps its last code)
        uint32_t fl = 0;
        for (uint32_t k = lane; k < nrows; k += 32) fl |= sm_meta[st][k].e[IB_NONE].flag;
        const bool absent = __any_sync(FULL, fl != 0);
        uint32_t cnt = 0;
        // The adds of one sample form a chain; the look-ups of the NEXT eight rows are written between them so that the
        // in-order issue has something to do while an add is under way.
        uint32_t k = 0;
        if (!absent && nrows == IB_TILE) {
            Ent xa[8], xb[8];                                          // (two sets taking turns: no register is copied)
#pragma unroll
            for (int j = 0; j < 8; ++j) xa[j] = entry(ms + j * 64, cs[j * 32]);
#pragma unroll 1
            for (k = 8; k + 16 <= IB_TILE; k += 16) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    xb[j] = entry(ms + (k + j) * 64, cs[(k + j) * 32]);
                    sum = dadd(sum, xa[j].x); cnt += xa[j].inc;
                }
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    xa[j] = entry(ms + (k + 8 + j) * 64, cs[(k + 8 + j) * 32]);
                    sum = dadd(sum, xb[j].x); cnt += xb[j].inc;
                }
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) {                            // rows IB_TILE-8 .. IB_TILE-1 come in while the set before them is added
                xb[j] = entry(ms + (IB_TILE - 8 + j) * 64, cs[(IB_TILE - 8 + j) * 32]);
                sum = dadd(sum, xa[j].x); cnt += xa[j].inc;
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) { sum = dadd(sum, xb[j].x); cnt += xb[j].inc; }
            last = cs[(IB_TILE - 1) * 32];
            k = IB_TILE;
        }
        for (; k < nrows; ++k) {
            uint32_t off = cs[k * 32u];
            off = (off == 16u * IB_ABSENT) ? last : off; last = off;
            const Ent e = entry(ms + k * 64, off);
            sum = dadd(sum, e.x); cnt += e.inc;
        }
        used += cnt & 0xFFFFu; het += cnt >> 16;
        __syncwarp();
    }
    if (live) { S.sum[s] = sum; S.het[s] = het; S.used[s] = used; S.last[s] = (uint8_t)(last >> 4); }
    if (s == 0) S.variants = (fresh ? 0ULL : S.variants) + P.stats->rows;
}

// K3c: closes the chunk (order guard) and, behind the last chunk, writes the rows "name \t F \n" (:641-667): NA without a
// used site, 1.000000 when nothing was expected, else 1 - observed / expected with six truncated decimals (:205-240).
__global__ void __launch_bounds__(1024)
ib_finish_kernel(const KParams P) {
    __shared__ unsigned long long s_warp[32];
    __shared__ unsigned long long s_carry;
    __shared__ int s_state;
    const uint32_t tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    IbState &S = *P.ib;
    if (tid == 0) {
        int st = 0;                                                  // 0 = go on, 1 = leave
        if (P.stats->overflow) st = 1;
        else if (S.seq == P.ib_seq) S.seq = P.ib_seq + 1;            // this launch applied the chunk
        else if (S.seq != P.ib_seq + 1) { P.stats->overflow = OV_IB_ORDER; st = 1; }   // an earlier chunk is being run again: so will this one
        if (st || !P.is_final) P.stats->bytes_out = 0;
        s_state = st; s_carry = 0;
    }
    __syncthreads();
    if (s_state || !P.is_final) return;
    const bool none_used = S.variants == 0;
    for (uint32_t base = 0; base < P.n_sel; base += 1024) {
        const uint32_t s = base + tid;
        char num[40]; uint32_t nl = 0, name_n = 0;
        if (s < P.n_sel) {
            name_n = P.name_off[s + 1] - P.name_off[s];              // the name and its tab
            if (none_used || S.used[s] == 0) { num[0] = 'N'; num[1] = 'A'; nl = 2; }
            else {
                const double e = S.sum[s];
                if (e <= 0.0) { const char one[] = "1.000000"; for (int k = 0; k < 8; ++k) num[k] = one[k]; nl = 8; }
                else nl = (uint32_t)fmt_p_file(dsub(1.0, ddiv((double)S.het[s], e)), num);
            }
        }
        const unsigned long long len = s < P.n_sel ? (unsigned long long)name_n + nl + 1u : 0ULL;
        unsigned long long incl = len;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const unsigned long long t = __shfl_up_sync(FULL, incl, o); if ((int)lane >= o) incl += t; }
        if (lane == 31) s_warp[wid] = incl;
        __syncthreads();
        if (wid == 0) {
            unsigned long long v = s_warp[lane], iv = v;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) { const unsigned long long t = __shfl_up_sync(FULL, iv, o); if ((int)lane >= o) iv += t; }
            s_warp[lane] = iv - v;
        }
        __syncthreads();
        const unsigned long long off = s_carry + s_warp[wid] + incl - len;
        if (s < P.n_sel && off + len <= P.text_cap) {
            uint8_t *o = P.out + off;
            const uint8_t *nm = P.names + P.name_off[s];
            for (uint32_t k = 0; k < name_n; ++k) o[k] = nm[k];
            for (uint32_t k = 0; k < nl; ++k) o[name_n + k] = (uint8_t)num[k];
            o[name_n + nl] = '\n';
        }
        __syncthreads();
        if (tid == 1023) s_carry = off + len;
        __syncthreads();
    }
    if (tid == 0) {
        P.stats->bytes_out = s_carry;
        if (s_carry > P.text_cap) P.stats->overflow = OV_OUTPUT;
    }
}

// hwe_pvalue() of vcfx_numfmt.cuh over an array of (homRef, het, homAlt) triples: the measuring stick for the one
// operation of the path that is not bit-identical by construction (exp)
__global__ void __launch_bounds__(256)
hwe_pvalue_kernel(const int32_t *__restrict__ counts, size_t n, double *__restrict__ out) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        out[i] = hwe_pvalue(counts[3 * i], counts[3 * i + 1], counts[3 * i + 2]);
}

}  // namespace vcfx
