/*
 * vcfx_cuda.h — C ABI of libvcfx_cuda, the B200 (sm_100a) implementation of VCFX's shared
 * hot path:  VCF bytes -> line/field scan -> FORMAT/GT parse -> per-variant reduce -> text.
 *
 * The reference (jorgeMFS/VCFX v1.1.4) has no library boundary for this path: each tool
 * carries a private copy of the same loop.  Every entry point below therefore names the
 * reference code it stands in for; INTEGRATION.md shows the change a maintainer makes in
 * each tool's main() to call it.
 *
 *   reference loop being replaced                               op
 *   ----------------------------------------------------------  ------------------------
 *   VCFX_variant_counter.cpp:317-389 countVariantsMmap,         VCFX_OP_VARIANT_COUNT
 *     :204-221 countVariants, :223-290 countVariantsGzip
 *   VCFX_allele_freq_calc.cpp:342-472 processMmap,              VCFX_OP_ALLELE_FREQ
 *     :477-557 processStdin
 *   VCFX_hwe_tester.cpp:455-559 performHWE_Mmap,                VCFX_OP_HWE
 *     :565-608 performHWE_Stdin
 *   VCFX_missing_detector.cpp:450-589 processMmapZeroCopy,      VCFX_OP_MISSING_DETECT
 *     :860-911 detectMissingGenotypes
 *   VCFX_allele_counter.cpp:550-642 processChunk (+786-950),    VCFX_OP_ALLELE_COUNT
 *     :1122-1260 countAllelesStream, :1266-1468 countAllelesUnified
 *
 * The "mode" selects which of the two behaviours of a tool is reproduced: the reference
 * formats numbers and skips lines differently when it mmaps a file (-i FILE) and when it
 * reads stdin (SURVEY.md finding 1).  Output is byte-identical to the reference tool run in
 * that mode; the fixed header row of each tool is written by the caller, not by the library.
 *
 * Conventions: plain pointers and sizes, no C++ types, no exceptions; every function returns
 * 0 or a negative vcfx_err; the library never prints and never falls back to the CPU
 * (no device => VCFX_E_NO_DEVICE).  One context drives one GPU; a context is used by one
 * thread at a time; contexts are independent, so one process can hold one per GPU.
 */
#ifndef VCFX_CUDA_H
#define VCFX_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VCFX_CUDA_ABI_VERSION 3

typedef struct vcfx_ctx vcfx_ctx;

typedef enum {
    VCFX_OP_VARIANT_COUNT  = 0,
    VCFX_OP_ALLELE_FREQ    = 1,
    VCFX_OP_HWE            = 2,
    VCFX_OP_MISSING_DETECT = 3,
    VCFX_OP_ALLELE_COUNT   = 4,
    VCFX_OP_PHASE_CHECK    = 7,   /* VCFX_phase_checker.cpp:470-558 filterPhaseCheckedMmap, :563-650 processVCF (SURVEY §8 f2); vcfx_cuda_short_lines
                                     then returns, per dropped line, (offset of the line in the chunk << 2 | reason): 0 unphased, 1 before
                                     the header, 2 fewer than ten columns, 3 no GT key */
    VCFX_OP_INBREEDING     = 8,   /* VCFX_inbreeding_calculator.cpp:456-668 calculateInbreedingMmap, :670-826 calculateInbreedingStdin
                                     (SURVEY §8 f3, a sample-axis reduction): cfg.n_sel / sel_names / sel_name_off = the samples of the
                                     "#CHROM" line in column order (sel_col is not used); the per-sample sums live in the context from
                                     chunk to chunk and the text ("name \t F \n" per sample) comes with the chunk submitted as final */
    VCFX_OP_GENOTYPE_QUERY = 9,   /* VCFX_genotype_query.cpp:433-517 genotypeQueryMmap, :527-614 genotypeQueryStream (SURVEY §8 f2): cfg.sel_names =
                                     the -g argument, cfg.n_sel = its length in bytes (< 64); VCFX_F_GQ_STRICT = --strict.  The caller
                                     ends the input in front of a data line that comes before the "#CHROM" line and, in stdin mode,
                                     holds back '#' lines until a data line follows; vcfx_cuda_short_lines returns (offset << 2 | 2)
                                     for every line that earns "skipping line with <9 fields" */
    VCFX_OP_DOSAGE         = 10,  /* VCFX_dosage_calculator.cpp:375-591 processFileMmap, :209-366 calculateDosage (SURVEY §8 f2): a row
                                     "CHROM..ALT \t d,d,NA,.." per data line with ten columns; stats.short_lines = lines with fewer
                                     (one warning each).  The caller prints the header row and ends the run at a data line that
                                     comes before the "#CHROM" line.
                                     VCFX_F_DS_MATRIX: the same rows as a matrix instead of text, cfg.n_sel = W sample columns
                                     (0 is valid).  Output of a launch / chunk: rows x vcfx_ds_row, then at byte 16 x rows the
                                     rows x W int8 codes, row-major: 0 / 1 / 2 the dosage the text prints, -1 its "NA" (every
                                     column of a line without a GT key too), -2 for a column s >= n_cols the line does not have.
                                     Columns beyond W are dropped (n_cols keeps the true count; stats.flagged counts such rows).
                                     stats.rows = rows, stats.bytes_out = rows x (16 + W); short_lines, data_lines as for the text.
                                     run_device wants d_out 16-byte aligned (else VCFX_E_INVALID).
                                     VCFX_F_DS_BED: the same rows as PLINK 1 .bed rows (variant-major), W = cfg.n_sel (0 is
                                     valid), B = ceil(W / 4) bytes a row.  Output: rows x vcfx_ds_row, then at byte 16 x rows
                                     the rows x B packed bytes, row-major; stats.bytes_out = rows x (16 + B), stats.flagged
                                     as for the matrix.  Sample s sits in byte s >> 2 at bits 2 (s & 3) and 2 (s & 3) + 1, with
                                     A1 = ALT and A2 = REF: matrix code 2 -> 00 (hom A1), 1 -> 10 (het), 0 -> 11 (hom A2),
                                     -1 and -2 -> 01 (missing), s >= W -> 00 (padding).  A multi-allelic line keeps the
                                     dosage rule (every allele > 0 counts): A1 stands for "any non-REF allele".  Cannot be
                                     combined with VCFX_F_DS_MATRIX (VCFX_E_INVALID from create); run_device wants d_out
                                     16-byte aligned */
    VCFX_OP_INDEX          = 6,   /* VCFX_indexer.cpp:205-322 createVCFIndexMmap, :329-443 createVCFIndex (SURVEY §8 f4) */
    VCFX_OP_NONREF_FILTER  = 5    /* VCFX_nonref_filter.cpp:458-548 filterNonRefMmap, :553-631 filterNonRef (SURVEY §8 f2) */
} vcfx_op;

typedef enum {
    VCFX_MODE_FILE  = 0,   /* semantics of `tool -i FILE` (mmap path of the reference)  */
    VCFX_MODE_STDIN = 1    /* semantics of `tool < FILE`  (getline path of the reference) */
} vcfx_mode;

typedef enum {
    VCFX_OK               =  0,
    VCFX_E_INVALID        = -1,   /* bad argument / call order                         */
    VCFX_E_NO_DEVICE      = -2,   /* no usable CUDA device: there is no CPU fallback   */
    VCFX_E_CUDA           = -3,   /* a CUDA call failed (see vcfx_cuda_last_error)     */
    VCFX_E_NOMEM          = -4,
    VCFX_E_BUSY           = -5,   /* every pipeline slot is in flight: drain an output */
    VCFX_E_EMPTY          = -6,   /* nothing in flight                                 */
    VCFX_E_OUTPUT_TOO_BIG = -7,   /* one chunk's output exceeds the output capacity    */
    VCFX_E_UNSUPPORTED    = -8
} vcfx_err;

/* variants of an op (cfg.flags): the bits are per op */
#define VCFX_F_GQ_STRICT         0x01u  /* genotype_query --strict: byte-for-byte comparison (:277-279)               */
#define VCFX_F_IB_GLOBAL         0x01u  /* inbreeding_calculator --freq-mode global (:596-604)                 */
#define VCFX_F_IB_SKIP_BOUNDARY  0x02u  /* --skip-boundary (:614-620)                                          */
#define VCFX_F_IB_COUNT_BOUNDARY 0x04u  /* --count-boundary-as-used                                            */
#define VCFX_F_AC_AGGREGATE   0x01u  /* -a: one row per variant (countAllelesUnified :1440-1461)          */
#define VCFX_F_AC_BINARY      0x02u  /* -b: int8 {ref,alt} per selected sample (:1444-1449)               */
#define VCFX_F_DS_MATRIX      0x01u  /* dosage_calculator: int8 variants x samples matrix instead of text (see VCFX_OP_DOSAGE) */
#define VCFX_F_DS_BED         0x02u  /* dosage_calculator: PLINK 1 .bed rows, 2 bits a call, instead of text (see VCFX_OP_DOSAGE) */
#define VCFX_F_AC_FORWARD     0x04u  /* stdin / unified column walk: forward only, stop at the first absent
                                        column (:1222-1229, :1416-1423); without it: processChunk's random
                                        access with 0/0 padding and int8 storage (:610-627)               */

typedef struct {
    int32_t  device;          /* CUDA device ordinal                                            */
    int32_t  op;              /* vcfx_op                                                        */
    int32_t  mode;            /* vcfx_mode                                                      */
    uint32_t flags;
    size_t   chunk_bytes;     /* capacity of one pinned input slot (0 = 64 MiB)                 */
    size_t   out_bytes;       /* capacity of one output slot (0 = sized from op and chunk)      */
    int32_t  n_slots;         /* chunks in flight, 1..8 (0 = 3)                                 */
    int32_t  tile_bytes;      /* bytes of input owned by one warp, multiple of 512 (0 = chosen per
                                 launch from the chunk size, 32..256 KiB)                       */
    void    *stream;          /* optional cudaStream_t for the device-resident entry point      */
    /* VCFX_OP_ALLELE_COUNT: the selected sample columns, in output order */
    uint32_t        n_sel;          /* number of selected samples                               */
    const uint32_t *sel_col;        /* [n_sel] 0-based sample column (field 9 + col)            */
    const char     *sel_names;      /* concatenated names, each followed by '\t'                */
    const uint32_t *sel_name_off;   /* [n_sel + 1] offsets into sel_names                       */
} vcfx_cfg;

/* VCFX_OP_DOSAGE with VCFX_F_DS_MATRIX or VCFX_F_DS_BED: the metadata of one row (16 bytes, the rows in file order) */
typedef struct vcfx_ds_row {
    uint64_t line_offset;      /* offset of the row's line in the whole input: info.file_offset + offset in the chunk */
    uint32_t n_cols;           /* sample columns of the line (may exceed W)                                           */
    uint32_t flags;            /* bit 0: the line has no GT key (the text prints "NA" alone; every code is -1)         */
} vcfx_ds_row;

/* what the caller knows about the chunk it submits */
typedef struct {
    uint64_t data_valid_from;  /* ALLELE_FREQ: data lines starting below this chunk offset precede
                                  the first "#CHROM" line and are skipped with a warning
                                  (allele_freq_calc.cpp:382-386); 0 = header already seen       */
    int32_t  is_final;         /* last chunk: the final line may lack its '\n'                   */
    int32_t  reserved;
    uint64_t file_offset;      /* ABI 2: offset of the chunk's first byte in the whole input (VCFX_OP_INDEX prints absolute offsets) */
    uint64_t format_cache_from;/* ABI 3, VCFX_OP_PHASE_CHECK in file mode: data lines starting below this chunk offset are checked
                                  while the reference's FORMAT cache is still ("", GT index 0) — no line with a non-empty FORMAT
                                  column was looked at before them — so an empty FORMAT column means "GT is the first key" there
                                  (VCFX_phase_checker.cpp:486-488, :313-316); 0 = a non-empty FORMAT was already seen */
} vcfx_chunk_info;

typedef struct {
    uint64_t bytes_in;
    uint64_t bytes_out;
    uint64_t lines;            /* lines in the chunk (a final unterminated line counts)          */
    uint64_t data_lines;       /* lines the tool treats as records                               */
    uint64_t rows;             /* rows written / variants counted                                */
    uint64_t flagged;          /* MISSING_DETECT: lines rewritten                                */
    uint64_t pre_header;       /* ALLELE_FREQ: data lines before #CHROM (one warning each)       */
    uint64_t short_lines;      /* VARIANT_COUNT: <8 columns; ALLELE_FREQ stdin: <9 fields        */
    uint64_t first_short_line; /* 1-based line number inside the chunk of the first one, 0=none  */
    uint64_t n_events;         /* short-line events recorded (see vcfx_cuda_short_lines)         */
    uint64_t dots_terminated;  /* MISSING_DETECT: '\n'-terminated lines with a '.' after the 9th
                                  tab (the reference's pre-scan, missing_detector.cpp:347-369)   */
    uint64_t last_unterminated_flagged; /* MISSING_DETECT: length of the rewritten final line when
                                  that line had no '\n' and was flagged, else 0                   */
    float    kernel_ms;        /* device time of this chunk's kernels (CUDA events)              */
    float    reserved;
} vcfx_chunk_stats;

int  vcfx_cuda_abi_version(void);
int  vcfx_cuda_device_count(int *n);
const char *vcfx_cuda_strerror(int err);
const char *vcfx_cuda_last_error(const vcfx_ctx *ctx);   /* text of the last CUDA failure */

int  vcfx_cuda_create(const vcfx_cfg *cfg, vcfx_ctx **out);
void vcfx_cuda_destroy(vcfx_ctx *ctx);

/* ---- streaming path: host buffers in, host text out (replaces the per-line loops) --------
 * acquire_input  : a pinned buffer of cfg.chunk_bytes to fill (read(2)/memcpy straight in).
 * submit         : nbytes of it become a chunk.  A chunk must start at a line start and,
 *                  unless info->is_final, end with '\n'.  Asynchronous: H2D copy, kernels and
 *                  the D2H copy of the text run on the context's streams.
 * next_output    : blocks for the OLDEST chunk in flight and returns its text (order
 *                  preserving).  The pointer stays valid until the next acquire/submit.     */
int vcfx_cuda_acquire_input(vcfx_ctx *ctx, char **buf, size_t *cap);
int vcfx_cuda_submit(vcfx_ctx *ctx, size_t nbytes, const vcfx_chunk_info *info);
/* submit_shared  : run THIS context's op on the chunk most recently submitted to `primary` (same
 *                  device), reading the bytes that are already in the primary's device slot: one
 *                  upload feeds several tools (e.g. variant_counter next to allele_freq_calc).
 *                  Drain this context before the primary takes `n_slots` further chunks; a chunk
 *                  whose output outgrows its slot is re-run and must still find the bytes there.  */
int vcfx_cuda_submit_shared(vcfx_ctx *ctx, vcfx_ctx *primary, const vcfx_chunk_info *info);
int vcfx_cuda_next_output(vcfx_ctx *ctx, const char **text, size_t *n, vcfx_chunk_stats *stats);
/* set_line_hint  : typical bytes per data line (0 = let the library measure it on the host buffers it
 *                  is given).  A tile's owner re-reads about one line around every tile border, so
 *                  inputs with very long lines (FORMAT GT:AD:DP:GQ:PL x thousands of samples) get
 *                  larger tiles.  Only needed by run_device callers, whose bytes the host never sees:
 *                  the reference tools have no such knob, it changes no result.                   */
int vcfx_cuda_set_line_hint(vcfx_ctx *ctx, size_t line_bytes);
/* submit_host    : like acquire + memcpy + submit, but the chunk is copied to the device straight
 *                  from the caller's buffer (an mmap'ed/pinned region gives the full PCIe rate).
 *                  The buffer must stay unchanged until next_output has returned this chunk.   */
int vcfx_cuda_submit_host(vcfx_ctx *ctx, const void *host, size_t nbytes, const vcfx_chunk_info *info);
int vcfx_cuda_in_flight(const vcfx_ctx *ctx);

/* 1-based line numbers (inside the chunk last returned by next_output) of lines with too few
 * columns, ascending; at most `cap` are copied, the total is stats.n_events
 * (variant_counter.cpp:373-380 prints one message per such line). */
int vcfx_cuda_short_lines(vcfx_ctx *ctx, uint64_t *line_no, size_t cap, size_t *n);

/* ---- device-resident path: for callers that already hold the bytes in HBM -----------------
 * d_in must be 16-byte aligned and readable for nbytes + VCFX_DEVICE_PAD bytes (the library
 * writes '\n' into the first 64 bytes of that pad; the kernels keep up to eight 512-byte windows
 * in flight per warp and so read up to 4,100 bytes past the window that holds the last byte).
 * d_out receives the text (out_cap bytes).
 * Runs on cfg.stream (or the context's own stream), asynchronously; calls may be queued back to
 * back; vcfx_cuda_sync waits and fills stats of the LAST one.  Used by bench.py for the
 * kernel-only figure. */
#define VCFX_DEVICE_PAD 8192
int vcfx_cuda_run_device(vcfx_ctx *ctx, void *d_in, size_t nbytes, const vcfx_chunk_info *info,
                         void *d_out, size_t out_cap);
int vcfx_cuda_sync(vcfx_ctx *ctx, vcfx_chunk_stats *stats);

/* hwe_tester's p-value (VCFX_hwe_tester.cpp:278-315 chi2_pvalue_1df + calculateHWE_chisq) evaluated ON THE DEVICE
 * for n (hom_ref, het, hom_alt) triples: counts[3*i .. 3*i+2] -> pvalues[i] (host arrays).  It is the same device
 * code the row formatter runs; exported so that the difference to the reference's libm arithmetic can be measured
 * and reported (BASELINE.json: any HWE p-value difference must stay within 1e-12 relative and be reported). */
int vcfx_cuda_hwe_pvalues(int device, const int32_t *counts, size_t n, double *pvalues);

/* ---- pairwise relatedness: KING-robust kinship counts from PLINK 1 .bed rows, on the tensor cores ------------------
 * An accumulator of its own (no vcfx_cfg, no op).  Each .bed row (VCFX_F_DS_BED's layout: sample s at bits 2 (s & 3) of
 * byte s >> 2) gives every sample four 0/1 indicators for the variant:
 *
 *     code  meaning                                                    plane
 *     11    hom A2 (REF/REF)                                           A
 *     10    het                                                        H
 *     00    hom A1 (ALT/ALT; on a multi-allelic line "any non-REF")    B
 *     01    missing                                                    none
 *
 * and C = A | H | B ("called").  The bits of samples s >= n_samples in a row's last byte are padding and are ignored
 * whatever their value (a .bed writes 00 there, which would read as hom A1).  Over all rows added, for every ordered pair
 * (i, j), four uint32 counts:
 *     CC[i][j]  both called (NSNP)                HH[i][j]  both het (HETHET)
 *     AB[i][j]  i hom A2 and j hom A1, so IBS0(i, j) = AB[i][j] + AB[j][i]
 *     HC[i][j]  i het and j called, so HET1 = HC[i][j] and HET2 = HC[j][i]
 * KING's between-family robust kinship for i < j, in double, is then
 *     kinship = 0.5 - (HET1 + HET2 - 2 HETHET + 4 IBS0) / (4.0 * min(HET1, HET2))
 * (the division first, then the subtraction), NA when min(HET1, HET2) = 0.  The numerator is the sum of (x_i - x_j)^2 over
 * the jointly called sites, so the het counts are restricted to jointly called sites; duplicates give exactly 0.5.
 * Haploid and multi-allelic calls count as the .bed encodes them.  The counts are integer products (int8 MMAs with s32
 * accumulation), so they are exact; a run takes at most UINT32_MAX rows in all.
 * Memory on the device: the four planes (at most about 1 GiB), one slab of rows (vcfx_cuda_king_slab_rows of them) and
 * 16 x s_pad^2 bytes of counts, s_pad = n_samples rounded up to 256. */
typedef struct vcfx_king vcfx_king;
/* no device: VCFX_E_NO_DEVICE; n_samples = 0 or above 2,097,152 (s_pad past 2^21, the most a tile word indexes):
   VCFX_E_INVALID, before anything is allocated; counts that do not fit the device: VCFX_E_NOMEM.  Every copy and kernel
   runs on `stream`, a cudaStream_t of that device (NULL: the default stream) */
int  vcfx_cuda_king_create(int device, uint32_t n_samples, void *stream, vcfx_king **out);
void vcfx_cuda_king_destroy(vcfx_king *k);
/* n_rows PLINK 1 .bed rows of ceil(n_samples / 4) bytes, back to back.  on_device: a pointer into k's device (enqueued on
   k's stream) else host memory (may be reused when the call returns).  0 rows is valid.  A call that would take the rows
   added past UINT32_MAX is refused (VCFX_E_INVALID) and adds nothing.  Rows are gathered into slabs; a full slab is
   turned into counts on the spot, the rest by vcfx_cuda_king_counts. */
int  vcfx_cuda_king_add(vcfx_king *k, const void *rows, uint64_t n_rows, int on_device);
/* waits; writes CC, HH, AB, HC as four row-major n x n uint32 matrices, in that order, to host or device memory
   (dst_on_device); rows_added (may be NULL) gets the rows added so far.  More rows may be added afterwards. */
int  vcfx_cuda_king_counts(vcfx_king *k, uint32_t *dst, int dst_on_device, uint64_t *rows_added);
/* rows of one slab (a multiple of 128): the planes workspace holds this many variants for all samples */
uint64_t vcfx_cuda_king_slab_rows(const vcfx_king *k);

#ifdef __cplusplus
}
#endif
#endif /* VCFX_CUDA_H */
