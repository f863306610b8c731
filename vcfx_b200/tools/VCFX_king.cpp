// VCFX_king — KING-robust kinship of every pair of samples of a VCF (PREFIX.kin0).  It has no counterpart in the reference
// toolkit.  The calls are VCFX_dosage_calculator's, packed two bits each on the GPU as PLINK 1 .bed rows (VCFX_OP_DOSAGE +
// VCFX_F_DS_BED, as VCFX_plink_bed writes them); each chunk's rows go to one relatedness accumulator on the first device
// (vcfx_cuda_king_*, the pair counts as int8 MMAs on the tensor cores), and the host prints one line per pair at the end.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fcntl.h>
#include <getopt.h>
#include <string>
#include <unistd.h>
#include <vector>

#include "vcfx_host.h"

static void display_help() {
    fputs("VCFX_king: KING-robust kinship of every pair of samples of a VCF.\n\n"
          "Usage:\n"
          "  VCFX_king --out PREFIX [--min-kinship X] [-q] [-i input.vcf | input.vcf | < input.vcf]\n\n"
          "Options:\n"
          "  -o, --out PREFIX     Write PREFIX.kin0 (required)\n"
          "  -m, --min-kinship X  Keep only the pairs whose kinship is >= X (NA pairs are dropped)\n"
          "  -i, --input FILE     Input VCF file (default: the positional argument, else stdin)\n"
          "  -q, --quiet          Suppress the warning for each line with fewer than 10 fields\n"
          "  -h, --help           Display this help message and exit\n\n"
          "Description:\n"
          "  PREFIX.kin0 has a header line '#ID1 ID2 NSNP HETHET IBS0 HET1 HET2 KINSHIP' and one\n"
          "  line per pair of samples (i < j in column order, i outer), tab-separated.  Over the\n"
          "  variants where both samples are called: NSNP sites, HETHET both het, IBS0 one hom\n"
          "  REF and the other hom ALT, HET1 / HET2 the first / second sample het.  KINSHIP is\n"
          "  KING's between-family robust estimator (Manichaikul et al., Bioinformatics 2010)\n"
          "  0.5 - (HET1 + HET2 - 2 HETHET + 4 IBS0) / (4 min(HET1, HET2)), printed with %.6g,\n"
          "  or NA when min(HET1, HET2) = 0.  Duplicates give 0.5, parent-offspring and full\n"
          "  sibs about 0.25, unrelated samples about 0 or below.\n"
          "  The calls are VCFX_dosage_calculator's, read as VCFX_plink_bed packs them: on a\n"
          "  multi-allelic line every allele > 0 counts as ALT, a haploid call counts as the\n"
          "  dosage it gives, and a missing call, a line without a GT key or a missing column\n"
          "  is not called.  Lines with fewer than 10 fields are skipped; columns beyond the\n"
          "  #CHROM line's samples are dropped (one warning).  File and stdin input are read the\n"
          "  same way.  This tool has no counterpart in the reference VCFX toolkit.\n\n"
          "Example:\n"
          "  VCFX_king --out cohort --min-kinship 0.0884 -i cohort.vcf\n", stdout);
}

static const char SHORT_WARNING[] = "Warning: Skipping VCF line with fewer than 10 fields.\n";

int main(int argc, char *argv[]) {
    for (int i = 1; i < argc; ++i) if (!strcmp(argv[i], "--help") || !strcmp(argv[i], "-h")) { display_help(); return 0; }
    const char *input = nullptr, *prefix = nullptr;
    bool quiet = false, filter = false;
    double min_kinship = 0;
    static struct option long_opts[] = {{"help", no_argument, nullptr, 'h'}, {"input", required_argument, nullptr, 'i'},
                                        {"out", required_argument, nullptr, 'o'}, {"min-kinship", required_argument, nullptr, 'm'},
                                        {"quiet", no_argument, nullptr, 'q'}, {nullptr, 0, nullptr, 0}};
    int c;
    while ((c = getopt_long(argc, argv, "hi:o:m:q", long_opts, nullptr)) != -1) {
        switch (c) {
        case 'i': input = optarg; break;
        case 'o': prefix = optarg; break;
        case 'q': quiet = true; break;
        case 'm': {
            char *end = nullptr;
            min_kinship = strtod(optarg, &end);
            if (!*optarg || *end) { fprintf(stderr, "Error: invalid --min-kinship value '%s'\n", optarg); return 1; }
            filter = true;
            break;
        }
        default: display_help(); return 1;
        }
    }
    if (!input && optind < argc) input = argv[optind];
    if (!prefix || !*prefix) { fputs("Error: --out PREFIX is required.\n", stderr); return 1; }

    int fd = 0;
    if (input) {
        fd = open(input, O_RDONLY);
        if (fd < 0) { fprintf(stderr, "Error: cannot open file '%s'\n", input); return 1; }
    }
    vcfxh::Source src(fd);
    std::string head;
    std::vector<std::string> names;
    if (!vcfxh::read_sample_header(src, head, names, ".kin0")) return 1;
    const uint32_t W = (uint32_t)names.size();
    const size_t B = ((size_t)W + 3) / 4, row_bytes = 16 + B;

    vcfxh::AsideFiles outs;
    outs.prefix = prefix;
    outs.ext = {".kin0"};
    if (!outs.open_all()) { outs.discard(); return 1; }

    vcfxh::RunOptions opt;
    opt.op = VCFX_OP_DOSAGE;
    opt.mode = VCFX_MODE_FILE;
    opt.flags = VCFX_F_DS_BED;
    opt.n_sel = W;
    opt.preface = head;
    opt.out_fd = outs.fd[0];                              // (nothing reaches it: the hook keeps every piece)
    int device = 0;
    opt.first_device = &device;
    vcfx_king *king = nullptr;
    int king_rc = VCFX_OK;
    auto ensure_king = [&]() {
        if (!king && W && king_rc == VCFX_OK) king_rc = vcfx_cuda_king_create(device, W, nullptr, &king);
        return king_rc == VCFX_OK;
    };
    // per chunk, in file order: its packed rows into the accumulator (the rows of a chunk are copied before add returns)
    opt.on_output = [&](const char *, size_t, uint64_t, const char **out, size_t *n) {
        const size_t k = *n / row_bytes;
        if (k && (!ensure_king() || (king_rc = vcfx_cuda_king_add(king, *out + 16 * k, k, 0)) != VCFX_OK)) return false;
        *n = 0;
        return true;
    };
    vcfxh::Totals tot;
    std::string err;
    int rc = vcfxh::run_stream(src, opt, tot, err);
    if (input) close(fd);
    std::vector<uint32_t> cnt;
    if (rc == VCFX_OK && W && ensure_king()) {
        cnt.resize(4 * (size_t)W * W);
        king_rc = vcfx_cuda_king_counts(king, cnt.data(), 0, nullptr);
    }
    if (rc == VCFX_OK && king_rc != VCFX_OK) rc = king_rc;
    if (rc != VCFX_OK) {
        fprintf(stderr, "Error: %s\n", king_rc != VCFX_OK ? vcfx_cuda_strerror(king_rc) : err.c_str());
        outs.discard(); vcfxh::finish(1);
    }

    // PREFIX.kin0: CC, HH, AB, HC are n x n row-major
    const size_t nn = (size_t)W * W;
    const uint32_t *CC = cnt.data(), *HH = CC + nn, *AB = HH + nn, *HC = AB + nn;
    std::string text = "#ID1\tID2\tNSNP\tHETHET\tIBS0\tHET1\tHET2\tKINSHIP\n";
    bool ok = true;
    char num[64];
    for (uint32_t i = 0; i < W && ok; ++i) {
        for (uint32_t j = i + 1; j < W; ++j) {
            const uint64_t nsnp = CC[(size_t)i * W + j], hethet = HH[(size_t)i * W + j];
            const uint64_t ibs0 = (uint64_t)AB[(size_t)i * W + j] + AB[(size_t)j * W + i];
            const uint64_t het1 = HC[(size_t)i * W + j], het2 = HC[(size_t)j * W + i];
            const uint64_t m = std::min(het1, het2);
            double kin = 0;
            if (m) kin = 0.5 - (double)(int64_t)(het1 + het2 + 4 * ibs0 - 2 * hethet) / (4.0 * (double)m);
            if (filter && (!m || !(kin >= min_kinship))) continue;
            text += names[i]; text += '\t'; text += names[j];
            snprintf(num, sizeof num, "\t%llu\t%llu\t%llu\t%llu\t%llu\t", (unsigned long long)nsnp, (unsigned long long)hethet,
                     (unsigned long long)ibs0, (unsigned long long)het1, (unsigned long long)het2);
            text += num;
            if (m) { snprintf(num, sizeof num, "%.6g\n", kin); text += num; }
            else text += "NA\n";
        }
        if (text.size() > (8u << 20)) { ok = vcfxh::write_all(outs.fd[0], text.data(), text.size()); text.clear(); }
    }
    if (!ok || !vcfxh::write_all(outs.fd[0], text.data(), text.size())) {
        fprintf(stderr, "Error: cannot write '%s.kin0'\n", prefix);
        outs.discard(); vcfxh::finish(1);
    }
    if (!outs.commit()) { outs.discard(); vcfxh::finish(1); }
    if (!quiet)
        for (uint64_t i = 0; i < tot.short_lines; ++i) fputs(SHORT_WARNING, stderr);
    if (tot.flagged)
        fprintf(stderr, "Warning: %llu variant line(s) have more sample columns than the #CHROM line names; the extra columns were dropped.\n",
                (unsigned long long)tot.flagged);
    vcfxh::finish(0);
}
