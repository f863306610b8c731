// VCFX_plink_bed — PLINK 1 binary genotypes (PREFIX.bed, PREFIX.bim, PREFIX.fam) from a VCF.  It has no counterpart in the
// reference toolkit: its calls are VCFX_dosage_calculator's, packed two bits each on the GPU by libvcfx_cuda
// (VCFX_OP_DOSAGE + VCFX_F_DS_BED, see include/vcfx_cuda.h).  The host reads the "#CHROM" line for the samples, cuts the
// .bim fields from each chunk's own bytes at the rows' line offsets, and writes the packed rows behind the .bed magic in
// file order.  Every file is written under a private name and renamed at the end: a run that fails leaves none behind.
#include <cctype>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fcntl.h>
#include <getopt.h>
#include <string>
#include <sys/stat.h>
#include <unistd.h>
#include <vector>

#include "vcfx_host.h"

static void display_help() {
    fputs("VCFX_plink_bed: Write the genotypes of a VCF as PLINK 1 binary files (.bed, .bim, .fam).\n\n"
          "Usage:\n"
          "  VCFX_plink_bed --out PREFIX [-q] [-i input.vcf | input.vcf | < input.vcf]\n\n"
          "Options:\n"
          "  -o, --out PREFIX  Write PREFIX.bed, PREFIX.bim and PREFIX.fam (required)\n"
          "  -i, --input FILE  Input VCF file (default: the positional argument, else stdin)\n"
          "  -q, --quiet       Suppress the warning for each line with fewer than 10 fields\n"
          "  -h, --help        Display this help message and exit\n\n"
          "Description:\n"
          "  The calls are VCFX_dosage_calculator's: the number of alleles > 0 in a sample's GT.\n"
          "  A1 is ALT and A2 is REF, so a reader that counts A1 alleles gets the dosage back.\n"
          "  On a multi-allelic line every allele > 0 counts: A1 stands for \"any non-REF allele\"\n"
          "  and ALT in the .bim is the line's whole ALT column.  A missing call (\"NA\"), a line\n"
          "  without a GT key and a line with fewer sample columns than the #CHROM line give\n"
          "  missing calls; columns beyond the #CHROM line's samples are dropped (one warning).\n"
          "  Lines with fewer than 10 fields are skipped.  The .bed is variant-major; the .fam\n"
          "  gives each sample its name as family and individual ID.  File and stdin input are\n"
          "  read the same way ('\\r' before '\\n' is dropped).  This tool has no counterpart in\n"
          "  the reference VCFX toolkit.\n\n"
          "Example:\n"
          "  VCFX_plink_bed --out cohort -i cohort.vcf\n", stdout);
}

static const char SHORT_WARNING[] = "Warning: Skipping VCF line with fewer than 10 fields.\n";

namespace {

// PREFIX.bed / .bim / .fam, each written under a private name until commit()
struct Outputs {
    std::string prefix;
    const char *ext[3] = {".bed", ".bim", ".fam"};
    int fd[3] = {-1, -1, -1};
    std::string tmp[3];
    bool open_all() {
        for (int i = 0; i < 3; ++i) {
            tmp[i] = prefix + ext[i] + "." + std::to_string((long)getpid()) + ".part";
            fd[i] = open(tmp[i].c_str(), O_WRONLY | O_CREAT | O_TRUNC | O_EXCL, 0666);
            if (fd[i] < 0) { fprintf(stderr, "Error: cannot create '%s%s'\n", prefix.c_str(), ext[i]); return false; }
        }
        return true;
    }
    void discard() {
        for (int i = 0; i < 3; ++i) {
            if (fd[i] >= 0) { close(fd[i]); fd[i] = -1; }
            if (!tmp[i].empty()) unlink(tmp[i].c_str());
        }
    }
    bool commit() {
        for (int i = 0; i < 3; ++i) {
            const int rc = close(fd[i]);
            fd[i] = -1;
            if (rc != 0) { fprintf(stderr, "Error: cannot write '%s%s'\n", prefix.c_str(), ext[i]); return false; }
        }
        for (int i = 0; i < 3; ++i)
            if (rename(tmp[i].c_str(), (prefix + ext[i]).c_str()) != 0) {
                fprintf(stderr, "Error: cannot create '%s%s'\n", prefix.c_str(), ext[i]);
                for (int j = 0; j < i; ++j) unlink((prefix + ext[j]).c_str());
                return false;
            }
        return true;
    }
};

// the first five fields of a tab-separated line (a row's line has ten or more)
void cut_fields(const char *p, const char *end, const char *f[5], size_t len[5]) {
    for (int i = 0; i < 5; ++i) {
        const char *t = static_cast<const char *>(memchr(p, '\t', (size_t)(end - p)));
        const char *e = t ? t : end;
        f[i] = p; len[i] = (size_t)(e - p);
        p = t ? t + 1 : end;
    }
}

}  // namespace

int main(int argc, char *argv[]) {
    for (int i = 1; i < argc; ++i) if (!strcmp(argv[i], "--help") || !strcmp(argv[i], "-h")) { display_help(); return 0; }
    const char *input = nullptr, *prefix = nullptr;
    bool quiet = false;
    static struct option long_opts[] = {{"help", no_argument, nullptr, 'h'}, {"input", required_argument, nullptr, 'i'},
                                        {"out", required_argument, nullptr, 'o'}, {"quiet", no_argument, nullptr, 'q'},
                                        {nullptr, 0, nullptr, 0}};
    int c;
    while ((c = getopt_long(argc, argv, "hi:o:q", long_opts, nullptr)) != -1) {
        switch (c) {
        case 'i': input = optarg; break;
        case 'o': prefix = optarg; break;
        case 'q': quiet = true; break;
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

    // ---- up to the first data line: the first "#CHROM" line names the samples (dosage_calculator's file-mode rule)
    vcfxh::Source src(fd);
    std::string head, chrom;
    bool found_chrom = false;
    {
        std::string buf(1 << 16, '\0');
        size_t scan = 0;
        bool eof = false;
        for (;;) {
            size_t nl;
            while ((nl = head.find('\n', scan)) == std::string::npos && !eof) {
                long r = src.read(&buf[0], buf.size());
                if (r < 0) { fputs("Error: read error\n", stderr); return 1; }
                if (r == 0) { eof = true; break; }
                head.append(buf.data(), (size_t)r);
            }
            if (scan >= head.size()) break;
            size_t end = (nl == std::string::npos) ? head.size() : nl;
            if (end > scan && head[end - 1] == '\r') --end;
            if (end > scan) {
                if (head[scan] != '#') {
                    if (!found_chrom) { fputs("Error: VCF header (#CHROM) not found before variant records.\n", stderr); return 1; }
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
    if (!found_chrom) { fputs("Error: no #CHROM header line in the input.\n", stderr); return 1; }
    std::vector<std::string> names;
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
            fprintf(stderr, "Error: sample %zu ('%s') is empty or contains a blank; .fam is whitespace-delimited.\n", i + 1, names[i].c_str());
            return 1;
        }
    }
    const uint32_t W = (uint32_t)names.size();
    const size_t B = ((size_t)W + 3) / 4, row_bytes = 16 + B;

    Outputs outs;
    outs.prefix = prefix;
    if (!outs.open_all()) { outs.discard(); return 1; }
    std::string fam;
    for (const std::string &n : names) fam += n + "\t" + n + "\t0\t0\t0\t-9\n";
    static const char MAGIC[3] = {0x6c, 0x1b, 0x01};
    if (!vcfxh::write_all(outs.fd[2], fam.data(), fam.size()) || !vcfxh::write_all(outs.fd[0], MAGIC, 3)) {
        fputs("Error: cannot write the output files\n", stderr); outs.discard(); return 1;
    }

    vcfxh::RunOptions opt;
    opt.op = VCFX_OP_DOSAGE;
    opt.mode = VCFX_MODE_FILE;
    opt.flags = VCFX_F_DS_BED;
    opt.n_sel = W;
    opt.preface = head;
    opt.out_fd = outs.fd[0];
    std::string hook_err, bim;
    uint64_t rows = 0;
    // per chunk: a .bim line per row, cut from the chunk's bytes; the packed part of the piece goes on to the .bed
    opt.on_output = [&](const char *chunk, size_t nbytes, uint64_t file_offset, const char **out, size_t *n) {
        const size_t k = *n / row_bytes;
        bim.clear();
        for (size_t i = 0; i < k; ++i) {
            vcfx_ds_row r;
            memcpy(&r, *out + 16 * i, sizeof r);
            const char *line = chunk + (r.line_offset - file_offset);
            const char *f[5]; size_t len[5];
            cut_fields(line, chunk + nbytes, f, len);
            bim.append(f[0], len[0]); bim += '\t'; bim.append(f[2], len[2]); bim += "\t0\t"; bim.append(f[1], len[1]);
            bim += '\t'; bim.append(f[4], len[4]); bim += '\t'; bim.append(f[3], len[3]); bim += '\n';
        }
        if (!vcfxh::write_all(outs.fd[1], bim.data(), bim.size())) { hook_err = "cannot write '" + outs.prefix + ".bim'"; return false; }
        rows += k;
        *out += 16 * k; *n = k * B;
        return true;
    };
    vcfxh::Totals tot;
    std::string err;
    const int rc = vcfxh::run_stream(src, opt, tot, err);
    if (input) close(fd);
    if (rc != VCFX_OK) {
        fprintf(stderr, "Error: %s\n", hook_err.empty() ? err.c_str() : hook_err.c_str());
        outs.discard(); vcfxh::finish(1);
    }
    struct stat st;                                      // the ordered writer reports no failure of its own: check the size
    if (fstat(outs.fd[0], &st) != 0 || (uint64_t)st.st_size != 3 + rows * B) {
        fprintf(stderr, "Error: cannot write '%s.bed'\n", prefix);
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
