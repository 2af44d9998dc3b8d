// host_api.cpp -- C ABI of libnimpress_host.so (include/nimpress_host.h) and the command line.
#include <cstring>
#include <unistd.h>
#include <iostream>
#include <string>
#include <vector>

#include "../../include/nimpress_host.h"
#include "driver.hpp"
#include "fast_inflate.hpp"
#include "stats.hpp"

using namespace nph;

struct nph_result { ScoreResult r; };

static thread_local std::string g_err;

const char *nph_last_error(void) { return g_err.c_str(); }

static ScoreParams to_params(const nph_params *p) {
    ScoreParams q;
    q.imp_locus = p->imp_locus; q.imp_missing = p->imp_missing; q.imp_sample = p->imp_sample;
    q.ignorefilt = p->ignorefilt != 0; q.use_cov = p->use_cov != 0; q.device = p->device; q.exact_order = p->exact_order != 0;
    q.mincs = p->mincs; q.maxmis = p->maxmis; q.afmisp = p->afmisp;
    for (int d = 0; d < 32; d++) if (((uint32_t)p->device_mask >> d) & 1u) q.devices.push_back(d);
    q.use_ds = p->use_ds != 0;
    q.use_pl = p->use_pl != 0;
    if (p->samples_path) q.samples_path = p->samples_path;
    q.exclude_samples = p->exclude_samples != 0;
    return q;
}

// samples a scoring call would score: the file's, or the kept ones under --samples
static int64_t scored_samples(const VariantSource &vcf, const ScoreParams &q) {
    if (q.samples_path.empty()) return vcf.n_samples();
    const std::vector<int64_t> keep = sample_subset(vcf.samples(), q.samples_path, q.exclude_samples);
    return keep.empty() ? vcf.n_samples() : (int64_t)keep.size();
}

// open(ScoreFile) + loadBedIntervals as main() sequences them (:728-740)
static int load_inputs(const char *score_path, const char *bed_path, ScoreParams &q, ScoreFile &sf, GenomeIntervals &cov,
                       std::string *fatal) {
    if (!sf.load(score_path)) return NPH_EOPEN_SCORE;
    if (q.use_cov && bed_path) {
        if (!cov.load(bed_path) && fatal)            // the reference logs FATAL but carries on (:739-740)
            *fatal += std::string("FATAL Could not open coverage BED file ") + bed_path + "\n";
    }
    return NPH_OK;
}

int nph_compute_polygenic_scores(const char *score_path, const char *genotype_path, const char *bed_path,
                                 const nph_params *p, nph_result **out) {
    if (!score_path || !genotype_path || !p || !out) return NPH_EINPUT;
    return nph_compute_polygenic_scores_files(&score_path, 1, &genotype_path, 1, bed_path, p, out);
}

int nph_compute_polygenic_scores_multi(const char *const *score_paths, int32_t n_scores, const char *genotype_path,
                                       const char *bed_path, const nph_params *p, nph_result **out) {
    if (!genotype_path) return NPH_EINPUT;
    return nph_compute_polygenic_scores_files(score_paths, n_scores, &genotype_path, 1, bed_path, p, out);
}

int nph_compute_polygenic_scores_files(const char *const *score_paths, int32_t n_scores, const char *const *genotype_paths,
                                       int32_t n_genotypes, const char *bed_path, const nph_params *p, nph_result **out) {
    if (!score_paths || n_scores < 1 || !genotype_paths || n_genotypes < 1 || !p || !out) return NPH_EINPUT;
    for (int32_t k = 0; k < n_scores; k++) out[k] = nullptr;
    try {
        ScoreParams q = to_params(p);
        std::vector<std::string> geno;
        for (int32_t f = 0; f < n_genotypes; f++) {
            if (!genotype_paths[f]) return NPH_EINPUT;
            geno.push_back(genotype_paths[f]);
        }
        // main() opens the VCF first (:728): an unreadable genotype file wins over an unreadable score file
        for (const std::string &g : geno) {
            std::unique_ptr<VariantSource> probe = open_variant_source(g, true);
            if (!probe) { g_err = "Could not open input VCF file " + g; return NPH_EOPEN_VCF; }
        }
        std::vector<ScoreFile> files((size_t)n_scores);
        std::vector<const ScoreFile *> ptrs;
        GenomeIntervals cov;
        std::string fatal;
        for (int32_t k = 0; k < n_scores; k++) {
            if (!files[k].load(score_paths[k])) { g_err = std::string("Could not open polygenic score file ") + score_paths[k]; return NPH_EOPEN_SCORE; }
            ptrs.push_back(&files[k]);
        }
        // the reference logs FATAL but carries on (:739-740)
        if (q.use_cov && bed_path && !cov.load(bed_path)) fatal = std::string("FATAL Could not open coverage BED file ") + bed_path + "\n";
        std::vector<ScoreResult> rs;
        std::string unopened = geno[0];
        if (!compute_polygenic_scores_files(ptrs, geno, cov, q, rs, &unopened)) {
            g_err = "Could not open input VCF file " + unopened;
            return NPH_EOPEN_VCF;
        }
        for (int32_t k = 0; k < n_scores; k++) {
            out[k] = new nph_result();
            out[k]->r = std::move(rs[k]);
            out[k]->r.warnings = fatal + out[k]->r.warnings;
        }
        return NPH_OK;
    } catch (const InputError &e) {
        g_err = e.what();
        return NPH_EINPUT;
    } catch (const std::exception &e) {
        g_err = e.what();
        return NPH_EGPU;
    }
}

int64_t nph_result_n_samples(const nph_result *r) { return (int64_t)r->r.scores.size(); }
int64_t nph_result_n_loci(const nph_result *r) { return (int64_t)r->r.loci.size(); }
int64_t nph_result_nloci_used(const nph_result *r) { return r->r.nloci; }
int64_t nph_result_rounds(const nph_result *r) { return r->r.rounds; }
int64_t nph_result_devices(const nph_result *r) { return r->r.devices; }
int64_t nph_result_records_read(const nph_result *r) { return r->r.records_read; }
int64_t nph_result_index_seeks(const nph_result *r) { return r->r.index_seeks; }
const double *nph_result_scores(const nph_result *r) { return r->r.scores.data(); }
const npc_locus *nph_result_loci(const nph_result *r) { return r->r.loci.data(); }
const char *nph_result_sample(const nph_result *r, int64_t i) { return r->r.samples[(size_t)i].c_str(); }
const char *nph_result_warnings(const nph_result *r) { return r->r.warnings.c_str(); }
void nph_result_free(nph_result *r) { delete r; }

int nph_plan(const char *score_path, const char *genotype_path, const char *bed_path, const nph_params *p,
             int32_t *kind_out, int32_t *eaidx_out, int64_t cap, int64_t *n_rows_out, int64_t *n_samples_out) {
    try {
        ScoreParams q = to_params(p);
        std::unique_ptr<VariantSource> vcf = open_variant_source(genotype_path);
        if (!vcf) return NPH_EOPEN_VCF;
        const int64_t n_scored = scored_samples(*vcf, q);
        ScoreFile sf; GenomeIntervals cov;
        int rc = load_inputs(score_path, bed_path, q, sf, cov, nullptr);
        if (rc) return rc;
        if ((int64_t)sf.entries.size() > cap) return NPH_ECAPACITY;
        Matcher M(sf, cov, q);
        VariantRecord rec;
        while (vcf->next(rec)) M.match(rec);
        M.finish();
        for (size_t i = 0; i < sf.entries.size(); i++) { kind_out[i] = M.kind[i]; eaidx_out[i] = M.eaidx[i]; }
        *n_rows_out = (int64_t)sf.entries.size();
        *n_samples_out = n_scored;
        return NPH_OK;
    } catch (const InputError &e) {
        g_err = e.what();
        return NPH_EINPUT;
    }
}

int nph_plan_indexed(const char *score_path, const char *genotype_path, const char *bed_path, const nph_params *p,
                     int32_t *kind_out, int32_t *eaidx_out, int64_t cap, int64_t *n_rows_out, int64_t *n_samples_out,
                     int64_t *records_read_out, int64_t *index_seeks_out) {
    return nph_plan_files(score_path, &genotype_path, 1, bed_path, p, kind_out, eaidx_out, cap, n_rows_out, n_samples_out,
                          records_read_out, index_seeks_out);
}

int nph_plan_files(const char *score_path, const char *const *genotype_paths, int32_t n_genotypes, const char *bed_path,
                   const nph_params *p, int32_t *kind_out, int32_t *eaidx_out, int64_t cap, int64_t *n_rows_out,
                   int64_t *n_samples_out, int64_t *records_read_out, int64_t *index_seeks_out) {
    try {
        if (!genotype_paths || n_genotypes < 1) return NPH_EINPUT;
        ScoreParams q = to_params(p);
        ScoreFile sf; GenomeIntervals cov;
        int rc = load_inputs(score_path, bed_path, q, sf, cov, nullptr);
        if (rc) return rc;
        if ((int64_t)sf.entries.size() > cap) return NPH_ECAPACITY;
        Matcher M(sf, cov, q);
        GenotypeFiles files(std::vector<std::string>(genotype_paths, genotype_paths + n_genotypes));
        std::string unopened;
        if (!files.open(q, &unopened)) { g_err = "Could not open input VCF file " + unopened; return NPH_EOPEN_VCF; }     // the driver's order: index first
        Spans spans;
        M.add_spans(spans);
        VariantRecord rec;
        int64_t nrec = 0, seeks = 0;
        for (size_t f = 0; f < files.paths.size(); f++) {
            if (!files.prepare(f, spans)) { g_err = "Could not open input VCF file " + files.paths[f]; return NPH_EOPEN_VCF; }
            VariantSource &vcf = *files.src[f];
            while (vcf.next(rec)) { nrec++; M.match(rec); }
            seeks += vcf.seeks();
            files.src[f].reset();
        }
        M.finish();
        for (size_t i = 0; i < sf.entries.size(); i++) { kind_out[i] = M.kind[i]; eaidx_out[i] = M.eaidx[i]; }
        *n_rows_out = (int64_t)sf.entries.size();
        *n_samples_out = (int64_t)files.names.size();
        if (records_read_out) *records_read_out = nrec;
        if (index_seeks_out) *index_seeks_out = seeks;
        return NPH_OK;
    } catch (const InputError &e) {
        g_err = e.what();
        return NPH_EINPUT;
    }
}

int nph_read_gt(const char *genotype_path, uint8_t *out, int64_t row_bytes, int64_t max_records, int64_t *n_records,
                int64_t *n_samples, int32_t *width, int32_t *ploidy) {
    try {
        std::unique_ptr<VariantSource> vcf = open_variant_source(genotype_path);
        if (!vcf) return NPH_EOPEN_VCF;
        if (const char *e = getenv("NIMPRESS_READ_DS")) if (*e && *e != '0') vcf->set_dosage_mode(true);   // tests: FORMAT/DS instead of GT
        if (const char *e = getenv("NIMPRESS_READ_PL")) if (*e && *e != '0') vcf->set_pl_mode(true);       // tests: FORMAT/PL rows
        int bgen_layout = NPC_GT_DOSE255;                                                                   // BGEN rows
        if (const char *e = getenv("NIMPRESS_READ_DOSE32")) if (*e && *e != '0') bgen_layout = NPC_GT_DOSE32;
        VariantRecord rec;
        int64_t k = 0;
        *n_samples = vcf->n_samples();
        while (vcf->next(rec)) {
            if (k >= max_records) return NPH_ECAPACITY;
            if (rec.has_gt && vcf->fixed_layout() == NPC_GT_DOSE255) {
                // BGEN: converted by the source's workers straight into the output row, as the driver has it done
                if (npc_gt_row_bytes(vcf->n_samples(), 2, bgen_layout) > row_bytes) { vcf->wait_rows(); return NPH_ECAPACITY; }
                vcf->load_gt_into(rec, out + k * row_bytes, bgen_layout, 2);
                *width = rec.gt_width; *ploidy = rec.ploidy;
            } else if (rec.has_gt) {
                vcf->load_gt(rec);
                const int64_t bytes = npc_gt_row_bytes(vcf->n_samples(), rec.ploidy, rec.gt_width);
                if (bytes > row_bytes) return NPH_ECAPACITY;
                memcpy(out + k * row_bytes, rec.gt, (size_t)bytes);
                *width = rec.gt_width; *ploidy = rec.ploidy;
            }
            k++;
        }
        vcf->wait_rows();
        *n_records = k;
        return NPH_OK;
    } catch (const InputError &e) {
        g_err = e.what();
        return NPH_EINPUT;
    }
}

int nph_fast_inflate(const uint8_t *in, int64_t in_len, uint8_t *out, int64_t out_len) {
    static thread_local FastInflateTables t;
    return fast_inflate(in, (size_t)in_len, out, (size_t)out_len, t) ? 1 : 0;
}

double nph_dbinom(int64_t x, int64_t n, double p) { return dbinom(x, n, p); }
double nph_pbinom(int64_t x, int64_t n, double p) { return pbinom(x, n, p); }
double nph_betai(double a, double b, double x) { return betai(a, b, x); }
double nph_binom_test(int64_t x, int64_t n, double p) { return binom_test(x, n, p); }

int nph_format_float(double v, char *buf, int32_t buflen) {
    std::string s = format_float_nim(v);
    if ((int32_t)s.size() + 1 > buflen) return -1;
    memcpy(buf, s.c_str(), s.size() + 1);
    return (int)s.size();
}

// ------------------------------------------------------------------------------------------
// command line -- main() of the reference (src/nimpress.nim:652-753), docopt usage text :653-706
// ------------------------------------------------------------------------------------------

static const char *USAGE =
    "Compute polygenic scores from a VCF/BCF, a PLINK 1 binary fileset or a BGEN v1.2 file.\n\n"
    "Usage:\n"
    "  nimpress [options] <scoredef> <genotypes.vcf|.bcf|.bed>\n"
    "  nimpress [options] <scoredef1>,<scoredef2>,... <genotypes.vcf|.bcf|.bed>   (one pass, a \"#score\" line per file; not in the reference)\n"
    "  nimpress [options] <scoredef> <genotypes.bgen>\n"
    "  nimpress [options] <scoredef>[,<scoredef>...] <genotypes> [<genotypes> ...]   (several genotype files, e.g. one per\n"
    "                     chromosome: scored exactly as their concatenation; not in the reference)\n"
    "  nimpress (-h | --help)\n"
    "  nimpress --version\n\n"
    "Options:\n"
    "  -h --help          Show this screen.\n"
    "  --version          Show version.\n"
    "  --cov=<path>       Path to a BED file supplying genome regions that have been\n"
    "                     genotyped in the genotypes.vcf file.\n"
    "  --imp-locus=<m>    Imputation to apply for whole loci which are either not\n"
    "                     in the sequenced BED regions, or fail (too many samples\n"
    "                     with missing genotype, as set by --maxmis, or a FILTER field\n"
    "                     other than \".\" / \"PASS\" if --ignorefilt is not set). Valid\n"
    "                     values are ps, homref, fail, ignore [default: ps].\n"
    "  --imp-missing=<m>  Imputation to apply for loci which are in the sequenced BED\n"
    "                     regions (and thus should have been genotyped), but are\n"
    "                     completely missing from the VCF. Valid values are homref,\n"
    "                     ignore [default: homref].\n"
    "  --imp-sample=<m>   Imputation to apply for an individual sample with missing\n"
    "                     genotype. Valid values are ps, homref, fail, int_fail,\n"
    "                     int_ps [default: int_ps].\n"
    "  --maxmis=<f>       Maximum fraction of samples with missing genotypes allowed\n"
    "                     at a locus [default: 0.05].\n"
    "  --mincs=<n>        Minimum number of genotyped samples at a locus for internal\n"
    "                     imputation [default: 100].\n"
    "  --afmisp=<f>       p-value threshold for warning about allele frequency\n"
    "                     mismatch [default: 0.001].\n"
    "  --ignorefilt       Ignore the VCF FILTER field.\n"
    "  --device=<n>       CUDA device to score on [default: 0] (not a reference option).\n"
    "  --devices=<list>   Several CUDA devices, e.g. 0-7 or 0,2,3: the score file is split into\n"
    "                     contiguous ranges, one per device, and the partial sums are combined\n"
    "                     in range order (not a reference option).\n"
    "  --dosage           Score FORMAT/DS (expected ALT-allele dosage, one float per sample) instead of\n"
    "                     FORMAT/GT (not a reference option: the reference lists it under Future).\n"
    "                     Not with a PLINK fileset; with a BGEN file it changes nothing.\n"
    "  --pl               Score FORMAT/PL (phred-scaled genotype likelihoods) as the posterior expected\n"
    "                     dosage under a Hardy-Weinberg prior at the score file's EAF, instead of\n"
    "                     FORMAT/GT (not a reference option).  Biallelic records only (split others\n"
    "                     with bcftools norm -m-); diploid and haploid samples.  Not with --dosage, a\n"
    "                     PLINK fileset or a BGEN file.  No AF-mismatch warnings.\n"
    "PLINK 1 fileset (not a reference input): X.bed with X.bim and X.fam, recognised by its magic bytes.\n"
    "  REF = A2 (.bim column 6), ALT = A1 (column 5), sample names = .fam IID; FILTER is always \".\".\n"
    "BGEN v1.2 file (not a reference input): layout 2, 1-16 bits per probability, uncompressed or zlib,\n"
    "  haploid and diploid samples, biallelic variants, recognised by its magic bytes.  Scored as expected\n"
    "  ALT dosages.  REF = allele 1, ALT = allele 2, CHROM compared literally; sample names = the embedded\n"
    "  identifiers, else column 2 (ID_2) of X.sample beside X.bgen; FILTER is always \".\".  No AF-mismatch\n"
    "  warnings for its loci.\n"
    "  --exact-order      Add every locus to the running sums in score-file order, bit for bit\n"
    "                     like the reference (default: sum tiles of four loci first; same\n"
    "                     products, scores equal to ~1e-15 relative) (not a reference option).\n"
    "  --samples=<file>   Score only the samples named in <file>, one name per line (VCF/BCF header\n"
    "                     name, .fam IID, BGEN identifier or .sample ID_2), in the genotype file's\n"
    "                     order: exactly what a genotype file holding only them gives, cohort EAF,\n"
    "                     --maxmis and WARN lines included (not a reference option).\n"
    "  --samples=^<file>  Score every sample except those named in <file>; names the genotype file\n"
    "                     lacks are ignored (not a reference option).\n"
    "Several genotype files (not a reference input): VCF/BCF files (text and BCF may be mixed), PLINK 1 filesets\n"
    "  or BGEN files, one kind per run, read in the order given; a site in two files is matched in the earlier one.\n"
    "  Every file must carry the same samples in the same order, or, with --samples, keep the same samples in the\n"
    "  same order.\n";

static int parse_enum(const std::string &v, std::initializer_list<const char *> names) {   // Nim parseEnum: style-insensitive beyond the first char is not reproduced
    int i = 0;
    for (const char *nm : names) { if (v == nm) return i; i++; }
    throw InputError("invalid enum value: " + v);
}

// "0-3", "0,2,5", "1" -> bit mask of CUDA devices
static uint32_t parse_device_list(const std::string &v) {
    uint32_t mask = 0;
    for (size_t a = 0; a <= v.size();) {
        size_t b = v.find(',', a);
        if (b == std::string::npos) b = v.size();
        const std::string item = v.substr(a, b - a);
        const size_t dash = item.find('-');
        const int64_t lo = parse_int_nim(dash == std::string::npos ? item : item.substr(0, dash), "--devices");
        const int64_t hi = dash == std::string::npos ? lo : parse_int_nim(item.substr(dash + 1), "--devices");
        if (lo < 0 || hi > 31 || hi < lo) throw InputError("--devices: device indices are 0..31, ranges lo-hi");
        for (int64_t d = lo; d <= hi; d++) mask |= 1u << d;
        a = b + 1;
    }
    if (!mask) throw InputError("--devices: empty list");
    return mask;
}

// WARN lines, then one `name<TAB>$score` line per sample (:752-753), formatted into one buffer
static void print_result(const nph_result *r) {
    std::string out = r->r.warnings;
    const std::vector<double> &s = r->r.scores;
    size_t names = 0;
    for (const std::string &nm : r->r.samples) names += nm.size();
    out.reserve(out.size() + names + s.size() * 28);
    char buf[48];
    for (size_t i = 0; i < s.size(); i++) {
        out += r->r.samples[i];
        out += '\t';
        out.append(buf, (size_t)format_float_nim_to(s[i], buf));
        out += '\n';
    }
    std::cout.write(out.data(), (std::streamsize)out.size());
}

int nph_main(int argc, char **argv) {
    nph_params p = { NPC_LOCUS_PS, NPC_MISSING_HOMREF, NPC_SAMPLE_INT_PS, 0, 0, 0, 0, 0, 100, 0.05, 0.001, 0, 0, nullptr, 0 };
    std::string cov, samples_list;
    std::vector<std::string> pos;                          // <scoredef>, then the genotype files
    try {
        for (int i = 1; i < argc; i++) {
            std::string a = argv[i];
            auto val = [&](const char *opt) -> std::string {      // --opt=value or --opt value
                const size_t l = strlen(opt);
                if (a.size() > l && a[l] == '=') return a.substr(l + 1);
                if (i + 1 >= argc) throw InputError(std::string(opt) + " requires an argument");
                return argv[++i];
            };
            auto is = [&](const char *opt) { const size_t l = strlen(opt); return a.compare(0, l, opt) == 0 && (a.size() == l || a[l] == '='); };
            if (a == "-h" || a == "--help") { std::cout << USAGE; return 0; }
            else if (a == "--version") { std::cout << "nimpress 1.0.0\n"; return 0; }        // :708
            else if (is("--cov")) { cov = val("--cov"); p.use_cov = 1; }
            else if (is("--imp-locus")) p.imp_locus = parse_enum(val("--imp-locus"), { "ps", "homref", "fail", "ignore" });
            else if (is("--imp-missing")) p.imp_missing = parse_enum(val("--imp-missing"), { "homref", "ignore" });
            else if (is("--imp-sample")) p.imp_sample = parse_enum(val("--imp-sample"), { "ps", "homref", "fail", "int_ps", "int_fail" });
            else if (is("--maxmis")) p.maxmis = parse_float_nim(val("--maxmis"), "--maxmis");
            else if (is("--mincs")) p.mincs = parse_int_nim(val("--mincs"), "--mincs");
            else if (is("--afmisp")) p.afmisp = parse_float_nim(val("--afmisp"), "--afmisp");
            else if (is("--devices")) p.device_mask = (int32_t)parse_device_list(val("--devices"));
            else if (is("--device")) p.device = (int)parse_int_nim(val("--device"), "--device");
            else if (is("--samples")) {
                samples_list = val("--samples");
                p.exclude_samples = !samples_list.empty() && samples_list[0] == '^';
                if (p.exclude_samples) samples_list.erase(0, 1);
                if (samples_list.empty()) throw InputError("--samples requires a file name");
            }
            else if (a == "--ignorefilt") p.ignorefilt = 1;
            else if (a == "--exact-order") p.exact_order = 1;
            else if (a == "--dosage") p.use_ds = 1;
            else if (a == "--pl") p.use_pl = 1;
            else if (a.size() > 1 && a[0] == '-') throw InputError("unknown option " + a);
            else pos.push_back(a);
        }
        if (pos.size() < 2) throw InputError("expected <scoredef> <genotypes> [<genotypes> ...]");
        if (!samples_list.empty()) p.samples_path = samples_list.c_str();
    } catch (const InputError &e) {
        std::cerr << e.what() << "\n" << "Usage:\n  nimpress [options] <scoredef>[,<scoredef>...] <genotypes> [<genotypes> ...]\n";
        return 1;
    }
    std::vector<const char *> geno;                        // several genotype files: scored as their concatenation (DESIGN.md 4.12)
    for (size_t f = 1; f < pos.size(); f++) geno.push_back(pos[f].c_str());
    const char *bed = p.use_cov ? cov.c_str() : nullptr;
    // several score files, one pass (not a reference feature) -- unless the whole argument names a file, as it would for the reference
    if (pos[0].find(',') != std::string::npos && access(pos[0].c_str(), F_OK) != 0) {
        std::vector<std::string> paths;
        for (size_t a = 0; a <= pos[0].size();) { size_t b = pos[0].find(',', a); if (b == std::string::npos) b = pos[0].size(); if (b > a) paths.push_back(pos[0].substr(a, b - a)); a = b + 1; }
        std::vector<const char *> cp;
        for (auto &s : paths) cp.push_back(s.c_str());
        std::vector<nph_result *> rs(paths.size(), nullptr);
        int rc = nph_compute_polygenic_scores_files(cp.data(), (int32_t)cp.size(), geno.data(), (int32_t)geno.size(), bed, &p, rs.data());
        if (rc == NPH_EOPEN_VCF || rc == NPH_EOPEN_SCORE) { std::cout << "FATAL " << nph_last_error() << "\n"; return 255; }
        if (rc) { std::cerr << "nimpress: " << nph_last_error() << "\n"; return 1; }
        for (size_t k = 0; k < rs.size(); k++) {           // per file: a "#score" line, then the reference's output for it
            std::cout << "#score\t" << paths[k] << "\n";
            print_result(rs[k]);
            nph_result_free(rs[k]);
        }
        return 0;
    }
    nph_result *r = nullptr;
    const char *score = pos[0].c_str();
    int rc = nph_compute_polygenic_scores_files(&score, 1, geno.data(), (int32_t)geno.size(), bed, &p, &r);
    // "FATAL Could not open input VCF file <path>" (:729-730), "FATAL Could not open polygenic score file <path>" (:733-734)
    if (rc == NPH_EOPEN_VCF || rc == NPH_EOPEN_SCORE) { std::cout << "FATAL " << nph_last_error() << "\n"; return 255; }
    if (rc) { std::cerr << "nimpress: " << nph_last_error() << "\n"; return 1; }
    print_result(r);
    nph_result_free(r);
    return 0;
}
