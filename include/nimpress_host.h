/*
 * nimpress_host.h -- C ABI of libnimpress_host.so: the C++ host of the B200 scoring engine.
 *
 * The reference's host language is Nim, which this build environment does not have; the host
 * is therefore C++ and mirrors the reference's own entry points:
 *
 *   nph_compute_polygenic_scores  <->  computePolygenicScores  (src/nimpress.nim:592-649) after
 *                                      open(VCF) / open(ScoreFile) / loadBedIntervals
 *                                      (:233-244, :278-308), as tests/test_set1.nim:37-44 calls it
 *   nph_main                      <->  main()                  (src/nimpress.nim:652-753)
 *   nph_plan                      <->  the genotype-free half of getImputedDosages: coverage
 *                                      (:526), findVariant (:353-364), eaidx (:375-379), the
 *                                      FILTER test (:553) -- CPU only, for tests
 *   nph_binom_test ...            <->  binomTest / dbinom / pbinom / betai (:54-188)
 *
 * Everything genotype-shaped goes through libnimpress_cuda.so (include/nimpress_cuda.h); this
 * library never computes a score on the CPU.
 */
/*
 * Environment (diagnostics and tests; none is needed in normal use):
 *   NIMPRESS_THREADS=<n>     BGZF inflate threads (default min(cores - 1, 32); 1 = one thread, block by block)
 *   NIMPRESS_ZLIB_ONLY=1     inflate BGZF blocks with zlib instead of this library's own DEFLATE decoder
 *   NIMPRESS_NO_INDEX=1      never use <genotypes>.tbi / .csi;  NIMPRESS_FORCE_INDEX=1  use it whatever it saves
 *   NIMPRESS_TIMING=1        phase wall times on stderr
 *   NIMPRESS_SLAB_ROWS=<n>   cap the device-resident genotype rows (tests: forces scoring in rounds)
 *   NIMPRESS_SPLIT=<k>       with one device: k contexts on it, combined by npc_reduce (tests of the multi-GPU path on one GPU)
 *   NIMPRESS_READ_PL=1       nph_read_gt on a VCF / BCF: FORMAT/PL of every record as a packed PL row (NPC_GT_PL) instead
 *                            of its GT
 *   NIMPRESS_READ_DOSE32=1   nph_read_gt on a BGEN file: every block as a 32-bit dosage row (NPC_GT_DOSE32) instead of a
 *                            2-byte one (NPC_GT_DOSE255, which refuses other bit depths and haploid samples)
 */
#ifndef NIMPRESS_HOST_H
#define NIMPRESS_HOST_H
#include <stdint.h>

#include "nimpress_cuda.h"

#ifdef __cplusplus
extern "C" {
#endif

#define NPH_OK          0
#define NPH_EOPEN_VCF  -1   /* reference: "FATAL Could not open input VCF file", quit(-1)            */
#define NPH_EOPEN_SCORE -2  /* reference: "FATAL Could not open polygenic score file", quit(-1)      */
#define NPH_EINPUT     -3   /* malformed input: the reference's doAssert / ValueError paths (exit 1) */
#define NPH_ECAPACITY  -4   /* caller buffer too small                                               */
#define NPH_EGPU       -5   /* CUDA library / device failure                                          */

typedef struct {
    int32_t imp_locus;      /* NPC_LOCUS_*   */
    int32_t imp_missing;    /* NPC_MISSING_* */
    int32_t imp_sample;     /* NPC_SAMPLE_*  */
    int32_t ignorefilt;
    int32_t use_cov;        /* restrictToCoveredRgns */
    int32_t device;
    int32_t exact_order;    /* 1: npc_set_exact_order(ctx, 1) -- the reference's summation order bit for bit */
    int32_t device_mask;    /* != 0: score on every CUDA device whose bit is set (ascending order): the score rows are split
                               into contiguous ranges, one per device, combined in range order by npc_reduce; `device` is then
                               ignored.  0: one device, `device`.  Several score files at once: every file is cut into ranges of its own,
                               device d scores range d of every file, the host adds each file's partial sums in device order. */
    int64_t mincs;
    double  maxmis;
    double  afmisp;
    int32_t use_ds;         /* 1: score FORMAT/DS (fp32 expected ALT dosage, biallelic effect alleles) instead of FORMAT/GT --
                               npc_set_dosage_rows; not in the reference (README.md:162-165 "Future") */
    int32_t use_pl;         /* 1: score FORMAT/PL (phred-scaled genotype likelihoods of biallelic VCF / BCF records) as posterior
                               expected dosages at the score file's eaf (NPC_GT_PL rows, DESIGN.md 4.10) instead of FORMAT/GT;
                               not with use_ds, a PLINK fileset or a BGEN file; not in the reference */
    const char *samples_path; /* NULL: score every sample.  Else a list of sample names, one per line (the whole line, a trailing
                               \r stripped, blank lines skipped), matched against the names the results carry (VCF / BCF header,
                               .fam IID, BGEN identifier or .sample ID_2): only the listed samples are scored, in the genotype
                               file's order, exactly as a genotype file holding only them would be (cohort EAF, --maxmis, WARN
                               lines; DESIGN.md 4.11).  An unknown or twice-listed name, a name the file holds twice, an empty
                               subset or an unreadable list is NPH_EINPUT.  Not in the reference (plink --keep, bcftools -S) */
    int32_t exclude_samples;  /* 1: score the samples the list does NOT name (plink --remove, bcftools -S ^FILE); names the file
                               lacks are ignored */
    int32_t observed;       /* 1: also count, per sample, the score rows of class OK at which the sample has a called genotype
                               (nph_result_observed; DESIGN.md 4.13); scores and records are the same either way.  Not in the
                               reference (PLINK's CNT, PRSice's CNT, pgsc_calc's DENOM) */
} nph_params;

typedef struct nph_result nph_result;

/* Scores every sample of genotype_path (VCF text or BCF; plain, gzip or BGZF) against
 * score_path; bed_path may be NULL.  On NPH_OK *out owns the result. */
int nph_compute_polygenic_scores(const char *score_path, const char *genotype_path, const char *bed_path,
                                 const nph_params *p, nph_result **out);
/* Several score files over ONE pass of the genotype file (BASELINE config 4).  out[k] is what
 * nph_compute_polygenic_scores returns for score_paths[k] alone -- the reference's way to get it
 * is one nimpress process per score file.  On failure nothing is returned in out. */
int nph_compute_polygenic_scores_multi(const char *const *score_paths, int32_t n_scores, const char *genotype_path,
                                       const char *bed_path, const nph_params *p, nph_result **out);
/* Several genotype files (e.g. one per chromosome or chunk), read in the order given: exactly what one run over their
 * concatenation gives -- the records of file 1, then file 2, ..., with the common sample list (DESIGN.md 4.12).  out[k]
 * is what score_paths[k] gets.  The files are VCF text / BCF (mixed freely), or all PLINK 1 filesets, or all BGEN; they
 * carry the same samples in the same order, or keep the same sequence of samples under samples_path (applied to each
 * file on its own).  Mixed kinds and differing samples are NPH_EINPUT naming the file; NPH_EOPEN_VCF names the first
 * file that cannot be opened (nph_last_error).  All genotype files are opened before the score files. */
int nph_compute_polygenic_scores_files(const char *const *score_paths, int32_t n_scores, const char *const *genotype_paths,
                                       int32_t n_genotypes, const char *bed_path, const nph_params *p, nph_result **out);
int64_t nph_result_n_samples(const nph_result *r);
int64_t nph_result_n_loci(const nph_result *r);          /* score rows                      */
int64_t nph_result_nloci_used(const nph_result *r);      /* loci in the sum (the divisor/2) */
int64_t nph_result_rounds(const nph_result *r);          /* 1 = exact reference summation order */
int64_t nph_result_devices(const nph_result *r);         /* GPUs that scored this result             */
int64_t nph_result_records_read(const nph_result *r);    /* records the reader handed to the matcher         */
int64_t nph_result_index_seeks(const nph_result *r);     /* > 0: the file's .tbi / .csi index was used        */
const double *nph_result_scores(const nph_result *r);
/* Per sample: score rows of class OK (klass 0) at which the sample has a called genotype, i.e. nloci minus the loci imputed
 * for it (DESIGN.md 4.13).  NULL exactly when nph_params.observed was not set (never NULL when it was, even for no samples). */
const int64_t *nph_result_observed(const nph_result *r);
const npc_locus *nph_result_loci(const nph_result *r);   /* score-file order */
const char *nph_result_sample(const nph_result *r, int64_t i);
const char *nph_result_warnings(const nph_result *r);    /* "WARN ...\n" lines, reference order */
void nph_result_free(nph_result *r);
const char *nph_last_error(void);

/* CPU only: per score row kind (NPC_KIND_*) and eaidx after coverage / lookup / FILTER; *n_samples_out the samples a
 * scoring call would score (the kept ones under samples_path). */
int nph_plan(const char *score_path, const char *genotype_path, const char *bed_path, const nph_params *p,
             int32_t *kind_out, int32_t *eaidx_out, int64_t cap, int64_t *n_rows_out, int64_t *n_samples_out);
/* The same through the reader the scoring calls use: when <genotypes>.tbi / .csi exists, the file is
 * BGZF and the score's loci cover little of it, only the stretches around the loci are read (the
 * reference reaches every locus by an index query, src/nimpress.nim:358); otherwise the file is
 * streamed.  kind / eaidx are identical either way.  NIMPRESS_NO_INDEX=1 disables the index,
 * NIMPRESS_FORCE_INDEX=1 uses it whatever the coverage. */
int nph_plan_indexed(const char *score_path, const char *genotype_path, const char *bed_path, const nph_params *p,
                     int32_t *kind_out, int32_t *eaidx_out, int64_t cap, int64_t *n_rows_out, int64_t *n_samples_out,
                     int64_t *records_read_out, int64_t *index_seeks_out);
/* nph_plan_indexed over several genotype files, read as their concatenation (nph_compute_polygenic_scores_files): each
 * file takes its index-driven pass or is streamed on its own; records_read and index_seeks are sums over the files. */
int nph_plan_files(const char *score_path, const char *const *genotype_paths, int32_t n_genotypes, const char *bed_path,
                   const nph_params *p, int32_t *kind_out, int32_t *eaidx_out, int64_t cap, int64_t *n_rows_out,
                   int64_t *n_samples_out, int64_t *records_read_out, int64_t *index_seeks_out);

/* CPU only: raw GT payload of every record of a VCF/BCF, for reader tests.  Record r occupies
 * out[r*row_bytes ..]; returns the record count, width and ploidy of the LAST record read. */
int nph_read_gt(const char *genotype_path, uint8_t *out, int64_t row_bytes, int64_t max_records,
                int64_t *n_records, int64_t *n_samples, int32_t *width, int32_t *ploidy);

/* The pool's raw-DEFLATE decoder on one buffer (tests): `in` readable 16 bytes beyond in_len, `out` writable
 * 16 bytes beyond out_len; 1 = decoded exactly out_len bytes and the stream ended, 0 = not (the reader then uses zlib). */
int nph_fast_inflate(const uint8_t *in, int64_t in_len, uint8_t *out, int64_t out_len);

double nph_dbinom(int64_t x, int64_t n, double p);
double nph_pbinom(int64_t x, int64_t n, double p);
double nph_betai(double a, double b, double x);
double nph_binom_test(int64_t x, int64_t n, double p);
int nph_format_float(double v, char *buf, int32_t buflen);   /* Nim `$`(float), the output format */

/* The command line of the reference: nimpress [options] <scoredef> <genotypes.vcf> (and, beyond it, several score files
 * and several genotype files: <scoredef>[,<scoredef>...] <genotypes> [<genotypes> ...]); prints the
 * reference's WARN lines and `sample<TAB>score` lines to stdout; returns the process exit code
 * (0, 1 on malformed input / bad option, 255 when a file cannot be opened). */
int nph_main(int argc, char **argv);

#ifdef __cplusplus
}
#endif
#endif
