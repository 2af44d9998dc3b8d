/*
 * nimpress_cuda.h -- C ABI of libnimpress_cuda.so, the B200 (sm_100a) scoring engine.
 *
 * The reference (mpinese/nimpress, one Nim file) has no plugin or FFI interface of its own;
 * its scoring path is the body of `computePolygenicScores` (src/nimpress.nim:592-649) and the
 * procs it calls per locus.  This library sits exactly where those procs sit, so that a host
 * (Nim via {.importc, dynlib.}, C++, or ctypes) keeps file reading / locus matching and hands
 * the per-locus genotype work to the GPU:
 *
 *   reference proc (src/nimpress.nim)                replaced by
 *   ------------------------------------------------ -------------------------------------
 *   getRawDosages        :367-391  (GT decode)        count + accumulate kernels (npc_score_block*)
 *   tallyAlleles         :32-47    (ngt/nmiss/neff)   count kernel, integer-exact
 *   getImputedDosages    :565-571  (--maxmis rule)    decide kernel (IEEE fp64 divide + strict >)
 *   imputeLocusDosages   :417-447  (locus constant)   decide kernel (constant rows)
 *   absent-variant rule  :536-551                     decide kernel (kind = NPC_KIND_ABSENT)
 *   imputeSampleDosages  :450-481  (per-sample fill)  decide kernel + accumulate LUT
 *   scores[i] += d*beta  :639-641                     accumulate kernel, fp64, score-row order
 *   scores /= 2*nloci; += offset :643-649             npc_finish
 *
 * What stays on the host: coverage lookup (:313-345), findVariant (:353-364), the FILTER
 * string test (:553) and eaidx (:375-379); they enter as npc_row.kind / npc_row.eaidx.
 *
 * Conventions: plain C, no exceptions across the boundary.  Every call returns 0 (NPC_OK) or
 * a negative NPC_E* code; npc_last_error() gives the text.  One producer thread per context,
 * one context per GPU.  The library owns device memory and its pinned staging ring; buffers
 * passed by pointer belong to the caller and may be reused when the call returns.  There is
 * no CPU fallback: without a usable sm_100 device npc_create fails with NPC_ECUDA.
 *
 * Genotype rows are raw BCF FORMAT/GT payloads, untouched: per sample `ploidy` values of
 * `gt_width` bytes (1, 2 or 4), value = (allele+1)<<1 | phased, 0|phase = missing allele,
 * width-specific sentinels missing = MIN, vector_end = MIN+1 (both ignored, and a vector_end
 * ends the sample), rows `row_stride` bytes apart (row_stride % 16 == 0).
 *
 * Or, for a context created with gt_width = NPC_GT_BED (ploidy 2), rows of a PLINK 1 `.bed` fileset as stored:
 * 2 bits per sample, low bits first, ceil(n/4) bytes per row (DESIGN.md 4.7, npc_bed.cuh).
 *
 * Or, for a context created with gt_width = NPC_GT_DOSE255 (ploidy 2), fixed-point dosage rows as the host makes them
 * from a BGEN v1.2 file (layout 2, 8-bit probabilities, diploid, biallelic; DESIGN.md 4.8, npc_dose255.cuh): n
 * little-endian uint16 per row, k = 255 x the expected ALT dosage (unphased: 510 - 2*P(hom allele 1) - P(het);
 * phased: (255 - h0) + (255 - h1), all in units of 1/255), 0..510; any value above 510 (the host writes 0xFFFF) is a
 * missing sample.  A row whose effect allele is REF (eaidx 0) uses k' = 510 - k.  Tally: nmiss, and
 * neff_num = sum of k' over called samples as an exact integer; the reference's real tally is neff = fl(neff_num / 255)
 * and npc_locus.neff reports neff_num (units of 1/255).  Accumulate: scores[s] += fl(fl(k'/255) * beta) (cm for a
 * missing sample) in score-row order, the reference's chain, in every mode.  Hard calls (k = 0, 255, 510) therefore
 * score bit for bit as the same genotypes in int8 GT rows in exact order.
 *
 * Or, for a context created with gt_width = NPC_GT_DOSE32 (ploidy 2), 32-bit fixed-point dosage rows as the host makes
 * them from a BGEN v1.2 file at any bit depth B from 1 to 16, haploid and diploid samples (DESIGN.md 4.9,
 * npc_dose32.cuh): a 16-byte row header, uint32 D = 2^B - 1 then 12 zero bytes, then n little-endian uint32 words, one
 * per sample: bits 0-23 k = D x the expected ALT dosage, bits 24-25 the ploidy p (1 or 2), bit 31 missing (the host
 * writes 0xFFFFFFFF).  A sample is called when bit 31 is clear, p is 1 or 2 and k <= p*D; every other word is a missing
 * sample.  The host writes unphased diploid: 2D - 2*b0 - b1; phased diploid: (D - h0) + (D - h1); haploid: D - b0.  A
 * row whose effect allele is REF (eaidx 0) uses k' = p*D - k.  Tally: nmiss, and neff_num = sum of k' over called
 * samples as an exact integer; neff = fl(neff_num / D) and npc_locus.neff reports neff_num (units of 1/D of that row).
 * Accumulate: scores[s] += fl(fl(k'/D) * beta) (cm for a missing sample) in score-row order, the reference's chain, in
 * every mode.  With D = 255 and diploid samples a row scores bit for bit as the same NPC_GT_DOSE255 row; hard calls
 * (k' = 0, D, 2D) score bit for bit as the same genotypes in int8 GT rows in exact order, haploid samples included.
 *
 * Or, for a context created with gt_width = NPC_GT_PL (ploidy 2), FORMAT/PL rows as the host packs them from a biallelic
 * VCF or BCF record's phred-scaled genotype likelihoods (DESIGN.md 4.10, npc_pl.cuh; NOT in the reference, parity
 * unpinned): n little-endian uint32 words, one per sample.  With m the sample's smallest PL, j the index of its first
 * occurrence and x_g = PL_g - m: bits 0-11 a and bits 12-23 b, the x of the two other genotypes in genotype order, each
 * saturated at 4095 (b = 0 for a haploid sample); bits 24-25 j; bits 26-27 the ploidy (1: 2 PL values, 2: 3 values).
 * The host writes 0xFFFFFFFF for a missing sample; any word with bit 31 set, a ploidy outside {1, 2} or j > ploidy is a
 * missing sample.  All in fp64, round to nearest, no FMA contraction, with p = npc_row.eaf and q = fl(1 - p):
 *   w_g = T[x_g], T[x] = fl(10^(-x/10)) correctly rounded (npc_pl_weight_table), 0 from x = 3237 on;
 *   prior by c = effect-allele copies of g (ALT: c = g; REF: c = 2 - g diploid, 1 - g haploid): diploid pi(0) = fl(q*q),
 *   pi(1) = fl(2*fl(p*q)), pi(2) = fl(p*p); haploid pi(0) = q, pi(1) = p; p NaN or outside [0, 1]: every sample missing;
 *   u_g = fl(pi(c_g) * w_g); den = u_0 + u_1 (+ u_2) left to right; num = fl(u_1 + 2*u_2) (diploid, ALT), fl(2*u_0 + u_1)
 *   (diploid, REF), u_1 (haploid, ALT), u_0 (haploid, REF); the sample is called iff den > 0, then d = fl(num / den).
 * Tally, decision and accumulate as FORMAT/DS rows (npc_set_dosage_rows): nmiss an integer, neff = the fp64 sum of the
 * called d in chunks of 8 samples left to right, a 32-way butterfly, blocks of 256 left to right, npc_locus.neff its IEEE
 * bits; scores[s] += fl(d * beta) (cm for a missing sample) in score-row order, the reference's chain, in every mode.
 * Decisive PLs (every other x >= 3237, 0 < eaf < 1, no underflow in the priors) give d in {0, 1, 2} exactly: such rows
 * score bit for bit as the same genotypes in int8 GT rows in exact order, haploid samples included.
 */
/*
 * Environment (diagnostics and tests; none is needed in normal use):
 *   NPC_FUSED=0              two-kernel sequence instead of the fused tile kernel
 *   NPC_EXACT=1              exact-order mode for every context (as npc_set_exact_order)
 *   NPC_TILE_K / _SR / _SC / _L / _A / _GR / _GD   launch shape of the fused tile kernel (chunks per thread, raw
 *                            stages, index tiles, lag, decider warps, row groups, tiles per decider pass)
 *   NPC_TILE_LONG_MB=<MB>    what counts as a long launch, which may split the grid differently (default 1536, or 192 when short launches split the rows too)
 *   NPC_MULTI=0 | 1          npc_score_resident_multi: never / always the tensor-core contraction (default: >= 3 definitions)
 *   NPC_MULTI_PARTS=<n>      split of a tile's entry range over work units in the contraction (default: chosen from the tile count)
 *   NPC_TIMING=1             phase wall times of npc_score_resident_multi on stderr
 *   NPC_TRACE=1              keep %globaltimer stamps of the tile kernel's CTA 0 (npc_trace)
 */
#ifndef NIMPRESS_CUDA_H
#define NIMPRESS_CUDA_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NPC_OK            0
#define NPC_EINVAL       -1   /* bad argument                                  */
#define NPC_ECUDA        -2   /* CUDA runtime error, or no sm_100 device       */
#define NPC_ENOMEM       -3   /* host or device allocation failed              */
#define NPC_ESTATE       -4   /* call out of sequence (e.g. slot not acquired) */
#define NPC_EUNSUPPORTED -5

/* ImputeMethodLocus / Missing / Sample, declaration order of src/nimpress.nim:412-414 */
enum { NPC_LOCUS_PS = 0, NPC_LOCUS_HOMREF = 1, NPC_LOCUS_FAIL = 2, NPC_LOCUS_IGNORE = 3 };
enum { NPC_MISSING_HOMREF = 0, NPC_MISSING_IGNORE = 1 };
enum { NPC_SAMPLE_PS = 0, NPC_SAMPLE_HOMREF = 1, NPC_SAMPLE_FAIL = 2, NPC_SAMPLE_INT_PS = 3,
       NPC_SAMPLE_INT_FAIL = 4 };

/* npc_row.kind: what the host already decided for the score row.  Same numbering as the
 * class reported back in npc_locus.klass; NPC_CLASS_MAXMIS is only ever an output. */
enum { NPC_KIND_GT = 0,      /* record found, FILTER passes: decode its genotypes          */
       NPC_KIND_NOTCOV = 1,  /* --cov given and locus not covered      (:526-531)           */
       NPC_KIND_ABSENT = 2,  /* findVariant returned nil               (:536-551)           */
       NPC_KIND_FILTER = 3,  /* FILTER not in {".","PASS"}, !ignorefilt (:553-558)          */
       NPC_CLASS_MAXMIS = 4  /* nmissing/n > maxmis                     (:565-571)          */ };

/* gt_width of a context whose rows are PLINK 1 `.bed` rows (SNP-major): ploidy must be 2.  Per sample a 2-bit code,
 * sample s in bits 2*(s%4) of byte s/4: 00 = homozygous A1, 01 = missing, 10 = heterozygous, 11 = homozygous A2, with
 * A2 = REF (eaidx 0) and A1 = the one ALT (eaidx 1); the padding codes of a row's last byte are ignored.  Every
 * npc_score_block* / npc_score_resident call takes such rows (npc_score_resident_multi scores one definition at a time);
 * a GT-kind row names eaidx 0 or 1.  The split count / accumulate calls return NPC_EUNSUPPORTED. */
#define NPC_GT_BED 0

/* gt_width of a context whose rows are fixed-point dosage rows (2 bytes per sample, see above): ploidy must be 2.  Every
 * npc_score_block* / npc_score_resident call takes such rows (npc_score_resident_multi scores one definition at a time);
 * a GT-kind row names eaidx 0 (REF) or 1 (the ALT).  npc_set_exact_order changes nothing: the sums always follow the
 * reference's chain.  The split count / accumulate calls return NPC_EUNSUPPORTED. */
#define NPC_GT_DOSE255 255

/* gt_width of a context whose rows are 32-bit fixed-point dosage rows (a 16-byte header, then 4 bytes per sample, see
 * above): ploidy must be 2.  Calls, effect alleles, exact order and the split calls as for NPC_GT_DOSE255. */
#define NPC_GT_DOSE32 32

/* gt_width of a context whose rows are FORMAT/PL rows (4 bytes per sample, see above): ploidy must be 2.  Calls, effect
 * alleles, exact order and the split calls as for NPC_GT_DOSE255. */
#define NPC_GT_PL 10

/* Bytes of one genotype row of n samples in a layout (gt_width 1, 2, 4, NPC_GT_BED, NPC_GT_DOSE255, NPC_GT_DOSE32 or
 * NPC_GT_PL). */
int64_t npc_gt_row_bytes(int64_t n_samples, int32_t ploidy, int32_t gt_width);

/* The weights of FORMAT/PL rows, no device needed: out[x] = T[x] = fl(10^(-x/10)) correctly rounded for x = 0 .. n - 1
 * (0 from x = 3237 on), the table the PL kernels use. */
int npc_pl_weight_table(double *out, int32_t n);

typedef struct npc_ctx npc_ctx;

typedef struct {
    int32_t imp_locus;     /* NPC_LOCUS_*   (--imp-locus,   default ps)     */
    int32_t imp_missing;   /* NPC_MISSING_* (--imp-missing, default homref) */
    int32_t imp_sample;    /* NPC_SAMPLE_*  (--imp-sample,  default int_ps) */
    int32_t reserved;
    int64_t mincs;         /* --mincs  (default 100)  */
    double  maxmis;        /* --maxmis (default 0.05) */
} npc_policy;

/* One score-file row, in score-file order (ScoreEntry, src/nimpress.nim:221-228, after the
 * host-side lookup).  Several rows may name the same gt_row (different effect alleles). */
typedef struct {
    int32_t gt_row;        /* row of this block's genotype slab; -1 when kind != NPC_KIND_GT */
    int32_t eaidx;         /* 0 = REF is the effect allele, k = k-th ALT (:375-379)          */
    double  beta;
    double  eaf;
    int32_t ref_is_ea;     /* refseq == easeq: the homref dosage is 2.0 instead of 0.0       */
    int32_t kind;          /* NPC_KIND_*                                                     */
} npc_row;

/* Per-row outcome, bit-exact against the reference's decision for that locus. */
typedef struct {
    int32_t klass;         /* 0 OK, else NPC_KIND_NOTCOV/ABSENT/FILTER or NPC_CLASS_MAXMIS   */
    int32_t used;          /* 1 = entered the sum and nloci (getImputedDosages returned true) */
    int32_t eaidx;         /* echo; -1 when the locus had no record                          */
    int32_t reserved;
    int64_t ngt;           /* tallyAlleles (:32-47) as exact integers; -1 when not tallied   */
    int64_t nmiss;
    int64_t neff;
    double  imputed;       /* OK: dosage given to missing samples; else the locus constant   */
} npc_locus;

/* ---- lifetime ------------------------------------------------------------------------- */

/* n_samples: samples held by THIS context (the whole cohort, or this GPU's slab when the
 * sample axis is sharded).  max_rows_per_block bounds both genotype rows and score rows of
 * one npc_score_block* call.  n_slots >= 2 pinned staging slots (0 = no staging ring: only
 * the *_device entry points are usable). */
int  npc_create(npc_ctx **out, int device, int64_t n_samples, int32_t ploidy, int32_t gt_width,
                int64_t max_rows_per_block, int32_t n_slots);
/* The same with the pinned staging slots sized separately: staging_rows (<= max_rows_per_block) rows per
 * slot bound npc_score_block / npc_stage_upload, max_rows_per_block still bounds the score rows of one
 * launch.  A host that uploads into the resident slab wants small slots (pinning costs ~1 ms per MB)
 * and large launches. */
int  npc_create2(npc_ctx **out, int device, int64_t n_samples, int32_t ploidy, int32_t gt_width,
                 int64_t max_rows_per_block, int32_t n_slots, int64_t staging_rows);
/* A context that scores n_keep of the n_row_samples samples its staged rows carry: keep[0..n_keep) ascending, distinct,
 * < n_row_samples.  n_samples of the context is n_keep: sums, tallies, --maxmis, scores_out, launch shapes.  Staging slots
 * (npc_stage_acquire) hold rows of n_row_samples samples; npc_score_block and npc_stage_upload compact them on the device.
 * The *_device entry points, npc_resident_adopt and npc_score_resident_multi take compact rows (the context's layout).
 * A compact row is byte for byte the row of a file holding only the kept samples, in the same order (DESIGN.md 4.11), so
 * scoring through such a context gives exactly what a context of n_keep samples gives on that file.  NPC_EINVAL for
 * a keep list that breaks these rules. */
int npc_create_subset(npc_ctx **out, int device, int64_t n_row_samples, const int64_t *keep, int64_t n_keep, int32_t ploidy,
                      int32_t gt_width, int64_t max_rows_per_block, int32_t n_slots, int64_t staging_rows);
/* The compaction alone, for rows already in device memory (src rows of n_row_samples, dst rows of n_keep; both 16-byte
 * aligned, strides multiples of 16 holding a whole row).  Asynchronous, on the context's stream (npc_set_stream).
 * NPC_ESTATE for a context not created by npc_create_subset. */
int npc_gather_rows_device(npc_ctx *ctx, const void *src, int64_t src_stride, int64_t n_rows, void *dst, int64_t dst_stride);
/* Replaces the keep list of a context made by npc_create_subset, for rows uploaded after this call: keep[0..n_keep)
 * ascending, distinct, below n_row_samples of the context; n_keep must equal the context's.  Rows staged or uploaded
 * before the call (npc_stage_upload, npc_score_block, npc_gather_rows_device) are compacted with the list they were
 * uploaded under: the call waits for those gathers, so flush a half-filled staging slot first.  Several genotype files
 * whose rows carry different samples score through one context this way (DESIGN.md 4.12).  NPC_ESTATE for a context
 * not made by npc_create_subset, NPC_EINVAL for a bad list. */
int npc_set_keep(npc_ctx *ctx, const int64_t *keep, int64_t n_keep);
void npc_destroy(npc_ctx *ctx);
const char *npc_last_error(const npc_ctx *ctx);   /* ctx may be NULL: text of the last npc_create failure */

/* Launch on an existing CUDA stream (cudaStream_t as void*) instead of the context's own;
 * NULL restores the internal stream (so the legacy default stream, whose handle is 0, must be
 * named as cudaStreamLegacy).  For callers that time or order work themselves. */
int npc_set_stream(npc_ctx *ctx, void *cuda_stream);

int npc_set_policy(npc_ctx *ctx, const npc_policy *p);

/* Cohort size used by the --maxmis rule when the sample axis is sharded across contexts
 * (defaults to n_samples). */
int npc_set_cohort_size(npc_ctx *ctx, int64_t n_total);

/* Zero the per-sample sums, nloci and the locus log (and the observed counts, npc_set_observed): start of a
 * computePolygenicScores call (src/nimpress.nim:626-632). */
int npc_reset(npc_ctx *ctx);

/* Not in the reference (DESIGN 4.13).  on != 0: from now on every scoring launch (npc_score_block, npc_score_block_device,
 * npc_score_resident, npc_accumulate_block_device) also adds, per sample, the number of its score rows whose record has
 * class OK (klass 0) and at which the sample has a called genotype -- one with no nmiss count in the layout's tally --
 * into a per-context vector of int64 counts: one more kernel on the context's stream per launch.  Rows of the other
 * classes never count (their dosage is the locus constant).  Loci, not alleles: PLINK's ALLELE_CT is twice this for
 * diploid calls.  npc_reset zeroes the vector; on = 0 stops adding to it.  Off (the default) launches nothing more. */
int npc_set_observed(npc_ctx *ctx, int32_t on);
/* Waits for the submitted work, then copies the context's n_samples counts out.  Variant-sharded contexts: add them
 * (integers: any order).  NPC_ESTATE when npc_set_observed was never turned on. */
int npc_observed(npc_ctx *ctx, int64_t *out);

/* ---- streaming blocks from host memory (pinned, double-buffered) ---------------------- */

/* Blocks until a staging slot is free, then lends it: the caller copies up to
 * max_rows_per_block raw GT rows to gt_host + r * row_stride. */
int npc_stage_acquire(npc_ctx *ctx, int32_t *slot, void **gt_host, int64_t *row_stride);

/* Asynchronous: H2D copy of n_gt_rows rows of `slot`, then for the n_rows score rows
 * count -> decide -> accumulate, in row order.  The slot returns to the ring when the GPU is
 * done with it.  `rows` is copied before the call returns. */
int npc_score_block(npc_ctx *ctx, int32_t slot, int64_t n_gt_rows, const npc_row *rows, int64_t n_rows);

/* ---- blocks already resident in device memory ------------------------------------------ */

/* Same work on a device-resident slab (gt_dev % 16 == 0).  rows: host pointer, or a device
 * pointer when rows_on_device != 0.  Asynchronous. */
int npc_score_block_device(npc_ctx *ctx, const void *gt_dev, int64_t row_stride, int64_t n_gt_rows,
                           const npc_row *rows, int64_t n_rows, int32_t rows_on_device);

/* Split form for a sample-sharded cohort: (1) per-row (nmiss, neff) of this context's slab
 * into counts_dev[n_rows][2] (int64, device), (2) the caller sums counts across contexts
 * (exact integers: any order), (3) decide + accumulate with the summed counts. */
int npc_count_block_device(npc_ctx *ctx, const void *gt_dev, int64_t row_stride, int64_t n_gt_rows,
                           const npc_row *rows, int64_t n_rows, int32_t rows_on_device,
                           int64_t *counts_dev);
int npc_accumulate_block_device(npc_ctx *ctx, const void *gt_dev, int64_t row_stride, int64_t n_gt_rows,
                                const npc_row *rows, int64_t n_rows, int32_t rows_on_device,
                                const int64_t *counts_dev);

/* ---- resident slab: upload first, then score in exact score-file order ----------------- */

/* The reference adds loci to every sample's sum in score-file order, while records arrive in
 * genotype-file order.  A host that wants the reference's summation order bit for bit uploads
 * the matched records' GT rows into a device slab as they stream past (staging ring -> slab),
 * then submits the score rows in score-file order, npc_row.gt_row naming slab rows.  Scoring is
 * two orders of magnitude faster than PCIe, so deferring it costs nothing.
 *
 * npc_resident_reserve: (re)allocate the slab for capacity_rows rows of the context's
 * row_stride; *granted_rows may come back smaller when device memory is short (the caller then
 * scores and refills in rounds). */
int npc_resident_reserve(npc_ctx *ctx, int64_t capacity_rows, int64_t *granted_rows);
/* Asynchronous: copy n_gt_rows staged rows of `slot` to slab rows dst_row.. and return the slot
 * to the ring when the copy is done. */
/* Use caller-owned device memory as the resident slab instead (genotypes already on the GPU):
 * n_gt_rows rows of row_stride bytes (16-byte aligned, a multiple of 16, >= a whole row).  The
 * context never frees it; it must stay valid until the context is destroyed or another slab is
 * reserved / adopted.  npc_stage_upload needs row_stride equal to the staging ring's. */
int npc_resident_adopt(npc_ctx *ctx, const void *gt_dev, int64_t row_stride, int64_t n_gt_rows);
int npc_stage_upload(npc_ctx *ctx, int32_t slot, int64_t n_gt_rows, int64_t dst_row);
/* Asynchronous: count -> decide -> accumulate for n_rows score rows over the slab, in order
 * (any n_rows: split internally into launches of at most max_rows_per_block rows). */
int npc_score_resident(npc_ctx *ctx, const npc_row *rows, int64_t n_rows);

/* Several score definitions over the same resident slab in one call (BASELINE config 4; the
 * reference runs its whole pipeline once per score file, src/nimpress.nim:652-753 per process).
 * For each k < n_scores the outcome is what npc_reset; npc_score_resident(rows[k], n_rows[k]);
 * npc_finish(offsets[k], scores_out[k], &nloci_out[k], loci_out[k], n_rows[k]) gives:
 * scores_out[k][n_samples] normalised, loci_out[k][n_rows[k]] in row order (loci_out or
 * loci_out[k] may be NULL).  Synchronous; the context's own running sums and locus log are
 * overwritten, and its observed counts (npc_set_observed) are left zero.  offsets == NULL: scores_out[k] receives the raw partial sums instead (what
 * npc_partial gives) -- for variant-sharded cohorts, where the caller adds the shards' partials
 * per definition in shard order and applies npc_normalise once.
 *   With three or more definitions on an int8 diploid slab (and exact order off) the sums are
 * formed as one dense contraction on the tensor cores (npc_multi.cuh): the genotypes are read
 * once for the tallies and once per 18 definitions (16 when some imputed contribution is NaN)
 * instead of once per definition.  Per-locus
 * records and nloci are bit-equal to the one-by-one path.  Scores come from exact integer
 * arithmetic on coefficients rounded to a fixed-point grid: per sample they are within
 * 2^-52 * (the definition's largest |coefficient|) per unit of plane value (dosage 0/1/2, 1 for
 * a missing call) per row, plus fp64 rounding, of the exact sum -- an absolute bound, not a
 * relative one (DESIGN 4.5).  Inputs it does not represent (effect-allele index > 62, a
 * definition naming one slab row with one allele more than four times, a coefficient that is
 * infinite or above 1.79e308, more than 2^22 distinct (row, allele) entries) take the one-by-one
 * path.  npc_multi_contractions counts the calls the contraction served. */
int npc_score_resident_multi(npc_ctx *ctx, int32_t n_scores, const npc_row *const *rows, const int64_t *n_rows,
                             const double *offsets, double *const *scores_out, int64_t *nloci_out,
                             npc_locus *const *loci_out);
/* npc_score_resident_multi, and per definition the count of scored loci that used each sample's own genotype
 * (npc_set_observed, DESIGN 4.13): observed_out[k][n_samples], or nothing when observed_out or observed_out[k] is NULL.
 * The counts come from the definitions' records, one pass over the slab per group of up to 8 definitions, whichever
 * path (contraction or one by one) scored them: the same integers either way.  The context's own observed vector
 * (npc_set_observed) is not added to; like its running sums, it is reset: both multi calls leave it zero, on either path. */
int npc_score_resident_multi_observed(npc_ctx *ctx, int32_t n_scores, const npc_row *const *rows, const int64_t *n_rows,
                                      const double *offsets, double *const *scores_out, int64_t *nloci_out,
                                      npc_locus *const *loci_out, int64_t *const *observed_out);

/* ---- results ---------------------------------------------------------------------------- */

/* Waits for all submitted blocks.  scores_out[n_samples] = sum / (2*nloci) + offset
 * (:643-649; nloci == 0 gives NaN like the reference).  loci_out (may be NULL) receives the
 * per-row outcomes of every row submitted since npc_reset, in submission order. */
int npc_finish(npc_ctx *ctx, double offset, double *scores_out, int64_t *nloci_out,
               npc_locus *loci_out, int64_t loci_cap, int64_t *n_loci_out);

/* Variant-sharded cohorts: each context yields its raw partial sums and nloci; the caller
 * adds partials in shard order and applies npc_normalise once. */
int npc_partial(npc_ctx *ctx, double *sums_out, int64_t *nloci_out,
                npc_locus *loci_out, int64_t loci_cap, int64_t *n_loci_out);
int npc_partial_device_ptr(npc_ctx *ctx, double **sums_dev, int64_t **nloci_dev);
/* sums[i] = sums[i] / (2*nloci) + offset on host memory: the reference's epilogue. */
void npc_normalise(double *sums, int64_t n, int64_t nloci, double offset);

/* ---- several GPUs: the combine of a variant-sharded run (SURVEY.md 8b/8e) ------------------- */

/* Replaces nothing the reference has -- it is single-process, single-threaded -- but is what makes
 * `scores[i] += dosages[i]*beta` over ALL loci (src/nimpress.nim:634-641) and the one normalisation
 * (:643-649) come out of several GPUs: the score rows are partitioned into contiguous ranges in
 * score-file order, context k scores range k over all samples, and the combine adds the raw partial
 * sums in context order -- total[s] = ((p0[s] + p1[s]) + p2[s]) + ... -- a fixed order, so the result
 * does not depend on the transport or on the number of ranks that computed each partial.  nloci is
 * summed; a NaN in any partial propagates like the reference's.
 *
 * npc_reduce: ONE process, one context per GPU (ctxs[0..n_ctx) in score-file order of their ranges,
 * all with the same n_samples).  Waits for every context's submitted work; one kernel on ctxs[0]'s
 * device reads the other partials through NVLink peer mappings (bridged by peer copies when the
 * devices cannot map each other).  offset != NULL: scores_out[s] = total / (2*nloci) + *offset (the
 * reference's epilogue); offset == NULL: the raw total.  Synchronous.  Per-locus records stay with
 * the context that scored the row (npc_partial). */
int npc_reduce(npc_ctx *const *ctxs, int32_t n_ctx, const double *offset, double *scores_out, int64_t *nloci_out);

/* One process PER GPU: NCCL, bound at run time with dlopen("libnccl.so.2") -- no link-time dependency;
 * NPC_EUNSUPPORTED when the library is absent.  Rank 0 calls npc_comm_unique_id and hands the 128
 * bytes to the other ranks by whatever channel the host has; every rank then calls npc_comm_init
 * (collective), and after scoring its range npc_comm_combine (collective, rank order = score-file
 * order): all-gather of the partial sums over NVLink, the same fixed-order add on every rank, an
 * all-reduce of nloci.  scores_out and nloci_out both NULL: asynchronous on the context's stream,
 * the result stays on the device (npc_combined_device_ptr). */
int npc_comm_unique_id(uint8_t *id128);
int npc_comm_init(npc_ctx *ctx, const uint8_t *id128, int32_t rank, int32_t world);
int npc_comm_combine(npc_ctx *ctx, const double *offset, double *scores_out, int64_t *nloci_out);
int npc_combined_device_ptr(npc_ctx *ctx, double **scores_dev, int64_t **nloci_dev);
/* Sample-sharded cohorts over NCCL: sums counts_dev[n_rows][2] (what npc_count_block_device wrote on each rank's
 * slab of the samples) over the ranks, in place, on the context's stream -- exact integers, any order.  Then
 * npc_set_cohort_size(total) + npc_accumulate_block_device; every rank keeps the scores of its own samples. */
int npc_comm_sum_counts(npc_ctx *ctx, int64_t *counts_dev, int64_t n_rows);

/* Kernels this context has launched since creation (bench.py's gpu_launches). */
int64_t npc_launch_count(const npc_ctx *ctx);
int64_t npc_multi_contractions(const npc_ctx *ctx);

/* Summation order of the int8 diploid fused kernels.  on = 0 (default): a tile of four score
 * rows is summed first and then added to each sample's running sum -- same rounded products
 * fl(dosage*beta) as the reference, different association, scores within a few ulp of the running
 * sum (<= 1e-12 relative in the tests; contract 1e-9).  on = 1: every product is added in
 * score-row order like `scores[i] += dosages[i]*beta` (src/nimpress.nim:639-640): bit-identical
 * to the reference's chain, at about 85% of the default mode's speed.  The generic (int16/int32/
 * other ploidy) kernels and the split count/accumulate calls are always exact. */
int npc_set_exact_order(npc_ctx *ctx, int32_t on);

/* FORMAT/DS rows instead of hard calls (SURVEY.md 8f-4; NOT in the reference, which reads GT only --
 * src/nimpress.nim:384 -- and lists dosage input under "Future", README.md:162-165).  The context must
 * have been created with ploidy = 1, gt_width = 4: a row is n_samples BCF floats, the expected dosage of
 * the ALT allele (missing 0x7F800001, vector_end 0x7F800002 and NaN = no call).  Raw dosage = ds for
 * eaidx 1, 2 - ds for eaidx 0; everything after that is the reference's logic on a real-valued dosage:
 * tallies (npc_locus.neff then holds the IEEE-754 bits of the fp64 sum of called dosages, added in the
 * fixed order npc_dosage.cuh defines), --maxmis, locus / sample imputation, scores[s] += fl(d*beta) in
 * score-row order.  All npc_score_block* / npc_score_resident calls then take such rows; the split
 * count / accumulate calls and npc_score_resident_multi's contraction do not (the latter scores one by
 * one). */
int npc_set_dosage_rows(npc_ctx *ctx, int32_t on);

/* Which kernels npc_score_block* uses for this context: shape[0] = 2 for the fused tile kernel in
 * its default mode, 1 in exact-order mode (int8 / int16 diploid cohorts that fit one resident pass),
 * 3 for cohorts too wide for that (> ~1.2 M samples per GPU: tally + decide over all samples, then the
 * tile kernel in "decided" mode once per slab of the sample axis), 4 for NPC_GT_BED rows (k_count_chunks,
 * k_decide, k_accum_bed; then shape[1] = CTAs of the accumulate pass, shape[2] = warps per CTA,
 * shape[3] = samples per thread, shape[4] = rows per tile: 4 in the default mode, 1 in exact order),
 * 5 for NPC_GT_DOSE255 rows (k_count_chunks, k_decide, k_accum_dose255; then shape[1] = CTAs of the
 * accumulate pass, shape[2] = warps per CTA, shape[3] = 8 samples per thread), 6 for NPC_GT_DOSE32 rows (k_count_chunks,
 * k_decide, k_accum_dose32; shape[1..3] as for 5, with 4 samples per thread), 7 for NPC_GT_PL rows (k_count_pl,
 * k_decide, k_accum_pl; shape[1..3] as for 6), 0 for the count/decide/accumulate sequence; then grid (tile kernel: sample slabs * 1000 + row
 * groups), consumer warps, chunks per thread, rows
 * per tile, raw stages * 1000 + index-ring tiles, lag * 100 + tiles per decider pass * 10 + decider warps, dynamic
 * shared-memory bytes. */
int npc_kernel_shape(const npc_ctx *ctx, int32_t shape[8]);
/* The same for a launch of n_rows score rows: in the default mode a launch of >= 1.5 GB of genotypes (192 MB for cohorts whose short launches split the rows too) may use another
 * split of the grid (more row groups, better-filled warps) than a short one; npc_kernel_shape = npc_kernel_shape2(ctx, 0, ..). */
int npc_kernel_shape2(const npc_ctx *ctx, int64_t n_rows, int32_t shape[8]);
/* The launch-shape choice alone, no device needed (host arithmetic; used by the CPU tests to check every cohort size):
 * what a context of n_samples diploid samples of gt_width bytes on a GPU with num_sms SMs and max_smem bytes of
 * shared memory per CTA would launch for a block of n_rows rows.  plan = { mode (0: generic kernels, 2: tile kernel,
 * 1: exact order, 3: decided-mode slabs), sample slabs, row groups, chunks per thread K, consumer warps, cells * 16 W bytes,
 * raw stages, index-ring tiles, lag, decider warps, tiles per decider pass, shared-memory bytes, threads per CTA, most
 * consumer warps of the kernel instance, sample slabs of the wide mode, samples per such slab }. */
int npc_plan_shape(int64_t n_samples, int32_t gt_width, int32_t num_sms, int32_t max_smem, int64_t n_rows, int32_t exact,
                   int32_t plan[16]);
/* NPC_TRACE=1 at npc_create: %globaltimer stamps (ns) of CTA 0 of the last tile-kernel launch -- launch start, code
 * tables ready, first tile counted, last tile counted, last tile accumulated, sums stored -- for the launch-floor
 * analysis of short launches (profiles/). */
int npc_trace(npc_ctx *ctx, uint64_t out[8]);
/* ---- utilities (tests / bench) ----------------------------------------------------------- */

/* Deterministic synthetic cohort written straight into device memory: int8 diploid GT rows
 * for variants v0..v0+n_rows, a pure function of (seed, variant, sample); per-row arrays are
 * device pointers.  Byte-identical to the oracle's generator. */
int npc_synth_fill_device(npc_ctx *ctx, void *gt_dev, int64_t row_stride, int64_t v0, int64_t n_rows,
                          uint64_t seed, const uint32_t *af_thr16_dev, const uint32_t *miss_thr24_dev,
                          const int32_t *alt_code_dev);

int npc_version(void);
/* Create the CUDA context of `device` (driver initialisation + primary context: most of a short run's start-up),
 * so that a host can do it on a thread of its own while it parses its inputs. */
int npc_warmup(int device);

#ifdef __cplusplus
}
#endif
#endif
