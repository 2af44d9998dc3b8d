// driver.hpp -- host side of computePolygenicScores (src/nimpress.nim:592-649) over the CUDA
// C ABI.  The host keeps what the reference does per locus on strings and files -- coverage
// lookup, findVariant, the FILTER test, eaidx -- and hands decode / tally / decision /
// imputation / accumulation to libnimpress_cuda.
#pragma once
#include <cstdint>
#include <memory>
#include <string>
#include <unordered_map>
#include <vector>

#include "../../include/nimpress_cuda.h"
#include "inputs.hpp"
#include "variant_source.hpp"

namespace nph {

// enums mirror ImputeMethodLocus / Missing / Sample (src/nimpress.nim:412-414)
struct ScoreParams {
    int imp_locus = NPC_LOCUS_PS;          // --imp-locus   [default: ps]
    int imp_missing = NPC_MISSING_HOMREF;  // --imp-missing [default: homref]
    int imp_sample = NPC_SAMPLE_INT_PS;    // --imp-sample  [default: int_ps]
    double maxmis = 0.05;                  // --maxmis
    double afmisp = 0.001;                 // --afmisp
    int64_t mincs = 100;                   // --mincs
    bool ignorefilt = false;               // --ignorefilt
    bool use_cov = false;                  // --cov given (restrictToCoveredRgns)
    int device = 0;                        // CUDA device (not a reference option)
    std::vector<int> devices;              // several GPUs: the score rows are split into contiguous ranges, one per device (empty: `device`)
    bool exact_order = false;              // npc_set_exact_order: bit-for-bit reference summation order
    bool use_ds = false;                   // score FORMAT/DS (fp32 expected ALT dosage) instead of FORMAT/GT -- not a reference option
    bool use_pl = false;                   // score FORMAT/PL as posterior expected dosages (NPC_GT_PL rows) -- not a reference option
    std::string samples_path;              // --samples: a list of sample names (empty: every sample) -- not a reference option
    bool exclude_samples = false;          // --samples=^FILE: score every sample the list does not name
};

struct ScoreResult {
    std::vector<std::string> samples;
    std::vector<double> scores;            // per sample, after /(2*nloci) and +offset
    std::vector<npc_locus> loci;           // per score row, score-file order
    int64_t nloci = 0;
    std::string warnings;                  // the "WARN ..." lines the reference logs, in its order
    int64_t devices = 1;                   // GPUs that scored (npc_reduce combined their partial sums when > 1)
    int64_t records_read = 0, records_matched = 0, rounds = 0, index_seeks = 0;   // index_seeks > 0: the .tbi / .csi index was used
};

// Host-side part of getImputedDosages that needs no genotypes: coverage (:526), the streaming
// equivalent of findVariant (:353-364: first record in file order overlapping contig:pos-stop with
// REF == refseq and the effect allele equal to REF or present in ALT), eaidx (:375-379) and the
// FILTER test (:553).  Pure CPU: unit-tested without a GPU.
class Matcher {
public:
    Matcher(const ScoreFile &score, const GenomeIntervals &cov, const ScoreParams &p);
    // entries settled by this record (their kind / eaidx / filter text are set); empty if none
    const std::vector<int64_t> &match(const VariantRecord &rec);
    const std::vector<int64_t> &match_last() const { return hits_; }   // what the last match() returned
    void finish();                                  // everything still pending is ABSENT (:536)
    bool has_contig(const std::string &c) const { return index_.count(c) != 0; }
    int64_t n_lookup() const { return n_lookup_; }
    // 1-based inclusive [pos, stop] of every entry that needs a record lookup, per contig (for the index-driven reader)
    void add_spans(std::unordered_map<std::string, std::vector<std::pair<int64_t, int64_t>>> &spans) const;

    static constexpr int32_t PENDING = -1;
    std::vector<int32_t> kind, eaidx;               // per score entry; kind is NPC_KIND_* or PENDING
    std::vector<std::string> filter_text;           // FILTER string of the matched record (FILTER rows)
    std::vector<uint8_t> contig_in_bed;
private:
    struct ContigIndex { std::vector<std::pair<int64_t, int64_t>> by_pos; int64_t max_reflen = 1; };
    const std::vector<ScoreEntry> &E_;
    bool ignorefilt_;
    std::unordered_map<std::string, ContigIndex> index_;
    std::vector<int64_t> hits_;
    int64_t n_lookup_ = 0;
};

// --samples: the samples of `file_samples` (the genotype file's names, in its order) to score, as ascending indices; an
// empty result means every sample (also when the list keeps them all).  The list file holds one name per line (the whole
// line, a trailing \r stripped, blank lines skipped).  A keep list naming a sample the file lacks or naming one twice, a
// listed name occurring more than once in the file, an empty subset or an unreadable list throw InputError; names of an
// exclude list that the file lacks are ignored.
std::vector<int64_t> sample_subset(const std::vector<std::string> &file_samples, const std::string &list_path, bool exclude);

using Spans = std::unordered_map<std::string, std::vector<std::pair<int64_t, int64_t>>>;   // per contig, 1-based inclusive

// The genotype files of one run, read one after the other as their concatenation (DESIGN.md 4.12).
struct GenotypeFiles {
    std::vector<std::string> paths;
    std::vector<uint8_t> seekable;                     // per file: try its index-driven pass when it is read
    std::vector<std::unique_ptr<VariantSource>> src;   // per file while open: file 0 from open(), the others from prepare()
    int kind = VariantSource::NO_FIXED_LAYOUT;         // the files' common fixed_layout()
    std::vector<std::vector<int64_t>> keep;            // per file: its scored samples, ascending; empty: every file scores all of its samples
    std::vector<std::string> names;                    // the scored samples, in order
    int64_t n_row = 0;                                 // samples of the widest file

    explicit GenotypeFiles(const std::vector<std::string> &paths) : paths(paths), seekable(paths.size(), 1) {}
    // Opens every file in turn, checks that they are of one kind (VCF text and BCF, or PLINK 1 filesets, or BGEN) and
    // resolves --samples per file; the kept names must be the same sequence in every file.  Only file 0 stays open.  false,
    // with *unopened = its path, at the first file that cannot be opened; InputError for mixed kinds or differing samples.
    bool open(const ScoreParams &p, std::string *unopened);
    void set_modes(bool ds, bool pl);                  // set_dosage_mode / set_pl_mode of every source, also of one reopened later
    // Before file f is read: open it if it is closed, restrict it to these spans by its .tbi / .csi when seekable[f] and the
    // index allows it, otherwise (re)open it to be streamed (false: it cannot be opened).
    bool prepare(size_t f, const Spans &spans);
private:
    bool reopen(size_t f, bool block_mode);
    bool ds_ = false, pl_ = false;
    std::vector<uint8_t> opened_seekable_;             // per file: its source reads block by block (no inflate pool)
};

// Throws InputError where the reference raises; std::runtime_error on CUDA / library failure.
// false: the genotype file cannot be opened (the reference: FATAL + quit(-1), :728-730).
bool compute_polygenic_scores(const ScoreFile &score, const std::string &genotype_path, const GenomeIntervals &cov,
                              const ScoreParams &p, ScoreResult &out);

// Several score files over ONE pass of the genotype file (BASELINE config 4).  Each result is what
// compute_polygenic_scores gives for that file alone (the reference: one nimpress run per file).
bool compute_polygenic_scores_multi(const std::vector<const ScoreFile *> &scores, const std::string &genotype_path,
                                    const GenomeIntervals &cov, const ScoreParams &p, std::vector<ScoreResult> &outs);

// The same over several genotype files, exactly as over their concatenation (DESIGN.md 4.12).  false: a genotype file
// cannot be opened (*unopened, when given, names it).
bool compute_polygenic_scores_files(const std::vector<const ScoreFile *> &scores, const std::vector<std::string> &genotype_paths,
                                    const GenomeIntervals &cov, const ScoreParams &p, std::vector<ScoreResult> &outs,
                                    std::string *unopened = nullptr);

}  // namespace nph
