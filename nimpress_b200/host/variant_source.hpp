// variant_source.hpp -- streaming reader of VCF text / BCF2, plain, gzip or BGZF, written against
// zlib only.  It stands in for what the reference gets from hts-nim/htslib (third-party, not in
// the reference tree): sample names, and per record CHROM, POS, rlen, REF, ALT, FILTER and the
// FORMAT/GT payload.  For BCF the GT payload is handed out as the raw typed-value bytes of the
// record -- exactly the slab the CUDA kernels decode -- without widening or per-sample parsing;
// for VCF text the GT strings are encoded the way htslib's vcf_parse_format encodes them.
#pragma once
#include <zlib.h>

#include <cstdint>
#include <cstdio>
#include <memory>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

#include "util.hpp"

namespace nph {

class BgzfPool;
struct FastInflateTables;                                      // multi-threaded BGZF block inflater (variant_source.cpp)

// Byte stream over a plain / gzip / BGZF file.  BGZF (concatenated <= 64 KiB gzip members with a
// `BC` extra field giving each member's size) is inflated by a pool of worker threads, blocks
// delivered in file order; plain gzip falls back to one sequential zlib stream.  This is the
// replacement for htslib's bgzf reader (which the reference uses single-threaded, hts-nim's
// default threads = 0).  NIMPRESS_THREADS sets the pool size (default: min(cores - 1, 32); 1 = sequential).
class InflateStream {
public:
    InflateStream();
    ~InflateStream();
    // seekable: BGZF read one block at a time by one sequential zlib stream, so that the position is
    // known as a virtual offset and seek_virtual can jump (the reader's index-driven region mode)
    bool open(const std::string &path, bool seekable = false);
    bool is_bgzf() const { return bgzf_; }
    void seek_virtual(uint64_t voff);                 // block file offset << 16 | offset inside the inflated block
    uint64_t tell_virtual() const { return (block_coff_ << 16) | (uint64_t)out_pos_; }
    int64_t file_size() const { return file_size_; }
    size_t read(void *dst, size_t n);                 // up to n bytes; 0 at end of stream
    bool read_exact(void *dst, size_t n);
    bool skip(size_t n);                              // false: the stream ended first
    bool getline(std::string &line);                  // strips \n and a preceding \r
    bool peek(void *dst, size_t n);                   // look ahead without consuming (n <= 64)
    int threads() const { return threads_; }
private:
    bool fill();
    FILE *fp_ = nullptr;
    bool compressed_ = false, zinit_ = false, eof_ = false, bgzf_ = false, block_mode_ = false;
    uint64_t block_coff_ = 0, in_file_off_ = 0;       // block mode: file offset of the current block / of the next byte to fread
    int64_t file_size_ = 0;
    z_stream zs_{};
    std::vector<uint8_t> in_, out_;
    size_t out_pos_ = 0, out_len_ = 0;
    const uint8_t *cur() const { return pool_ ? pool_data_ : out_.data(); }
    std::unique_ptr<BgzfPool> pool_;
    std::unique_ptr<FastInflateTables> tabs_;
    const uint8_t *pool_data_ = nullptr;
    int threads_ = 1;
};

struct VariantRecord {
    int32_t contig_id = -1;
    const std::string *contig = nullptr;
    int64_t pos = 0;                                  // 1-based
    int64_t rlen = 0;                                 // reference span used for overlap (REF length or INFO/END)
    std::string ref;
    std::vector<std::string> alts;
    std::string filter;                               // ".", "PASS" or ';'-joined names
    bool has_gt = false;
    int gt_width = 1, ploidy = 0;                     // bytes per value, values per sample            } after
    const uint8_t *gt = nullptr;                      // n_samples * ploidy * gt_width bytes, until next() } load_gt()
    int64_t end() const { return pos + rlen - 1; }    // 1-based inclusive
};

class RegionIndex;

class VariantSource {
public:
    VariantSource();
    virtual ~VariantSource();
    // false at end of file; throws InputError on corrupt input.  With regions set (use_regions) only
    // records that can overlap one of them are returned, the rest of the file is skipped by seeking.
    bool next(VariantRecord &rec);
    // Restrict the pass to records overlapping these 1-based inclusive spans per contig, using the
    // file's .tbi / .csi index.  false (and nothing changes) when there is no usable index, the file is
    // not BGZF, or the spans cover so much of the file that streaming it with the inflate pool is faster.
    bool use_regions(const std::unordered_map<std::string, std::vector<std::pair<int64_t, int64_t>>> &spans, const std::string &path);
    int64_t seeks() const { return seeks_; }
    // Fills rec.gt / ploidy / gt_width of the record next() just returned (rec.has_gt tells whether
    // it has a GT field).  Text VCF parses its genotype columns only here; BCF has them already.
    virtual void load_gt(VariantRecord &) {}
    // The same, but when the record's GT layout is (want_width, want_ploidy) the payload is written to dst and rec.gt = dst
    // (true); otherwise as load_gt (false: rec.gt points into the reader's buffer, the caller converts or restarts).
    virtual bool load_gt_into(VariantRecord &rec, uint8_t *dst, int want_width, int want_ploidy) {
        (void)dst; (void)want_width; (void)want_ploidy;
        load_gt(rec);
        return false;
    }
    // FORMAT/DS instead of FORMAT/GT (not a reference feature: README.md:162-165 lists dosage input under "Future"):
    // load_gt / load_gt_into then deliver one BCF float per value, gt_width = 4, ploidy = values per sample.
    virtual void set_dosage_mode(bool on) { dosage_ = on; }
    // FORMAT/PL instead of FORMAT/GT (not a reference feature, DESIGN.md 4.10): load_gt / load_gt_into then deliver one packed
    // uint32 word per sample (npc_pl.cuh), gt_width = NPC_GT_PL, ploidy = 2.  A sample with a PL count other than 2 or 3
    // (or none), or a negative PL, throws InputError naming the variant.
    void set_pl_mode(bool on) { pl_ = on; }
    // The one device layout this source's rows come in, or NO_FIXED_LAYOUT for VCF / BCF (whose layout follows the records):
    // NPC_GT_BED for a PLINK 1 fileset (.bed rows as stored, ploidy 2, ceil(n/4) bytes), NPC_GT_DOSE255 for a BGEN file
    // (one uint16 dosage numerator per sample, ploidy 2).  A BGEN file also delivers NPC_GT_DOSE32 rows when load_gt_into
    // asks for them, and throws NeedsDose32 where a matched block does not fit NPC_GT_DOSE255 rows.
    static constexpr int NO_FIXED_LAYOUT = -1;
    virtual int fixed_layout() const { return NO_FIXED_LAYOUT; }
    // Rows that load_gt_into handed to worker threads are complete once this returns; a worker's InputError is rethrown
    // here.  Call before the rows' bytes are read.
    virtual void wait_rows() {}
    bool dosage_mode() const { return dosage_; }
    bool pl_mode() const { return pl_; }
    const std::vector<std::string> &samples() const { return samples_; }
    int64_t n_samples() const { return (int64_t)samples_.size(); }
protected:
    virtual bool next_raw(VariantRecord &rec) = 0;
    virtual InflateStream *stream() = 0;
    virtual int contig_rank(const VariantRecord &rec) const = 0;      // position of the record's contig in the index's order, -1 unknown
    virtual int contig_rank(const std::string &name) const = 0;
    virtual void after_seek() {}                                      // forget whatever of the previous record was still unread
    virtual bool index_names_contigs() const { return true; }         // text VCF: the index must carry the contig names
    std::vector<std::string> samples_;
    std::unique_ptr<RegionIndex> index_;
    bool dosage_ = false, pl_ = false;
private:
    struct Region { int ref; int64_t beg0, end0; };                   // 0-based half open
    std::vector<Region> regions_;
    size_t region_ = 0;
    bool filtering_ = false, positioned_ = false;
    int64_t seeks_ = 0;
};

// A matched BGEN genotype block that 2-byte dosage rows (NPC_GT_DOSE255) cannot hold and 32-bit rows (NPC_GT_DOSE32) can:
// a bit depth other than 8, or samples that are not all diploid.  The driver restarts its pass with NPC_GT_DOSE32 rows;
// to any other caller it is the InputError that names the variant.
struct NeedsDose32 : InputError {
    using InputError::InputError;
};

// nullptr: the file cannot be opened or is neither VCF, BCF, a PLINK 1 .bed nor a BGEN file (the reference: open() == false);
// for a .bed also when its .bim or .fam sibling cannot be opened, for a BGEN file without sample identifiers when its
// .sample cannot be opened.  A malformed fileset or BGEN header throws InputError (see PlinkSource, BgenSource).
// seekable: read BGZF block by block with one zlib stream so that VariantSource::use_regions can jump (no inflate pool).
std::unique_ptr<VariantSource> open_variant_source(const std::string &path, bool seekable = false);

}  // namespace nph
