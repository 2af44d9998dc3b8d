// region_index.hpp -- tabix (.tbi) and CSI (.csi) indexes, read only.
//
// The reference reaches every score locus with an index query (findVariant, src/nimpress.nim:353-364:
// genotypeVcf.query(contig:pos-stop) through hts-nim / htslib), so a 700-locus score on a genome-wide
// file touches a few hundred BGZF blocks.  This engine streams the file instead and needs no index;
// when one is present AND the score's loci cover little of the file, the reader uses it to skip the
// stretches no locus can overlap.  Which records reach the matcher then differs, what it matches does
// not: a record overlapping a locus is never skipped (the index names the first record overlapping a
// window / bin, and records are sorted by start).
#pragma once
#include <cstdint>
#include <memory>
#include <string>
#include <unordered_map>
#include <utility>
#include <vector>

namespace nph {

class RegionIndex {
public:
    static constexpr uint64_t NONE = ~0ull;
    // <path>.tbi, then <path>.csi; nullptr when neither exists or parses
    static std::unique_ptr<RegionIndex> load(const std::string &data_path);
    // whether load() can find an index for data_path at all: <data_path>.tbi or .csi, not older than the data file
    static bool present(const std::string &data_path);
    // Virtual file offset (BGZF: block offset << 16 | offset in block) from which every record of
    // reference `ref` overlapping [beg0, end0) (0-based, half open) lies at or after; NONE: no such record.
    uint64_t query_start(int ref, int64_t beg0, int64_t end0) const;
    const std::vector<std::string> &names() const { return names_; }     // tabix: contig names in index order; CSI of a BCF: empty
    int n_ref() const { return (int)refs_.size(); }
private:
    struct Bin { uint64_t loff = 0; std::vector<std::pair<uint64_t, uint64_t>> chunks; };
    struct Ref { std::unordered_map<uint32_t, Bin> bins; std::vector<uint64_t> ioff; };
    bool parse(const std::vector<uint8_t> &d, bool csi);
    std::vector<std::string> names_;
    std::vector<Ref> refs_;
    bool csi_ = false;
    int min_shift_ = 14, depth_ = 5;
};

}  // namespace nph
