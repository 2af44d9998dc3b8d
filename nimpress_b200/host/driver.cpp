#include "driver.hpp"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <fstream>
#include <stdexcept>
#include <future>
#include <map>
#include <mutex>
#include <thread>
#include <unordered_map>
#include <unordered_set>

#include "region_index.hpp"
#include "stats.hpp"

namespace nph {

namespace {

struct Ctx {                                       // RAII over npc_ctx
    npc_ctx *h = nullptr;
    ~Ctx() { if (h) npc_destroy(h); }
    void ck(int rc, const char *what) const {
        if (rc != NPC_OK) throw std::runtime_error(std::string(what) + ": " + npc_last_error(h) + " (rc " + std::to_string(rc) + ")");
    }
};

// Re-encode one record's GT payload into the context layout (width w_dst, ploidy p_dst): wider
// integers with the sentinels translated, missing trailing values padded with vector_end --
// exactly the values htslib would hand the reference after widening.
bool convert_gt(const VariantRecord &rec, int64_t n, int w_dst, int p_dst, uint8_t *dst) {
    if (rec.ploidy > p_dst || rec.gt_width > w_dst) return false;
    auto load = [&](int64_t j) -> int64_t {
        if (rec.gt_width == 1) { int8_t v = ((const int8_t *)rec.gt)[j]; return v == INT8_MIN ? INT64_MIN : v == INT8_MIN + 1 ? INT64_MIN + 1 : v; }
        if (rec.gt_width == 2) { int16_t v; memcpy(&v, rec.gt + 2 * j, 2); return v == INT16_MIN ? INT64_MIN : v == INT16_MIN + 1 ? INT64_MIN + 1 : v; }
        int32_t v; memcpy(&v, rec.gt + 4 * j, 4); return v == INT32_MIN ? INT64_MIN : v == INT32_MIN + 1 ? INT64_MIN + 1 : v;
    };
    auto store = [&](int64_t j, int64_t v) {
        if (w_dst == 1) ((int8_t *)dst)[j] = v == INT64_MIN ? INT8_MIN : v == INT64_MIN + 1 ? INT8_MIN + 1 : (int8_t)v;
        else if (w_dst == 2) { int16_t t = v == INT64_MIN ? INT16_MIN : v == INT64_MIN + 1 ? INT16_MIN + 1 : (int16_t)v; memcpy(dst + 2 * j, &t, 2); }
        else { int32_t t = v == INT64_MIN ? INT32_MIN : v == INT64_MIN + 1 ? INT32_MIN + 1 : (int32_t)v; memcpy(dst + 4 * j, &t, 4); }
    };
    for (int64_t i = 0; i < n; i++)
        for (int k = 0; k < p_dst; k++) store(i * p_dst + k, k < rec.ploidy ? load(i * rec.ploidy + k) : INT64_MIN + 1);
    return true;
}

}  // namespace

Matcher::Matcher(const ScoreFile &score, const GenomeIntervals &cov, const ScoreParams &p)
    : E_(score.entries), ignorefilt_(p.ignorefilt) {
    const int64_t nE = (int64_t)E_.size();
    kind.assign(nE, PENDING); eaidx.assign(nE, -1); filter_text.assign(nE, std::string()); contig_in_bed.assign(nE, 1);
    for (int64_t i = 0; i < nE; i++) {
        if (p.use_cov) {                                            // :526, isVariantCovered :313-345
            contig_in_bed[i] = cov.has_contig(E_[i].contig);
            if (!cov.covers(E_[i])) { kind[i] = NPC_KIND_NOTCOV; continue; }   // the reference never looks these up
        }
        ContigIndex &ci = index_[E_[i].contig];
        ci.by_pos.emplace_back(E_[i].pos, i);
        ci.max_reflen = std::max<int64_t>(ci.max_reflen, (int64_t)E_[i].refseq.size());
    }
    for (auto &kv : index_) std::sort(kv.second.by_pos.begin(), kv.second.by_pos.end());
}

const std::vector<int64_t> &Matcher::match(const VariantRecord &rec) {
    hits_.clear();
    auto it = index_.find(*rec.contig);
    if (it == index_.end()) return hits_;
    const ContigIndex &ci = it->second;
    // entries overlapping [rec.pos, rec.end()]: entry.pos <= rec.end and entry.stop >= rec.pos
    auto lo = std::lower_bound(ci.by_pos.begin(), ci.by_pos.end(), std::make_pair(rec.pos - ci.max_reflen + 1, (int64_t)-1));
    for (auto q = lo; q != ci.by_pos.end() && q->first <= rec.end(); ++q) {
        const int64_t i = q->second;
        if (kind[i] != PENDING) continue;                           // an earlier record already matched: first one wins
        const ScoreEntry &e = E_[i];
        if (e.stop() < rec.pos || rec.ref != e.refseq) continue;
        int ea = -1;
        if (e.easeq == e.refseq) ea = 0;
        else for (size_t a = 0; a < rec.alts.size(); a++) if (rec.alts[a] == e.easeq) { ea = (int)a + 1; break; }
        if (ea < 0) continue;
        eaidx[i] = ea;
        const bool filt = !ignorefilt_ && rec.filter != "." && rec.filter != "PASS";          // :553
        kind[i] = filt ? NPC_KIND_FILTER : NPC_KIND_GT;
        if (filt) filter_text[i] = rec.filter;
        hits_.push_back(i);
    }
    return hits_;
}

void Matcher::add_spans(std::unordered_map<std::string, std::vector<std::pair<int64_t, int64_t>>> &spans) const {
    for (const auto &kv : index_) {
        auto &v = spans[kv.first];
        for (const auto &q : kv.second.by_pos) v.emplace_back(E_[q.second].pos, E_[q.second].stop());
    }
}

void Matcher::finish() {
    for (auto &k : kind) if (k == PENDING) k = NPC_KIND_ABSENT;
}

std::vector<int64_t> sample_subset(const std::vector<std::string> &file_samples, const std::string &list_path, bool exclude) {
    std::ifstream in(list_path, std::ios::binary);
    if (!in) throw InputError("--samples: cannot read the sample list " + list_path);
    std::vector<std::string> names;
    for (std::string line; std::getline(in, line);) {
        if (!line.empty() && line.back() == '\r') line.pop_back();
        if (!line.empty()) names.push_back(line);
    }
    if (in.bad()) throw InputError("--samples: cannot read the sample list " + list_path);
    std::unordered_map<std::string, int64_t> index;                  // name -> its index, -1 when the file has it twice
    for (int64_t i = 0; i < (int64_t)file_samples.size(); i++) {
        auto ins = index.emplace(file_samples[i], i);
        if (!ins.second) ins.first->second = -1;
    }
    std::vector<uint8_t> listed(file_samples.size(), 0);
    for (const std::string &nm : names) {
        auto it = index.find(nm);
        if (it == index.end()) {
            if (exclude) continue;                                   // a withdrawal list may name samples of other files
            throw InputError("--samples: sample " + nm + " is not in the genotype file");
        }
        if (it->second < 0) throw InputError("--samples: sample " + nm + " occurs more than once in the genotype file");
        if (listed[it->second] && !exclude) throw InputError("--samples: sample " + nm + " is listed twice");
        listed[it->second] = 1;
    }
    std::vector<int64_t> keep;
    for (int64_t i = 0; i < (int64_t)file_samples.size(); i++) if (listed[i] != exclude) keep.push_back(i);
    if (keep.empty()) throw InputError("--samples: no sample of the genotype file is left to score");
    if ((int64_t)keep.size() == (int64_t)file_samples.size()) keep.clear();        // every sample: the plain path
    return keep;
}

namespace {

const char *kind_name(int fixed) {
    return fixed == NPC_GT_BED ? "a PLINK 1 fileset" : fixed == NPC_GT_DOSE255 ? "BGEN" : "VCF/BCF";
}

// first position at which two name lists differ (the shorter one's length when one is a prefix of the other), -1 if equal
int64_t first_difference(const std::vector<std::string> &a, const std::vector<std::string> &b) {
    const size_t m = std::min(a.size(), b.size());
    for (size_t i = 0; i < m; i++) if (a[i] != b[i]) return (int64_t)i;
    return a.size() == b.size() ? -1 : (int64_t)m;
}

std::string name_at(const std::vector<std::string> &v, int64_t i) {
    return i < (int64_t)v.size() ? v[(size_t)i] : "(none: " + std::to_string(v.size()) + " samples)";
}

}  // namespace

bool GenotypeFiles::open(const ScoreParams &p, std::string *unopened) {
    const size_t F = paths.size();
    src.clear(); src.resize(F);
    opened_seekable_.assign(F, 0);
    n_row = 0;
    keep.assign(F, std::vector<int64_t>());
    std::vector<int64_t> n_file(F);
    std::vector<std::string> kept0;                                            // the names file 0 scores
    bool all = true;                                                           // every file scores all of its samples
    for (size_t f = 0; f < F; f++) {
        // Checked one at a time: a later file is opened (seekable, which starts no inflate threads), checked and closed
        // again, so that hundreds of chunk files do not hold their buffers and descriptors at once; prepare() reopens it.
        std::unique_ptr<VariantSource> v = open_variant_source(paths[f], f == 0 ? seekable[f] != 0 : true);
        if (!v) { if (unopened) *unopened = paths[f]; return false; }
        if (f == 0) kind = v->fixed_layout();
        else if (v->fixed_layout() != kind)
            throw InputError("genotype files " + paths[0] + " (" + kind_name(kind) + ") and " + paths[f] + " (" + kind_name(v->fixed_layout()) +
                             ") are of different kinds: one run reads VCF/BCF files, PLINK 1 filesets or BGEN files");
        n_file[f] = v->n_samples();
        n_row = std::max(n_row, n_file[f]);
        const std::vector<std::string> &s = v->samples();
        if (!p.samples_path.empty()) {
            try {
                keep[f] = sample_subset(s, p.samples_path, p.exclude_samples);
            } catch (const InputError &e) {
                if (F == 1) throw;
                throw InputError("genotype file " + paths[f] + ": " + e.what());
            }
        }
        std::vector<std::string> kept;
        if (keep[f].empty()) kept = s;
        else { all = false; for (int64_t i : keep[f]) kept.push_back(s[(size_t)i]); }
        if (f == 0) {
            kept0 = std::move(kept);
            opened_seekable_[0] = seekable[0];
            src[0] = std::move(v);                                             // file 0 is read next: keep it open
            continue;
        }
        const int64_t d = first_difference(kept0, kept);
        if (d < 0) continue;
        if (p.samples_path.empty())
            throw InputError("genotype file " + paths[f] + ": sample " + std::to_string(d + 1) + " is " + name_at(kept, d) + ", in " + paths[0] +
                             " it is " + name_at(kept0, d) + ": files scored together carry the same samples in the same order "
                             "(--samples=FILE scores the samples it names from every file)");
        throw InputError("--samples: genotype file " + paths[f] + " keeps " + name_at(kept, d) + " as sample " + std::to_string(d + 1) + ", " +
                         paths[0] + " keeps " + name_at(kept0, d) + ": the kept samples must be the same, in the same order, in every file");
    }
    if (kind != VariantSource::NO_FIXED_LAYOUT) seekable.assign(F, 0);          // rows read by offset: no index pass
    names = std::move(kept0);
    if (all) keep.clear();
    else for (size_t f = 0; f < F; f++)
        if (keep[f].empty()) for (int64_t i = 0; i < n_file[f]; i++) keep[f].push_back(i);
    return true;
}

void GenotypeFiles::set_modes(bool ds, bool pl) {
    ds_ = ds; pl_ = pl;
    for (auto &s : src) if (s) { s->set_dosage_mode(ds); s->set_pl_mode(pl); }
}

bool GenotypeFiles::reopen(size_t f, bool block_mode) {
    src[f] = open_variant_source(paths[f], block_mode);
    if (!src[f]) return false;
    opened_seekable_[f] = block_mode;
    src[f]->set_dosage_mode(ds_); src[f]->set_pl_mode(pl_);
    return true;
}

bool GenotypeFiles::prepare(size_t f, const Spans &spans) {
    if (!src[f]) {
        // no .tbi / .csi beside the file: use_regions() would refuse, so open it to be streamed straight away
        if (seekable[f] && !RegionIndex::present(paths[f])) seekable[f] = 0;
        if (!reopen(f, seekable[f] != 0)) return false;
    }
    if (seekable[f]) {
        if (src[f]->use_regions(spans, paths[f])) return true;
        seekable[f] = 0;                                                       // streamed, with the inflate pool, from now on
    } else if (!opened_seekable_[f] || kind != VariantSource::NO_FIXED_LAYOUT) {
        return true;
    }
    return reopen(f, false);
}

namespace {

// NIMPRESS_TIMING=1: phase wall times on stderr
struct PhaseTimer {
    bool on = getenv("NIMPRESS_TIMING") != nullptr;
    std::chrono::steady_clock::time_point t = std::chrono::steady_clock::now();
    void mark(const char *what) {
        auto now = std::chrono::steady_clock::now();
        if (on) fprintf(stderr, "[nimpress timing] %-28s %8.1f ms\n", what, std::chrono::duration<double, std::milli>(now - t).count());
        t = now;
    }
};

// CUDA driver + primary-context creation is most of a short run's start-up (~1 s per process on the boxes seen):
// it is started once per device on a thread of its own as soon as a scoring call begins -- while the inputs are
// opened, indexed and, when there is a .tbi / .csi, consulted -- and waited for only where a context is needed.
std::mutex g_warm_mutex;
std::map<int, std::shared_future<void>> g_warm;
void start_warm(int device) {
    std::lock_guard<std::mutex> g(g_warm_mutex);
    if (!g_warm.count(device)) g_warm[device] = std::async(std::launch::async, [device] { npc_warmup(device); }).share();
}
void wait_warm(int device) {
    std::shared_future<void> f;
    {
        std::lock_guard<std::mutex> g(g_warm_mutex);
        auto it = g_warm.find(device);
        if (it == g_warm.end()) return;
        f = it->second;
    }
    f.wait();
}

struct LayoutOverflow { int width, ploidy; };      // a matched record does not fit the context's GT layout
struct SlabOverflow {};                            // several score files, and their matched rows exceed device memory
struct CannotOpen { std::string path; };           // a genotype file that opened before could not be reopened to be streamed

// The row format of one pass: what the staging rows and the contexts hold
struct RowLayout {
    int width = 1, ploidy = 2;                     // BCF's usual GT layout: int8, diploid
    bool ds = false, pl = false;                   // FORMAT/DS rows (one float per sample), FORMAT/PL rows (one packed word per sample)
    // dosage rows (FORMAT/DS, FORMAT/PL, BGEN): the effect-allele tally is not an integer allele count
    bool real_tally() const { return ds || pl || width == NPC_GT_DOSE255 || width == NPC_GT_DOSE32; }
};

// The layout a pass over genotype files of this kind (GenotypeFiles::kind) starts with; dose32: a BGEN pass met a block
// that only 32-bit dosage rows hold.  InputError when the files cannot give the rows p asks for.
RowLayout row_layout(int kind, const ScoreParams &p, bool dose32) {
    if (p.use_ds && p.use_pl) throw InputError("--pl and --dosage: score either FORMAT/PL or FORMAT/DS");
    if (kind == NPC_GT_BED && p.use_ds) throw InputError("--dosage: a PLINK fileset holds hard calls only, no FORMAT/DS");
    if (kind == NPC_GT_BED && p.use_pl) throw InputError("--pl: a PLINK fileset holds hard calls only, no FORMAT/PL");
    if (kind == NPC_GT_DOSE255 && p.use_pl) throw InputError("--pl: a BGEN file holds genotype probabilities, no FORMAT/PL");
    RowLayout L;
    if (kind != VariantSource::NO_FIXED_LAYOUT) L.width = dose32 ? NPC_GT_DOSE32 : kind;   // BGEN rows are dosages already: --dosage changes nothing
    else if (p.use_ds) { L.width = 4; L.ploidy = 1; L.ds = true; }
    else if (p.use_pl) { L.width = NPC_GT_PL; L.pl = true; }
    return L;
}

// WARN lines of one score file, in the reference's order (:326, :527-530, :538-541, :554-557, :567-570, :575-579)
// real_tally: RowLayout::real_tally() of the pass
std::string make_warnings(const ScoreFile &score, const Matcher &M, const std::vector<npc_locus> &loci, int64_t n, const ScoreParams &p,
                          bool real_tally) {
    std::string w;
    const std::vector<ScoreEntry> &E = score.entries;
    for (int64_t i = 0; i < (int64_t)E.size(); i++) {
        const ScoreEntry &e = E[i];
        const npc_locus &L = loci[i];
        const std::string id = e.contig + ":" + std::to_string(e.pos) + ":" + e.refseq + ":" + e.easeq;
        const std::string span = e.contig + ":" + std::to_string(e.pos) + "-" + std::to_string(e.stop());
        if (L.klass == NPC_KIND_NOTCOV) {
            if (!M.contig_in_bed[i]) w += "WARN Contig " + e.contig + " not present within the coverage BED file.\n";
            w += "WARN Locus " + span + " is not covered by the sequence coverage BED.  Imputing all dosages at this locus.\n";
        } else if (L.klass == NPC_KIND_ABSENT) {
            if (!std::isnan(e.eaf) && binom_test(0, n * 2, e.eaf) < p.afmisp)
                w += "WARN Variant " + id + " cohort EAF is 0 in " + std::to_string(n) + " samples.  This is highly unlikely given polygenic score EAF of " +
                     format_float_nim(e.eaf) + "\n";
        } else if (L.klass == NPC_KIND_FILTER) {
            w += "WARN Variant " + id + " has a FILTER flag set (value \"" + M.filter_text[i] + "\").  Imputing all dosages at this locus.\n";
        } else if (L.klass == NPC_CLASS_MAXMIS) {
            const double missingrate = (double)L.nmiss / (double)n;
            w += "WARN Locus " + span + " has " + format_float_nim(missingrate * 100) +
                 "% of samples missing a genotype. This exceeds the missingness threshold; imputing all dosages at this locus.\n";
        } else if (real_tally) {
            // dosage rows: the tally is a real number, the reference's exact binomial test is not defined on it
        } else if (!std::isnan(e.eaf) && binom_test(L.neff, (n - L.nmiss) * 2, e.eaf) < p.afmisp) {
            w += "WARN Variant " + id + " cohort EAF is " + format_float_nim((double)L.neff / (double)((n - L.nmiss) * 2)) + " in " +
                 std::to_string(n) + " samples.  This is highly unlikely given polygenic score EAF of " + format_float_nim(e.eaf) + "\n";
        }
    }
    return w;
}

// One score file's side of a pass
struct ScoreState {
    const ScoreFile &score;
    Matcher M;
    int D;                                         // devices of the pass
    std::vector<int64_t> slab_row;                 // per entry: row of its device's resident slab
    std::vector<uint8_t> done;                     // per entry: taken by a round
    ScoreState(const ScoreFile &s, const GenomeIntervals &cov, const ScoreParams &p, int D)
        : score(s), M(s, cov, p), D(D), slab_row(s.entries.size(), -1), done(s.entries.size(), 0) {}
    // entry i belongs to device i * D / (entries): contiguous ranges of EVERY file in its own order
    int dev_of(int64_t i) const {
        return D == 1 ? 0 : (int)std::min<int64_t>(D - 1, i * D / std::max<int64_t>((int64_t)score.entries.size(), 1));
    }
};

// Rows of each device's ranges that need a record (an upper bound when score files share records).  One device and
// several score files: entries with the same (contig, pos, ref, ea) settle on the same record, so a key counts once.
std::vector<int64_t> lookup_counts(const std::vector<ScoreState> &ps, int D) {
    const bool dedup = D == 1 && ps.size() > 1;
    std::vector<int64_t> c(D, 0);
    std::unordered_set<std::string> keys;
    for (const ScoreState &s : ps)
        for (int64_t i = 0; i < (int64_t)s.score.entries.size(); i++) if (s.M.kind[i] == Matcher::PENDING) {
            const ScoreEntry &e = s.score.entries[i];
            c[s.dev_of(i)]++;
            if (dedup) keys.insert(e.contig + "\t" + std::to_string(e.pos) + "\t" + e.refseq + "\t" + e.easeq);
        }
    if (dedup) c[0] = (int64_t)keys.size();
    return c;
}

// The rows of score file s that a round takes on device d, in score-file order: a final round takes every row not taken
// yet, an earlier one the rows whose genotypes sit in the slab.  Their entry indices are appended to submitted.
void collect_rows(ScoreState &s, int d, bool final_round, std::vector<npc_row> &rows, std::vector<int64_t> &submitted) {
    const std::vector<ScoreEntry> &E = s.score.entries;
    rows.clear();
    for (int64_t i = 0; i < (int64_t)E.size(); i++) {
        if (s.done[i] || s.dev_of(i) != d) continue;
        const int32_t kind = s.M.kind[i];
        if (!final_round && !(kind == NPC_KIND_GT && s.slab_row[i] >= 0)) continue;
        npc_row r;
        r.gt_row = kind == NPC_KIND_GT ? (int32_t)s.slab_row[i] : -1;
        r.eaidx = s.M.eaidx[i]; r.beta = E[i].beta; r.eaf = E[i].eaf;
        r.ref_is_ea = E[i].ref_is_ea() ? 1 : 0; r.kind = kind;
        rows.push_back(r);
        submitted.push_back(i);
        s.done[i] = 1;
    }
}

// What the contexts of a pass are created with, and the file being read
struct Pass {
    const ScoreParams &p;
    const RowLayout &lay;
    int64_t n, n_row, row_bytes;                   // scored samples, samples of the widest file, bytes of a staging row
    VariantSource *src;                            // the file being read (after the stream: the last one)
    // its keep list, nullptr when every file scores all of its samples: a context opened lazily takes it; one opened after
    // the stream receives no rows, so any file's list serves it
    const int64_t *keep;
    double waited_ms = 0.0;                        // spent opening contexts
};

// Devices: one context per GPU.  With several, the score rows are partitioned into contiguous ranges in
// score-file order (a contig / region partition for a sorted score file): context d scores range d over all
// samples, a matched record is uploaded to the device(s) whose ranges name it, and the partial sums are
// combined in range order by npc_reduce.  Several score files at once: every file is cut into D ranges of its own,
// device d scores range d of every file in one npc_score_resident_multi call (raw partial sums), and the host adds
// the partials of each file in device order and normalises once.
struct Device {
    Pass *pass = nullptr;
    int d = 0, id = 0;                             // index in the pass, CUDA device
    int64_t lookup = 0;                            // rows of its ranges that need a record
    Ctx ctx;
    bool opened = false;
    int32_t slot = -1; uint8_t *stage = nullptr; int64_t stride = 0, staged = 0, slab_base = 0, slab_cap = 0, block_rows = 1, rounds = 0;
    int64_t taken = -1;                            // slab row of the last row take_row() handed out
    std::vector<npc_row> rows; std::vector<int64_t> submitted;   // one score file: this device's rows, entry index of each

    // A context is opened when its first row arrives (or at the end, for its constant rows): contexts come up one after
    // the other inside the driver (~1 s each), and a sorted file reaches the later ranges later -- the first device's
    // rows stream while the others' contexts are still being created.
    void open() {
        if (opened) return;
        const auto t0 = std::chrono::steady_clock::now();
        wait_warm(id);
        const Pass &P = *pass;
        // staging slots of ~8 MB: big enough for efficient H2D copies, small enough that pinning three of them per
        // device does not dominate a short run (pinning costs ~1 ms per MB); scoring launches are sized separately
        const int64_t want = std::max<int64_t>(lookup, 1);
        block_rows = std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>(4096, (8ll << 20) / P.row_bytes + 1), want));
        const int64_t launch_rows = std::max<int64_t>(block_rows, 32768);
        if (!P.keep) ctx.ck(npc_create2(&ctx.h, id, P.n, P.lay.ploidy, P.lay.width, launch_rows, 3, block_rows), "npc_create");
        else ctx.ck(npc_create_subset(&ctx.h, id, P.n_row, P.keep, P.n, P.lay.ploidy, P.lay.width, launch_rows, 3, block_rows),
                    "npc_create_subset");
        const npc_policy pol = { P.p.imp_locus, P.p.imp_missing, P.p.imp_sample, 0, P.p.mincs, P.p.maxmis };
        ctx.ck(npc_set_policy(ctx.h, &pol), "npc_set_policy");
        if (P.lay.ds) ctx.ck(npc_set_dosage_rows(ctx.h, 1), "npc_set_dosage_rows");
        if (P.p.exact_order) ctx.ck(npc_set_exact_order(ctx.h, 1), "npc_set_exact_order");
        if (P.p.observed) ctx.ck(npc_set_observed(ctx.h, 1), "npc_set_observed");      // rounds add up in the context
        ctx.ck(npc_reset(ctx.h), "npc_reset");
        int64_t slab_want = want;
        if (const char *e = getenv("NIMPRESS_SLAB_ROWS")) if (*e) slab_want = std::max<int64_t>(1, std::min<int64_t>(slab_want, atoll(e)));   // tests: force rounds
        ctx.ck(npc_resident_reserve(ctx.h, slab_want, &slab_cap), "npc_resident_reserve");
        pass->waited_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        opened = true;
    }
    // The next staging row (its slab row in `taken`).  A full slab is scored (one score file, ps[0]; several throw
    // SlabOverflow) and refilled from row 0; a slot is acquired when none is held.
    uint8_t *take_row(std::vector<ScoreState> &ps) {
        open();
        if (slab_base + staged >= slab_cap) {
            if (ps.size() > 1) throw SlabOverflow();
            score_round(ps[0], false);
            slab_base = 0;
        }
        if (slot < 0) {
            void *ptr;
            ctx.ck(npc_stage_acquire(ctx.h, &slot, &ptr, &stride), "npc_stage_acquire");
            stage = (uint8_t *)ptr; staged = 0;
        }
        taken = slab_base + staged;
        return stage + staged++ * stride;
    }
    void flush() {                                 // uploads the held slot once the reader's workers have filled its rows
        if (slot < 0) return;
        pass->src->wait_rows();
        ctx.ck(npc_stage_upload(ctx.h, slot, staged, slab_base), "npc_stage_upload");
        slab_base += staged; staged = 0; slot = -1;
    }
    // A round scores rows over the resident slab in score-file order.  The normal case is ONE final round per device
    // holding every row of its range: exactly the reference's loop order (:634-641).  Only when the matched genotype rows
    // exceed device memory are there earlier rounds; those take the rows whose genotypes sit in the slab, and the
    // summation order then differs from the reference's by a reordering of terms (scores agree to ~1 ulp of the partial
    // sums, not bit for bit).  One score file only.
    void score_round(ScoreState &s, bool final_round) {
        flush();
        collect_rows(s, d, final_round, rows, submitted);
        if (!rows.empty()) ctx.ck(npc_score_resident(ctx.h, rows.data(), (int64_t)rows.size()), "npc_score_resident");
        rounds++;
    }
};

std::string record_at(const VariantRecord &rec) { return "record " + *rec.contig + ":" + std::to_string(rec.pos); }

// Fills one staging row from the record src just returned (row_bytes: a row of the file's own samples).  InputError for
// a record these rows cannot take, LayoutOverflow when it needs a wider GT layout.
void load_row(VariantRecord &rec, VariantSource &src, const RowLayout &lay, size_t row_bytes, uint8_t *dst) {
    if (lay.pl && rec.alts.size() != 1)
        throw InputError(record_at(rec) + ": FORMAT/PL rows take biallelic records only (" + std::to_string(rec.alts.size()) +
                         " ALT alleles; split them with bcftools norm -m-)");
    // BCF with the context's layout: the GT payload goes from the inflated blocks straight into the pinned row
    const bool direct = src.load_gt_into(rec, dst, lay.width, lay.ploidy);
    if (!rec.has_gt || !rec.gt)
        throw InputError(record_at(rec) + (lay.pl ? " has no PL field" : lay.ds ? " has no DS field" : " has no GT field"));
    if (lay.ds && (rec.ploidy != 1 || rec.gt_width != 4))
        throw InputError(record_at(rec) + ": FORMAT/DS with several values per sample is not supported");
    if (direct) return;
    if (rec.ploidy > lay.ploidy || rec.gt_width > lay.width)
        throw LayoutOverflow{ std::max(rec.gt_width, lay.width), std::max(rec.ploidy, lay.ploidy) };
    if (rec.gt_width == lay.width && rec.ploidy == lay.ploidy) memcpy(dst, rec.gt, row_bytes);
    else convert_gt(rec, src.n_samples(), lay.width, lay.ploidy, dst);
}

// One streaming pass over the genotype files, one after the other (findVariant :353-364, eaidx :375-379): a record whose
// genotypes a score file needs is staged once on every device whose ranges name it.  Sets the record counters of outs.
void stream_files(GenotypeFiles &files, const Spans &spans, Pass &P, std::vector<ScoreState> &ps, std::vector<Device> &devs,
                  std::vector<ScoreResult> &outs) {
    VariantRecord rec;
    int64_t records_read = 0, records_matched = 0, seeks = 0;
    for (size_t cur = 0; cur < files.src.size(); cur++) {
        if (cur > 0) {
            if (!files.prepare(cur, spans)) throw CannotOpen{ files.paths[cur] };
            P.src = files.src[cur].get();
            if (P.keep) {                             // staged rows of the previous file are compacted with its list
                P.keep = files.keep[cur].data();
                for (Device &v : devs) if (v.opened) {
                    v.flush();
                    v.ctx.ck(npc_set_keep(v.ctx.h, P.keep, P.n), "npc_set_keep");
                }
            }
        }
        VariantSource &src = *P.src;
        const size_t file_row_bytes = (size_t)npc_gt_row_bytes(src.n_samples(), P.lay.ploidy, P.lay.width);   // the front of a staging row
        while (src.next(rec)) {
            records_read++;
            bool any = false;
            uint32_t need_dev = 0;                    // devices that take the record's genotypes
            for (ScoreState &s : ps)
                for (int64_t i : s.M.match(rec)) {
                    any = true;
                    if (s.M.kind[i] == NPC_KIND_GT) need_dev |= 1u << s.dev_of(i);
                }
            if (!any) continue;
            records_matched++;
            if (!need_dev) continue;                  // FILTER-failed: never decoded (:553-558)
            const uint8_t *first = nullptr;
            for (size_t d = 0; d < devs.size(); d++) {
                if (!((need_dev >> d) & 1u)) continue;
                uint8_t *dst = devs[d].take_row(ps);
                if (first) {                          // a record named by two ranges: same bytes
                    src.wait_rows();
                    memcpy(dst, first, file_row_bytes);
                } else {
                    load_row(rec, src, P.lay, file_row_bytes, dst);
                    first = dst;
                }
            }
            for (ScoreState &s : ps)
                for (int64_t i : s.M.match_last()) if (s.M.kind[i] == NPC_KIND_GT) {
                    if (P.lay.ds && s.M.eaidx[i] > 1)
                        throw InputError(record_at(rec) + ": FORMAT/DS rows take the REF or the first ALT as effect allele");
                    s.slab_row[i] = devs[s.dev_of(i)].taken;
                }
            for (Device &v : devs) if (v.slot >= 0 && v.staged == v.block_rows) v.flush();
        }
        src.wait_rows();                              // BGEN workers may still be writing this file's rows into pinned slots
        seeks += src.seeks();
        if (cur + 1 < files.src.size()) { files.src[cur].reset(); P.src = nullptr; }
    }
    for (size_t k = 0; k < ps.size(); k++) {
        ps[k].M.finish();
        outs[k].records_read = records_read; outs[k].records_matched = records_matched; outs[k].index_seeks = seeks;
    }
}

// One score file: every device scores the rest of its range in a final round.  One device's npc_finish gives the scores;
// with several, npc_reduce combines their partial sums in range order and npc_partial gives each one's locus records.
void score_single(ScoreState &s, std::vector<Device> &devs, int64_t n, ScoreResult &out) {
    const int D = (int)devs.size();
    std::vector<npc_ctx *> hs;
    for (Device &v : devs) {
        v.score_round(s, true);
        out.rounds = std::max(out.rounds, v.rounds);
        hs.push_back(v.ctx.h);
    }
    out.scores.assign(n, 0.0);
    out.devices = D;
    if (D > 1) devs[0].ctx.ck(npc_reduce(hs.data(), D, &s.score.offset, out.scores.data(), &out.nloci), "npc_reduce");
    std::vector<double> scratch(D > 1 ? (size_t)std::max<int64_t>(n, 1) : 0);
    for (Device &v : devs) {
        std::vector<npc_locus> log(v.submitted.size());
        int64_t nlog = 0, nl = 0;
        if (D == 1)
            v.ctx.ck(npc_finish(v.ctx.h, s.score.offset, out.scores.data(), &out.nloci, log.data(), (int64_t)log.size(), &nlog), "npc_finish");
        else v.ctx.ck(npc_partial(v.ctx.h, scratch.data(), &nl, log.data(), (int64_t)log.size(), &nlog), "npc_partial");
        if (nlog != (int64_t)v.submitted.size()) throw std::runtime_error("locus log length mismatch");
        for (size_t j = 0; j < log.size(); j++) out.loci[v.submitted[j]] = log[j];
    }
    if (!devs[0].pass->p.observed) return;
    // integer counts: the devices' vectors add up in any order
    out.has_observed = true;
    out.observed.assign((size_t)n, 0);
    std::vector<int64_t> obs((size_t)n);
    for (Device &v : devs) {
        v.ctx.ck(npc_observed(v.ctx.h, obs.data()), "npc_observed");
        for (int64_t i = 0; i < n; i++) out.observed[(size_t)i] += obs[(size_t)i];
    }
}

// Several score files: device d scores range d of every file in one npc_score_resident_multi call.  One device gives the
// normalised scores straight away; several give raw partial sums, device 0's into the scores and the others' added to
// them in device order (= score-file order of the ranges), normalised once.
void score_multi(std::vector<ScoreState> &ps, std::vector<Device> &devs, int64_t n, std::vector<ScoreResult> &outs) {
    const int S = (int)ps.size(), D = (int)devs.size();
    const bool observed = devs[0].pass->p.observed;
    std::vector<std::vector<double>> part(S);
    std::vector<std::vector<int64_t>> obs(S);
    for (int k = 0; k < S; k++) {
        outs[k].scores.assign(n, 0.0); outs[k].rounds = 1; outs[k].devices = D;
        if (D > 1) part[k].assign((size_t)n, 0.0);
        if (observed) { outs[k].has_observed = true; outs[k].observed.assign((size_t)n, 0); obs[k].assign((size_t)n, 0); }
    }
    for (Device &v : devs) {
        v.flush();
        std::vector<std::vector<npc_row>> rows(S);
        std::vector<std::vector<int64_t>> entries(S);
        std::vector<std::vector<npc_locus>> log(S);
        std::vector<const npc_row *> row_ptr(S);
        std::vector<int64_t> n_rows(S), nloci(S);
        std::vector<double> offsets(S);
        std::vector<double *> sc(S);
        std::vector<npc_locus *> log_ptr(S);
        std::vector<int64_t *> obs_ptr(S);
        for (int k = 0; k < S; k++) {
            obs_ptr[k] = observed ? obs[k].data() : nullptr;
            collect_rows(ps[k], v.d, true, rows[k], entries[k]);
            row_ptr[k] = rows[k].data(); n_rows[k] = (int64_t)rows[k].size(); offsets[k] = ps[k].score.offset;
            sc[k] = v.d == 0 ? outs[k].scores.data() : part[k].data();
            log[k].resize(rows[k].size()); log_ptr[k] = log[k].data();
        }
        // one device: normalised scores; several: raw partial sums (offsets = NULL)
        v.ctx.ck(npc_score_resident_multi_observed(v.ctx.h, S, row_ptr.data(), n_rows.data(), D == 1 ? offsets.data() : nullptr, sc.data(),
                                                   nloci.data(), log_ptr.data(), observed ? obs_ptr.data() : nullptr),
                 "npc_score_resident_multi");
        for (int k = 0; k < S; k++) {
            outs[k].nloci += nloci[k];
            if (observed) for (int64_t i = 0; i < n; i++) outs[k].observed[(size_t)i] += obs[k][(size_t)i];
            for (size_t j = 0; j < log[k].size(); j++) outs[k].loci[entries[k][j]] = log[k][j];
            if (v.d > 0) for (int64_t i = 0; i < n; i++) outs[k].scores[i] += part[k][i];
        }
    }
    if (D > 1) for (int k = 0; k < S; k++) npc_normalise(outs[k].scores.data(), n, outs[k].nloci, ps[k].score.offset);
}

// One pass over the genotype files with a fixed row layout, for one score file or several at once
// (BASELINE config 4: every score file sees the same record stream, a record any of them matches
// is uploaded once, and the resident slab is then scored for each file).  Throws LayoutOverflow
// when a matched record needs a wider layout (the caller restarts the pass with it) and
// SlabOverflow when several files are given and their rows do not fit device memory.
// The genotype files are read one after the other as one record stream (DESIGN.md 4.12).  files.keep: the samples each
// file scores, empty for all.  The reader's rows carry a file's own samples, at the front of staging rows sized for the
// widest file (n_row); the devices compact them to the n kept ones (npc_create_subset, npc_set_keep at each file), which
// is all that the contexts, scores and WARN lines see.
void run_pass(const std::vector<const ScoreFile *> &scores, GenotypeFiles &files, const GenomeIntervals &cov, const ScoreParams &p,
              const RowLayout &lay, std::vector<ScoreResult> &outs) {
    const int S = (int)scores.size();
    const int64_t n = (int64_t)files.names.size();
    PhaseTimer timer;
    std::vector<int> dev_ids = p.devices.empty() ? std::vector<int>{ p.device } : p.devices;
    if (const char *e = getenv("NIMPRESS_SPLIT")) if (*e && dev_ids.size() == 1 && atoi(e) > 1)      // tests: several contexts on one GPU
        dev_ids.assign((size_t)std::min(atoi(e), 16), dev_ids[0]);
    const int D = (int)dev_ids.size();
    outs.assign(S, ScoreResult());
    std::vector<ScoreState> ps;
    ps.reserve(S);
    for (int k = 0; k < S; k++) {
        outs[k].samples = files.names;
        outs[k].loci.assign(scores[k]->entries.size(), npc_locus());
        ps.emplace_back(*scores[k], cov, p, D);
    }
    const std::vector<int64_t> lookup = lookup_counts(ps, D);
    Spans spans;                                      // an index next to a file and few loci: read only where loci are
    if (std::count(files.seekable.begin(), files.seekable.end(), 1)) for (const ScoreState &s : ps) s.M.add_spans(spans);
    if (!files.prepare(0, spans)) throw CannotOpen{ files.paths[0] };
    timer.mark("coverage + entry index");

    Pass P{ p, lay, n, files.n_row, std::max<int64_t>(16, npc_gt_row_bytes(files.n_row, lay.ploidy, lay.width)), files.src[0].get(),
            files.keep.empty() ? nullptr : files.keep[0].data() };
    std::vector<Device> devs(D);
    for (int d = 0; d < D; d++) {
        devs[d].pass = &P; devs[d].d = d; devs[d].id = dev_ids[d]; devs[d].lookup = lookup[d];
    }
    // rows still being converted by the source's workers land in the devices' pinned slots: let them finish before the
    // slots go, whichever way this pass ends
    struct RowsGuard {
        VariantSource *&v;
        ~RowsGuard() { try { if (v) v->wait_rows(); } catch (...) {} }
    } rows_guard{ P.src };
    devs[0].open();
    timer.mark("first GPU context + buffers");

    stream_files(files, spans, P, ps, devs, outs);
    timer.mark("stream + match + upload");
    const ScoreResult &o = outs[0];
    if (timer.on) fprintf(stderr, "[nimpress timing] records read %lld, matched %lld, index seeks %lld%s\n", (long long)o.records_read,
                          (long long)o.records_matched, (long long)o.index_seeks, o.index_seeks ? " (.tbi / .csi used)" : "");

    for (Device &v : devs) v.open();
    if (timer.on && D > 1) fprintf(stderr, "[nimpress timing] waited for GPU contexts + buffers, all devices %8.1f ms\n", P.waited_ms);
    if (S == 1) score_single(ps[0], devs, n, outs[0]);
    else score_multi(ps, devs, n, outs);
    timer.mark("score + finish (GPU)");
    for (int k = 0; k < S; k++) outs[k].warnings = make_warnings(*scores[k], ps[k].M, outs[k].loci, n, p, lay.real_tally());
    timer.mark("WARN lines (binomial tests)");
}

}  // namespace

bool compute_polygenic_scores_files(const std::vector<const ScoreFile *> &scores, const std::vector<std::string> &genotype_paths,
                                    const GenomeIntervals &cov, const ScoreParams &p, std::vector<ScoreResult> &outs, std::string *unopened) {
    for (int d : (p.devices.empty() ? std::vector<int>{ p.device } : p.devices)) start_warm(d);
    RowLayout lay = row_layout(VariantSource::NO_FIXED_LAYOUT, p, false);   // --pl with --dosage fails before any file is opened
    GenotypeFiles files(genotype_paths);            // each file first tries the index-driven pass (needs <file>.tbi / .csi)
    bool dose32 = false;                            // a BGEN pass met a block that only 32-bit dosage rows hold
    for (int attempt = 0; attempt < 6; attempt++) {
        // every file is (re)opened and its --samples list resolved before any context: a bad list fails without a device
        if (!files.open(p, unopened)) return false;
        // PLINK filesets, BGEN files: rows in a layout of their own, read by offset (no index pass); VCF/BCF rows keep
        // the layout the last LayoutOverflow grew them to
        if (files.kind != VariantSource::NO_FIXED_LAYOUT) lay = row_layout(files.kind, p, dose32);
        files.set_modes(lay.ds, lay.pl);
        try {
            run_pass(scores, files, cov, p, lay, outs);
            return true;
        } catch (const CannotOpen &e) {
            if (unopened) *unopened = e.path;
            return false;
        } catch (const LayoutOverflow &o) {         // rare: wider integers or higher ploidy -- rerun every file with that layout
            lay.width = o.width; lay.ploidy = o.ploidy;
        } catch (const NeedsDose32 &e) {            // BGEN at another bit depth or with haploid samples: rerun with 32-bit rows
            dose32 = true;
            if (getenv("NIMPRESS_TIMING")) fprintf(stderr, "[nimpress timing] restart with 32-bit dosage rows: %s\n", e.what());
        } catch (const SlabOverflow &) {            // too many rows for one resident slab: one score file at a time
            files.src.clear();
            outs.assign(scores.size(), ScoreResult());
            for (size_t k = 0; k < scores.size(); k++) {
                std::vector<ScoreResult> one;
                if (!compute_polygenic_scores_files({ scores[k] }, genotype_paths, cov, p, one, unopened)) return false;
                outs[k] = std::move(one[0]);
            }
            return true;
        }
    }
    throw std::runtime_error("GT layout kept growing between passes");
}

}  // namespace nph
