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
    for (auto &kv : index_) { std::sort(kv.second.by_pos.begin(), kv.second.by_pos.end()); n_lookup_ += (int64_t)kv.second.by_pos.size(); }
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

// WARN lines of one score file, in the reference's order (:326, :527-530, :538-541, :554-557, :567-570, :575-579)
// real_tally: dosage rows (FORMAT/DS, BGEN), whose effect-allele tally is not an integer allele count
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

// One pass over the genotype file with a fixed GT layout, for one score file or several at once
// (BASELINE config 4: every score file sees the same record stream, a record any of them matches
// is uploaded once, and the resident slab is then scored for each file).  Throws LayoutOverflow
// when a matched record needs a wider layout (the caller restarts the pass with it) and
// SlabOverflow when several files are given and their rows do not fit device memory.
// The genotype files are read one after the other as one record stream (DESIGN.md 4.12).  files.keep: the samples each
// file scores, empty for all.  The reader's rows carry a file's own samples, at the front of staging rows sized for the
// widest file (n_row); the devices compact them to the n kept ones (npc_create_subset, npc_set_keep at each file), which
// is all that the contexts, scores and WARN lines see.
void run_pass(const std::vector<const ScoreFile *> &scores, GenotypeFiles &files, const GenomeIntervals &cov, const ScoreParams &p,
              int gt_width, int ploidy, std::vector<ScoreResult> &outs) {
    const int S = (int)scores.size();
    const int64_t n_row = files.n_row, n = (int64_t)files.names.size();
    const std::vector<std::string> &names = files.names;
    const bool subset = !files.keep.empty();
    size_t cur = 0;                                   // the file being read
    // the keep list of the file being read (or, after the stream, of the last one): a context opened lazily takes it; one
    // opened after the stream receives no rows, so any file's list serves it
    const int64_t *keep_now = subset ? files.keep[0].data() : nullptr;
    struct PerScore {
        std::unique_ptr<Matcher> M;
        std::vector<int64_t> slab_row;              // per entry: row of its device's resident slab
        std::vector<uint8_t> done;
        std::vector<npc_row> rows;
    };
    std::vector<PerScore> ps(S);
    outs.assign(S, ScoreResult());

    PhaseTimer timer;
    int64_t n_lookup = 0;
    {   // entries with the same (contig, pos, ref, ea) settle on the same record: count keys once
        std::unordered_map<std::string, int> keys;
        for (int k = 0; k < S; k++) {
            outs[k].samples = names;
            ps[k].M.reset(new Matcher(*scores[k], cov, p));
            const int64_t nE = (int64_t)scores[k]->entries.size();
            ps[k].slab_row.assign(nE, -1); ps[k].done.assign(nE, 0);
            if (S == 1) { n_lookup = ps[k].M->n_lookup(); break; }
            for (int64_t i = 0; i < nE; i++) if (ps[k].M->kind[i] == Matcher::PENDING) {
                const ScoreEntry &e = scores[k]->entries[i];
                keys.emplace(e.contig + "\t" + std::to_string(e.pos) + "\t" + e.refseq + "\t" + e.easeq, 0);
            }
        }
        if (S > 1) n_lookup = (int64_t)keys.size();
    }
    Spans spans;                                      // an index next to a file and few loci: read only where loci are
    if (std::count(files.seekable.begin(), files.seekable.end(), 1))
        for (int k = 0; k < S; k++) ps[k].M->add_spans(spans);
    if (!files.prepare(0, spans)) throw CannotOpen{ files.paths[0] };
    VariantSource *vcf = files.src[0].get();
    timer.mark("coverage + entry index");

    // Devices: one context per GPU.  With several, the score rows are partitioned into contiguous ranges in
    // score-file order (a contig / region partition for a sorted score file): context d scores range d over all
    // samples, a matched record is uploaded to the device(s) whose ranges name it, and the partial sums are
    // combined in range order by npc_reduce.  Several score files at once: every file is cut into D ranges of its own,
    // device d scores range d of every file in one npc_score_resident_multi call (raw partial sums), and the host adds
    // the partials of each file in device order and normalises once.
    std::vector<int> dev_ids = p.devices.empty() ? std::vector<int>{ p.device } : p.devices;
    if (const char *e = getenv("NIMPRESS_SPLIT")) if (*e && dev_ids.size() == 1 && atoi(e) > 1)      // tests: several contexts on one GPU
        dev_ids.assign((size_t)std::min(atoi(e), 16), dev_ids[0]);
    const int D = (int)dev_ids.size();
    // entry i of score file k belongs to device i * D / (entries of k): contiguous ranges of EVERY file in its own order
    auto dev_of = [&](int k, int64_t i) -> int {
        return D == 1 ? 0 : (int)std::min<int64_t>(D - 1, i * D / std::max<int64_t>((int64_t)scores[k]->entries.size(), 1));
    };
    std::vector<int64_t> dev_lookup(D, 0);            // rows of each device's ranges that need a record (an upper bound when files share records)
    if (D == 1) dev_lookup[0] = n_lookup;
    else for (int k = 0; k < S; k++)
        for (int64_t i = 0; i < (int64_t)scores[k]->entries.size(); i++) if (ps[k].M->kind[i] == Matcher::PENDING) dev_lookup[dev_of(k, i)]++;

    // staging slots of ~8 MB: big enough for efficient H2D copies, small enough that pinning three of them per
    // device does not dominate a short run (pinning costs ~1 ms per MB); scoring launches are sized separately
    const int64_t row_bytes = std::max<int64_t>(16, npc_gt_row_bytes(n_row, ploidy, gt_width));
    struct Dev {
        Ctx ctx;
        int32_t slot = -1; uint8_t *stage = nullptr; int64_t stride = 0, staged = 0, slab_base = 0, slab_cap = 0, block_rows = 1;
        std::vector<npc_row> rows; std::vector<int64_t> submitted;   // S == 1: this device's rows, entry index of each
        std::string err;
    };
    std::vector<Dev> devs(D);
    // rows still being converted by the source's workers land in the devices' pinned slots: let them finish before the
    // slots go, whichever way this pass ends
    struct RowsGuard {
        VariantSource *&v;
        ~RowsGuard() { try { if (v) v->wait_rows(); } catch (...) {} }
    } rows_guard{ vcf };
    npc_policy pol = { p.imp_locus, p.imp_missing, p.imp_sample, 0, p.mincs, p.maxmis };
    auto open_dev = [&](int d) {
        Dev &v = devs[d];
        try {
            const int64_t want = std::max<int64_t>(dev_lookup[d], 1);
            v.block_rows = std::max<int64_t>(1, std::min<int64_t>(std::min<int64_t>(4096, (8ll << 20) / row_bytes + 1), want));
            const int64_t launch_rows = std::max<int64_t>(v.block_rows, 32768);
            if (!subset) v.ctx.ck(npc_create2(&v.ctx.h, dev_ids[d], n, ploidy, gt_width, launch_rows, 3, v.block_rows), "npc_create");
            else v.ctx.ck(npc_create_subset(&v.ctx.h, dev_ids[d], n_row, keep_now, n, ploidy, gt_width, launch_rows, 3,
                                            v.block_rows), "npc_create_subset");
            v.ctx.ck(npc_set_policy(v.ctx.h, &pol), "npc_set_policy");
            if (p.use_ds) v.ctx.ck(npc_set_dosage_rows(v.ctx.h, 1), "npc_set_dosage_rows");
            if (p.exact_order) v.ctx.ck(npc_set_exact_order(v.ctx.h, 1), "npc_set_exact_order");
            v.ctx.ck(npc_reset(v.ctx.h), "npc_reset");
            int64_t slab_want = want;
            if (const char *e = getenv("NIMPRESS_SLAB_ROWS")) if (*e) slab_want = std::max<int64_t>(1, std::min<int64_t>(slab_want, atoll(e)));   // tests: force rounds
            v.ctx.ck(npc_resident_reserve(v.ctx.h, slab_want, &v.slab_cap), "npc_resident_reserve");
        } catch (const std::exception &e) { v.err = e.what(); }
    };
    // A device is opened when its first row arrives (or at the end, for its constant rows): contexts come up one after
    // the other inside the driver (~1 s each), and a sorted file reaches the later ranges later -- the first device's
    // rows stream while the others' contexts are still being created.
    std::vector<uint8_t> opened(D, 0);
    double waited_ms = 0.0;
    auto ensure_open = [&](int d) {
        if (opened[d]) return;
        const auto t0 = std::chrono::steady_clock::now();
        wait_warm(dev_ids[d]);
        open_dev(d);
        waited_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        if (!devs[d].err.empty()) throw std::runtime_error(devs[d].err);
        opened[d] = 1;
    };
    ensure_open(0);
    timer.mark("first GPU context + buffers");

    auto flush_stage = [&](Dev &v) {
        if (v.slot < 0) return;
        vcf->wait_rows();
        v.ctx.ck(npc_stage_upload(v.ctx.h, v.slot, v.staged, v.slab_base), "npc_stage_upload");
        v.slab_base += v.staged; v.staged = 0; v.slot = -1;
    };
    // the rows of score k that a round takes on device d, in score-file order
    auto collect_rows = [&](int k, int d, bool final_round, std::vector<npc_row> &rows, std::vector<int64_t> &submitted) {
        PerScore &q = ps[k];
        const std::vector<ScoreEntry> &E = scores[k]->entries;
        rows.clear();
        for (int64_t i = 0; i < (int64_t)E.size(); i++) {
            if (q.done[i] || dev_of(k, i) != d) continue;
            const int32_t kind = q.M->kind[i];
            if (!final_round && !(kind == NPC_KIND_GT && q.slab_row[i] >= 0)) continue;
            npc_row r;
            r.gt_row = kind == NPC_KIND_GT ? (int32_t)q.slab_row[i] : -1;
            r.eaidx = q.M->eaidx[i]; r.beta = E[i].beta; r.eaf = E[i].eaf;
            r.ref_is_ea = E[i].ref_is_ea() ? 1 : 0; r.kind = kind;
            rows.push_back(r);
            submitted.push_back(i);
            q.done[i] = 1;
        }
    };
    // A round scores rows over a device's resident slab in score-file order.  The normal case is ONE
    // final round per device holding every row of its range: exactly the reference's loop order
    // (:634-641).  Only when the matched genotype rows exceed device memory are there earlier rounds;
    // those take the rows whose genotypes sit in the slab, and the summation order then differs from
    // the reference's by a reordering of terms (scores agree to ~1 ulp of the partial sums, not bit for bit).
    std::vector<int64_t> rounds(D, 0);
    auto score_round = [&](int d, bool final_round) {     // one score file only
        Dev &v = devs[d];
        flush_stage(v);
        collect_rows(0, d, final_round, v.rows, v.submitted);
        if (!v.rows.empty()) v.ctx.ck(npc_score_resident(v.ctx.h, v.rows.data(), (int64_t)v.rows.size()), "npc_score_resident");
        rounds[d]++;
    };

    // ---- one streaming pass over the genotype files (findVariant :353-364, eaidx :375-379) ---
    VariantRecord rec;
    int64_t records_read = 0, records_matched = 0, seeks = 0;
    std::vector<int64_t> rec_row(D);                   // slab row this record got on each device, -1 = not uploaded there
    for (cur = 0; cur < files.src.size(); cur++) {
        if (cur > 0) {
            if (!files.prepare(cur, spans)) throw CannotOpen{ files.paths[cur] };
            vcf = files.src[cur].get();
            if (subset) {                                 // staged rows of the previous file are compacted with its list
                keep_now = files.keep[cur].data();
                for (int d = 0; d < D; d++) if (opened[d]) {
                    flush_stage(devs[d]);
                    devs[d].ctx.ck(npc_set_keep(devs[d].ctx.h, keep_now, n), "npc_set_keep");
                }
            }
        }
        const size_t file_row_bytes = (size_t)npc_gt_row_bytes(vcf->n_samples(), ploidy, gt_width);   // the front of a staging row
        while (vcf->next(rec)) {
            records_read++;
            bool any = false, need_gt = false;
            uint32_t need_dev = 0;
            for (int k = 0; k < S; k++) {
                const std::vector<int64_t> &hits = ps[k].M->match(rec);
                for (int64_t i : hits) {
                    any = true;
                    if (ps[k].M->kind[i] == NPC_KIND_GT) { need_gt = true; need_dev |= 1u << dev_of(k, i); }
                }
            }
            if (!any) continue;
            records_matched++;
            if (!need_gt) continue;                                     // FILTER-failed: never decoded (:553-558)
            const uint8_t *first = nullptr;
            for (int d = 0; d < D; d++) {
                rec_row[d] = -1;
                if (!((need_dev >> d) & 1u)) continue;
                ensure_open(d);
                Dev &v = devs[d];
                if (v.slab_base + v.staged >= v.slab_cap) {             // slab full: score its rows, start over
                    if (S > 1) throw SlabOverflow();
                    score_round(d, false);
                    v.slab_base = 0;
                }
                if (v.slot < 0) {
                    void *ptr;
                    v.ctx.ck(npc_stage_acquire(v.ctx.h, &v.slot, &ptr, &v.stride), "npc_stage_acquire");
                    v.stage = (uint8_t *)ptr; v.staged = 0;
                }
                uint8_t *dst = v.stage + v.staged * v.stride;
                if (first) {                                            // a record named by two ranges: same bytes
                    vcf->wait_rows();
                    memcpy(dst, first, file_row_bytes);
                }
                else {
                    if (p.use_pl && rec.alts.size() != 1)
                        throw InputError("record " + *rec.contig + ":" + std::to_string(rec.pos) + ": FORMAT/PL rows take biallelic records only (" +
                                         std::to_string(rec.alts.size()) + " ALT alleles; split them with bcftools norm -m-)");
                    // BCF with the context's layout: the GT payload goes from the inflated blocks straight into the pinned row
                    const bool direct = vcf->load_gt_into(rec, dst, gt_width, ploidy);
                    if (!rec.has_gt || !rec.gt)
                        throw InputError("record " + *rec.contig + ":" + std::to_string(rec.pos) +
                                         (p.use_pl ? " has no PL field" : p.use_ds ? " has no DS field" : " has no GT field"));
                    if (p.use_ds && (rec.ploidy != 1 || rec.gt_width != 4))
                        throw InputError("record " + *rec.contig + ":" + std::to_string(rec.pos) + ": FORMAT/DS with several values per sample is not supported");
                    if (!direct) {
                        if (rec.ploidy > ploidy || rec.gt_width > gt_width)
                            throw LayoutOverflow{ std::max(rec.gt_width, gt_width), std::max(rec.ploidy, ploidy) };
                        if (rec.gt_width == gt_width && rec.ploidy == ploidy) memcpy(dst, rec.gt, file_row_bytes);
                        else convert_gt(rec, vcf->n_samples(), gt_width, ploidy, dst);
                    }
                    first = dst;
                }
                rec_row[d] = v.slab_base + v.staged;
                v.staged++;
            }
            for (int k = 0; k < S; k++) for (int64_t i : ps[k].M->match_last())
                if (ps[k].M->kind[i] == NPC_KIND_GT) {
                    if (p.use_ds && ps[k].M->eaidx[i] > 1)
                        throw InputError("record " + *rec.contig + ":" + std::to_string(rec.pos) + ": FORMAT/DS rows take the REF or the first ALT as effect allele");
                    ps[k].slab_row[i] = rec_row[dev_of(k, i)];
                }
            for (int d = 0; d < D; d++) if (devs[d].slot >= 0 && devs[d].staged == devs[d].block_rows) flush_stage(devs[d]);
        }
        vcf->wait_rows();                                 // BGEN workers may still be writing this file's rows into pinned slots
        seeks += vcf->seeks();
        if (cur + 1 < files.src.size()) { files.src[cur].reset(); vcf = nullptr; }
    }
    for (int k = 0; k < S; k++) {
        ps[k].M->finish();
        outs[k].records_read = records_read; outs[k].records_matched = records_matched; outs[k].index_seeks = seeks;
    }
    timer.mark("stream + match + upload");
    if (timer.on) fprintf(stderr, "[nimpress timing] records read %lld, matched %lld, index seeks %lld%s\n", (long long)records_read,
                          (long long)records_matched, (long long)seeks, seeks ? " (.tbi / .csi used)" : "");

    // ---- score the slab(s), collect results ----------------------------------------------------
    std::vector<std::vector<npc_locus>> logs(S);
    std::vector<std::vector<int64_t>> order(S);          // entry index of every log record
    for (int d = 0; d < D; d++) ensure_open(d);
    if (timer.on && D > 1) fprintf(stderr, "[nimpress timing] waited for GPU contexts + buffers, all devices %8.1f ms\n", waited_ms);
    if (S == 1) {
        for (int d = 0; d < D; d++) score_round(d, true);
        outs[0].scores.assign(n, 0.0);
        outs[0].rounds = *std::max_element(rounds.begin(), rounds.end());
        outs[0].devices = D;
        if (D == 1) {
            Dev &v = devs[0];
            logs[0].resize(v.submitted.size());
            int64_t nlog = 0;
            v.ctx.ck(npc_finish(v.ctx.h, scores[0]->offset, outs[0].scores.data(), &outs[0].nloci, logs[0].data(), (int64_t)logs[0].size(), &nlog), "npc_finish");
            if (nlog != (int64_t)v.submitted.size()) throw std::runtime_error("locus log length mismatch");
            order[0] = v.submitted;
        } else {
            std::vector<npc_ctx *> hs(D);
            for (int d = 0; d < D; d++) hs[d] = devs[d].ctx.h;
            const double off = scores[0]->offset;
            devs[0].ctx.ck(npc_reduce(hs.data(), D, &off, outs[0].scores.data(), &outs[0].nloci), "npc_reduce");
            std::vector<double> scratch((size_t)std::max<int64_t>(n, 1));
            for (int d = 0; d < D; d++) {
                Dev &v = devs[d];
                std::vector<npc_locus> lg(v.submitted.size());
                int64_t nlog = 0, nl = 0;
                v.ctx.ck(npc_partial(v.ctx.h, scratch.data(), &nl, lg.data(), (int64_t)lg.size(), &nlog), "npc_partial");
                if (nlog != (int64_t)v.submitted.size()) throw std::runtime_error("locus log length mismatch");
                logs[0].insert(logs[0].end(), lg.begin(), lg.end());
                order[0].insert(order[0].end(), v.submitted.begin(), v.submitted.end());
            }
        }
    } else {
        std::vector<int64_t> nloci_tot(S, 0);
        std::vector<std::vector<double>> part(S);
        for (int k = 0; k < S; k++) { outs[k].scores.assign(n, 0.0); outs[k].rounds = 1; outs[k].devices = D; if (D > 1) part[k].assign((size_t)n, 0.0); }
        for (int d = 0; d < D; d++) {
            Dev &v = devs[d];
            flush_stage(v);
            std::vector<std::vector<npc_row>> drows(S);
            std::vector<std::vector<npc_locus>> dlog(S);
            std::vector<const npc_row *> rows(S);
            std::vector<int64_t> n_rows(S), nloci(S);
            std::vector<double> offsets(S);
            std::vector<double *> sc(S);
            std::vector<npc_locus *> lg(S);
            for (int k = 0; k < S; k++) {
                collect_rows(k, d, true, drows[k], order[k]);
                rows[k] = drows[k].data(); n_rows[k] = (int64_t)drows[k].size(); offsets[k] = scores[k]->offset;
                sc[k] = D == 1 ? outs[k].scores.data() : part[k].data();
                dlog[k].resize(drows[k].size()); lg[k] = dlog[k].data();
            }
            // one device: normalised scores straight away; several: raw partial sums (offsets = NULL), combined below
            v.ctx.ck(npc_score_resident_multi(v.ctx.h, S, rows.data(), n_rows.data(), D == 1 ? offsets.data() : nullptr, sc.data(), nloci.data(), lg.data()),
                     "npc_score_resident_multi");
            for (int k = 0; k < S; k++) {
                nloci_tot[k] += nloci[k];
                logs[k].insert(logs[k].end(), dlog[k].begin(), dlog[k].end());
                if (D > 1) {
                    double *tot = outs[k].scores.data();
                    const double *pk = part[k].data();
                    if (d == 0) memcpy(tot, pk, (size_t)n * sizeof(double));
                    else for (int64_t i = 0; i < n; i++) tot[i] += pk[i];            // device order = score-file order of the ranges
                }
            }
        }
        for (int k = 0; k < S; k++) {
            outs[k].nloci = nloci_tot[k];
            if (D > 1) npc_normalise(outs[k].scores.data(), n, nloci_tot[k], scores[k]->offset);
        }
    }
    timer.mark("score + finish (GPU)");
    for (int k = 0; k < S; k++) {
        outs[k].loci.assign(scores[k]->entries.size(), npc_locus());
        for (size_t j = 0; j < order[k].size(); j++) outs[k].loci[order[k][j]] = logs[k][j];
        outs[k].warnings = make_warnings(*scores[k], *ps[k].M, outs[k].loci, n, p,
                                         p.use_ds || p.use_pl || gt_width == NPC_GT_DOSE255 || gt_width == NPC_GT_DOSE32);
    }
    timer.mark("WARN lines (binomial tests)");
}

}  // namespace

bool compute_polygenic_scores_files(const std::vector<const ScoreFile *> &scores, const std::vector<std::string> &genotype_paths,
                                    const GenomeIntervals &cov, const ScoreParams &p, std::vector<ScoreResult> &outs, std::string *unopened) {
    for (int d : (p.devices.empty() ? std::vector<int>{ p.device } : p.devices)) start_warm(d);
    int width = 1, ploidy = 2;                      // BCF's usual GT layout: int8, diploid
    if (p.use_ds && p.use_pl) throw InputError("--pl and --dosage: score either FORMAT/PL or FORMAT/DS");
    if (p.use_ds) { width = 4; ploidy = 1; }        // FORMAT/DS: one float per sample
    if (p.use_pl) { width = NPC_GT_PL; ploidy = 2; }   // FORMAT/PL: one packed word per sample
    GenotypeFiles files(genotype_paths);            // each file first tries the index-driven pass (needs <file>.tbi / .csi)
    bool dose32 = false;                            // a BGEN pass met a block that only 32-bit dosage rows hold
    for (int attempt = 0; attempt < 6; attempt++) {
        // every file is (re)opened and its --samples list resolved before any context: a bad list fails without a device
        if (!files.open(p, unopened)) return false;
        // PLINK filesets, BGEN files: rows in a layout of their own, read by offset (no index pass)
        const int fixed = files.kind;
        ScoreParams q = p;
        if (fixed == NPC_GT_BED && p.use_ds) throw InputError("--dosage: a PLINK fileset holds hard calls only, no FORMAT/DS");
        if (fixed == NPC_GT_BED && p.use_pl) throw InputError("--pl: a PLINK fileset holds hard calls only, no FORMAT/PL");
        if (fixed == NPC_GT_DOSE255 && p.use_pl) throw InputError("--pl: a BGEN file holds genotype probabilities, no FORMAT/PL");
        if (fixed != VariantSource::NO_FIXED_LAYOUT) {
            width = dose32 ? NPC_GT_DOSE32 : fixed; ploidy = 2;
            q.use_ds = false;                       // BGEN rows are dosages already: --dosage changes nothing
        }
        files.set_modes(q.use_ds, q.use_pl);
        try {
            run_pass(scores, files, cov, q, width, ploidy, outs);
            return true;
        } catch (const CannotOpen &e) {
            if (unopened) *unopened = e.path;
            return false;
        } catch (const LayoutOverflow &o) {         // rare: wider integers or higher ploidy -- rerun every file with that layout
            width = o.width; ploidy = o.ploidy;
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

bool compute_polygenic_scores_multi(const std::vector<const ScoreFile *> &scores, const std::string &genotype_path,
                                    const GenomeIntervals &cov, const ScoreParams &p, std::vector<ScoreResult> &outs) {
    return compute_polygenic_scores_files(scores, { genotype_path }, cov, p, outs);
}

bool compute_polygenic_scores(const ScoreFile &score, const std::string &genotype_path, const GenomeIntervals &cov,
                              const ScoreParams &p, ScoreResult &out) {
    std::vector<ScoreResult> outs;
    if (!compute_polygenic_scores_multi({ &score }, genotype_path, cov, p, outs)) return false;
    out = std::move(outs[0]);
    return true;
}

}  // namespace nph
