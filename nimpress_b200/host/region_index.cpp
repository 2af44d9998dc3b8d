#include "region_index.hpp"

#include <sys/stat.h>

#include <algorithm>
#include <cstring>

#include "variant_source.hpp"

namespace nph {

namespace {
struct Cur {
    const uint8_t *p, *e;
    bool ok = true;
    template <typename T> T get() {
        T v{};
        if ((size_t)(e - p) < sizeof(T)) { ok = false; p = e; return v; }
        memcpy(&v, p, sizeof(T)); p += sizeof(T);
        return v;
    }
};
}  // namespace

bool RegionIndex::present(const std::string &data_path) {
    struct stat si, sd;
    if (stat(data_path.c_str(), &sd) != 0) return false;
    for (const char *ext : { ".tbi", ".csi" })
        if (stat((data_path + ext).c_str(), &si) == 0 && si.st_mtime >= sd.st_mtime) return true;
    return false;
}

std::unique_ptr<RegionIndex> RegionIndex::load(const std::string &data_path) {
    for (int k = 0; k < 2; k++) {
        const std::string path = data_path + (k == 0 ? ".tbi" : ".csi");
        struct stat si, sd;                                         // an index older than its data file is not trusted (htslib warns; here: stream)
        if (stat(path.c_str(), &si) != 0 || stat(data_path.c_str(), &sd) != 0 || si.st_mtime < sd.st_mtime) continue;
        InflateStream s;
        if (!s.open(path)) continue;
        std::vector<uint8_t> d;
        try {
            uint8_t buf[1 << 16];
            for (size_t got; (got = s.read(buf, sizeof buf)) > 0;) d.insert(d.end(), buf, buf + got);
        } catch (const InputError &) { continue; }
        auto idx = std::unique_ptr<RegionIndex>(new RegionIndex());
        if (idx->parse(d, k == 1)) return idx;
    }
    return nullptr;
}

// tabix: "TBI\1" n_ref format col_seq col_beg col_end meta skip l_nm names | per ref: n_bin {bin n_chunk {beg end}} n_intv {ioff}
// CSI:   "CSI\1" min_shift depth l_aux aux n_ref | per ref: n_bin {bin loffset n_chunk {beg end}}     (aux of a tabix-made CSI = the tabix header fields)
bool RegionIndex::parse(const std::vector<uint8_t> &d, bool csi) {
    Cur c{ d.data(), d.data() + d.size() };
    csi_ = csi;
    uint8_t magic[4];
    for (auto &m : magic) m = c.get<uint8_t>();
    if (!c.ok || memcmp(magic, csi ? "CSI\1" : "TBI\1", 4) != 0) return false;
    auto read_names = [&](Cur &q, int32_t l_nm) {
        if (l_nm < 0 || (size_t)(q.e - q.p) < (size_t)l_nm) { q.ok = false; return; }
        const char *s = (const char *)q.p, *e = s + l_nm;
        while (s < e) { size_t l = strnlen(s, e - s); names_.emplace_back(s, l); s += l + 1; }
        q.p += l_nm;
    };
    int32_t n_ref = 0;
    if (!csi) {
        n_ref = c.get<int32_t>();
        for (int i = 0; i < 6; i++) c.get<int32_t>();               // format, col_seq, col_beg, col_end, meta, skip
        read_names(c, c.get<int32_t>());
    } else {
        min_shift_ = c.get<int32_t>(); depth_ = c.get<int32_t>();
        const int32_t l_aux = c.get<int32_t>();
        if (l_aux < 0 || (size_t)(c.e - c.p) < (size_t)l_aux || min_shift_ < 1 || min_shift_ > 30 || depth_ < 1 || depth_ > 10) return false;
        if (l_aux >= 28) {                                          // tabix meta: 6 x int32, l_nm, names
            Cur a{ c.p, c.p + l_aux };
            for (int i = 0; i < 6; i++) a.get<int32_t>();
            read_names(a, a.get<int32_t>());
        }
        c.p += l_aux;
        n_ref = c.get<int32_t>();
    }
    if (!c.ok || n_ref < 0 || n_ref > (1 << 24)) return false;
    refs_.resize(n_ref);
    for (int r = 0; r < n_ref; r++) {
        const int32_t n_bin = c.get<int32_t>();
        if (!c.ok || n_bin < 0) return false;
        for (int b = 0; b < n_bin; b++) {
            const uint32_t bin = c.get<uint32_t>();
            Bin B;
            if (csi) B.loff = c.get<uint64_t>();
            const int32_t n_chunk = c.get<int32_t>();
            if (!c.ok || n_chunk < 0 || (size_t)(c.e - c.p) < (size_t)n_chunk * 16) return false;
            B.chunks.resize(n_chunk);
            for (auto &ch : B.chunks) { ch.first = c.get<uint64_t>(); ch.second = c.get<uint64_t>(); }
            refs_[r].bins.emplace(bin, std::move(B));
        }
        if (!csi) {
            const int32_t n_intv = c.get<int32_t>();
            if (!c.ok || n_intv < 0 || (size_t)(c.e - c.p) < (size_t)n_intv * 8) return false;
            refs_[r].ioff.resize(n_intv);
            for (auto &o : refs_[r].ioff) o = c.get<uint64_t>();
        }
    }
    return c.ok;
}

uint64_t RegionIndex::query_start(int ref, int64_t beg0, int64_t end0) const {
    if (ref < 0 || ref >= (int)refs_.size() || end0 <= beg0) return NONE;
    if (beg0 < 0) beg0 = 0;
    const Ref &R = refs_[ref];
    if (!csi_) {
        // linear index: smallest offset of the records overlapping each 16 kb window; empty windows are 0
        // (or back-filled by the writer): fall back to the nearest earlier window, else the contig's start
        if (R.ioff.empty()) return NONE;
        int64_t w = beg0 >> 14;
        if (w >= (int64_t)R.ioff.size()) return NONE;               // beyond the last record's end
        while (w > 0 && R.ioff[w] == 0) w--;
        if (R.ioff[w] != 0) return R.ioff[w];
        uint64_t first = NONE;                                      // nothing before either: the first chunk of the contig
        const uint32_t meta_bin = ((1u << (3 * (depth_ + 1))) - 1u) / 7u + 1u;   // 37450 for depth 5: its "chunks" are record counts, not offsets
        for (const auto &kv : R.bins) {
            if (kv.first == meta_bin) continue;
            for (const auto &ch : kv.second.chunks) first = std::min(first, ch.first);
        }
        return first;
    }
    // CSI (htslib hts_itr_query): the lower bound comes from the loffset of the deepest bin containing beg
    // (or, when absent, its previous sibling / parent); candidates are the chunks of every overlapping bin
    auto first_of = [](int l) { return ((1u << (3 * l)) - 1u) / 7u; };
    const int64_t maxpos = (int64_t)1 << (min_shift_ + 3 * depth_);
    if (beg0 >= maxpos) return NONE;
    end0 = std::min(end0, maxpos);
    uint64_t min_off = 0;
    {
        uint32_t bin = first_of(depth_) + (uint32_t)(beg0 >> min_shift_);
        for (;;) {
            auto it = R.bins.find(bin);
            if (it != R.bins.end()) { min_off = it->second.loff; break; }
            if (bin == 0) break;
            const uint32_t parent = (bin - 1) >> 3, first = (parent << 3) + 1;
            bin = bin > first ? bin - 1 : parent;
        }
    }
    uint64_t best = NONE;
    for (int l = 0; l <= depth_; l++) {
        const int s = min_shift_ + 3 * (depth_ - l);
        const uint32_t t = first_of(l);
        for (uint32_t b = t + (uint32_t)(beg0 >> s); b <= t + (uint32_t)((end0 - 1) >> s); b++) {
            auto it = R.bins.find(b);
            if (it == R.bins.end()) continue;
            for (const auto &ch : it->second.chunks) if (ch.second > min_off) best = std::min(best, std::max(ch.first, min_off));
        }
    }
    return best;
}

}  // namespace nph
