#include "variant_source.hpp"
#include "region_index.hpp"
#include "fast_inflate.hpp"
#include "../../include/nimpress_cuda.h"

#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <algorithm>
#include <atomic>
#include <climits>
#include <condition_variable>
#include <cstring>
#include <deque>
#include <map>
#include <mutex>
#include <thread>
#include <unordered_map>

namespace nph {

// ------------------------------------------------------------------------------------------
// InflateStream
// ------------------------------------------------------------------------------------------

// ------------------------------------------------------------------------------------------
// BgzfPool: a reader thread cuts the file into BGZF blocks (18-byte header, BSIZE in the `BC`
// extra field), worker threads inflate them (raw deflate, independent streams), the consumer takes
// them in file order from a ring of slots.
// ------------------------------------------------------------------------------------------

class BgzfPool {
public:
    BgzfPool(FILE *fp, int n_workers) : fp_(fp), ring_((size_t)n_workers * 4) {
        reader_ = std::thread([this] { read_loop(); });
        for (int i = 0; i < n_workers; i++) workers_.emplace_back([this] { work_loop(); });
    }
    ~BgzfPool() {
        { std::lock_guard<std::mutex> g(m_); stop_ = true; }
        cv_job_.notify_all(); cv_free_.notify_all(); cv_done_.notify_all();
        reader_.join();
        for (auto &t : workers_) t.join();
    }
    // next inflated block, in order; false at end of file.  The returned buffer stays valid until the next call.
    bool next(const uint8_t *&data, size_t &len) {
        std::unique_lock<std::mutex> g(m_);
        if (held_) { ring_[(rd_ - 1) % ring_.size()].state = FREE; held_ = false; cv_free_.notify_all(); }
        for (;;) {
            Slot &s = ring_[rd_ % ring_.size()];
            if (rd_ < wr_ && s.state == DONE) {
                if (!s.error.empty()) throw InputError(s.error);
                data = s.out.data(); len = s.out_len; rd_++; held_ = true;
                return true;
            }
            if (eof_ && rd_ == wr_) { if (!error_.empty()) throw InputError(error_); return false; }
            cv_done_.wait(g);
        }
    }
private:
    enum { FREE = 0, QUEUED = 1, BUSY = 2, DONE = 3 };
    struct Slot { std::vector<uint8_t> in, out; size_t in_len = 0, out_len = 0; int state = FREE; std::string error; };
    void read_loop() {
        for (;;) {
            size_t idx;
            {
                std::unique_lock<std::mutex> g(m_);
                cv_free_.wait(g, [this] { return stop_ || ring_[wr_ % ring_.size()].state == FREE; });
                if (stop_) return;
                idx = wr_ % ring_.size();
            }
            Slot &s = ring_[idx];
            uint8_t hdr[18];
            size_t got = fread(hdr, 1, 18, fp_);
            std::string err;
            size_t bsize = 0;
            if (got == 0) { finish(""); return; }
            if (got != 18 || hdr[0] != 0x1f || hdr[1] != 0x8b || !(hdr[3] & 4) || hdr[12] != 'B' || hdr[13] != 'C')
                err = "BGZF: malformed block header";
            else {
                bsize = (size_t)(hdr[16] | (hdr[17] << 8)) + 1;
                const size_t xlen = (size_t)(hdr[10] | (hdr[11] << 8));
                if (xlen < 6 || bsize < 12 + xlen + 8) err = "BGZF: bad block size";      // xlen < 6: no room for the BC subfield we just read
                else {
                    const size_t rest = bsize - 18;                 // remaining extra fields + deflate data + CRC32 + ISIZE
                    if (s.in.size() < rest + 16) s.in.resize(std::max<size_t>(rest + 16, (1 << 16) + 64));   // + the decoder's read-ahead
                    if (fread(s.in.data(), 1, rest, fp_) != rest) err = "BGZF: truncated block";
                    else {
                        const size_t skip = xlen - 6;               // extra subfields beyond BC
                        s.in_len = rest; s.out_len = skip;          // out_len doubles as the payload offset for the worker
                    }
                }
            }
            if (!err.empty()) { finish(err); return; }
            {
                std::lock_guard<std::mutex> g(m_);
                s.state = QUEUED; s.error.clear(); wr_++;
            }
            cv_job_.notify_one();
        }
    }
    void finish(const std::string &err) {
        std::lock_guard<std::mutex> g(m_);
        eof_ = true; error_ = err;
        cv_done_.notify_all(); cv_job_.notify_all();
    }
    void work_loop() {
        z_stream zs;
        memset(&zs, 0, sizeof zs);
        inflateInit2(&zs, -15);
        std::unique_ptr<FastInflateTables> tabs(new FastInflateTables);
        const char *zo = getenv("NIMPRESS_ZLIB_ONLY");
        const bool zlib_only = zo && *zo && *zo != '0';
        for (;;) {
            Slot *s = nullptr;
            {
                std::unique_lock<std::mutex> g(m_);
                for (;;) {
                    if (stop_) { inflateEnd(&zs); return; }
                    for (size_t k = job_; k < wr_; k++)
                        if (ring_[k % ring_.size()].state == QUEUED) { s = &ring_[k % ring_.size()]; s->state = BUSY; if (k == job_) job_++; break; }
                    if (s) break;
                    while (job_ < wr_ && ring_[job_ % ring_.size()].state != QUEUED) job_++;
                    if (job_ < wr_) continue;
                    if (eof_) { inflateEnd(&zs); return; }
                    cv_job_.wait(g);
                }
            }
            const size_t off = s->out_len, tail = 8;
            uint32_t isize, want_crc;
            memcpy(&want_crc, s->in.data() + s->in_len - 8, 4);
            memcpy(&isize, s->in.data() + s->in_len - 4, 4);
            if (s->out.size() < (size_t)isize + 16) s->out.resize(std::max<size_t>((size_t)isize + 16, (1 << 16) + 16));
            std::string err;
            // this engine's own decoder first (fast_inflate.hpp); zlib when it declines or the CRC disagrees
            bool ok = !zlib_only && isize && s->in_len >= off + tail &&
                      fast_inflate(s->in.data() + off, s->in_len - off - tail, s->out.data(), isize, *tabs) &&
                      (uint32_t)crc32(0L, s->out.data(), isize) == want_crc;
            if (!ok && isize) {
                inflateReset(&zs);
                zs.next_in = s->in.data() + off; zs.avail_in = (uInt)(s->in_len - off - tail);
                zs.next_out = s->out.data(); zs.avail_out = (uInt)s->out.size();
                const int rc = inflate(&zs, Z_FINISH);
                if (rc != Z_STREAM_END || zs.total_out != isize) err = "BGZF: corrupt deflate data";
                else if ((uint32_t)crc32(0L, s->out.data(), isize) != want_crc) err = "BGZF: CRC32 mismatch";
            }
            {
                std::lock_guard<std::mutex> g(m_);
                s->out_len = isize; s->error = err; s->state = DONE;
            }
            cv_done_.notify_all();
        }
    }
    FILE *fp_;
    std::vector<Slot> ring_;
    std::mutex m_;
    std::condition_variable cv_job_, cv_free_, cv_done_;
    size_t wr_ = 0, rd_ = 0, job_ = 0;
    bool eof_ = false, stop_ = false, held_ = false;
    std::string error_;
    std::thread reader_;
    std::vector<std::thread> workers_;
};

InflateStream::InflateStream() = default;

InflateStream::~InflateStream() {
    pool_.reset();
    if (zinit_) inflateEnd(&zs_);
    if (fp_) fclose(fp_);
}

bool InflateStream::open(const std::string &path, bool seekable) {
    fp_ = fopen(path.c_str(), "rb");
    if (!fp_) return false;
    fseek(fp_, 0, SEEK_END);
    file_size_ = (int64_t)ftell(fp_);
    fseek(fp_, 0, SEEK_SET);
    unsigned char magic[18] = { 0 };
    size_t got = fread(magic, 1, 18, fp_);
    fseek(fp_, 0, SEEK_SET);
    compressed_ = got >= 2 && magic[0] == 0x1f && magic[1] == 0x8b;
    const bool bgzf = got == 18 && compressed_ && (magic[3] & 4) && magic[12] == 'B' && magic[13] == 'C';
    bgzf_ = bgzf;
    // all cores but one (the reader's own thread walks the records and copies the GT payloads), at most 32
    const unsigned hc = std::max(1u, std::thread::hardware_concurrency());
    int want = (int)std::min<unsigned>(hc > 2 ? hc - 1 : hc, 32u);
    if (const char *e = getenv("NIMPRESS_THREADS")) if (*e) want = std::max(1, atoi(e));
    block_mode_ = bgzf && (seekable || want == 1);     // one thread: block by block with this engine's decoder
    if (bgzf && want > 1 && !block_mode_) {
        threads_ = want;
        pool_ = std::make_unique<BgzfPool>(fp_, want);
        return true;
    }
    in_.resize(block_mode_ ? 128 << 10 : 1 << 20);    // seekable: a jump costs one read of two blocks, not a megabyte
    out_.resize(4 << 20);
    if (compressed_) {
        memset(&zs_, 0, sizeof zs_);
        if (inflateInit2(&zs_, 15 + 16) != Z_OK) return false;
        zinit_ = true;
    }
    return true;
}

bool InflateStream::fill() {
    out_pos_ = out_len_ = 0;
    if (eof_) return false;
    if (pool_) {                                      // blocks arrive inflated, in order; empty blocks (EOF marker) are skipped
        const uint8_t *d; size_t l;
        do {
            if (!pool_->next(d, l)) { eof_ = true; return false; }
        } while (l == 0);
        pool_data_ = d; out_len_ = l;
        return true;
    }
    if (!compressed_) {
        out_len_ = fread(out_.data(), 1, out_.size(), fp_);
        if (out_len_ == 0) eof_ = true;
        return out_len_ > 0;
    }
    if (block_mode_) {                                // exactly one BGZF block per fill: the position stays a virtual offset
        for (;;) {
            block_coff_ = in_file_off_;
            uint8_t hdr[18];
            const size_t got = fread(hdr, 1, 18, fp_);
            if (got == 0) { eof_ = true; return false; }
            if (got != 18 || hdr[0] != 0x1f || hdr[1] != 0x8b || !(hdr[3] & 4) || hdr[12] != 'B' || hdr[13] != 'C')
                throw InputError("BGZF: malformed block header");
            const size_t bsize = (size_t)(hdr[16] | (hdr[17] << 8)) + 1, xlen = (size_t)(hdr[10] | (hdr[11] << 8));
            if (bsize < 12 + xlen + 8 || xlen < 6) throw InputError("BGZF: bad block size");
            const size_t rest = bsize - 18, off = xlen - 6;         // remaining extra fields, deflate data, CRC32, ISIZE
            if (in_.size() < rest + 16) in_.resize(rest + 16);
            if (fread(in_.data(), 1, rest, fp_) != rest) throw InputError("BGZF: truncated block");
            in_file_off_ += bsize;
            uint32_t want_crc, isize;
            memcpy(&want_crc, in_.data() + rest - 8, 4);
            memcpy(&isize, in_.data() + rest - 4, 4);
            if (isize == 0) continue;                               // empty blocks (the EOF marker) are skipped
            if (out_.size() < (size_t)isize + 16) out_.resize((size_t)isize + 16);
            if (!tabs_) tabs_.reset(new FastInflateTables);
            const char *zo = getenv("NIMPRESS_ZLIB_ONLY");
            bool ok = !(zo && *zo && *zo != '0') && rest >= off + 8 &&
                      fast_inflate(in_.data() + off, rest - off - 8, out_.data(), isize, *tabs_) &&
                      (uint32_t)crc32(0L, out_.data(), isize) == want_crc;
            if (!ok) {                                              // zlib, raw deflate
                if (inflateReset2(&zs_, -15) != Z_OK) throw InputError("zlib: inflateReset failed");
                zs_.next_in = in_.data() + off; zs_.avail_in = (uInt)(rest - off - 8);
                zs_.next_out = out_.data(); zs_.avail_out = (uInt)out_.size();
                const int rc = inflate(&zs_, Z_FINISH);
                if (rc != Z_STREAM_END || zs_.total_out != isize) throw InputError("BGZF: corrupt deflate data");
                if ((uint32_t)crc32(0L, out_.data(), isize) != want_crc) throw InputError("BGZF: CRC32 mismatch");
            }
            out_len_ = isize;
            return true;
        }
    }
    zs_.next_out = out_.data();
    zs_.avail_out = (uInt)out_.size();
    while (zs_.avail_out == out_.size()) {            // until something was produced
        if (zs_.avail_in == 0) {
            zs_.next_in = in_.data();
            zs_.avail_in = (uInt)fread(in_.data(), 1, in_.size(), fp_);
            if (zs_.avail_in == 0) { eof_ = true; break; }
        }
        int rc = inflate(&zs_, Z_NO_FLUSH);
        if (rc == Z_STREAM_END) {                     // next BGZF block / gzip member
            if (inflateReset(&zs_) != Z_OK) throw InputError("zlib: inflateReset failed");
        } else if (rc != Z_OK && rc != Z_BUF_ERROR) {
            throw InputError(std::string("zlib: corrupt compressed stream: ") + (zs_.msg ? zs_.msg : "?"));
        }
    }
    out_len_ = out_.size() - zs_.avail_out;
    return out_len_ > 0;
}

void InflateStream::seek_virtual(uint64_t voff) {
    if (!block_mode_) throw InputError("seek on a stream that was not opened seekable");
    const uint64_t coff = voff >> 16;
    if (fseek(fp_, (long)coff, SEEK_SET) != 0) throw InputError("index points outside the file");
    in_file_off_ = coff;
    eof_ = false;
    out_pos_ = out_len_ = 0;
    if (!fill()) return;                              // at or past the end: the next read reports end of stream
    out_pos_ = std::min<size_t>((size_t)(voff & 0xFFFF), out_len_);
}

size_t InflateStream::read(void *dst, size_t n) {
    size_t done = 0;
    while (done < n) {
        if (out_pos_ == out_len_ && !fill()) break;
        size_t k = std::min(n - done, out_len_ - out_pos_);
        memcpy((uint8_t *)dst + done, cur() + out_pos_, k);
        out_pos_ += k;
        done += k;
    }
    return done;
}

bool InflateStream::read_exact(void *dst, size_t n) { return read(dst, n) == n; }

bool InflateStream::skip(size_t n) {                  // advance without copying
    while (n) {
        if (out_pos_ == out_len_ && !fill()) return false;
        const size_t k = std::min(n, out_len_ - out_pos_);
        out_pos_ += k; n -= k;
    }
    return true;
}

bool InflateStream::peek(void *dst, size_t n) {
    if (out_pos_ == out_len_ && !fill()) return false;
    if (out_len_ - out_pos_ < n) return false;        // only used at the very start of the stream
    memcpy(dst, cur() + out_pos_, n);
    return true;
}

bool InflateStream::getline(std::string &line) {
    line.clear();
    bool any = false;
    for (;;) {
        if (out_pos_ == out_len_ && !fill()) break;
        any = true;
        const uint8_t *b = cur() + out_pos_;
        const uint8_t *nl = (const uint8_t *)memchr(b, '\n', out_len_ - out_pos_);
        if (nl) {
            line.append((const char *)b, nl - b);
            out_pos_ += (nl - b) + 1;
            break;
        }
        line.append((const char *)b, out_len_ - out_pos_);
        out_pos_ = out_len_;
    }
    if (!any) return false;
    if (!line.empty() && line.back() == '\r') line.pop_back();
    return true;
}

// ------------------------------------------------------------------------------------------
// shared: encode GT values into the narrowest BCF integer width, pad with vector_end
// ------------------------------------------------------------------------------------------

static void pack_gt(const std::vector<int32_t> &vals, const std::vector<int> &counts, int64_t n, int ploidy,
                    std::vector<uint8_t> &out, int &width) {
    int32_t mx = 0;
    for (int32_t v : vals) mx = std::max(mx, v);
    width = mx <= INT8_MAX ? 1 : mx <= INT16_MAX ? 2 : 4;
    out.assign((size_t)n * ploidy * width, 0);
    size_t src = 0;
    for (int64_t i = 0; i < n; i++) {
        for (int k = 0; k < ploidy; k++) {
            const bool have = k < counts[i];
            const int32_t v = have ? vals[src + k] : 0;
            const size_t j = (size_t)i * ploidy + k;
            if (width == 1) ((int8_t *)out.data())[j] = have ? (int8_t)v : (int8_t)(INT8_MIN + 1);
            else if (width == 2) ((int16_t *)out.data())[j] = have ? (int16_t)v : (int16_t)(INT16_MIN + 1);
            else ((int32_t *)out.data())[j] = have ? v : INT32_MIN + 1;
        }
        src += counts[i];
    }
}

// INFO/END=<n> overrides the REF length for overlap (htslib vcf_parse / tabix readrec)
static int64_t rlen_from_info(const char *info, size_t len, int64_t pos, int64_t dflt) {
    size_t i = 0;
    while (i < len) {
        size_t e = i;
        while (e < len && info[e] != ';') e++;
        if (e - i > 4 && !memcmp(info + i, "END=", 4)) {
            long long end = atoll(std::string(info + i + 4, e - i - 4).c_str());
            return end >= pos ? end - pos + 1 : dflt;
        }
        i = e + 1;
    }
    return dflt;
}

// ------------------------------------------------------------------------------------------
// FORMAT/PL rows (DESIGN.md 4.10) -- not a reference input
// ------------------------------------------------------------------------------------------

// One sample's PL values -> its word of an NPC_GT_PL row: a | b << 12 | j << 24 | ploidy << 26 with m the smallest PL, j
// the index of its first occurrence, a, b the other genotypes' PL - m in genotype order, saturated at 4095 (T is 0 from
// 3237 on, so nothing is lost).  No value or any missing value: a missing sample.
static uint32_t pl_word(const int64_t *v, int cnt, bool missing, const VariantRecord &rec, const std::string &sample) {
    if (missing || cnt == 0) return 0xFFFFFFFFu;
    auto bad = [&](const std::string &m) {
        return InputError("record " + *rec.contig + ":" + std::to_string(rec.pos) + ": FORMAT/PL of sample " + sample + ": " + m);
    };
    if (cnt != 2 && cnt != 3)
        throw bad(std::to_string(cnt) + " values (a biallelic record has 3 for a diploid sample, 2 for a haploid one)");
    int j = 0;
    for (int g = 0; g < cnt; g++) {
        if (v[g] < 0) throw bad("negative value " + std::to_string(v[g]));
        if (v[g] < v[j]) j = g;
    }
    uint32_t x[2] = { 0, 0 };
    for (int g = 0, k = 0; g < cnt; g++)
        if (g != j) x[k++] = (uint32_t)std::min<int64_t>(v[g] - v[j], 4095);
    return x[0] | x[1] << 12 | (uint32_t)j << 24 | (uint32_t)(cnt - 1) << 26;
}

// A BCF PL field (per sample `len` integers of esz bytes, missing = MIN and vector_end = MIN + 1 of the width) -> n words
static void pack_pl_typed(const uint8_t *q, size_t esz, uint32_t len, int64_t n, uint8_t *dst, const VariantRecord &rec,
                          const std::vector<std::string> &samples) {
    for (int64_t i = 0; i < n; i++) {
        int64_t v[3];
        int cnt = 0;
        bool missing = false;
        for (uint32_t k = 0; k < len; k++) {
            const uint8_t *e = q + ((size_t)i * len + k) * esz;
            int64_t x, miss, vend;
            if (esz == 1) { x = (int8_t)*e; miss = INT8_MIN; vend = INT8_MIN + 1; }
            else if (esz == 2) { int16_t t; memcpy(&t, e, 2); x = t; miss = INT16_MIN; vend = INT16_MIN + 1; }
            else { int32_t t; memcpy(&t, e, 4); x = t; miss = INT32_MIN; vend = INT32_MIN + 1; }
            if (x == vend) break;
            if (x == miss) missing = true;
            else if (cnt < 3) v[cnt] = x;
            cnt++;
        }
        const uint32_t w = pl_word(v, cnt, missing, rec, samples[i]);
        memcpy(dst + 4 * i, &w, 4);
    }
}

// ------------------------------------------------------------------------------------------
// VCF text
// ------------------------------------------------------------------------------------------

class VcfTextSource : public VariantSource {
public:
    explicit VcfTextSource(std::unique_ptr<InflateStream> s) : in_(std::move(s)) {}
    bool read_header() {
        while (in_->getline(line_)) {
            if (line_.size() >= 2 && line_[0] == '#' && line_[1] == '#') continue;
            if (!line_.empty() && line_[0] == '#') {
                std::vector<std::string> f = split_char(line_, '\t');
                for (size_t i = 9; i < f.size(); i++) samples_.push_back(f[i]);
                return true;
            }
            return false;                              // data before the #CHROM line
        }
        return false;
    }
    InflateStream *stream() override { return in_.get(); }
    bool index_names_contigs() const override { return index_ && !index_->names().empty(); }
    int contig_rank(const VariantRecord &rec) const override { return contig_rank(*rec.contig); }
    int contig_rank(const std::string &name) const override {
        if (!index_) return -1;
        if (rank_.empty()) for (size_t i = 0; i < index_->names().size(); i++) rank_.emplace(index_->names()[i], (int)i);
        auto it = rank_.find(name);
        return it == rank_.end() ? -1 : it->second;
    }
    bool next_raw(VariantRecord &rec) override {
        for (;;) {
            if (!in_->getline(line_)) return false;
            if (!line_.empty()) break;
        }
        // split the 9 fixed columns in place
        const char *p = line_.data(), *end = p + line_.size();
        const char *col[10];
        size_t len[10];
        int nc = 0;
        while (nc < 9 && p <= end) {
            const char *t = (const char *)memchr(p, '\t', end - p);
            col[nc] = p; len[nc] = (t ? t : end) - p; nc++;
            if (!t) { p = end + 1; break; }
            p = t + 1;
        }
        if (nc < 8) throw InputError("VCF: record with fewer than 8 columns");
        contig_.assign(col[0], len[0]);
        rec.contig = &contig_; rec.contig_id = -1;
        rec.pos = parse_int_nim(std::string(col[1], len[1]), "VCF POS");
        rec.ref.assign(col[3], len[3]);
        rec.alts.clear();
        if (!(len[4] == 1 && col[4][0] == '.')) rec.alts = split_char(std::string(col[4], len[4]), ',');
        rec.filter.assign(col[6], len[6]);
        rec.rlen = rlen_from_info(col[7], len[7], rec.pos, (int64_t)rec.ref.size());
        rec.has_gt = false; rec.gt = nullptr; rec.ploidy = 0; rec.gt_width = 1;
        if (nc < 9 || samples_.empty()) return true;
        // FORMAT: index of GT
        int gt_idx = -1, k = 0;
        for (const char *q = col[8], *qe = col[8] + len[8]; q <= qe; k++) {
            const char *t = (const char *)memchr(q, ':', qe - q);
            size_t l = (t ? t : qe) - q;
            const char c0 = pl_ ? 'P' : dosage_ ? 'D' : 'G', c1 = pl_ ? 'L' : dosage_ ? 'S' : 'T';
            if (l == 2 && q[0] == c0 && q[1] == c1) gt_idx = k;
            if (!t) break;
            q = t + 1;
        }
        if (gt_idx < 0) return true;
        // the genotype columns are parsed only if the caller asks (load_gt): most records of a
        // genome-wide file match no score row
        rec.has_gt = true;
        gt_p_ = p; gt_idx_ = gt_idx; gt_loaded_ = false;
        return true;
    }
    bool load_gt_into(VariantRecord &rec, uint8_t *dst, int want_width, int want_ploidy) override {
        if (!pl_ || want_width != NPC_GT_PL || want_ploidy != 2 || !rec.has_gt || gt_loaded_) {
            load_gt(rec);
            return false;
        }
        gt_loaded_ = true;
        load_pl(rec, dst);
        return true;
    }
    void load_gt(VariantRecord &rec) override {
        if (!rec.has_gt || gt_loaded_) return;
        gt_loaded_ = true;
        const char *p = gt_p_, *end = line_.data() + line_.size();
        const int64_t n = n_samples();
        if (pl_) {
            gt_.resize((size_t)n * 4);
            load_pl(rec, gt_.data());
            return;
        }
        if (dosage_) {                                   // DS sub-field of every sample -> BCF floats ("." = missing)
            gt_.resize((size_t)n * 4);
            int maxv = 1;
            for (int64_t i = 0; i < n; i++) {
                const char *s = p <= end ? p : end, *se = end;
                if (p <= end) {
                    const char *t = (const char *)memchr(p, '\t', end - p);
                    se = t ? t : end;
                    p = t ? t + 1 : end + 1;
                }
                for (int f = 0; f < gt_idx_ && s < se; f++) {
                    const char *t = (const char *)memchr(s, ':', se - s);
                    s = t ? t + 1 : se;
                }
                const char *fe = (const char *)memchr(s, ':', se - s);
                if (!fe) fe = se;
                if (memchr(s, ',', fe - s)) maxv = 2;             // Number=A with several ALTs: the caller refuses
                uint32_t bits = 0x7F800001u;
                if (s < fe && !(fe - s == 1 && *s == '.')) {
                    const float v = (float)parse_float_nim(std::string(s, fe - s), "FORMAT/DS");
                    memcpy(&bits, &v, 4);
                }
                memcpy(gt_.data() + 4 * i, &bits, 4);
            }
            rec.ploidy = maxv; rec.gt_width = 4; rec.gt = gt_.data();
            return;
        }
        // fast path: every sample is "a/b" or "a|b" with one-character alleles and GT the first
        // sub-field -- written straight as int8 (allele+1)<<1|phased (htslib vcf_parse_format)
        if (gt_idx_ == 0 && p <= end) {
            gt_.resize((size_t)n * 2);
            int8_t *out = (int8_t *)gt_.data();
            const char *s = p;
            int64_t i = 0;
            for (; i < n; i++) {
                if (end - s < 3) break;
                const char c0 = s[0], sep = s[1], c1 = s[2];
                const bool ok0 = c0 == '.' || (c0 >= '0' && c0 <= '9'), ok1 = c1 == '.' || (c1 >= '0' && c1 <= '9');
                if (!ok0 || !ok1 || (sep != '/' && sep != '|')) break;
                const char *t = s + 3;
                if (t < end && *t != '\t') {
                    if (*t != ':') break;                          // longer allele number or another ploidy
                    t = (const char *)memchr(t, '\t', end - t);
                    if (!t) t = end;
                }
                out[2 * i] = c0 == '.' ? 0 : (int8_t)((c0 - '0' + 1) << 1);
                out[2 * i + 1] = (int8_t)((c1 == '.' ? 0 : ((c1 - '0' + 1) << 1)) | (sep == '|'));
                s = t + 1;
                if (t >= end && i + 1 < n) { i++; break; }
            }
            if (i == n) { rec.ploidy = 2; rec.gt_width = 1; rec.gt = gt_.data(); return; }
        }
        // general path: per-sample GT strings -> (allele+1)<<1|phased, any ploidy, any allele number
        vals_.clear(); counts_.assign(n, 0);
        int maxp = 1;
        const int gt_idx = gt_idx_;
        for (int64_t i = 0; i < n; i++) {
            const char *s = p <= end ? p : end, *se = end;
            if (p <= end) {
                const char *t = (const char *)memchr(p, '\t', end - p);
                se = t ? t : end;
                p = t ? t + 1 : end + 1;
            }
            for (int f = 0; f < gt_idx && s < se; f++) {          // skip to sub-field gt_idx
                const char *t = (const char *)memchr(s, ':', se - s);
                s = t ? t + 1 : se;
            }
            int l = 0, phased = 0;
            for (;;) {
                if (s < se && *s == '.') { s++; vals_.push_back(phased); l++; }
                else if (s < se && *s >= '0' && *s <= '9') {
                    uint32_t v = 0;
                    while (s < se && *s >= '0' && *s <= '9') v = v * 10 + (uint32_t)(*s++ - '0');
                    vals_.push_back((int32_t)(((v + 1) << 1) | (uint32_t)phased)); l++;
                } else break;
                if (s >= se) break;
                phased = *s == '|';
                if (*s != '|' && *s != '/') break;
                s++;
            }
            if (!l) { vals_.push_back(0); l = 1; }                // empty field = one missing allele
            counts_[i] = l;
            maxp = std::max(maxp, l);
        }
        pack_gt(vals_, counts_, n, maxp, gt_, rec.gt_width);
        rec.ploidy = maxp; rec.gt = gt_.data();
    }
private:
    // PL sub-field of every sample -> packed words in dst ("." or an absent sub-field = a missing sample)
    void load_pl(VariantRecord &rec, uint8_t *dst) {
        const char *p = gt_p_, *end = line_.data() + line_.size();
        const int64_t n = n_samples();
        for (int64_t i = 0; i < n; i++) {
            const char *s = p <= end ? p : end, *se = end;
            if (p <= end) {
                const char *t = (const char *)memchr(p, '\t', end - p);
                se = t ? t : end;
                p = t ? t + 1 : end + 1;
            }
            for (int f = 0; f < gt_idx_ && s < se; f++) {
                const char *t = (const char *)memchr(s, ':', se - s);
                s = t ? t + 1 : se;
            }
            const char *fe = (const char *)memchr(s, ':', se - s);
            if (!fe) fe = se;
            int64_t v[3];
            int cnt = 0;
            bool missing = false;
            while (s < fe) {
                const char *c = (const char *)memchr(s, ',', fe - s);
                if (!c) c = fe;
                if (c - s == 1 && *s == '.') missing = true;
                else {
                    const char *d = s;
                    const bool neg = *d == '-';
                    if (neg || *d == '+') d++;
                    if (d == c || c - d > 10)
                        throw InputError("record " + *rec.contig + ":" + std::to_string(rec.pos) + ": FORMAT/PL of sample " + samples_[i] +
                                         ": value \"" + std::string(s, c - s) + "\" is not an integer");
                    int64_t x = 0;
                    for (; d < c; d++) {
                        if (*d < '0' || *d > '9')
                            throw InputError("record " + *rec.contig + ":" + std::to_string(rec.pos) + ": FORMAT/PL of sample " + samples_[i] +
                                         ": value \"" + std::string(s, c - s) + "\" is not an integer");
                        x = x * 10 + (*d - '0');
                    }
                    if (cnt < 3) v[cnt] = neg ? -x : x;
                }
                cnt++;
                s = c + 1;
                if (c == fe) break;
            }
            const uint32_t w = pl_word(v, cnt, missing, rec, samples_[i]);
            memcpy(dst + 4 * i, &w, 4);
        }
        rec.ploidy = 2; rec.gt_width = NPC_GT_PL; rec.gt = dst;
    }
    std::unique_ptr<InflateStream> in_;
    std::string line_, contig_;
    const char *gt_p_ = nullptr;
    int gt_idx_ = -1;
    bool gt_loaded_ = true;
    mutable std::unordered_map<std::string, int> rank_;
    std::vector<int32_t> vals_;
    std::vector<int> counts_;
    std::vector<uint8_t> gt_;
};

// ------------------------------------------------------------------------------------------
// BCF2
// ------------------------------------------------------------------------------------------

class BcfSource : public VariantSource {
public:
    explicit BcfSource(std::unique_ptr<InflateStream> s) : in_(std::move(s)) {}
    bool read_header() {
        uint8_t magic[5];
        uint32_t l_text = 0;
        if (!in_->read_exact(magic, 5) || memcmp(magic, "BCF\2", 4) != 0) return false;
        if (!in_->read_exact(&l_text, 4)) return false;
        std::string text(l_text, '\0');
        if (!in_->read_exact(&text[0], l_text)) return false;
        parse_header(text);
        return true;
    }
    InflateStream *stream() override { return in_.get(); }
    void after_seek() override { indiv_left_ = 0; gt_done_ = true; }
    int contig_rank(const VariantRecord &rec) const override { return rec.contig_id; }       // CSI reference ids = header contig ids
    int contig_rank(const std::string &name) const override {
        for (size_t i = 0; i < contigs_.size(); i++) if (contigs_[i] == name) return (int)i;
        return -1;
    }
    bool next_raw(VariantRecord &rec) override {
        // the per-sample block of the previous record is consumed only on demand (load_gt / load_gt_into):
        // a record no score row matches costs no copy of its genotypes at all
        if (indiv_left_ && !in_->skip(indiv_left_)) throw InputError("BCF: truncated record");
        indiv_left_ = 0;
        uint32_t lens[2];
        size_t got = in_->read(lens, 8);
        if (got == 0) return false;
        if (got != 8) throw InputError("BCF: truncated record header");
        shared_.resize(lens[0]);
        if (!in_->read_exact(shared_.data(), lens[0])) throw InputError("BCF: truncated record");
        indiv_left_ = lens[1];
        if (lens[0] < 24) throw InputError("BCF: shared block too short");
        const uint8_t *p = shared_.data(), *e = p + shared_.size();
        int32_t chrom, pos0, rlen; uint32_t nai, nfs;
        memcpy(&chrom, p, 4); memcpy(&pos0, p + 4, 4); memcpy(&rlen, p + 8, 4);
        memcpy(&nai, p + 16, 4); memcpy(&nfs, p + 20, 4);
        p += 24;
        const uint32_t n_allele = nai >> 16, n_info = nai & 0xFFFF, n_fmt = nfs >> 24, n_sample = nfs & 0xFFFFFF;
        (void)n_info;
        if (chrom < 0 || (size_t)chrom >= contigs_.size() || contigs_[chrom].empty()) throw InputError("BCF: CHROM id not in header");
        rec.contig_id = chrom; rec.contig = &contigs_[chrom];
        rec.pos = (int64_t)pos0 + 1; rec.rlen = rlen;
        skip_typed(p, e);                                          // ID
        rec.ref.clear(); rec.alts.clear();
        for (uint32_t a = 0; a < n_allele; a++) {
            std::string s = read_typed_string(p, e);
            if (a == 0) rec.ref = std::move(s); else rec.alts.push_back(std::move(s));
        }
        // FILTER: typed int vector of dictionary ids
        {
            int type; uint32_t len;
            read_desc(p, e, type, len);
            rec.filter.clear();
            if (len == 0) rec.filter = ".";
            for (uint32_t i = 0; i < len; i++) {
                int32_t id = read_int(p, e, type);
                if (i) rec.filter += ';';
                rec.filter += dict_name(id);
            }
        }
        // FORMAT fields are looked at when the genotypes are asked for
        rec.has_gt = n_fmt > 0 && n_sample > 0; rec.gt = nullptr; rec.ploidy = 0; rec.gt_width = 1;
        n_fmt_ = n_fmt; n_sample_ = n_sample; gt_done_ = false;
        return true;
    }
    // whole per-sample block into indiv_, GT located inside it
    void load_gt(VariantRecord &rec) override {
        if (gt_done_) return;
        gt_done_ = true;
        indiv_.resize(indiv_left_);
        if (!in_->read_exact(indiv_.data(), indiv_left_)) throw InputError("BCF: truncated record");
        indiv_left_ = 0;
        rec.has_gt = false; rec.gt = nullptr; rec.ploidy = 0; rec.gt_width = 1;
        const uint8_t *q = indiv_.data(), *qe = q + indiv_.size();
        for (uint32_t f = 0; f < n_fmt_ && q < qe; f++) {
            int kt; uint32_t kl;
            read_desc(q, qe, kt, kl);
            int32_t key = read_int(q, qe, kt);
            int type; uint32_t len;
            read_desc(q, qe, type, len);
            const size_t esz = type == 1 ? 1 : type == 2 ? 2 : type == 3 ? 4 : type == 5 ? 4 : type == 7 ? 1 : 0;
            const size_t bytes = (size_t)n_sample_ * len * esz;
            if (q + bytes > qe) throw InputError("BCF: FORMAT field overruns the record");
            if (wanted(key, type)) {
                if ((int64_t)n_sample_ != n_samples()) throw InputError("BCF: record sample count differs from header");
                rec.has_gt = true; rec.gt = q; rec.gt_width = (int)esz; rec.ploidy = (int)len;
            }
            q += bytes;
        }
        pack_pl(rec, nullptr);
    }
    // The GT payload straight from the inflated blocks into dst (the pinned staging row) when its layout is the wanted
    // one: the only copy the genotypes make on the host.  The field headers in front of it are a few bytes each.
    bool load_gt_into(VariantRecord &rec, uint8_t *dst, int want_width, int want_ploidy) override {
        if (gt_done_) return false;
        uint8_t hdr[16];
        size_t left = indiv_left_;
        for (uint32_t f = 0; f < n_fmt_ && left; f++) {
            // key (typed int) and the type descriptor: read what a short header needs, byte by byte where lengths chain
            size_t h = 0;
            auto need = [&](size_t n) { if (left < n || !in_->read_exact(hdr + h, n)) throw InputError("BCF: truncated record"); h += n; left -= n; };
            need(1);
            const int kt = hdr[0] & 0xF;
            if ((hdr[0] >> 4) != 1 || (kt != 1 && kt != 2 && kt != 3)) { finish_general(rec, hdr, h, left); return false; }
            const size_t ksz = kt == 1 ? 1 : kt == 2 ? 2 : 4;
            need(ksz);
            const uint8_t *kp = hdr + 1;
            const int32_t key = read_int(kp, hdr + h, kt);
            const size_t d0 = h;
            need(1);
            int type = hdr[d0] & 0xF; uint32_t len = hdr[d0] >> 4;
            if (len == 15) {                                                // long vector: the length follows as a typed int
                need(1);
                const int lt = hdr[d0 + 1] & 0xF;
                if ((hdr[d0 + 1] >> 4) != 1 || (lt != 1 && lt != 2 && lt != 3)) { finish_general(rec, hdr, h, left); return false; }
                need(lt == 1 ? 1 : lt == 2 ? 2 : 4);
                const uint8_t *lp = hdr + d0 + 2;
                len = (uint32_t)read_int(lp, hdr + h, lt);
            }
            const size_t esz = type == 1 ? 1 : type == 2 ? 2 : type == 3 ? 4 : type == 5 ? 4 : type == 7 ? 1 : 0;
            const size_t bytes = (size_t)n_sample_ * len * esz;
            if (bytes > left) throw InputError("BCF: FORMAT field overruns the record");
            if (wanted(key, type)) {
                if ((int64_t)n_sample_ != n_samples()) throw InputError("BCF: record sample count differs from header");
                gt_done_ = true;
                rec.has_gt = true; rec.gt_width = (int)esz; rec.ploidy = (int)len;
                const bool direct = !pl_ && (int)esz == want_width && (int)len == want_ploidy;
                uint8_t *to = dst;
                if (!direct) { indiv_.resize(bytes); to = indiv_.data(); }
                if (!in_->read_exact(to, bytes)) throw InputError("BCF: truncated record");
                rec.gt = to;
                indiv_left_ = left - bytes;                                 // later fields: skipped when the next record is read
                if (pl_) return pack_pl(rec, want_width == NPC_GT_PL && want_ploidy == 2 ? dst : nullptr);
                return direct;
            }
            if (!in_->skip(bytes)) throw InputError("BCF: truncated record");
            left -= bytes;
        }
        indiv_left_ = left; gt_done_ = true;
        rec.has_gt = false; rec.gt = nullptr;
        return false;
    }
private:
    static void read_desc(const uint8_t *&p, const uint8_t *e, int &type, uint32_t &len) {
        if (p >= e) throw InputError("BCF: truncated typed value");
        const uint8_t d = *p++;
        type = d & 0xF; len = d >> 4;
        if (len == 15) {
            int t2; uint32_t l2;
            read_desc(p, e, t2, l2);
            len = (uint32_t)read_int(p, e, t2);
        }
    }
    static int32_t read_int(const uint8_t *&p, const uint8_t *e, int type) {
        int32_t v = 0;
        if (type == 1) { if (p + 1 > e) goto bad; v = (int8_t)*p; p += 1; }
        else if (type == 2) { if (p + 2 > e) goto bad; int16_t t; memcpy(&t, p, 2); v = t; p += 2; }
        else if (type == 3) { if (p + 4 > e) goto bad; memcpy(&v, p, 4); p += 4; }
        else throw InputError("BCF: expected an integer typed value");
        return v;
    bad:
        throw InputError("BCF: truncated integer");
    }
    static void skip_typed(const uint8_t *&p, const uint8_t *e) {
        int type; uint32_t len;
        read_desc(p, e, type, len);
        const size_t esz = type == 1 ? 1 : type == 2 ? 2 : type == 3 ? 4 : type == 5 ? 4 : type == 7 ? 1 : 0;
        if (p + (size_t)len * esz > e) throw InputError("BCF: truncated typed value");
        p += (size_t)len * esz;
    }
    static std::string read_typed_string(const uint8_t *&p, const uint8_t *e) {
        int type; uint32_t len;
        read_desc(p, e, type, len);
        if (type != 7 && len != 0) throw InputError("BCF: expected a string typed value");
        if (p + len > e) throw InputError("BCF: truncated string");
        std::string s((const char *)p, len);
        p += len;
        while (!s.empty() && s.back() == '\0') s.pop_back();
        return s;
    }
    const std::string &dict_name(int32_t id) const {
        static const std::string unknown = "?";
        return id >= 0 && (size_t)id < dict_.size() && !dict_[id].empty() ? dict_[id] : unknown;
    }
    // ID=..., optional IDX=... of one ##KEY=<...> line
    static bool meta_id(const std::string &line, size_t lt, std::string &id, int &idx) {
        idx = -1;
        size_t p = line.find("ID=", lt);
        if (p == std::string::npos) return false;
        size_t e = line.find_first_of(",>", p);
        id = line.substr(p + 3, (e == std::string::npos ? line.size() : e) - p - 3);
        size_t q = line.find("IDX=", lt);
        if (q != std::string::npos) idx = atoi(line.c_str() + q + 4);
        return true;
    }
    void parse_header(const std::string &text) {
        std::unordered_map<std::string, int> seen;
        auto add_dict = [&](const std::string &id, int idx) {
            auto it = seen.find(id);
            if (it != seen.end()) return;
            if (idx < 0) idx = (int)dict_next_++;
            else dict_next_ = std::max<size_t>(dict_next_, (size_t)idx + 1);
            if (dict_.size() <= (size_t)idx) dict_.resize(idx + 1);
            dict_[idx] = id;
            seen[id] = idx;
        };
        add_dict("PASS", 0);
        size_t b = 0;
        while (b < text.size()) {
            size_t e = text.find('\n', b);
            if (e == std::string::npos) e = text.size();
            std::string line = text.substr(b, e - b);
            while (!line.empty() && (line.back() == '\r' || line.back() == '\0')) line.pop_back();
            b = e + 1;
            if (line.rfind("##", 0) == 0) {
                size_t eq = line.find("=<");
                if (eq == std::string::npos) continue;
                const std::string key = line.substr(2, eq - 2);
                std::string id; int idx;
                if (!meta_id(line, eq, id, idx)) continue;
                if (key == "contig") {
                    if (idx < 0) idx = (int)contig_next_++;
                    else contig_next_ = std::max<size_t>(contig_next_, (size_t)idx + 1);
                    if (contigs_.size() <= (size_t)idx) contigs_.resize(idx + 1);
                    contigs_[idx] = id;
                } else if (key == "FILTER" || key == "INFO" || key == "FORMAT") {
                    add_dict(id, idx);
                }
            } else if (!line.empty() && line[0] == '#') {
                std::vector<std::string> f = split_char(line, '\t');
                for (size_t i = 9; i < f.size(); i++) samples_.push_back(f[i]);
            }
        }
        auto it = seen.find("GT");
        gt_key_ = it == seen.end() ? -1 : it->second;
        it = seen.find("DS");
        ds_key_ = it == seen.end() ? -1 : it->second;
        it = seen.find("PL");
        pl_key_ = it == seen.end() ? -1 : it->second;
    }
    // the FORMAT field the caller reads: GT (typed ints), in dosage mode DS (floats), in PL mode PL (typed ints)
    bool wanted(int32_t key, int type) const {
        if (pl_) return key == pl_key_ && (type == 1 || type == 2 || type == 3);
        return dosage_ ? (key == ds_key_ && type == 5) : (key == gt_key_ && (type == 1 || type == 2 || type == 3));
    }
    std::unique_ptr<InflateStream> in_;
    std::vector<std::string> contigs_, dict_;
    size_t dict_next_ = 0, contig_next_ = 0;
    // an unusual field header inside load_gt_into: put the bytes read so far back in front and take the general path
    void finish_general(VariantRecord &rec, const uint8_t *hdr, size_t h, size_t left) {
        indiv_.resize(h + left);
        memcpy(indiv_.data(), hdr, h);
        if (!in_->read_exact(indiv_.data() + h, left)) throw InputError("BCF: truncated record");
        // fields already skipped are gone; the general parser starts at this field
        indiv_left_ = 0; gt_done_ = true;
        rec.has_gt = false; rec.gt = nullptr; rec.ploidy = 0; rec.gt_width = 1;
        const uint8_t *q = indiv_.data(), *qe = q + indiv_.size();
        while (q < qe) {
            int kt; uint32_t kl;
            read_desc(q, qe, kt, kl);
            int32_t key = read_int(q, qe, kt);
            int type; uint32_t len;
            read_desc(q, qe, type, len);
            const size_t esz = type == 1 ? 1 : type == 2 ? 2 : type == 3 ? 4 : type == 5 ? 4 : type == 7 ? 1 : 0;
            const size_t bytes = (size_t)n_sample_ * len * esz;
            if (q + bytes > qe) throw InputError("BCF: FORMAT field overruns the record");
            if (wanted(key, type)) { rec.has_gt = true; rec.gt = q; rec.gt_width = (int)esz; rec.ploidy = (int)len; }
            q += bytes;
        }
        pack_pl(rec, nullptr);
    }
    // PL mode: the typed integers rec.gt points at -> packed words in dst, or in pl_buf_ when dst is null; true when
    // written to dst.  Nothing to do in the other modes or without a PL field.
    bool pack_pl(VariantRecord &rec, uint8_t *dst) {
        if (!pl_ || !rec.has_gt || !rec.gt) return false;
        const int64_t n = n_samples();
        if (!dst) { pl_buf_.resize((size_t)n * 4); }
        uint8_t *to = dst ? dst : pl_buf_.data();
        pack_pl_typed(rec.gt, (size_t)rec.gt_width, (uint32_t)rec.ploidy, n, to, rec, samples_);
        rec.gt = to; rec.gt_width = NPC_GT_PL; rec.ploidy = 2;
        return dst != nullptr;
    }
    std::vector<uint8_t> pl_buf_;
    int32_t gt_key_ = -1, ds_key_ = -1, pl_key_ = -1;
    size_t indiv_left_ = 0;
    uint32_t n_fmt_ = 0, n_sample_ = 0;
    bool gt_done_ = true;
    std::vector<uint8_t> shared_, indiv_;
};

// ------------------------------------------------------------------------------------------
// PLINK 1 binary fileset (.bed + .bim + .fam), DESIGN.md 4.7 -- not a reference input
// ------------------------------------------------------------------------------------------

// The .bim is read whole at open (it sizes and checks the .bed); next() walks its lines in file order, and a row of the
// .bed is read by offset only when the driver asks for it (load_gt / load_gt_into): a few hundred scored loci on a
// genome-wide fileset read a few hundred rows, no index needed.  Per line: CHROM = column 1 (compared literally),
// POS = column 4, ALT = A1 (column 5; "0" = no ALT), REF = A2 (column 6), rlen = len(REF), FILTER ".".
class PlinkSource : public VariantSource {
public:
    ~PlinkSource() override { if (fd_ >= 0) ::close(fd_); }
    // false: a sibling file cannot be opened.  Throws InputError on a malformed fileset.
    bool open(const std::string &bed_path, uint8_t mode) {
        if (mode == 0x00) throw InputError("PLINK .bed " + bed_path + ": individual-major mode (mode byte 00) is not supported");
        if (mode != 0x01) throw InputError("PLINK .bed " + bed_path + ": unknown mode byte");
        const std::string prefix = bed_path.size() > 4 && bed_path.compare(bed_path.size() - 4, 4, ".bed") == 0
                                       ? bed_path.substr(0, bed_path.size() - 4) : bed_path;
        FILE *fam = fopen((prefix + ".fam").c_str(), "rb");
        if (!fam) return false;
        FILE *bim = fopen((prefix + ".bim").c_str(), "rb");
        if (!bim) { fclose(fam); return false; }
        std::string line;
        auto getline = [&line](FILE *f) {
            line.clear();
            int ch;
            while ((ch = fgetc(f)) != EOF && ch != '\n') line += (char)ch;
            if (!line.empty() && line.back() == '\r') line.pop_back();
            return ch != EOF || !line.empty();
        };
        auto fields = [&line]() {
            std::vector<std::string> f;
            size_t i = 0;
            while (i < line.size()) {
                while (i < line.size() && (line[i] == ' ' || line[i] == '\t')) i++;
                size_t j = i;
                while (j < line.size() && line[j] != ' ' && line[j] != '\t') j++;
                if (j > i) f.emplace_back(line, i, j - i);
                i = j;
            }
            return f;
        };
        int64_t ln = 0;
        while (getline(fam)) {
            ln++;
            std::vector<std::string> f = fields();
            if (f.empty()) continue;
            if (f.size() < 2) { fclose(fam); fclose(bim); throw InputError("PLINK .fam line " + std::to_string(ln) + ": fewer than 2 columns"); }
            samples_.push_back(f[1]);                                   // IID
        }
        fclose(fam);
        std::unordered_map<std::string, int32_t> ids;
        ln = 0;
        try {
            while (getline(bim)) {
                ln++;
                std::vector<std::string> f = fields();
                if (f.empty()) continue;
                const std::string where = "PLINK .bim line " + std::to_string(ln);
                if (f.size() < 6) throw InputError(where + ": fewer than 6 columns");
                Line L;
                auto it = ids.find(f[0]);
                if (it == ids.end()) { it = ids.emplace(f[0], (int32_t)contigs_.size()).first; contigs_.push_back(f[0]); }
                L.contig = it->second;
                L.pos = parse_int_nim(f[3], (where + " POS").c_str());
                if (L.pos < 1) throw InputError(where + ": bad POS " + f[3]);
                L.alt = f[4]; L.ref = f[5];
                lines_.push_back(std::move(L));
            }
        } catch (...) { fclose(bim); throw; }
        fclose(bim);
        fd_ = ::open(bed_path.c_str(), O_RDONLY);
        if (fd_ < 0) return false;
        struct stat st;
        if (fstat(fd_, &st) != 0) return false;
        row_bytes_ = npc_gt_row_bytes((int64_t)samples_.size(), 2, NPC_GT_BED);
        const int64_t want = 3 + (int64_t)lines_.size() * row_bytes_;
        if ((int64_t)st.st_size != want)
            throw InputError("PLINK .bed " + bed_path + " holds " + std::to_string((long long)st.st_size) + " bytes; " +
                             std::to_string(lines_.size()) + " variants x " + std::to_string(samples_.size()) + " samples need " + std::to_string(want));
        return true;
    }
    int fixed_layout() const override { return NPC_GT_BED; }
    void load_gt(VariantRecord &rec) override {
        buf_.resize((size_t)std::max<int64_t>(row_bytes_, 1));
        read_row(buf_.data());
        fill(rec, buf_.data());
    }
    bool load_gt_into(VariantRecord &rec, uint8_t *dst, int want_width, int want_ploidy) override {
        if (want_width != NPC_GT_BED || want_ploidy != 2) { load_gt(rec); return false; }
        read_row(dst);
        fill(rec, dst);
        return true;
    }
protected:
    bool next_raw(VariantRecord &rec) override {
        if (cur_ + 1 >= (int64_t)lines_.size()) { cur_ = (int64_t)lines_.size(); return false; }
        const Line &L = lines_[(size_t)++cur_];
        rec.contig_id = L.contig; rec.contig = &contigs_[(size_t)L.contig];
        rec.pos = L.pos; rec.ref = L.ref; rec.rlen = (int64_t)L.ref.size();
        rec.alts.clear();
        if (L.alt != "0") rec.alts.push_back(L.alt);
        rec.filter = ".";
        rec.has_gt = true; rec.gt = nullptr; rec.gt_width = NPC_GT_BED; rec.ploidy = 2;
        return true;
    }
    InflateStream *stream() override { return nullptr; }               // no index-driven mode: use_regions returns false
    int contig_rank(const VariantRecord &rec) const override { return rec.contig_id; }
    int contig_rank(const std::string &) const override { return -1; }
private:
    struct Line { int32_t contig; int64_t pos; std::string ref, alt; };
    void read_row(uint8_t *dst) {
        const int64_t off = 3 + cur_ * row_bytes_;
        int64_t got = 0;
        while (got < row_bytes_) {
            const ssize_t r = pread(fd_, dst + got, (size_t)(row_bytes_ - got), (off_t)(off + got));
            if (r <= 0) throw InputError("PLINK .bed: read failed at byte " + std::to_string((long long)(off + got)));
            got += r;
        }
    }
    void fill(VariantRecord &rec, const uint8_t *row) const { rec.has_gt = true; rec.gt = row; rec.gt_width = NPC_GT_BED; rec.ploidy = 2; }
    std::vector<std::string> contigs_;
    std::vector<Line> lines_;
    std::vector<uint8_t> buf_;
    int64_t cur_ = -1, row_bytes_ = 0;
    int fd_ = -1;
};

// ------------------------------------------------------------------------------------------
// BGEN v1.2, layout 2, 1 to 16 bits per probability (DESIGN.md 4.8, 4.9) -- not a reference input
// ------------------------------------------------------------------------------------------

// One genotype block -> one row of fixed-point dosages, in either layout:
//   NPC_GT_DOSE255  8 bits, diploid: per sample k = 255 x the expected ALT dosage as a little-endian uint16, 0xFFFF for a
//                   missing sample.  A well-formed block these rows cannot hold throws NeedsDose32.
//   NPC_GT_DOSE32   1 to 16 bits, haploid and diploid samples: the row header (uint32 D = 2^B - 1, 12 zero bytes), then
//                   per sample the uint32 word k | ploidy << 24, 0xFFFFFFFF for a missing sample (npc_dose32.cuh).
// Each thread that converts blocks has one of these: its own file descriptor, inflate tables and buffers.
class BgenBlockReader {
public:
    BgenBlockReader(const std::string &path, int64_t n, bool compressed) : n_(n), compressed_(compressed) {
        fd_ = ::open(path.c_str(), O_RDONLY);
        if (fd_ < 0) throw InputError("BGEN " + path + ": cannot reopen the file");
    }
    ~BgenBlockReader() { if (fd_ >= 0) ::close(fd_); }
    BgenBlockReader(const BgenBlockReader &) = delete;
    BgenBlockReader &operator=(const BgenBlockReader &) = delete;
    // off / C: file offset and length of the genotype block after its C field; what: the variant, for messages
    // layout: NPC_GT_DOSE255 or NPC_GT_DOSE32
    void convert(int64_t off, uint32_t C, uint8_t *dst, const std::string &what, int layout) {
        in_.resize((size_t)C + 16);
        int64_t got = 0;
        while (got < (int64_t)C) {
            const ssize_t r = pread(fd_, in_.data() + got, (size_t)(C - got), (off_t)(off + got));
            if (r <= 0) throw InputError("BGEN: read failed in the genotype block of " + what);
            got += r;
        }
        const uint8_t *p = in_.data();
        size_t len = C;
        if (compressed_) {
            if (C < 4) throw InputError("BGEN: genotype block of " + what + " is too short");
            uint32_t D;
            memcpy(&D, in_.data(), 4);
            out_.resize((size_t)D + 16);
            // a zlib stream: 2-byte header, raw deflate, Adler-32.  This engine's decoder first, zlib where it does not finish.
            const uint8_t *z = in_.data() + 4;
            const size_t zl = C - 4;
            bool ok = zl >= 6 && (z[0] & 0x0F) == 8 && !(z[1] & 0x20) && fast_inflate(z + 2, zl - 6, out_.data(), D, tabs_);
            if (ok) {
                const uint32_t want = (uint32_t)z[zl - 4] << 24 | (uint32_t)z[zl - 3] << 16 | (uint32_t)z[zl - 2] << 8 | z[zl - 1];
                ok = (uint32_t)adler32(1L, out_.data(), D) == want;
            }
            if (!ok) {
                uLongf dl = D;
                if (uncompress(out_.data(), &dl, z, (uLong)zl) != Z_OK || dl != D)
                    throw InputError("BGEN: corrupt compressed genotype block of " + what);
            }
            p = out_.data(); len = D;
        }
        if (layout == NPC_GT_DOSE32) decode32(p, len, dst, what);
        else decode(p, len, dst, what);
    }
private:
    InputError bad(const std::string &what, const std::string &m) const { return InputError("BGEN: variant " + what + ": " + m); }
    // NeedsDose32 when the block is well-formed; decode32 refuses it otherwise
    NeedsDose32 needs32(const uint8_t *p, size_t len, const std::string &what, const std::string &m) const {
        decode32(p, len, nullptr, what);
        return NeedsDose32("BGEN: variant " + what + ": " + m + " (needs 32-bit dosage rows)");
    }
    void decode(const uint8_t *p, size_t len, uint8_t *dst, const std::string &what) const {
        if (len < 8) throw bad(what, "genotype block too short");
        uint32_t N; uint16_t K;
        memcpy(&N, p, 4); memcpy(&K, p + 4, 2);
        const int pmin = p[6], pmax = p[7];
        if ((int64_t)N != n_) throw bad(what, "genotype block holds " + std::to_string(N) + " samples, the header " + std::to_string(n_));
        if (K != 2) throw bad(what, std::to_string(K) + " alleles (only biallelic variants are supported)");
        if (pmin != 2 || pmax != 2) throw needs32(p, len, what, "ploidy " + std::to_string(pmin) + ".." + std::to_string(pmax));
        if (len < 8 + (size_t)n_ + 2) throw bad(what, "genotype block too short");
        const uint8_t *ploidy = p + 8, *q = p + 8 + n_;
        const bool phased = q[0] != 0;
        const int B = q[1];
        if (B != 8) throw needs32(p, len, what, std::to_string(B) + " bits per probability");
        if (len < 8 + (size_t)n_ + 2 + 2 * (size_t)n_) throw bad(what, "genotype block too short");
        const uint8_t *pr = q + 2;
        for (int64_t i = 0; i < n_; i++) {
            const uint32_t a = pr[2 * i], b = pr[2 * i + 1];
            uint32_t k;
            if (ploidy[i] & 0x80) k = 0xFFFF;
            else if (phased) k = 510 - a - b;                             // (255 - h0) + (255 - h1)
            else {
                if (a + b > 255) throw bad(what, "sample " + std::to_string(i) + ": P(hom allele 1) + P(het) > 1");
                k = 510 - 2 * a - b;                                      // P(het) + 2 P(hom allele 2), in 1/255
            }
            const uint16_t v = (uint16_t)k;
            memcpy(dst + 2 * i, &v, 2);
        }
    }
    // dst == nullptr: check the block only.  Each sample stores `ploidy` values of B bits (phased or not, K = 2), packed
    // back to back least-significant bit first; a missing sample still occupies its values.
    void decode32(const uint8_t *p, size_t len, uint8_t *dst, const std::string &what) const {
        if (len < 8) throw bad(what, "genotype block too short");
        uint32_t N; uint16_t K;
        memcpy(&N, p, 4); memcpy(&K, p + 4, 2);
        const int pmin = p[6], pmax = p[7];
        if ((int64_t)N != n_) throw bad(what, "genotype block holds " + std::to_string(N) + " samples, the header " + std::to_string(n_));
        if (K != 2) throw bad(what, std::to_string(K) + " alleles (only biallelic variants are supported)");
        if (pmax > 2) throw bad(what, "ploidy " + std::to_string(pmin) + ".." + std::to_string(pmax) + " (only haploid and diploid samples are supported)");
        if (len < 8 + (size_t)n_ + 2) throw bad(what, "genotype block too short");
        const uint8_t *ploidy = p + 8, *q = p + 8 + n_;
        const bool phased = q[0] != 0;
        const int B = q[1];
        if (B < 1 || B > 16) throw bad(what, std::to_string(B) + " bits per probability (1 to 16 are supported)");
        uint64_t values = 0;
        for (int64_t i = 0; i < n_; i++) {
            const int pl = ploidy[i] & 0x3F;
            if (pl < pmin || pl > pmax)
                throw bad(what, "sample " + std::to_string(i) + ": ploidy " + std::to_string(pl) + " outside " + std::to_string(pmin) + ".." + std::to_string(pmax));
            values += (uint64_t)pl;
        }
        if (len - (8 + (size_t)n_ + 2) < (values * (uint64_t)B + 7) / 8)
            throw bad(what, "genotype block too short for " + std::to_string(n_) + " samples at " + std::to_string(B) + " bits");
        const uint32_t D = (1u << B) - 1, mask = D;
        const uint8_t *src = q + 2;
        uint64_t acc = 0;
        int have = 0;
        auto next = [&]() -> uint32_t {                                   // the next B-bit value of the stream
            while (have < B) { acc |= (uint64_t)*src++ << have; have += 8; }
            const uint32_t v = (uint32_t)acc & mask;
            acc >>= B; have -= B;
            return v;
        };
        if (dst) {
            memset(dst, 0, 16);
            memcpy(dst, &D, 4);
        }
        for (int64_t i = 0; i < n_; i++) {
            const int pl = ploidy[i] & 0x3F;
            uint32_t w = 0xFFFFFFFFu;
            if (pl == 1) {
                const uint32_t a = next();
                w = (D - a) | 1u << 24;                                   // P(allele 2), in 1/D
            } else if (pl == 2) {
                const uint32_t a = next(), b = next();
                if (phased) w = (2 * D - a - b) | 2u << 24;               // (D - h0) + (D - h1)
                else {
                    if (a + b > D && !(ploidy[i] & 0x80)) throw bad(what, "sample " + std::to_string(i) + ": P(hom allele 1) + P(het) > 1");
                    w = (2 * D - 2 * a - b) | 2u << 24;                   // P(het) + 2 P(hom allele 2), in 1/D
                }
            }
            if (ploidy[i] & 0x80) w = 0xFFFFFFFFu;
            if (dst) memcpy(dst + 16 + 4 * i, &w, 4);
        }
    }
    int fd_ = -1;
    int64_t n_;
    bool compressed_;
    std::vector<uint8_t> in_, out_;
    FastInflateTables tabs_;
};

// The header and sample identifiers are read at open; next() walks the variant headers and skips each genotype block by
// its length (there is no index: a .bgi is an SQLite file).  A block is read and converted only when a score row matched
// its variant (load_gt / load_gt_into).  load_gt_into hands the block to a pool of NIMPRESS_THREADS workers and returns;
// wait_rows() waits for every block posted so far, and rethrows a worker's InputError (before a worker's NeedsDose32, so
// that which of them is thrown does not depend on the workers' timing).  Per variant: CHROM = chromosome (compared
// literally), POS, REF = allele 1, ALT = allele 2 (and any further alleles), rlen = len(REF), FILTER ".".
class BgenSource : public VariantSource {
public:
    ~BgenSource() override {
        {
            std::lock_guard<std::mutex> g(mu_);
            stop_ = true;
        }
        cv_.notify_all();
        for (auto &t : workers_) t.join();
        if (fp_) fclose(fp_);
    }
    // false: the file cannot be read, or the .sample it needs cannot be opened.  Throws InputError on a malformed file.
    bool open(const std::string &path) {
        path_ = path;
        fp_ = fopen(path.c_str(), "rb");
        if (!fp_) return false;
        fseeko(fp_, 0, SEEK_END);
        size_ = (int64_t)ftello(fp_);
        fseeko(fp_, 0, SEEK_SET);
        const std::string where = "BGEN " + path;
        uint32_t offset, LH, M, N, flags;
        if (!rd(&offset, 4) || !rd(&LH, 4) || !rd(&M, 4) || !rd(&N, 4)) throw InputError(where + ": truncated header");
        if (LH < 20) throw InputError(where + ": header length " + std::to_string(LH) + " < 20");
        if (offset < LH) throw InputError(where + ": variant data offset " + std::to_string(offset) + " lies inside the header block");
        if ((int64_t)LH + 4 > size_ || fseeko(fp_, (off_t)LH, SEEK_SET) != 0 || !rd(&flags, 4)) throw InputError(where + ": truncated header");
        const int comp = flags & 3, layout = (flags >> 2) & 15;
        if (comp == 2) throw InputError(where + ": zstd-compressed genotype blocks are not supported");
        if (comp == 3) throw InputError(where + ": unknown compression " + std::to_string(comp));
        if (layout != 2) throw InputError(where + ": layout " + std::to_string(layout) + " is not supported (layout 2 only)");
        compressed_ = comp == 1;
        n_ = N; m_ = M;
        if (flags & 0x80000000u) {                                        // sample identifier block
            uint32_t LSI, NS;
            if (!rd(&LSI, 4) || !rd(&NS, 4)) throw InputError(where + ": truncated sample identifier block");
            if (NS != N) throw InputError(where + ": " + std::to_string(NS) + " sample identifiers for " + std::to_string(N) + " samples");
            for (uint32_t i = 0; i < N; i++) samples_.push_back(str16(where + ": truncated sample identifier block"));
        } else {
            const std::string stem = path.size() > 5 && path.compare(path.size() - 5, 5, ".bgen") == 0 ? path.substr(0, path.size() - 5) : path;
            FILE *sf = fopen((stem + ".sample").c_str(), "rb");
            if (!sf) return false;
            std::string line;
            int64_t ln = 0;
            for (;;) {
                line.clear();
                int ch;
                while ((ch = fgetc(sf)) != EOF && ch != '\n') line += (char)ch;
                if (ch == EOF && line.empty()) break;
                if (++ln <= 2) continue;                                 // header line, type line
                size_t i = 0;
                std::string cols[2];
                for (int c = 0; c < 2; c++) {
                    while (i < line.size() && isspace((unsigned char)line[i])) i++;
                    const size_t j0 = i;
                    while (i < line.size() && !isspace((unsigned char)line[i])) i++;
                    cols[c] = line.substr(j0, i - j0);
                }
                if (cols[0].empty() && cols[1].empty()) continue;
                if (cols[1].empty()) { fclose(sf); throw InputError(where + ": .sample line " + std::to_string(ln) + " has fewer than 2 columns"); }
                samples_.push_back(cols[1]);                             // ID_2
            }
            fclose(sf);
            if ((int64_t)samples_.size() != (int64_t)N)
                throw InputError(where + ": the .sample file names " + std::to_string(samples_.size()) + " samples, the header " + std::to_string(N));
        }
        pos_ = 4 + (int64_t)offset;
        if (pos_ > size_ || fseeko(fp_, (off_t)pos_, SEEK_SET) != 0) throw InputError(where + ": truncated before the first variant");
        const unsigned hc = std::max(1u, std::thread::hardware_concurrency());
        threads_ = (int)std::min<unsigned>(hc > 2 ? hc - 1 : hc, 32u);
        if (const char *e = getenv("NIMPRESS_THREADS")) if (*e) threads_ = std::max(1, atoi(e));
        return true;
    }
    int fixed_layout() const override { return NPC_GT_DOSE255; }
    void load_gt(VariantRecord &rec) override {
        buf_.resize((size_t)std::max<int64_t>(2 * n_, 1));
        inline_reader().convert(blk_off_, blk_len_, buf_.data(), what_, NPC_GT_DOSE255);
        fill(rec, buf_.data(), NPC_GT_DOSE255);
    }
    bool load_gt_into(VariantRecord &rec, uint8_t *dst, int want_width, int want_ploidy) override {
        if ((want_width != NPC_GT_DOSE255 && want_width != NPC_GT_DOSE32) || want_ploidy != 2) { load_gt(rec); return false; }
        if (threads_ <= 1) inline_reader().convert(blk_off_, blk_len_, dst, what_, want_width);
        else {
            std::lock_guard<std::mutex> g(mu_);
            if (workers_.empty())
                for (int t = 0; t < threads_; t++) workers_.emplace_back([this] { work(); });
            jobs_.push_back(Job{ blk_off_, blk_len_, dst, what_, want_width });
            pending_++;
            cv_.notify_one();
        }
        fill(rec, dst, want_width);
        return true;
    }
    void wait_rows() override {
        std::unique_lock<std::mutex> lk(mu_);
        done_.wait(lk, [this] { return pending_ == 0; });
        std::string e;
        if (!err_.empty()) { e.swap(err_); need32_.clear(); throw InputError(e); }
        if (!need32_.empty()) { e.swap(need32_); throw NeedsDose32(e); }
    }
protected:
    bool next_raw(VariantRecord &rec) override {
        if (read_ >= m_) return false;
        const std::string where = "BGEN " + path_ + ": variant block " + std::to_string(read_ + 1) + " of " + std::to_string(m_);
        const std::string trunc = where + " is truncated";
        id_ = str16(trunc);
        str16(trunc);                                                     // rsid
        std::string chrom = str16(trunc);
        uint32_t pos; uint16_t K;
        if (!rd(&pos, 4) || !rd(&K, 2)) throw InputError(trunc);
        rec.alts.clear();
        rec.ref.clear();
        for (uint16_t a = 0; a < K; a++) {
            uint32_t L;
            if (!rd(&L, 4) || pos_ + (int64_t)L > size_) throw InputError(trunc);
            std::string s(L, '\0');
            if (L && !rd(&s[0], L)) throw InputError(trunc);
            if (a == 0) rec.ref = std::move(s); else rec.alts.push_back(std::move(s));
        }
        uint32_t C;
        if (!rd(&C, 4)) throw InputError(trunc);
        blk_off_ = pos_; blk_len_ = C;
        if (pos_ + (int64_t)C > size_ || fseeko(fp_, (off_t)(pos_ + C), SEEK_SET) != 0) throw InputError(trunc);
        pos_ += C;
        read_++;
        auto it = ids_.find(chrom);
        if (it == ids_.end()) { it = ids_.emplace(chrom, (int32_t)contigs_.size()).first; contigs_.push_back(chrom); }
        rec.contig_id = it->second; rec.contig = &contigs_[(size_t)it->second];
        rec.pos = pos; rec.rlen = (int64_t)rec.ref.size(); rec.filter = ".";
        rec.has_gt = true; rec.gt = nullptr; rec.gt_width = NPC_GT_DOSE255; rec.ploidy = 2;
        what_ = chrom + ":" + std::to_string(pos) + " (" + id_ + ")";
        return true;
    }
    InflateStream *stream() override { return nullptr; }               // no index-driven mode: use_regions returns false
    int contig_rank(const VariantRecord &rec) const override { return rec.contig_id; }
    int contig_rank(const std::string &) const override { return -1; }
private:
    struct Job { int64_t off; uint32_t len; uint8_t *dst; std::string what; int layout; };
    bool rd(void *dst, size_t n) {
        if (fread(dst, 1, n, fp_) != n) return false;
        pos_ += (int64_t)n;
        return true;
    }
    std::string str16(const std::string &err) {
        uint16_t L;
        if (!rd(&L, 2)) throw InputError(err);
        std::string s(L, '\0');
        if (L && !rd(&s[0], L)) throw InputError(err);
        return s;
    }
    BgenBlockReader &inline_reader() {
        if (!inline_) inline_ = std::make_unique<BgenBlockReader>(path_, n_, compressed_);
        return *inline_;
    }
    void fill(VariantRecord &rec, const uint8_t *row, int layout) const { rec.has_gt = true; rec.gt = row; rec.gt_width = layout; rec.ploidy = 2; }
    void work() {
        std::unique_ptr<BgenBlockReader> r;
        for (;;) {
            Job j;
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [this] { return stop_ || !jobs_.empty(); });
                if (jobs_.empty()) return;
                j = std::move(jobs_.front());
                jobs_.pop_front();
            }
            std::string e, e32;
            try {
                if (!r) r = std::make_unique<BgenBlockReader>(path_, n_, compressed_);
                r->convert(j.off, j.len, j.dst, j.what, j.layout);
            } catch (const NeedsDose32 &x) { e32 = x.what(); }
            catch (const InputError &x) { e = x.what(); }
            std::lock_guard<std::mutex> g(mu_);
            if (!e.empty() && err_.empty()) err_ = e;
            if (!e32.empty() && need32_.empty()) need32_ = e32;
            if (--pending_ == 0) done_.notify_all();
        }
    }
    std::string path_, id_, what_;
    FILE *fp_ = nullptr;
    int64_t size_ = 0, pos_ = 0, n_ = 0, m_ = 0, read_ = 0, blk_off_ = 0;
    uint32_t blk_len_ = 0;
    bool compressed_ = false;
    std::vector<std::string> contigs_;
    std::unordered_map<std::string, int32_t> ids_;
    std::vector<uint8_t> buf_;
    std::unique_ptr<BgenBlockReader> inline_;
    int threads_ = 1;
    std::mutex mu_;
    std::condition_variable cv_, done_;
    std::deque<Job> jobs_;
    int64_t pending_ = 0;
    bool stop_ = false;
    std::string err_, need32_;
    std::vector<std::thread> workers_;
};

// ------------------------------------------------------------------------------------------
// index-driven region mode
// ------------------------------------------------------------------------------------------

VariantSource::VariantSource() = default;
VariantSource::~VariantSource() = default;

bool VariantSource::use_regions(const std::unordered_map<std::string, std::vector<std::pair<int64_t, int64_t>>> &spans,
                                const std::string &path) {
    if (const char *e = getenv("NIMPRESS_NO_INDEX")) if (*e && *e != '0') return false;
    InflateStream *in = stream();
    if (!in || !in->is_bgzf()) return false;
    index_ = RegionIndex::load(path);
    if (!index_) return false;
    if (!index_names_contigs()) { index_.reset(); return false; }
    std::vector<Region> regs;
    for (const auto &kv : spans) {
        const int ref = contig_rank(kv.first);
        if (ref < 0 || ref >= index_->n_ref()) continue;            // contig not in the file: its loci stay unmatched, as when streaming
        for (const auto &sp : kv.second) regs.push_back(Region{ ref, sp.first - 1, sp.second });
    }
    std::sort(regs.begin(), regs.end(), [](const Region &a, const Region &b) { return a.ref != b.ref ? a.ref < b.ref : a.beg0 < b.beg0; });
    std::vector<Region> merged;                                       // spans closer than one 16 kb index window are one region
    for (const Region &r : regs) {
        if (!merged.empty() && merged.back().ref == r.ref && r.beg0 <= merged.back().end0 + (1 << 14)) merged.back().end0 = std::max(merged.back().end0, r.end0);
        else merged.push_back(r);
    }
    // Jumping reads block by block with one zlib stream (no inflate pool: several times slower per byte than
    // streaming).  Estimate the compressed bytes the regions need from the index itself -- from the first record
    // of a region to the first record at its end, plus a block -- and use the index only when that is a small
    // part of the file.
    const char *force = getenv("NIMPRESS_FORCE_INDEX");
    if (!(force && *force && *force != '0')) {
        int64_t est = 0;
        for (const Region &r : merged) {
            const uint64_t v0 = index_->query_start(r.ref, r.beg0, r.end0);
            if (v0 == RegionIndex::NONE) continue;
            const uint64_t v1 = index_->query_start(r.ref, r.end0, r.end0 + 1);
            const int64_t c0 = (int64_t)(v0 >> 16), c1 = v1 == RegionIndex::NONE ? in->file_size() : (int64_t)(v1 >> 16);
            est += std::max<int64_t>(c1 - c0, 0) + (64 << 10);
        }
        if (est * 8 > in->file_size()) { index_.reset(); return false; }
    }
    // The pass below walks the regions in header-contig order and only ever seeks forward.  htslib merely
    // requires each contig's records to be contiguous, so a file may hold its contig blocks in another order
    // than its header names them (and index fine): the regions' first records must then be visited in FILE
    // order, which the rank-ordered walk cannot do -- stream such a file instead of silently missing loci.
    {
        uint64_t last = 0;
        for (const Region &r : merged) {
            const uint64_t v0 = index_->query_start(r.ref, r.beg0, r.end0);
            if (v0 == RegionIndex::NONE) continue;
            if (v0 < last) { index_.reset(); return false; }
            last = v0;
        }
    }
    regions_ = std::move(merged);
    region_ = 0; filtering_ = true; positioned_ = false;
    return true;
}

bool VariantSource::next(VariantRecord &rec) {
    if (!filtering_) return next_raw(rec);
    InflateStream *in = stream();
    for (;;) {
        if (region_ >= regions_.size()) return false;
        if (!positioned_) {                                           // entering regions_[region_]: jump if its first record lies ahead
            const Region &R = regions_[region_];
            const uint64_t v = index_->query_start(R.ref, R.beg0, R.end0);
            if (v == RegionIndex::NONE) { region_++; continue; }
            if (v > in->tell_virtual()) { in->seek_virtual(v); after_seek(); seeks_++; }
            positioned_ = true;
        }
        if (!next_raw(rec)) return false;
        for (;;) {                                                    // place the record against the current region
            const Region &R = regions_[region_];
            const int rank = contig_rank(rec);
            const bool past = rank > R.ref || (rank == R.ref && rec.pos - 1 >= R.end0);
            if (!past) {
                if (rank == R.ref && rec.end() > R.beg0) return true; // overlaps (rec.end() is 1-based inclusive = 0-based exclusive)
                break;                                                // before the region (or a contig the index does not know): keep reading
            }
            if (++region_ >= regions_.size()) return false;
            const Region &N = regions_[region_];
            const uint64_t v = index_->query_start(N.ref, N.beg0, N.end0);
            if (v == RegionIndex::NONE) { positioned_ = false; break; }
            if (v > in->tell_virtual()) { in->seek_virtual(v); after_seek(); seeks_++; positioned_ = true; break; }   // this record lies before the next region's first
            positioned_ = true;                                       // no jump: the same record may belong to the next region
        }
        if (!positioned_) continue;
    }
}

std::unique_ptr<VariantSource> open_variant_source(const std::string &path, bool seekable) {
    {   // a PLINK 1 .bed is recognised by its magic bytes 6c 1b, then the mode byte, a BGEN file by "bgen" at bytes 16-19
        // (not by the file name)
        uint8_t m[20] = { 0 };
        FILE *f = fopen(path.c_str(), "rb");
        if (!f) return nullptr;
        const size_t got = fread(m, 1, 20, f);
        fclose(f);
        if (got >= 3 && m[0] == 0x6c && m[1] == 0x1b) {
            auto src = std::make_unique<PlinkSource>();
            if (!src->open(path, m[2])) return nullptr;
            return src;
        }
        if (got == 20 && !memcmp(m + 16, "bgen", 4)) {
            auto src = std::make_unique<BgenSource>();
            if (!src->open(path)) return nullptr;
            return src;
        }
    }
    auto s = std::make_unique<InflateStream>();
    if (!s->open(path, seekable)) return nullptr;
    uint8_t magic[5] = { 0 };
    try {
        if (!s->peek(magic, 5)) return nullptr;
        if (!memcmp(magic, "BCF\2", 4)) {
            auto src = std::make_unique<BcfSource>(std::move(s));
            if (!src->read_header()) return nullptr;
            return src;
        }
        if (magic[0] != '#') return nullptr;
        auto src = std::make_unique<VcfTextSource>(std::move(s));
        if (!src->read_header()) return nullptr;
        return src;
    } catch (const InputError &) {
        return nullptr;
    }
}

}  // namespace nph
