// npc_api.cu -- C ABI of libnimpress_cuda.so (include/nimpress_cuda.h): contexts, the pinned
// double-buffered staging ring, stream/event plumbing and kernel launches.  No CPU fallback:
// every entry point either runs the CUDA kernels or fails.
#include <algorithm>
#include <array>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <chrono>
#include <cmath>
#include <string>
#include <unordered_map>
#include <vector>

#include "npc_fused5.cuh"
#include "npc_multi.cuh"
#include "npc_reduce.cuh"
#include "npc_dosage.cuh"
#include "npc_bed.cuh"
#include "npc_dose255.cuh"
#include "npc_dose32.cuh"
#include "npc_pl.cuh"
#include "npc_subset.cuh"
#include "npc_observed.cuh"

using namespace npc;

static thread_local std::string g_create_error;

// The layout of a context's genotype rows, set once from gt_width by npc_create*; npc_set_dosage_rows switches a ploidy-1,
// width-4 context between GT and DS.
enum class Layout { GT, DS, BED, DOSE255, DOSE32, PL };

// What the launcher knows of each layout, indexed by Layout.
struct LayoutInfo {
    const char *name;                       // in error messages
    int32_t sample_bits;                    // bits per sample of a row (0: ploidy x width bytes)
    int32_t header;                         // bytes of a row before its first sample
    bool diploid;                           // the context's ploidy must be 2
    bool one_alt;                           // a decoded row names REF (eaidx 0) or the one ALT (eaidx 1)
    bool real_tally;                        // tally: one count word a row (missing samples), the called dosages' block sums in d_ds_part
    int32_t mode;                           // npc_kernel_shape mode (0: the GT path's choice, launch_mode)
    int32_t threads, per_thread;            // accumulate pass of modes 4-7: threads per CTA, samples per thread
    int32_t chunk;                          // k_count_chunks: samples per 16-byte chunk (0: another tally)
};
static constexpr LayoutInfo LAYOUTS[] = {
    { "BCF GT rows", 0, 0, false, false, false, 0, 0, 0, 0 },
    { "FORMAT/DS rows", 0, 0, false, false, true, 0, 0, 0, 0 },
    { "PLINK .bed rows", 2, Bed::HEADER, true, true, false, 4, BED_THREADS, 8, Bed::PER16 },
    { "BGEN dosage rows", 16, Dose255::HEADER, true, true, false, 5, D255_THREADS, 8, Dose255::PER16 },
    { "BGEN dosage rows", 32, Dose32::HEADER, true, true, false, 6, D32_THREADS, 4, Dose32::PER16 },
    { "FORMAT/PL rows", 32, 0, true, true, true, 7, PL_THREADS, 4, 0 },
};
static const LayoutInfo &info(Layout l) { return LAYOUTS[(int)l]; }

// The layout of a gt_width; false for none.
static bool layout_of(int32_t gt_width, Layout &l) {
    switch (gt_width) {
    case 1: case 2: case 4: l = Layout::GT; return true;
    case NPC_GT_BED: l = Layout::BED; return true;
    case NPC_GT_DOSE255: l = Layout::DOSE255; return true;
    case NPC_GT_DOSE32: l = Layout::DOSE32; return true;
    case NPC_GT_PL: l = Layout::PL; return true;
    }
    return false;
}

static int64_t row_bytes(Layout l, int64_t n_samples, int32_t ploidy, int32_t width) {
    const LayoutInfo &L = info(l);
    return L.sample_bits ? L.header + (n_samples * L.sample_bits + 7) / 8 : n_samples * ploidy * width;
}

struct npc_ctx {
    int device = 0;
    int64_t n = 0;
    Layout layout = Layout::GT;
    int32_t ploidy = 2, width = 1;          // width: bytes of a GT allele value (1, 2 or 4); 0 in the other layouts
    int64_t max_rows = 0;
    int64_t staging_rows = 0;               // rows per pinned staging slot (<= max_rows)
    int32_t n_slots = 0;
    int64_t row_stride = 0;                 // of the context's rows (the staging ring's too, unless a subset context)
    int64_t stage_stride = 0;               // of the staging ring's rows: n_row samples
    // subset context (npc_create_subset, npc_subset.cuh): staged rows carry n_row samples, the context scores the n of them
    // that d_keep names; rows are compacted on the device after the H2D copy (into d_gt / the slab, from d_raw)
    bool sub = false;
    int64_t n_row = 0;
    std::vector<int32_t> keep;              // the kept sample indices until create_impl uploads them
    int32_t *d_keep = nullptr;              // n ascending sample indices, zero-padded to a multiple of SUB_PAD
    std::vector<uint8_t *> d_raw;           // per staging slot: its full rows on the device
    cudaStream_t own_stream = nullptr, stream = nullptr, copy_stream = nullptr;
    std::vector<uint8_t *> h_gt, d_gt;
    std::vector<cudaEvent_t> ev_h2d, ev_done;
    std::vector<int> slot_state;            // 0 free, 1 lent to the caller, 2 in flight
    int next_slot = 0;
    double *d_sums = nullptr, *d_out = nullptr;
    ull *d_nloci = nullptr, *d_counts = nullptr;
    npc_row *d_rows = nullptr;
    RowP *d_rowp = nullptr;
    npc_locus *d_log = nullptr;
    int64_t log_cap = 0, log_len = 0;
    Policy pol{};
    int64_t launches = 0;
    std::string err;
    // fused tile kernel (int8 diploid): launch shapes fixed per context
    struct TileCfg {
        bool ok = false;
        int Gs = 1, Gr = 1, K = 1, nc = 1, slab = 0, Sr = 3, Sc = 16, L = 15, A = 2, GD = 8;
        uint32_t smem = 0;
    };
    TileCfg fast;                           // default: sample slabs x row groups, tile-wise summation
    TileCfg fast_long;                      // default mode, long launches (fast_config): the best-filled split, however many row groups
    TileCfg exact_cfg;                      // npc_set_exact_order: 1-D grid, reference summation order
    // cohorts too wide for one resident pass (> ~1.2 M samples): tally + decide over all samples first, then the tile
    // kernel in "decided" mode over wide_slabs slabs of wide_n samples each (both shapes: default / exact order)
    TileCfg wide, wide_exact;
    int64_t wide_n = 0;
    int wide_slabs = 0;
    bool exact = false;
    int num_sms = 0;
    double *d_partials = nullptr;           // [fast.Gr - 1][n] partial sums of row groups 1..
    uint8_t *d_slab = nullptr;              // resident slab (npc_resident_reserve / npc_resident_adopt)
    bool slab_owned = false;
    int64_t slab_stride = 0;
    int64_t slab_rows = 0;
    cudaEvent_t ev_slab = nullptr;          // last scoring launch that read the slab
    ull *d_fcounts = nullptr;               // [2][max_rows] arrivals | nmiss | neff words of the fused kernel: a double buffer, each launch
                                            // clears the half the next one uses (pair kernel)
    int fcounts_half = 0;
    int64_t fcounts_dirty[2] = { 0, 0 };    // words of each half written since it was last cleared
    ull *d_trace = nullptr;                 // NPC_TRACE: 8 %globaltimer stamps of the last pair-kernel launch
    uint8_t *d_multi_scratch = nullptr;     // arena of npc_score_resident_multi's contraction
    size_t multi_scratch_bytes = 0;
    bool multi_attr_set = false;
    int64_t multi_contractions = 0;         // npc_score_resident_multi calls served by the tensor-core contraction
    double *d_ds_part = nullptr;            // FORMAT/DS and FORMAT/PL rows: [max_rows][n_blocks] block sums of the tally pass
    double *d_bed_tab = nullptr;            // PLINK .bed rows, per batch of BED_RB rows: the accumulate pass's value tables
    int32_t *d_bed_off = nullptr;           // ... and the slab row of every row it loads
    // cross-GPU combine (npc_reduce.cuh)
    cudaEvent_t ev_multi = nullptr;         // npc_score_resident_multi: orders its copy-stream work against the compute stream
    cudaEvent_t ev_reduce = nullptr;        // "this context's partial sums are final"
    ull *d_nloci_total = nullptr;           // combined nloci, next to d_out (the combined scores)
    double *d_bridge = nullptr;             // npc_reduce without peer access: [n_ctx - 1][n] copies of the other partials
    size_t bridge_bytes = 0;
    void *comm = nullptr;                   // ncclComm_t of npc_comm_init
    int comm_rank = 0, comm_world = 1;
    double *d_gather = nullptr;             // [world][n] all-gathered partial sums
    // per-sample observed counts (npc_observed.cuh): while `observed`, every scoring launch adds its OK rows' counts to d_obs
    bool observed = false;
    ull *d_obs = nullptr;
    uint8_t *d_obs_scratch = nullptr;       // npc_score_resident_multi_observed: a group's entries, weights and counts
    size_t obs_scratch_bytes = 0;
};

static npc::NcclApi g_nccl;

#define NPC_CUDA(ctx, call)                                                                       \
    do {                                                                                          \
        cudaError_t e_ = (call);                                                                  \
        if (e_ != cudaSuccess) {                                                                  \
            (ctx)->err = std::string(#call) + ": " + cudaGetErrorString(e_);                      \
            return e_ == cudaErrorMemoryAllocation ? NPC_ENOMEM : NPC_ECUDA;                      \
        }                                                                                         \
    } while (0)

static int fail(npc_ctx *ctx, int code, const char *msg) {
    ctx->err = msg;
    return code;
}

extern "C" int npc_version(void) { return 200; }

extern "C" int64_t npc_gt_row_bytes(int64_t n_samples, int32_t ploidy, int32_t gt_width) {
    Layout l = Layout::GT;
    layout_of(gt_width, l);
    return row_bytes(l, n_samples, ploidy, gt_width);
}

static int64_t ctx_row_bytes(const npc_ctx *c, int64_t n_samples) { return row_bytes(c->layout, n_samples, c->ploidy, c->width); }

extern "C" int npc_pl_weight_table(double *out, int32_t n) {
    static const double tab[PL_TN] = { NPC_PL_TABLE_VALUES };
    if (n < 0 || (n && !out)) return NPC_EINVAL;
    for (int32_t x = 0; x < n; x++) out[x] = x < PL_TN ? tab[x] : 0.0;
    return NPC_OK;
}

extern "C" int npc_warmup(int device) {
    if (cudaSetDevice(device) != cudaSuccess || cudaFree(nullptr) != cudaSuccess) { cudaGetLastError(); return NPC_ECUDA; }
    return NPC_OK;
}

extern "C" const char *npc_last_error(const npc_ctx *ctx) {
    return ctx ? ctx->err.c_str() : g_create_error.c_str();
}

extern "C" void npc_destroy(npc_ctx *ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    for (auto p : ctx->h_gt) if (p) cudaFreeHost(p);
    for (auto p : ctx->d_gt) if (p) cudaFree(p);
    for (auto p : ctx->d_raw) if (p) cudaFree(p);
    cudaFree(ctx->d_keep);
    for (auto e : ctx->ev_h2d) if (e) cudaEventDestroy(e);
    for (auto e : ctx->ev_done) if (e) cudaEventDestroy(e);
    cudaFree(ctx->d_sums); cudaFree(ctx->d_out); cudaFree(ctx->d_nloci); cudaFree(ctx->d_counts);
    cudaFree(ctx->d_rows); cudaFree(ctx->d_rowp); cudaFree(ctx->d_log); cudaFree(ctx->d_fcounts); cudaFree(ctx->d_trace); if (ctx->slab_owned) cudaFree(ctx->d_slab); cudaFree(ctx->d_partials); cudaFree(ctx->d_multi_scratch);
    if (ctx->ev_slab) cudaEventDestroy(ctx->ev_slab);
    if (ctx->ev_reduce) cudaEventDestroy(ctx->ev_reduce);
    if (ctx->ev_multi) cudaEventDestroy(ctx->ev_multi);
    cudaFree(ctx->d_nloci_total); cudaFree(ctx->d_bridge); cudaFree(ctx->d_gather); cudaFree(ctx->d_ds_part); cudaFree(ctx->d_bed_tab); cudaFree(ctx->d_bed_off);
    cudaFree(ctx->d_obs); cudaFree(ctx->d_obs_scratch);
    if (ctx->comm && g_nccl.lib) g_nccl.CommDestroy(ctx->comm);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    if (ctx->copy_stream) cudaStreamDestroy(ctx->copy_stream);
    delete ctx;
}

static int env_int(const char *name, int dflt) {
    const char *v = getenv(name);
    return v && *v ? atoi(v) : dflt;
}

// NCMAX of the k_fused_pair instance that runs nc warps of K chunks per thread: 24 or 28 for int8 GT at K = 1, else 16.
static int instance_warps(int width, int K, int nc) {
    if (width != 1 || K != 1) return 16;
    return nc > F5_NC_WIDE ? F5_NC_MAX : nc > 16 ? F5_NC_WIDE : 16;
}

static const void *tile_kernel(int K, bool exact, int width, int nc) {
    if (width == 2) {
        if (K == 1) return exact ? (const void *)k_fused_pair<1, true, 2> : (const void *)k_fused_pair<1, false, 2>;
        return exact ? (const void *)k_fused_pair<2, true, 2> : (const void *)k_fused_pair<2, false, 2>;
    }
    const int inst = instance_warps(width, K, nc);
    if (inst == F5_NC_MAX) return exact ? (const void *)k_fused_pair<1, true, 1, F5_NC_MAX> : (const void *)k_fused_pair<1, false, 1, F5_NC_MAX>;
    if (inst == F5_NC_WIDE) return exact ? (const void *)k_fused_pair<1, true, 1, F5_NC_WIDE> : (const void *)k_fused_pair<1, false, 1, F5_NC_WIDE>;
    if (K == 1) return exact ? (const void *)k_fused_pair<1, true> : (const void *)k_fused_pair<1, false>;
    return exact ? (const void *)k_fused_pair<2, true> : (const void *)k_fused_pair<2, false>;
}

// Consumer shape for a CTA that owns nch chunks (of 8 samples) of every row: K chunks per thread, nc warps.  One chunk
// per thread as long as the warps fit the SM's registers (int8 GT: up to 24 warps on the 72-register instance, cohorts
// up to ~909,000 samples per GPU), two (up to 16 warps) above that.
static bool tile_shape(int width, int64_t nch, int &K, int64_t &nc) {
    const int max1 = width == 1 ? F5_NC_MAX : 16;
    K = env_int("NPC_TILE_K", 0);
    if (K != 1 && K != 2) K = nch <= 32 * max1 ? 1 : 2;
    nc = (nch + 32 * K - 1) / (32 * K);
    return nc <= (K == 1 ? max1 : 16);                // else: cohort too wide for one resident pass
}

// The sample axis of C chunks under `gr` row groups: gs slabs (one CTA each, gs * gr CTAs at most one per SM) of nch chunks,
// and the consumer shape that holds a slab.  False when no such split exists.
static bool slab_split(const npc_ctx *c, int64_t C, int gr, int &gs, int64_t &nch, int &K, int64_t &nc) {
    gs = (int)std::min<int64_t>(c->num_sms / gr, std::max<int64_t>(1, C / 32));
    if (gs < 1) return false;
    nch = (C + gs - 1) / gs;
    return tile_shape(c->width, nch, K, nc);
}

// Launch shape of the tile kernel for `gr` row groups: Gs sample slabs (one CTA each), a raw ring of Sr
// stages (one chunk set of 4 rows each; ~110 KB of loads in flight per SM), the rest of shared memory as
// index-ring slots, lag L = Sc - 1 tiles, A decider warps deciding GD tiles per pass.
static bool tile_config(const npc_ctx *c, int gr, int max_smem, npc_ctx::TileCfg &t, int64_t n_samples = -1) {
    int gs, K; int64_t nch, nc;
    if (!slab_split(c, ((n_samples < 0 ? c->n : n_samples) + 7) / 8, gr, gs, nch, K, nc)) return false;
    const int W = c->width;                            // 1 or 2 (int16 GT)
    const int slab = (int)(nc * 32 * K * 16 * W);
    int Sr = env_int("NPC_TILE_SR", 0), Sc = env_int("NPC_TILE_SC", 0), L = env_int("NPC_TILE_L", 0), A = env_int("NPC_TILE_A", 2);
    int GD = env_int("NPC_TILE_GD", 0);
    const int stage = F5_R * slab / K;                 // bytes of a raw stage
    auto smem_of = [&](int sr, int sc) { return (int)Fused5Smem::make(sr, sc, slab, (int)nc, K, W).total; };
    // K = 2: one raw stage per chunk set, ~110 KB of them, at least 3
    // (a quarter stage of slack: 19-20 warps, 38-40 KB stages, measured 0.93 / 0.965 on three stages against 0.91 / 0.94 on two)
    if (Sr <= 0) Sr = std::max(K == 2 ? 3 : 2, std::min(8, (112 * 1024 + stage / 4) / stage));
    if (Sc <= 0) {
        Sc = 32;
        while (Sc > 2 && smem_of(Sr, Sc) > max_smem) Sc--;
    }
    while (Sr > (K == 2 ? 3 : 2) && smem_of(Sr, Sc) > max_smem) Sr--;
    // Deciders work on groups of GD tiles and the first tile of a group waits for the last: the lag must cover a
    // whole group plus the grid-wide round trip of the tally word (~6 us under load; a tile streams in
    // 4 * slab bytes / 42 GB/s per SM).  8 tiles per pass where the rings leave that much lag, else 4.
    if (GD != 4 && GD != 8) {
        const double tile_us = 4.0 * slab / 41.9e3;
        GD = Sc - 1 >= 8 + 1 + (int)std::ceil(6.0 / tile_us) ? 8 : 4;
    }
    if (smem_of(Sr, Sc) > max_smem || Sc < GD + 2) return false;
    if (L <= GD || L > Sc - 1) L = Sc - 1;
    t.Gs = gs; t.Gr = gr; t.K = K; t.nc = (int)nc; t.slab = slab; t.Sr = Sr; t.Sc = Sc; t.L = L; t.GD = GD;
    t.A = std::max(1, std::min(2, A));
    t.smem = (uint32_t)smem_of(Sr, Sc);
    t.ok = true;
    return true;
}

// Choose the grids of the tile kernel.  Default mode: Gs sample slabs x Gr row groups -- a cohort too
// small to give every SM ~14 consumer warps from the sample axis alone (< ~500k samples) also splits
// the rows into contiguous groups whose partial sums are added in group order afterwards.  Exact
// order: Gr = 1.  NPC_TILE_{K,SR,SC,L,A,GR} override for tuning; NPC_FUSED=0 forces the two-kernel path.
// Pure host arithmetic (no CUDA call): fills c->fast, fast_long, exact_cfg, wide, wide_exact from n, width, ploidy, the SM
// count and the shared memory a CTA may take.  npc_plan_shape exposes it so that the choice can be tested for every
// cohort size without a device (tests/test_shape_plan.py).
static void plan_shapes(npc_ctx *c, int num_sms, int max_smem) {
    c->fast.ok = c->fast_long.ok = c->exact_cfg.ok = c->wide.ok = c->wide_exact.ok = false;
    if ((c->width != 1 && c->width != 2) || c->ploidy != 2 || c->n == 0 || c->n >= (1ll << 27) || env_int("NPC_FUSED", 1) == 0) return;
    c->num_sms = num_sms;
    const int64_t C = (c->n + 7) / 8;
    const int force_gr = env_int("NPC_TILE_GR", 0);
    // candidates in the order of preference: the score of round 1 (SMs used x warps kept busy), a larger number of row
    // groups only when it is worth 8 %; the first candidate whose rings fit shared memory is taken (the fuzz of round 2
    // found cohorts whose best-scoring split did not fit and silently lost the fused path)
    std::vector<std::pair<double, int>> cand;
    for (int gr = 1; gr <= 16; gr++) {
        int gs, k; int64_t nch, nc;
        if (!slab_split(c, C, gr, gs, nch, k, nc) || (force_gr && gr != force_gr)) continue;
        const double score = (double)gs * gr * std::min<int64_t>(nc * k, 14) * ((double)nch / (double)(nc * 32 * k));
        cand.emplace_back(score, gr);
    }
    {
        // round 1's rule: walk gr upwards, move on only for an 8 % better score
        std::vector<int> order;
        double best = -1.0;
        for (const auto &sc : cand) if (sc.first > best * 1.08) { best = sc.first; order.insert(order.begin(), sc.second); }
        for (const auto &sc : cand) if (std::find(order.begin(), order.end(), sc.second) == order.end()) order.push_back(sc.second);
        for (int gr : order) if (tile_config(c, gr, max_smem, c->fast)) break;
    }
    // Long launches take the split with the best-filled warps even for a few per cent (bench shard, 500,000 samples: 74 slabs x
    // 2 row groups on 27 warps fill 97.8 % of the lanes, 148 x 1 on 14 warps 94.3 %: 0.938 against 0.920 of the
    // roofline); short ones keep round 1's rule -- more row groups leave a CTA fewer tiles to hide ramp-up and
    // drain behind, and k_add_partials grows with them.
    if (c->fast.ok && !force_gr) {
        double have = 0.0, best = 0.0; int best_gr = 0;
        for (const auto &sc : cand) { if (sc.second == c->fast.Gr) have = sc.first; if (sc.first > best) { best = sc.first; best_gr = sc.second; } }
        if (best_gr && best_gr != c->fast.Gr && best > have * 1.02) tile_config(c, best_gr, max_smem, c->fast_long);
    }
    tile_config(c, 1, max_smem, c->exact_cfg);
    if (!c->fast.ok && c->width == 1) {
        // no shape holds a whole row's share in one CTA: the fewest equal slabs (multiples of 1024 samples) the tile kernel can hold
        for (int S = 2; S <= 64 && !c->wide.ok; S++) {
            const int64_t ns = ((c->n + S - 1) / S + 1023) / 1024 * 1024;
            if (tile_config(c, 1, max_smem, c->wide, ns) && tile_config(c, 1, max_smem, c->wide_exact, ns)) { c->wide_n = ns; c->wide_slabs = (int)((c->n + ns - 1) / ns); }
            else c->wide.ok = c->wide_exact.ok = false;
        }
        // ONE decider warp: in decided mode the local "tile counted" barrier is the deciders' only gate, and a warp that
        // takes every A-th group of 8 tiles would wait on a ring slot's barrier 8*A tiles apart -- with 8*A > Sc it
        // skips a phase of that slot and the parity test passes a whole ring turn early (in the normal mode the poll
        // of the grid-wide tally word is the real gate, so the early pass is harmless there)
        c->wide.A = c->wide_exact.A = 1;
    }
}

static int fused_configure(npc_ctx *c, const cudaDeviceProp &prop) {
    const int max_smem = (int)prop.sharedMemPerBlockOptin;
    plan_shapes(c, prop.multiProcessorCount, max_smem);
    if (!c->fast.ok && !c->exact_cfg.ok && !c->wide.ok) return NPC_OK;
    const std::pair<const npc_ctx::TileCfg *, bool> cfgs[] = {
        { &c->fast, false }, { &c->fast_long, false }, { &c->exact_cfg, true }, { &c->wide, false }, { &c->wide_exact, true } };
    for (const auto &[t, exact] : cfgs) {
        if (!t->ok) continue;
        // the device's maximum, not this shape's need: the attribute belongs to the kernel function, which other contexts
        // of the process (and this context's other shapes) launch with other sizes
        cudaError_t e = cudaFuncSetAttribute(tile_kernel(t->K, exact, c->width, t->nc), cudaFuncAttributeMaxDynamicSharedMemorySize, max_smem);
        if (e != cudaSuccess) { c->err = std::string("cudaFuncSetAttribute: ") + cudaGetErrorString(e); return NPC_ECUDA; }
    }
    const size_t words = 2 * (size_t)std::max<int64_t>(c->max_rows, 1);
    NPC_CUDA(c, cudaMalloc(&c->d_fcounts, words * sizeof(ull)));
    NPC_CUDA(c, cudaMemset(c->d_fcounts, 0, words * sizeof(ull)));
    if (env_int("NPC_TRACE", 0)) { NPC_CUDA(c, cudaMalloc(&c->d_trace, 8 * sizeof(ull))); NPC_CUDA(c, cudaMemset(c->d_trace, 0, 8 * sizeof(ull))); }
    const int max_gr = std::max(c->fast.ok ? c->fast.Gr : 1, c->fast_long.ok ? c->fast_long.Gr : 1);
    if (max_gr > 1) NPC_CUDA(c, cudaMalloc(&c->d_partials, (size_t)(max_gr - 1) * (size_t)c->n * sizeof(double)));
    c->exact = env_int("NPC_EXACT", 0) != 0;
    return NPC_OK;
}

static int create_impl(npc_ctx *c) {
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(c, NPC_ECUDA, "no CUDA device: libnimpress_cuda has no CPU fallback");
    if (c->device < 0 || c->device >= ndev) return fail(c, NPC_EINVAL, "device index out of range");
    NPC_CUDA(c, cudaSetDevice(c->device));
    cudaDeviceProp prop;
    NPC_CUDA(c, cudaGetDeviceProperties(&prop, c->device));
    if (prop.major != 10) return fail(c, NPC_ECUDA, "device is not sm_100 (B200): kernels are built for sm_100a only");
    NPC_CUDA(c, cudaStreamCreateWithFlags(&c->own_stream, cudaStreamNonBlocking));
    NPC_CUDA(c, cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking));
    c->stream = c->own_stream;
    const int64_t n1 = std::max<int64_t>(c->n, 1), r1 = std::max<int64_t>(c->max_rows, 1);
    NPC_CUDA(c, cudaMalloc(&c->d_sums, n1 * sizeof(double)));
    NPC_CUDA(c, cudaMalloc(&c->d_out, n1 * sizeof(double)));
    NPC_CUDA(c, cudaMalloc(&c->d_nloci, sizeof(ull)));
    NPC_CUDA(c, cudaMalloc(&c->d_counts, r1 * 2 * sizeof(ull)));
    NPC_CUDA(c, cudaMalloc(&c->d_rows, r1 * sizeof(npc_row)));
    NPC_CUDA(c, cudaMalloc(&c->d_rowp, r1 * sizeof(RowP)));
    c->log_cap = std::max<int64_t>(r1, 1024);
    NPC_CUDA(c, cudaMalloc(&c->d_log, c->log_cap * sizeof(npc_locus)));
    c->row_stride = ((ctx_row_bytes(c, c->n) + 127) / 128) * 128;
    if (c->row_stride == 0) c->row_stride = 128;
    c->stage_stride = c->row_stride;
    if (c->sub) {
        c->stage_stride = std::max<int64_t>(128, ((ctx_row_bytes(c, c->n_row) + 127) / 128) * 128);
        c->keep.resize((size_t)((c->n + SUB_PAD - 1) / SUB_PAD * SUB_PAD), 0);
        NPC_CUDA(c, cudaMalloc(&c->d_keep, c->keep.size() * sizeof(int32_t)));
        NPC_CUDA(c, cudaMemcpy(c->d_keep, c->keep.data(), c->keep.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
        std::vector<int32_t>().swap(c->keep);
    }
    c->h_gt.assign(c->n_slots, nullptr); c->d_gt.assign(c->n_slots, nullptr); c->d_raw.assign(c->n_slots, nullptr);
    c->ev_h2d.assign(c->n_slots, nullptr); c->ev_done.assign(c->n_slots, nullptr);
    c->slot_state.assign(c->n_slots, 0);
    for (int s = 0; s < c->n_slots; s++) {
        // pinned host slots only: the device copy of a slot is allocated when npc_score_block first needs it
        // (the resident path uploads straight into the slab)
        const size_t bytes = (size_t)c->stage_stride * (size_t)std::max<int64_t>(c->staging_rows, 1);
        // (write-combined memory was measured no faster: the H2D copy runs at the PCIe rate either way)
        NPC_CUDA(c, cudaHostAlloc((void **)&c->h_gt[s], bytes, cudaHostAllocDefault));
        NPC_CUDA(c, cudaEventCreateWithFlags(&c->ev_h2d[s], cudaEventDisableTiming));
        NPC_CUDA(c, cudaEventCreateWithFlags(&c->ev_done[s], cudaEventDisableTiming));
    }
    NPC_CUDA(c, cudaMemsetAsync(c->d_sums, 0, n1 * sizeof(double), c->stream));
    NPC_CUDA(c, cudaMemsetAsync(c->d_nloci, 0, sizeof(ull), c->stream));
    NPC_CUDA(c, cudaStreamSynchronize(c->stream));
    return fused_configure(c, prop);
}

extern "C" int npc_create(npc_ctx **out, int device, int64_t n_samples, int32_t ploidy, int32_t gt_width,
                          int64_t max_rows_per_block, int32_t n_slots) {
    return npc_create2(out, device, n_samples, ploidy, gt_width, max_rows_per_block, n_slots, max_rows_per_block);
}

// keep == nullptr: a context over n_samples samples (npc_create2); else over keep[0..n_samples) of rows of n_row samples
static int create_ctx(npc_ctx **out, int device, int64_t n_row, const int64_t *keep, int64_t n_samples, int32_t ploidy,
                      int32_t gt_width, int64_t max_rows_per_block, int32_t n_slots, int64_t staging_rows) {
    if (!out) return NPC_EINVAL;
    *out = nullptr;
    Layout layout = Layout::GT;
    if (n_samples < 0 || ploidy < 1 || ploidy > 64 || !layout_of(gt_width, layout) || (info(layout).diploid && ploidy != 2) ||
        max_rows_per_block < 1 || n_slots < 0 || n_slots == 1 || staging_rows < 1 || staging_rows > max_rows_per_block) {
        g_create_error = "npc_create: invalid argument";
        return NPC_EINVAL;
    }
    npc_ctx *c = new npc_ctx();
    c->n_row = n_row;
    if (keep) {
        c->sub = true;
        c->keep.resize((size_t)n_samples);
        for (int64_t i = 0; i < n_samples; i++) c->keep[(size_t)i] = (int32_t)keep[i];
    }
    c->device = device; c->n = n_samples; c->ploidy = ploidy; c->layout = layout; c->width = layout == Layout::GT ? gt_width : 0;
    c->max_rows = max_rows_per_block; c->n_slots = n_slots; c->staging_rows = staging_rows;
    c->pol.imp_locus = NPC_LOCUS_PS; c->pol.imp_missing = NPC_MISSING_HOMREF; c->pol.imp_sample = NPC_SAMPLE_INT_PS;
    c->pol.mincs = 100; c->pol.maxmis = 0.05; c->pol.n_total = n_samples;      // defaults of main (:670-687)
    int rc = create_impl(c);
    if (rc != NPC_OK) {
        g_create_error = c->err;
        npc_destroy(c);
        return rc;
    }
    *out = c;
    return NPC_OK;
}

extern "C" int npc_create2(npc_ctx **out, int device, int64_t n_samples, int32_t ploidy, int32_t gt_width,
                           int64_t max_rows_per_block, int32_t n_slots, int64_t staging_rows) {
    return create_ctx(out, device, n_samples, nullptr, n_samples, ploidy, gt_width, max_rows_per_block, n_slots, staging_rows);
}

extern "C" int npc_create_subset(npc_ctx **out, int device, int64_t n_row_samples, const int64_t *keep, int64_t n_keep,
                                 int32_t ploidy, int32_t gt_width, int64_t max_rows_per_block, int32_t n_slots,
                                 int64_t staging_rows) {
    if (!out) return NPC_EINVAL;
    *out = nullptr;
    // int32 indices on the device; ascending and distinct, so that a compact row keeps the file's sample order
    bool ok = keep && n_keep >= 1 && n_row_samples >= n_keep && n_row_samples <= INT32_MAX;
    for (int64_t i = 0; ok && i < n_keep; i++) ok = keep[i] >= 0 && keep[i] < n_row_samples && (i == 0 || keep[i] > keep[i - 1]);
    if (!ok) {
        g_create_error = "npc_create_subset: keep must hold 1 .. n_row_samples ascending, distinct indices below n_row_samples";
        return NPC_EINVAL;
    }
    return create_ctx(out, device, n_row_samples, keep, n_keep, ploidy, gt_width, max_rows_per_block, n_slots, staging_rows);
}

extern "C" int npc_set_stream(npc_ctx *ctx, void *cuda_stream) {
    if (!ctx) return NPC_EINVAL;
    ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    return NPC_OK;
}

extern "C" int npc_set_policy(npc_ctx *ctx, const npc_policy *p) {
    if (!ctx || !p) return NPC_EINVAL;
    if (p->imp_locus < 0 || p->imp_locus > 3 || p->imp_missing < 0 || p->imp_missing > 1 || p->imp_sample < 0 ||
        p->imp_sample > 4)
        return fail(ctx, NPC_EINVAL, "npc_set_policy: unknown imputation method");
    ctx->pol.imp_locus = p->imp_locus; ctx->pol.imp_missing = p->imp_missing; ctx->pol.imp_sample = p->imp_sample;
    ctx->pol.mincs = p->mincs; ctx->pol.maxmis = p->maxmis;
    return NPC_OK;
}

extern "C" int npc_set_cohort_size(npc_ctx *ctx, int64_t n_total) {
    if (!ctx || n_total < 0) return NPC_EINVAL;
    ctx->pol.n_total = n_total;
    return NPC_OK;
}

extern "C" int npc_reset(npc_ctx *ctx) {
    if (!ctx) return NPC_EINVAL;
    NPC_CUDA(ctx, cudaSetDevice(ctx->device));
    NPC_CUDA(ctx, cudaMemsetAsync(ctx->d_sums, 0, std::max<int64_t>(ctx->n, 1) * sizeof(double), ctx->stream));
    NPC_CUDA(ctx, cudaMemsetAsync(ctx->d_nloci, 0, sizeof(ull), ctx->stream));
    if (ctx->d_obs) NPC_CUDA(ctx, cudaMemsetAsync(ctx->d_obs, 0, std::max<int64_t>(ctx->n, 1) * sizeof(ull), ctx->stream));
    ctx->log_len = 0;
    return NPC_OK;
}

extern "C" int64_t npc_launch_count(const npc_ctx *ctx) { return ctx ? ctx->launches : 0; }
extern "C" int64_t npc_multi_contractions(const npc_ctx *ctx) { return ctx ? ctx->multi_contractions : 0; }

extern "C" int npc_trace(npc_ctx *ctx, uint64_t out[8]) {
    if (!ctx || !out) return NPC_EINVAL;
    if (!ctx->d_trace) return fail(ctx, NPC_ESTATE, "npc_trace: set NPC_TRACE=1 before npc_create");
    NPC_CUDA(ctx, cudaSetDevice(ctx->device));
    NPC_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    NPC_CUDA(ctx, cudaMemcpy(out, ctx->d_trace, 8 * sizeof(ull), cudaMemcpyDeviceToHost));
    return NPC_OK;
}

// A launch of at least this many genotype bytes counts as long (fast_long).  Measured crossover (500,000 samples, 148 x 1
// against 74 x 2): the extra k_add_partials launch and the shorter per-CTA tile runs cost more than the fuller warps gain
// below ~1.5 GB.  When the short split has row groups of its own the partial sums are added anyway and the better-filled
// split wins from ~200 MB on (250,000 samples, 74 x 2 against 49 x 3: +3.5 % at 256 MB, +5.5 % at 1 GB).
// NPC_TILE_LONG_MB overrides.
static const npc_ctx::TileCfg &fast_config(const npc_ctx *c, int64_t n_rows) {
    if (!c->fast_long.ok) return c->fast;
    const int64_t long_bytes = (int64_t)env_int("NPC_TILE_LONG_MB", c->fast.Gr > 1 ? 192 : 1536) << 20;
    return n_rows * c->row_stride >= long_bytes ? c->fast_long : c->fast;
}

// What a launch of n_rows rows runs (launch_block), and what npc_kernel_shape2 and npc_plan_shape report: 0 the generic
// tally, decide, accumulate sequence, 1 the tile kernel in exact order, 2 in default order, 3 tally + decide, then the tile
// kernel in decided mode over the wide slabs (only where no resident shape fits), 4 the sequence on PLINK .bed rows, 5 the
// sequence on fixed-point dosage rows (BGEN), 6 the sequence on 32-bit fixed-point dosage rows (BGEN at any bit depth),
// 7 the sequence on FORMAT/PL rows.
// t: the tile kernel's shape in modes 1-3.
static int launch_mode(const npc_ctx *c, bool exact, int64_t n_rows, const npc_ctx::TileCfg *&t) {
    t = nullptr;
    if (const int mode = info(c->layout).mode) return mode;
    t = exact ? &c->exact_cfg : &fast_config(c, n_rows);
    if (t->ok) return exact ? 1 : 2;
    t = exact ? &c->wide_exact : &c->wide;
    return t->ok ? 3 : 0;
}

extern "C" int npc_kernel_shape2(const npc_ctx *ctx, int64_t n_rows, int32_t shape[8]) {
    if (!ctx || !shape || n_rows < 0) return NPC_EINVAL;
    memset(shape, 0, 8 * sizeof(int32_t));
    const npc_ctx::TileCfg *t;
    shape[0] = launch_mode(ctx, ctx->exact, n_rows, t);
    if (shape[0] >= 4) {
        const LayoutInfo &L = info(ctx->layout);
        const int64_t per_cta = (int64_t)L.threads * L.per_thread;
        shape[1] = (int32_t)((ctx->n + per_cta - 1) / per_cta); shape[2] = L.threads / 32; shape[3] = L.per_thread;
        if (ctx->layout == Layout::BED) shape[4] = ctx->exact ? 1 : 4;
    } else if (shape[0]) {
        shape[1] = t->Gs * 1000 + t->Gr; shape[2] = t->nc; shape[3] = t->K;
        shape[4] = F5_R; shape[5] = t->Sr * 1000 + t->Sc; shape[6] = t->L * 100 + t->GD * 10 + t->A; shape[7] = (int32_t)t->smem;
    }
    return NPC_OK;
}
extern "C" int npc_kernel_shape(const npc_ctx *ctx, int32_t shape[8]) { return npc_kernel_shape2(ctx, 0, shape); }

extern "C" int npc_plan_shape(int64_t n_samples, int32_t gt_width, int32_t num_sms, int32_t max_smem, int64_t n_rows, int32_t exact,
                              int32_t plan[16]) {
    if (!plan || n_samples < 0 || num_sms < 1 || max_smem < 1 || n_rows < 0) return NPC_EINVAL;
    npc_ctx *c = new npc_ctx;
    c->n = n_samples; c->ploidy = 2; c->width = gt_width;
    c->row_stride = ((npc_gt_row_bytes(c->n, c->ploidy, c->width) + 127) / 128) * 128;
    plan_shapes(c, num_sms, max_smem);
    const npc_ctx::TileCfg *t;
    const int mode = launch_mode(c, exact != 0, n_rows, t);
    memset(plan, 0, 16 * sizeof(int32_t));
    if (mode) {
        const int32_t v[16] = { mode, t->Gs, t->Gr, t->K, t->nc, t->slab, t->Sr, t->Sc, t->L, t->A, t->GD, (int32_t)t->smem,
                                (t->nc + 2 + t->A) * 32, instance_warps(c->width, t->K, t->nc),
                                mode == 3 ? c->wide_slabs : 1, mode == 3 ? (int32_t)c->wide_n : (int32_t)std::min<int64_t>(c->n, INT32_MAX) };
        memcpy(plan, v, sizeof(v));
    }
    delete c;
    return NPC_OK;
}

extern "C" int npc_set_dosage_rows(npc_ctx *ctx, int32_t on) {
    if (!ctx) return NPC_EINVAL;
    const bool can = ctx->width == 4 && ctx->ploidy == 1;                   // a GT or DS context
    if (on && !can)
        return fail(ctx, NPC_EINVAL, "npc_set_dosage_rows: create the context with ploidy 1 and gt_width 4 (one fp32 DS value per sample)");
    if (can) ctx->layout = on ? Layout::DS : Layout::GT;
    return NPC_OK;
}

extern "C" int npc_set_exact_order(npc_ctx *ctx, int32_t on) {
    if (!ctx) return NPC_EINVAL;
    ctx->exact = on != 0;
    return NPC_OK;
}

// ---- internals ---------------------------------------------------------------------------

static int ensure_log(npc_ctx *c, int64_t extra) {
    if (c->log_len + extra <= c->log_cap) return NPC_OK;
    int64_t cap = std::max(c->log_cap * 2, c->log_len + extra);
    npc_locus *nl = nullptr;
    NPC_CUDA(c, cudaMalloc(&nl, cap * sizeof(npc_locus)));
    NPC_CUDA(c, cudaMemcpyAsync(nl, c->d_log, c->log_len * sizeof(npc_locus), cudaMemcpyDeviceToDevice, c->stream));
    NPC_CUDA(c, cudaStreamSynchronize(c->stream));
    cudaFree(c->d_log);
    c->d_log = nl; c->log_cap = cap;
    return NPC_OK;
}

static int check_block(npc_ctx *c, const void *gt, int64_t row_stride, int64_t n_gt_rows, const npc_row *rows,
                       int64_t n_rows) {
    if (!c) return NPC_EINVAL;
    if (n_rows < 0 || n_gt_rows < 0 || n_rows > c->max_rows || n_gt_rows > c->max_rows)
        return fail(c, NPC_EINVAL, "block larger than max_rows_per_block");
    if (n_rows && !rows) return fail(c, NPC_EINVAL, "rows is NULL");
    if (n_gt_rows && (!gt || ((uintptr_t)gt & 15) || (row_stride & 15) || row_stride < ctx_row_bytes(c, c->n)))
        return fail(c, NPC_EINVAL, "genotype slab must be 16-byte aligned with row_stride % 16 == 0 and >= the bytes of a row");
    return NPC_OK;
}

// .bed, BGEN and PL rows carry one ALT: a decoded row names REF (0) or that ALT (1).  Checked where the rows are on the host.
static int check_one_alt(npc_ctx *c, const npc_row *rows, int64_t n_rows, int on_device) {
    if (!info(c->layout).one_alt || on_device) return NPC_OK;
    for (int64_t i = 0; i < n_rows; i++)
        if (rows[i].kind == NPC_KIND_GT && rows[i].gt_row >= 0 && rows[i].eaidx != 0 && rows[i].eaidx != 1)
            return fail(c, NPC_EINVAL, (std::string(info(c->layout).name) +
                                        ": the effect allele of a genotype row is REF (eaidx 0) or the one ALT (eaidx 1)").c_str());
    return NPC_OK;
}

// rows -> d_rows on the compute stream.  A pageable source is staged by the runtime before the
// call returns, so the caller may reuse `rows` immediately.
static int upload_rows(npc_ctx *c, const npc_row *rows, int64_t n_rows, int on_device, const npc_row **d_rows) {
    if (on_device) { *d_rows = rows; return NPC_OK; }
    NPC_CUDA(c, cudaMemcpyAsync(c->d_rows, rows, n_rows * sizeof(npc_row), cudaMemcpyHostToDevice, c->stream));
    *d_rows = c->d_rows;
    return NPC_OK;
}

// Blocks per row of the tally kernels (256 threads, rows of `units`): cheap to run but not free to schedule, so up to 64 units
// per thread (5.8 TB/s on an 8 GB slab against 4.6 TB/s at 4), fewer only to keep ~4096 blocks, at least min_units a block.
static unsigned tally_grid_y(int64_t units, int64_t n_rows, int64_t min_units) {
    const int64_t s_min = (units + 16383) / 16384, s_max = (units + min_units - 1) / min_units, want = (4096 + n_rows - 1) / n_rows;
    return (unsigned)std::min<int64_t>(std::max<int64_t>(std::min(std::max(want, s_min), s_max), 1), 65535);
}

// Tallies of n_rows rows into counts: two words a row; for FORMAT/DS and FORMAT/PL rows the missing count alone, the
// block sums of the called dosages go to d_ds_part.
static int launch_tally(npc_ctx *c, const uint8_t *gt, int64_t row_stride, const npc_row *d_rows, int64_t n_rows,
                        ull *counts) {
    const LayoutInfo &L = info(c->layout);
    NPC_CUDA(c, cudaMemsetAsync(counts, 0, n_rows * (L.real_tally ? 1 : 2) * sizeof(ull), c->stream));
    if (n_rows == 0 || c->n == 0) return NPC_OK;
    const int64_t n_blocks = (c->n + DS_BLOCK - 1) / DS_BLOCK;
    if (L.real_tally && !c->d_ds_part)
        NPC_CUDA(c, cudaMalloc(&c->d_ds_part, (size_t)std::max<int64_t>(c->max_rows, 1) * (size_t)n_blocks * sizeof(double)));
    void (*chunks)(const uint8_t *, int64_t, const npc_row *, int64_t, ull *) = nullptr;
    switch (c->layout) {
    case Layout::GT:
        if (c->width == 1 && c->ploidy == 2) {
            const unsigned slabs = tally_grid_y((c->n + 7) / 8, n_rows, 1024);               // units: chunks of 8 samples
            k_count_i8x2<<<dim3((unsigned)n_rows, slabs), 256, 0, c->stream>>>(gt, row_stride, d_rows, c->n, counts);
        } else {
            dim3 grid((unsigned)n_rows, tally_grid_y(c->n, n_rows, 2048));                    // units: samples
            if (c->width == 1) k_count_generic<int8_t><<<grid, 256, 0, c->stream>>>(gt, row_stride, d_rows, c->n, c->ploidy, counts);
            else if (c->width == 2) k_count_generic<int16_t><<<grid, 256, 0, c->stream>>>(gt, row_stride, d_rows, c->n, c->ploidy, counts);
            else k_count_generic<int32_t><<<grid, 256, 0, c->stream>>>(gt, row_stride, d_rows, c->n, c->ploidy, counts);
        }
        c->launches++;
        break;
    case Layout::DS:
        for (int64_t r0 = 0; r0 < n_rows; r0 += 65535) {                                        // grid y: at most 65,535 rows
            const int64_t nr = std::min<int64_t>(65535, n_rows - r0);
            k_count_ds<<<dim3((unsigned)((n_blocks + 7) / 8), (unsigned)nr), 256, 0, c->stream>>>(gt, row_stride, d_rows + r0, c->n, n_blocks,
                                                                                               c->d_ds_part + r0 * n_blocks, counts + r0);
            c->launches++;
        }
        break;
    case Layout::PL: {
        // a CTA loads T once and takes every gridDim.y-th row: about 4096 CTAs in all
        const unsigned gx = (unsigned)((n_blocks + 7) / 8);
        const unsigned gy = (unsigned)std::min<int64_t>(n_rows, std::max<int64_t>(1, (4096 + gx - 1) / gx));
        k_count_pl<<<dim3(gx, gy), 256, 0, c->stream>>>(gt, row_stride, d_rows, n_rows, c->n, n_blocks, c->d_ds_part, counts);
        c->launches++;
        break;
    }
    case Layout::BED: chunks = k_count_chunks<Bed>; break;
    case Layout::DOSE255: chunks = k_count_chunks<Dose255>; break;
    case Layout::DOSE32: chunks = k_count_chunks<Dose32>; break;
    }
    if (chunks) {
        const unsigned slabs = tally_grid_y((c->n + L.chunk - 1) / L.chunk, n_rows, 1024);     // units: chunks
        chunks<<<dim3((unsigned)n_rows, slabs), 256, 0, c->stream>>>(gt, row_stride, d_rows, c->n, counts);
        c->launches++;
    }
    NPC_CUDA(c, cudaGetLastError());
    return NPC_OK;
}

// The decision for each of n_rows tallied rows: its contributions to d_rowp, its record appended to the locus log.  gt: the
// rows' slab, whose row headers hold the denominators of 32-bit dosage rows
static int launch_decide(npc_ctx *c, const uint8_t *gt, int64_t row_stride, const npc_row *d_rows, int64_t n_rows, const ull *counts) {
    if (n_rows == 0) return NPC_OK;
    int rc = ensure_log(c, n_rows);
    if (rc) return rc;
    auto decide = k_decide<CountTally>;
    switch (c->layout) {
    case Layout::GT: case Layout::BED: break;
    case Layout::DS: decide = k_decide<DsTally>; break;
    case Layout::DOSE255: decide = k_decide<Dose255::Tally>; break;
    case Layout::DOSE32: decide = k_decide<Dose32::Tally>; break;
    case Layout::PL: decide = k_decide<PlTally>; break;
    }
    const TallyIn in = { gt, row_stride, counts, c->d_ds_part, (c->n + DS_BLOCK - 1) / DS_BLOCK };
    decide<<<(unsigned)((n_rows + 127) / 128), 128, 0, c->stream>>>(in, d_rows, n_rows, c->pol, c->n, c->d_rowp, c->d_log + c->log_len,
                                                                  c->d_nloci);
    c->launches++;
    NPC_CUDA(c, cudaGetLastError());
    c->log_len += n_rows;
    return NPC_OK;
}

// The decided rows' contributions (d_rowp) added to the sums
static int launch_accum(npc_ctx *c, const uint8_t *gt, int64_t row_stride, int64_t n_rows) {
    if (n_rows == 0 || c->n == 0) return NPC_OK;
    const LayoutInfo &L = info(c->layout);
    const unsigned grid = L.threads ? (unsigned)((c->n + L.threads * L.per_thread - 1) / (L.threads * L.per_thread)) : 0;   // modes 4-7
    switch (c->layout) {
    case Layout::GT:
        if (c->width == 1 && c->ploidy == 2) {
            const int64_t nchunks = (c->n + 7) / 8;
            k_accum_i8x2<64, 8><<<(unsigned)((nchunks + 255) / 256), 256, 0, c->stream>>>(gt, row_stride, c->d_rowp, n_rows,
                                                                                         c->n, c->d_sums);
        } else {
            const unsigned grid = (unsigned)((c->n + 255) / 256);
            if (c->width == 1) k_accum_generic<int8_t><<<grid, 256, 0, c->stream>>>(gt, row_stride, c->d_rowp, n_rows, c->n, c->ploidy, c->d_sums);
            else if (c->width == 2) k_accum_generic<int16_t><<<grid, 256, 0, c->stream>>>(gt, row_stride, c->d_rowp, n_rows, c->n, c->ploidy, c->d_sums);
            else k_accum_generic<int32_t><<<grid, 256, 0, c->stream>>>(gt, row_stride, c->d_rowp, n_rows, c->n, c->ploidy, c->d_sums);
        }
        break;
    case Layout::DS:
        k_accum_ds<<<(unsigned)((c->n + 255) / 256), 256, 0, c->stream>>>(gt, row_stride, c->d_rowp, n_rows, c->n, c->d_sums);
        break;
    case Layout::BED: {
        const int64_t n_batches = (n_rows + BED_RB - 1) / BED_RB, E = c->exact ? BED_RB * 4 : BED_RB * 8;
        if (!c->d_bed_tab) {
            const int64_t max_batches = (std::max<int64_t>(c->max_rows, 1) + BED_RB - 1) / BED_RB;
            NPC_CUDA(c, cudaMalloc(&c->d_bed_tab, (size_t)max_batches * BED_RB * 8 * sizeof(double)));
            NPC_CUDA(c, cudaMalloc(&c->d_bed_off, (size_t)max_batches * BED_RB * sizeof(int32_t)));
        }
        const unsigned pgrid = (unsigned)((n_batches * E + 255) / 256);
        if (c->exact) {
            k_bed_prep<true><<<pgrid, 256, 0, c->stream>>>(c->d_rowp, n_rows, n_batches, c->d_bed_tab, c->d_bed_off);
            k_accum_bed<true><<<grid, BED_THREADS, 0, c->stream>>>(gt, row_stride, c->d_bed_tab, c->d_bed_off, n_rows, c->n, c->d_sums);
        } else {
            k_bed_prep<false><<<pgrid, 256, 0, c->stream>>>(c->d_rowp, n_rows, n_batches, c->d_bed_tab, c->d_bed_off);
            k_accum_bed<false><<<grid, BED_THREADS, 0, c->stream>>>(gt, row_stride, c->d_bed_tab, c->d_bed_off, n_rows, c->n, c->d_sums);
        }
        c->launches++;                                                                          // k_bed_prep
        break;
    }
    case Layout::DOSE255:
        k_accum_dose255<<<grid, D255_THREADS, 0, c->stream>>>(gt, row_stride, c->d_rowp, n_rows, c->n, c->d_sums);
        break;
    case Layout::DOSE32:
        k_accum_dose32<<<grid, D32_THREADS, 0, c->stream>>>(gt, row_stride, c->d_rowp, n_rows, c->n, c->d_sums);
        break;
    case Layout::PL:
        k_accum_pl<<<grid, PL_THREADS, 0, c->stream>>>(gt, row_stride, c->d_rowp, n_rows, c->n, c->d_sums);
        break;
    }
    c->launches++;
    NPC_CUDA(c, cudaGetLastError());
    return NPC_OK;
}

// The observed pass (npc_observed.cuh) over n_ent entries: out[g * n + s] += called(entry, s) x weight.  w == nullptr: a
// group of one weighted by the records in log; else OBS_G definitions, w[g * n_ent + e].
template <class L>
static int observed_launch(npc_ctx *c, const uint8_t *gt, int64_t row_stride, const npc_row *ent, const npc_locus *log,
                           const uint32_t *w, int64_t n_ent, ull *out) {
    const unsigned gx = (unsigned)((c->n + (int64_t)L::P * OBS_THREADS - 1) / ((int64_t)L::P * OBS_THREADS));
    // the entries split over gridDim.y until ~16 CTAs an SM, at least 64 entries each
    const int64_t sms = c->num_sms > 0 ? c->num_sms : 148;
    const int64_t gy = std::max<int64_t>(1, std::min<int64_t>({ (sms * 16 + gx - 1) / gx, (n_ent + 63) / 64, 65535 }));
    const int64_t per_y = (n_ent + gy - 1) / gy;
    auto k = w ? k_observed<L, OBS_G> : k_observed<L, 1>;
    k<<<dim3(gx, (unsigned)((n_ent + per_y - 1) / per_y)), OBS_THREADS, 0, c->stream>>>(gt, row_stride, c->ploidy, ent, log, w, n_ent, per_y,
                                                                                     c->n, out);
    c->launches++;
    NPC_CUDA(c, cudaGetLastError());
    return NPC_OK;
}

static int launch_observed(npc_ctx *c, const uint8_t *gt, int64_t row_stride, const npc_row *ent, const npc_locus *log,
                           const uint32_t *w, int64_t n_ent, ull *out) {
    if (n_ent == 0 || c->n == 0) return NPC_OK;
    switch (c->layout) {
    case Layout::GT:
        if (c->width == 1 && c->ploidy == 2) return observed_launch<ObsI8x2>(c, gt, row_stride, ent, log, w, n_ent, out);
        if (c->width == 1) return observed_launch<ObsGT<int8_t>>(c, gt, row_stride, ent, log, w, n_ent, out);
        if (c->width == 2) return observed_launch<ObsGT<int16_t>>(c, gt, row_stride, ent, log, w, n_ent, out);
        return observed_launch<ObsGT<int32_t>>(c, gt, row_stride, ent, log, w, n_ent, out);
    case Layout::DS: return observed_launch<ObsDs>(c, gt, row_stride, ent, log, w, n_ent, out);
    case Layout::BED: return observed_launch<ObsBed>(c, gt, row_stride, ent, log, w, n_ent, out);
    case Layout::DOSE255: return observed_launch<ObsDose255>(c, gt, row_stride, ent, log, w, n_ent, out);
    case Layout::DOSE32: return observed_launch<ObsDose32>(c, gt, row_stride, ent, log, w, n_ent, out);
    case Layout::PL: return observed_launch<ObsPl>(c, gt, row_stride, ent, log, w, n_ent, out);
    }
    return NPC_OK;
}

// After a launch's scoring sequence: its n_rows rows and their records (the last n_rows of the log) into d_obs
static int observe_launch(npc_ctx *c, const uint8_t *gt, int64_t row_stride, const npc_row *d_rows, int64_t n_rows) {
    if (!c->observed || n_rows == 0) return NPC_OK;
    return launch_observed(c, gt, row_stride, d_rows, c->d_log + c->log_len - n_rows, nullptr, n_rows, c->d_obs);
}

// The tile kernel's parameters for shape t over every sample and one row group; each mode then sets its own fields
static FusedParams fused_params(const npc_ctx *c, const npc_ctx::TileCfg &t, const uint8_t *gt, int64_t row_stride,
                                const npc_row *d_rows, int64_t n_rows) {
    FusedParams P;
    memset(&P, 0, sizeof(P));
    P.gt = gt; P.row_stride = row_stride; P.n = c->n; P.rows = d_rows; P.n_rows = n_rows; P.pol = c->pol;
    P.sums = c->d_sums; P.nloci = c->d_nloci;
    P.Sr = t.Sr; P.Sc = t.Sc; P.L = t.L; P.A = t.A; P.nc = t.nc; P.slab_stride = t.slab; P.GD = t.GD;
    P.Gs = t.Gs; P.Gr = 1;
    return P;
}

// One cooperative launch of the tile kernel: P.Gs sample slabs x P.Gr row groups
static int launch_tile(npc_ctx *c, const npc_ctx::TileCfg &t, bool exact, FusedParams &P) {
    void *args[] = { &P };
    NPC_CUDA(c, cudaLaunchCooperativeKernel(tile_kernel(t.K, exact, c->width, t.nc), dim3(P.Gs * P.Gr), dim3((t.nc + 2 + t.A) * 32), args, t.smem, c->stream));
    c->launches++;
    return NPC_OK;
}

// count -> decide -> accumulate in one persistent cooperative launch (npc_fused5.cuh)
static int launch_fused(npc_ctx *c, const npc_ctx::TileCfg &t, bool exact, const uint8_t *gt, int64_t row_stride,
                        const npc_row *d_rows, int64_t n_rows) {
    if (n_rows == 0) return NPC_OK;
    int rc = ensure_log(c, n_rows);
    if (rc) return rc;
    const int64_t tiles = (n_rows + F5_R - 1) / F5_R;
    FusedParams P = fused_params(c, t, gt, row_stride, d_rows, n_rows);
    P.Gr = exact ? 1 : (int)std::max<int64_t>(1, std::min<int64_t>(t.Gr, tiles / 16));   // >= 16 tiles per row group
    P.partials = c->d_partials;
    // the tally words are a double buffer: this launch counts into half h and clears the words of half h ^ 1 the next one uses
    const int64_t half_words = std::max<int64_t>(c->max_rows, 1), h = c->fcounts_half;
    P.counts = c->d_fcounts + h * half_words; P.log = c->d_log + c->log_len; P.trace = c->d_trace;
    P.counts_next = c->d_fcounts + (h ^ 1) * half_words; P.n_zero = c->fcounts_dirty[h ^ 1];
    c->fcounts_dirty[h ^ 1] = 0;
    c->fcounts_dirty[h] = n_rows;
    c->fcounts_half ^= 1;
    if ((rc = launch_tile(c, t, exact, P))) return rc;
    // Row groups > 1: a second, wide kernel adds the groups' partial sums in group order.  (Folding this into the tile
    // kernel -- the last group of a slab to finish adds them -- was measured in round 2: one CTA per slab doing
    // Gr - 1 dependent L2 reads per sample took 12 us where this kernel takes ~4, launch included.)
    if (P.Gr > 1) {
        k_add_partials<<<(unsigned)((c->n + 255) / 256), 256, 0, c->stream>>>(c->d_sums, c->d_partials, c->n, P.Gr - 1);
        c->launches++;
        NPC_CUDA(c, cudaGetLastError());
    }
    c->log_len += n_rows;
    return NPC_OK;
}

// Cohorts too wide for one resident pass: tally + decide over all samples (the two kernels of the generic sequence),
// then the tile kernel in "decided" mode once per slab of the sample axis -- it decodes and accumulates, the deciders
// read the rows' contributions from d_rowp.  The slab is read twice (4 B/genotype), the second time at the tile
// kernel's rate instead of k_accum's.
static int launch_wide(npc_ctx *c, const npc_ctx::TileCfg &t, bool exact, const uint8_t *gt, int64_t row_stride,
                       const npc_row *d_rows, int64_t n_rows) {
    if (n_rows == 0) return NPC_OK;
    int rc = launch_tally(c, gt, row_stride, d_rows, n_rows, c->d_counts);
    if (!rc) rc = launch_decide(c, gt, row_stride, d_rows, n_rows, c->d_counts);
    if (rc) return rc;
    FusedParams P = fused_params(c, t, gt, row_stride, d_rows, n_rows);
    P.decided = c->d_rowp;
    for (int s = 0; s < c->wide_slabs; s++) {
        const int64_t s0 = (int64_t)s * c->wide_n, ns = std::min<int64_t>(c->wide_n, c->n - s0);
        if (ns <= 0) break;
        P.gt = gt + s0 * 2; P.n = ns; P.sums = c->d_sums + s0;
        if ((rc = launch_tile(c, t, exact, P))) return rc;
    }
    return NPC_OK;
}

static int launch_block(npc_ctx *c, const uint8_t *gt, int64_t row_stride, const npc_row *d_rows, int64_t n_rows) {
    const npc_ctx::TileCfg *t;
    int rc;
    switch (launch_mode(c, c->exact, n_rows, t)) {
    case 1: case 2: rc = launch_fused(c, *t, c->exact, gt, row_stride, d_rows, n_rows); break;
    case 3: rc = launch_wide(c, *t, c->exact, gt, row_stride, d_rows, n_rows); break;
    default:                                                                                    // 0, 4, 5, 6, 7
        rc = launch_tally(c, gt, row_stride, d_rows, n_rows, c->d_counts);
        if (!rc) rc = launch_decide(c, gt, row_stride, d_rows, n_rows, c->d_counts);
        if (!rc) rc = launch_accum(c, gt, row_stride, n_rows);
    }
    return rc ? rc : observe_launch(c, gt, row_stride, d_rows, n_rows);
}

// ---- subset contexts: compaction ------------------------------------------------------------

// n_rows full rows (n_row samples, src_stride apart) -> compact rows of the context's layout (dst_stride apart), on stream st
static int launch_gather(npc_ctx *c, const uint8_t *src, int64_t src_stride, int64_t n_rows, uint8_t *dst, int64_t dst_stride,
                         cudaStream_t st) {
    if (n_rows == 0) return NPC_OK;
    const LayoutInfo &L = info(c->layout);
    const bool bed = c->layout == Layout::BED;
    const int64_t E = L.sample_bits ? L.sample_bits / 8 : (int64_t)c->ploidy * c->width;             // bytes per sample (.bed: 0)
    const int hdr = L.header;
    // threads per row: one per 16 output bytes (2- and 4-byte samples), 4 bytes (.bed) or unit; a grid-stride loop beyond
    const int64_t per_row = bed ? (c->n + 15) / 16 : (E == 2 || E == 4) ? (c->n * E + 15) / 16 : c->n * (E % 4 ? E : E / 4);
    const unsigned gx = (unsigned)std::max<int64_t>(1, std::min<int64_t>((per_row + SUB_THREADS - 1) / SUB_THREADS, 1024));
    for (int64_t r0 = 0; r0 < n_rows; r0 += 65535) {                                            // grid y: at most 65,535 rows
        const dim3 grid(gx, (unsigned)std::min<int64_t>(65535, n_rows - r0));
        const uint8_t *s = src + r0 * src_stride;
        uint8_t *d = dst + r0 * dst_stride;
        if (bed) k_gather_bed<<<grid, SUB_THREADS, 0, st>>>(s, src_stride, d, dst_stride, c->d_keep, c->n);
        else if (E == 2) k_gather_vec<uint16_t><<<grid, SUB_THREADS, 0, st>>>(s, src_stride, d, dst_stride, c->d_keep, c->n, hdr);
        else if (E == 4) k_gather_vec<uint32_t><<<grid, SUB_THREADS, 0, st>>>(s, src_stride, d, dst_stride, c->d_keep, c->n, hdr);
        else if (E % 4 == 0) k_gather_unit<uint32_t><<<grid, SUB_THREADS, 0, st>>>(s, src_stride, d, dst_stride, c->d_keep, c->n, (int)(E / 4));
        else k_gather_unit<uint8_t><<<grid, SUB_THREADS, 0, st>>>(s, src_stride, d, dst_stride, c->d_keep, c->n, (int)E);
        c->launches++;
        NPC_CUDA(c, cudaGetLastError());
    }
    return NPC_OK;
}

extern "C" int npc_gather_rows_device(npc_ctx *ctx, const void *src, int64_t src_stride, int64_t n_rows, void *dst, int64_t dst_stride) {
    if (!ctx) return NPC_EINVAL;
    if (!ctx->sub) return fail(ctx, NPC_ESTATE, "npc_gather_rows_device: the context was not created with npc_create_subset");
    if (n_rows < 0 || (n_rows && (!src || !dst)) || ((uintptr_t)src & 15) || ((uintptr_t)dst & 15) || (src_stride & 15) || (dst_stride & 15) ||
        src_stride < ctx_row_bytes(ctx, ctx->n_row) || dst_stride < ctx_row_bytes(ctx, ctx->n))
        return fail(ctx, NPC_EINVAL, "npc_gather_rows_device: rows must be 16-byte aligned, strides multiples of 16 holding a whole row");
    NPC_CUDA(ctx, cudaSetDevice(ctx->device));
    return launch_gather(ctx, (const uint8_t *)src, src_stride, n_rows, (uint8_t *)dst, dst_stride, ctx->stream);
}

extern "C" int npc_set_keep(npc_ctx *ctx, const int64_t *keep, int64_t n_keep) {
    if (!ctx) return NPC_EINVAL;
    if (!ctx->sub) return fail(ctx, NPC_ESTATE, "npc_set_keep: the context was not created with npc_create_subset");
    bool ok = keep && n_keep == ctx->n;
    for (int64_t i = 0; ok && i < n_keep; i++) ok = keep[i] >= 0 && keep[i] < ctx->n_row && (i == 0 || keep[i] > keep[i - 1]);
    if (!ok) return fail(ctx, NPC_EINVAL, "npc_set_keep: keep must hold the context's n ascending, distinct indices below n_row_samples");
    std::vector<int32_t> h((size_t)((ctx->n + SUB_PAD - 1) / SUB_PAD * SUB_PAD), 0);
    for (int64_t i = 0; i < n_keep; i++) h[(size_t)i] = (int32_t)keep[i];
    NPC_CUDA(ctx, cudaSetDevice(ctx->device));
    // the gathers of rows uploaded so far (copy stream) and of npc_gather_rows_device (the context's stream) read d_keep:
    // let them finish, then replace it with a blocking copy
    NPC_CUDA(ctx, cudaStreamSynchronize(ctx->copy_stream));
    NPC_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    NPC_CUDA(ctx, cudaMemcpy(ctx->d_keep, h.data(), h.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    return NPC_OK;
}

// A subset context's H2D copy of a slot's n_gt_rows full rows, compacted into dst (dst_stride apart); on the copy stream
static int upload_compact(npc_ctx *c, int32_t slot, int64_t n_gt_rows, uint8_t *dst, int64_t dst_stride) {
    if (!c->d_raw[slot]) NPC_CUDA(c, cudaMalloc(&c->d_raw[slot], (size_t)c->stage_stride * (size_t)std::max<int64_t>(c->staging_rows, 1)));
    NPC_CUDA(c, cudaMemcpyAsync(c->d_raw[slot], c->h_gt[slot], (size_t)n_gt_rows * c->stage_stride, cudaMemcpyHostToDevice, c->copy_stream));
    return launch_gather(c, c->d_raw[slot], c->stage_stride, n_gt_rows, dst, dst_stride, c->copy_stream);
}

// ---- staged blocks -----------------------------------------------------------------------

extern "C" int npc_stage_acquire(npc_ctx *ctx, int32_t *slot, void **gt_host, int64_t *row_stride) {
    if (!ctx || !slot || !gt_host || !row_stride) return NPC_EINVAL;
    if (ctx->n_slots == 0) return fail(ctx, NPC_ESTATE, "context was created without a staging ring");
    NPC_CUDA(ctx, cudaSetDevice(ctx->device));
    const int s = ctx->next_slot;
    if (ctx->slot_state[s] == 1) return fail(ctx, NPC_ESTATE, "all staging slots are lent out: submit one first");
    if (ctx->slot_state[s] == 2) {
        NPC_CUDA(ctx, cudaEventSynchronize(ctx->ev_done[s]));
        ctx->slot_state[s] = 0;
    }
    ctx->slot_state[s] = 1;
    ctx->next_slot = (s + 1) % ctx->n_slots;
    *slot = s; *gt_host = ctx->h_gt[s]; *row_stride = ctx->stage_stride;
    return NPC_OK;
}

extern "C" int npc_score_block(npc_ctx *ctx, int32_t slot, int64_t n_gt_rows, const npc_row *rows, int64_t n_rows) {
    if (!ctx) return NPC_EINVAL;
    if (slot < 0 || slot >= ctx->n_slots || ctx->slot_state[slot] != 1)
        return fail(ctx, NPC_ESTATE, "slot was not acquired");
    if (n_gt_rows > ctx->staging_rows) return fail(ctx, NPC_EINVAL, "more genotype rows than a staging slot holds");
    NPC_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!ctx->d_gt[slot]) NPC_CUDA(ctx, cudaMalloc(&ctx->d_gt[slot], (size_t)ctx->row_stride * (size_t)std::max<int64_t>(ctx->staging_rows, 1)));
    int rc = check_block(ctx, ctx->d_gt[slot], ctx->row_stride, n_gt_rows, rows, n_rows);
    if (!rc) rc = check_one_alt(ctx, rows, n_rows, 0);
    if (rc) return rc;
    if (n_gt_rows && ctx->sub) {
        if ((rc = upload_compact(ctx, slot, n_gt_rows, ctx->d_gt[slot], ctx->row_stride))) return rc;
    } else if (n_gt_rows)
        NPC_CUDA(ctx, cudaMemcpyAsync(ctx->d_gt[slot], ctx->h_gt[slot], (size_t)n_gt_rows * ctx->row_stride,
                                      cudaMemcpyHostToDevice, ctx->copy_stream));
    NPC_CUDA(ctx, cudaEventRecord(ctx->ev_h2d[slot], ctx->copy_stream));
    NPC_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_h2d[slot], 0));
    const npc_row *d_rows;
    if ((rc = upload_rows(ctx, rows, n_rows, 0, &d_rows))) return rc;
    if ((rc = launch_block(ctx, ctx->d_gt[slot], ctx->row_stride, d_rows, n_rows))) return rc;
    // npc_stage_acquire waits on ev_done before lending the slot again, so the next H2D into
    // it cannot overtake these kernels and copies into OTHER slots overlap them freely
    NPC_CUDA(ctx, cudaEventRecord(ctx->ev_done[slot], ctx->stream));
    ctx->slot_state[slot] = 2;
    return NPC_OK;
}

// ---- device-resident blocks ----------------------------------------------------------------

extern "C" int npc_score_block_device(npc_ctx *ctx, const void *gt_dev, int64_t row_stride, int64_t n_gt_rows,
                                      const npc_row *rows, int64_t n_rows, int32_t rows_on_device) {
    int rc = check_block(ctx, gt_dev, row_stride, n_gt_rows, rows, n_rows);
    if (!rc) rc = check_one_alt(ctx, rows, n_rows, rows_on_device);
    if (rc) return rc;
    NPC_CUDA(ctx, cudaSetDevice(ctx->device));
    const npc_row *d_rows;
    if ((rc = upload_rows(ctx, rows, n_rows, rows_on_device, &d_rows))) return rc;
    return launch_block(ctx, (const uint8_t *)gt_dev, row_stride, d_rows, n_rows);
}

// The split calls' checks and row upload: hard-call rows of the BCF layouts only
static int split_prologue(npc_ctx *c, const void *gt_dev, int64_t row_stride, int64_t n_gt_rows, const npc_row *rows,
                          int64_t n_rows, int32_t rows_on_device, const int64_t *counts_dev, const npc_row **d_rows) {
    int rc = check_block(c, gt_dev, row_stride, n_gt_rows, rows, n_rows);
    if (rc) return rc;
    if (!counts_dev) return fail(c, NPC_EINVAL, "counts_dev is NULL");
    if (c->layout != Layout::GT)
        return fail(c, NPC_EUNSUPPORTED, (std::string("the split count / accumulate calls take BCF GT rows, not ") + info(c->layout).name).c_str());
    NPC_CUDA(c, cudaSetDevice(c->device));
    return upload_rows(c, rows, n_rows, rows_on_device, d_rows);
}

extern "C" int npc_count_block_device(npc_ctx *ctx, const void *gt_dev, int64_t row_stride, int64_t n_gt_rows,
                                      const npc_row *rows, int64_t n_rows, int32_t rows_on_device,
                                      int64_t *counts_dev) {
    const npc_row *d_rows;
    int rc = split_prologue(ctx, gt_dev, row_stride, n_gt_rows, rows, n_rows, rows_on_device, counts_dev, &d_rows);
    return rc ? rc : launch_tally(ctx, (const uint8_t *)gt_dev, row_stride, d_rows, n_rows, (ull *)counts_dev);
}

extern "C" int npc_accumulate_block_device(npc_ctx *ctx, const void *gt_dev, int64_t row_stride, int64_t n_gt_rows,
                                           const npc_row *rows, int64_t n_rows, int32_t rows_on_device,
                                           const int64_t *counts_dev) {
    const npc_row *d_rows;
    int rc = split_prologue(ctx, gt_dev, row_stride, n_gt_rows, rows, n_rows, rows_on_device, counts_dev, &d_rows);
    if (!rc) rc = launch_decide(ctx, (const uint8_t *)gt_dev, row_stride, d_rows, n_rows, (const ull *)counts_dev);
    if (!rc) rc = launch_accum(ctx, (const uint8_t *)gt_dev, row_stride, n_rows);
    return rc ? rc : observe_launch(ctx, (const uint8_t *)gt_dev, row_stride, d_rows, n_rows);
}

// ---- resident slab ---------------------------------------------------------------------------

extern "C" int npc_resident_reserve(npc_ctx *ctx, int64_t capacity_rows, int64_t *granted_rows) {
    if (!ctx || capacity_rows < 0) return NPC_EINVAL;
    NPC_CUDA(ctx, cudaSetDevice(ctx->device));
    NPC_CUDA(ctx, cudaDeviceSynchronize());
    if (ctx->d_slab && ctx->slab_owned) cudaFree(ctx->d_slab);
    ctx->d_slab = nullptr; ctx->slab_rows = 0; ctx->slab_owned = false;
    if (!ctx->ev_slab) NPC_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_slab, cudaEventDisableTiming));
    size_t free_b = 0, total_b = 0;
    NPC_CUDA(ctx, cudaMemGetInfo(&free_b, &total_b));
    const int64_t budget = (int64_t)(free_b - std::min<size_t>(free_b, (size_t)1 << 30)) / ctx->row_stride;   // keep 1 GiB spare
    int64_t rows = std::min(capacity_rows, budget);
    if (rows < 1 && capacity_rows > 0) return fail(ctx, NPC_ENOMEM, "no device memory for a resident slab");
    if (rows > 0) NPC_CUDA(ctx, cudaMalloc(&ctx->d_slab, (size_t)rows * ctx->row_stride));
    ctx->slab_rows = rows; ctx->slab_owned = rows > 0; ctx->slab_stride = ctx->row_stride;
    if (granted_rows) *granted_rows = rows;
    return NPC_OK;
}

extern "C" int npc_resident_adopt(npc_ctx *ctx, const void *gt_dev, int64_t row_stride, int64_t n_gt_rows) {
    if (!ctx || n_gt_rows < 0 || (n_gt_rows && !gt_dev)) return NPC_EINVAL;
    if (((uintptr_t)gt_dev & 15) || (row_stride & 15) || row_stride < ctx_row_bytes(ctx, ctx->n))
        return fail(ctx, NPC_EINVAL, "npc_resident_adopt: slab must be 16-byte aligned, row_stride a multiple of 16 holding a whole row");
    NPC_CUDA(ctx, cudaSetDevice(ctx->device));
    NPC_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->d_slab && ctx->slab_owned) cudaFree(ctx->d_slab);
    if (!ctx->ev_slab) NPC_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_slab, cudaEventDisableTiming));
    ctx->d_slab = (uint8_t *)gt_dev; ctx->slab_rows = n_gt_rows; ctx->slab_owned = false; ctx->slab_stride = row_stride;
    return NPC_OK;
}

extern "C" int npc_stage_upload(npc_ctx *ctx, int32_t slot, int64_t n_gt_rows, int64_t dst_row) {
    if (!ctx) return NPC_EINVAL;
    if (slot < 0 || slot >= ctx->n_slots || ctx->slot_state[slot] != 1) return fail(ctx, NPC_ESTATE, "slot was not acquired");
    if (n_gt_rows < 0 || n_gt_rows > ctx->staging_rows || dst_row < 0 || dst_row + n_gt_rows > ctx->slab_rows)
        return fail(ctx, NPC_EINVAL, "npc_stage_upload: rows outside the resident slab");
    if (ctx->slab_stride != ctx->row_stride) return fail(ctx, NPC_ESTATE, "npc_stage_upload: the adopted slab has another row stride");
    NPC_CUDA(ctx, cudaSetDevice(ctx->device));
    // a scoring launch may still be reading the slab rows we are about to overwrite
    NPC_CUDA(ctx, cudaStreamWaitEvent(ctx->copy_stream, ctx->ev_slab, 0));
    if (n_gt_rows && ctx->sub) {
        if (int rc = upload_compact(ctx, slot, n_gt_rows, ctx->d_slab + dst_row * ctx->row_stride, ctx->row_stride)) return rc;
    } else if (n_gt_rows)
        NPC_CUDA(ctx, cudaMemcpyAsync(ctx->d_slab + dst_row * ctx->row_stride, ctx->h_gt[slot], (size_t)n_gt_rows * ctx->row_stride,
                                      cudaMemcpyHostToDevice, ctx->copy_stream));
    NPC_CUDA(ctx, cudaEventRecord(ctx->ev_h2d[slot], ctx->copy_stream));
    NPC_CUDA(ctx, cudaEventRecord(ctx->ev_done[slot], ctx->copy_stream));      // the slot is free once copied
    ctx->slot_state[slot] = 2;
    return NPC_OK;
}

extern "C" int npc_score_resident(npc_ctx *ctx, const npc_row *rows, int64_t n_rows) {
    if (!ctx || n_rows < 0 || (n_rows && !rows)) return NPC_EINVAL;
    NPC_CUDA(ctx, cudaSetDevice(ctx->device));
    for (int64_t i = 0; i < n_rows; i++)
        if (rows[i].kind == NPC_KIND_GT && rows[i].gt_row >= ctx->slab_rows)
            return fail(ctx, NPC_EINVAL, "npc_score_resident: gt_row outside the resident slab");
    if (int rc = check_one_alt(ctx, rows, n_rows, 0)) return rc;
    // every upload issued so far must have landed
    for (int s = 0; s < ctx->n_slots; s++) NPC_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, ctx->ev_h2d[s], 0));
    for (int64_t r0 = 0; r0 < n_rows; r0 += ctx->max_rows) {
        const int64_t nr = std::min(ctx->max_rows, n_rows - r0);
        const npc_row *d_rows;
        int rc = upload_rows(ctx, rows + r0, nr, 0, &d_rows);
        if (rc) return rc;
        if ((rc = launch_block(ctx, ctx->d_slab, ctx->slab_stride, d_rows, nr))) return rc;
    }
    NPC_CUDA(ctx, cudaEventRecord(ctx->ev_slab, ctx->stream));
    return NPC_OK;
}

// ---- results -------------------------------------------------------------------------------

// sums (n doubles from the device array `sums`), nloci and the locus log to the host; returns when they have landed
static int copy_out(npc_ctx *c, const double *sums, double *sums_out, int64_t *nloci_out, npc_locus *loci_out, int64_t loci_cap,
                    int64_t *n_loci_out) {
    if (c->n) NPC_CUDA(c, cudaMemcpyAsync(sums_out, sums, c->n * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    ull nl = 0;
    NPC_CUDA(c, cudaMemcpyAsync(&nl, c->d_nloci, sizeof(ull), cudaMemcpyDeviceToHost, c->stream));
    if (n_loci_out) *n_loci_out = c->log_len;
    if (loci_out) {
        if (loci_cap < c->log_len) return fail(c, NPC_EINVAL, "loci_out too small");
        NPC_CUDA(c, cudaMemcpyAsync(loci_out, c->d_log, c->log_len * sizeof(npc_locus), cudaMemcpyDeviceToHost, c->stream));
    }
    NPC_CUDA(c, cudaStreamSynchronize(c->stream));
    if (nloci_out) *nloci_out = (int64_t)nl;
    return NPC_OK;
}

extern "C" int npc_finish(npc_ctx *ctx, double offset, double *scores_out, int64_t *nloci_out, npc_locus *loci_out,
                          int64_t loci_cap, int64_t *n_loci_out) {
    if (!ctx || !scores_out) return NPC_EINVAL;
    NPC_CUDA(ctx, cudaSetDevice(ctx->device));
    if (ctx->n) {
        k_finalize<<<(unsigned)((ctx->n + 255) / 256), 256, 0, ctx->stream>>>(ctx->d_sums, ctx->n, ctx->d_nloci, offset, ctx->d_out);
        ctx->launches++;
        NPC_CUDA(ctx, cudaGetLastError());
    }
    return copy_out(ctx, ctx->d_out, scores_out, nloci_out, loci_out, loci_cap, n_loci_out);
}

// ---- several score definitions over the resident slab ------------------------------------------

// one fused pass per definition: exactly npc_reset + npc_score_resident + npc_finish each
static int multi_one_by_one(npc_ctx *ctx, int32_t n_scores, const npc_row *const *rows, const int64_t *n_rows, const double *offsets,
                            double *const *scores_out, int64_t *nloci_out, npc_locus *const *loci_out) {
    for (int32_t k = 0; k < n_scores; k++) {
        int rc = npc_reset(ctx);
        if (rc) return rc;
        if ((rc = npc_score_resident(ctx, rows[k], n_rows[k]))) return rc;
        int64_t nlog = 0;
        npc_locus *lg = loci_out ? loci_out[k] : nullptr;
        rc = offsets ? npc_finish(ctx, offsets[k], scores_out[k], nloci_out ? &nloci_out[k] : nullptr, lg, lg ? n_rows[k] : 0, &nlog)
                     : npc_partial(ctx, scores_out[k], nloci_out ? &nloci_out[k] : nullptr, lg, lg ? n_rows[k] : 0, &nlog);
        if (rc) return rc;
    }
    return NPC_OK;
}


// The dense contraction (npc_multi.cuh).  Returns 1 when the input is outside what it represents
// (the caller then scores one by one), 0 on success, < 0 on error.
static int multi_contract(npc_ctx *c, int32_t S, const npc_row *const *rows, const int64_t *n_rows, const double *offsets,
                          double *const *scores_out, int64_t *nloci_out, npc_locus *const *loci_out) {
    const bool timing = getenv("NPC_TIMING") != nullptr;         // phase wall times on stderr (each phase drained first)
    auto t_last = std::chrono::steady_clock::now();
    auto mark = [&](const char *what) {
        if (!timing) return;
        cudaStreamSynchronize(c->stream);
        auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "[npc multi] %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(now - t_last).count());
        t_last = now;
    };
    // ---- entries: one per (slab row, effect allele) any definition uses -------------------------
    std::vector<int64_t> row0(S + 1, 0);
    for (int k = 0; k < S; k++) row0[k + 1] = row0[k] + n_rows[k];
    const int64_t R = row0[S];
    std::vector<npc_row> erows;
    std::vector<int32_t> ent((size_t)R, -1), score_of((size_t)R, 0);
    // per slab row: the entry of effect alleles 0..3 directly, a chain only for rarer alleles.  (Building this table on
    // eight host threads, each owning a range of slab rows and scanning every definition, was measured in round 2: 1.85 ms
    // against 1.2-1.4 ms for this loop at 18 x 20,000 rows -- thread start-up and eight scans cost more than they save.)
    std::vector<int32_t> direct((size_t)c->slab_rows * 4, -1), head, next, last_score, repeats;
    erows.reserve((size_t)std::min<int64_t>(R, c->slab_rows * 2));
    for (int k = 0; k < S; k++)
        for (int64_t i = 0; i < n_rows[k]; i++) {
            const npc_row &r = rows[k][i];
            const int64_t j = row0[k] + i;
            score_of[j] = k;
            if (r.kind != NPC_KIND_GT || r.gt_row < 0) continue;
            if (r.gt_row >= c->slab_rows) return fail(c, NPC_EINVAL, "npc_score_resident_multi: gt_row outside the resident slab");
            if (r.eaidx < 0 || r.eaidx > 62) return 1;               // no int8 code can match: leave it to the general path
            int32_t e;
            if (r.eaidx < 4) e = direct[(size_t)r.gt_row * 4 + r.eaidx];
            else {
                if (head.empty()) head.assign((size_t)c->slab_rows, -1);
                e = head[r.gt_row];
                while (e >= 0 && erows[e].eaidx != r.eaidx) e = next[e];
            }
            if (e < 0) {
                e = (int32_t)erows.size();
                npc_row er = r; er.kind = NPC_KIND_GT;
                erows.push_back(er); last_score.push_back(-1); repeats.push_back(0); next.push_back(-1);
                if (r.eaidx < 4) direct[(size_t)r.gt_row * 4 + r.eaidx] = e;
                else { next[e] = head[r.gt_row]; head[r.gt_row] = e; }
            }
            ent[j] = e;
            if (last_score[e] != k) { last_score[e] = k; repeats[e] = 0; }
            if (++repeats[e] > 4) return 1;                          // fixed-point headroom covers 4 repeats
        }
    const int64_t E = (int64_t)erows.size();
    if (E == 0 || E > (1 << 22)) return 1;
    const int32_t n_kb = (int32_t)((E + npc::MC_ENT - 1) / npc::MC_ENT);
    const int64_t Ep = (int64_t)n_kb * npc::MC_ENT;
    std::vector<int32_t> entry_row((size_t)Ep, erows[0].gt_row);
    // low byte: (eaidx + 1) << 1, the byte an allele of the effect allele carries; bits 8..: byte offset of the entry's pair table.
    // Padding entries: a pattern no allele byte equals (0xFE) and the no-match table.
    std::vector<uint32_t> entry_pat((size_t)Ep, 0xFEu | ((uint32_t)(3 * npc::MC_TAB_STRIDE) << 8));
    for (int64_t e = 0; e < E; e++) {
        entry_row[e] = erows[e].gt_row;
        entry_pat[e] = (uint32_t)((erows[e].eaidx + 1) << 1) | ((uint32_t)(std::min(erows[e].eaidx, 3) * npc::MC_TAB_STRIDE) << 8);
    }

    mark("entries (host)");
    const int64_t n_tiles = (c->n + npc::MC_N - 1) / npc::MC_N;
    const int64_t sms = c->num_sms > 0 ? c->num_sms : 148;
    // split the k-blocks of a tile over `parts` work units when that evens out the last round
    // (782 tiles on 148 SMs: 6 rounds for 5.3 rounds of work; in thirds 16 rounds of 1/3 = 5.33)
    int parts = 1;
    {
        double best = (double)((n_tiles + sms - 1) / sms);
        const char *e = getenv("NPC_MULTI_PARTS");
        for (int p = 2; p <= 4 && n_kb / p >= 16; p++) {
            const double cost = (double)((n_tiles * p + sms - 1) / sms) / p * 1.01;      // a little for the extra epilogues
            if (cost < best) { best = cost; parts = p; }
        }
        if (e && *e) parts = std::max(1, std::min(atoi(e), std::max(1, n_kb)));
    }
    const int kb_per_part = (n_kb + parts - 1) / parts;
    parts = (n_kb + kb_per_part - 1) / kb_per_part;                     // no empty part
    // scratch: one arena kept by the context, grown when a call needs more
    const int Sg = std::min<int>(S, npc::MC_SCORES);
    size_t need = 0;
    auto reserve = [&](size_t bytes) { size_t off = need; need += (std::max<size_t>(bytes, 16) + 255) & ~(size_t)255; return off; };
    const size_t o_erows = reserve(E * sizeof(npc_row)), o_ecounts = reserve(2 * E * sizeof(ull)), o_entry_row = reserve(Ep * 4),
                 o_entry_pat = reserve(Ep * 4), o_all = reserve(R * sizeof(npc_row)), o_ent = reserve(R * 4), o_score_of = reserve(R * 4),
                 o_counts = reserve(2 * R * sizeof(ull)), o_rowp = reserve(R * sizeof(RowP)), o_log = reserve(R * sizeof(npc_locus)),
                 o_nloci = reserve(S * sizeof(ull)), o_row0 = reserve((S + 1) * 8), o_scale = reserve(S * sizeof(MultiScale)),
                 o_fexp = reserve(S * 4), o_coef = reserve((size_t)Sg * 2 * Ep * 8), o_pois = reserve((size_t)Sg * Ep),
                 o_A = reserve((size_t)n_kb * npc::MC_A_STAGE), o_out = reserve((size_t)Sg * c->n * 8),
                 o_part = reserve(parts > 1 ? (size_t)parts * Sg * c->n * 8 : 16);
    if (need > c->multi_scratch_bytes) {
        NPC_CUDA(c, cudaStreamSynchronize(c->stream));
        cudaFree(c->d_multi_scratch); c->d_multi_scratch = nullptr; c->multi_scratch_bytes = 0;
        if (cudaMalloc(&c->d_multi_scratch, need) != cudaSuccess) { cudaGetLastError(); return 1; }   // no room: one by one needs none
        c->multi_scratch_bytes = need;
    }
    uint8_t *base = c->d_multi_scratch;
    npc_row *d_erows = (npc_row *)(base + o_erows), *d_all = (npc_row *)(base + o_all);
    ull *d_ecounts = (ull *)(base + o_ecounts), *d_counts = (ull *)(base + o_counts), *d_nloci = (ull *)(base + o_nloci);
    int32_t *d_entry_row = (int32_t *)(base + o_entry_row), *d_ent = (int32_t *)(base + o_ent), *d_score_of = (int32_t *)(base + o_score_of),
            *d_fexp = (int32_t *)(base + o_fexp);
    uint32_t *d_entry_pat = (uint32_t *)(base + o_entry_pat);
    RowP *d_rowp = (RowP *)(base + o_rowp); npc_locus *d_log = (npc_locus *)(base + o_log); int64_t *d_row0 = (int64_t *)(base + o_row0);
    MultiScale *d_scale = (MultiScale *)(base + o_scale); long long *d_coef = (long long *)(base + o_coef);
    uint8_t *d_pois = base + o_pois, *d_A = base + o_A; double *d_out = (double *)(base + o_out), *d_part = (double *)(base + o_part);
    cudaStream_t st = c->stream;
    mark("scratch arena");
    NPC_CUDA(c, cudaMemcpyAsync(d_erows, erows.data(), E * sizeof(npc_row), cudaMemcpyHostToDevice, st));
    for (int s = 0; s < c->n_slots; s++) NPC_CUDA(c, cudaStreamWaitEvent(st, c->ev_h2d[s], 0));   // every upload has landed

    // ---- tallies once per entry: launched first, so that the pass over the slab (the long pole) runs while the host
    // pushes the row tables of every definition through the copy stream
    int rc = launch_tally(c, c->d_slab, c->slab_stride, d_erows, E, d_ecounts);
    if (rc) return rc;
    cudaStream_t cs = c->copy_stream;
    if (!c->ev_multi) NPC_CUDA(c, cudaEventCreateWithFlags(&c->ev_multi, cudaEventDisableTiming));
    NPC_CUDA(c, cudaMemcpyAsync(d_entry_row, entry_row.data(), Ep * sizeof(int32_t), cudaMemcpyHostToDevice, cs));
    NPC_CUDA(c, cudaMemcpyAsync(d_entry_pat, entry_pat.data(), Ep * sizeof(uint32_t), cudaMemcpyHostToDevice, cs));
    for (int k = 0; k < S; k++) if (n_rows[k])
        NPC_CUDA(c, cudaMemcpyAsync(d_all + row0[k], rows[k], n_rows[k] * sizeof(npc_row), cudaMemcpyHostToDevice, cs));
    NPC_CUDA(c, cudaMemcpyAsync(d_ent, ent.data(), R * sizeof(int32_t), cudaMemcpyHostToDevice, cs));
    NPC_CUDA(c, cudaMemcpyAsync(d_score_of, score_of.data(), R * sizeof(int32_t), cudaMemcpyHostToDevice, cs));
    NPC_CUDA(c, cudaMemcpyAsync(d_row0, row0.data(), (S + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, cs));
    NPC_CUDA(c, cudaMemsetAsync(d_nloci, 0, S * sizeof(ull), cs));
    NPC_CUDA(c, cudaEventRecord(c->ev_multi, cs));
    NPC_CUDA(c, cudaStreamWaitEvent(st, c->ev_multi, 0));
    mark("tally kernel + row tables H2D");

    // ---- decisions per definition (the same k_decide as every path) -----------------------------
    if (R) {
        k_multi_gather<<<(unsigned)((R + 255) / 256), 256, 0, st>>>(d_ent, R, d_ecounts, d_counts);
        c->launches++;
    }
    for (int k = 0; k < S; k++) if (n_rows[k]) {
        const TallyIn in = { nullptr, 0, d_counts + 2 * row0[k], nullptr, 0 };
        k_decide<CountTally><<<(unsigned)((n_rows[k] + 127) / 128), 128, 0, st>>>(in, d_all + row0[k], n_rows[k], c->pol, c->n,
                                                                                 d_rowp + row0[k], d_log + row0[k], d_nloci + k);
        c->launches++;
    }
    k_multi_scale<<<S, 256, 0, st>>>(d_rowp, d_row0, d_scale);
    c->launches++;
    NPC_CUDA(c, cudaGetLastError());
    std::vector<MultiScale> scale(S);
    std::vector<ull> nloci(S);
    NPC_CUDA(c, cudaMemcpyAsync(scale.data(), d_scale, S * sizeof(MultiScale), cudaMemcpyDeviceToHost, st));
    NPC_CUDA(c, cudaMemcpyAsync(nloci.data(), d_nloci, S * sizeof(ull), cudaMemcpyDeviceToHost, st));
    NPC_CUDA(c, cudaEventRecord(c->ev_multi, st));
    NPC_CUDA(c, cudaStreamSynchronize(st));
    // the per-locus records go home on the copy stream while the contraction runs
    NPC_CUDA(c, cudaStreamWaitEvent(cs, c->ev_multi, 0));
    for (int k = 0; k < S; k++) if (loci_out && loci_out[k] && n_rows[k])
        NPC_CUDA(c, cudaMemcpyAsync(loci_out[k], d_log + row0[k], n_rows[k] * sizeof(npc_locus), cudaMemcpyDeviceToHost, cs));
    mark("decide + scale");
    std::vector<int32_t> fexp(S, 0);
    int rps = npc::MC_DIGITS;
    for (int k = 0; k < S; k++) {
        if (scale[k].flags & 1) return 1;
        if (scale[k].flags & 2) rps = npc::MC_DIGITS + 1;                // some imputed contribution is NaN: add the counter rows
        int ex = 0;
        if (scale[k].maxabs > 0) { frexp(scale[k].maxabs, &ex); fexp[k] = 52 - ex; }
        if (fexp[k] > 900 || fexp[k] < -900) return 1;
    }
    NPC_CUDA(c, cudaMemcpyAsync(d_fexp, fexp.data(), S * sizeof(int32_t), cudaMemcpyHostToDevice, st));

    // ---- contraction -------------------------------------------------------------------------------
    if (!c->multi_attr_set) {                                           // per device, hence per context
        NPC_CUDA(c, cudaFuncSetAttribute(k_multi_contract, cudaFuncAttributeMaxDynamicSharedMemorySize, npc::MC_SMEM));
        c->multi_attr_set = true;
    }
    const unsigned grid = (unsigned)std::min<int64_t>(n_tiles * parts, sms);
    const int per_launch = npc::MC_M / rps;                             // 18 definitions of 7 rows, or 16 of 8
    for (int k0 = 0; k0 < S; k0 += per_launch) {
        const int ng = std::min(per_launch, S - k0);
        NPC_CUDA(c, cudaMemsetAsync(d_coef, 0, (size_t)ng * 2 * Ep * sizeof(long long), st));
        NPC_CUDA(c, cudaMemsetAsync(d_pois, 0, (size_t)ng * Ep, st));
        const int64_t ra = row0[k0], rb = row0[k0 + ng];
        if (rb > ra) {
            k_multi_coef<<<(unsigned)((rb - ra + 255) / 256), 256, 0, st>>>(d_rowp + ra, d_ent + ra, d_score_of + ra, rb - ra, k0, d_fexp + k0, Ep,
                                                                           d_coef, d_pois);
            c->launches++;
        }
        k_multi_digits<<<dim3((unsigned)n_kb, npc::MC_M), 128, 0, st>>>(d_coef, d_pois, Ep, ng, rps, d_A);
        c->launches++;
        MultiParams P;
        memset(&P, 0, sizeof(P));
        P.gt = c->d_slab; P.row_stride = c->slab_stride; P.n = c->n;
        P.entry_row = d_entry_row; P.entry_pat = d_entry_pat; P.A = d_A; P.n_kb = n_kb; P.n_scores = ng; P.rps = rps;
        P.parts = parts; P.kb_per_part = kb_per_part; P.partial = d_part;
        for (int k = 0; k < ng; k++) {
            P.sc_lo[k] = ldexp(1.0, -fexp[k0 + k]); P.sc_hi[k] = ldexp(1.0, 32 - fexp[k0 + k]);
            P.consts[k] = scale[k0 + k].consts;
            P.denom[k] = offsets ? (double)(int64_t)nloci[k0 + k] * 2.0 : 1.0;       // no offsets: raw partial sums (x / 1 + 0 = x)
            P.offset[k] = offsets ? offsets[k0 + k] : 0.0;
            P.out[k] = d_out + (size_t)k * c->n;
        }
        mark("digit tiles");
        k_multi_contract<<<grid, npc::MC_THREADS, npc::MC_SMEM, st>>>(P);
        c->launches++;
        NPC_CUDA(c, cudaGetLastError());
        if (parts > 1) {
            k_multi_finish<<<dim3((unsigned)((c->n + 255) / 256), (unsigned)ng), 256, 0, st>>>(P);
            c->launches++;
            NPC_CUDA(c, cudaGetLastError());
        }
        mark("contraction kernel");
        for (int k = 0; k < ng; k++)
            NPC_CUDA(c, cudaMemcpyAsync(scores_out[k0 + k], d_out + (size_t)k * c->n, c->n * sizeof(double), cudaMemcpyDeviceToHost, st));
        NPC_CUDA(c, cudaStreamSynchronize(st));
        mark("scores D2H");
    }
    NPC_CUDA(c, cudaEventRecord(c->ev_slab, st));
    NPC_CUDA(c, cudaStreamSynchronize(cs));                                // the records have landed
    for (int k = 0; k < S; k++) if (nloci_out) nloci_out[k] = (int64_t)nloci[k];
    return 0;
}

static int score_multi(npc_ctx *ctx, int32_t n_scores, const npc_row *const *rows, const int64_t *n_rows, const double *offsets,
                       double *const *scores_out, int64_t *nloci_out, npc_locus *const *loci_out) {
    // the contraction pays one tally pass + one pass per 16 definitions; below three definitions the fused kernel is as cheap
    const char *env = getenv("NPC_MULTI");
    const int min_scores = env && *env ? (atoi(env) ? 1 : 1 << 30) : 3;
    if (n_scores >= min_scores && !ctx->exact && ctx->width == 1 && ctx->ploidy == 2 && ctx->n > 0 && ctx->d_slab) {
        const int rc = multi_contract(ctx, n_scores, rows, n_rows, offsets, scores_out, nloci_out, loci_out);
        if (rc <= 0) { if (rc == 0) ctx->multi_contractions++; return rc; }
    }
    return multi_one_by_one(ctx, n_scores, rows, n_rows, offsets, scores_out, nloci_out, loci_out);
}

// Observed counts of the definitions with observed_out[k] != NULL from their records (loci[k]), OBS_G definitions per pass
// over the slab.  An entry is a slab row (FORMAT/PL: a slab row, effect allele and eaf, which decide whether a sample is
// called); its weight for a definition is the number of the definition's OK rows that name it.
static int multi_observed(npc_ctx *c, int32_t S, const npc_row *const *rows, const int64_t *n_rows, npc_locus *const *loci,
                          int64_t *const *observed_out) {
    std::vector<int32_t> defs;
    for (int32_t k = 0; k < S; k++) if (observed_out[k]) defs.push_back(k);
    const bool pl = c->layout == Layout::PL;
    const int64_t n1 = std::max<int64_t>(c->n, 1);
    for (size_t k0 = 0; k0 < defs.size(); k0 += OBS_G) {
        const size_t ng = std::min<size_t>(OBS_G, defs.size() - k0);
        std::vector<npc_row> ent;
        std::vector<std::array<uint32_t, OBS_G>> wt;
        std::vector<int32_t> by_row((size_t)c->slab_rows, -1);
        std::unordered_map<std::string, int32_t> by_key;                // FORMAT/PL entries
        for (size_t g = 0; g < ng; g++) {
            const int32_t k = defs[k0 + g];
            for (int64_t i = 0; i < n_rows[k]; i++) {
                const npc_row &r = rows[k][i];
                const npc_locus &rec = loci[k][i];
                if (rec.klass != 0 || !rec.used || r.kind != NPC_KIND_GT || r.gt_row < 0) continue;
                int32_t *slot = &by_row[(size_t)r.gt_row];
                if (pl) {
                    std::string key((const char *)&r.gt_row, 4);
                    key.append((const char *)&r.eaidx, 4).append((const char *)&r.eaf, 8);
                    slot = &by_key.emplace(key, -1).first->second;
                }
                if (*slot < 0) {
                    *slot = (int32_t)ent.size();
                    ent.push_back(r);
                    wt.push_back({});
                }
                wt[(size_t)*slot][g]++;
            }
        }
        const int64_t E = (int64_t)ent.size();
        std::vector<uint32_t> w((size_t)(OBS_G * E));
        for (int64_t e = 0; e < E; e++) for (int g = 0; g < OBS_G; g++) w[(size_t)(g * E + e)] = wt[(size_t)e][g];
        const size_t o_out = 0, o_ent = OBS_G * n1 * sizeof(ull), o_w = o_ent + ((E * sizeof(npc_row) + 255) & ~(size_t)255);
        const size_t need = o_w + std::max<size_t>(w.size() * sizeof(uint32_t), 16);
        if (need > c->obs_scratch_bytes) {
            NPC_CUDA(c, cudaStreamSynchronize(c->stream));
            cudaFree(c->d_obs_scratch); c->d_obs_scratch = nullptr; c->obs_scratch_bytes = 0;
            NPC_CUDA(c, cudaMalloc(&c->d_obs_scratch, need));
            c->obs_scratch_bytes = need;
        }
        ull *d_out = (ull *)(c->d_obs_scratch + o_out);
        npc_row *d_ent = (npc_row *)(c->d_obs_scratch + o_ent);
        uint32_t *d_w = (uint32_t *)(c->d_obs_scratch + o_w);
        NPC_CUDA(c, cudaMemsetAsync(d_out, 0, OBS_G * n1 * sizeof(ull), c->stream));
        if (E) {
            NPC_CUDA(c, cudaMemcpyAsync(d_ent, ent.data(), E * sizeof(npc_row), cudaMemcpyHostToDevice, c->stream));
            NPC_CUDA(c, cudaMemcpyAsync(d_w, w.data(), w.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, c->stream));
            if (int rc = launch_observed(c, c->d_slab, c->slab_stride, d_ent, nullptr, d_w, E, d_out)) return rc;
        }
        for (size_t g = 0; g < ng; g++)
            if (c->n) NPC_CUDA(c, cudaMemcpyAsync(observed_out[defs[k0 + g]], d_out + g * n1, c->n * sizeof(ull), cudaMemcpyDeviceToHost, c->stream));
        NPC_CUDA(c, cudaStreamSynchronize(c->stream));                      // the host tables above go out of scope
    }
    NPC_CUDA(c, cudaEventRecord(c->ev_slab, c->stream));
    return NPC_OK;
}

// The context's own observed counts after a multi call: zero whichever path scored (the one-by-one path resets the
// context per definition, the contraction does not touch it)
static int zero_observed(npc_ctx *c) {
    if (c->d_obs) NPC_CUDA(c, cudaMemsetAsync(c->d_obs, 0, std::max<int64_t>(c->n, 1) * sizeof(ull), c->stream));
    return NPC_OK;
}

extern "C" int npc_score_resident_multi_observed(npc_ctx *ctx, int32_t n_scores, const npc_row *const *rows, const int64_t *n_rows,
                                                 const double *offsets, double *const *scores_out, int64_t *nloci_out,
                                                 npc_locus *const *loci_out, int64_t *const *observed_out) {
    if (!ctx || n_scores < 0 || (n_scores && (!rows || !n_rows || !scores_out))) return NPC_EINVAL;
    for (int32_t k = 0; k < n_scores; k++) if (n_rows[k] < 0 || (n_rows[k] && !rows[k]) || !scores_out[k]) return NPC_EINVAL;
    NPC_CUDA(ctx, cudaSetDevice(ctx->device));
    bool want = false;
    for (int32_t k = 0; observed_out && k < n_scores; k++) want = want || observed_out[k];
    // the counts come from one pass per group below, whichever path scored: the per-launch pass stays off meanwhile
    const bool hook = ctx->observed;
    ctx->observed = false;
    if (!want) {
        const int rc = score_multi(ctx, n_scores, rows, n_rows, offsets, scores_out, nloci_out, loci_out);
        ctx->observed = hook;
        return rc ? rc : zero_observed(ctx);
    }
    if (!ctx->ev_slab) NPC_CUDA(ctx, cudaEventCreateWithFlags(&ctx->ev_slab, cudaEventDisableTiming));
    std::vector<std::vector<npc_locus>> own((size_t)n_scores);                // records of definitions the caller does not take
    std::vector<npc_locus *> loci((size_t)n_scores);
    for (int32_t k = 0; k < n_scores; k++) {
        if (loci_out && loci_out[k]) loci[k] = loci_out[k];
        else { own[k].resize((size_t)n_rows[k]); loci[k] = own[k].data(); }
    }
    int rc = score_multi(ctx, n_scores, rows, n_rows, offsets, scores_out, nloci_out, loci.data());
    ctx->observed = hook;
    if (!rc) rc = multi_observed(ctx, n_scores, rows, n_rows, loci.data(), observed_out);
    return rc ? rc : zero_observed(ctx);
}

extern "C" int npc_score_resident_multi(npc_ctx *ctx, int32_t n_scores, const npc_row *const *rows, const int64_t *n_rows,
                                        const double *offsets, double *const *scores_out, int64_t *nloci_out,
                                        npc_locus *const *loci_out) {
    return npc_score_resident_multi_observed(ctx, n_scores, rows, n_rows, offsets, scores_out, nloci_out, loci_out, nullptr);
}

extern "C" int npc_set_observed(npc_ctx *ctx, int32_t on) {
    if (!ctx) return NPC_EINVAL;
    if (on && !ctx->d_obs) {
        NPC_CUDA(ctx, cudaSetDevice(ctx->device));
        const size_t bytes = (size_t)std::max<int64_t>(ctx->n, 1) * sizeof(ull);
        NPC_CUDA(ctx, cudaMalloc(&ctx->d_obs, bytes));
        NPC_CUDA(ctx, cudaMemsetAsync(ctx->d_obs, 0, bytes, ctx->stream));
    }
    ctx->observed = on != 0;
    return NPC_OK;
}

extern "C" int npc_observed(npc_ctx *ctx, int64_t *out) {
    if (!ctx || !out) return NPC_EINVAL;
    if (!ctx->d_obs) return fail(ctx, NPC_ESTATE, "npc_observed: npc_set_observed was never turned on for this context");
    NPC_CUDA(ctx, cudaSetDevice(ctx->device));
    if (ctx->n) NPC_CUDA(ctx, cudaMemcpyAsync(out, ctx->d_obs, ctx->n * sizeof(ull), cudaMemcpyDeviceToHost, ctx->stream));
    NPC_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return NPC_OK;
}

extern "C" int npc_partial(npc_ctx *ctx, double *sums_out, int64_t *nloci_out, npc_locus *loci_out, int64_t loci_cap,
                           int64_t *n_loci_out) {
    if (!ctx || !sums_out) return NPC_EINVAL;
    NPC_CUDA(ctx, cudaSetDevice(ctx->device));
    return copy_out(ctx, ctx->d_sums, sums_out, nloci_out, loci_out, loci_cap, n_loci_out);
}

extern "C" int npc_partial_device_ptr(npc_ctx *ctx, double **sums_dev, int64_t **nloci_dev) {
    if (!ctx) return NPC_EINVAL;
    if (sums_dev) *sums_dev = ctx->d_sums;
    if (nloci_dev) *nloci_dev = (int64_t *)ctx->d_nloci;
    return NPC_OK;
}

extern "C" void npc_normalise(double *sums, int64_t n, int64_t nloci, double offset) {
    // host mirror of k_finalize; volatile keeps the two roundings apart under any -ffp-contract
    const double denom = (double)nloci * 2.0;
    for (int64_t i = 0; i < n; i++) {
        volatile double q = sums[i] / denom;
        sums[i] = q + offset;
    }
}

// ---- several GPUs ---------------------------------------------------------------------------------

static int ensure_combine_buffers(npc_ctx *c) {
    if (!c->ev_reduce) NPC_CUDA(c, cudaEventCreateWithFlags(&c->ev_reduce, cudaEventDisableTiming));
    if (!c->d_nloci_total) NPC_CUDA(c, cudaMalloc(&c->d_nloci_total, sizeof(ull)));
    return NPC_OK;
}

extern "C" int npc_reduce(npc_ctx *const *ctxs, int32_t n_ctx, const double *offset, double *scores_out, int64_t *nloci_out) {
    if (!ctxs || n_ctx < 1 || !ctxs[0]) return NPC_EINVAL;
    npc_ctx *root = ctxs[0];
    if (n_ctx > REDUCE_MAX) return fail(root, NPC_EINVAL, "npc_reduce: too many contexts");
    for (int k = 0; k < n_ctx; k++) {
        if (!ctxs[k] || ctxs[k]->n != root->n) return fail(root, NPC_EINVAL, "npc_reduce: contexts must hold the same samples");
        for (int j = 0; j < k; j++) if (ctxs[j] == ctxs[k]) return fail(root, NPC_EINVAL, "npc_reduce: a context is listed twice");
    }
    ReduceParams P;
    memset(&P, 0, sizeof(P));
    P.n_parts = n_ctx; P.normalise = offset ? 1 : 0; P.offset = offset ? *offset : 0.0;
    // every context's partial sums are final when its stream reaches this point
    for (int k = 1; k < n_ctx; k++) {
        npc_ctx *c = ctxs[k];
        NPC_CUDA(c, cudaSetDevice(c->device));
        int rc = ensure_combine_buffers(c);
        if (rc) return rc;
        NPC_CUDA(c, cudaEventRecord(c->ev_reduce, c->stream));
    }
    NPC_CUDA(root, cudaSetDevice(root->device));
    int rc = ensure_combine_buffers(root);
    if (rc) return rc;
    int n_bridge = 0;
    std::vector<int> bridged(n_ctx, 0);
    for (int k = 1; k < n_ctx; k++) {
        npc_ctx *c = ctxs[k];
        NPC_CUDA(root, cudaStreamWaitEvent(root->stream, c->ev_reduce, 0));
        if (c->device == root->device) continue;
        int can = 0;
        NPC_CUDA(root, cudaDeviceCanAccessPeer(&can, root->device, c->device));
        if (can) {
            cudaError_t e = cudaDeviceEnablePeerAccess(c->device, 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
            else if (e != cudaSuccess) { cudaGetLastError(); can = 0; }
        }
        if (!can) bridged[k] = ++n_bridge;
    }
    const size_t nbytes = (size_t)std::max<int64_t>(root->n, 1) * sizeof(double);
    if (n_bridge && root->bridge_bytes < (size_t)n_bridge * (nbytes + 256)) {
        NPC_CUDA(root, cudaStreamSynchronize(root->stream));
        cudaFree(root->d_bridge); root->d_bridge = nullptr; root->bridge_bytes = 0;
        NPC_CUDA(root, cudaMalloc(&root->d_bridge, (size_t)n_bridge * (nbytes + 256)));
        root->bridge_bytes = (size_t)n_bridge * (nbytes + 256);
    }
    for (int k = 0; k < n_ctx; k++) {
        npc_ctx *c = ctxs[k];
        if (!bridged[k]) { P.part[k] = c->d_sums; P.nloci[k] = c->d_nloci; continue; }
        uint8_t *slot = (uint8_t *)root->d_bridge + (size_t)(bridged[k] - 1) * (nbytes + 256);      // [n doubles][nloci]
        NPC_CUDA(root, cudaMemcpyPeerAsync(slot, root->device, c->d_sums, c->device, (size_t)root->n * sizeof(double), root->stream));
        NPC_CUDA(root, cudaMemcpyPeerAsync(slot + nbytes, root->device, c->d_nloci, c->device, sizeof(ull), root->stream));
        P.part[k] = (const double *)slot; P.nloci[k] = (const ull *)(slot + nbytes);
    }
    const unsigned grid = (unsigned)std::min<int64_t>(std::max<int64_t>((root->n + 255) / 256, 1), 148 * 8);
    k_combine<<<grid, 256, 0, root->stream>>>(P, root->n, root->d_out, root->d_nloci_total);
    root->launches++;
    NPC_CUDA(root, cudaGetLastError());
    ull nl = 0;
    if (scores_out && root->n)
        NPC_CUDA(root, cudaMemcpyAsync(scores_out, root->d_out, (size_t)root->n * sizeof(double), cudaMemcpyDeviceToHost, root->stream));
    NPC_CUDA(root, cudaMemcpyAsync(&nl, root->d_nloci_total, sizeof(ull), cudaMemcpyDeviceToHost, root->stream));
    NPC_CUDA(root, cudaStreamSynchronize(root->stream));
    if (nloci_out) *nloci_out = (int64_t)nl;
    return NPC_OK;
}

extern "C" int npc_comm_unique_id(uint8_t *id128) {
    if (!id128) return NPC_EINVAL;
    if (!g_nccl.load()) { g_create_error = g_nccl.err; return NPC_EUNSUPPORTED; }
    NcclId id;
    const int r = g_nccl.GetUniqueId(&id);
    if (r) { g_create_error = std::string("ncclGetUniqueId: ") + g_nccl.GetErrorString(r); return NPC_ECUDA; }
    memcpy(id128, id.internal, 128);
    return NPC_OK;
}

extern "C" int npc_comm_init(npc_ctx *ctx, const uint8_t *id128, int32_t rank, int32_t world) {
    if (!ctx || !id128 || world < 1 || rank < 0 || rank >= world) return NPC_EINVAL;
    if (world > REDUCE_MAX) return fail(ctx, NPC_EINVAL, "npc_comm_init: too many ranks");
    if (!g_nccl.load()) return fail(ctx, NPC_EUNSUPPORTED, g_nccl.err.c_str());
    NPC_CUDA(ctx, cudaSetDevice(ctx->device));
    if (ctx->comm) { g_nccl.CommDestroy(ctx->comm); ctx->comm = nullptr; }
    NcclId id;
    memcpy(id.internal, id128, 128);
    const int r = g_nccl.CommInitRank(&ctx->comm, world, id, rank);
    if (r) { ctx->comm = nullptr; ctx->err = std::string("ncclCommInitRank: ") + g_nccl.GetErrorString(r); return NPC_ECUDA; }
    ctx->comm_rank = rank; ctx->comm_world = world;
    cudaFree(ctx->d_gather); ctx->d_gather = nullptr;
    NPC_CUDA(ctx, cudaMalloc(&ctx->d_gather, (size_t)world * (size_t)std::max<int64_t>(ctx->n, 1) * sizeof(double)));
    return ensure_combine_buffers(ctx);
}

extern "C" int npc_comm_combine(npc_ctx *ctx, const double *offset, double *scores_out, int64_t *nloci_out) {
    if (!ctx) return NPC_EINVAL;
    if (!ctx->comm) return fail(ctx, NPC_ESTATE, "npc_comm_combine: npc_comm_init was not called");
    NPC_CUDA(ctx, cudaSetDevice(ctx->device));
    const int W = ctx->comm_world;
    int r = 0;
    if (ctx->n) r = g_nccl.AllGather(ctx->d_sums, ctx->d_gather, (size_t)ctx->n, NCCL_FLOAT64, ctx->comm, ctx->stream);
    if (!r) r = g_nccl.AllReduce(ctx->d_nloci, ctx->d_nloci_total, 1, NCCL_UINT64, NCCL_SUM, ctx->comm, ctx->stream);
    if (r) { ctx->err = std::string("NCCL: ") + g_nccl.GetErrorString(r); return NPC_ECUDA; }
    ReduceParams P;
    memset(&P, 0, sizeof(P));
    P.n_parts = W; P.normalise = offset ? 1 : 0; P.offset = offset ? *offset : 0.0;
    for (int k = 0; k < W; k++) P.part[k] = ctx->d_gather + (size_t)k * ctx->n;
    // nloci: the all-reduced total lives in d_nloci_total; the kernel reads it as a one-element "shard" list
    P.n_parts = W;
    k_combine_total<<<(unsigned)std::min<int64_t>(std::max<int64_t>((ctx->n + 255) / 256, 1), 148 * 8), 256, 0, ctx->stream>>>(
        P, ctx->n, ctx->d_out, ctx->d_nloci_total);
    ctx->launches++;
    NPC_CUDA(ctx, cudaGetLastError());
    if (!scores_out && !nloci_out) return NPC_OK;                        // asynchronous: results stay on the device (npc_combined_device_ptr)
    ull nl = 0;
    if (scores_out && ctx->n)
        NPC_CUDA(ctx, cudaMemcpyAsync(scores_out, ctx->d_out, (size_t)ctx->n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    NPC_CUDA(ctx, cudaMemcpyAsync(&nl, ctx->d_nloci_total, sizeof(ull), cudaMemcpyDeviceToHost, ctx->stream));
    NPC_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (nloci_out) *nloci_out = (int64_t)nl;
    return NPC_OK;
}

extern "C" int npc_comm_sum_counts(npc_ctx *ctx, int64_t *counts_dev, int64_t n_rows) {
    if (!ctx || !counts_dev || n_rows < 0) return NPC_EINVAL;
    if (!ctx->comm) return fail(ctx, NPC_ESTATE, "npc_comm_sum_counts: npc_comm_init was not called");
    NPC_CUDA(ctx, cudaSetDevice(ctx->device));
    if (n_rows == 0) return NPC_OK;
    const int r = g_nccl.AllReduce(counts_dev, counts_dev, (size_t)n_rows * 2, NCCL_UINT64, NCCL_SUM, ctx->comm, ctx->stream);
    if (r) { ctx->err = std::string("NCCL: ") + g_nccl.GetErrorString(r); return NPC_ECUDA; }
    return NPC_OK;
}

extern "C" int npc_combined_device_ptr(npc_ctx *ctx, double **scores_dev, int64_t **nloci_dev) {
    if (!ctx) return NPC_EINVAL;
    NPC_CUDA(ctx, cudaSetDevice(ctx->device));
    int rc = ensure_combine_buffers(ctx);
    if (rc) return rc;
    if (scores_dev) *scores_dev = ctx->d_out;
    if (nloci_dev) *nloci_dev = (int64_t *)ctx->d_nloci_total;
    return NPC_OK;
}

extern "C" int npc_synth_fill_device(npc_ctx *ctx, void *gt_dev, int64_t row_stride, int64_t v0, int64_t n_rows,
                                     uint64_t seed, const uint32_t *af_thr16_dev, const uint32_t *miss_thr24_dev,
                                     const int32_t *alt_code_dev) {
    if (!ctx || !gt_dev || ((uintptr_t)gt_dev & 15) || (row_stride & 15) || row_stride < ctx->n * 2 || n_rows < 0)
        return ctx ? fail(ctx, NPC_EINVAL, "npc_synth_fill_device: bad slab") : NPC_EINVAL;
    if (ctx->width != 1 || ctx->ploidy != 2) return fail(ctx, NPC_EUNSUPPORTED, "synthetic cohort is int8 diploid");
    NPC_CUDA(ctx, cudaSetDevice(ctx->device));
    const int64_t nchunks = (ctx->n + 7) / 8;
    const unsigned gx = (unsigned)std::min<int64_t>(std::max<int64_t>((nchunks + 255) / 256, 1), 4096);
    for (int64_t r0 = 0; r0 < n_rows; r0 += 65535) {
        const int64_t nr = std::min<int64_t>(65535, n_rows - r0);
        k_synth<<<dim3(gx, (unsigned)nr), 256, 0, ctx->stream>>>((uint8_t *)gt_dev + r0 * row_stride, row_stride, ctx->n,
                                                                v0 + r0, seed, af_thr16_dev + r0, miss_thr24_dev + r0,
                                                                alt_code_dev + r0);
        ctx->launches++;
        NPC_CUDA(ctx, cudaGetLastError());
    }
    return NPC_OK;
}
