// npc_observed.cuh -- per sample, the scored loci that used the sample's own genotype (DESIGN.md 4.13).
//
// NOT IN THE REFERENCE, whose output is `sample<TAB>score`.  observed[s] counts the score rows whose locus record has class
// OK (klass 0, used 1) and at which sample s is called, with multiplicity: a sample is called exactly when the layout's
// tally does not count it in nmiss.  Rows of the other classes never count: their dosage is the locus constant.
//
// The pass runs after a launch's scoring sequence, on the same stream, and only when asked for (npc_set_observed,
// npc_score_resident_multi_observed).  It reads each entry's slab row once per launch with the access pattern of the
// layout's accumulate kernel: a thread owns L::P samples of every row (one 16-byte streaming load; 2 bytes of a .bed
// row; one sample of a generic GT row) and adds called(row, s) x w[g][entry] into integer registers for the G
// definitions of a group.  Entries are staged in shared memory OBS_RB at a time, OBS_U loads in flight per thread;
// gridDim.y splits the entries, and every CTA adds its registers into the 64-bit counts with atomics -- integers, so
// the result does not depend on the split or the order.
//
// Weights: w[g * n_ent + e], or, when w is NULL (a group of one), 1 for an entry whose record log[e] is OK, else 0.
// An entry no definition weighs is not read.  A thread's counters hold one CTA's share of a launch: less than 2^32
// as long as a definition has fewer than 2^32 score rows.
#pragma once
#include "npc_kernels.cuh"
#include "npc_bed.cuh"
#include "npc_dose255.cuh"
#include "npc_dose32.cuh"
#include "npc_dosage.cuh"
#include "npc_pl.cuh"

namespace npc {

constexpr int OBS_G = 8;                          // definitions per launch of a group: 8 x 8 counters per thread on int8 rows, no spills
constexpr int OBS_THREADS = 128;
constexpr int OBS_RB = 32;                        // entries staged per batch
constexpr int OBS_U = 4;                          // loads in flight per thread

// Each layout type: P samples per thread, Ctx made once per entry from its slab row and npc_row, load() of thread t's
// share of a row, called() -> bit k set when sample P t + k is called.  TAB: the FORMAT/PL weight table in shared memory.
struct NoCtx {};

struct ObsI8x2 {                                  // int8 diploid GT: the tally's fast chunks, else its exact decode
    static constexpr int P = 8;
    static constexpr bool TAB = false;
    using Ctx = NoCtx;
    using Word = uint4;
    __device__ static Ctx make(const uint8_t *, const npc_row &) { return {}; }
    __device__ static Word load(const uint8_t *row, int64_t t, int) { return ldg_stream(reinterpret_cast<const uint4 *>(row) + t); }
    __device__ static uint32_t called(const Word &w, const Ctx &, const double *) {
        const uint32_t ww[4] = { w.x, w.y, w.z, w.w };
        uint32_t m = 0;
        if (chunk_is_fast(w)) {
            // every byte < 16: an allele is missing when its code bits (pack_idx8) are 0; called = both bytes of a sample non-zero
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const uint32_t c = ww[k] & 0x0E0E0E0Eu;
                const uint32_t nz = (c + 0x7F7F7F7Fu) & 0x80808080u;
                const uint32_t both = nz & (nz >> 8);
                m |= ((both >> 7) & 1u) << (2 * k) | ((both >> 23) & 1u) << (2 * k + 1);
            }
        } else {
#pragma unroll
            for (int k = 0; k < 8; k++) {
                const uint32_t h = (ww[k >> 1] >> ((k & 1) * 16)) & 0xFFFFu;
                m |= (uint32_t)(slow_off8(h, 0) != (64u + 3u) * 8u) << k;
            }
        }
        return m;
    }
};

template <typename T>
struct ObsGT {                                    // GT rows of any width and ploidy: decode_sample, one sample per thread
    static constexpr int P = 1;
    static constexpr bool TAB = false;
    using Ctx = NoCtx;
    using Word = uint32_t;
    __device__ static Ctx make(const uint8_t *, const npc_row &) { return {}; }
    __device__ static Word load(const uint8_t *row, int64_t t, int ploidy) {
        int d; bool miss;
        decode_sample<T>(reinterpret_cast<const T *>(row) + t * ploidy, ploidy, 0, d, miss);
        return miss ? 0u : 1u;
    }
    __device__ static uint32_t called(const Word &w, const Ctx &, const double *) { return w; }
};

struct ObsBed {                                   // .bed: any code but 01; 8 samples = 16 bits, as k_accum_bed reads them
    static constexpr int P = 8;
    static constexpr bool TAB = false;
    using Ctx = NoCtx;
    using Word = uint32_t;
    __device__ static Ctx make(const uint8_t *, const npc_row &) { return {}; }
    __device__ static Word load(const uint8_t *row, int64_t t, int) { return __ldg(reinterpret_cast<const uint16_t *>(row) + t); }
    __device__ static uint32_t called(const Word &w, const Ctx &, const double *) {
        const uint32_t lo = w & 0x5555u, hi = (w >> 1) & 0x5555u;
        const uint32_t c = ~(lo & ~hi) & 0x5555u;                          // bit 2k: sample k is not 01
        uint32_t m = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) m |= ((c >> (2 * k)) & 1u) << k;
        return m;
    }
};

struct ObsDose255 {                               // BGEN 2-byte rows: k <= D255_MAX
    static constexpr int P = 8;
    static constexpr bool TAB = false;
    using Ctx = NoCtx;
    using Word = uint4;
    __device__ static Ctx make(const uint8_t *, const npc_row &) { return {}; }
    __device__ static Word load(const uint8_t *row, int64_t t, int) { return ldg_stream(reinterpret_cast<const uint4 *>(row) + t); }
    __device__ static uint32_t called(const Word &w, const Ctx &, const double *) {
        const uint32_t ww[4] = { w.x, w.y, w.z, w.w };
        uint32_t m = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) m |= (uint32_t)(((ww[k >> 1] >> ((k & 1) * 16)) & 0xFFFFu) <= D255_MAX) << k;
        return m;
    }
};

struct ObsDose32 {                                // BGEN 32-bit rows: d32_sample with the row's D
    static constexpr int P = 4;
    static constexpr bool TAB = false;
    struct Ctx { uint32_t D; };
    using Word = uint4;
    __device__ static Ctx make(const uint8_t *row, const npc_row &) { return { d32_den(row) }; }
    __device__ static Word load(const uint8_t *row, int64_t t, int) {
        return ldg_stream(reinterpret_cast<const uint4 *>(row + Dose32::HEADER) + t);
    }
    __device__ static uint32_t called(const Word &w, const Ctx &c, const double *) {
        const uint32_t ww[4] = { w.x, w.y, w.z, w.w };
        uint32_t m = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) { uint32_t kk; m |= (uint32_t)d32_sample(ww[k], c.D, false, kk) << k; }
        return m;
    }
};

struct ObsDs {                                    // FORMAT/DS: not missing, not vector_end, not NaN
    static constexpr int P = 4;
    static constexpr bool TAB = false;
    using Ctx = NoCtx;
    using Word = uint4;
    __device__ static Ctx make(const uint8_t *, const npc_row &) { return {}; }
    __device__ static Word load(const uint8_t *row, int64_t t, int) { return ldg_stream(reinterpret_cast<const uint4 *>(row) + t); }
    __device__ static uint32_t called(const Word &w, const Ctx &, const double *) {
        const uint32_t ww[4] = { w.x, w.y, w.z, w.w };
        uint32_t m = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) m |= (uint32_t)!ds_missing(ww[k]) << k;
        return m;
    }
};

struct ObsPl {                                    // FORMAT/PL: den > 0 at the entry's eaf and effect allele
    static constexpr int P = 4;
    static constexpr bool TAB = true;
    struct Ctx { PlPrior pr; int32_t alt, ok; };
    using Word = uint4;
    __device__ static Ctx make(const uint8_t *, const npc_row &r) {
        Ctx c;
        c.alt = r.eaidx != 0;
        c.ok = pl_prior(r.eaf, c.alt != 0, c.pr);
        return c;
    }
    __device__ static Word load(const uint8_t *row, int64_t t, int) { return ldg_stream(reinterpret_cast<const uint4 *>(row) + t); }
    __device__ static uint32_t called(const Word &w, const Ctx &c, const double *tab) {
        if (!c.ok) return 0u;
        const uint32_t ww[4] = { w.x, w.y, w.z, w.w };
        uint32_t m = 0;
#pragma unroll
        for (int k = 0; k < 4; k++) { double d; m |= (uint32_t)pl_dosage(ww[k], tab, c.pr, c.alt != 0, d) << k; }
        return m;
    }
};

// out[g * n + s] += sum over entries e of this CTA's share of called(e, s) x weight(g, e); entries [y * per_y, (y + 1) * per_y)
template <class L, int G>
__global__ void __launch_bounds__(OBS_THREADS)
k_observed(const uint8_t *__restrict__ gt, int64_t row_stride, int ploidy, const npc_row *__restrict__ ent,
           const npc_locus *__restrict__ log, const uint32_t *__restrict__ w, int64_t n_ent, int64_t per_y, int64_t n,
           ull *__restrict__ out) {
    __shared__ double s_tab[L::TAB ? PL_TN + 1 : 1];
    __shared__ typename L::Ctx s_ctx[OBS_RB];
    __shared__ uint32_t s_w[OBS_RB][G];
    __shared__ int32_t s_row[OBS_RB];
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool active = t < (n + L::P - 1) / L::P;
    uint32_t cnt[G][L::P];
#pragma unroll
    for (int g = 0; g < G; g++)
#pragma unroll
        for (int k = 0; k < L::P; k++) cnt[g][k] = 0;
    if (L::TAB) pl_load_table(s_tab);
    const int64_t e_begin = (int64_t)blockIdx.y * per_y, e_end = min(n_ent, e_begin + per_y);
    for (int64_t e0 = e_begin; e0 < e_end; e0 += OBS_RB) {
        const int nb = (int)min((int64_t)OBS_RB, e_end - e0);
        __syncthreads();
        if (threadIdx.x < nb) {
            const int64_t e = e0 + threadIdx.x;
            const npc_row r = ent[e];
            uint32_t any = 0;
#pragma unroll
            for (int g = 0; g < G; g++) {
                const uint32_t wt = w ? w[g * n_ent + e] : (uint32_t)(log[e].klass == 0 && log[e].used);
                s_w[threadIdx.x][g] = wt;
                any |= wt;
            }
            const bool read = any && r.kind == NPC_KIND_GT && r.gt_row >= 0;
            s_row[threadIdx.x] = read ? r.gt_row : -1;
            if (read) s_ctx[threadIdx.x] = L::make(gt + (int64_t)r.gt_row * row_stride, r);
        }
        __syncthreads();
        if (!active) continue;
        for (int u0 = 0; u0 < nb; u0 += OBS_U) {
            typename L::Word wd[OBS_U];
#pragma unroll
            for (int u = 0; u < OBS_U; u++) {
                const int g = u0 + u < nb ? s_row[u0 + u] : -1;
                if (g >= 0) wd[u] = L::load(gt + (int64_t)g * row_stride, t, ploidy);
            }
#pragma unroll
            for (int u = 0; u < OBS_U; u++) {
                if (u0 + u >= nb) break;
                if (s_row[u0 + u] < 0) continue;                                  // block-uniform
                const uint32_t m = L::called(wd[u], s_ctx[u0 + u], s_tab);
#pragma unroll
                for (int g = 0; g < G; g++) {
                    const uint32_t wt = s_w[u0 + u][g];
#pragma unroll
                    for (int k = 0; k < L::P; k++) cnt[g][k] += wt & (0u - ((m >> k) & 1u));
                }
            }
        }
    }
    if (!active) return;
#pragma unroll
    for (int g = 0; g < G; g++)
#pragma unroll
        for (int k = 0; k < L::P; k++) {
            const int64_t s = t * L::P + k;
            if (s < n && cnt[g][k]) atomicAdd(&out[(int64_t)g * n + s], (ull)cnt[g][k]);
        }
}

}  // namespace npc
