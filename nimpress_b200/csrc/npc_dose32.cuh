// npc_dose32.cuh -- 32-bit fixed-point dosage rows from BGEN v1.2 files at any bit depth (DESIGN.md 4.9).
//
// NOT IN THE REFERENCE, which reads VCF / BCF hard calls only.  At B bits per probability (1..16) a BGEN dosage is an
// exact rational with denominator D = 2^B - 1.  The host writes each matched block as one row: a 16-byte header (uint32
// D, 12 bytes of zero), then one little-endian uint32 word per sample:
//
//   bits 0-23   k = D x the expected ALT dosage        bits 24-25   ploidy p (1 or 2)        bit 31   missing
//
// A sample is called when bit 31 is clear, p is 1 or 2 and k <= p*D; any other word is a missing sample (the host writes
// 0xFFFFFFFF).  Then, as for NPC_GT_DOSE255 rows (npc_dose255.cuh):
//
//   raw dosage   k' = k (effect allele = ALT, eaidx 1) or p*D - k (effect allele = REF, eaidx 0); dosage fl(k'/D)
//   tally        nmiss and neff_num = sum of k' over called samples, both exact integers (64-bit atomics: the result
//                does not depend on the order of the adds).  neff = fl(neff_num / D) goes to decide_row_real unchanged;
//                the locus record reports neff_num, in units of 1/D of its row.
//   accumulate   scores[s] = fl(scores[s] + fl(fl(k'/D) * beta)) (cm for a missing sample, c0 for a constant row), rows
//                in score-row order: the reference's chain in every mode.
//
// fl(k'/D) is the only place the accumulate pass turns k' into a dosage (d32_quot).  A table of it, as npc_dose255.cuh
// keeps, would take 131,071 entries at D = 65,535, so it is computed: q0 = fl(k' r) with r = fl(1/D), the exact residual
// e = k' - q0 D by one FMA, q = fl(q0 + e r) by another.  That equals the correctly rounded k'/D for every k' in 0..2D
// and every B in 1..16 (tests/test_bgen_bits_gpu.py checks all 262,124 of them on the device).
//
// With D = 255 and diploid samples these rows score bit for bit as the same NPC_GT_DOSE255 rows; hard calls (k' = 0, D,
// 2D) score bit for bit as the same genotypes in int8 GT rows in exact order, haploid samples included.
//
// Both passes read the row: 4 B per genotype each, 8 B in all.  A thread of the accumulate pass owns 4 samples (one
// 16-byte load per row) and keeps their sums in fp64 registers across the launch; the loads of the next batch of D32_RB
// rows are issued before the current batch is added.
#pragma once
#include "npc_kernels.cuh"

namespace npc {

constexpr int D32_THREADS = 128;                  // accumulate pass: threads per CTA (4 samples each)
constexpr int D32_RB = 8;                         // rows per batch

// The row's D, from its header.
__device__ __forceinline__ uint32_t d32_den(const uint8_t *__restrict__ row) {
    return __ldg(reinterpret_cast<const uint32_t *>(row));
}

// One sample word -> k' (eaidx 0: p*D - k); false for a missing sample.
__device__ __forceinline__ bool d32_sample(uint32_t w, uint32_t D, bool ref, uint32_t &kk) {
    const uint32_t p = (w >> 24) & 3u, k = w & 0xFFFFFFu;
    kk = ref ? p * D - k : k;
    return !(w >> 31) && (p == 1u || p == 2u) && k <= p * D;
}

// fl(k'/D), correctly rounded, for integers 0 <= k' <= 2D < 2^17; r = fl(1/D).
__device__ __forceinline__ double d32_quot(uint32_t kk, double D, double r) {
    const double k = (double)kk;
    const double q0 = __dmul_rn(k, r);
    const double e = __fma_rn(-q0, D, k);                                  // exact: q0 is within an ulp of k'/D
    return __fma_rn(e, r, q0);
}

// The layout type of k_count_chunks and k_decide (npc_kernels.cuh).
struct Dose32 {
    static constexpr int PER16 = 4, HEADER = 16;  // samples per 16-byte word, bytes before the first sample word

    // tallyAlleles (:32-47) with D and the flip from the row.  Per thread: tally_grid_y gives a thread at most 64 chunks,
    // 256 samples x 2 x 65,535 < 2^25; a warp's sum of ne can pass 2^32, which k_count_chunks' 64-bit reduction holds.
    struct Count {
        uint32_t D;
        bool ref;
        __device__ Count(const uint8_t *row, const npc_row &r) : D(d32_den(row)), ref(r.eaidx == 0) {}
        __device__ void operator()(const uint4 &w, int64_t left, uint32_t &nm, uint32_t &ne) const {
            const int valid = (int)min((int64_t)4, left);
            const uint32_t ww[4] = { w.x, w.y, w.z, w.w };
#pragma unroll
            for (int k = 0; k < 4; k++) {
                if (k >= valid) break;
                uint32_t kk;
                if (d32_sample(ww[k], D, ref, kk)) ne += kk;
                else nm++;
            }
        }
    };

    // The common decision on the integer tallies: neff = fl(neff_num / D), the record reports neff_num.  RowP::pad carries
    // the row's D to the accumulate pass.
    struct Tally : RowTally {
        uint32_t D;
        __device__ Tally(const TallyIn &in, const npc_row &row, int64_t r) {
            D = row.kind == NPC_KIND_GT && row.gt_row >= 0 ? d32_den(in.gt + (int64_t)row.gt_row * in.row_stride) : 1u;
            const ull num = in.counts[2 * r + 1];
            nmiss = in.counts[2 * r]; neff = __ddiv_rn((double)num, (double)D); neff_rec = (long long)num;
        }
        __device__ void extra(const npc_row &, RowP &out) const { out.pad = (int32_t)D; }
    };
};

// Staged per row: mode word (0 dropped, 1 constant, 2 decode with k' = k, 3 decode with k' = p*D - k), beta (c0 for a
// constant row), cm and D; the slab row of every row whose loads go out (-1: not read).
__device__ __forceinline__ void d32_stage(const RowP *__restrict__ rowp, int64_t r, int64_t n_rows, int32_t &mode,
                                          double &beta, double &cm, uint32_t &D) {
    mode = 0; beta = 0.0; cm = 0.0; D = 1;
    if (r >= n_rows) return;
    const RowP &rp = rowp[r];
    if (rp.mode == MODE_CONST) { mode = 1; beta = rp.c0; }
    else if (rp.mode == MODE_DECODE) { mode = rp.eaidx == 0 ? 3 : 2; beta = rp.beta; cm = rp.cm; D = (uint32_t)rp.pad; }
}
__device__ __forceinline__ int32_t d32_off(const RowP *__restrict__ rowp, int64_t r, int64_t n_rows) {
    return r < n_rows && rowp[r].mode == MODE_DECODE ? rowp[r].gt_row : -1;
}

// Loop of batch b: the loads of batch b + 1 go out first (their slab rows wait in shared memory), then this thread's
// share of batch b + 1's row words and batch b + 2's slab rows is fetched into registers, batch b is added, the
// fetched share is stored to the other buffer, one barrier -- the scheme of k_accum_dose255.
__global__ void __launch_bounds__(D32_THREADS, 4)
k_accum_dose32(const uint8_t *__restrict__ gt, int64_t row_stride, const RowP *__restrict__ rowp, int64_t n_rows, int64_t n,
               double *__restrict__ sums) {
    __shared__ double s_beta[2][D32_RB], s_cm[2][D32_RB], s_rcp[2][D32_RB];
    __shared__ uint32_t s_den[2][D32_RB];
    __shared__ int32_t s_mode[2][D32_RB], s_off[2][D32_RB];
    const int64_t n_batches = (n_rows + D32_RB - 1) / D32_RB;
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;    // owns samples 4t .. 4t+3
    const int64_t nw = (n + 3) >> 2;
    const bool active = t < nw;
    const int valid = active ? (int)min((int64_t)4, n - t * 4) : 0;
    double acc[4];
#pragma unroll
    for (int k = 0; k < 4; k++) acc[k] = k < valid ? sums[t * 4 + k] : 0.0;
    const uint4 *col = reinterpret_cast<const uint4 *>(gt + Dose32::HEADER) + (active ? t : 0);
    const int64_t stride16 = row_stride >> 4;
    if (threadIdx.x < D32_RB) {
        uint32_t D;
        d32_stage(rowp, threadIdx.x, n_rows, s_mode[0][threadIdx.x], s_beta[0][threadIdx.x], s_cm[0][threadIdx.x], D);
        s_den[0][threadIdx.x] = D; s_rcp[0][threadIdx.x] = __drcp_rn((double)D);
        s_off[0][threadIdx.x] = d32_off(rowp, threadIdx.x, n_rows);
        s_off[1][threadIdx.x] = d32_off(rowp, D32_RB + threadIdx.x, n_rows);
    }
    __syncthreads();
    uint4 w[D32_RB], wn[D32_RB];
#pragma unroll
    for (int u = 0; u < D32_RB; u++) {
        const int g = s_off[0][u];
        w[u] = g >= 0 && active ? ldg_stream(col + (int64_t)g * stride16) : make_uint4(0, 0, 0, 0);
    }
    for (int64_t b = 0; b < n_batches; b++) {
        const int cur = (int)(b & 1), nxt = cur ^ 1;
        const bool more = b + 1 < n_batches;
#pragma unroll
        for (int u = 0; u < D32_RB; u++) {
            const int g = more ? s_off[nxt][u] : -1;
            wn[u] = g >= 0 && active ? ldg_stream(col + (int64_t)g * stride16) : make_uint4(0, 0, 0, 0);
        }
        int32_t mn = 0, on = -1;
        double bn = 0.0, cn = 0.0;
        uint32_t dn = 1;
        if (threadIdx.x < D32_RB) {
            d32_stage(rowp, (b + 1) * D32_RB + threadIdx.x, n_rows, mn, bn, cn, dn);
            on = d32_off(rowp, (b + 2) * D32_RB + threadIdx.x, n_rows);
        }
#pragma unroll
        for (int u = 0; u < D32_RB; u++) {
            const int mode = s_mode[cur][u];                                    // warp-uniform
            if (mode == 1) {
                const double c = s_beta[cur][u];
#pragma unroll
                for (int k = 0; k < 4; k++) acc[k] = __dadd_rn(acc[k], c);
            } else if (mode >= 2) {
                const double beta = s_beta[cur][u], cm = s_cm[cur][u], r = s_rcp[cur][u];
                const uint32_t D = s_den[cur][u];
                const double Dd = (double)D;
                const uint32_t ww[4] = { w[u].x, w[u].y, w[u].z, w[u].w };
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    uint32_t kk;
                    const bool called = d32_sample(ww[k], D, mode == 3, kk);
                    const double c = __dmul_rn(d32_quot(kk, Dd, r), beta);
                    acc[k] = __dadd_rn(acc[k], called ? c : cm);
                }
            }
        }
        if (threadIdx.x < D32_RB) {
            s_mode[nxt][threadIdx.x] = mn; s_beta[nxt][threadIdx.x] = bn; s_cm[nxt][threadIdx.x] = cn;
            s_den[nxt][threadIdx.x] = dn; s_rcp[nxt][threadIdx.x] = __drcp_rn((double)dn);
            s_off[cur][threadIdx.x] = on;                                      // batch b + 2 uses buffer (b + 2) & 1 = cur
        }
        __syncthreads();
#pragma unroll
        for (int u = 0; u < D32_RB; u++) w[u] = wn[u];
    }
#pragma unroll
    for (int k = 0; k < 4; k++)
        if (k < valid) sums[t * 4 + k] = acc[k];
}

}  // namespace npc
