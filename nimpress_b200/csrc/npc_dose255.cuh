// npc_dose255.cuh -- fixed-point dosage rows from BGEN v1.2 files (DESIGN.md 4.8).
//
// NOT IN THE REFERENCE, which reads VCF / BCF hard calls only.  The host inflates a matched BGEN genotype block and
// writes, per sample, k = 255 x the expected ALT dosage as a little-endian uint16 (0..510; above 510 = missing, the
// host writes 0xFFFF).  At 8 bits per probability that dosage is an exact rational with denominator 255, so:
//
//   raw dosage   k' = k (effect allele = ALT, eaidx 1) or 510 - k (effect allele = REF, eaidx 0); dosage fl(k'/255)
//   tally        nmiss and neff_num = sum of k' over called samples, both exact integers (64-bit atomics: the result
//                does not depend on the order of the adds).  The reference's real tally is neff = fl(neff_num / 255),
//                and decide_row_real takes it unchanged, so --maxmis, the locus constants and the imputed dosage
//                fl(neff / ngt) are what they are for every other row.  The locus record reports neff_num.
//   accumulate   scores[s] = fl(scores[s] + fl(fl(k'/255) * beta)) (cm for a missing sample, c0 for a constant row),
//                rows in score-row order: the reference's chain (:639-640) in every mode.  The running sums stay in
//                d_sums across launches, so launch cuts and staging blocks give the same bits.
//
// fl(k/255) is exactly 0, 1 and 2 for k = 0, 255 and 510, and fl(255 x / 255) = x for an integer x below 2^53, so a
// file of hard calls scores bit for bit as the same genotypes in int8 GT rows in exact order.
//
// Both passes read the row: 2 B per genotype each, 4 B in all.  A thread of the accumulate pass owns 8 samples (one
// 16-byte load per row) and keeps their sums in fp64 registers across the launch; the loads of the next batch of
// D255_RB rows are issued before the current batch is added.  Per genotype: one shared-memory lookup of fl(k'/255),
// one DMUL and one DADD.
#pragma once
#include "npc_kernels.cuh"

namespace npc {

constexpr int D255_THREADS = 128;                 // accumulate pass: threads per CTA (8 samples each)
constexpr int D255_RB = 8;                        // rows per batch
constexpr uint32_t D255_MAX = 510;                // 255 x the largest dosage; anything above is a missing sample

// tallyAlleles (:32-47) on dosage rows: one 16-byte load = 8 samples, four in flight per thread.
__global__ void __launch_bounds__(256)
k_count_dose255(const uint8_t *__restrict__ gt, int64_t row_stride, const npc_row *__restrict__ rows, int64_t n,
                ull *__restrict__ counts) {
    const int r = blockIdx.x;
    const npc_row row = rows[r];
    if (row.kind != NPC_KIND_GT || row.gt_row < 0) return;
    __shared__ ull s_m, s_e;
    if (threadIdx.x == 0) { s_m = 0; s_e = 0; }
    __syncthreads();
    const uint4 *base = reinterpret_cast<const uint4 *>(gt + (int64_t)row.gt_row * row_stride);
    const int64_t nchunks = (n + 7) >> 3;
    const uint32_t flip = row.eaidx == 0 ? D255_MAX : 0u;            // k' = |k - flip|
    uint32_t nm = 0, ne = 0;         // per thread: tally_grid_y gives a thread at most 64 chunks, 512 samples x 510
    constexpr int U = 4;
    for (int64_t c0 = (int64_t)blockIdx.y * blockDim.x * U + threadIdx.x; c0 < nchunks; c0 += (int64_t)gridDim.y * blockDim.x * U) {
        uint4 wv[U];
#pragma unroll
        for (int u = 0; u < U; u++) {
            const int64_t c = c0 + (int64_t)u * blockDim.x;
            wv[u] = c < nchunks ? ldg_stream(base + c) : make_uint4(0, 0, 0, 0);
        }
#pragma unroll
        for (int u = 0; u < U; u++) {
            const int64_t c = c0 + (int64_t)u * blockDim.x;
            if (c >= nchunks) break;
            const int valid = (int)min((int64_t)8, n - c * 8);
            const uint32_t ww[4] = { wv[u].x, wv[u].y, wv[u].z, wv[u].w };
#pragma unroll
            for (int k = 0; k < 8; k++) {
                if (k >= valid) break;
                const uint32_t v = (ww[k >> 1] >> ((k & 1) * 16)) & 0xFFFFu;
                if (v > D255_MAX) nm++;
                else ne += (uint32_t)abs((int)v - (int)flip);
            }
        }
    }
    const ull m64 = __reduce_add_sync(0xffffffffu, nm), e64 = __reduce_add_sync(0xffffffffu, ne);
    if ((threadIdx.x & 31) == 0) { atomicAdd(&s_m, m64); atomicAdd(&s_e, e64); }
    __syncthreads();
    if (threadIdx.x == 0) { atomicAdd(&counts[2 * r], s_m); atomicAdd(&counts[2 * r + 1], s_e); }
}

// The common decision on the integer tallies: neff = fl(neff_num / 255), the record reports neff_num.
__global__ void __launch_bounds__(128)
k_decide_dose255(const npc_row *__restrict__ rows, int64_t n_rows, const ull *__restrict__ counts, Policy p,
                 int64_t n_local, RowP *__restrict__ rowp, npc_locus *__restrict__ log, ull *__restrict__ nloci) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int used = 0;
    if (r < n_rows) {
        RowP out; npc_locus rec;
        const ull num = counts[2 * r + 1];
        decide_row_real(p, rows[r], counts[2 * r], __ddiv_rn((double)num, 255.0), (long long)num, n_local, out, rec);
        rowp[r] = out;
        log[r] = rec;
        used = rec.used;
    }
    used = __reduce_add_sync(0xffffffffu, used);
    if ((threadIdx.x & 31) == 0 && used) atomicAdd(nloci, (ull)used);
}

// Staged per row: mode word (0 dropped, 1 constant, 2 decode with k' = k, 3 decode with k' = 510 - k), beta (c0 for a
// constant row) and cm; the slab row of every row whose loads go out (-1: not read).
__device__ __forceinline__ void d255_stage(const RowP *__restrict__ rowp, int64_t r, int64_t n_rows, int32_t &mode,
                                           double &beta, double &cm) {
    mode = 0; beta = 0.0; cm = 0.0;
    if (r >= n_rows) return;
    const RowP &rp = rowp[r];
    if (rp.mode == MODE_CONST) { mode = 1; beta = rp.c0; }
    else if (rp.mode == MODE_DECODE) { mode = rp.eaidx == 0 ? 3 : 2; beta = rp.beta; cm = rp.cm; }
}
__device__ __forceinline__ int32_t d255_off(const RowP *__restrict__ rowp, int64_t r, int64_t n_rows) {
    return r < n_rows && rowp[r].mode == MODE_DECODE ? rowp[r].gt_row : -1;
}

// Loop of batch b: the loads of batch b + 1 go out first (their slab rows wait in shared memory), then this thread's
// share of batch b + 1's row words and batch b + 2's slab rows is fetched into registers, batch b is added, the
// fetched share is stored to the other buffer, one barrier -- the scheme of k_accum_bed.
__global__ void __launch_bounds__(D255_THREADS, 4)
k_accum_dose255(const uint8_t *__restrict__ gt, int64_t row_stride, const RowP *__restrict__ rowp, int64_t n_rows, int64_t n,
                double *__restrict__ sums) {
    __shared__ double s_d[512];                                           // fl(k/255), k = 0..510 (entry 511 unused)
    __shared__ double s_beta[2][D255_RB], s_cm[2][D255_RB];
    __shared__ int32_t s_mode[2][D255_RB], s_off[2][D255_RB];
    const int64_t n_batches = (n_rows + D255_RB - 1) / D255_RB;
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;    // owns samples 8t .. 8t+7
    const int64_t nw = (n + 7) >> 3;
    const bool active = t < nw;
    const int valid = active ? (int)min((int64_t)8, n - t * 8) : 0;
    double acc[8];
#pragma unroll
    for (int k = 0; k < 8; k++) acc[k] = k < valid ? sums[t * 8 + k] : 0.0;
    const uint4 *col = reinterpret_cast<const uint4 *>(gt) + (active ? t : 0);
    const int64_t stride16 = row_stride >> 4;
    for (int i = threadIdx.x; i < 512; i += D255_THREADS) s_d[i] = __ddiv_rn((double)min(i, (int)D255_MAX), 255.0);
    if (threadIdx.x < D255_RB) {
        d255_stage(rowp, threadIdx.x, n_rows, s_mode[0][threadIdx.x], s_beta[0][threadIdx.x], s_cm[0][threadIdx.x]);
        s_off[0][threadIdx.x] = d255_off(rowp, threadIdx.x, n_rows);
        s_off[1][threadIdx.x] = d255_off(rowp, D255_RB + threadIdx.x, n_rows);
    }
    __syncthreads();
    uint4 w[D255_RB], wn[D255_RB];
#pragma unroll
    for (int u = 0; u < D255_RB; u++) {
        const int g = s_off[0][u];
        w[u] = g >= 0 && active ? ldg_stream(col + (int64_t)g * stride16) : make_uint4(0, 0, 0, 0);
    }
    for (int64_t b = 0; b < n_batches; b++) {
        const int cur = (int)(b & 1), nxt = cur ^ 1;
        const bool more = b + 1 < n_batches;
#pragma unroll
        for (int u = 0; u < D255_RB; u++) {
            const int g = more ? s_off[nxt][u] : -1;
            wn[u] = g >= 0 && active ? ldg_stream(col + (int64_t)g * stride16) : make_uint4(0, 0, 0, 0);
        }
        int32_t mn = 0, on = -1;
        double bn = 0.0, cn = 0.0;
        if (threadIdx.x < D255_RB) {
            d255_stage(rowp, (b + 1) * D255_RB + threadIdx.x, n_rows, mn, bn, cn);
            on = d255_off(rowp, (b + 2) * D255_RB + threadIdx.x, n_rows);
        }
#pragma unroll
        for (int u = 0; u < D255_RB; u++) {
            const int mode = s_mode[cur][u];                                    // warp-uniform
            if (mode == 1) {
                const double c = s_beta[cur][u];
#pragma unroll
                for (int k = 0; k < 8; k++) acc[k] = __dadd_rn(acc[k], c);
            } else if (mode >= 2) {
                const double beta = s_beta[cur][u], cm = s_cm[cur][u];
                const int flip = mode == 3 ? (int)D255_MAX : 0;
                const uint32_t ww[4] = { w[u].x, w[u].y, w[u].z, w[u].w };
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    const uint32_t v = (ww[k >> 1] >> ((k & 1) * 16)) & 0xFFFFu;
                    const int kk = abs((int)min(v, D255_MAX + 1) - flip);     // k', or 1 / 511 for a missing sample
                    const double c = __dmul_rn(s_d[kk], beta);
                    acc[k] = __dadd_rn(acc[k], v > D255_MAX ? cm : c);
                }
            }
        }
        if (threadIdx.x < D255_RB) {
            s_mode[nxt][threadIdx.x] = mn; s_beta[nxt][threadIdx.x] = bn; s_cm[nxt][threadIdx.x] = cn;
            s_off[cur][threadIdx.x] = on;                                      // batch b + 2 uses buffer (b + 2) & 1 = cur
        }
        __syncthreads();
#pragma unroll
        for (int u = 0; u < D255_RB; u++) w[u] = wn[u];
    }
#pragma unroll
    for (int k = 0; k < 8; k++)
        if (k < valid) sums[t * 8 + k] = acc[k];
}

}  // namespace npc
