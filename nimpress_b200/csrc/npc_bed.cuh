// npc_bed.cuh -- PLINK 1 `.bed` rows: 2 bits per sample instead of a BCF GT payload (DESIGN.md 4.7).
//
// NOT IN THE REFERENCE, which reads VCF / BCF only.  A `.bed` row (SNP-major) holds the same hard calls as a
// biallelic diploid GT row, so every decision is the reference's: only the decode differs.
//
//   layout      ceil(n/4) bytes per row, sample s in bits 2*(s%4) of byte s/4.  The codes of the last byte past
//               sample n-1 are padding (PLINK writes 00) and are never counted or stored.
//   code        00 hom A1, 01 missing, 10 het, 11 hom A2; A2 = REF (eaidx 0), A1 = the one ALT (eaidx 1):
//               dosage for eaidx 1 = 2 / NaN / 1 / 0, for eaidx 0 = 0 / NaN / 1 / 2.
//   k_count_bed (nmiss, neff) per score row from masks and popc over 32-bit words (16 samples), as exact integers.
//   k_decide    unchanged (npc_kernels.cuh).
//   k_accum_bed the 2-bit code indexes the row's value table {contribution of code 0, 1, 2, 3}: no decode.
//               A CONST row's table holds its constant in every entry, a dropped row's holds +0.0.
//     EXACT     acc = acc + T_r[c_r], row by row: the reference's chain (:639-640), bit for bit.
//     default   tiles of four rows from the launch's first row; T01[c0 | c1 << 2] = T0[c0] + T1[c1] and
//               T23[c2 | c3 << 2] = T2[c2] + T3[c3], then acc = (acc + T01) + T23 -- the tile kernel's association
//               (tests/util_order.py default_order_scores with one row group), one DADD per two genotypes.
//
// Both passes read the row (0.25 B per genotype each, 0.5 B in all).  A thread owns 8 samples (16 bits) of every row
// and keeps their sums in registers; a batch of BED_RB rows is loaded before the previous batch is added, so
// 2 * BED_RB rows' loads are in flight per thread -- the sample axis alone gives only ~13 warps per SM at 500,000
// samples.  k_bed_prep writes each batch's tables and slab rows beforehand, so that the accumulate pass issues a
// batch's loads without waiting on any row record.
#pragma once
#include "npc_kernels.cuh"

namespace npc {

constexpr int BED_THREADS = 128;                  // accumulate pass: threads per CTA (8 samples each)
constexpr int BED_RB = 32;                        // rows per batch (8 tiles of four)

// contribution of 2-bit code c for a decided row
__device__ __forceinline__ double bed_value(const RowP &rp, int c) {
    if (rp.mode == MODE_SKIP) return 0.0;
    if (rp.mode == MODE_CONST) return rp.c0;
    if (c == 1) return rp.cm;
    if (c == 2) return rp.c1;
    return (c == 0) == (rp.eaidx == 1) ? rp.c2 : rp.c0;          // 00 = two A1 (ALT) alleles, 11 = two A2 (REF)
}

// tallyAlleles (:32-47) on 2-bit rows.  One 16-byte load = 64 samples; four in flight per thread.
__global__ void __launch_bounds__(256)
k_count_bed(const uint8_t *__restrict__ gt, int64_t row_stride, const npc_row *__restrict__ rows, int64_t n,
            ull *__restrict__ counts) {
    const int r = blockIdx.x;
    const npc_row row = rows[r];
    if (row.kind != NPC_KIND_GT || row.gt_row < 0) return;
    __shared__ ull s_m, s_e;
    if (threadIdx.x == 0) { s_m = 0; s_e = 0; }
    __syncthreads();
    const uint4 *base = reinterpret_cast<const uint4 *>(gt + (int64_t)row.gt_row * row_stride);
    const int64_t nchunks = (n + 63) >> 6;
    const bool alt = row.eaidx == 1;
    uint32_t nm = 0, ne = 0;                      // per thread: < 2^32 for any cohort below 2^25 samples per thread
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
            const uint32_t ww[4] = { wv[u].x, wv[u].y, wv[u].z, wv[u].w };
#pragma unroll
            for (int k = 0; k < 4; k++) {
                const int64_t left = n - (c * 64 + k * 16);               // samples of this word still in the row
                const uint32_t m = left >= 16 ? 0x55555555u : left <= 0 ? 0u : 0x55555555u & ((1u << (2 * left)) - 1u);
                const uint32_t lo = ww[k] & m, hi = (ww[k] >> 1) & m;
                nm += __popc(lo & ~hi);                                   // 01
                // effect alleles: ALT = A1 counts 2 for 00 and 1 for 10; REF = A2 counts 1 for 10 and 2 for 11
                ne += alt ? __popc(m & ~lo & ~hi) + __popc(m & ~lo) : __popc(hi) + __popc(lo & hi);
            }
        }
    }
    const ull m64 = __reduce_add_sync(0xffffffffu, nm), e64 = __reduce_add_sync(0xffffffffu, ne);
    if ((threadIdx.x & 31) == 0) { atomicAdd(&s_m, m64); atomicAdd(&s_e, e64); }
    __syncthreads();
    if (threadIdx.x == 0) { atomicAdd(&counts[2 * r], s_m); atomicAdd(&counts[2 * r + 1], s_e); }
}

// Per batch of BED_RB rows, what the accumulate pass reads: the value tables (EXACT: [row][code], 4 per row; default:
// [tile][half][pair index], 32 per tile) and the slab row of every row it loads (-1: constant or dropped row, or past
// the launch's end -- every table entry equal, so the row is not read).  One thread per table entry.
template <bool EXACT>
__global__ void __launch_bounds__(256)
k_bed_prep(const RowP *__restrict__ rowp, int64_t n_rows, int64_t n_batches, double *__restrict__ tab, int32_t *__restrict__ off) {
    constexpr int E = EXACT ? BED_RB * 4 : BED_RB * 8;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_batches * E) return;
    const int64_t b = i / E;
    const int x = (int)(i - b * E);
    const int64_t r0 = b * BED_RB;
    if (x < BED_RB) {
        const int64_t r = r0 + x;
        off[r] = r < n_rows && rowp[r].mode == MODE_DECODE ? rowp[r].gt_row : -1;
    }
    if (EXACT) {
        const int64_t r = r0 + (x >> 2);
        tab[i] = r < n_rows ? bed_value(rowp[r], x & 3) : 0.0;
    } else {
        const int64_t ra = r0 + 2 * (x >> 4);                             // rows ra, ra + 1 of a tile half
        const int c = x & 15;
        const double va = ra < n_rows ? bed_value(rowp[ra], c & 3) : 0.0;
        const double vb = ra + 1 < n_rows ? bed_value(rowp[ra + 1], c >> 2) : 0.0;
        tab[i] = __dadd_rn(va, vb);
    }
}

// Loop of batch b: the loads of batch b + 1 go out first (their slab rows wait in shared memory), then this thread's
// share of batch b + 1's tables and batch b + 2's slab rows is fetched into registers, batch b is added, the fetched
// share is stored to the other shared-memory buffer, one barrier.
template <bool EXACT>
__global__ void __launch_bounds__(BED_THREADS, 4)
k_accum_bed(const uint8_t *__restrict__ gt, int64_t row_stride, const double *__restrict__ tab, const int32_t *__restrict__ off,
            int64_t n_rows, int64_t n, double *__restrict__ sums) {
    constexpr int E = EXACT ? BED_RB * 4 : BED_RB * 8;                    // table entries per batch
    constexpr int EPT = E / BED_THREADS;
    __shared__ double s_tab[2][E];
    __shared__ int32_t s_off[2][BED_RB];
    const int64_t n_batches = (n_rows + BED_RB - 1) / BED_RB;
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;    // owns samples 8t .. 8t+7
    const int64_t nw = (n + 7) >> 3;
    const bool active = t < nw;
    const int valid = active ? (int)min((int64_t)8, n - t * 8) : 0;
    double acc[8];
#pragma unroll
    for (int k = 0; k < 8; k++) acc[k] = k < valid ? sums[t * 8 + k] : 0.0;
    const uint16_t *col = reinterpret_cast<const uint16_t *>(gt) + (active ? t : 0);
    const int64_t stride2 = row_stride >> 1;
    // prologue: tables of batch 0, slab rows of batches 0 and 1
#pragma unroll
    for (int e = 0; e < EPT; e++) s_tab[0][threadIdx.x + e * BED_THREADS] = tab[threadIdx.x + e * BED_THREADS];
    if (threadIdx.x < BED_RB) {
        s_off[0][threadIdx.x] = off[threadIdx.x];
        s_off[1][threadIdx.x] = n_batches > 1 ? off[BED_RB + threadIdx.x] : -1;
    }
    __syncthreads();
    uint32_t w[BED_RB], wn[BED_RB];
#pragma unroll
    for (int u = 0; u < BED_RB; u++) {
        const int g = s_off[0][u];
        w[u] = g >= 0 && active ? (uint32_t)__ldg(col + (int64_t)g * stride2) : 0u;
    }
    for (int64_t b = 0; b < n_batches; b++) {
        const int cur = (int)(b & 1), nxt = cur ^ 1;
        const bool more = b + 1 < n_batches;
#pragma unroll
        for (int u = 0; u < BED_RB; u++) {
            const int g = more ? s_off[nxt][u] : -1;
            wn[u] = g >= 0 && active ? (uint32_t)__ldg(col + (int64_t)g * stride2) : 0u;
        }
        double tn[EPT];
        int32_t on = -1;
#pragma unroll
        for (int e = 0; e < EPT; e++) tn[e] = more ? tab[(b + 1) * E + threadIdx.x + e * BED_THREADS] : 0.0;
        if (threadIdx.x < BED_RB && b + 2 < n_batches) on = off[(b + 2) * BED_RB + threadIdx.x];
        const char *tb = reinterpret_cast<const char *>(s_tab[cur]);
        if (EXACT) {
            const int nb = (int)min((int64_t)BED_RB, n_rows - b * BED_RB);
#pragma unroll
            for (int u = 0; u < BED_RB; u++) {
                if (u >= nb) break;
                const char *tr = tb + u * 32;
#pragma unroll
                for (int k = 0; k < 8; k++)
                    acc[k] = __dadd_rn(acc[k], *reinterpret_cast<const double *>(tr + ((w[u] << 3 >> (2 * k)) & 0x18u)));
            }
        } else {
            const int nt = (int)min((int64_t)BED_RB / 4, (n_rows - b * BED_RB + 3) / 4);
#pragma unroll
            for (int q = 0; q < BED_RB / 4; q++) {
                if (q >= nt) break;
                const uint32_t w0 = w[4 * q], w1 = w[4 * q + 1], w2 = w[4 * q + 2], w3 = w[4 * q + 3];
                // nibble j of e01 = c0 | c1 << 2 of sample 2j, of o01 the same of sample 2j + 1 (likewise rows 2, 3)
                const uint32_t e01 = (w0 & 0x3333u) | ((w1 & 0x3333u) << 2), o01 = ((w0 >> 2) & 0x3333u) | (w1 & 0xCCCCu);
                const uint32_t e23 = (w2 & 0x3333u) | ((w3 & 0x3333u) << 2), o23 = ((w2 >> 2) & 0x3333u) | (w3 & 0xCCCCu);
                const char *t01 = tb + q * 256, *t23 = t01 + 128;
#pragma unroll
                for (int j = 0; j < 4; j++) {
                    const double a0 = *reinterpret_cast<const double *>(t01 + ((e01 >> (4 * j)) & 15u) * 8);
                    const double b0 = *reinterpret_cast<const double *>(t23 + ((e23 >> (4 * j)) & 15u) * 8);
                    const double a1 = *reinterpret_cast<const double *>(t01 + ((o01 >> (4 * j)) & 15u) * 8);
                    const double b1 = *reinterpret_cast<const double *>(t23 + ((o23 >> (4 * j)) & 15u) * 8);
                    acc[2 * j] = __dadd_rn(__dadd_rn(acc[2 * j], a0), b0);
                    acc[2 * j + 1] = __dadd_rn(__dadd_rn(acc[2 * j + 1], a1), b1);
                }
            }
        }
#pragma unroll
        for (int e = 0; e < EPT; e++) s_tab[nxt][threadIdx.x + e * BED_THREADS] = tn[e];
        if (threadIdx.x < BED_RB) s_off[cur][threadIdx.x] = on;              // batch b + 2 uses buffer (b + 2) & 1 = cur
        __syncthreads();
#pragma unroll
        for (int u = 0; u < BED_RB; u++) w[u] = wn[u];
    }
#pragma unroll
    for (int k = 0; k < 8; k++)
        if (k < valid) sums[t * 8 + k] = acc[k];
}

}  // namespace npc
