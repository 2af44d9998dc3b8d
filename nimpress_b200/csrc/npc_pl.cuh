// npc_pl.cuh -- FORMAT/PL rows: phred-scaled genotype likelihoods scored as posterior expected dosages (DESIGN.md 4.10).
//
// NOT IN THE REFERENCE, which reads GT only; its README lists DS and PL "soft PS" under "Future" (README.md:162-165).
// The reference's PS imputes a missing sample with 2 eaf, the expected dosage under the score file's allele frequency;
// here a sample's dosage is the posterior expected dosage given its likelihoods, with the same Hardy-Weinberg prior at
// that eaf.  The posterior depends on the score row's eaf, so it is formed here, per (score row, sample).
//
// Row layout (gt_width NPC_GT_PL, 4 B per sample): one little-endian uint32 word per sample, packed by the host from the
// sample's PL values in VCF genotype order (3 values: diploid 0/0, 0/1, 1/1; 2 values: haploid 0, 1):
//
//   bits 0-11   a     bits 12-23   b     bits 24-25   j     bits 26-27   ploidy P (1 or 2)     bit 31   missing
//
// with m the smallest PL, j the index of its first occurrence, x_g = PL_g - m, and a, b the x of the other genotypes in
// genotype order, each saturated at 4095 (b = 0 for a haploid sample).  The host writes 0xFFFFFFFF for a missing
// sample; any word with bit 31 set, P outside {1, 2} or j > P is a missing sample.
//
// Per sample, all in fp64, round to nearest, no FMA (p = npc_row.eaf, q = fl(1 - p)):
//   weights      w_g = T[x_g], T[x] = fl(10^(-x/10)) correctly rounded (npc_pl_table.cuh; 0 from x = 3237 on)
//   prior        by c = effect-allele copies of genotype g: diploid pi(0) = fl(q q), pi(1) = fl(2 fl(p q)),
//                pi(2) = fl(p p); haploid pi(0) = q, pi(1) = p.  p NaN or outside [0, 1]: every sample is missing
//   posterior    u_g = fl(pi(c_g) w_g); den = u_0 + u_1 (+ u_2) left to right; num = fl(u_1 + 2 u_2) (diploid, effect
//                allele ALT), fl(2 u_0 + u_1) (diploid, REF), u_1 (haploid, ALT), u_0 (haploid, REF).  Called iff
//                den > 0; d = fl(num / den)
//   tally        as FORMAT/DS rows (npc_dosage.cuh): nmiss an integer, neff = the fp64 sum of the called d in chunks of
//                8 samples, a 32-way butterfly, blocks of 256 left to right; k_decide_pl = k_decide_ds + the row's eaf
//   accumulate   scores[s] = fl(scores[s] + fl(d beta)) (cm for a missing sample, c0 for a constant row), rows in
//                score-row order: the reference's chain in every mode.
//
// Decisive PLs (every other x >= 3237, 0 < eaf < 1, no underflow in the priors) give d in {0, 1, 2} exactly, so such
// rows score bit for bit as the same genotypes in int8 GT rows in exact order, haploid samples included.
//
// Both passes read the row (4 B per genotype each, 8 B in all) and hold T (25.9 KB) in shared memory.  Per genotype and
// pass: two table lookups, five fp64 multiplies or adds and one correctly rounded fp64 divide.
#pragma once
#include "npc_dosage.cuh"
#include "npc_pl_table.cuh"

namespace npc {

constexpr int PL_TN = NPC_PL_TABLE_N;             // T[PL_TN] = 0 ends the table: every x >= PL_TN reads it
constexpr int PL_THREADS = 128;                   // accumulate pass: threads per CTA (4 samples each)
constexpr int PL_RB = 6;                          // accumulate pass: rows per batch (8 spills at 4 CTAs per SM)
constexpr uint32_t PL_MISSING = 0xFFFFFFFFu;

__device__ const double g_pl_tab[PL_TN + 1] = { NPC_PL_TABLE_VALUES, 0.0 };

// The row's priors by genotype index: g0..g2 of a diploid sample, h0, h1 of a haploid one.  False: p is NaN or
// outside [0, 1] (every sample of the row is missing).
struct PlPrior { double g0, g1, g2, h0, h1; };
__device__ __forceinline__ bool pl_prior(double p, bool alt, PlPrior &pr) {
    const double q = __dsub_rn(1.0, p);
    const double p0 = __dmul_rn(q, q), p1 = __dmul_rn(2.0, __dmul_rn(p, q)), p2 = __dmul_rn(p, p);
    pr.g0 = alt ? p0 : p2; pr.g1 = p1; pr.g2 = alt ? p2 : p0;
    pr.h0 = alt ? q : p; pr.h1 = alt ? p : q;
    return p >= 0.0 && p <= 1.0;
}

// One sample word -> its posterior expected dosage d; false for a missing sample.  tab: T in shared memory.
__device__ __forceinline__ bool pl_dosage(uint32_t w, const double *tab, const PlPrior &pr, bool alt, double &d) {
    const uint32_t a = w & 0xFFFu, b = (w >> 12) & 0xFFFu, j = (w >> 24) & 3u, P = (w >> 26) & 3u;
    const bool ok = !(w >> 31) && (P == 1u || P == 2u) && j <= P;
    const double wa = tab[min(a, (uint32_t)PL_TN)], wb = tab[min(b, (uint32_t)PL_TN)];
    const double w0 = j == 0u ? 1.0 : wa, w1 = j == 0u ? wa : j == 1u ? 1.0 : wb, w2 = j == 2u ? 1.0 : wb;
    const bool dip = P == 2u;
    const double u0 = __dmul_rn(dip ? pr.g0 : pr.h0, w0), u1 = __dmul_rn(dip ? pr.g1 : pr.h1, w1);
    const double u2 = dip ? __dmul_rn(pr.g2, w2) : 0.0;                  // haploid: den + 0 = den
    const double den = __dadd_rn(__dadd_rn(u0, u1), u2);
    const double num = dip ? __dadd_rn(u1, __dmul_rn(2.0, alt ? u2 : u0)) : (alt ? u1 : u0);
    d = __ddiv_rn(num, den);
    return ok && den > 0.0;
}

__device__ __forceinline__ void pl_load_table(double *s_tab) {
    for (int i = threadIdx.x; i <= PL_TN; i += blockDim.x) s_tab[i] = g_pl_tab[i];
}

// The tally of k_count_ds on PL rows: one warp per (row, block of 256 samples), a lane per chunk of 8 samples summed
// left to right, the butterfly over the 32 chunks.  A CTA loads T once and then takes rows blockIdx.y, + gridDim.y, ...
// part[r * n_blocks + b] = block sum; miss[r] += missing samples.
__global__ void __launch_bounds__(256)
k_count_pl(const uint8_t *__restrict__ gt, int64_t row_stride, const npc_row *__restrict__ rows, int64_t n_rows, int64_t n,
           int64_t n_blocks, double *__restrict__ part, ull *__restrict__ miss) {
    __shared__ double s_tab[PL_TN + 1];
    pl_load_table(s_tab);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t b = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (b >= n_blocks) return;
    const int64_t s0 = b * DS_BLOCK + lane * 8;
    for (int64_t r = blockIdx.y; r < n_rows; r += gridDim.y) {
        const npc_row row = rows[r];
        if (row.kind != NPC_KIND_GT || row.gt_row < 0) continue;
        const uint32_t *base = reinterpret_cast<const uint32_t *>(gt + (int64_t)row.gt_row * row_stride);
        const bool alt = row.eaidx != 0;
        PlPrior pr;
        const bool valid_eaf = pl_prior(row.eaf, alt, pr);
        uint32_t w[8];
        if (s0 + 8 <= n) {
            const uint4 x = ldg_stream(reinterpret_cast<const uint4 *>(base + s0)), y = ldg_stream(reinterpret_cast<const uint4 *>(base + s0) + 1);
            w[0] = x.x; w[1] = x.y; w[2] = x.z; w[3] = x.w; w[4] = y.x; w[5] = y.y; w[6] = y.z; w[7] = y.w;
        } else {
#pragma unroll
            for (int k = 0; k < 8; k++) w[k] = s0 + k < n ? base[s0 + k] : PL_MISSING;
        }
        double sum = 0.0;
        uint32_t nm = 0;
#pragma unroll
        for (int k = 0; k < 8; k++) {
            if (s0 + k >= n) break;
            double d;
            if (pl_dosage(w[k], s_tab, pr, alt, d) && valid_eaf) sum = __dadd_rn(sum, d);
            else nm++;
        }
        for (int o = 16; o; o >>= 1) sum = __dadd_rn(sum, __shfl_xor_sync(0xffffffffu, sum, o));
        nm = __reduce_add_sync(0xffffffffu, nm);
        if (lane == 0) {
            part[r * n_blocks + b] = sum;
            if (nm) atomicAdd(&miss[r], (ull)nm);
        }
    }
}

// k_decide_ds, and a decoded row carries its eaf in RowP::c0 (unused by this format) to the accumulate pass
__global__ void __launch_bounds__(128)
k_decide_pl(const npc_row *__restrict__ rows, int64_t n_rows, const double *__restrict__ part, int64_t n_blocks,
            const ull *__restrict__ miss, Policy p, int64_t n_local, RowP *__restrict__ rowp, npc_locus *__restrict__ log,
            ull *__restrict__ nloci) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int used = 0;
    if (r < n_rows) {
        const npc_row row = rows[r];
        double neff = 0.0;
        if (row.kind == NPC_KIND_GT && row.gt_row >= 0)
            for (int64_t b = 0; b < n_blocks; b++) neff = __dadd_rn(neff, part[r * n_blocks + b]);
        RowP out; npc_locus rec;
        decide_row_real(p, row, miss[r], neff, __double_as_longlong(neff), n_local, out, rec);
        if (out.mode == MODE_DECODE) out.c0 = row.eaf;
        rowp[r] = out;
        log[r] = rec;
        used = rec.used;
    }
    used = __reduce_add_sync(0xffffffffu, used);
    if ((threadIdx.x & 31) == 0 && used) atomicAdd(nloci, (ull)used);
}

// Staged per row: mode (0 dropped, 1 constant, 2 decode with effect allele ALT, 3 decode with REF), beta (the constant
// of a constant row; cm for a decoded row whose eaf makes every sample missing), cm and the priors.
struct PlStage { double beta, cm, g0, g1, g2, h0, h1; int32_t mode, off; };
__device__ __forceinline__ void pl_stage(const RowP *__restrict__ rowp, int64_t r, int64_t n_rows, PlStage &s) {
    s.mode = 0; s.beta = 0.0; s.cm = 0.0; s.g0 = s.g1 = s.g2 = s.h0 = s.h1 = 0.0;
    if (r >= n_rows) return;
    const RowP &rp = rowp[r];
    if (rp.mode == MODE_CONST) { s.mode = 1; s.beta = rp.c0; }
    else if (rp.mode == MODE_DECODE) {
        const bool alt = rp.eaidx != 0;
        PlPrior pr;
        if (pl_prior(rp.c0, alt, pr)) {
            s.mode = alt ? 2 : 3; s.beta = rp.beta; s.cm = rp.cm;
            s.g0 = pr.g0; s.g1 = pr.g1; s.g2 = pr.g2; s.h0 = pr.h0; s.h1 = pr.h1;
        } else {
            s.mode = 1; s.beta = rp.cm;
        }
    }
}
__device__ __forceinline__ int32_t pl_off(const RowP *__restrict__ rowp, int64_t r, int64_t n_rows) {
    if (r >= n_rows || rowp[r].mode != MODE_DECODE) return -1;
    PlPrior pr;
    return pl_prior(rowp[r].c0, true, pr) ? rowp[r].gt_row : -1;
}

// Loop of batch b: the loads of batch b + 1 go out first (their slab rows wait in shared memory), then the first PL_RB
// threads stage batch b + 1's rows and batch b + 2's slab rows into the buffers batch b does not read, batch b is added,
// one barrier -- the scheme of k_accum_dose32, with the staging written straight to shared memory to save registers.  A thread owns 4 samples (one
// 16-byte load per row) with their sums in fp64 registers across the launch.
__global__ void __launch_bounds__(PL_THREADS, 4)
k_accum_pl(const uint8_t *__restrict__ gt, int64_t row_stride, const RowP *__restrict__ rowp, int64_t n_rows, int64_t n,
           double *__restrict__ sums) {
    __shared__ double s_tab[PL_TN + 1];
    __shared__ PlStage s_st[2][PL_RB];
    __shared__ int32_t s_off[2][PL_RB];
    const int64_t n_batches = (n_rows + PL_RB - 1) / PL_RB;
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;    // owns samples 4t .. 4t+3
    const int64_t nw = (n + 3) >> 2;
    const bool active = t < nw;
    const int valid = active ? (int)min((int64_t)4, n - t * 4) : 0;
    double acc[4];
#pragma unroll
    for (int k = 0; k < 4; k++) acc[k] = k < valid ? sums[t * 4 + k] : 0.0;
    const uint4 *col = reinterpret_cast<const uint4 *>(gt) + (active ? t : 0);
    const int64_t stride16 = row_stride >> 4;
    pl_load_table(s_tab);
    if (threadIdx.x < PL_RB) {
        pl_stage(rowp, threadIdx.x, n_rows, s_st[0][threadIdx.x]);
        s_off[0][threadIdx.x] = pl_off(rowp, threadIdx.x, n_rows);
        s_off[1][threadIdx.x] = pl_off(rowp, PL_RB + threadIdx.x, n_rows);
    }
    __syncthreads();
    uint4 w[PL_RB], wn[PL_RB];
#pragma unroll
    for (int u = 0; u < PL_RB; u++) {
        const int g = s_off[0][u];
        w[u] = g >= 0 && active ? ldg_stream(col + (int64_t)g * stride16) : make_uint4(0, 0, 0, 0);
    }
    for (int64_t b = 0; b < n_batches; b++) {
        const int cur = (int)(b & 1), nxt = cur ^ 1;
        const bool more = b + 1 < n_batches;
#pragma unroll
        for (int u = 0; u < PL_RB; u++) {
            const int g = more ? s_off[nxt][u] : -1;
            wn[u] = g >= 0 && active ? ldg_stream(col + (int64_t)g * stride16) : make_uint4(0, 0, 0, 0);
        }
        if (threadIdx.x < PL_RB) {                                              // neither buffer is read in this batch
            pl_stage(rowp, (b + 1) * PL_RB + threadIdx.x, n_rows, s_st[nxt][threadIdx.x]);
            s_off[cur][threadIdx.x] = pl_off(rowp, (b + 2) * PL_RB + threadIdx.x, n_rows);   // batch b + 2 uses buffer cur
        }
#pragma unroll
        for (int u = 0; u < PL_RB; u++) {
            const PlStage &st = s_st[cur][u];
            const int mode = st.mode;                                           // warp-uniform
            if (mode == 1) {
                const double c = st.beta;
#pragma unroll
                for (int k = 0; k < 4; k++) acc[k] = __dadd_rn(acc[k], c);
            } else if (mode >= 2) {
                const bool alt = mode == 2;
                const PlPrior pr = { st.g0, st.g1, st.g2, st.h0, st.h1 };
                const double beta = st.beta, cm = st.cm;
                const uint32_t ww[4] = { w[u].x, w[u].y, w[u].z, w[u].w };
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    double d;
                    const bool called = pl_dosage(ww[k], s_tab, pr, alt, d);
                    acc[k] = __dadd_rn(acc[k], called ? __dmul_rn(d, beta) : cm);
                }
            }
        }
        __syncthreads();
#pragma unroll
        for (int u = 0; u < PL_RB; u++) w[u] = wn[u];
    }
#pragma unroll
    for (int k = 0; k < 4; k++)
        if (k < valid) sums[t * 4 + k] = acc[k];
}

}  // namespace npc
