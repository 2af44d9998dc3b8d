// npc_dosage.cuh -- FORMAT/DS rows: fp32 expected ALT-allele dosages instead of hard calls (SURVEY.md 8f-4).
//
// NOT IN THE REFERENCE.  nimpress reads GT only (src/nimpress.nim:384-391); dosage input is listed under
// "Future" in its README (README.md:162-165).  north_star names "optional DS dosages", so the path exists,
// with the reference's own per-locus logic applied to a real-valued raw dosage:
//
//   raw dosage   ds (BCF float; missing 0x7F800001, vector_end 0x7F800002 and NaN = no call -> NaN dosage);
//                effect allele = ALT (eaidx 1): d = double(ds); effect allele = REF (eaidx 0): d = 2.0 - double(ds)
//                (both exact in fp64).  One value per sample (biallelic records).
//   tallyAlleles (:32-47) ngenotyped / nmissing as integers; neffectallele = sum of the called dosages in fp64.
//                The reference's sum is sequential; a GPU cannot reproduce a 500,000-term sequential fp64 chain
//                at speed, so the ORDER IS DEFINED HERE (and restated by the oracle): samples in chunks of 8,
//                each chunk summed left to right from +0.0; 32 consecutive chunk sums (a block of 256 samples)
//                combined by the butterfly v[i] += v[i ^ o], o = 16, 8, 4, 2, 1; block sums added left to right.
//   decision / imputation / accumulation: decide_row as for GT rows (missing rate, locus constant, neff/ngt),
//                then scores[s] += fl(d * beta) (fl(imputed * beta) for a missing sample) in score-row order:
//                the reference's chain (:639-640), bit for bit against the oracle.
//
// Roofline: 4 B per (variant, sample) cell read twice (tally pass, accumulate pass): HBM-bound, at most 50 % of
// the 4 B/cell roofline by construction; a fused variant is what comes next if the format sees use.
#pragma once
#include "npc_kernels.cuh"

namespace npc {

constexpr int DS_BLOCK = 256;                     // samples per tally block (one warp: 32 chunks of 8)

__device__ __forceinline__ bool ds_missing(uint32_t bits) {
    return bits == 0x7F800001u || bits == 0x7F800002u || (bits & 0x7FFFFFFFu) > 0x7F800000u;
}
__device__ __forceinline__ double ds_dosage(uint32_t bits, int eaidx) {
    const double d = (double)__uint_as_float(bits);
    return eaidx == 0 ? __dsub_rn(2.0, d) : d;
}

// One warp per (row, block of 256 samples): chunk sums left to right, butterfly over the 32 chunks.
// part[r * n_blocks + b] = block sum; miss[r] += missing samples (integer atomics: exact, order-free).
__global__ void __launch_bounds__(256)
k_count_ds(const uint8_t *__restrict__ gt, int64_t row_stride, const npc_row *__restrict__ rows, int64_t n, int64_t n_blocks,
           double *__restrict__ part, ull *__restrict__ miss) {
    const int r = blockIdx.y;
    const npc_row row = rows[r];
    if (row.kind != NPC_KIND_GT || row.gt_row < 0) return;
    const int lane = threadIdx.x & 31;
    const int64_t b = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (b >= n_blocks) return;
    const uint32_t *base = reinterpret_cast<const uint32_t *>(gt + (int64_t)row.gt_row * row_stride);
    const int64_t s0 = b * DS_BLOCK + lane * 8;
    double sum = 0.0;
    uint32_t nm = 0;
    uint32_t w[8];
    if (s0 + 8 <= n) {
        const uint4 a = ldg_stream(reinterpret_cast<const uint4 *>(base + s0)), c = ldg_stream(reinterpret_cast<const uint4 *>(base + s0) + 1);
        w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w; w[4] = c.x; w[5] = c.y; w[6] = c.z; w[7] = c.w;
    } else {
#pragma unroll
        for (int k = 0; k < 8; k++) w[k] = s0 + k < n ? base[s0 + k] : 0x7F800002u;
    }
#pragma unroll
    for (int k = 0; k < 8; k++) {
        if (s0 + k >= n) break;
        if (ds_missing(w[k])) nm++;
        else sum = __dadd_rn(sum, ds_dosage(w[k], row.eaidx));
    }
    for (int o = 16; o; o >>= 1) sum = __dadd_rn(sum, __shfl_xor_sync(0xffffffffu, sum, o));
    nm = __reduce_add_sync(0xffffffffu, nm);
    if (lane == 0) {
        part[(int64_t)r * n_blocks + b] = sum;
        if (nm) atomicAdd(&miss[r], (ull)nm);
    }
}

// The tally of k_decide for dosage rows: block sums left to right -> neff; the record holds its IEEE-754 bits.
struct DsTally : RowTally {
    __device__ DsTally(const TallyIn &in, const npc_row &row, int64_t r) {
        neff = 0.0;
        if (row.kind == NPC_KIND_GT && row.gt_row >= 0)
            for (int64_t b = 0; b < in.n_blocks; b++) neff = __dadd_rn(neff, in.part[r * in.n_blocks + b]);
        nmiss = in.counts[r]; neff_rec = __double_as_longlong(neff);
    }
};

// scores[s] += contribution(row, s), rows in order: the reference's chain
__global__ void __launch_bounds__(256)
k_accum_ds(const uint8_t *__restrict__ gt, int64_t row_stride, const RowP *__restrict__ rowp, int64_t n_rows, int64_t n,
           double *__restrict__ sums) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    double acc = sums[s];
    for (int64_t r = 0; r < n_rows; r++) {
        const RowP rp = rowp[r];
        if (rp.mode == MODE_CONST) acc = __dadd_rn(acc, rp.c0);
        else if (rp.mode == MODE_DECODE) {
            const uint32_t bits = reinterpret_cast<const uint32_t *>(gt + (int64_t)rp.gt_row * row_stride)[s];
            acc = __dadd_rn(acc, ds_missing(bits) ? rp.cm : __dmul_rn(ds_dosage(bits, rp.eaidx), rp.beta));
        }
    }
    sums[s] = acc;
}

}  // namespace npc
