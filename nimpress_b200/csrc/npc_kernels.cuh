// npc_kernels.cuh -- sm_100a kernels of the nimpress scoring path.
//
// Data layout in HBM: a block is a slab of raw BCF FORMAT/GT rows, one row per VCF record,
// row r at gt + r*row_stride, sample-major inside the row (sample s at s*ploidy*width).  The
// per-sample sums live in one fp64 array `sums[n_samples]` for the whole run.
//
// Per score row the reference does: decode -> tally -> decide -> impute -> accumulate
// (src/nimpress.nim:367-391, 32-47, 565-571, 417-481, 639-641).  Here:
//   k_count_*   decode + tally: exact integer (nmiss, neff) per score row
//   k_decide    the fp64 decision (IEEE divide, strict >) and the four possible contributions
//               of the row: c[d] = fl(d*beta) for dosage d, cm = fl(imputed*beta)
//   k_accum_*   sums[s] = fl(sums[s] + c[code(s)]) in score-row order: the very same rounded
//               product and rounded add as `scores[i] += dosages[i]*beta`, so one context
//               reproduces the reference's per-sample fp64 chain bit for bit.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
#include "../../include/nimpress_cuda.h"

namespace npc {

enum { MODE_SKIP = 0, MODE_CONST = 1, MODE_DECODE = 2 };

// Decided row: what the accumulate pass needs.  64 bytes.
struct RowP {
    double c0, c1, c2, cm;   // DECODE: contribution of dosage 0/1/2 and of a missing sample; CONST: c0 = constant
    double beta;             // generic-ploidy path: contribution of dosage d is fl(d*beta)
    int32_t mode;
    int32_t eaidx;
    int32_t gt_row;
    int32_t pad;             // 32-bit dosage rows: the row's denominator D (npc_dose32.cuh); 0 elsewhere
};

struct Policy {
    int32_t imp_locus, imp_missing, imp_sample, pad;
    int64_t mincs;
    double maxmis;
    int64_t n_total;         // cohort size for the --maxmis rule
};

typedef unsigned long long ull;

// ------------------------------------------------------------------------------------------
// decode helpers
// ------------------------------------------------------------------------------------------

template <typename T> struct Sent;
template <> struct Sent<int8_t>  { static constexpr int miss = INT8_MIN,  vend = INT8_MIN + 1; };
template <> struct Sent<int16_t> { static constexpr int miss = INT16_MIN, vend = INT16_MIN + 1; };
template <> struct Sent<int32_t> { static constexpr int miss = INT32_MIN, vend = INT32_MIN + 1; };

// getRawDosages (src/nimpress.nim:384-391) for one sample, on the stored width.  The
// width-specific missing / vector_end sentinels are what htslib widens to the int32 ones:
// both are ignored by the reference's comparison, and a vector_end ends the sample.
template <typename T>
__device__ __forceinline__ void decode_sample(const T *p, int ploidy, int eaidx, int &d, bool &miss) {
    d = 0;
    miss = false;
    for (int k = 0; k < ploidy; k++) {
        int raw = (int)p[k];
        if (raw == Sent<T>::vend) break;
        if (raw == Sent<T>::miss) continue;
        int val = raw < 0 ? raw : (raw >> 1) - 1;     // hts-nim Allele.value
        if (val == eaidx) d++;
        else if (val == -1) miss = true;              // NaN is sticky under a later += 1
    }
}

// Fast int8 diploid decode.  When every byte of a 16-byte chunk (8 samples) is < 16 -- alleles
// REF..ALT6, no sentinel -- each byte is a nibble (allele+1)<<1|phase.  Dropping the phase bit
// leaves a 3-bit code per allele (0 = missing, k = allele k-1) and a 6-bit index per sample,
// code0 | code1<<3, into a 64-entry per-row table.  One word holds two samples:
//   m = w & 0x0E0E0E0E ; p = m*33 = m + (m<<5)  (carry-free)  ->  index of sample 0 at bits
//   6..11, of sample 1 at bits 22..27 ; (p>>3) & 0x01F801F8 = the two indices times 8, one per
//   16-bit half: byte offsets into a table of doubles.
// Entries 64..67 are the canonical codes (dosage 0, 1, 2, missing) used by the exact slow path.
constexpr int LUT_N = 68;
__device__ __forceinline__ uint32_t pack_idx8(uint32_t w) {
    uint32_t m = w & 0x0E0E0E0Eu;
    uint32_t p = m * 33u;
    return (p >> 3) & 0x01F801F8u;
}
__device__ __forceinline__ bool chunk_is_fast(const uint4 &w) {
    return (((w.x | w.y) | (w.z | w.w)) & 0xF0F0F0F0u) == 0u;
}
// exact decode of one int8 diploid sample held in the low 16 bits of h -> canonical index * 8
__device__ __forceinline__ uint32_t slow_off8(uint32_t h, int eaidx) {
    int8_t a[2] = { (int8_t)(h & 0xFF), (int8_t)((h >> 8) & 0xFF) };
    int d; bool miss;
    decode_sample<int8_t>(a, 2, eaidx, d, miss);
    return (uint32_t)(64 + (miss ? 3 : d)) * 8u;
}
// table entry for index i (0..67) given T = eaidx+1: dosage code 0,1,2 or 3 = missing
__device__ __forceinline__ int lut_code(int i, int T) {
    if (i >= 64) return i - 64;
    int c0 = i & 7, c1 = i >> 3;
    if (c0 == 0 || c1 == 0) return 3;
    return (c0 == T) + (c1 == T);
}

__device__ __forceinline__ uint4 ldg_stream(const uint4 *p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

// ------------------------------------------------------------------------------------------
// count: tallyAlleles as integers.  counts[r] = {nmiss, neff} (zeroed by the caller)
// ------------------------------------------------------------------------------------------

template <typename T>
__global__ void __launch_bounds__(256)
k_count_generic(const uint8_t *__restrict__ gt, int64_t row_stride, const npc_row *__restrict__ rows,
                int64_t n, int ploidy, ull *__restrict__ counts) {
    const int r = blockIdx.x;
    const npc_row row = rows[r];
    if (row.kind != NPC_KIND_GT || row.gt_row < 0) return;
    const T *base = reinterpret_cast<const T *>(gt + (int64_t)row.gt_row * row_stride);
    ull nmiss = 0, neff = 0;
    const int64_t step = (int64_t)gridDim.y * blockDim.x;
    int64_t s = (int64_t)blockIdx.y * blockDim.x + threadIdx.x;
    if (ploidy <= 2) {
        // haploid / diploid: four samples' values in registers before any is decoded (the loop is latency-bound otherwise)
        constexpr int U = 4;
        for (; s + (U - 1) * step < n; s += U * step) {
            T v[U][2];
#pragma unroll
            for (int u = 0; u < U; u++)
#pragma unroll
                for (int k = 0; k < 2; k++) v[u][k] = k < ploidy ? base[(s + u * step) * ploidy + k] : (T)Sent<T>::vend;
#pragma unroll
            for (int u = 0; u < U; u++) {
                int d; bool miss;
                decode_sample<T>(v[u], 2, row.eaidx, d, miss);
                if (miss) nmiss++; else neff += d;
            }
        }
    }
    for (; s < n; s += step) {
        int d; bool miss;
        decode_sample<T>(base + s * ploidy, ploidy, row.eaidx, d, miss);
        if (miss) nmiss++; else neff += d;
    }
    __shared__ ull s_m, s_e;
    if (threadIdx.x == 0) { s_m = 0; s_e = 0; }
    __syncthreads();
    for (int o = 16; o; o >>= 1) {
        nmiss += __shfl_xor_sync(0xffffffffu, nmiss, o);
        neff += __shfl_xor_sync(0xffffffffu, neff, o);
    }
    if ((threadIdx.x & 31) == 0) { atomicAdd(&s_m, nmiss); atomicAdd(&s_e, neff); }
    __syncthreads();
    if (threadIdx.x == 0) { atomicAdd(&counts[2 * r], s_m); atomicAdd(&counts[2 * r + 1], s_e); }
}

// int8 diploid: 16-byte streaming loads, 8 samples per load, table-driven tally.
__global__ void __launch_bounds__(256)
k_count_i8x2(const uint8_t *__restrict__ gt, int64_t row_stride, const npc_row *__restrict__ rows,
             int64_t n, ull *__restrict__ counts) {
    const int r = blockIdx.x;
    const npc_row row = rows[r];
    if (row.kind != NPC_KIND_GT || row.gt_row < 0) return;
    __shared__ uint2 s_cnt[LUT_N];               // 8-byte stride so the pack_idx8 offsets apply
    __shared__ uint32_t s_m, s_e;
    if (threadIdx.x < LUT_N) {
        int c = lut_code(threadIdx.x, row.eaidx + 1);
        s_cnt[threadIdx.x] = make_uint2(c == 3 ? 0x10000u : (uint32_t)c, 0u);
    }
    if (threadIdx.x == 0) { s_m = 0; s_e = 0; }
    __syncthreads();
    const uint4 *base = reinterpret_cast<const uint4 *>(gt + (int64_t)row.gt_row * row_stride);
    const char *lut = reinterpret_cast<const char *>(s_cnt);
    const int64_t nchunks = (n + 7) >> 3;
    uint32_t acc = 0;                            // low half: effect alleles, high half: missing samples
    uint32_t nm = 0, ne = 0;
    // four independent 16-byte loads in flight per thread before any of them is used
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
            const uint4 w = wv[u];
            const int valid = (int)min((int64_t)8, n - c * 8);
            uint32_t ww[4] = { w.x, w.y, w.z, w.w };
            if (valid == 8 && chunk_is_fast(w)) {
#pragma unroll
                for (int k = 0; k < 4; k++) {
                    uint32_t o = pack_idx8(ww[k]);
                    acc += *reinterpret_cast<const uint32_t *>(lut + (o & 0xFFFFu));
                    acc += *reinterpret_cast<const uint32_t *>(lut + (o >> 16));
                }
            } else {
#pragma unroll
                for (int k = 0; k < 8; k++) {
                    if (k < valid) {
                        uint32_t h = (ww[k >> 1] >> ((k & 1) * 16)) & 0xFFFFu;
                        acc += *reinterpret_cast<const uint32_t *>(lut + slow_off8(h, row.eaidx));
                    }
                }
            }
            if (acc & 0x80008000u) { ne += acc & 0xFFFFu; nm += acc >> 16; acc = 0; }   // keep halves from overflowing
        }
    }
    ne += acc & 0xFFFFu; nm += acc >> 16;
    nm = __reduce_add_sync(0xffffffffu, nm);
    ne = __reduce_add_sync(0xffffffffu, ne);
    if ((threadIdx.x & 31) == 0) { atomicAdd(&s_m, nm); atomicAdd(&s_e, ne); }
    __syncthreads();
    if (threadIdx.x == 0) { atomicAdd(&counts[2 * r], (ull)s_m); atomicAdd(&counts[2 * r + 1], (ull)s_e); }
}

// Rows read as 16-byte chunks of L::PER16 samples after L::HEADER bytes (.bed and fixed-point dosage rows): one CTA per row
// and slab of the sample axis, four chunks in flight per thread.  L::Count, made once per row, adds one chunk to the
// thread's (nmiss, neff) words; a warp sums them in 64 bits, then shared and global 64-bit atomics (order-free).
template <class L>
__global__ void __launch_bounds__(256)
k_count_chunks(const uint8_t *__restrict__ gt, int64_t row_stride, const npc_row *__restrict__ rows, int64_t n,
               ull *__restrict__ counts) {
    const int r = blockIdx.x;
    const npc_row row = rows[r];
    if (row.kind != NPC_KIND_GT || row.gt_row < 0) return;
    __shared__ ull s_m, s_e;
    if (threadIdx.x == 0) { s_m = 0; s_e = 0; }
    __syncthreads();
    const uint8_t *p = gt + (int64_t)row.gt_row * row_stride;
    const typename L::Count count(p, row);
    const uint4 *base = reinterpret_cast<const uint4 *>(p + L::HEADER);
    const int64_t nchunks = (n + L::PER16 - 1) / L::PER16;
    uint32_t nm = 0, ne = 0;
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
            count(wv[u], n - c * L::PER16, nm, ne);
        }
    }
    ull m64 = nm, e64 = ne;
    for (int o = 16; o; o >>= 1) {
        m64 += __shfl_xor_sync(0xffffffffu, m64, o);
        e64 += __shfl_xor_sync(0xffffffffu, e64, o);
    }
    if ((threadIdx.x & 31) == 0) { atomicAdd(&s_m, m64); atomicAdd(&s_e, e64); }
    __syncthreads();
    if (threadIdx.x == 0) { atomicAdd(&counts[2 * r], s_m); atomicAdd(&counts[2 * r + 1], s_e); }
}

// ------------------------------------------------------------------------------------------
// decide: one thread per score row.  Everything the reference decides in fp64 is decided here
// with the same IEEE operations on the same integers.
// ------------------------------------------------------------------------------------------

// imputeLocusDosages (:417-447): false = locus dropped
__device__ __forceinline__ bool locus_value(const Policy &p, const npc_row &row, double &v) {
    if (p.imp_locus == NPC_LOCUS_IGNORE) return false;
    if (p.imp_locus == NPC_LOCUS_PS) v = __dmul_rn(row.eaf, 2.0);
    else if (p.imp_locus == NPC_LOCUS_HOMREF) v = row.ref_is_ea ? 2.0 : 0.0;
    else v = __longlong_as_double(0x7FF8000000000000LL);
    return true;
}

// neff: the effect-allele tally as the reference holds it, a double (an exact integer for GT rows, a real
// number for FORMAT/DS rows, npc_dosage.cuh); neff_rec: what the locus record reports for it
__device__ __forceinline__ void decide_row_real(const Policy &p, const npc_row &row, ull nmiss_u, double neff, long long neff_rec,
                                                int64_t n_local, RowP &out, npc_locus &rec) {
    const double qnan = __longlong_as_double(0x7FF8000000000000LL);
    out.c0 = out.c1 = out.c2 = out.cm = 0.0;
    out.beta = row.beta; out.eaidx = row.eaidx; out.gt_row = row.gt_row; out.pad = 0;
    rec.eaidx = -1; rec.reserved = 0; rec.ngt = rec.nmiss = rec.neff = -1; rec.imputed = qnan;
    double v = qnan;
    bool used = false, constant = false;
    int klass = row.kind;
    if (row.kind == NPC_KIND_NOTCOV) {                                   // :526-531
        used = constant = locus_value(p, row, v);
    } else if (row.kind == NPC_KIND_FILTER) {                            // :553-558 (never decoded: gt_row may be -1)
        rec.eaidx = row.eaidx;
        used = constant = locus_value(p, row, v);
    } else if (row.kind == NPC_KIND_ABSENT || row.gt_row < 0) {          // :536-551
        klass = NPC_KIND_ABSENT;
        if (p.imp_missing == NPC_MISSING_HOMREF) { v = row.ref_is_ea ? 2.0 : 0.0; used = constant = true; }
    } else {
        rec.eaidx = row.eaidx;
        const double nmiss = (double)nmiss_u;
        const double ngt = (double)(p.n_total - (int64_t)nmiss_u);
        rec.ngt = p.n_total - (int64_t)nmiss_u; rec.nmiss = (int64_t)nmiss_u; rec.neff = neff_rec;
        const double missingrate = __ddiv_rn(nmiss, (double)p.n_total);  // :565
        if (missingrate > p.maxmis) {                                    // :566-571
            klass = NPC_CLASS_MAXMIS;
            used = constant = locus_value(p, row, v);
        } else {                                                         // :582-583, imputeSampleDosages :460-477
            klass = 0;
            used = true;
            switch (p.imp_sample) {
            case NPC_SAMPLE_PS: v = __dmul_rn(row.eaf, 2.0); break;
            case NPC_SAMPLE_HOMREF: v = row.ref_is_ea ? 2.0 : 0.0; break;
            case NPC_SAMPLE_FAIL: v = qnan; break;
            default:
                if (ngt >= (double)p.mincs) v = __ddiv_rn(neff, ngt);
                else v = p.imp_sample == NPC_SAMPLE_INT_PS ? __dmul_rn(row.eaf, 2.0) : qnan;
            }
            out.c0 = __dmul_rn(0.0, row.beta);                           // dosages[i]*beta (:640)
            out.c1 = __dmul_rn(1.0, row.beta);
            out.c2 = __dmul_rn(2.0, row.beta);
            out.cm = __dmul_rn(v, row.beta);
        }
    }
    (void)n_local;
    if (constant) out.c0 = __dmul_rn(v, row.beta);
    out.mode = !used ? MODE_SKIP : constant ? MODE_CONST : MODE_DECODE;
    rec.klass = klass; rec.used = used ? 1 : 0; rec.imputed = v;
}

__device__ __forceinline__ void decide_row(const Policy &p, const npc_row &row, ull nmiss_u, ull neff_u,
                                           int64_t n_local, RowP &out, npc_locus &rec) {
    decide_row_real(p, row, nmiss_u, (double)neff_u, (long long)neff_u, n_local, out, rec);
}

// What the tally pass left for k_decide: integer layouts two words a row in counts, real-valued ones (FORMAT/DS, FORMAT/PL)
// the missing count in counts and n_blocks block sums a row in part; gt, row_stride: the slab, for rows with a header.
struct TallyIn {
    const uint8_t *gt;
    int64_t row_stride;
    const ull *counts;
    const double *part;
    int64_t n_blocks;
};

// A row's tally as decide_row_real takes it.  Each layout's tally type derives from it, fills it from (TallyIn, row, r) in
// its constructor and may hide extra(), which sets a RowP field the layout's accumulate pass needs beyond the decision.
struct RowTally {
    ull nmiss;
    double neff;
    long long neff_rec;
    __device__ void extra(const npc_row &, RowP &) const {}
};

// GT and .bed rows: counts[2r] = nmiss, counts[2r+1] = neff.
struct CountTally : RowTally {
    __device__ CountTally(const TallyIn &in, const npc_row &, int64_t r) {
        nmiss = in.counts[2 * r]; neff = (double)in.counts[2 * r + 1]; neff_rec = (long long)in.counts[2 * r + 1];
    }
};

template <class T>
__global__ void __launch_bounds__(128)
k_decide(TallyIn in, const npc_row *__restrict__ rows, int64_t n_rows, Policy p, int64_t n_local, RowP *__restrict__ rowp,
         npc_locus *__restrict__ log, ull *__restrict__ nloci) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int used = 0;
    if (r < n_rows) {
        const npc_row row = rows[r];
        const T t(in, row, r);
        RowP out; npc_locus rec;
        decide_row_real(p, row, t.nmiss, t.neff, t.neff_rec, n_local, out, rec);
        t.extra(row, out);
        rowp[r] = out;
        log[r] = rec;
        used = rec.used;
    }
    used = __reduce_add_sync(0xffffffffu, used);
    if ((threadIdx.x & 31) == 0 && used) atomicAdd(nloci, (ull)used);
}

// ------------------------------------------------------------------------------------------
// accumulate: sums[s] += contribution(row, s) for the rows of the block IN ORDER
// ------------------------------------------------------------------------------------------

template <typename T>
__global__ void __launch_bounds__(256)
k_accum_generic(const uint8_t *__restrict__ gt, int64_t row_stride, const RowP *__restrict__ rowp,
                int64_t n_rows, int64_t n, int ploidy, double *__restrict__ sums) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    double acc = sums[s];
    int64_t r = 0;
    if (ploidy <= 2) {
        // haploid / diploid: the values of four rows are loaded before the first is added -- the adds stay in row order
        // (the reference's chain), only the loads run ahead
        constexpr int U = 4;
        for (; r + U <= n_rows; r += U) {
            T v[U][2];
            int mode[U];
#pragma unroll
            for (int u = 0; u < U; u++) {
                mode[u] = rowp[r + u].mode;
                const T *p = reinterpret_cast<const T *>(gt + (int64_t)rowp[r + u].gt_row * row_stride) + s * ploidy;
#pragma unroll
                for (int k = 0; k < 2; k++) v[u][k] = (mode[u] == MODE_DECODE && k < ploidy) ? p[k] : (T)Sent<T>::vend;
            }
#pragma unroll
            for (int u = 0; u < U; u++) {
                const RowP &rp = rowp[r + u];
                if (mode[u] == MODE_CONST) acc = __dadd_rn(acc, rp.c0);
                else if (mode[u] == MODE_DECODE) {
                    int d; bool miss;
                    decode_sample<T>(v[u], 2, rp.eaidx, d, miss);
                    acc = __dadd_rn(acc, miss ? rp.cm : __dmul_rn((double)d, rp.beta));
                }
            }
        }
    }
    for (; r < n_rows; r++) {
        const RowP rp = rowp[r];
        if (rp.mode == MODE_CONST) acc = __dadd_rn(acc, rp.c0);
        else if (rp.mode == MODE_DECODE) {
            const T *p = reinterpret_cast<const T *>(gt + (int64_t)rp.gt_row * row_stride) + s * ploidy;
            int d; bool miss;
            decode_sample<T>(p, ploidy, rp.eaidx, d, miss);
            acc = __dadd_rn(acc, miss ? rp.cm : __dmul_rn((double)d, rp.beta));
        }
    }
    sums[s] = acc;
}

// int8 diploid.  A thread owns one 16-byte chunk = 8 consecutive samples and keeps their sums
// in registers across all rows of the block; rows are taken RB at a time: their tables are
// built in shared memory, then each row costs one 16-byte load, and per sample 3 integer ops,
// one 8-byte shared load and one DADD.
template <int RB, int U>
__global__ void __launch_bounds__(256)
k_accum_i8x2(const uint8_t *__restrict__ gt, int64_t row_stride, const RowP *__restrict__ rowp,
             int64_t n_rows, int64_t n, double *__restrict__ sums) {
    __shared__ double s_lut[RB][LUT_N];
    __shared__ int32_t s_mode[RB], s_gtrow[RB], s_eaidx[RB];
    const int64_t chunk = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t nchunks = (n + 7) >> 3;
    const bool active = chunk < nchunks;
    const int valid = active ? (int)min((int64_t)8, n - chunk * 8) : 0;
    double acc[8];
#pragma unroll
    for (int k = 0; k < 8; k++) acc[k] = k < valid ? sums[chunk * 8 + k] : 0.0;
    const uint4 *col = reinterpret_cast<const uint4 *>(gt) + (active ? chunk : 0);
    const int64_t stride16 = row_stride >> 4;

    for (int64_t r0 = 0; r0 < n_rows; r0 += RB) {
        const int nb = (int)min((int64_t)RB, n_rows - r0);
        __syncthreads();
        for (int i = threadIdx.x; i < nb * LUT_N; i += blockDim.x) {
            const int rr = i / LUT_N, e = i - rr * LUT_N;
            const RowP &rp = rowp[r0 + rr];
            const int code = lut_code(e, rp.eaidx + 1);
            s_lut[rr][e] = (rp.mode == MODE_CONST || code == 0) ? rp.c0 : code == 1 ? rp.c1 : code == 2 ? rp.c2 : rp.cm;
            if (e == 0) { s_mode[rr] = rp.mode; s_gtrow[rr] = rp.gt_row; s_eaidx[rr] = rp.eaidx; }
        }
        __syncthreads();
        if (!active) continue;
        for (int rb = 0; rb < nb; rb += U) {
            uint4 w[U];
#pragma unroll
            for (int u = 0; u < U; u++)
                if (rb + u < nb && s_mode[rb + u] == MODE_DECODE)
                    w[u] = ldg_stream(col + (int64_t)s_gtrow[rb + u] * stride16);
#pragma unroll
            for (int u = 0; u < U; u++) {
                if (rb + u >= nb) break;
                const int mode = s_mode[rb + u];
                if (mode == MODE_DECODE) {
                    const char *lut = reinterpret_cast<const char *>(&s_lut[rb + u][0]);
                    const uint32_t ww[4] = { w[u].x, w[u].y, w[u].z, w[u].w };
                    if (chunk_is_fast(w[u])) {
#pragma unroll
                        for (int k = 0; k < 4; k++) {
                            const uint32_t o = pack_idx8(ww[k]);
                            acc[2 * k] = __dadd_rn(acc[2 * k], *reinterpret_cast<const double *>(lut + (o & 0xFFFFu)));
                            acc[2 * k + 1] = __dadd_rn(acc[2 * k + 1], *reinterpret_cast<const double *>(lut + (o >> 16)));
                        }
                    } else {
                        const int ea = s_eaidx[rb + u];
#pragma unroll
                        for (int k = 0; k < 8; k++) {
                            const uint32_t h = (ww[k >> 1] >> ((k & 1) * 16)) & 0xFFFFu;
                            acc[k] = __dadd_rn(acc[k], *reinterpret_cast<const double *>(lut + slow_off8(h, ea)));
                        }
                    }
                } else if (mode == MODE_CONST) {
                    const double c = s_lut[rb + u][0];
#pragma unroll
                    for (int k = 0; k < 8; k++) acc[k] = __dadd_rn(acc[k], c);
                }
            }
        }
    }
#pragma unroll
    for (int k = 0; k < 8; k++)
        if (k < valid) sums[chunk * 8 + k] = acc[k];
}

// computePolygenicScores epilogue (:643-649): a rounded divide, then a rounded add.
__global__ void k_finalize(const double *__restrict__ sums, int64_t n, const ull *__restrict__ nloci,
                           double offset, double *__restrict__ out) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    const double denom = __dmul_rn((double)(int64_t)*nloci, 2.0);
    out[s] = __dadd_rn(__ddiv_rn(sums[s], denom), offset);
}

// ------------------------------------------------------------------------------------------
// synthetic cohort (tests / bench): identical bytes to oracle/nimpress_oracle.c orc_synth_fill
// ------------------------------------------------------------------------------------------

__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
    x += 0x9E3779B97F4A7C15ULL;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
    return x ^ (x >> 31);
}

__global__ void __launch_bounds__(256)
k_synth(uint8_t *__restrict__ gt, int64_t row_stride, int64_t n, int64_t v0, uint64_t seed,
        const uint32_t *__restrict__ af_thr16, const uint32_t *__restrict__ miss_thr24,
        const int32_t *__restrict__ alt_code) {
    const int64_t r = blockIdx.y;
    const uint64_t vkey = seed + (uint64_t)(v0 + r) * 0xD1B54A32D192ED03ULL;
    const uint32_t aft = af_thr16[r], mt = miss_thr24[r];
    const uint32_t alt = (uint32_t)((alt_code[r] + 1) << 1) & 0xFF;
    uint8_t *row = gt + r * row_stride;
    const int64_t nchunks = (n + 7) >> 3;
    for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < nchunks; c += (int64_t)gridDim.x * blockDim.x) {
        uint32_t ww[4] = { 0, 0, 0, 0 };
#pragma unroll
        for (int k = 0; k < 8; k++) {
            const int64_t s = c * 8 + k;
            if (s < n) {
                const uint64_t x = splitmix64(vkey + (uint64_t)s * 0x8CB92BA72F3D8DD7ULL);
                const uint32_t u0 = (uint32_t)(x & 0xFFFF), u1 = (uint32_t)((x >> 16) & 0xFFFF);
                const uint32_t um = (uint32_t)((x >> 32) & 0xFFFFFF), ph = (uint32_t)((x >> 56) & 1);
                uint32_t a0 = u0 < aft ? alt : 2u, a1 = (u1 < aft ? alt : 2u) | ph;
                if (um < mt) { a0 = 0; if (((x >> 57) & 7) != 0) a1 = ph; }
                ww[k >> 1] |= (a0 | (a1 << 8)) << ((k & 1) * 16);
            }
        }
        if (c * 8 + 8 <= n) *reinterpret_cast<uint4 *>(row + c * 16) = make_uint4(ww[0], ww[1], ww[2], ww[3]);
        else
            for (int k = 0; k < 8 && c * 8 + k < n; k++) {
                const uint32_t h = (ww[k >> 1] >> ((k & 1) * 16)) & 0xFFFF;
                row[(c * 8 + k) * 2] = (uint8_t)(h & 0xFF);
                row[(c * 8 + k) * 2 + 1] = (uint8_t)(h >> 8);
            }
    }
}

}  // namespace npc
