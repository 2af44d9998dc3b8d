// npc_multi.cuh -- several score definitions over one resident slab as ONE dense contraction
// (BASELINE.json configs[3]; north_star: "when several score files are evaluated in one pass it
// becomes a true dense contraction (scores x variants . variants x samples), and only then is a
// tensor-core path used, with its tolerance stated").
//
// The reference scores one file per process (src/nimpress.nim:652-753); per score k, for every
// row classed OK it adds dosage*beta, or imputed*beta for a missing sample (:639-641, :450-481).
// With d[e,s] = called dosage (0 when missing) and m[e,s] = missing indicator of slab entry e
// (= one genotype row decoded for one effect allele):
//
//     sum[k,s] = SUM_e  beta[k,e] * d[e,s] + cm[k,e] * m[e,s]            cm = fl(imputed*beta)
//
// is a [scores x 2E] . [2E x samples] product.  It is evaluated EXACTLY in integers on the 5th-gen
// tensor cores: every coefficient is scaled by a per-score power of two to a 56-bit fixed-point
// integer and split into seven balanced base-256 digits; tcgen05.mma.kind::i8 multiplies the digit
// rows (operand A, int8) with the d / m planes (operand B, int8 values 0,1,2) into int32
// accumulators in tensor memory; the epilogue recombines the seven digit sums as two int64 and
// converts once.  The only approximation is the fixed-point rounding of the coefficients: with
// F = 52 - ex (max|c| = m * 2^ex, 0.5 <= m < 1) a coefficient is off by at most half a quantum,
// 2^(ex-53) <= 2^-52 * max|c| of its score, reached when max|c| is a power of two.  Stated tolerance,
// absolute: per sample, 2^-52 * max|c| times the sum of the plane values (dosage 0/1/2, 1 for a
// missing call) over the score's rows, plus fp64 rounding of the constant sum, the conversion, the
// k-split adds and the normalisation.  The errors add up over rows, so no relative bound holds: a
// score whose coefficients span many binades loses its smallest ones (tests/test_multi_exact_gpu.py
// checks this bound against the exact sum).  Per-locus records and nloci come from the same k_decide
// as every other path: bit-equal.
//
// When some imputed contribution is NaN (--imp-sample=fail / int_fail, eaf = NaN) an eighth row per
// score counts, per sample, the missing calls at those entries: count > 0 -> score NaN, as the
// reference's NaN propagation gives.  128 accumulator rows hold 18 scores of 7 rows or 16 of 8.
//
// Kernel k_multi_contract: persistent, one CTA per SM, a tile = 256 samples x all entries.
//   warps 4..7   producers: per k-block (64 entries) 64 TMA bulk copies of 512 B (one per genotype row
//                segment; a warp issues one copy at a time, hence four warps) + the 64 effect-allele
//                patterns into a 3-stage raw ring
//   warp 9       loads the 16 KB digit tile A of the k-block (prebuilt in global memory as the smem
//                image, L2-resident) into its own 3-stage ring
//   warps 10..25 converters: raw GT bytes -> d / m planes with byte-wise SWAR compares, written as
//                operand B, MN-major (the samples of a plane row contiguous: no transpose), 128-byte
//                swizzle, 2-stage ring
//   warp 8       one thread issues 4 x tcgen05.mma (M=128, N=256, K=32) per k-block; tcgen05.commit
//                releases the A / B stages and, after the last k-block, hands the accumulator over
//   warps 0..3   epilogue: tcgen05.ld -> smem (all 128 rows) -> int64 recombination -> normalise
//                (:643-649) -> coalesced stores; two accumulators (2 x 256 TMEM columns) so the
//                epilogue of tile t overlaps the main loop of tile t+1
#pragma once
#include "npc_fused5.cuh"   // the pair index (F5_PACK_W) and the shared PTX helpers

namespace npc {

constexpr int MC_M = 128;                    // UMMA M: rows_per_score rows for each score
constexpr int MC_N = 256;                    // UMMA N: samples per tile
constexpr int MC_ENT = 64;                   // entries per k-block -> 128 plane rows = one 128-byte swizzle row of K
constexpr int MC_SCORES = 18;                // scores per launch: 18 x 7 digit rows, or 16 x (7 digits + NaN counter)
constexpr int MC_DIGITS = 7;
constexpr int MC_RS = 3, MC_BS = 2, MC_AS = 3, MC_TS = 2;   // ring depths: raw, B, A, accumulators
constexpr int MC_PITCH = 528;                // raw row pitch in a stage: 512 + 16 so that rows g, g+1, .. hit distinct banks
constexpr int MC_RAW_STAGE = MC_ENT * MC_PITCH + MC_ENT * 4;   // + the effect-allele byte patterns of the 64 entries
constexpr int MC_A_STAGE = MC_M * 128, MC_B_STAGE = MC_N * 128;
constexpr int MC_CW = 16;                    // converter warps: one 8-entry x 4-sample-quad step each per k-block
constexpr int MC_PW = 4;                     // raw producer warps: a bulk copy is issued by one thread at a time per warp
constexpr int MC_W_MMA = 4 + MC_PW, MC_W_A = MC_W_MMA + 1, MC_FIRST_CW = MC_W_A + 1;   // warps 0..3 epilogue, 4..7 producers, 8 MMA, 9 A loader, 10.. converters
constexpr int MC_THREADS = (MC_FIRST_CW + MC_CW) * 32;
constexpr int MC_EPI_COLS = 16;              // accumulator columns per epilogue step
constexpr int MC_EPI_PITCH = MC_EPI_COLS + 1; // words; conflict-free transpose
constexpr int MC_OFF_B = 0;
constexpr int MC_OFF_A = MC_OFF_B + MC_BS * MC_B_STAGE;
constexpr int MC_OFF_RAW = MC_OFF_A + MC_AS * MC_A_STAGE;
constexpr int MC_OFF_EPI = MC_OFF_RAW + MC_RS * MC_RAW_STAGE;
constexpr int MC_OFF_BAR = MC_OFF_EPI + 4 * 32 * MC_EPI_PITCH * 4;
constexpr int MC_NBAR = 2 * MC_RS + 2 * MC_BS + 2 * MC_AS + 2 * MC_TS;
constexpr int MC_OFF_TMEM = MC_OFF_BAR + MC_NBAR * 8;
// converters' pair tables (round 2): [T-1 (3 = no allele matches)][66*c0 + c1 + 4*c2 + 16*c3] -> bytes {d(s0), d(s1), m(s0), m(s1)} of
// the two samples of a raw word, the index of npc_fused5.cuh.  Tables are 1184 bytes apart = 1152 + a QUARTER of a bank row:
// a warp's lookup mixes entries (lanes g) with effect allele REF and ALT1, i.e. tables 0 and 1, and the 16 REF / ALT1
// combinations of a table sit in banks {7..14, 23..30} -- a set that a 16-bank shift maps onto itself (measured: 1.63
// wavefronts per lookup with a 64-byte shift) and an 8-bank shift maps onto its complement
constexpr int MC_TAB_STRIDE = 1184;
constexpr int MC_OFF_TAB = (MC_OFF_TMEM + 16 + 127) & ~127;
constexpr int MC_SMEM = MC_OFF_TAB + 4 * MC_TAB_STRIDE + 1024;   // + slack to align the base to 1024 (swizzle atom)

struct MultiParams {
    const uint8_t *gt; int64_t row_stride; int64_t n;
    const int32_t *entry_row;                // [n_kb*64] slab row of each entry (padding entries: any valid row)
    const uint32_t *entry_pat;               // [n_kb*64] low byte: (eaidx+1)<<1; bits 8..: byte offset of the entry's pair table (min(eaidx, 3) * MC_TAB_STRIDE)
    const uint8_t *A;                        // [n_kb][16 KB] digit tiles, already in the swizzled smem layout
    int32_t n_kb, n_scores;
    int32_t rps, parts;                      // rows per score: 7 digits, or 8 = 7 digits + NaN counter; parts: see below
    int32_t kb_per_part, pad;
    // parts > 1: the k-blocks of a tile are split over `parts` work units so that the number of units
    // is close to a multiple of the grid (782 tiles on 148 SMs is 6 rounds for 5.3 rounds of work); a
    // unit then stores its raw partial sum to partial[part][score][sample] and k_multi_finish adds the
    // parts in order, adds the constants and normalises
    double *partial;
    double sc_lo[MC_SCORES], sc_hi[MC_SCORES];   // 2^-F and 2^(32-F) of each score's fixed-point scale
    double consts[MC_SCORES];                // sum of the constant (whole-locus) contributions, NaN if any is NaN
    double denom[MC_SCORES];                 // 2 * nloci
    double offset[MC_SCORES];
    double *out[MC_SCORES];                  // device, [n] each
};

// ---- tcgen05 wrappers ------------------------------------------------------------------------
__device__ __forceinline__ uint64_t l2_evict_last_policy() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
// K-major operand, 128-byte swizzle: row r (M or N index) at r*128, its 16-byte chunk c at ((c ^ (r&7)) << 4);
// 8 rows = one 1024-byte atom, atoms 1024 bytes apart (stride byte offset); descriptor version 1.
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
// MN-major operand (the N = 256 samples of a K row contiguous), 128-byte swizzle: two column blocks of 128 samples,
// 16 KB apart (leading byte offset); in a block K row r at r*128 with its 16-byte chunk c at ((c ^ (r&7)) << 4);
// 8 K rows = one 1024-byte atom (stride byte offset).  Layout verified by tools/probe/umma_i8_probe.cu.
__device__ __forceinline__ uint64_t umma_desc_sw128_mn(uint32_t saddr) {
    return (uint64_t)((saddr >> 4) & 0x3FFFu) | ((uint64_t)(16384 >> 4) << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
// D = S32, A = B = signed 8-bit, A K-major, B MN-major (bit 16), N = 256, M = 128
constexpr uint32_t MC_IDESC = (2u << 4) | (1u << 7) | (1u << 10) | (1u << 16) | ((uint32_t)(MC_N >> 3) << 17) | ((uint32_t)(MC_M >> 4) << 24);
__device__ __forceinline__ void umma_i8(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t accumulate) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
                 ::"r"(tmem_d), "l"(da), "l"(db), "r"(MC_IDESC), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,"
                 "%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
                   "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]), "=r"(v[17]), "=r"(v[18]),
                   "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]),
                   "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&v)[16]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), "=r"(v[9]),
                   "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15])
                 : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void sts_u32(uint32_t addr, uint32_t v) {
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

// d and m of four samples of one genotype row.  w0, w1: the eight GT bytes (sample-major allele pairs);
// pat: (eaidx+1)<<1 in every byte.  Returns dosage bytes (0 where the sample is missing) and missing bytes (0/1).
// convert4_fast -- all bytes non-negative (the common case): per byte, bits 1..6 are allele+1 (0 = missing); a byte x is zero iff
// (x + 0x7F) has bit 7 clear, carry-free since x <= 0x7E.  convert4_exact -- otherwise (sentinels, invalid codes): decode_sample.
__device__ __forceinline__ void convert4_fast(uint32_t w0, uint32_t w1, uint32_t pat, uint32_t &d4, uint32_t &m4) {
    const uint32_t a0 = __byte_perm(w0, w1, 0x6420), a1 = __byte_perm(w0, w1, 0x7531);   // first / second allele of the 4 samples
    const uint32_t ne0 = ((a0 ^ pat) & 0x7E7E7E7Eu) + 0x7F7F7F7Fu, ne1 = ((a1 ^ pat) & 0x7E7E7E7Eu) + 0x7F7F7F7Fu;   // bit 7: allele != effect allele
    const uint32_t nz0 = (a0 & 0x7E7E7E7Eu) + 0x7F7F7F7Fu, nz1 = (a1 & 0x7E7E7E7Eu) + 0x7F7F7F7Fu;                   // bit 7: allele called
    const uint32_t called = nz0 & nz1 & 0x80808080u;                                       // bit 7: both alleles called
    d4 = ((~ne0 & called) >> 7) + ((~ne1 & called) >> 7);
    m4 = (called >> 7) ^ 0x01010101u;
}
__device__ __forceinline__ void convert4_exact(uint32_t w0, uint32_t w1, int eaidx, uint32_t &d4, uint32_t &m4) {
    d4 = 0; m4 = 0;
#pragma unroll
    for (int i = 0; i < 4; i++) {
        const uint32_t h = ((i < 2 ? w0 : w1) >> ((i & 1) * 16)) & 0xFFFFu;
        int8_t a[2] = { (int8_t)(h & 0xFF), (int8_t)(h >> 8) };
        int d; bool miss;
        decode_sample<int8_t>(a, 2, eaidx, d, miss);
        d4 |= (uint32_t)(miss ? 0 : d) << (8 * i);
        m4 |= (uint32_t)(miss ? 1 : 0) << (8 * i);
    }
}

__global__ void __launch_bounds__(MC_THREADS, 1) k_multi_contract(const __grid_constant__ MultiParams P) {
    extern __shared__ uint8_t mc_smem_raw[];
    const uint32_t base = (smem_u32(mc_smem_raw) + 1023u) & ~1023u;
    const uint32_t sB = base + MC_OFF_B, sA = base + MC_OFF_A, sRaw = base + MC_OFF_RAW, sEpi = base + MC_OFF_EPI;
    const uint32_t bars = base + MC_OFF_BAR, sTmem = base + MC_OFF_TMEM;
    // barrier map
    const uint32_t raw_full = bars, raw_empty = raw_full + 8 * MC_RS, b_full = raw_empty + 8 * MC_RS, b_empty = b_full + 8 * MC_BS;
    const uint32_t a_full = b_empty + 8 * MC_BS, a_empty = a_full + 8 * MC_AS, t_full = a_empty + 8 * MC_AS, t_empty = t_full + 8 * MC_TS;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int64_t n_units = ((P.n + MC_N - 1) / MC_N) * P.parts;     // unit = (sample tile, part of the k-blocks)

    if (tid == 0) {
        for (int i = 0; i < MC_RS; i++) { mbar_init(raw_full + 8 * i, MC_PW); mbar_init(raw_empty + 8 * i, MC_CW); }
        for (int i = 0; i < MC_BS; i++) { mbar_init(b_full + 8 * i, MC_CW); mbar_init(b_empty + 8 * i, 1); }
        for (int i = 0; i < MC_AS; i++) { mbar_init(a_full + 8 * i, 1); mbar_init(a_empty + 8 * i, 1); }
        for (int i = 0; i < MC_TS; i++) { mbar_init(t_full + 8 * i, 1); mbar_init(t_empty + 8 * i, 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int i = tid; i < 4 * 256; i += MC_THREADS) {
        const int cc = i & 255, Tm = i >> 8, T = Tm < 3 ? Tm + 1 : 99;
        const int c0 = cc & 3, c1 = (cc >> 2) & 3, c2 = (cc >> 4) & 3, c3 = cc >> 6;
        const uint32_t s0 = f5_code(c0, c1, T), s1 = f5_code(c2, c3, T);
        const uint32_t e = (s0 == 3u ? 0u : s0) | ((s1 == 3u ? 0u : s1) << 8) | ((s0 == 3u ? 1u : 0u) << 16) | ((s1 == 3u ? 1u : 0u) << 24);
        sts_u32(base + MC_OFF_TAB + Tm * MC_TAB_STRIDE + 4 * (66 * c0 + c1 + 4 * c2 + 16 * c3), e);
    }
    if (warp == MC_W_MMA) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(sTmem) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem = lds_u32(sTmem);

    if (warp >= 4 && warp < 4 + MC_PW) {
        // ===== raw producers: warp pw brings entries pw*16 .. pw*16+15 of every k-block =====
        const uint64_t pol_stream = l2_evict_first_policy(), pol_keep = l2_evict_last_policy();
        constexpr int PER = MC_ENT / MC_PW;
        const int pw = warp - 4, el = pw * PER + (lane % PER);
        uint32_t it = 0;
        for (int64_t unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
            const int64_t tile = unit / P.parts;
            const int kb_lo = (int)(unit % P.parts) * P.kb_per_part, kb_hi = min(P.n_kb, kb_lo + P.kb_per_part);
            const int64_t byte0 = tile * (MC_N * 2);
            const uint32_t seg = (uint32_t)min((int64_t)(MC_N * 2), P.row_stride - byte0);      // multiple of 16: row_stride is
            int32_t r0 = P.entry_row[kb_lo * MC_ENT + el];
            for (int kb = kb_lo; kb < kb_hi; kb++, it++) {
                const uint32_t rs = it % MC_RS;
                const uint32_t stage = sRaw + rs * MC_RAW_STAGE;
                mbar_wait(raw_empty + 8 * rs, ((it / MC_RS) & 1) ^ 1);
                if (lane == 0) mbar_arrive_expect_tx(raw_full + 8 * rs, seg * PER + (pw == 0 ? MC_ENT * 4 : 0));
                __syncwarp();
                if (lane < PER) tma_load_1d(stage + el * MC_PITCH, P.gt + (int64_t)r0 * P.row_stride + byte0, seg, raw_full + 8 * rs, pol_stream);
                if (pw == 0 && lane == 0) tma_load_1d(stage + MC_ENT * MC_PITCH, P.entry_pat + (int64_t)kb * MC_ENT, MC_ENT * 4, raw_full + 8 * rs, pol_keep);
                if (kb + 1 < kb_hi) r0 = P.entry_row[(kb + 1) * MC_ENT + el];
                __syncwarp();
            }
        }
    } else if (warp == MC_W_A) {
        // ===== digit-tile loader: its own ring, so that it never holds the raw producer back =====
        if (lane == 0) {
            const uint64_t pol_keep = l2_evict_last_policy();
            uint32_t it = 0;
            for (int64_t unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
                const int kb_lo = (int)(unit % P.parts) * P.kb_per_part, kb_hi = min(P.n_kb, kb_lo + P.kb_per_part);
                for (int kb = kb_lo; kb < kb_hi; kb++, it++) {
                    const uint32_t as = it % MC_AS;
                    mbar_wait(a_empty + 8 * as, ((it / MC_AS) & 1) ^ 1);
                    mbar_arrive_expect_tx(a_full + 8 * as, MC_A_STAGE);
                    tma_load_1d(sA + as * MC_A_STAGE, P.A + (int64_t)kb * MC_A_STAGE, MC_A_STAGE, a_full + 8 * as, pol_keep);
                }
            }
        }
    } else if (warp == MC_W_MMA) {
        // ===== MMA issuer: one thread =====
        if (lane == 0) {
            uint32_t it = 0, tcount = 0;
            for (int64_t unit = blockIdx.x; unit < n_units; unit += gridDim.x, tcount++) {
                const int kb_lo = (int)(unit % P.parts) * P.kb_per_part, kb_hi = min(P.n_kb, kb_lo + P.kb_per_part);
                const uint32_t ts = tcount % MC_TS;
                mbar_wait(t_empty + 8 * ts, ((tcount / MC_TS) & 1) ^ 1);
                tc_fence_after();
                const uint32_t acc = tmem + ts * MC_N;
                for (int kb = kb_lo; kb < kb_hi; kb++, it++) {
                    const uint32_t bs = it % MC_BS, as = it % MC_AS;
                    mbar_wait(a_full + 8 * as, (it / MC_AS) & 1);
                    mbar_wait(b_full + 8 * bs, (it / MC_BS) & 1);
                    tc_fence_after();
                    const uint64_t da = umma_desc_sw128(sA + as * MC_A_STAGE), db = umma_desc_sw128_mn(sB + bs * MC_B_STAGE);
#pragma unroll
                    for (int ks = 0; ks < 4; ks++)                       // K = 32 per instruction: A +32 bytes in its rows, B 32 K rows (4 KB) further
                        umma_i8(acc, da + 2 * ks, db + 256 * ks, ((kb - kb_lo) | ks) != 0);
                    umma_commit(b_empty + 8 * bs);
                    umma_commit(a_empty + 8 * as);
                }
                umma_commit(t_full + 8 * ts);
            }
        }
    } else if (warp >= MC_FIRST_CW) {
        // ===== converters =====
        const int cw = warp - MC_FIRST_CW, g = lane & 7, qsub = lane >> 3;
        uint32_t it = 0;
        for (int64_t unit = blockIdx.x; unit < n_units; unit += gridDim.x) {
            const int kb_lo = (int)(unit % P.parts) * P.kb_per_part, kb_hi = min(P.n_kb, kb_lo + P.kb_per_part);
            for (int kb = kb_lo; kb < kb_hi; kb++, it++) {
                const uint32_t rs = it % MC_RS, bs = it % MC_BS;
                const uint32_t stage = sRaw + rs * MC_RAW_STAGE, bt = sB + bs * MC_B_STAGE;
                mbar_wait(raw_full + 8 * rs, (it / MC_RS) & 1);
                mbar_wait(b_empty + 8 * bs, ((it / MC_BS) & 1) ^ 1);
                uint32_t pat[8];
#pragma unroll
                for (int j = 0; j < 8; j++) pat[j] = lds_u32(stage + MC_ENT * MC_PITCH + (g + 8 * j) * 4);
                {
                    const int q = cw * 4 + qsub;                         // sample quad 0..63 of the tile
                    uint32_t D[8], M[8];
                    uint2 w[8];
#pragma unroll
                    for (int j = 0; j < 8; j++) w[j] = lds_v2(stage + (g + 8 * j) * MC_PITCH + q * 8);   // entry g + 8j of the k-block
                    const uint32_t any = ((w[0].x | w[0].y) | (w[1].x | w[1].y)) | ((w[2].x | w[2].y) | (w[3].x | w[3].y)) |
                                         ((w[4].x | w[4].y) | (w[5].x | w[5].y)) | ((w[6].x | w[6].y) | (w[7].x | w[7].y));
                    if ((any & 0xF8F8F8F8u) == 0u) {
                        // every allele is REF, ALT1, ALT2 or missing: two samples per table lookup (the pair index of the fused
                        // kernel), the entry's bytes are the two dosages and the two missing flags
                        const uint32_t tab0 = base + MC_OFF_TAB;
#pragma unroll
                        for (int j = 0; j < 8; j++) {
                            const uint32_t tb = tab0 + (pat[j] >> 8);
                            const uint32_t e01 = lds_u32(__dp4a(w[j].x & 0x06060606u, F5_PACK_W, tb)), e23 = lds_u32(__dp4a(w[j].y & 0x06060606u, F5_PACK_W, tb));
                            D[j] = __byte_perm(e01, e23, 0x5410);
                            M[j] = __byte_perm(e01, e23, 0x7632);
                        }
                    } else if ((any & 0x80808080u) == 0u) {              // more alleles, but no sentinel and no invalid code: byte-wise SWAR compares
#pragma unroll
                        for (int j = 0; j < 8; j++) convert4_fast(w[j].x, w[j].y, (pat[j] & 0xFFu) * 0x01010101u, D[j], M[j]);
                    } else {
#pragma unroll
                        for (int j = 0; j < 8; j++) convert4_exact(w[j].x, w[j].y, (int)((pat[j] & 0xFFu) >> 1) - 1, D[j], M[j]);
                    }
                    // operand B, MN-major: K row 16j + 8*plane + g (entry g + 8j; plane 0 = dosage, 1 = missing) holds the
                    // tile's 256 samples contiguously, so a thread's four samples of a plane are one word: no transpose.
                    // Lanes g = 0..7 write eight consecutive K rows -> eight different swizzled chunks: conflict-free.
                    const uint32_t col = bt + (uint32_t)(q >> 5) * 16384u + ((uint32_t)q & 3u) * 4u;
                    const uint32_t chunk = ((uint32_t)(q & 31) >> 2) ^ (uint32_t)g;
#pragma unroll
                    for (int j = 0; j < 8; j++) {
                        sts_u32(col + (uint32_t)(16 * j + g) * 128u + (chunk << 4), D[j]);
                        sts_u32(col + (uint32_t)(16 * j + 8 + g) * 128u + (chunk << 4), M[j]);
                    }
                }
                fence_async_smem();                                      // these generic-proxy writes are read by the tensor core
                __syncwarp();
                if (lane == 0) { mbar_arrive(b_full + 8 * bs); mbar_arrive(raw_empty + 8 * rs); }
            }
        }
    } else {
        // ===== epilogue: warp w reads TMEM lanes 32w..32w+31 (rows of the digit tile) =====
        uint32_t tcount = 0;
        const int col = tid & 15, grp = tid >> 4;                            // column of the step, score group 0..7
        for (int64_t unit = blockIdx.x; unit < n_units; unit += gridDim.x, tcount++) {
            const int64_t tile = unit / P.parts;
            const int part = (int)(unit % P.parts);
            const uint32_t ts = tcount % MC_TS;
            mbar_wait(t_full + 8 * ts, (tcount / MC_TS) & 1);
            tc_fence_after();
            for (int c0 = 0; c0 < MC_N; c0 += MC_EPI_COLS) {
                uint32_t v[MC_EPI_COLS];
                tmem_ld16(tmem + ((uint32_t)(warp * 32) << 16) + ts * MC_N + c0, v);
#pragma unroll
                for (int j = 0; j < MC_EPI_COLS; j++) sts_u32(sEpi + (tid * MC_EPI_PITCH + j) * 4, v[j]);
                asm volatile("bar.sync 1, 128;" ::: "memory");               // the four epilogue warps: rows of one score may span two of them
                const int64_t s = tile * MC_N + c0 + col;
#pragma unroll
                for (int kq = 0; kq < (MC_SCORES + 7) / 8; kq++) {
                    const int k = grp + 8 * kq;
                    if (k < P.n_scores) {
                        int32_t x[8];
#pragma unroll
                        for (int j = 0; j < 8; j++) x[j] = j < P.rps ? (int32_t)lds_u32(sEpi + ((k * P.rps + j) * MC_EPI_PITCH + col) * 4) : 0;
                        const long long lo = (long long)x[0] + ((long long)x[1] << 8) + ((long long)x[2] << 16) + ((long long)x[3] << 24);
                        const long long hi = (long long)x[4] + ((long long)x[5] << 8) + ((long long)x[6] << 16);
                        double sum = __dadd_rn(__dmul_rn((double)hi, P.sc_hi[k]), __dmul_rn((double)lo, P.sc_lo[k]));
                        if (x[7] != 0) sum = __longlong_as_double(0x7FF8000000000000ll);
                        if (s < P.n) {
                            if (P.parts == 1) P.out[k][s] = __dadd_rn(__ddiv_rn(__dadd_rn(sum, P.consts[k]), P.denom[k]), P.offset[k]);   // :643-649
                            else P.partial[((int64_t)part * P.n_scores + k) * P.n + s] = sum;
                        }
                    }
                }
                asm volatile("bar.sync 1, 128;" ::: "memory");
            }
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(t_empty + 8 * ts);
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == MC_W_MMA) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}

// parts > 1: out[k][s] = normalise(partial[0][k][s] + partial[1][k][s] + ... + consts[k])
__global__ void k_multi_finish(const __grid_constant__ MultiParams P) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int k = blockIdx.y;
    if (s >= P.n) return;
    double sum = P.partial[(int64_t)k * P.n + s];
    for (int p = 1; p < P.parts; p++) sum = __dadd_rn(sum, P.partial[((int64_t)p * P.n_scores + k) * P.n + s]);
    P.out[k][s] = __dadd_rn(__ddiv_rn(__dadd_rn(sum, P.consts[k]), P.denom[k]), P.offset[k]);
}

// ---- coefficient preparation -------------------------------------------------------------------

// counts of a score row = counts of its slab entry
__global__ void k_multi_gather(const int32_t *__restrict__ ent, int64_t n_rows, const ull *__restrict__ ecounts, ull *__restrict__ counts) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    const int32_t e = ent[r];
    counts[2 * r] = e >= 0 ? ecounts[2 * e] : 0;
    counts[2 * r + 1] = e >= 0 ? ecounts[2 * e + 1] : 0;
}

struct MultiScale { double maxabs; double consts; int32_t flags; int32_t pad; };   // flags bit 0: not representable -> caller falls back; bit 1: has NaN cm

// One block per score: largest |coefficient| over its OK rows, the ordered sum of its constant rows
// (fixed order: 256 contiguous chunks, then the chunk sums left to right), and the fallback flag.
__global__ void __launch_bounds__(256) k_multi_scale(const RowP *__restrict__ rowp, const int64_t *__restrict__ row0, MultiScale *__restrict__ out) {
    const int k = blockIdx.x;
    const int64_t a = row0[k], b = row0[k + 1];
    const int64_t per = (b - a + 255) / 256;
    const int64_t lo = a + threadIdx.x * per, hi = min(b, lo + per);
    double mx = 0.0, cs = 0.0;
    int flags = 0;
    for (int64_t r = lo; r < hi; r++) {
        const RowP rp = rowp[r];
        if (rp.mode == MODE_CONST) cs = __dadd_rn(cs, rp.c0);
        else if (rp.mode == MODE_DECODE) {
            if (rp.c1 != rp.c1) cs = __dadd_rn(cs, __longlong_as_double(0x7FF8000000000000ll));   // beta NaN: every sample NaN, as in the reference
            else if (!(fabs(rp.c1) <= 1.79e308)) flags |= 1;             // beta +-inf or near DBL_MAX: +-inf, NaN only at dosage 0 -> one by one
            else {
                mx = fmax(mx, fabs(rp.c1));
                if (rp.cm == rp.cm) { if (fabs(rp.cm) > 1.79e308) flags |= 1; else mx = fmax(mx, fabs(rp.cm)); }
                else flags |= 2;                                      // a NaN imputed contribution: the launch needs the NaN counter rows
            }
        }
    }
    __shared__ double s_mx[256], s_cs[256];
    __shared__ int s_fl;
    if (threadIdx.x == 0) s_fl = 0;
    __syncthreads();
    s_mx[threadIdx.x] = mx; s_cs[threadIdx.x] = cs;
    if (flags) atomicOr(&s_fl, flags);
    __syncthreads();
    if (threadIdx.x == 0) {
        double m = 0.0, c = 0.0;
        for (int i = 0; i < 256; i++) { m = fmax(m, s_mx[i]); c = __dadd_rn(c, s_cs[i]); }
        MultiScale o; o.maxabs = m; o.consts = c; o.flags = s_fl; o.pad = 0;
        out[k] = o;
    }
}

// coef[(k*2 + plane) * E + e] += round(c * 2^F_k): exact integer adds, so repeated rows of one score commute
__global__ void k_multi_coef(const RowP *__restrict__ rowp, const int32_t *__restrict__ ent, const int32_t *__restrict__ score_of, int64_t n_rows,
                             int k0, const int32_t *__restrict__ fexp, int64_t E, long long *__restrict__ coef, uint8_t *__restrict__ pois) {
    const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= n_rows) return;
    const RowP rp = rowp[r];
    const int32_t e = ent[r];
    if (rp.mode != MODE_DECODE || e < 0) return;
    if (rp.c1 != rp.c1) return;                                        // beta NaN: counted as a NaN constant by k_multi_scale
    const int k = score_of[r] - k0;                                    // score within this launch
    const int F = fexp[k];
    atomicAdd((ull *)&coef[((int64_t)k * 2 + 0) * E + e], (ull)__double2ll_rn(scalbn(rp.c1, F)));
    if (rp.cm == rp.cm) atomicAdd((ull *)&coef[((int64_t)k * 2 + 1) * E + e], (ull)__double2ll_rn(scalbn(rp.cm, F)));
    else pois[(int64_t)k * E + e] = 1;
}

// digit tiles: image kb, row R = score*rps + digit (digit 7 = NaN counter), K byte kbyte = 16*j + 8*plane + g  <->  entry kb*64 + g + 8j
__global__ void __launch_bounds__(128) k_multi_digits(const long long *__restrict__ coef, const uint8_t *__restrict__ pois, int64_t E, int n_scores,
                                                     int rps, uint8_t *__restrict__ A) {
    const int kb = blockIdx.x, R = blockIdx.y, kbyte = threadIdx.x;
    const int k = R / rps, dg = R % rps, j = kbyte >> 4, plane = (kbyte >> 3) & 1, g = kbyte & 7;
    const int64_t e = (int64_t)kb * MC_ENT + g + 8 * j;
    int8_t val = 0;
    if (k < n_scores && e < E) {
        if (dg == 7) val = plane ? (int8_t)pois[(int64_t)k * E + e] : 0;
        else {
            long long v = coef[((int64_t)k * 2 + plane) * E + e];
            int d = 0;
            for (int i = 0; i <= dg; i++) { d = (int)(((v + 128) & 255) - 128); v = (v - d) >> 8; }   // balanced base-256 digits
            val = (int8_t)d;
        }
    }
    A[(int64_t)kb * MC_A_STAGE + R * 128 + (((kbyte >> 4) ^ (R & 7)) << 4) + (kbyte & 15)] = (uint8_t)val;
}

}  // namespace npc
