// npc_fused.cuh -- shared pieces of the fused persistent tile kernel (npc_fused5.cuh): launch
// parameters, the packed tally word, the PTX wrappers for mbarrier / TMA bulk copies / relaxed
// global loads and REDs / shared-memory loads with raw 32-bit addresses, and k_add_partials.
#pragma once
#include "npc_kernels.cuh"

namespace npc {

struct FusedParams {
    const uint8_t *gt;
    int64_t row_stride;
    int64_t n;                 // samples of this context
    const npc_row *rows;
    int64_t n_rows;
    Policy pol;
    double *sums;
    ull *counts;               // [n_rows] arrivals<<56 | nmiss<<28 | neff, zeroed before the launch
    npc_locus *log;
    ull *nloci;
    int32_t Sr, Sc, L, A;      // raw stages, index-ring tiles, count->accumulate lag (tiles), decider warps
    int32_t nc;                // consumer warps
    int32_t GD;                // pair kernel: tiles a decider pass covers (8 = one row per lane; 4 when the lag is short)
    int32_t slab_stride;       // bytes per row in a raw stage = nc*32*K*16 (every consumer thread has a cell)
    // tile kernel only: the grid is Gs sample slabs x Gr row groups (Gr = 1: every CTA sees every row).
    // Group g > 0 accumulates into partials[(g-1)*n ..]; k_add_partials folds them in group order.
    int32_t Gs, Gr;
    double *partials;
    // pair kernel: the tally words of the NEXT launch (the other half of a double buffer), cleared by this one so
    // that no memset sits between launches; n_zero words.  nullptr: the caller cleared `counts` itself.
    ull *counts_next;
    int64_t n_zero;
    // NPC_TRACE: %globaltimer stamps of CTA 0 (launch start, tables ready, first tile counted, last tile counted,
    // last tile accumulated, sums stored), for the low-n launch-floor analysis; nullptr = off
    ull *trace;
    // pair kernel, cohorts too wide for one resident pass: the rows were tallied and decided beforehand (k_count_* +
    // k_decide over ALL samples) and this launch covers one slab of the sample axis: no tallies are published, the
    // deciders take the rows' contributions from decided[row] instead of polling the grid.  nullptr: the normal mode.
    const RowP *decided;
};

constexpr int FUSED_CNT_BITS = 28;
constexpr ull FUSED_CNT_MASK = (1ull << FUSED_CNT_BITS) - 1;
// The tally table of a row depends only on T = eaidx+1.  Fast-path codes are alleles REF..ALT6
// (T <= 7); for T >= 8 no fast-path code can match, so table 8 serves every larger T.
constexpr uint32_t FUSED_CNT_TABLES = 8;
constexpr uint32_t FUSED_CNT_STRIDE = 256;     // one-byte entries; a PRMT forms (index byte | table << 8)

// ---- PTX helpers --------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_%=:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"
        "@p bra DONE_%=;\n"
        "bra WAIT_%=;\n"
        "DONE_%=:\n"
        "}\n" ::"r"(bar), "r"(parity), "r"(0x989680u) : "memory");   // suspend-time hint: sleep in hardware, do not spin
}
// TMA bulk copy global -> shared, completion counted in bytes on an mbarrier; the slab is read
// once, so it is marked evict-first in L2.
__device__ __forceinline__ void tma_load_1d(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
        ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "l"(policy) : "memory");
}
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ ull ld_relaxed_gpu_u64(const ull *p) {
    ull v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void red_relaxed_gpu_add_u64(ull *p, ull v) {
    asm volatile("red.relaxed.gpu.global.add.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ uint32_t lds_u8(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint32_t lds_u32(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ double lds_f64(uint32_t addr) {
    double v;
    asm volatile("ld.shared.f64 %0, [%1];" : "=d"(v) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint4 lds_v4(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
    return v;
}
__device__ __forceinline__ uint2 lds_v2(uint32_t addr) {
    uint2 v;
    asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(addr));
    return v;
}
__device__ __forceinline__ void sts_v2(uint32_t addr, uint32_t a, uint32_t b) {
    asm volatile("st.shared.v2.u32 [%0], {%1,%2};" ::"r"(addr), "r"(a), "r"(b) : "memory");
}
__device__ __forceinline__ void sts_v1(uint32_t addr, uint32_t a) {
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(a) : "memory");
}
__device__ __forceinline__ void red_shared_add_u32(uint32_t addr, uint32_t v) {
    asm volatile("red.shared.add.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

// sums[s] = ((sums[s] + p0[s]) + p1[s]) + ...: the row groups' partial sums, in group (= row) order
__global__ void k_add_partials(double *__restrict__ sums, const double *__restrict__ partials, int64_t n, int n_partials) {
    const int64_t s = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n) return;
    double a = sums[s];
    for (int g = 0; g < n_partials; g++) a = __dadd_rn(a, partials[(int64_t)g * n + s]);
    sums[s] = a;
}

}  // namespace npc
