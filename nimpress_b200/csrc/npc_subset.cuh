// npc_subset.cuh -- on-device row compaction for contexts that score a subset of the samples their rows carry
// (npc_create_subset, DESIGN.md 4.11).
//
// NOT IN THE REFERENCE, which scores every sample of its VCF.  The host reads and uploads full rows of n_row samples as
// it always does; after the H2D copy one gather writes the kept samples keep[0..n_keep) (ascending, distinct) into
// rows of the context's own layout.  A compact row is byte for byte the row the reader would have made from a file
// holding only the kept samples, apart from stride padding (written as zeros) and the padding codes of a .bed row's last
// byte.  The scoring kernels never see the difference.
//
//   k_gather_vec<T>  layouts of 2 or 4 bytes per sample (int8 diploid GT, int16 haploid GT, FORMAT/DS, NPC_GT_DOSE255,
//                    NPC_GT_DOSE32, NPC_GT_PL, int32 haploid GT): a thread gathers 16 / sizeof(T) kept samples and
//                    writes them with one 16-byte store.  `hdr` bytes at the front of the row (NPC_GT_DOSE32: 16) are
//                    copied unchanged.
//   k_gather_unit<U> any other whole number of bytes per sample (1 .. 256): one thread per output unit of U.
//   k_gather_bed     2-bit .bed codes: output byte j holds kept samples 4j .. 4j+3; a thread writes 4 bytes.
//
// The keep list on the device is padded with zeros to a multiple of SUB_PAD entries, so that the vector loads of a
// row's last chunk stay inside it; positions at or past n_keep are written as zeros.
#pragma once
#include <cstdint>

namespace npc {

constexpr int SUB_THREADS = 256;
constexpr int64_t SUB_PAD = 64;                   // keep-list padding: >= the samples of one thread's chunk in every kernel

template <typename T>
__global__ void __launch_bounds__(SUB_THREADS)
k_gather_vec(const uint8_t *__restrict__ src, int64_t src_stride, uint8_t *__restrict__ dst, int64_t dst_stride,
             const int32_t *__restrict__ keep, int64_t n_keep, int hdr) {
    constexpr int PER = 16 / (int)sizeof(T);      // samples per thread: 8 (2-byte) or 4 (4-byte)
    const int64_t r = blockIdx.y;
    const uint8_t *s = src + r * src_stride;
    uint8_t *d = dst + r * dst_stride;
    if (hdr && blockIdx.x == 0 && threadIdx.x == 0)
        *reinterpret_cast<uint4 *>(d) = *reinterpret_cast<const uint4 *>(s);
    const T *se = reinterpret_cast<const T *>(s + hdr);
    const int64_t n_chunks = (n_keep + PER - 1) / PER;
    for (int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; c < n_chunks; c += (int64_t)gridDim.x * blockDim.x) {
        int32_t idx[PER];
        const int4 *kp = reinterpret_cast<const int4 *>(keep + c * PER);
#pragma unroll
        for (int q = 0; q < PER / 4; q++) {
            const int4 k = __ldg(kp + q);
            idx[4 * q] = k.x; idx[4 * q + 1] = k.y; idx[4 * q + 2] = k.z; idx[4 * q + 3] = k.w;
        }
        T v[PER];
#pragma unroll
        for (int q = 0; q < PER; q++) v[q] = c * PER + q < n_keep ? __ldg(se + idx[q]) : (T)0;
        uint4 out;
        memcpy(&out, v, 16);
        *reinterpret_cast<uint4 *>(d + hdr + c * 16) = out;
    }
}

template <typename U>
__global__ void __launch_bounds__(SUB_THREADS)
k_gather_unit(const uint8_t *__restrict__ src, int64_t src_stride, uint8_t *__restrict__ dst, int64_t dst_stride,
              const int32_t *__restrict__ keep, int64_t n_keep, int units) {
    const int64_t r = blockIdx.y;
    const U *s = reinterpret_cast<const U *>(src + r * src_stride);
    U *d = reinterpret_cast<U *>(dst + r * dst_stride);
    const int64_t n_units = n_keep * units;
    for (int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; j < n_units; j += (int64_t)gridDim.x * blockDim.x) {
        const int64_t i = j / units;
        d[j] = __ldg(s + (int64_t)__ldg(keep + i) * units + (j - i * units));
    }
}

__global__ void __launch_bounds__(SUB_THREADS)
k_gather_bed(const uint8_t *__restrict__ src, int64_t src_stride, uint8_t *__restrict__ dst, int64_t dst_stride,
             const int32_t *__restrict__ keep, int64_t n_keep) {
    const int64_t r = blockIdx.y;
    const uint8_t *s = src + r * src_stride;
    uint8_t *d = dst + r * dst_stride;
    const int64_t n_words = (n_keep + 15) / 16;   // 16 samples = 4 output bytes per thread
    for (int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; w < n_words; w += (int64_t)gridDim.x * blockDim.x) {
        const int4 *kp = reinterpret_cast<const int4 *>(keep + w * 16);
        uint32_t out = 0;
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int4 k = __ldg(kp + q);
            const int32_t idx[4] = { k.x, k.y, k.z, k.w };
#pragma unroll
            for (int b = 0; b < 4; b++) {
                const int t = 4 * q + b;
                if (w * 16 + t < n_keep) out |= (uint32_t)((__ldg(s + (idx[b] >> 2)) >> (2 * (idx[b] & 3))) & 3u) << (2 * t);
            }
        }
        *reinterpret_cast<uint32_t *>(d + w * 4) = out;   // a last word past the row's bytes is stride padding
    }
}

}  // namespace npc
