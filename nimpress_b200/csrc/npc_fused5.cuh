// npc_fused5.cuh -- the default roofline kernel ("pair lookup"): count -> decide -> accumulate in one
// persistent cooperative launch.  A TMA raw ring feeds COUNT, a grid-wide tally dependency gates
// DECIDE, and ACCUMULATE runs over tiles of four score rows; every genotype byte is read from HBM
// exactly once.  The consumer warps are bound by the instructions they issue, not by waiting (the
// round-1 tile kernel issued 336 per (tile, warp), 75 of them for the tallies alone), so every step
// below is built to issue few:
//
//  * COUNT looks up TWO samples at a time.  A 32-bit word of the raw row holds two diploid int8
//    samples (4 allele bytes).  On the fast path (every byte < 8: alleles REF, ALT1, ALT2 or missing,
//    no sentinel) each byte carries its allele code (allele+1, 0 = missing) in bits 1-2, and ONE
//    byte-wise dot product, dp4a(w & 0x06060606, {132, 2, 8, 32}, table), is the address of the pair's
//    4-byte entry: a mask, an IDP.4A and an LDS.32 per two genotypes.  The entry index is
//    66*c0 + c1 + 4*c2 + 16*c3: injective over all 256 code
//    combinations, and -- unlike the plain base-4 index, whose top digit never reaches the bank
//    bits -- the 16 combinations of REF / ALT1 alleles fall into 16 different banks, so the lookups of a
//    warp are conflict-free on ordinary data (measured with base-4: 1.85 wavefronts per lookup).
//  * The entry holds the pair's two dosage codes already placed for the row's position in the tile
//    (top byte) and the pair's tally contribution in 6-bit fields (bits 0-23): entries of rows (0,1)
//    and of rows (2,3) are simply ADDED -- per word that gives the index-ring byte of both samples,
//    and the sum over the chunk's four words gives the tallies of two rows in one register.
//  * Tallies leave the warp with two RED.shared.add.u32 per chunk into per-lane counters (three
//    warps share a counter: 6-bit fields hold 3 x 16), no warp reduction, no lane-0 epilogue; the
//    publisher warp, which has time to spare, does the cross-lane sum once per tile.
//  * DECIDE builds, per tile, two 16-entry fp64 tables T01[b0|b1<<2] = v0[b0]+v1[b1] and
//    T23[b2|b3<<2] = v2[b2]+v3[b3] of the rows' contributions (constant rows and dropped rows fold
//    in as constants).  16 doubles span exactly the 32 banks: every lookup is conflict-free (one
//    256-entry table was measured at 3-way conflicts: its hot entries share 9 of 16 bank pairs).
//  * ACCUMULATE: sums[s] = (sums[s] + T01[..]) + T23[..] -- two LDS.64 and two DADD per sample per
//    four genotypes, no per-row branches.  The index-ring byte of a sample pair is
//    [sample 0: rows a,b | sample 1: rows a,b], one byte for rows (0,1) and one for rows (2,3).
//
//  * Wide cohorts.  One chunk (8 samples) per consumer thread up to 28 warps (~1.06 M samples on 148 CTAs); above that
//    two chunk SETS per tile (K = 2), each set a raw stage of its own, so the ring holds 3-4 half-tile stages where two
//    whole tiles would leave no room for the index ring.  Where the index ring is short (a tile of 1 M samples is 11 KB
//    of ring and 1.4 us of streaming) the deciders take 4 tiles per pass instead of 8: the first tile of a pass waits
//    for its last to be counted by the whole grid, and that wait must fit the lag.
//
// Rounding: the contributions of rows (0,1) and of rows (2,3) of a tile are added to each other
// first and then, in that order, to the running sum.  Every addend is still the reference's rounded
// product fl(dosage*beta); only the association differs from the reference's left-to-right chain
// (src/nimpress.nim:639-640), so scores agree to a few ulp of the running sum (tests assert <= 1e-12
// relative; the contract is 1e-9).  The result is deterministic; the association depends on how the
// rows are cut into launches and row groups (DESIGN 4.1), not on the sample slabs.
//
// EXACT = true (npc_set_exact_order) keeps everything above except the pre-summing: the tile's
// block holds the four rows' 4-entry tables and ACCUMULATE does one lookup and one DADD per
// genotype, rows in order -- the same rounded products and the same rounded adds as
// `scores[i] += dosages[i]*beta` (src/nimpress.nim:640), bit for bit.  It runs on a 1-D grid (every
// CTA sees every row) so that the per-sample chain is the reference's.
#pragma once
#include "npc_fused.cuh"

namespace npc {

constexpr int F5_NC_WIDE = 24;                // consumer warps of the K = 1 "wide" instance (72 registers); all others: 16
constexpr int F5_NC_MAX = 28;                 // ... and of the widest one: 32 warps per CTA, 64 registers (24 bytes of spills)
constexpr int F5_R = 4;                       // rows per tile
constexpr uint32_t F5_NT = 4;                 // tables per parity: T = 1, 2, 3 and "no allele matches" (T >= 4)
constexpr uint32_t F5_TAB_BYTES = 1152;       // 262 four-byte entries (index <= 3 * 87), padded to a multiple of 128
constexpr uint32_t F5_PACK_W = 0x20080284u;   // dp4a weights of bytes 0..3 of (w & 0x06060606): 4 * index = 132*b0 + 2*b1 + 8*b2 + 32*b3
constexpr int F5_GROUP = 3;                   // (warp, chunk) pairs per tally counter: 3 * 16 < 64

struct Fused5Smem {
    uint32_t code, vtab, vrow, bars, cnt, rflags, rtb, reaidx, idx, data, total;
    __host__ __device__ static int groups(int nc, int K) { return (nc * K + F5_GROUP - 1) / F5_GROUP; }
    __host__ __device__ static Fused5Smem make(int Sr, int Sc, int slab_stride, int nc, int K, int W = 1) {
        Fused5Smem m;
        uint32_t o = 0;
        m.code = o;   o += F5_NT * 2u * F5_TAB_BYTES;                    // first: 1024-byte aligned
        m.vtab = o;   o += (uint32_t)Sc * 256u;                          // 256-byte aligned: T01 at +0, T23 at +128
        m.vrow = o;   o += 6u * 128u * 8u;                               // per decider warp: 32 rows x 4 values
        m.bars = o;   o += (2u * Sr + 2u * Sc) * 8u;            o = (o + 127u) & ~127u;
        m.cnt = o;    o += (uint32_t)Sc * (uint32_t)groups(nc, K) * 256u;   // [tile slot][group][rows 01 | rows 23][lane]
        m.rflags = o; o += (uint32_t)Sr * 4u;                   o = (o + 127u) & ~127u;
        m.rtb = o;    o += (uint32_t)Sr * 16u;                  o = (o + 127u) & ~127u;
        m.reaidx = o; o += (uint32_t)Sr * 16u;                  o = (o + 127u) & ~127u;
        m.idx = o;    o += (uint32_t)Sc * (uint32_t)(slab_stride / (2 * W));  o = (o + 127u) & ~127u;   // one byte per sample per tile
        m.data = o;   o += (uint32_t)Sr * F5_R * (uint32_t)(slab_stride / K);    // a raw stage: one chunk set (1/K of the slab) of R rows
        m.total = o;
        return m;
    }
};

__device__ __forceinline__ ull globaltimer_ns() {
    ull t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// dosage code of one sample from its two allele codes (allele+1, 0 = missing): 0, 1, 2 or 3 = missing
__device__ __forceinline__ uint32_t f5_code(int ca, int cb, int T) {
    if (ca == 0 || cb == 0) return 3u;
    return (uint32_t)((ca == T) + (cb == T));
}
// what one sample adds to its word's entry: code placed for (row parity q, sample-in-word s), tally fields
__device__ __forceinline__ uint32_t f5_sample_entry(uint32_t c, int q, int s) {
    return (c << (24 + 2 * q + 4 * s)) | ((c == 3u ? 0u : c) << (6 * q)) | ((c == 3u ? 1u : 0u) << (12 + 6 * q));
}
// exact decode (any bytes) of the sample in the low 16 bits of h -> dosage code
__device__ __forceinline__ uint32_t f5_slow_code(uint32_t h, int eaidx) {
    int8_t a[2] = { (int8_t)(h & 0xFF), (int8_t)((h >> 8) & 0xFF) };
    int d; bool miss;
    decode_sample<int8_t>(a, 2, eaidx, d, miss);
    return miss ? 3u : (uint32_t)d;
}
// fast path: the entry of the two samples of word w in the row's table
__device__ __forceinline__ uint32_t f5_pair_entry(uint32_t w, uint32_t table) {
    return lds_u32(__dp4a(w & 0x06060606u, F5_PACK_W, table));             // table + 4 * (66*c0 + c1 + 4*c2 + 16*c3)
}
// int16 GT: a sample is one 32-bit word (two halfwords, each < 8 on the fast path, so their high bytes are zero);
// (w0 | w1 << 8) & 0x06060606 has bytes [c0(s0), c0(s1), c1(s0), c1(s1)] * 2 -- the same table, other weights
constexpr uint32_t F5_PACK_W16 = 0x20020884u;
__device__ __forceinline__ uint32_t f5_pair_entry16(uint32_t w0, uint32_t w1, uint32_t table) {
    return lds_u32(__dp4a((w0 | (w1 << 8)) & 0x06060606u, F5_PACK_W16, table));
}
__device__ __forceinline__ uint32_t f5_slow_code16(uint32_t word, int eaidx) {
    int16_t a[2] = { (int16_t)(word & 0xFFFF), (int16_t)(word >> 16) };
    int d; bool miss;
    decode_sample<int16_t>(a, 2, eaidx, d, miss);
    return miss ? 3u : (uint32_t)d;
}

// W = bytes per stored allele value: 1 (int8, the usual BCF GT) or 2 (int16: records with more than 63 alleles)
// NCMAX = most consumer warps the instance is launched with (+ producer + publisher + <= 2 deciders): 16 keeps up to 96
// registers per thread; the K = 1 instances for 17-24 and 25-28 warps are held to 72 and 64 (measured: each ~3 % slower than
// the next one up at equal warp count, but 0.95-0.99 of the roofline at 800-950 k samples where two chunks per thread on
// 11-13 warps reach 0.81-0.88, and 27 warps on half as many sample slabs beat 14 at 500 k because their lanes are fuller)
template <int K, bool EXACT, int W = 1, int NCMAX = 16>
__global__ void __launch_bounds__((NCMAX + 4) * 32, 1)
k_fused_pair(const FusedParams P) {
    constexpr int R = F5_R;
    constexpr uint32_t CELL = 16u * W;                 // bytes of a chunk (8 diploid samples) in a raw row
    constexpr uint32_t HI_MASK = W == 1 ? 0xF8F8F8F8u : 0xFFF8FFF8u;   // any value >= 8 (ALT3.., sentinels) leaves the fast path
    extern __shared__ __align__(1024) uint8_t smem[];
    const int Sr = P.Sr, Sc = P.Sc, L = P.L, NC = P.nc, A = P.A;
    const int NG = Fused5Smem::groups(NC, K);
    const Fused5Smem M = Fused5Smem::make(Sr, Sc, P.slab_stride, NC, K, W);
    const uint32_t sb = smem_u32(smem);
    const uint32_t bar_full = sb + M.bars, bar_rempty = bar_full + 8u * Sr, bar_cnt = bar_rempty + 8u * Sr, bar_lut = bar_cnt + 8u * Sc;
    uint32_t *s_rflags = reinterpret_cast<uint32_t *>(smem + M.rflags);
    uint32_t *s_rtb = reinterpret_cast<uint32_t *>(smem + M.rtb);
    int32_t *s_reaidx = reinterpret_cast<int32_t *>(smem + M.reaidx);
    const uint32_t cnt_slot = (uint32_t)NG * 256u;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // grid = Gs sample slabs x Gr row groups: this CTA owns chunk range `slab` of the sample axis and
    // the contiguous tile range [tile_lo, tile_lo + n_tiles) of the rows
    const int Gs = P.Gs, slab_id = (int)blockIdx.x % Gs, grp = (int)blockIdx.x / Gs;
    const int64_t all_tiles = (P.n_rows + R - 1) / R;
    const int64_t tile_lo = all_tiles * grp / P.Gr, n_tiles = all_tiles * (grp + 1) / P.Gr - tile_lo;
    const int64_t row_lo = tile_lo * R;

    const int64_t C = (P.n + 7) >> 3;
    const int64_t q_ = C / Gs, rem = C % Gs;
    const int64_t c0 = (int64_t)slab_id * q_ + min((int64_t)slab_id, rem);
    const int nch = (int)(q_ + ((int64_t)slab_id < rem ? 1 : 0));
    const uint32_t slab_bytes = (uint32_t)nch * CELL;
    const uint32_t hslab = (uint32_t)P.slab_stride / K;             // bytes per row of a raw stage (one chunk set)

    if (threadIdx.x == 0) {
        for (int s = 0; s < Sr; s++) { mbar_init(bar_full + 8u * s, 1); mbar_init(bar_rempty + 8u * s, NC); }
        for (int s = 0; s < Sc; s++) { mbar_init(bar_cnt + 8u * s, NC); mbar_init(bar_lut + 8u * s, 1); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (uint32_t i = threadIdx.x; i < (uint32_t)Sc * cnt_slot / 4u; i += blockDim.x)
        reinterpret_cast<uint32_t *>(smem + M.cnt)[i] = 0u;
    // Lanes past the slab's last chunk.  K = 1: they run along on the cells past the bytes the TMA copies write, which
    // nothing ever writes -- zero ("missing": every lane looks up the same entry, a broadcast) just that tail of the
    // ring, not the whole ring: ~1 us off every launch.  Their tallies are not published, their sums not stored.
    // K = 2: a stage alternates between the two chunk sets, its tail would hold an older set's genotypes and the idle
    // lanes' lookups would collide with the others' -- there they sit the loop bodies out.
    // (Measured both ways: predicating costs the K = 1 shapes with a partly filled warp 5 %, running along costs the
    // K = 2 shapes 3 %.)
    if (K == 1) {
        const uint32_t tail16 = (hslab - slab_bytes) / 16u;
        for (uint32_t i = threadIdx.x; i < (uint32_t)Sr * R * tail16; i += blockDim.x)
            reinterpret_cast<uint4 *>(smem + M.data + (i / tail16) * hslab + slab_bytes)[i % tail16] = make_uint4(0, 0, 0, 0);
    }
    if (P.counts_next)
        for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < P.n_zero; i += (int64_t)gridDim.x * blockDim.x) P.counts_next[i] = 0ull;
    if (P.trace && blockIdx.x == 0 && threadIdx.x == 0) P.trace[0] = globaltimer_ns();
    npc_row first_meta;                                  // producer: the first 32 rows' metadata, in flight across the barrier
    if (warp == NC) {
        const int64_t r = row_lo + lane;
        if (r < min(P.n_rows, (tile_lo + n_tiles) * R)) first_meta = P.rows[r];
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();

    if (warp == NC) {
        // ================= producer ============================================================
        // Row metadata is read 32 rows (8 tiles) at a time, one row per lane, and the NEXT group is
        // already in flight while this one is issued.
        const uint64_t pol = l2_evict_first_policy();
        constexpr int G = 32 / R;                                    // tiles per metadata group
        int s = 0; uint32_t ph = 0;
        const int64_t row_hi = min(P.n_rows, (tile_lo + n_tiles) * R);      // this group's rows: [row_lo, row_hi)
        npc_row nxt = first_meta;
        for (int64_t t0 = 0; t0 < n_tiles; t0 += G) {
            const npc_row cur = nxt;
            const int64_t my_row = row_lo + t0 * R + lane;
            const bool have = my_row < row_hi;
            {
                const int64_t r = my_row + 32;
                if (r < row_hi) nxt = P.rows[r];
            }
            const bool is_gt = have && cur.kind == NPC_KIND_GT && cur.gt_row >= 0;
            const bool is_odd = is_gt && cur.eaidx < 0;              // no table represents it: exact decode
            const uint32_t gt_all = __ballot_sync(0xffffffffu, is_gt), odd_all = __ballot_sync(0xffffffffu, is_odd);
            const int ng = (int)min((int64_t)G, n_tiles - t0);
            const int T = is_gt ? cur.eaidx + 1 : 99;
            const uint32_t my_tb = sb + M.code + (uint32_t)((T >= 1 && T <= 3 ? T - 1 : 3) * 2 + (lane & 1)) * F5_TAB_BYTES;
            for (int j = 0; j < ng; j++) {
                const uint32_t gt_mask = (gt_all >> (R * j)) & ((1u << R) - 1u);
                const bool mine = (lane / R) == j;                   // lanes R*j .. R*j+R-1 own this tile's rows
#pragma unroll
                for (int k = 0; k < K; k++) {                        // one raw stage per chunk set of the tile
                    const uint32_t lo = (uint32_t)k * hslab;
                    const uint32_t bytes = slab_bytes > lo ? min(slab_bytes - lo, hslab) : 0u;
                    mbar_wait(bar_rempty + 8u * s, ph ^ 1u);
                    if (mine) { s_reaidx[s * R + (lane % R)] = is_gt ? cur.eaidx : 0; s_rtb[s * R + (lane % R)] = my_tb; }
                    if (lane == 0) s_rflags[s] = gt_mask | (((odd_all >> (R * j)) & ((1u << R) - 1u)) << 4);
                    __syncwarp();
                    if (lane == 0) mbar_arrive_expect_tx(bar_full + 8u * s, (uint32_t)__popc(gt_mask) * bytes);
                    __syncwarp();
                    if (mine && is_gt && bytes)
                        tma_load_1d(sb + M.data + (uint32_t)(s * R + (lane % R)) * hslab,
                                    P.gt + (int64_t)cur.gt_row * P.row_stride + c0 * CELL + lo, bytes, bar_full + 8u * s, pol);
                    if (++s == Sr) { s = 0; ph ^= 1u; }
                }
            }
        }
    } else if (warp == NC + 1) {
        // ================= publisher ===========================================================
        // per tile: sum the per-lane counters of every group (and clear them), reduce over the lanes, one
        // 64-bit RED per row: tallies and arrival count in the same word, so the data is the flag
        int s = 0; uint32_t ph = 0;
        for (int64_t t = 0; t < (P.decided ? 0 : n_tiles); t++) {
            mbar_wait(bar_cnt + 8u * s, ph);
            const uint32_t base = sb + M.cnt + (uint32_t)s * cnt_slot + (uint32_t)lane * 4u;
            uint32_t d01 = 0, m01 = 0, d23 = 0, m23 = 0;             // 16-bit halves: row a | row b
            for (int g = 0; g < NG; g++) {
                const uint32_t a = lds_u32(base + (uint32_t)g * 256u), b = lds_u32(base + (uint32_t)g * 256u + 128u);
                sts_v1(base + (uint32_t)g * 256u, 0u); sts_v1(base + (uint32_t)g * 256u + 128u, 0u);
                d01 += (a & 0x3Fu) | ((a & 0xFC0u) << 10);  m01 += ((a >> 12) & 0x3Fu) | ((a & 0xFC0000u) >> 2);
                d23 += (b & 0x3Fu) | ((b & 0xFC0u) << 10);  m23 += ((b >> 12) & 0x3Fu) | ((b & 0xFC0000u) >> 2);
            }
            __threadfence_block();                                   // the counters are clear before the grid can learn of this tile
            d01 = __reduce_add_sync(0xffffffffu, d01); m01 = __reduce_add_sync(0xffffffffu, m01);
            d23 = __reduce_add_sync(0xffffffffu, d23); m23 = __reduce_add_sync(0xffffffffu, m23);
            const int nr = (int)min((int64_t)R, P.n_rows - (tile_lo + t) * R);
            if (lane < nr) {
                const uint32_t dd = lane < 2 ? d01 : d23, mm = lane < 2 ? m01 : m23;
                const ull eff = (lane & 1) ? (dd >> 16) : (dd & 0xFFFFu), miss = (lane & 1) ? (mm >> 16) : (mm & 0xFFFFu);
                red_relaxed_gpu_add_u64(P.counts + (tile_lo + t) * R + lane, (1ull << 56) | (miss << FUSED_CNT_BITS) | eff);
            }
            if (++s == Sc) { s = 0; ph ^= 1u; }
        }
    } else if (warp > NC + 1) {
        // ================= deciders ============================================================
        // One pass decides a GROUP of GD tiles, one row per lane (GD = 8: 32 rows): the global round trip
        // of the tally word (microseconds under load) is paid once per group, not once per tile.  The
        // first tile of a group waits for the last one to be counted everywhere, so the lag L must cover
        // GD tiles plus that round trip: shapes whose rings leave a short lag (wide cohorts: a tile of
        // 1M samples is 1.4 us of streaming and 11 KB of ring) run with GD = 4.
        // Groups rotate over the A decider warps.
        const int a = warp - NC - 2;
        const int GD = P.GD;                                         // tiles per group
        double *vrow = reinterpret_cast<double *>(smem + M.vrow) + a * 128;      // [row in group][code]
        const int64_t n_groups = (n_tiles + GD - 1) / GD;
        for (int64_t g = a; g < n_groups; g += A) {
            const int64_t t0 = g * GD;
            const int ng = (int)min((int64_t)GD, n_tiles - t0);
            const int64_t my_row = (tile_lo + t0) * R + lane;
            const bool have = lane < ng * R && my_row < P.n_rows;
            npc_row row;
            if (have) row = P.rows[my_row];                          // in flight while we wait
            {   // the grid cannot have arrived before this CTA has: sleep on the local barrier of the group's last tile first
                const int64_t tl = t0 + ng - 1;
                mbar_wait(bar_cnt + 8u * (uint32_t)(tl % Sc), (uint32_t)((tl / Sc) & 1));
            }
            double v0 = 0.0, v1 = 0.0, v2 = 0.0, v3 = 0.0;           // a dropped row adds +0.0: the identity
            int used = 0;
            if (have && P.decided) {
                const RowP rp = P.decided[my_row];
                if (rp.mode == MODE_DECODE) { v0 = rp.c0; v1 = rp.c1; v2 = rp.c2; v3 = rp.cm; }
                else if (rp.mode == MODE_CONST) { v0 = v1 = v2 = v3 = rp.c0; }
            } else if (have) {
                const ull *word = P.counts + my_row;
                ull v = ld_relaxed_gpu_u64(word);
                while ((v >> 56) != (ull)Gs) { __nanosleep(500); v = ld_relaxed_gpu_u64(word); }      // all slabs of this row group
                RowP rp; npc_locus rec;
                decide_row(P.pol, row, (v >> FUSED_CNT_BITS) & FUSED_CNT_MASK, v & FUSED_CNT_MASK, P.n, rp, rec);
                used = rec.used;
                if (slab_id == 0) P.log[my_row] = rec;
                if (rp.mode == MODE_DECODE) { v0 = rp.c0; v1 = rp.c1; v2 = rp.c2; v3 = rp.cm; }
                else if (rp.mode == MODE_CONST) { v0 = v1 = v2 = v3 = rp.c0; }
            }
            vrow[lane * 4 + 0] = v0; vrow[lane * 4 + 1] = v1; vrow[lane * 4 + 2] = v2; vrow[lane * 4 + 3] = v3;
            if (slab_id == 0 && !P.decided) {
                used = __reduce_add_sync(0xffffffffu, used);
                if (lane == 0 && used) atomicAdd(P.nloci, (ull)used);
            }
            __syncwarp();
            // per tile, default order: lanes 0..15 build T01[lane] = v0[lane&3] + v1[lane>>2], lanes 16..31
            // T23 from rows 2, 3.  Exact order: no pre-summing -- lanes 0..15 copy row (lane>>2)'s four
            // contributions to bytes 32*row + 8*code of the tile's block.
            const int h = lane >> 4, e = lane & 15;
            for (int j = 0; j < ng; j++) {
                const int s = (int)((t0 + j) % Sc);
                double *tab = reinterpret_cast<double *>(smem + M.vtab) + s * 32;
                if (EXACT) {
                    if (lane < 16) tab[lane] = vrow[j * R * 4 + lane];
                } else {
                    const double *vr = vrow + (j * R + 2 * h) * 4;
                    tab[lane] = __dadd_rn(vr[e & 3], vr[4 + (e >> 2)]);
                }
            }
            __syncwarp();
            if (lane < ng) mbar_arrive(bar_lut + 8u * (uint32_t)((t0 + lane) % Sc));
            __syncwarp();
        }
    } else {
        // ================= consumers ===========================================================
        // The code tables are the consumers' alone: they build them while the producer's first copies are in
        // flight, then meet on a named barrier of their own.
        // pair tables [T-1 (3 = no match)][row parity q][66*c0 + c1 + 4*c2 + 16*c3], c_k the allele code of byte k of
        // the word (sample 0 = bytes 0,1; sample 1 = bytes 2,3); the six unused entries of a table are never read
        for (uint32_t i = threadIdx.x; i < F5_NT * 2u * 256u; i += (uint32_t)NC * 32u) {
            const int cc = (int)(i & 255u), q = (int)((i >> 8) & 1u), Tm = (int)(i >> 9);
            const int T = Tm < 3 ? Tm + 1 : 99;
            const int c0 = cc & 3, c1 = (cc >> 2) & 3, c2 = (cc >> 4) & 3, c3 = cc >> 6;
            const uint32_t s0 = f5_code(c0, c1, T), s1 = f5_code(c2, c3, T);
            reinterpret_cast<uint32_t *>(smem + M.code + (uint32_t)(Tm * 2 + q) * F5_TAB_BYTES)[66 * c0 + c1 + 4 * c2 + 16 * c3] =
                f5_sample_entry(s0, q, 0) + f5_sample_entry(s1, q, 1);
        }
        asm volatile("bar.sync 1, %0;" ::"r"(NC * 32) : "memory");
        if (P.trace && blockIdx.x == 0 && threadIdx.x == 0) P.trace[1] = globaltimer_ns();
        uint32_t cell[K], tailor[K], cnt_off[K];
        bool own[K];                           // lanes past the slab's last chunk sit the loop bodies out
        int valid[K];
        double acc[K][8];                      // natural sample order: acc[2w + s] = sample s of word w
#pragma unroll
        for (int k = 0; k < K; k++) {
            const int jc = lane + 32 * (warp + NC * k);
            cell[k] = (uint32_t)jc;
            const int64_t g = c0 + jc;
            valid[k] = jc < nch ? (int)min((int64_t)8, P.n - g * 8) : 0;
            own[k] = jc < nch;
            tailor[k] = (jc < nch && valid[k] < 8) ? 0xF8u : 0u;                        // a set bit of HI_MASK: the cohort's last, partial chunk decodes exactly
            cnt_off[k] = (uint32_t)((warp * K + k) / F5_GROUP) * 256u + (uint32_t)lane * 4u;
#pragma unroll
            for (int e = 0; e < 8; e++) acc[k][e] = (e < valid[k] && grp == 0) ? P.sums[g * 8 + e] : 0.0;
        }
        double *sums_out = grp == 0 ? P.sums : P.partials + (int64_t)(grp - 1) * P.n;
        const uint32_t slab = (uint32_t)P.slab_stride, islab = slab / (2u * W);
        const int nt = (int)n_tiles;
        int sr = 0, sc = 0, sa = 0;
        uint32_t ph_r = 0, ph_a = 0;
        for (int i = 0; i < nt + L; i++) {
            if (i < nt) {
                const uint32_t cnt_base = sb + M.cnt + (uint32_t)sc * cnt_slot;
#pragma unroll
                for (int k = 0; k < K; k++) {                    // one raw stage per chunk set: wait, count, release
                  mbar_wait(bar_full + 8u * sr, ph_r);
                  if (K == 1 || own[k]) {
                    const uint32_t flags = s_rflags[sr];             // bits 0-3: row has genotypes; bits 4-7: row needs the exact decode
                    const uint32_t d0 = sb + M.data + (uint32_t)(sr * R) * hslab + (uint32_t)(lane + 32 * warp) * CELL;
                    const uint4 tb4 = lds_v4(sb + M.rtb + (uint32_t)sr * 16u);
                    const uint32_t tb[R] = { tb4.x, tb4.y, tb4.z, tb4.w };
                    uint32_t ww[R][4 * W];                       // the chunk's raw words, row by row
                    uint32_t hi_bits = tailor[k];
#pragma unroll
                    for (int r = 0; r < R; r++)                  // all loads of the tile first: independent LDS.128
#pragma unroll
                        for (int h = 0; h < W; h++) {
                            const uint4 v = lds_v4(d0 + r * hslab + 16u * h);
                            ww[r][4 * h] = v.x; ww[r][4 * h + 1] = v.y; ww[r][4 * h + 2] = v.z; ww[r][4 * h + 3] = v.w;
                            hi_bits |= (v.x | v.y) | (v.z | v.w);
                        }
                    uint32_t A4[4], B4[4];                       // per sample pair: entries of rows (0,1) / rows (2,3) added
                    if (flags == 0xFu && (hi_bits & HI_MASK) == 0u) {
                        // common case, straight line: every row has genotypes and every value is < 8: 16 independent pair lookups
                        uint32_t e[R][4];
#pragma unroll
                        for (int r = 0; r < R; r++)
#pragma unroll
                            for (int j = 0; j < 4; j++)
                                e[r][j] = W == 1 ? f5_pair_entry(ww[r][j], tb[r]) : f5_pair_entry16(ww[r][(2 * j) % (4 * W)], ww[r][(2 * j + 1) % (4 * W)], tb[r]);
#pragma unroll
                        for (int j = 0; j < 4; j++) { A4[j] = e[0][j] + e[1][j]; B4[j] = e[2][j] + e[3][j]; }
                    } else {
#pragma unroll
                        for (int j = 0; j < 4; j++) A4[j] = B4[j] = 0u;
#pragma unroll
                        for (int r = 0; r < R; r++) {
                            if (!((flags >> r) & 1u)) continue;
                            uint32_t e[4], any = 0u;
#pragma unroll
                            for (int j = 0; j < 4 * W; j++) any |= ww[r][j];
                            const uint32_t row_hi = (any & HI_MASK) | tailor[k] | ((flags >> (4 + r)) & 1u);
                            if (row_hi == 0u) {
#pragma unroll
                                for (int j = 0; j < 4; j++)
                                    e[j] = W == 1 ? f5_pair_entry(ww[r][j], tb[r]) : f5_pair_entry16(ww[r][(2 * j) % (4 * W)], ww[r][(2 * j + 1) % (4 * W)], tb[r]);
                            } else {                             // exact decode, same entry format
                                const int vk = own[k] ? valid[k] : 8;
                                const int ea = s_reaidx[sr * R + r];
#pragma unroll
                                for (int j = 0; j < 4; j++) {
                                    e[j] = 0u;
#pragma unroll
                                    for (int s = 0; s < 2; s++)
                                        if (2 * j + s < vk)
                                            e[j] += f5_sample_entry(W == 1 ? f5_slow_code((ww[r][j] >> (16 * s)) & 0xFFFFu, ea)
                                                                           : f5_slow_code16(ww[r][(2 * j + s) % (4 * W)], ea), r & 1, s);
                                }
                            }
#pragma unroll
                            for (int j = 0; j < 4; j++) { if (r < 2) A4[j] += e[j]; else B4[j] += e[j]; }
                        }
                    }
                    // tallies of rows (0,1) / (2,3): the low 24 bits of the sums over the chunk's four words (four
                    // 6-bit fields: d_a, d_b, m_a, m_b); whatever the code bytes add up to stays in the top byte
                    const uint32_t SA = (A4[0] + A4[1]) + (A4[2] + A4[3]), SB = (B4[0] + B4[1]) + (B4[2] + B4[3]);
                    if (own[k] && !P.decided) {
                        red_shared_add_u32(cnt_base + cnt_off[k], SA);
                        red_shared_add_u32(cnt_base + cnt_off[k] + 128u, SB);
                    }
                    // the tile's code bytes (top byte of each word's sum) -> index ring: x = rows (0,1), y = rows (2,3)
                    const uint32_t x = __byte_perm(__byte_perm(A4[0], A4[1], 0x0073), __byte_perm(A4[2], A4[3], 0x0073), 0x5410);
                    const uint32_t y = __byte_perm(__byte_perm(B4[0], B4[1], 0x0073), __byte_perm(B4[2], B4[3], 0x0073), 0x5410);
                    sts_v2(sb + M.idx + (uint32_t)sc * islab + cell[k] * 8u, x, y);
                  }
                  __syncwarp();
                  if (lane == 0) mbar_arrive(bar_rempty + 8u * sr);
                  if (++sr == Sr) { sr = 0; ph_r ^= 1u; }
                }
                // tallies and index bytes of the tile written
                __syncwarp();
                if (lane == 0) mbar_arrive(bar_cnt + 8u * sc);
                if (++sc == Sc) sc = 0;
                if (P.trace && blockIdx.x == 0 && threadIdx.x == 0 && (i == 0 || i == nt - 1)) P.trace[i == 0 ? 2 : 3] = globaltimer_ns();
            }
            if (i >= L) {
                mbar_wait(bar_lut + 8u * sa, ph_a);
                const uint32_t thi = (sb + M.vtab + (uint32_t)sa * 256u) >> 8;     // bits 8.. of the slot's table block
#pragma unroll
                for (int k = 0; k < K; k++) {
                    if (K != 1 && !own[k]) continue;
                    const uint2 v = lds_v2(sb + M.idx + (uint32_t)sa * islab + cell[k] * 8u);
                    if (EXACT) {
                        // the reference's chain: one rounded add per row, rows in order.  Row r's table holds
                        // its 4 contributions at bytes 32r + 8*code; a dropped row adds +0.0 (the identity)
#pragma unroll
                        for (int r = 0; r < R; r++) {
                            const uint32_t xy = r < 2 ? v.x : v.y;
#pragma unroll
                            for (int s = 0; s < 2; s++) {
                                const int sh = 2 * (r & 1) + 4 * s;                // the code sits at bits sh, sh+1 of the word's byte
                                const uint32_t sv = sh == 0 ? xy << 3 : sh == 2 ? xy << 1 : sh == 4 ? xy >> 1 : xy >> 3;
                                const uint32_t off = (sv & 0x18181818u) | (0x20202020u * (uint32_t)r);
#pragma unroll
                                for (int j = 0; j < 4; j++)
                                    acc[k][2 * j + s] = __dadd_rn(acc[k][2 * j + s], lds_f64(__byte_perm(off, thi, 0x6540 + j)));
                            }
                        }
                    } else {
                        // byte offsets of 4 samples at once: T01 entry nibble * 8, T23 entry 128 + nibble * 8
                        const uint32_t a0 = (v.x & 0x0F0F0F0Fu) << 3, a1 = (v.x >> 1) & 0x78787878u;
                        const uint32_t b0 = ((v.y & 0x0F0F0F0Fu) << 3) | 0x80808080u, b1 = ((v.y >> 1) & 0x78787878u) | 0x80808080u;
#pragma unroll
                        for (int j = 0; j < 4; j++) {
                            const double p0 = lds_f64(__byte_perm(a0, thi, 0x6540 + j)), q0 = lds_f64(__byte_perm(b0, thi, 0x6540 + j));
                            const double p1 = lds_f64(__byte_perm(a1, thi, 0x6540 + j)), q1 = lds_f64(__byte_perm(b1, thi, 0x6540 + j));
                            acc[k][2 * j] = __dadd_rn(__dadd_rn(acc[k][2 * j], p0), q0);
                            acc[k][2 * j + 1] = __dadd_rn(__dadd_rn(acc[k][2 * j + 1], p1), q1);
                        }
                    }
                }
                if (++sa == Sc) { sa = 0; ph_a ^= 1u; }
            }
        }
        if (P.trace && blockIdx.x == 0 && threadIdx.x == 0) P.trace[4] = globaltimer_ns();
#pragma unroll
        for (int k = 0; k < K; k++) {
            const int64_t g = c0 + cell[k];
#pragma unroll
            for (int e = 0; e < 8; e++)
                if (e < valid[k]) sums_out[g * 8 + e] = acc[k][e];
        }
        if (P.trace && blockIdx.x == 0 && threadIdx.x == 0) P.trace[5] = globaltimer_ns();
    }
}

}  // namespace npc
