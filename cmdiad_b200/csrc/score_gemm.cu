// Patch -> bank nearest-neighbour search as a fused tcgen05 distance GEMM (reference features.py:186-190 + :227).
//
// torch.cdist computes d^2 = ||a||^2 + ||b||^2 - 2 a.b with a float32 GEMM and the reference then takes min/argmin over
// the materialised [P,R] matrix.  Here the contraction runs on the 5th-generation tensor cores and the distance matrix
// never exists; the tensor cores only PROPOSE candidates, every returned distance / index comes from an exact float32
// re-check (score_tail.cu):
//   * TERMS = 1 (default): fp16 roundings of the power-of-two-scaled operands, one kind::f16 MMA per K step.  The
//     certificate in refine_cert_kernel bounds the error and proves which rows cannot be the nearest neighbour.
//     TERMS = 3: FP32-equivalent split, every value = fp16 hi + fp16 lo (22 significand bits), a.b ~= hi.hi + hi.lo +
//     lo.hi, three MMAs per K step into ONE fp32 TMEM accumulator (1.5x the tensor time of a plain fp16 GEMM, half that
//     of 3xTF32) -- selectable mode and fallback of the default mode;
//   * warp-specialised persistent CTAs (one per SM): warp 0 = TMA producer (SWIZZLE_128B tiles into a 4- / 2-stage
//     ring), warp 1 = single-thread tcgen05.mma issuer (M=128 queries x N=256 bank rows, accumulators double-buffered in
//     all 512 TMEM columns), warp 2 = TMEM allocation, warps 4-11 = two epilogue groups (column halves);
//     CG = 2 (TERMS = 3 only): CTA pairs (cluster of 2, cta_group::2, M = 256), each CTA stages its query tile and half
//     of the bank tile;
//   * epilogue: tcgen05.ld 32 columns at a time, val = ||b||^2 - 2 a.b (the per-query ||a||^2 is constant under argmin),
//     two branch-free top-2 chains per thread (value, bank row), carried across all tiles of the producer in a list in
//     L2 (296 producers x P x 16 B); one thread == one query row, so no cross-lane reduction is needed;
//   * one launch sweeps all M tiles of a batch in n-major order: the bank streams from HBM exactly once per launch and
//     the (small) query operand is re-read from L2; the tile schedule spreads every query's rows over all CTAs.
// Algorithmic work: 2*P*R*D FLOP per image (TERMS = 3 issues 3x that).
#include <cuda.h>

#include <cstdlib>

#include "common.cuh"

namespace cmdb {

constexpr int BM = kScoreBM;      // 128 query rows  (UMMA M)
constexpr int BN = kScoreBN;      // 256 bank rows   (UMMA N)
constexpr int BK = kScoreBK;      // 64 fp16 = 128 B swizzle row
constexpr int UMMA_K = 16;
constexpr int kGemmCtlThreads = 128;  // warps 0-3: TMA / MMA / TMEM alloc / idle; then EG groups of 4 epilogue warps
constexpr uint32_t kTileABytes = BM * BK * 2;  // 16 KB
constexpr uint32_t kTileBBytes = BN * BK * 2;  // 32 KB
constexpr uint32_t kTmemCols = 512;

// TERMS = 3: FP32-equivalent split (hi.hi + hi.lo + lo.hi)     TERMS = 1: hi.hi only (certified pre-filter)
// CG = 1: one CTA per tile (96 / 48 KB per stage, 2 / 4 stages)
// CG = 2: CTA pair, tcgen05 cta_group::2: M = 256 (128 query rows per CTA), each CTA stages its own A tile and HALF of the
//         bank tile (64 / 32 KB per stage, 3 / 6 stages) -- the tensor core reads every bank element from shared memory
//         once per pair instead of once per CTA
template <int TERMS, int CG>
struct GemmSmem {  // offsets inside dynamic shared memory (1024-byte aligned base)
    static constexpr uint32_t kTileB = kTileBBytes / CG;
    static constexpr int kStages = (TERMS == 3 ? 2 : 4) * (CG == 2 ? 3 : 2) / 2;
    static constexpr uint32_t kStageBytes = (TERMS == 3 ? 2u : 1u) * (kTileABytes + kTileB);
    static constexpr uint32_t stage(int s) { return s * kStageBytes; }
    static constexpr uint32_t a_hi(int s) { return stage(s); }
    static constexpr uint32_t b_hi(int s) { return stage(s) + kTileABytes; }
    static constexpr uint32_t a_lo(int s) { return stage(s) + kTileABytes + kTileB; }
    static constexpr uint32_t b_lo(int s) { return stage(s) + 2 * kTileABytes + kTileB; }
    static constexpr uint32_t bnorm = kStages * kStageBytes;              // [2][BN] float
    static constexpr uint32_t bars = bnorm + 2 * BN * 4;                  // mbarriers
    static constexpr uint32_t total = bars + 128;
};

// ---------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"(bar),
        "r"(parity)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap *tmap, uint32_t bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// ---- CTA-pair (cta_group::2) forms
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t map_to_cta(uint32_t smem_addr, uint32_t rank) {  // shared::cluster address of a peer's smem
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_addr), "r"(rank));
    return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// both CTAs of the pair issue their loads; the transaction bytes are credited to the barrier `bar_cluster_addr`, which
// lives in the LEADER's shared memory
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap *tmap, uint32_t bar_cluster_addr, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
        "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar_cluster_addr), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t dst_smem, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst_smem), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_f16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
        "}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrives on the barrier at this shared-memory offset in BOTH CTAs of the pair once all prior MMAs have retired
__device__ __forceinline__ void umma_commit_pair(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
                 "h"((unsigned short)3)
                 : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, "
        "[%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start address >> 4 in [0,14),
// LBO in [16,30) (unused for a single swizzle atom along K), SBO = 8 rows * 128 B = 1024 B >> 4 in [32,46),
// version 1 in [46,48), layout type SWIZZLE_128B (2) in [61,64).
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFFu) >> 4);
    d |= (uint64_t)((8u * BK * 2u) >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}
// kind::f16 instruction descriptor (cute::UMMA::InstrDescriptor): D fp32 (bits 4-5 = 1), A/B fp16 (0), both K-major,
// N >> 3 in [17,23), M >> 4 in [24,29)
constexpr uint32_t kIdesc = (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
constexpr uint32_t kIdescPair = (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)((2 * BM) >> 4) << 24);  // M = 256 over 2 CTAs

// Tile schedule shared by the three warp roles: N tiles in order (the bank streams from HBM once); the mt M tiles of
// N tile n go to the consecutive CTAs (n*s + m) % G, where the stride s >= mt is the next integer coprime with G.
// With s == mt this is plain round-robin dealing; making s coprime with G keeps the load balanced (every G N-tiles each
// CTA receives exactly mt tiles) AND lets every CTA see ~R/G rows of every query whatever gcd(mt, G) is -- the
// certificate of the pre-filter (score_tail.cu) needs the rows inside a query's error band to land in different CTAs'
// top-2 lists.  (tile_stride, common.cuh; the host records the same schedule in GemmSched.)
// c: this CTA (or CTA pair), G: number of CTAs (pairs), mt: M tiles (M tile pairs) per N tile
struct TileIter {  // n, m: current tile; base: first M tile of this CTA inside N tile n
    int n, m, base, smod, G;
    __device__ __forceinline__ TileIter(int c, int G_, int mt, int stride) {
        G = G_;
        smod = stride % G;
        n = -1, m = mt, base = (c + smod) % G;
    }
    // incremental form of m = (c - n * stride) mod G: no division per step (a CTA walks over ALL N tiles, also the ones in
    // which it owns no M tile, so the step has to be cheap when mt is small)
    __device__ __forceinline__ bool next(int mt, int nt) {
        m += G;
        while (m >= mt) {
            if (++n >= nt) return false;
            base -= smod;
            if (base < 0) base += G;
            m = base;
        }
        return true;
    }
};

// running two smallest (value, bank row) of a stream visited in ascending row order: ties keep the lower row
struct Top2 {
    float b1, b2;
    int i1, i2;
};
__device__ __forceinline__ void top2_update(Top2 &t, float v, int col) {
    const bool c1 = v < t.b1, c2 = v < t.b2;
    t.i2 = c1 ? t.i1 : (c2 ? col : t.i2);
    t.b2 = fminf(t.b2, fmaxf(t.b1, v));
    t.i1 = c1 ? col : t.i1;
    t.b1 = fminf(t.b1, v);
}
// general insert (rows in any order): lexicographic (value, row); row < 0 = empty
__device__ __forceinline__ void top2_insert(Top2 &t, float v, int i) {
    if (i < 0) return;
    const bool c1 = t.i1 < 0 || v < t.b1 || (v == t.b1 && i < t.i1);
    const bool c2 = t.i2 < 0 || v < t.b2 || (v == t.b2 && i < t.i2);
    if (c1) t.b2 = t.b1, t.i2 = t.i1, t.b1 = v, t.i1 = i;
    else if (c2) t.b2 = v, t.i2 = i;
}
// 32 accumulator columns of one query row: v = ||b||^2 - 2 a.b, even columns feed list A, odd columns list B
__device__ __forceinline__ void top2_chunk(const uint32_t (&r)[32], float c, const float *bn, int col, Top2 &ta, Top2 &tb) {
#pragma unroll
    for (int k = 0; k < 32; k += 2) {
        top2_update(ta, fmaf(__uint_as_float(r[k]), c, bn[k]), col + k);
        top2_update(tb, fmaf(__uint_as_float(r[k + 1]), c, bn[k + 1]), col + k + 1);
    }
}

struct GemmParams {
    int mt;             // M tiles (padded query rows / 128) handled by this launch
    int m_base;         // first M tile of this launch inside the query operand / the candidate lists
    const int *m_count; // optional device-side query-row count that overrides mt (fallback launch over the compacted
                        // uncertified queries; 0 rows -> the kernel returns at once)
    int nt;             // N tiles (bank rows / 256)
    int kb;             // K blocks (D / 64)
    const float *bnorm; // [nt*256] ||b||^2, +inf on padding rows
    const int *q_scale_exp;
    int b_scale_exp;
    float4 *cand;       // [gridDim.x][cand_stride]: CTA c keeps its running top-2 of query row q at cand[c*cand_stride + q]
    int cand_stride;    // >= mt * 128
    int run;            // consecutive N tiles a unit processes for one M tile before it moves on: the running top-2 stays
                        // in registers across the run, so the lists are read / written once per RUN tiles (see score_gemm_run)
};

template <int TERMS, int EG, int CG>
__global__ void __launch_bounds__(kGemmCtlThreads + 128 * EG, 1)
score_gemm_kernel(const __grid_constant__ CUtensorMap tm_qhi, const __grid_constant__ CUtensorMap tm_qlo,
                  const __grid_constant__ CUtensorMap tm_bhi, const __grid_constant__ CUtensorMap tm_blo, GemmParams p) {
    using S = GemmSmem<TERMS, CG>;
    constexpr int kGemmThreads = kGemmCtlThreads + 128 * EG;
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    // SWIZZLE_128B tiles need 1024-byte alignment; the launch reserves 1 KB of slack for this round-up
    unsigned char *smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
    const uint32_t sbase = smem_u32(smem);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (p.m_count) {
        p.mt = (__ldg(p.m_count) + BM - 1) / BM;
        if (p.mt == 0) return;  // uniform over the grid, before any barrier / TMEM allocation
    }
    // CG == 2: the two CTAs of a cluster form a pair; the pair owns M tiles 2*mp and 2*mp + 1 (one per CTA) of its tiles
    const int rank = CG == 2 ? (int)cluster_ctarank() : 0;
    const int unit = (int)blockIdx.x / CG, n_units = (int)gridDim.x / CG;  // scheduling unit = CTA or CTA pair
    const int mt_units = (p.mt + CG - 1) / CG;
    const int stride = tile_stride(mt_units, n_units);
    const int nruns = (p.nt + p.run - 1) / p.run;  // the schedule deals (run of N tiles, M tile) pairs instead of single tiles
    // barriers: full[S::kStages], empty[S::kStages], tmem_full[2], tmem_empty[2], then the TMEM base address slot
    // (pair: full[] and tmem_empty[] are only used in the leader, rank 0; empty[] and tmem_full[] exist in both CTAs and
    // are signalled by the leader's multicast commits)
    const uint32_t bar_full = sbase + S::bars, bar_empty = bar_full + 8 * S::kStages;
    const uint32_t bar_tfull = bar_empty + 8 * S::kStages, bar_tempty = bar_tfull + 16;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(smem + S::bars + 8 * (2 * S::kStages + 4));
    float *bnorm_s = reinterpret_cast<float *>(smem + S::bnorm);
    // running per-query top-2 of this CTA: lives in global memory (L2), 2 KB read + written per tile, so one launch can
    // sweep any number of M tiles in n-major order (the bank is then read from HBM exactly once per launch)
    // (each epilogue warp group keeps its own list: producer id = EG * CTA + column group)
    float4 *state = p.cand + (size_t)blockIdx.x * EG * p.cand_stride;

    if (warp == 1 && lane == 0) {
        for (int s = 0; s < S::kStages; ++s) {
            mbar_init(bar_full + 8 * s, 1);
            mbar_init(bar_empty + 8 * s, 1);
        }
        for (int b = 0; b < 2; ++b) {
            mbar_init(bar_tfull + 8 * b, 1);
            mbar_init(bar_tempty + 8 * b, 4 * EG * CG);  // one arrival per epilogue warp (of both CTAs of a pair)
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        if constexpr (CG == 2) tmem_alloc_pair(smem_u32(tmem_slot), kTmemCols);
        else tmem_alloc(smem_u32(tmem_slot), kTmemCols);
    }
    for (int i = p.m_base * BM + threadIdx.x; i < (p.m_base + p.mt) * BM; i += kGemmThreads)
#pragma unroll
        for (int g = 0; g < EG; ++g)
            state[(size_t)g * p.cand_stride + i] = make_float4(INFINITY, __int_as_float(-1), INFINITY, __int_as_float(-1));
    __threadfence_block();
    tc_fence_before();
    __syncthreads();
    if constexpr (CG == 2) cluster_sync_all();  // the peer's barriers are initialised before anything is signalled there
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp == 0) {
        // ================= TMA producer (every CTA loads its own query tile and its share of the bank tile) =================
        if (lane == 0) {
            int stage = 0;
            uint32_t phase = 0;
            for (TileIter it(unit, n_units, mt_units, stride); it.next(mt_units, nruns);) {
              const int m = it.m * CG + rank;
              for (int n = it.n * p.run, n_end = min(p.nt, n + p.run); n < n_end; ++n) {
                const int a_row = (p.m_base + m) * BM, b_row = n * BN + rank * (BN / CG);
                for (int kb = 0; kb < p.kb; ++kb) {
                    mbar_wait(bar_empty + 8 * stage, phase ^ 1);
                    if constexpr (CG == 2) {
                        const uint32_t full = map_to_cta(bar_full + 8 * stage, 0);  // the leader's barrier
                        if (rank == 0) mbar_expect_tx(bar_full + 8 * stage, 2 * S::kStageBytes);
                        tma_load_2d_pair(sbase + S::a_hi(stage), &tm_qhi, full, kb * BK, a_row);
                        tma_load_2d_pair(sbase + S::b_hi(stage), &tm_bhi, full, kb * BK, b_row);
                        if constexpr (TERMS == 3) {
                            tma_load_2d_pair(sbase + S::a_lo(stage), &tm_qlo, full, kb * BK, a_row);
                            tma_load_2d_pair(sbase + S::b_lo(stage), &tm_blo, full, kb * BK, b_row);
                        }
                    } else {
                        const uint32_t full = bar_full + 8 * stage;
                        mbar_expect_tx(full, S::kStageBytes);
                        tma_load_2d(sbase + S::a_hi(stage), &tm_qhi, full, kb * BK, a_row);
                        tma_load_2d(sbase + S::b_hi(stage), &tm_bhi, full, kb * BK, b_row);
                        if constexpr (TERMS == 3) {
                            tma_load_2d(sbase + S::a_lo(stage), &tm_qlo, full, kb * BK, a_row);
                            tma_load_2d(sbase + S::b_lo(stage), &tm_blo, full, kb * BK, b_row);
                        }
                    }
                    if (++stage == S::kStages) stage = 0, phase ^= 1;
                }
              }
            }
        }
    } else if (warp == 1) {
        // ================= MMA issuer (one thread; in a pair only the leader CTA issues) =================
        if (lane == 0 && rank == 0) {
            int stage = 0;
            uint32_t phase = 0;
            int j = 0;
            for (TileIter it(unit, n_units, mt_units, stride); it.next(mt_units, nruns);)
              for (int n = it.n * p.run, n_end = min(p.nt, n + p.run); n < n_end; ++n, ++j) {
                const int buf = j & 1;
                mbar_wait(bar_tempty + 8 * buf, ((j >> 1) & 1) ^ 1);
                tc_fence_after();
                const uint32_t tmem_d = tmem_base + buf * BN;
                for (int kb = 0; kb < p.kb; ++kb) {
                    mbar_wait(bar_full + 8 * stage, phase);
                    tc_fence_after();
                    const uint64_t a_hi = make_sw128_desc(sbase + S::a_hi(stage));
                    const uint64_t a_lo = make_sw128_desc(sbase + S::a_lo(stage));
                    const uint64_t b_hi = make_sw128_desc(sbase + S::b_hi(stage));
                    const uint64_t b_lo = make_sw128_desc(sbase + S::b_lo(stage));
#pragma unroll
                    for (int ks = 0; ks < BK / UMMA_K; ++ks) {
                        const uint64_t adv = (uint64_t)((ks * UMMA_K * 2) >> 4);  // +32 B per K step inside the swizzle row
                        if constexpr (CG == 2) {
                            umma_f16_pair(tmem_d, a_hi + adv, b_hi + adv, kIdescPair, (kb | ks) != 0);
                            if constexpr (TERMS == 3) {
                                umma_f16_pair(tmem_d, a_hi + adv, b_lo + adv, kIdescPair, 1);
                                umma_f16_pair(tmem_d, a_lo + adv, b_hi + adv, kIdescPair, 1);
                            }
                        } else {
                            umma_f16(tmem_d, a_hi + adv, b_hi + adv, kIdesc, (kb | ks) != 0);
                            if constexpr (TERMS == 3) {
                                umma_f16(tmem_d, a_hi + adv, b_lo + adv, kIdesc, 1);
                                umma_f16(tmem_d, a_lo + adv, b_hi + adv, kIdesc, 1);
                            }
                        }
                    }
                    // frees the smem stage (in both CTAs of a pair) when these MMAs retire
                    if constexpr (CG == 2) umma_commit_pair(bar_empty + 8 * stage);
                    else umma_commit(bar_empty + 8 * stage);
                    if (++stage == S::kStages) stage = 0, phase ^= 1;
                }
                // accumulator complete
                if constexpr (CG == 2) umma_commit_pair(bar_tfull + 8 * buf);
                else umma_commit(bar_tfull + 8 * buf);
            }
        }
    } else if (warp >= 4) {
        // ================= epilogue: EG groups of 4 warps; thread == (query row, column group) =================
        // A warp may only touch the TMEM lane quarter warp % 4, so group g (warps 4+4g .. 7+4g) takes columns
        // [g, g+1) * 256/EG of every accumulator.  Each group owns a separate running list (no merge needed: the refine
        // kernels treat every (CTA, group) as one producer).  In a pair each CTA's TMEM holds the accumulator rows of its
        // own 128 queries against all 256 bank rows of the tile.
        const int quarter = warp & 3;            // TMEM lane quarter this warp may access
        const int half = (warp - 4) >> 2;        // column group of the accumulator
        const int row = quarter * 32 + lane;     // row inside the M tile
        const int et = threadIdx.x - kGemmCtlThreads;  // 0 .. 128*EG-1
        constexpr int kHalfCols = BN / EG;
        float4 *my_state = state + (size_t)half * p.cand_stride;
        const uint32_t tempty_leader = CG == 2 ? map_to_cta(bar_tempty, 0) : bar_tempty;
        auto release_tmem = [&](int buf) {  // one arrival per warp on the (leader's) tmem_empty barrier
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if constexpr (CG == 2) mbar_arrive_cluster(tempty_leader + 8 * buf);
                else mbar_arrive(bar_tempty + 8 * buf);
            }
        };
        int j = 0;
        for (TileIter it(unit, n_units, mt_units, stride); it.next(mt_units, nruns);) {
          const int m_tile = it.m * CG + rank;
          const bool valid = m_tile < p.mt;    // odd M-tile count: the pair's last second tile does not exist
          const int m_local = p.m_base + m_tile;
          float c = 0.f;
          // running top-2 of this producer for its query row: loaded once per run of N tiles, carried in registers
          Top2 ta{INFINITY, INFINITY, -1, -1};
          if (valid) {
              // -2 * 2^-(e_bank + e_query_row): undoes the operand scaling and applies the -2 of ||a-b||^2
              c = ldexpf(-2.f, -(p.b_scale_exp + __ldg(p.q_scale_exp + m_local * BM + row)));
              const float4 st = my_state[m_local * BM + row];
              ta = Top2{st.x, st.z, __float_as_int(st.y), __float_as_int(st.w)};
          }
          for (int n = it.n * p.run, n_end = min(p.nt, n + p.run); n < n_end; ++n, ++j) {
            const int buf = j & 1;
            float *bn = bnorm_s + buf * BN;
            // bank norms of this N tile (buffer `buf` was last read two tiles ago, before that tile's tmem_empty arrive)
#pragma unroll
            for (int g = 0; g < 2 / EG; ++g) bn[et + g * 128 * EG] = __ldg(p.bnorm + (size_t)n * BN + et + g * 128 * EG);
            // two independent running top-2 lists (even / odd columns) halve the dependent min/select chain; list A
            // continues this producer's state for the query, list B starts empty and is merged into A after the tile
            Top2 tb{INFINITY, INFINITY, -1, -1};
            mbar_wait(bar_tfull + 8 * buf, (j >> 1) & 1);
            tc_fence_after();
            asm volatile("bar.sync 1, %0;" ::"n"(128 * EG) : "memory");  // bn[] visible to all epilogue warps
            if (!valid) {
                release_tmem(buf);
                continue;
            }
            const uint32_t taddr = tmem_base + ((uint32_t)(quarter * 32) << 16) + buf * BN + half * kHalfCols;
            const int col0 = n * BN + half * kHalfCols;
            const float *bnh = bn + half * kHalfCols;
            // tcgen05.ld of chunk ch + 1 is in flight while chunk ch is processed (ping-pong register sets)
            uint32_t ra[32], rb[32];
            tmem_ld32(taddr, ra);
#pragma unroll 1
            for (int ch = 0; ch < kHalfCols / 32; ch += 2) {
                tmem_ld_wait();
                tmem_ld32(taddr + (ch + 1) * 32, rb);
                top2_chunk(ra, c, bnh + ch * 32, col0 + ch * 32, ta, tb);
                tmem_ld_wait();
                if (ch + 2 < kHalfCols / 32) tmem_ld32(taddr + (ch + 2) * 32, ra);
                else release_tmem(buf);  // this warp's part of the accumulator is in registers: hand the buffer back early
                top2_chunk(rb, c, bnh + (ch + 1) * 32, col0 + (ch + 1) * 32, ta, tb);
            }
            top2_insert(ta, tb.b1, tb.i1);
            top2_insert(ta, tb.b2, tb.i2);
          }
          if (valid) my_state[m_local * BM + row] = make_float4(ta.b1, __int_as_float(ta.i1), ta.b2, __int_as_float(ta.i2));
        }
    }
    tc_fence_before();
    __syncthreads();
    if constexpr (CG == 2) cluster_sync_all();  // the leader's MMAs read the peer's shared memory until the very end
    if (warp == 2) {
        tc_fence_after();
        if constexpr (CG == 2) tmem_dealloc_pair(tmem_base, kTmemCols);
        else tmem_dealloc(tmem_base, kTmemCols);
    }
}

// ---------------------------------------------------------------- query preparation
// One warp per query row: per-ROW power-of-two scale (max|q_row| -> [2^12, 2^13)), q * 2^e -> fp16 hi/lo; rows >= P are
// zero.  A per-row scale needs no grid-wide reduction (one launch, no host sync) and is free in the GEMM epilogue,
// where one thread owns one query row.  Also emits ||q|| and ||q - q_hi|| (true units, rounded up) for the certificate
// of the pre-filter.  Compact mode (list != nullptr): output row r is query list[r], r < *count (device-side count).
__global__ void __launch_bounds__(256) q_split_kernel(const float *__restrict__ q, int P, int P_pad, int dim,
                                                      __half *__restrict__ hi, __half *__restrict__ lo,
                                                      int *__restrict__ scale_exp_out, float *__restrict__ q_norm,
                                                      float *__restrict__ q_eps, const int *__restrict__ list,
                                                      const int *__restrict__ count) {
    const int lane = threadIdx.x & 31, dim4 = dim >> 2;
    if (count) {
        P = __ldg(count);
        P_pad = (P + BM - 1) / BM * BM;
    }
    for (int r = blockIdx.x * 8 + (threadIdx.x >> 5); r < P_pad; r += gridDim.x * 8) {
        uint2 *h = reinterpret_cast<uint2 *>(hi + (size_t)r * dim), *l = reinterpret_cast<uint2 *>(lo + (size_t)r * dim);
        const float *src = q + (size_t)((list && r < P) ? __ldg(list + r) : r) * dim;
        float amax = 0.f;
        if (r < P)
            for (int cc = lane; cc < dim4; cc += 32) {
                const float4 v = __ldg(reinterpret_cast<const float4 *>(src) + cc);
                amax = fmaxf(fmaxf(amax, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
            }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) amax = fmaxf(amax, __shfl_xor_sync(0xffffffffu, amax, o));
        int e = 0;
        if (amax > 0.f && amax < INFINITY) {
            int ex;
            frexpf(amax, &ex);
            e = 13 - ex;
        }
        if (lane == 0) scale_exp_out[r] = e;
        const float scale = ldexpf(1.f, e);
        float n2 = 0.f, e2 = 0.f;  // ||q * scale||^2 and ||q * scale - hi||^2 (the residuals are exact in float32)
        for (int cc = lane; cc < dim4; cc += 32) {
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (r < P) v = __ldg(reinterpret_cast<const float4 *>(src) + cc);
            v.x *= scale, v.y *= scale, v.z *= scale, v.w *= scale;
            __half2 h0 = __floats2half2_rn(v.x, v.y), h1 = __floats2half2_rn(v.z, v.w);
            const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
            const float r0 = v.x - f0.x, r1 = v.y - f0.y, r2 = v.z - f1.x, r3 = v.w - f1.y;
            n2 = fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, fmaf(v.w, v.w, n2))));
            e2 = fmaf(r0, r0, fmaf(r1, r1, fmaf(r2, r2, fmaf(r3, r3, e2))));
            __half2 l0 = __floats2half2_rn(r0, r1), l1 = __floats2half2_rn(r2, r3);
            h[cc] = make_uint2(*reinterpret_cast<unsigned int *>(&h0), *reinterpret_cast<unsigned int *>(&h1));
            l[cc] = make_uint2(*reinterpret_cast<unsigned int *>(&l0), *reinterpret_cast<unsigned int *>(&l1));
        }
        if (q_norm) {
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                n2 += __shfl_xor_sync(0xffffffffu, n2, o);
                e2 += __shfl_xor_sync(0xffffffffu, e2, o);
            }
            if (lane == 0) {  // float32 sums of <= 2^20 non-negative terms: 1e-3 relative slack covers their rounding
                const float inv = ldexpf(1.f, -e);
                q_norm[r] = __fmul_ru(__fsqrt_ru(n2), inv) * 1.001f;
                q_eps[r] = __fmul_ru(__fsqrt_ru(e2), inv) * 1.001f;
            }
        }
    }
}

// ---------------------------------------------------------------- tensor maps
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

// fp16 [rows, dim] row-major, box = [box_rows, 64] (128 B inner extent), SWIZZLE_128B
static int make_map(void **slot, const __half *base, long long rows, int dim, int box_rows) {
    EncodeTiledFn fn = get_encode_fn();
    CMDB_REQUIRE(fn != nullptr, CMDB_ERR_CUDA, "cuTensorMapEncodeTiled is not available from the driver");
    if (!*slot) *slot = aligned_alloc(64, sizeof(CUtensorMap));
    cuuint64_t gdim[2] = {(cuuint64_t)dim, (cuuint64_t)rows};
    cuuint64_t gstr[1] = {(cuuint64_t)dim * 2};
    cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = fn(reinterpret_cast<CUtensorMap *>(*slot), CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, (void *)base, gdim, gstr, box,
                    estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                    CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    CMDB_REQUIRE(r == CUDA_SUCCESS, CMDB_ERR_CUDA, "cuTensorMapEncodeTiled failed with CUresult %d", (int)r);
    return CMDB_OK;
}

int score_make_tensor_maps(cmdb_bank *b) {
    CMDB_CHECK(make_map(&b->tmap_hi, b->hi, b->fin_rows_pad, b->dim, BN));
    CMDB_CHECK(make_map(&b->tmap_lo, b->lo, b->fin_rows_pad, b->dim, BN));
    CMDB_CHECK(make_map(&b->tmap_hi2, b->hi, b->fin_rows_pad, b->dim, BN / 2));  // half tiles for the CTA-pair kernels
    CMDB_CHECK(make_map(&b->tmap_lo2, b->lo, b->fin_rows_pad, b->dim, BN / 2));
    return CMDB_OK;
}

void gemm_prefer_carveout() {
    CMDB_PREFER_MAX_SMEM(q_split_kernel);
    (void)cudaGetLastError();
}

template <typename... T>
static void free_dev(T *&...p) {
    ((cudaFree(p), p = nullptr), ...);
}

static void free_lane(Lane &l) {
    free_dev(l.q_hi, l.q_lo, l.q_scale_exp, l.cand, l.topk_keys, l.map_tmp, l.map_max, l.m_test, l.m_star, l.top3,
             l.done_counter, l.q_norm, l.q_eps, l.fail_list, l.fail_ctl, l.work_list, l.best_key);
    l.s_key = nullptr;   // lives inside the fail_ctl allocation
    if (l.fail_count_host) cudaFreeHost(l.fail_count_host);
    free(l.tmap_qhi), free(l.tmap_qlo);
    l.fail_count_host = nullptr, l.tmap_qhi = l.tmap_qlo = nullptr;
}

// callers make sure that no submitted call is outstanding: its results would be lost
void score_scratch_free(cmdb_bank *b) {
    // no copy or kernel may still be in flight into / out of the buffers
    if (b->copy_stream) cudaStreamSynchronize(b->copy_stream);
    if (b->d2h_stream) cudaStreamSynchronize(b->d2h_stream);
    for (const Lane &l : b->lane) {
        if (l.stream) cudaStreamSynchronize(l.stream);
        if (l.aux) cudaStreamSynchronize(l.aux);
    }
    for (ResultSlot &s : b->slot) {
        free_dev(s.q_f32, s.out_block);
        if (s.out_block_host) cudaFreeHost(s.out_block_host);
        s.out_block_host = nullptr;
    }
    for (Lane &l : b->lane) free_lane(l);
    b->layout = ScoreLayout();
    b->round.open = false;   // an open sharded round lived in these buffers
    b->last_fail_host = nullptr;
    b->fail_pending = false;
}

int score_max_batch(const cmdb_bank *b) {
    // reweight_kernel keeps B m_star rows (B*dim floats) + 8*B*3 keys in shared memory
    const int by_smem = (int)((160 * 1024) / (sizeof(float) * b->dim + 8 * 3 * sizeof(unsigned long long)));
    return std::max(1, std::min(32, by_smem));
}

ScoreCall score_call(cmdb_bank *b, int lane, int slot) {
    const ScoreLayout &L = b->layout;
    ResultSlot &rs = b->slot[slot];
    unsigned char *blk = rs.out_block;
    b->last_lane = lane;
    return ScoreCall{b, lane, slot, &b->lane[lane], &rs, b->lane[lane].stream, reinterpret_cast<TailResult *>(blk),
                     reinterpret_cast<float *>(blk + L.off_min_val), reinterpret_cast<long long *>(blk + L.off_min_idx),
                     reinterpret_cast<float *>(blk + L.off_map_out), reinterpret_cast<float *>(blk + L.off_map_pre),
                     blk + L.off_map_u8};
}

int score_mark(const ScoreCall &c, int stage, cudaStream_t st) {
    const cmdb_bank *b = c.b;
    if (b->timing && stage >= 0) CMDB_CUDA(cudaEventRecord(b->timing == 2 ? c.lane->ev_tl[stage] : b->ev[stage], st));
    return CMDB_OK;
}

int score_scratch_alloc(cmdb_bank *b, int B, int P_img, int out_hw) {
    const int p_pad = (B * P_img + BM - 1) / BM * BM;
    const int map_n = out_hw * out_hw;
    ScoreLayout &L = b->layout;
    if (L.cap_p >= p_pad && L.cap_b >= B && (int)L.map_stride >= map_n) return CMDB_OK;
    CMDB_REQUIRE(!b->any_pending(), CMDB_ERR_STATE,
                 "scoring: the scratch buffers have to grow while a submitted batch is outstanding; wait for it first");
    const int cap_p = std::max(p_pad, L.cap_p), cap_b = std::max(B, L.cap_b);
    const int map_cap = std::max(map_n, (int)L.map_stride);
    score_scratch_free(b);
    {
        static bool once = false;
        if (!once) {
            once = true;
            tail_prefer_carveout(), gemm_prefer_carveout(), api_prefer_carveout(), bank_prefer_carveout();
        }
    }
    const size_t D = b->dim;
    auto up = [](size_t v) { return (v + 255) & ~size_t(255); };
    L.map_stride = map_cap;
    L.off_min_val = up(sizeof(TailResult) * cap_b);
    L.off_min_idx = L.off_min_val + up(sizeof(float) * cap_p);
    L.off_map_out = L.off_min_idx + up(sizeof(long long) * cap_p);
    L.off_map_pre = L.off_map_out + up(sizeof(float) * map_cap * cap_b);
    L.off_map_u8 = L.off_map_pre + up(sizeof(float) * map_cap * cap_b);
    L.out_block_bytes = L.off_map_u8 + up((size_t)map_cap * cap_b);
    L.n_topk_blocks = b->num_sms * 4;
    // per slot: queries in, results out (mirrored by a pinned host block)
    for (ResultSlot &s : b->slot) {
        CMDB_CUDA(cudaMalloc(&s.q_f32, sizeof(float) * cap_p * D));
        CMDB_CUDA(cudaMalloc(&s.out_block, L.out_block_bytes));
        CMDB_CUDA(cudaMallocHost(&s.out_block_host, L.out_block_bytes));
    }
    for (Lane &l : b->lane) {
        CMDB_CUDA(cudaMalloc(&l.q_hi, sizeof(__half) * cap_p * D));
        CMDB_CUDA(cudaMalloc(&l.q_lo, sizeof(__half) * cap_p * D));
        CMDB_CUDA(cudaMalloc(&l.q_scale_exp, sizeof(int) * cap_p));
        CMDB_CUDA(cudaMalloc(&l.q_norm, sizeof(float) * cap_p));
        CMDB_CUDA(cudaMalloc(&l.q_eps, sizeof(float) * cap_p));
        CMDB_CUDA(cudaMalloc(&l.fail_list, sizeof(int) * cap_p));
        // control block (8 ints) and the per-image argmax keys behind it: one allocation, cleared by ONE memset per call
        CMDB_CUDA(cudaMalloc(&l.fail_ctl, 8 * sizeof(int) + sizeof(unsigned long long) * cap_b));
        l.s_key = reinterpret_cast<unsigned long long *>(l.fail_ctl + 8);
        CMDB_CUDA(cudaMalloc(&l.work_list, sizeof(int2) * kWorkCap));
        CMDB_CUDA(cudaMalloc(&l.best_key, sizeof(unsigned long long) * cap_p));
        CMDB_CUDA(cudaMallocHost(&l.fail_count_host, 2 * sizeof(int)));
        l.fail_count_host[0] = l.fail_count_host[1] = 0;
        CMDB_CUDA(cudaMalloc(&l.done_counter, sizeof(unsigned int)));
        CMDB_CUDA(cudaMemset(l.done_counter, 0, sizeof(unsigned int)));
        const size_t cand_bytes = sizeof(float4) * (size_t)cap_p * 2 * b->num_sms;
        CMDB_CUDA(cudaMalloc(&l.cand, cand_bytes));
        CMDB_CUDA(cudaMalloc(&l.map_tmp, (size_t)map_cap * cap_b));
        CMDB_CUDA(cudaMalloc(&l.map_max, sizeof(float) * cap_b * 17));
        CMDB_CUDA(cudaMalloc(&l.topk_keys, sizeof(unsigned long long) * 3 * L.n_topk_blocks * cap_b));
        CMDB_CUDA(cudaMalloc(&l.top3, sizeof(unsigned long long) * 3 * cap_b));
        CMDB_CUDA(cudaMalloc(&l.m_test, sizeof(float) * D * cap_b));
        CMDB_CUDA(cudaMalloc(&l.m_star, sizeof(float) * D * cap_b));
        CMDB_CHECK(make_map(&l.tmap_qhi, l.q_hi, cap_p, b->dim, BM));
        CMDB_CHECK(make_map(&l.tmap_qlo, l.q_lo, cap_p, b->dim, BM));
    }
    L.cap_p = cap_p, L.cap_b = cap_b;   // last: a failed allocation leaves the scratch to be rebuilt by the next call
    return CMDB_OK;
}

int score_query_prep(const ScoreCall &c, cudaStream_t st, int P, bool compact, int row0) {
    const cmdb_bank *b = c.b;
    const Lane &l = *c.lane;
    const int p_pad = (P + BM - 1) / BM * BM;
    const size_t o = (size_t)row0 * b->dim;
    q_split_kernel<<<std::min(b->num_sms * 2, (p_pad + 7) / 8), 256, 0, st>>>(
        c.slot->q_f32 + o, P, p_pad, b->dim, l.q_hi + o, l.q_lo + o, l.q_scale_exp + row0, compact ? nullptr : l.q_norm + row0,
        compact ? nullptr : l.q_eps + row0, compact ? l.fail_list : nullptr, compact ? l.fail_ctl + 2 : nullptr);
    CMDB_CUDA(cudaGetLastError());
    return CMDB_OK;
}

// fp16 split (+ norms for the certificate) of n explicit rows (n <= cap_p) into rows 0.. of the query operand
void q_split_rows(const ScoreCall &c, const float *rows_dev, int n) {
    const cmdb_bank *b = c.b;
    const Lane &l = *c.lane;
    const int p_pad = (n + BM - 1) / BM * BM;
    q_split_kernel<<<std::min(b->num_sms * 2, p_pad / 8), 256, 0, c.stream>>>(rows_dev, n, p_pad, b->dim, l.q_hi, l.q_lo,
                                                                              l.q_scale_exp, l.q_norm, l.q_eps, nullptr, nullptr);
}

// N tiles per visit of an M tile.  Longer runs cut the traffic of the candidate lists (read + written once per run instead of
// once per tile) but coarsen the work units: take the longest run whose busiest unit stays within 2 % of the ideal share.
static int score_gemm_run(int nt, int mt_units, int G) {
    // at least G runs per M tile, so that EVERY producer keeps seeing a share of every query's rows (the certificate wants the
    // rows near a query's minimum spread over many producers; idle producers made 1.7x more queries need a rescan)
    const double ideal = (double)nt * mt_units / G;
    for (int run = std::min(8, std::max(1, nt / G)); run >= 2; --run) {
        const long long nruns = (nt + run - 1) / run, pairs = nruns * mt_units;
        const long long makespan = (pairs + G - 1) / G * run;
        if ((double)makespan <= ideal * 1.02) return run;
    }
    return 1;
}

// x with (a * x) % m == 1 (a coprime with m; m = scheduling units of the GEMM, <= a few hundred); 0 for m == 1
static int mod_inverse(int a, int m) {
    a %= m;
    for (int x = 0; x < m; ++x)
        if ((a * x) % m == 1 % m) return x;
    return 0;
}

GemmSched gemm_sched(int nt, int mt, int num_sms, bool pair) {
    const int cg = pair ? 2 : 1, mt_units = (mt + cg - 1) / cg, G = num_sms / cg;
    const int stride = tile_stride(mt_units, G);
    return GemmSched{kGemmEpiGroups * num_sms, pair, G, stride, mod_inverse(stride, G), score_gemm_run(nt, mt_units, G), nt};
}

int score_gemm_candidates(const ScoreCall &c, cudaStream_t st, int P, int terms, bool compact, GemmSched *sched, int row0) {
    const cmdb_bank *b = c.b;
    const Lane &l = *c.lane;
    const int p_pad = (P + BM - 1) / BM * BM;

    GemmParams p{};
    p.nt = (int)(b->fin_rows_pad / BN);
    p.kb = b->dim / BK;
    p.bnorm = b->norm;
    p.q_scale_exp = l.q_scale_exp;
    p.b_scale_exp = b->scale_exp;
    p.cand = l.cand;
    p.cand_stride = b->layout.cap_p;
    p.mt = p_pad / BM;
    p.m_base = row0 / BM;
    p.m_count = compact ? l.fail_ctl + 2 : nullptr;
    // CTA pairs (cta_group::2), measured at 16 images x 200k x 768: the 3-term kernel gains 5 % from pairs (7.84 -> 7.42 ms),
    // the 1-term pre-filter loses 3 % (2.81 -> 2.90 ms; it is not limited by shared-memory reads, and a pair halves the
    // producers per query)
    const bool pair = !compact && b->num_sms % 2 == 0 && terms == 3 && p.mt >= 8;
    GemmSched s = gemm_sched(p.nt, p.mt, b->num_sms, pair);
    if (compact) s.stride = s.inv = 0, s.run = 1;  // sized on the device (m_count): single tiles, stride unknown here
    p.run = s.run;
    const int threads = kGemmCtlThreads + 128 * kGemmEpiGroups;
    auto launch = [&](auto kern, size_t smem, bool cluster2) -> int {
        CMDB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        cudaLaunchConfig_t cfg{};
        cfg.gridDim = dim3(b->num_sms), cfg.blockDim = dim3(threads), cfg.dynamicSmemBytes = smem, cfg.stream = st;
        cudaLaunchAttribute attr{};
        attr.id = cudaLaunchAttributeClusterDimension;
        attr.val.clusterDim.x = cluster2 ? 2 : 1, attr.val.clusterDim.y = 1, attr.val.clusterDim.z = 1;
        cfg.attrs = &attr, cfg.numAttrs = 1;
        // the pair kernels load HALF bank tiles (box of 128 rows)
        const CUtensorMap &mh = *reinterpret_cast<CUtensorMap *>(cluster2 ? b->tmap_hi2 : b->tmap_hi);
        const CUtensorMap &ml = *reinterpret_cast<CUtensorMap *>(cluster2 ? b->tmap_lo2 : b->tmap_lo);
        CMDB_CUDA(cudaLaunchKernelEx(&cfg, kern, *reinterpret_cast<CUtensorMap *>(l.tmap_qhi),
                                     *reinterpret_cast<CUtensorMap *>(l.tmap_qlo), mh, ml, p));
        return CMDB_OK;
    };
    if (pair) CMDB_CHECK(launch(score_gemm_kernel<3, kGemmEpiGroups, 2>, GemmSmem<3, 2>::total + 1024, true));
    else if (terms == 1) CMDB_CHECK(launch(score_gemm_kernel<1, kGemmEpiGroups, 1>, GemmSmem<1, 1>::total + 1024, false));
    else CMDB_CHECK(launch(score_gemm_kernel<3, kGemmEpiGroups, 1>, GemmSmem<3, 1>::total + 1024, false));
    *sched = s;
    return CMDB_OK;
}

}  // namespace cmdb
