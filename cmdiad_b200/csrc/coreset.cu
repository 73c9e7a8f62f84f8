// Greedy k-center coreset selection (reference features.py:372-425) as ONE persistent cooperative kernel.
//
// Per pick the reference launches >= 8 ATen kernels, materialises z - last as an [N,d'] temporary and syncs the host
// twice.  Here the whole loop of n-1 dependent picks runs inside one kernel:
//   * the projected bank z ([N,d'] half or double, natural row-major layout) is streamed once per pick
//     (N*d'*sizeof(T) algorithmic bytes per pick) and pinned in L2 as far as the persisting carve-out allows; rows are
//     statically split CTA -> 4-warp group -> warp (a warp owns one alignment class of its group's chunk), so the
//     running min-distance vector never leaves shared memory as long as the CTA's rows fit there;
//   * the distance ||z_i - last|| is evaluated in the CANONICAL reduction order documented in
//     oracle/coreset_oracle.c (the order of ATen's CUDA reduction for torch.linalg.norm on a contiguous [N,d'] tensor:
//     32 lanes per row, aligned 4-element vectors round-robin over lanes, 4 accumulators per lane, fma accumulate,
//     ((a0+a1)+a2)+a3, shfl_down-shaped tree, IEEE sqrt, one rounding to the storage type), so the selected indices
//     are bit-identical to the torch-CUDA reference, including its lowest-index tie-break;
//   * hot loop: two 4-row batches of loads in flight per warp (running per-lane pointers), HSUB2 + fma.rn.f32.f16
//     (SASS FHFMA), per-lane partials of 32 rows transposed through shared memory so the tree, sqrt, min and argmax
//     bookkeeping run lane-parallel (one row per lane) instead of as 5 shuffles per row;
//   * the per-pick grid-wide argmax is an all-gather of one self-flagged 64-bit word per CTA through L2 (relaxed
//     stores / relaxed polling, double-buffered by pick parity) -- no atomics, no fences, no host round trip;
//   * row-sharded mode (one process per GPU): CTA 0 of every GPU pushes its candidate key + row into all ranks'
//     mailboxes with plain NVLink stores of self-flagged 8-byte words (CUDA-IPC mapped peer memory, csrc/comm.cu); all
//     CTAs spin on their LOCAL mailbox -- no NCCL call, no system fence per pick; bounded spins turn a missing peer
//     into an error instead of a hang.
#include "common.cuh"

namespace cmdb {

constexpr int kCsThreads = 512;
constexpr int kCsWarps = kCsThreads / 32;

struct __align__(16) PickSlot {
    unsigned long long val;  // value bits (non-negative half/double order like unsigned integers)
    unsigned long long tag;  // (epoch << 32) | row
};

__device__ __forceinline__ void st_relaxed_u64(unsigned long long *p, unsigned long long v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ void st_release_u64(unsigned long long *p, unsigned long long v) {
    asm volatile("st.release.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_relaxed_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

__device__ __forceinline__ __half ld_volatile(const __half *p) {
    return __ushort_as_half(*reinterpret_cast<const volatile unsigned short *>(p));
}
__device__ __forceinline__ double ld_volatile(const double *p) { return *reinterpret_cast<const volatile double *>(p); }
__device__ __forceinline__ unsigned int ld_volatile(const unsigned int *p) { return *reinterpret_cast<const volatile unsigned int *>(p); }

__device__ __forceinline__ __half ld_cg(const __half *p) { return __ldcg(p); }
__device__ __forceinline__ double ld_cg(const double *p) { return __ldcg(p); }
__device__ __forceinline__ void st_cg(__half *p, __half v) { __stcg(p, v); }
__device__ __forceinline__ void st_cg(double *p, double v) { __stcg(p, v); }

template <typename T>
struct Traits;
template <>
struct Traits<__half> {
    using acc_t = float;
    static __device__ __forceinline__ unsigned long long bits(__half v) { return (unsigned long long)__half_as_ushort(v); }
    static __device__ __forceinline__ __half from_acc(float a) { return __float2half_rn(sqrtf(a)); }
    static __device__ __forceinline__ __half zero() { return __ushort_as_half((unsigned short)0); }
    static __device__ __forceinline__ __half from_bits(unsigned short b) { return __ushort_as_half(b); }
    static __device__ __forceinline__ __half from_bits64(unsigned long long) { return zero(); }  // float64 mailbox only
    static __device__ __forceinline__ bool lt(__half a, __half b) { return __half2float(a) < __half2float(b); }
    static __device__ __forceinline__ bool gt(__half a, __half b) { return __half2float(a) > __half2float(b); }
};
template <>
struct Traits<double> {
    using acc_t = double;
    static __device__ __forceinline__ unsigned long long bits(double v) { return (unsigned long long)__double_as_longlong(v); }
    static __device__ __forceinline__ double from_acc(double a) { return sqrt(a); }
    static __device__ __forceinline__ double zero() { return 0.0; }
    static __device__ __forceinline__ double from_bits(unsigned short) { return 0.0; }  // half mailbox only
    static __device__ __forceinline__ double from_bits64(unsigned long long b) { return __longlong_as_double((long long)b); }
    static __device__ __forceinline__ bool lt(double a, double b) { return a < b; }
    static __device__ __forceinline__ bool gt(double a, double b) { return a > b; }
};

// ---- one aligned 4-element vector: load + accumulate ----
struct HVec {
    __half2 a, b;
};
__device__ __forceinline__ HVec ldvec(const __half *p) {
    uint2 r = __ldg(reinterpret_cast<const uint2 *>(p));
    HVec v;
    v.a = *reinterpret_cast<__half2 *>(&r.x);
    v.b = *reinterpret_cast<__half2 *>(&r.y);
    return v;
}
struct DVec {
    double2 a, b;
};
__device__ __forceinline__ DVec ldvec(const double *p) {
    DVec v;
    v.a = __ldg(reinterpret_cast<const double2 *>(p));
    v.b = __ldg(reinterpret_cast<const double2 *>(p) + 1);
    return v;
}
__device__ __forceinline__ HVec zero_vec(const __half *) {
    HVec v;
    v.a = v.b = __half2(Traits<__half>::zero(), Traits<__half>::zero());
    return v;
}
__device__ __forceinline__ DVec zero_vec(const double *) {
    DVec v;
    v.a = v.b = make_double2(0.0, 0.0);
    return v;
}
// z - last is rounded to the storage type (half: HSUB2 == float subtract + RNE, see DESIGN.md), then fma-accumulated.
// fma.rn.f32.f16 (SASS FHFMA, sm_100) multiplies two halves exactly and adds in float with one rounding == fmaf on the
// converted values, without the two conversion instructions per element.
__device__ __forceinline__ void fhfma2(__half2 dv, float &a0, float &a1) {
    asm("{\n"
        ".reg .f16 lo, hi;\n"
        "mov.b32 {lo, hi}, %2;\n"
        "fma.rn.f32.f16 %0, lo, lo, %0;\n"
        "fma.rn.f32.f16 %1, hi, hi, %1;\n"
        "}"
        : "+f"(a0), "+f"(a1)
        : "r"(*reinterpret_cast<unsigned int *>(&dv)));
}
__device__ __forceinline__ void accum(const HVec &x, const HVec &l, float (&acc)[4]) {
    fhfma2(__hsub2(x.a, l.a), acc[0], acc[1]);
    fhfma2(__hsub2(x.b, l.b), acc[2], acc[3]);
}
__device__ __forceinline__ void accum(const DVec &x, const DVec &l, double (&acc)[4]) {
    double d;
    d = x.a.x - l.a.x, acc[0] = fma(d, d, acc[0]);
    d = x.a.y - l.a.y, acc[1] = fma(d, d, acc[1]);
    d = x.b.x - l.b.x, acc[2] = fma(d, d, acc[2]);
    d = x.b.y - l.b.y, acc[3] = fma(d, d, acc[3]);
}
__device__ __forceinline__ float sqdiff(__half x, __half l, float acc) {
    const unsigned short dv = __half_as_ushort(__hsub(x, l));
    asm("fma.rn.f32.f16 %0, %1, %1, %0;" : "+f"(acc) : "h"(dv));
    return acc;
}
__device__ __forceinline__ double sqdiff(double x, double l, double acc) {
    double d = x - l;
    return fma(d, d, acc);
}
__device__ __forceinline__ void set_elem(HVec &v, int j, __half x) {
    if (j == 0) v.a.x = x;
    else if (j == 1) v.a.y = x;
    else if (j == 2) v.b.x = x;
    else v.b.y = x;
}
__device__ __forceinline__ void set_elem(DVec &v, int j, double x) {
    if (j == 0) v.a.x = x;
    else if (j == 1) v.a.y = x;
    else if (j == 2) v.b.x = x;
    else v.b.y = x;
}

template <typename T>
struct VecOf;
template <>
struct VecOf<__half> {
    using type = HVec;
};
template <>
struct VecOf<double> {
    using type = DVec;
};

// geometry of one alignment class (shift s = (row*d) & 3) in the vectorised order
struct ClassGeom {
    int s, base, nfull, ntail, voff;  // voff: element offset of main vector 0 from the aligned row base (0 or 4)
};
__device__ __forceinline__ ClassGeom class_geom(int s, int d) {
    ClassGeom g;
    g.s = s;
    g.base = s ? 4 - s : 0;
    const int end = d - g.base;
    g.nfull = end >> 2;
    g.ntail = end & 3;
    g.voff = s ? 4 : 0;
    return g;
}

// `last` (the most recently selected row, in shared memory) arranged for one alignment class
template <typename T, int NV>
struct LastRegs {
    typename VecOf<T>::type main[NV];
    T head, tail;
};
template <typename T, int NV>
__device__ __forceinline__ void load_last(LastRegs<T, NV> &L, const T *last_sh, const ClassGeom &g, int lane, int d,
                                          bool vectorized) {
    if (vectorized) {
#pragma unroll
        for (int t = 0; t < NV; ++t) {
            const int v = lane + 32 * t;
            L.main[t] = zero_vec((const T *)nullptr);
            if (v < g.nfull) {
#pragma unroll
                for (int j = 0; j < 4; ++j) set_elem(L.main[t], j, last_sh[g.base + 4 * v + j]);
            }
        }
        L.head = (g.s > 0 && lane >= g.s && lane < 4) ? last_sh[lane - g.s] : Traits<T>::zero();
        L.tail = (lane < g.ntail) ? last_sh[g.base + 4 * g.nfull + lane] : Traits<T>::zero();
    } else {
        // d < 128: lane x owns elements x, x+32, x+64, x+96 -> accumulators 0..3 (kept in main[0])
        L.main[0] = zero_vec((const T *)nullptr);
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (lane + 32 * j < d) set_elem(L.main[0], j, last_sh[lane + 32 * j]);
        L.head = L.tail = Traits<T>::zero();
    }
}

// per-lane partial ((a0+a1)+a2)+a3 of row `rowp` (natural layout, element 0 at rowp) in the canonical order
template <typename T, int NV>
struct RowLoads {
    typename VecOf<T>::type main[NV];
    T head, tail;
};
template <typename T, int NV>
__device__ __forceinline__ void issue_loads(RowLoads<T, NV> &R, const T *rowp, const ClassGeom &g, int lane, int d,
                                            bool vectorized) {
    if (vectorized) {
        const T *vb = rowp - g.s + g.voff;  // 4-element aligned
#pragma unroll
        for (int t = 0; t < NV; ++t) {
            const int v = lane + 32 * t;
            if (v < g.nfull) R.main[t] = ldvec(vb + 4 * v);
            else R.main[t] = zero_vec((const T *)nullptr);
        }
        R.head = (g.s > 0 && lane >= g.s && lane < 4) ? __ldg(rowp + (lane - g.s)) : Traits<T>::zero();
        R.tail = (lane < g.ntail) ? __ldg(rowp + g.base + 4 * g.nfull + lane) : Traits<T>::zero();
    } else {
        R.main[0] = zero_vec((const T *)nullptr);
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (lane + 32 * j < d) set_elem(R.main[0], j, __ldg(rowp + lane + 32 * j));
        R.head = R.tail = Traits<T>::zero();
    }
}
template <typename T, int NV>
__device__ __forceinline__ typename Traits<T>::acc_t lane_partial(const RowLoads<T, NV> &R, const LastRegs<T, NV> &L,
                                                                   bool vectorized) {
    typename Traits<T>::acc_t acc[4] = {0, 0, 0, 0};
    if (vectorized) {
        acc[0] = sqdiff(R.head, L.head, acc[0]);  // lanes without a head element add fma(0,0,0) = 0
#pragma unroll
        for (int t = 0; t < NV; ++t) accum(R.main[t], L.main[t], acc);  // absent vectors are 0 - 0
        acc[0] = sqdiff(R.tail, L.tail, acc[0]);
    } else {
        accum(R.main[0], L.main[0], acc);
    }
    return ((acc[0] + acc[1]) + acc[2]) + acc[3];
}

struct CoresetParams {
    const void *z;               // [N,d] half or double
    void *mind;                  // [N] running min distances (global copy; shared memory is used when it fits)
    long long N;
    int d;
    long long n_select;
    long long *out_idx;          // [n_select]
    const long long *force_idx;  // optional teacher forcing
    PickSlot *slots;             // [2][gridDim.x]
    long long rows_per_cta;
    int mind_in_smem;
    // row-sharded mode (world > 1): rows are local, row_offset maps them to global rows; per pick the GPUs exchange
    // their candidate + its row through peer-mapped mailboxes
    long long row_offset;
    int world, rank;
    unsigned char *mb_peer[kMaxRanks];  // mailbox of every rank (mb_peer[rank] is local memory)
    unsigned int mb_keys_off;           // byte offset of the key slots inside a mailbox: [parity][source rank][source CTA]
    const void *z_full;                 // replica of the WHOLE projected bank [n_total, d] (storage type); local rows are a slice
    unsigned int mb_ready_off;          // byte offset of the per-rank "shard has arrived in your replica" flags (8 bytes each)
    unsigned long long ready_epoch;     // value those flags take for this call
    unsigned int *abort_flag;           // set when a peer did not answer in time
    long long spin_limit;               // clock64() ticks to wait for a peer
    size_t *l2_prev_limit;              // host side only: persisting-L2 carve-out found before the launch ...
    bool *l2_changed;                   // ... and whether launch_coreset enlarged it (restored by coreset_greedy_dev)
};

// per-warp constants of the streaming loop: every warp handles ONE alignment class (rows with row % 4 == warp % 4 of
// its 4-warp group's chunk), so the class geometry is computed once per kernel and `last` is re-staged once per pick
template <typename T, int NV>
struct WarpPlan {
    ClassGeom g;
    int main_off;   // element offset (from the row start) of this lane's first aligned main vector
    int head_off, tail_off;
    bool has_head, has_tail;
    bool vmain[NV];
    long long first, n_rows;  // rows first, first+4, ... (n_rows of them)
};

template <typename T, int NV>
__device__ __forceinline__ void issue_row(RowLoads<T, NV> &R, const T *rowp, const WarpPlan<T, NV> &w, int lane, int d,
                                          bool vectorized) {
    if (vectorized) {
        const T *vb = rowp + w.main_off;
#pragma unroll
        for (int t = 0; t < NV; ++t) {
            if (w.vmain[t]) R.main[t] = ldvec(vb + 128 * t);
            else R.main[t] = zero_vec((const T *)nullptr);
        }
        R.head = w.has_head ? __ldg(rowp + w.head_off) : Traits<T>::zero();
        R.tail = w.has_tail ? __ldg(rowp + w.tail_off) : Traits<T>::zero();
    } else {
        R.main[0] = zero_vec((const T *)nullptr);
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (lane + 32 * j < d) set_elem(R.main[0], j, __ldg(rowp + lane + 32 * j));
        R.head = R.tail = Traits<T>::zero();
    }
}

template <typename T>
struct Batch {
    static constexpr int rows = 4;
};
template <>
struct Batch<double> {
    static constexpr int rows = 2;  // 32-byte vectors: keep the register footprint of two batches in flight below 128
};

template <typename T, int NV>
__global__ void __launch_bounds__(kCsThreads, 1) coreset_kernel(CoresetParams p) {
    using acc_t = typename Traits<T>::acc_t;
    constexpr int RB = Batch<T>::rows;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    // layout: tile [kCsWarps][32][33] acc_t | last_sh [d] T | red (val,row) [32] | mind [rows_per_cta] T
    acc_t *tile_all = reinterpret_cast<acc_t *>(smem_raw);
    T *last_sh = reinterpret_cast<T *>(tile_all + kCsWarps * 32 * 33);
    unsigned long long *red_val = reinterpret_cast<unsigned long long *>(
        (reinterpret_cast<uintptr_t>(last_sh + p.d) + 15) & ~uintptr_t(15));
    unsigned long long *red_row = red_val + 32;
    T *mind_sh = reinterpret_cast<T *>(red_row + 32);

    const T *z = reinterpret_cast<const T *>(p.z);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int d = p.d;
    const bool vectorized = d >= 128;
    acc_t *tile = tile_all + warp * 32 * 33;

    // this CTA owns rows [cta_row0, cta_row1) and keeps their min-distances in shared memory when they fit, else in
    // global memory (L2, .cg accesses)
    const long long cta_row0 = (long long)blockIdx.x * p.rows_per_cta;
    const long long cta_row1 = min(p.N, cta_row0 + p.rows_per_cta);
    const long long cta_rows = max(0LL, cta_row1 - cta_row0);
    T *mind = p.mind_in_smem ? mind_sh : reinterpret_cast<T *>(p.mind) + cta_row0;
    const bool mind_global = !p.mind_in_smem;
    if (p.mind_in_smem)
        for (long long i = threadIdx.x; i < cta_rows; i += kCsThreads) mind_sh[i] = reinterpret_cast<T *>(p.mind)[cta_row0 + i];

    // ---- static work split: 4-warp groups share a contiguous chunk; warp (w & 3) takes its rows with row % 4 == w & 3 ----
    WarpPlan<T, NV> wp;
    auto plan_class = [&](int c) {  // geometry of the alignment class of global rows with row % 4 == c
        const int s = vectorized ? (int)(((long long)c * d) & 3) : 0;
        wp.g = class_geom(s, d);
        wp.main_off = wp.g.voff - s + 4 * lane;
        wp.has_head = s > 0 && lane >= s && lane < 4;
        wp.head_off = lane - s;
        wp.has_tail = lane < wp.g.ntail;
        wp.tail_off = wp.g.base + 4 * wp.g.nfull + lane;
#pragma unroll
        for (int t = 0; t < NV; ++t) wp.vmain[t] = lane + 32 * t < wp.g.nfull;
    };
    {
        constexpr int kGroups = kCsWarps / 4;
        const long long rows_per_group = (cta_rows + kGroups - 1) / kGroups;
        const long long g_row0 = cta_row0 + (warp >> 2) * rows_per_group;
        const long long g_row1 = min(cta_row1, g_row0 + rows_per_group);
        // alignment classes follow the GLOBAL row number (the reference's tensor is one contiguous [N,d] block); the
        // shard's buffer starts (row_offset*d) & 3 elements past a vector boundary so addresses agree with it
        const int c = warp & 3;  // this warp takes the local rows whose global row % 4 == c
        wp.first = g_row0 + ((c - (int)((g_row0 + p.row_offset) & 3)) & 3);
        wp.n_rows = wp.first < g_row1 ? (g_row1 - wp.first + 3) >> 2 : 0;
        plan_class(c);
    }
    const size_t rstride_b = (size_t)4 * d * sizeof(T);  // bytes between consecutive rows of this warp

    long long sel = 0;  // features.py:372 -- pick 0 is (global) row 0
    if (blockIdx.x == 0 && threadIdx.x == 0) p.out_idx[0] = 0;
    if (p.world > 1) {
        // the replica of the projected bank is complete once every rank's shard copy has landed: each rank's copy stream
        // sets its flag in our mailbox right after its rows (stream order), so one poll per peer suffices
        if (threadIdx.x < p.world) {
            const unsigned long long *f = reinterpret_cast<const unsigned long long *>(p.mb_peer[p.rank] + p.mb_ready_off) + threadIdx.x;
            const long long t0 = clock64();
            unsigned long long v;
            for (;;) {
                asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(f) : "memory");
                if (v == p.ready_epoch) break;
                if (clock64() - t0 > p.spin_limit) {
                    *p.abort_flag = 1u;
                    break;
                }
            }
        }
        __syncthreads();
        if (ld_volatile(p.abort_flag)) return;
    }

    for (long long pick = 1; pick < p.n_select; ++pick) {
        // ---- stage `last` = z[sel] in shared memory; owner CTA zeroes min_d[sel] (features.py:418-419) ----
        __syncthreads();
        {
            // sel is a GLOBAL row; row-sharded mode reads it from the local replica of the projected bank (no row exchange)
            const T *zsel = p.world > 1 ? reinterpret_cast<const T *>(p.z_full) : z;
            for (int e = threadIdx.x; e < d; e += kCsThreads) last_sh[e] = __ldg(zsel + sel * d + e);
        }
        {
            const long long sl = sel - p.row_offset;  // local row of the previous pick, if this shard owns it
            if (threadIdx.x == 0 && pick > 1 && sl >= cta_row0 && sl < cta_row1) {
                if (mind_global) st_cg(mind + (sl - cta_row0), Traits<T>::zero());
                else mind[sl - cta_row0] = Traits<T>::zero();
            }
        }
        __syncthreads();
        LastRegs<T, NV> L;
        load_last<T, NV>(L, last_sh, wp.g, lane, d, vectorized);

        T best_val = Traits<T>::zero();
        long long best_row = -1;
        // ---- distance pass: software-pipelined stream of full RB-row batches (two batches of loads in flight), running
        //      per-lane pointers instead of index arithmetic; the < RB leftover rows take a simple path ----
        auto finalize = [&](long long grp, int n_here) {
            __syncwarp();
            if (lane < n_here) {
                // shfl_down-shaped tree over the row's 32 lane partials, evaluated as 4 sub-trees of 8 to keep the
                // register footprint small while two batches of loads are in flight (same association as the shfl_down tree with offsets 1,2,4,8,16)
                acc_t q4[4];
#pragma unroll 1
                for (int blk = 0; blk < 4; ++blk) {
                    acc_t v[8];
#pragma unroll
                    for (int k = 0; k < 8; ++k) v[k] = tile[lane * 33 + blk * 8 + k];
                    q4[blk] = ((v[0] + v[1]) + (v[2] + v[3])) + ((v[4] + v[5]) + (v[6] + v[7]));
                }
                const T dist = Traits<T>::from_acc((q4[0] + q4[1]) + (q4[2] + q4[3]));
                const long long row = wp.first + 4 * (grp * 32 + lane);
                T m = mind_global ? ld_cg(mind + (row - cta_row0)) : mind[row - cta_row0];
                if (Traits<T>::lt(dist, m)) {  // torch.minimum (features.py:413)
                    m = dist;
                    if (mind_global) st_cg(mind + (row - cta_row0), m);
                    else mind[row - cta_row0] = m;
                }
                // argmax, ties -> lowest index (features.py:415)
                if (best_row < 0 || Traits<T>::gt(m, best_val) || (!Traits<T>::lt(m, best_val) && row < best_row)) {
                    best_val = m;
                    best_row = row;
                }
            }
            __syncwarp();
        };
        auto run_rows = [&]() {  // distance pass over rows wp.first, wp.first + 4, ... (wp.n_rows of them)
        if (vectorized) {
            RowLoads<T, NV> A[RB], B[RB];
            const char *pm = reinterpret_cast<const char *>(z + wp.first * d + wp.main_off);
            const char *ph = reinterpret_cast<const char *>(z + wp.first * d + wp.head_off);
            const char *pt = reinterpret_cast<const char *>(z + wp.first * d + wp.tail_off);
            auto issue = [&](RowLoads<T, NV>(&buf)[RB]) {
#pragma unroll
                for (int r = 0; r < RB; ++r) {
                    const T *rm = reinterpret_cast<const T *>(pm + r * rstride_b);
#pragma unroll
                    for (int t = 0; t < NV; ++t) {
                        if (wp.vmain[t]) buf[r].main[t] = ldvec(rm + 128 * t);
                        else buf[r].main[t] = zero_vec((const T *)nullptr);
                    }
                    buf[r].head = wp.has_head ? __ldg(reinterpret_cast<const T *>(ph + r * rstride_b)) : Traits<T>::zero();
                    buf[r].tail = wp.has_tail ? __ldg(reinterpret_cast<const T *>(pt + r * rstride_b)) : Traits<T>::zero();
                }
                pm += RB * rstride_b, ph += RB * rstride_b, pt += RB * rstride_b;
            };
            const long long nb_full = wp.n_rows / RB;
            if (nb_full > 0) issue(A);
            for (long long bi = 0; bi < nb_full; bi += 2) {
                if (bi + 1 < nb_full) issue(B);
                {
                    acc_t *trow = tile + (int)((bi * RB) & 31) * 33 + lane;
#pragma unroll
                    for (int r = 0; r < RB; ++r) trow[r * 33] = lane_partial<T, NV>(A[r], L, true);
                    if ((((bi + 1) * RB) & 31) == 0) finalize((bi * RB) >> 5, 32);
                }
                if (bi + 2 < nb_full) issue(A);
                if (bi + 1 < nb_full) {
                    acc_t *trow = tile + (int)(((bi + 1) * RB) & 31) * 33 + lane;
#pragma unroll
                    for (int r = 0; r < RB; ++r) trow[r * 33] = lane_partial<T, NV>(B[r], L, true);
                    if ((((bi + 2) * RB) & 31) == 0) finalize(((bi + 1) * RB) >> 5, 32);
                }
            }
            // leftover rows (< RB) and the last, partial group of 32
            for (long long k = nb_full * RB; k < wp.n_rows; ++k) {
                issue_row<T, NV>(A[0], z + (wp.first + 4 * k) * d, wp, lane, d, true);
                tile[(int)(k & 31) * 33 + lane] = lane_partial<T, NV>(A[0], L, true);
            }
            if (wp.n_rows & 31) finalize(wp.n_rows >> 5, (int)(wp.n_rows & 31));
        } else {
            // d < 128 (tiny test problems only): one row at a time
            RowLoads<T, NV> R;
            for (long long k = 0; k < wp.n_rows; ++k) {
                issue_row<T, NV>(R, z + (wp.first + 4 * k) * d, wp, lane, d, false);
                tile[(int)(k & 31) * 33 + lane] = lane_partial<T, NV>(R, L, false);
                if ((k & 31) == 31 || k == wp.n_rows - 1) finalize(k >> 5, (int)(k & 31) + 1);
            }
        }
        };
        run_rows();
        // ---- CTA argmax: warp shuffle, then shared memory ----
        unsigned long long bv = best_row < 0 ? 0ULL : Traits<T>::bits(best_val);
        unsigned long long br = best_row < 0 ? ~0ULL : (unsigned long long)best_row;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            unsigned long long ov = __shfl_xor_sync(0xffffffffu, bv, o), orow = __shfl_xor_sync(0xffffffffu, br, o);
            if (ov > bv || (ov == bv && orow < br)) bv = ov, br = orow;
        }
        if (lane == 0) red_val[warp] = bv, red_row[warp] = br;
        __syncthreads();
        long long argmax;
        if (p.world == 1) {
        PickSlot *slots = p.slots + (pick & 1) * gridDim.x;
        if (warp == 0) {
            bv = lane < kCsWarps ? red_val[lane] : 0ULL;
            br = lane < kCsWarps ? red_row[lane] : ~0ULL;
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                unsigned long long ov = __shfl_xor_sync(0xffffffffu, bv, o), orow = __shfl_xor_sync(0xffffffffu, br, o);
                if (ov > bv || (ov == bv && orow < br)) bv = ov, br = orow;
            }
            if (lane == 0) {
                if constexpr (sizeof(T) == 2) {
                    // half: value, row and pick number fit ONE self-flagged 64-bit word -> no fence on either side
                    st_relaxed_u64(&slots[blockIdx.x].tag,
                                   ((unsigned long long)(pick & 0xffff) << 48) | ((bv & 0xffffULL) << 32) | (br & 0xffffffffULL));
                } else {
                    st_relaxed_u64(&slots[blockIdx.x].val, bv);
                    st_release_u64(&slots[blockIdx.x].tag, ((unsigned long long)pick << 32) | (br & 0xffffffffULL));
                }
            }
        }
        // ---- grid all-gather of the per-CTA winners through L2 (relaxed polling) ----
        bv = 0ULL, br = ~0ULL;
        for (int c = threadIdx.x; c < (int)gridDim.x; c += kCsThreads) {
            unsigned long long tag, ov;
            if constexpr (sizeof(T) == 2) {
                do {
                    tag = ld_relaxed_u64(&slots[c].tag);
                } while ((tag >> 48) != (unsigned long long)(pick & 0xffff));
                ov = (tag >> 32) & 0xffffULL;
            } else {
                do {
                    tag = ld_relaxed_u64(&slots[c].tag);
                } while ((tag >> 32) != (unsigned long long)pick);
                asm volatile("fence.acq_rel.gpu;" ::: "memory");
                ov = ld_relaxed_u64(&slots[c].val);
            }
            const unsigned long long orow = (tag & 0xffffffffULL) == 0xffffffffULL ? ~0ULL : (tag & 0xffffffffULL);
            if (ov > bv || (ov == bv && orow < br)) bv = ov, br = orow;
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            unsigned long long ov = __shfl_xor_sync(0xffffffffu, bv, o), orow = __shfl_xor_sync(0xffffffffu, br, o);
            if (ov > bv || (ov == bv && orow < br)) bv = ov, br = orow;
        }
        __syncthreads();  // red_* reads of the CTA stage are done
        if (lane == 0) red_val[warp] = bv, red_row[warp] = br;
        __syncthreads();
        bv = red_val[0], br = red_row[0];
#pragma unroll
        for (int w = 1; w < kCsWarps; ++w) {
            const unsigned long long ov = red_val[w], orow = red_row[w];
            if (ov > bv || (ov == bv && orow < br)) bv = ov, br = orow;
        }
        argmax = (long long)br;  // local row == global row
        } else {
            // ---- row-sharded: ONE flat exchange per pick.  Every CTA of every GPU writes its candidate key straight into
            //      the mailboxes of all ranks (plain NVLink stores; the local rank's mailbox is written the same way), and
            //      every CTA polls the world x grid keys in its LOCAL mailbox.  LL-style protocol: each 8-byte word carries
            //      its own flag (the pick number), so neither side needs a system-scope fence, and slots are double-buffered
            //      by pick parity.  No second hop: the winning row itself is read from the local replica next pick.
            //        half  : one word   [63:48] pick & 0xffff | [47:32] value bits | [31:0] ~global_row
            //        double: three words [63:32] pick | value low half / value high half / ~global_row
            constexpr unsigned int kKeyBytes = sizeof(T) == 2 ? 8u : 32u;
            const unsigned int n_cta = gridDim.x;
            if (warp == 0) {
                bv = lane < kCsWarps ? red_val[lane] : 0ULL;
                br = lane < kCsWarps ? red_row[lane] : ~0ULL;
#pragma unroll
                for (int o = 16; o > 0; o >>= 1) {
                    unsigned long long ov = __shfl_xor_sync(0xffffffffu, bv, o), orow = __shfl_xor_sync(0xffffffffu, br, o);
                    if (ov > bv || (ov == bv && orow < br)) bv = ov, br = orow;
                }
                const unsigned long long inv = br == ~0ULL ? 0ULL : 0xffffffffULL - (unsigned long long)(br + p.row_offset);
                if (br == ~0ULL) bv = 0ULL;
                const size_t slot = p.mb_keys_off + (size_t)(((pick & 1) * p.world + p.rank) * n_cta + blockIdx.x) * kKeyBytes;
                if constexpr (sizeof(T) == 2) {
                    if (lane < p.world) {
                        const unsigned long long key = ((unsigned long long)(pick & 0xffff) << 48) | ((bv & 0xffffULL) << 32) | inv;
                        asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p.mb_peer[lane] + slot), "l"(key) : "memory");
                    }
                } else {
                    if (lane < 3 * p.world) {
                        const int r = lane / 3, k = lane % 3;
                        const unsigned long long part = k == 0 ? (bv & 0xffffffffULL) : k == 1 ? (bv >> 32) : inv;
                        const unsigned long long word = ((unsigned long long)(unsigned int)pick << 32) | part;
                        asm volatile("st.relaxed.sys.global.u64 [%0], %1;" ::"l"(p.mb_peer[r] + slot + 8 * k), "l"(word) : "memory");
                    }
                }
            }
            // poll the keys of all (rank, CTA) pairs in the local mailbox
            unsigned long long kval = 0ULL, kinv = 0ULL;
            int ok = 1;
            {
                const unsigned char *base = p.mb_peer[p.rank] + p.mb_keys_off + (size_t)((pick & 1) * p.world) * n_cta * kKeyBytes;
                const long long t0 = clock64();
                auto poll = [&](const unsigned char *q, int shift, unsigned long long want) {
                    unsigned long long w = 0ULL;
                    for (;;) {
                        asm volatile("ld.relaxed.sys.global.u64 %0, [%1];" : "=l"(w) : "l"(q) : "memory");
                        if ((w >> shift) == want) break;
                        if (clock64() - t0 > p.spin_limit || ld_volatile(p.abort_flag)) {
                            ok = 0;
                            break;
                        }
                    }
                    return w;
                };
                for (unsigned int k = threadIdx.x; k < (unsigned int)p.world * n_cta; k += kCsThreads) {
                    unsigned long long ov, oi;
                    if constexpr (sizeof(T) == 2) {
                        const unsigned long long key = poll(base + (size_t)k * kKeyBytes, 48, (unsigned long long)(pick & 0xffff));
                        ov = (key >> 32) & 0xffffULL, oi = key & 0xffffffffULL;
                    } else {
                        const unsigned long long want = (unsigned long long)(unsigned int)pick;
                        const unsigned char *q = base + (size_t)k * kKeyBytes;
                        const unsigned long long w0 = poll(q, 32, want), w1 = poll(q + 8, 32, want), w2 = poll(q + 16, 32, want);
                        ov = ((w1 & 0xffffffffULL) << 32) | (w0 & 0xffffffffULL), oi = w2 & 0xffffffffULL;
                    }
                    if (ov > kval || (ov == kval && oi > kinv)) kval = ov, kinv = oi;  // max value, ties -> lowest global row
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const unsigned long long ov = __shfl_xor_sync(0xffffffffu, kval, o), oi = __shfl_xor_sync(0xffffffffu, kinv, o);
                if (ov > kval || (ov == kval && oi > kinv)) kval = ov, kinv = oi;
            }
            ok = __all_sync(0xffffffffu, ok);
            __syncthreads();  // red_* reads of the CTA stage are done
            if (lane == 0) red_val[warp] = kval, red_row[warp] = kinv | (ok ? 0ULL : (1ULL << 63));
            __syncthreads();
            kval = red_val[0], kinv = red_row[0] & 0xffffffffULL;
            bool bad = (red_row[0] >> 63) != 0;
#pragma unroll
            for (int w = 1; w < kCsWarps; ++w) {
                const unsigned long long ov = red_val[w], oi = red_row[w] & 0xffffffffULL;
                bad |= (red_row[w] >> 63) != 0;
                if (ov > kval || (ov == kval && oi > kinv)) kval = ov, kinv = oi;
            }
            if (bad) {  // a peer did not answer in time: every CTA of every rank reaches the same verdict within the timeout
                if (threadIdx.x == 0) *p.abort_flag = 1u;
                return;
            }
            argmax = (long long)(0xffffffffULL - kinv);  // global row
        }
        if (blockIdx.x == 0 && threadIdx.x == 0) p.out_idx[pick] = argmax;
        sel = p.force_idx ? p.force_idx[pick] : argmax;
    }
    // final state of the min-distance vector (tests / diagnostics)
    __syncthreads();
    {
        const long long sl = sel - p.row_offset;
        if (threadIdx.x == 0 && p.n_select > 1 && sl >= cta_row0 && sl < cta_row1) mind[sl - cta_row0] = Traits<T>::zero();
    }
    __syncthreads();
    if (p.mind_in_smem)
        for (long long i = threadIdx.x; i < cta_rows; i += kCsThreads) reinterpret_cast<T *>(p.mind)[cta_row0 + i] = mind_sh[i];
}

// ---------------------------------------------------------------------------------------------------------------
// one distance pass (also the initial min-distance vector): out[i] = ||z_i - last||_2 in the canonical order
// ---------------------------------------------------------------------------------------------------------------
template <typename T, int NV>
__global__ void __launch_bounds__(256) rownorm_kernel(const T *__restrict__ z, const T *__restrict__ last, long long N,
                                                      int d, T *__restrict__ out_same, __half *__restrict__ out_half,
                                                      long long row_offset) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    T *last_sh = reinterpret_cast<T *>(smem_raw);
    for (int e = threadIdx.x; e < d; e += blockDim.x) last_sh[e] = last[e];
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const bool vectorized = d >= 128;
    const long long warps = (long long)gridDim.x * (blockDim.x >> 5);
    for (long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); row < N; row += warps) {
        const int s = vectorized ? (int)(((row + row_offset) * d) & 3) : 0;  // alignment class of the GLOBAL row
        const ClassGeom g = class_geom(s, d);
        LastRegs<T, NV> L;
        load_last<T, NV>(L, last_sh, g, lane, d, vectorized);
        RowLoads<T, NV> R;
        issue_loads<T, NV>(R, z + row * d, g, lane, d, vectorized);
        typename Traits<T>::acc_t v = lane_partial<T, NV>(R, L, vectorized);
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) v = v + __shfl_down_sync(0xffffffffu, v, off);
        if (lane == 0) {
            const T r = Traits<T>::from_acc(v);
            if (out_same) out_same[row] = r;
            // features.py:391 min_distances.half(): torch converts double -> float -> half
            if (out_half) out_half[row] = __float2half_rn((float)r);
        }
    }
}

// z64 -> half (torch .half(): double -> float -> half), natural layout
__global__ void __launch_bounds__(512) to_half_kernel(const double *__restrict__ z, long long n, __half *__restrict__ zh) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        zh[i] = __float2half_rn((float)z[i]);
}

template <typename T>
static int launch_rownorm(cudaStream_t st, int num_sms, const T *z, const T *last, long long N, int d, T *out_same,
                          __half *out_half, long long row_offset = 0) {
    const int nv = (d / 4 + 31) / 32;
    const int grid = (int)std::min<long long>((N + 7) / 8, (long long)num_sms * 8);
    const size_t smem = sizeof(T) * (size_t)d;
#define CMDB_RN(NVV)                                                                                   \
    case NVV:                                                                                          \
        rownorm_kernel<T, NVV><<<grid, 256, smem, st>>>(z, last, N, d, out_same, out_half, row_offset); \
        break;
    switch (d >= 128 ? nv : 1) {
        CMDB_RN(1) CMDB_RN(2) CMDB_RN(3) CMDB_RN(4) CMDB_RN(5) CMDB_RN(6) CMDB_RN(7) CMDB_RN(8)
        default:
            set_error("coreset: projected dim %d > 1024 is not supported", d);
            return CMDB_ERR_UNSUPPORTED;
    }
#undef CMDB_RN
    CMDB_CUDA(cudaGetLastError());
    return CMDB_OK;
}

// Where coreset_kernel keeps the running min-distance vector.  CTA c of `grid` owns rows [c * rows_per_cta,
// (c + 1) * rows_per_cta) and holds their min-distances in shared memory, behind the fixed part of its layout (transpose
// tiles, `last`, up to 16 bytes of alignment, the 64 reduction slots), as long as the whole block stays within 200 KB;
// otherwise they stay in global memory and every access goes through L2 (.cg).  force_global picks the second
// placement at any size (tests compare the two on the same bank).
struct CoresetPlan {
    long long rows_per_cta;
    bool mind_in_smem;
    size_t smem;  // dynamic shared memory of the launch
};
template <typename T>
static CoresetPlan coreset_plan(int grid, long long N, int d, bool force_global) {
    const size_t fixed = sizeof(typename Traits<T>::acc_t) * kCsWarps * 32 * 33 + sizeof(T) * (size_t)d + 16 + 64 * 8;
    CoresetPlan pl;
    pl.rows_per_cta = (N + grid - 1) / grid;
    pl.smem = fixed + sizeof(T) * (size_t)pl.rows_per_cta;
    pl.mind_in_smem = !force_global && pl.smem <= 200 * 1024;
    if (!pl.mind_in_smem) pl.smem = fixed;
    return pl;
}

int coreset_plan_info(int num_sms, int64_t N, int d, int dtype_mode, int64_t *rows_per_cta, int *mind_in_smem) {
    CMDB_REQUIRE(num_sms >= 1 && N >= 1 && d >= 1 && rows_per_cta && mind_in_smem, CMDB_ERR_INVALID, "coreset plan: bad arguments");
    CMDB_REQUIRE(dtype_mode == CMDB_CORESET_FP16 || dtype_mode == CMDB_CORESET_FP64, CMDB_ERR_INVALID,
                 "coreset plan: unknown dtype_mode %d", dtype_mode);
    const CoresetPlan pl = dtype_mode == CMDB_CORESET_FP16 ? coreset_plan<__half>(num_sms, N, d, false)
                                                           : coreset_plan<double>(num_sms, N, d, false);
    *rows_per_cta = pl.rows_per_cta;
    *mind_in_smem = pl.mind_in_smem ? 1 : 0;
    return CMDB_OK;
}

template <typename T>
static int launch_coreset(cmdb_bank *b, CoresetParams p, bool force_mind_global) {
    const int d = p.d;
    const int nv = d >= 128 ? (d / 4 + 31) / 32 : 1;
    int grid = b->num_sms;
    auto run = [&](auto kern) -> int {
        const CoresetPlan pl = coreset_plan<T>(grid, p.N, d, force_mind_global);
        p.rows_per_cta = pl.rows_per_cta;
        p.mind_in_smem = pl.mind_in_smem;
        const size_t smem = pl.smem;
        CMDB_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        int per_sm = 0;
        CMDB_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kCsThreads, smem));
        CMDB_REQUIRE(per_sm >= 1, CMDB_ERR_CUDA, "coreset: persistent kernel does not fit on an SM (smem %zu)", smem);
        CMDB_CUDA(cudaMemsetAsync(p.slots, 0, sizeof(PickSlot) * 2 * grid, b->handle_stream()));
        // The projected bank is re-read once per pick.  B200's L2 (126 MB) cannot hold a 120 MB cyclic sweep under its
        // default replacement (measured: 20 % hit rate), so pin as much of it as the persisting carve-out allows and
        // stream the rest: DRAM traffic per pick drops to roughly (1 - hitRatio) of the bank.
        int max_persist = 0, max_window = 0;
        cudaDeviceGetAttribute(&max_persist, cudaDevAttrMaxPersistingL2CacheSize, b->device);
        cudaDeviceGetAttribute(&max_window, cudaDevAttrMaxAccessPolicyWindowSize, b->device);
        const size_t z_bytes = sizeof(T) * (size_t)p.N * p.d;
        bool persisting = false;
        cudaStreamAttrValue attr{};
        if (max_persist > 0 && max_window > 0) {
            const size_t carve = std::min<size_t>(z_bytes, (size_t)max_persist);
            // the carve-out is process-wide device state: only ever GROW it here (another component of the host program
            // may have configured its own) and let coreset_greedy_dev restore the previous value when the loop is done
            size_t prev = 0;
            (void)cudaDeviceGetLimit(&prev, cudaLimitPersistingL2CacheSize);
            if (prev >= carve || cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, carve) == cudaSuccess) {
                if (prev < carve && p.l2_prev_limit) *p.l2_prev_limit = prev, *p.l2_changed = true;
                attr.accessPolicyWindow.base_ptr = const_cast<void *>(p.z);
                attr.accessPolicyWindow.num_bytes = std::min<size_t>(z_bytes, (size_t)max_window);
                attr.accessPolicyWindow.hitRatio =
                    (float)std::min(1.0, (double)carve / (double)attr.accessPolicyWindow.num_bytes);
                attr.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
                attr.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
                persisting = cudaStreamSetAttribute(b->handle_stream(), cudaStreamAttributeAccessPolicyWindow, &attr) == cudaSuccess;
            }
            (void)cudaGetLastError();
        }
        void *args[] = {&p};
        cudaError_t le = cudaLaunchCooperativeKernel((void *)kern, dim3(grid), dim3(kCsThreads), args, smem, b->handle_stream());
        if (persisting) {
            attr.accessPolicyWindow.num_bytes = 0;
            cudaStreamSetAttribute(b->handle_stream(), cudaStreamAttributeAccessPolicyWindow, &attr);
            // the carve-out is released by the caller after the kernel has finished (coreset_greedy_dev)
        }
        CMDB_CUDA(le);
        return CMDB_OK;
    };
#define CMDB_CS(NVV) \
    case NVV:        \
        return run(coreset_kernel<T, NVV>);
    switch (nv) {
        CMDB_CS(1) CMDB_CS(2) CMDB_CS(3) CMDB_CS(4) CMDB_CS(5) CMDB_CS(6) CMDB_CS(7) CMDB_CS(8)
        default:
            set_error("coreset: projected dim %d > 1024 is not supported", d);
            return CMDB_ERR_UNSUPPORTED;
    }
#undef CMDB_CS
}

// z_dev: float64 [N,d] projected rows of THIS shard; for a shard with row_offset != 0 the caller places row 0 of the
// buffer (row_offset*d) & 3 elements past a 32-byte boundary so that address alignment == global alignment class.
// force_mind_global: keep the min-distance vector in global memory even where it would fit shared memory (coreset_plan).
int coreset_greedy_dev(cmdb_bank *b, const double *z_dev, int64_t N, int d, int64_t n_select, int dtype_mode,
                       int64_t *out_idx_host, const int64_t *force_idx_host, void *out_min_last_host, const ShardCtx *sh,
                       bool force_mind_global) {
    const bool sharded = sh && sh->world > 1;
    const long long n_total = sharded ? sh->n_total : N;
    CMDB_REQUIRE(N >= 0 && n_total > 0 && d >= 32 && n_select >= 1 && n_select <= n_total, CMDB_ERR_INVALID,
                 "coreset: need N>0, d>=32, 1<=n_select<=N (N=%lld d=%d n=%lld)", (long long)n_total, d, (long long)n_select);
    CMDB_REQUIRE(n_total < (1LL << 32) - 1, CMDB_ERR_UNSUPPORTED, "coreset: N must fit 32 bits");
    CMDB_REQUIRE(dtype_mode == CMDB_CORESET_FP16 || dtype_mode == CMDB_CORESET_FP64, CMDB_ERR_INVALID,
                 "coreset: unknown dtype_mode %d", dtype_mode);
    CMDB_REQUIRE(!sharded || (!force_idx_host && N > 0), CMDB_ERR_UNSUPPORTED,
                 "coreset: the row-sharded loop needs non-empty shards and does not support teacher forcing");
    cudaStream_t st = b->handle_stream();
    long long *idx_dev = nullptr, *force_dev = nullptr;
    PickSlot *slots = nullptr;
    __half *zh_alloc = nullptr;
    double *z0_dev = nullptr;
    unsigned int *abort_dev = nullptr;
    void *mind = nullptr;
    int rc = CMDB_OK;
    size_t l2_prev = 0;
    bool l2_changed = false;
    auto cleanup = [&]() {  // every exit path: error returns included
        if (l2_changed) {
            // hand the persisting-L2 carve-out back exactly as it was found (cudaDeviceSetLimit is process-wide state);
            // lines other code had pinned are left alone -- only our own window was ever marked persisting
            (void)cudaStreamSynchronize(st);
            (void)cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, l2_prev);
            (void)cudaGetLastError();
            l2_changed = false;
        }
        cudaFree(idx_dev), cudaFree(force_dev), cudaFree(slots), cudaFree(zh_alloc), cudaFree(mind);
        cudaFree(z0_dev), cudaFree(abort_dev);
    };
#define CS_TRY(expr)                                                                                         \
    do {                                                                                                     \
        cudaError_t _e = (expr);                                                                             \
        if (_e != cudaSuccess) {                                                                             \
            set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e));                  \
            (void)cudaGetLastError();                                                                        \
            cleanup();                                                                                       \
            return CMDB_ERR_CUDA;                                                                            \
        }                                                                                                    \
    } while (0)
    CS_TRY(cudaMalloc(&idx_dev, sizeof(long long) * (size_t)n_select));
    CS_TRY(cudaMalloc(&slots, sizeof(PickSlot) * 2 * (size_t)b->num_sms));
    CS_TRY(cudaMalloc(&abort_dev, sizeof(unsigned int)));
    CS_TRY(cudaMemsetAsync(abort_dev, 0, sizeof(unsigned int), st));
    if (force_idx_host) {
        CS_TRY(cudaMalloc(&force_dev, sizeof(long long) * (size_t)n_select));
        CS_TRY(cudaMemcpyAsync(force_dev, force_idx_host, sizeof(long long) * (size_t)n_select, cudaMemcpyHostToDevice, st));
    }
    CoresetParams p{};
    p.N = N, p.d = d, p.n_select = n_select, p.out_idx = idx_dev, p.force_idx = force_dev, p.slots = slots;
    p.l2_prev_limit = &l2_prev, p.l2_changed = &l2_changed;
    p.world = 1, p.rank = 0, p.row_offset = 0, p.abort_flag = abort_dev, p.spin_limit = 20LL * 1000 * 1000 * 1000;  // ~10 s
    const double *first_row = z_dev;  // pick 0 = global row 0
    const size_t es = dtype_mode == CMDB_CORESET_FP16 ? sizeof(__half) : sizeof(double);
    unsigned char *mine_in_replica = nullptr;  // this shard's rows inside the local replica of the projected bank
    if (sharded) {
        p.world = sh->world, p.rank = sh->rank, p.row_offset = sh->row_offset;
        p.mb_keys_off = kCommKeysOff, p.mb_ready_off = kCommReadyOff, p.ready_epoch = 1ULL;
        for (int r = 0; r < kMaxRanks; ++r) p.mb_peer[r] = sh->peers[r];
        CMDB_REQUIRE(b->num_sms <= (int)kCommMaxCtas, CMDB_ERR_UNSUPPORTED, "coreset: %d SMs exceed the mailbox layout", b->num_sms);
        CS_TRY(cudaMalloc(&z0_dev, sizeof(double) * (d + 1)));
        CS_TRY(cudaMemcpyAsync(z0_dev, sh->z0_host, sizeof(double) * d, cudaMemcpyHostToDevice, st));
        CS_TRY(cudaMemcpyAsync(z0_dev + d, &p.ready_epoch, sizeof(unsigned long long), cudaMemcpyHostToDevice, st));
        first_row = z0_dev;
        p.z_full = sh->peers[sh->rank] + kCommHeaderBytes;
        mine_in_replica = sh->peers[sh->rank] + kCommHeaderBytes + es * (size_t)sh->row_offset * d;
    }
    // row-sharded: the kernel reads the local rows from the replica (the natural [n_total, d] layout, so address alignment ==
    // global alignment class with no padding); every rank copies its slice into all peers' replicas over NVLink and then
    // raises its flag there (stream order: the flag lands after the rows)
    auto publish_shard = [&]() -> cudaError_t {
        for (int r = 0; r < p.world; ++r) {
            cudaError_t e = cudaSuccess;
            if (r != p.rank)
                e = cudaMemcpyAsync(sh->peers[r] + kCommHeaderBytes + es * (size_t)sh->row_offset * d, mine_in_replica,
                                    es * (size_t)N * d, cudaMemcpyDeviceToDevice, st);
            if (e == cudaSuccess)
                e = cudaMemcpyAsync(sh->peers[r] + kCommReadyOff + 8 * (size_t)p.rank, z0_dev + d, 8, cudaMemcpyDeviceToDevice, st);
            if (e != cudaSuccess) return e;
        }
        return cudaSuccess;
    };
    if (dtype_mode == CMDB_CORESET_FP16) {
        __half *zh;
        if (sharded) {
            zh = reinterpret_cast<__half *>(mine_in_replica);
        } else {
            CS_TRY(cudaMalloc(&zh_alloc, sizeof(__half) * ((size_t)N * d + 4)));
            zh = zh_alloc;
        }
        CS_TRY(cudaMalloc(&mind, sizeof(__half) * (size_t)std::max<int64_t>(N, 1)));
        // features.py:378 initial distances in float64, then .half() (:389-391)
        rc = launch_rownorm<double>(st, b->num_sms, z_dev, first_row, N, d, nullptr, reinterpret_cast<__half *>(mind), p.row_offset);
        if (rc == CMDB_OK) {
            to_half_kernel<<<b->num_sms * 4, 512, 0, st>>>(z_dev, (long long)N * d, zh);
            CS_TRY(cudaGetLastError());
            if (sharded) CS_TRY(publish_shard());
            p.z = zh, p.mind = mind;
            rc = launch_coreset<__half>(b, p, force_mind_global);
        }
    } else {
        CS_TRY(cudaMalloc(&mind, sizeof(double) * (size_t)N));
        rc = launch_rownorm<double>(st, b->num_sms, z_dev, first_row, N, d, reinterpret_cast<double *>(mind), nullptr, p.row_offset);
        if (rc == CMDB_OK) {
            p.z = z_dev, p.mind = mind;
            if (sharded) {
                CS_TRY(cudaMemcpyAsync(mine_in_replica, z_dev, es * (size_t)N * d, cudaMemcpyDeviceToDevice, st));
                CS_TRY(publish_shard());
                p.z = mine_in_replica;
            }
            rc = launch_coreset<double>(b, p, force_mind_global);
        }
    }
    if (rc != CMDB_OK) {
        cleanup();
        return rc;
    }
    unsigned int aborted = 0;
    CS_TRY(cudaMemcpyAsync(out_idx_host, idx_dev, sizeof(long long) * (size_t)n_select, cudaMemcpyDeviceToHost, st));
    CS_TRY(cudaMemcpyAsync(&aborted, abort_dev, sizeof(aborted), cudaMemcpyDeviceToHost, st));
    if (out_min_last_host)
        CS_TRY(cudaMemcpyAsync(out_min_last_host, mind,
                               (dtype_mode == CMDB_CORESET_FP16 ? sizeof(__half) : sizeof(double)) * (size_t)N,
                               cudaMemcpyDeviceToHost, st));
    CS_TRY(cudaStreamSynchronize(st));
#undef CS_TRY
    cleanup();
    if (aborted) {
        set_error("coreset: a peer rank did not answer within the exchange timeout (all ranks must call "
                  "cmdb_coreset_select_sharded together)");
        return CMDB_ERR_CUDA;
    }
    return CMDB_OK;
}

int coreset_greedy(cmdb_bank *b, const double *z_dev, int64_t N, int d, int64_t n_select, int dtype_mode,
                   int64_t *out_idx_host) {
    return coreset_greedy_dev(b, z_dev, N, d, n_select, dtype_mode, out_idx_host, nullptr, nullptr, nullptr, false);
}

int coreset_rownorms(int device, const void *z_host, const void *last_host, int64_t n_rows, int d, int dtype_mode,
                     void *out_host) {
    CMDB_REQUIRE(z_host && last_host && out_host && n_rows > 0 && d >= 32, CMDB_ERR_INVALID, "rownorms: bad arguments");
    CMDB_CUDA(cudaSetDevice(device));
    int num_sms = kNumSMsDefault;
    cudaDeviceGetAttribute(&num_sms, cudaDevAttrMultiProcessorCount, device);
    const size_t es = dtype_mode == CMDB_CORESET_FP16 ? sizeof(__half) : sizeof(double);
    void *z = nullptr, *last = nullptr, *out = nullptr;
    cudaError_t e = cudaMalloc(&z, es * (size_t)n_rows * d);
    if (e == cudaSuccess) e = cudaMalloc(&last, es * (size_t)d);
    if (e == cudaSuccess) e = cudaMalloc(&out, es * (size_t)n_rows);
    if (e == cudaSuccess) e = cudaMemcpy(z, z_host, es * (size_t)n_rows * d, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(last, last_host, es * (size_t)d, cudaMemcpyHostToDevice);
    int rc = CMDB_OK;
    if (e == cudaSuccess) {
        if (dtype_mode == CMDB_CORESET_FP16)
            rc = launch_rownorm<__half>(nullptr, num_sms, (const __half *)z, (const __half *)last, n_rows, d, (__half *)out,
                                        nullptr);
        else
            rc = launch_rownorm<double>(nullptr, num_sms, (const double *)z, (const double *)last, n_rows, d, (double *)out,
                                        nullptr);
        if (rc == CMDB_OK) e = cudaMemcpy(out_host, out, es * (size_t)n_rows, cudaMemcpyDeviceToHost);
    }
    cudaFree(z);
    cudaFree(last);
    cudaFree(out);
    if (rc != CMDB_OK) return rc;
    CMDB_CUDA(e);
    return CMDB_OK;
}

}  // namespace cmdb
