// Everything of compute_single_s_s_map (reference features.py:225-297) after the distance GEMM:
//   refine_cert certificate of the pre-filter GEMM + exact float32 re-check of every candidate inside the error band
//               -> min_val / min_idx (:227) and the packed argmax key of min_val -> s_star / s_idx (:228-231);
//               rescan / fallback_decide / rescan_finish: exact rescan of producers the certificate could not clear
//   refine      (3-term and diagnostics modes) exact re-check of the 4 best candidates
//   select      m_test = patch[s_idx], m_star = bank[min_idx[s_idx]] (:235-251)
//   reweight    w_dist = ||m_star - bank_r|| for every bank row, 3 smallest (:239-254), m_star_knn, w, s (:275-290):
//               reweight_lookup (bank neighbour table), reweight_cert (batch through the tensor cores) or reweight_kernel
//               (CUDA-core sweep of the float32 bank)
//   upsample_blur  bilinear 28^2/56^2 -> 224^2 (:293-294) + KNNGaussianBlur (utils/utils.py:71-83): /max, 8-bit
//               truncation, Pillow's 3+3 pass integer box blur, /255, *max -- 16 row bands / 16 column bands per image
#include <math.h>

#include "common.cuh"

namespace cmdb {

// exact ||a - b||^2 in float32, one warp: lanes stride over float4s, xor-shuffle tree
__device__ __forceinline__ float warp_sqdist(const float *__restrict__ a, const float *__restrict__ b, int dim4, int lane) {
    float acc = 0.f;
    for (int c = lane; c < dim4; c += 32) {
        const float4 x = __ldg(reinterpret_cast<const float4 *>(a) + c), y = __ldg(reinterpret_cast<const float4 *>(b) + c);
        float d;
        d = x.x - y.x, acc = fmaf(d, d, acc);
        d = x.y - y.y, acc = fmaf(d, d, acc);
        d = x.z - y.z, acc = fmaf(d, d, acc);
        d = x.w - y.w, acc = fmaf(d, d, acc);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    return acc;
}

// four bank rows against one query at once: per row exactly the accumulation order and shuffle tree of warp_sqdist
// (bit-identical values), with the loads of all four rows in flight together (the re-checks are latency bound)
__device__ __forceinline__ void warp_sqdist4(const float *__restrict__ a, const float *__restrict__ b0, const float *__restrict__ b1,
                                             const float *__restrict__ b2, const float *__restrict__ b3, int dim4, int lane,
                                             float (&out)[4]) {
    float acc0 = 0.f, acc1 = 0.f, acc2 = 0.f, acc3 = 0.f;
#pragma unroll 3
    for (int c = lane; c < dim4; c += 32) {
        const float4 x = __ldg(reinterpret_cast<const float4 *>(a) + c);
        const float4 y0 = __ldg(reinterpret_cast<const float4 *>(b0) + c), y1 = __ldg(reinterpret_cast<const float4 *>(b1) + c);
        const float4 y2 = __ldg(reinterpret_cast<const float4 *>(b2) + c), y3 = __ldg(reinterpret_cast<const float4 *>(b3) + c);
        float d;
        d = x.x - y0.x, acc0 = fmaf(d, d, acc0), d = x.y - y0.y, acc0 = fmaf(d, d, acc0);
        d = x.z - y0.z, acc0 = fmaf(d, d, acc0), d = x.w - y0.w, acc0 = fmaf(d, d, acc0);
        d = x.x - y1.x, acc1 = fmaf(d, d, acc1), d = x.y - y1.y, acc1 = fmaf(d, d, acc1);
        d = x.z - y1.z, acc1 = fmaf(d, d, acc1), d = x.w - y1.w, acc1 = fmaf(d, d, acc1);
        d = x.x - y2.x, acc2 = fmaf(d, d, acc2), d = x.y - y2.y, acc2 = fmaf(d, d, acc2);
        d = x.z - y2.z, acc2 = fmaf(d, d, acc2), d = x.w - y2.w, acc2 = fmaf(d, d, acc2);
        d = x.x - y3.x, acc3 = fmaf(d, d, acc3), d = x.y - y3.y, acc3 = fmaf(d, d, acc3);
        d = x.z - y3.z, acc3 = fmaf(d, d, acc3), d = x.w - y3.w, acc3 = fmaf(d, d, acc3);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        acc0 += __shfl_xor_sync(0xffffffffu, acc0, o), acc1 += __shfl_xor_sync(0xffffffffu, acc1, o);
        acc2 += __shfl_xor_sync(0xffffffffu, acc2, o), acc3 += __shfl_xor_sync(0xffffffffu, acc3, o);
    }
    out[0] = acc0, out[1] = acc1, out[2] = acc2, out[3] = acc3;
}

// ---------------------------------------------------------------------------------------------------------------
// refine: one warp per query.  cand[c][q] = (val1, idx1, val2, idx2) from n_cand producers (approximate d^2 up to a
// per-query constant; idx < 0 = empty).  Takes the 4 best approximate candidates, recomputes their distance exactly
// and keeps the smallest (ties -> lowest row).
// ---------------------------------------------------------------------------------------------------------------
constexpr int kRefineTop = 4;

__global__ void __launch_bounds__(256) refine_kernel(const float4 *__restrict__ cand, int n_cand, int cand_stride,
                                                     const float *__restrict__ q, const float *__restrict__ bank, int dim,
                                                     int P, int P_img, long long row_offset, float *__restrict__ min_val,
                                                     long long *__restrict__ min_idx, unsigned long long *s_key,
                                                     const int *__restrict__ list, const int *__restrict__ count) {
    // P = total query rows of the batch (B images of P_img patches each); s_key[b] is image b's packed argmax.
    // Compact mode (list != nullptr): candidate column c belongs to query list[c], c < *count.
    const int lane = threadIdx.x & 31;
    const int qc = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);  // candidate column
    if (qc >= (count ? __ldg(count) : P)) return;
    const int qi = list ? __ldg(list + qc) : qc;
    // each lane keeps its own sorted top-4 (approx value, row) over the candidates it scans
    float tv[kRefineTop];
    int ti[kRefineTop];
#pragma unroll
    for (int k = 0; k < kRefineTop; ++k) tv[k] = INFINITY, ti[k] = -1;
    auto insert = [&](float v, int i) {
        if (i < 0) return;
#pragma unroll
        for (int k = 0; k < kRefineTop; ++k) {
            if (ti[k] == i) return;  // duplicates cannot happen across producers, cheap guard anyway
            if (v < tv[k] || (v == tv[k] && i < ti[k]) || ti[k] < 0) {
                float fv = tv[k];
                int fi = ti[k];
                tv[k] = v, ti[k] = i;
                v = fv, i = fi;
                if (i < 0) return;
            }
        }
    };
    for (int c = lane; c < n_cand; c += 32) {
        const float4 t = cand[(size_t)c * cand_stride + qc];
        insert(t.x, __float_as_int(t.y));
        insert(t.z, __float_as_int(t.w));
    }
    // warp-wide top-4: pop the global minimum 4 times
    int sel_idx[kRefineTop];
#pragma unroll
    for (int r = 0; r < kRefineTop; ++r) {
        float v = tv[0];
        int i = ti[0];
        if (i < 0) v = INFINITY;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const float ov = __shfl_xor_sync(0xffffffffu, v, o);
            const int oi = __shfl_xor_sync(0xffffffffu, i, o);
            if (oi >= 0 && (i < 0 || ov < v || (ov == v && oi < i))) v = ov, i = oi;
        }
        sel_idx[r] = i;
        if (i >= 0 && ti[0] == i) {  // owner pops
#pragma unroll
            for (int k = 0; k + 1 < kRefineTop; ++k) tv[k] = tv[k + 1], ti[k] = ti[k + 1];
            tv[kRefineTop - 1] = INFINITY, ti[kRefineTop - 1] = -1;
        }
    }
    float best = INFINITY;
    int best_i = -1;
#pragma unroll
    for (int r = 0; r < kRefineTop; ++r) {
        const int i = sel_idx[r];
        if (i < 0) continue;
        const float d2 = warp_sqdist(q + (size_t)qi * dim, bank + (size_t)i * dim, dim >> 2, lane);
        if (best_i < 0 || d2 < best || (d2 == best && i < best_i)) best = d2, best_i = i;
    }
    if (lane == 0) {
        const float dv = sqrtf(best);
        min_val[qi] = dv;
        min_idx[qi] = best_i < 0 ? -1 : (long long)best_i + row_offset;
        argmax_publish(s_key, qi, P_img, dv);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// certified refine (hi.hi pre-filter GEMM): one warp per query.  The epilogue's value of bank row r for query q is
//     v(q,r) = fl(||b_r||^2) - 2 * acc(q_hi . b_hi)        and the exact re-check is  f(q,r) = warp_sqdist(q, b_r).
// |v + ||q||^2 - f| <= E(q) for every bank row, with
//     E = 2 (eps_q * Bh + ||q|| * eps_b + kAccModel * (||q|| + eps_q) * Bh) + gamma * (||q|| + B)^2
//   eps_q = ||q - q_hi||, eps_b = max_r ||b_r - b_hi,r||, B = max ||b||, Bh = B + eps_b          (Cauchy-Schwarz on the
//   operand rounding), acc_model bounds the accumulation of the exact fp16 products in the tensor core (D/16 MMAs of
//   16 products each, every addend aligned to the largest exponent and truncated to >= 24 bits: <= (D/16 + 1) * 17 *
//   2^-23 relative to ||q_hi|| ||b_hi||; tests/test_gpu_score.py measures the real error against this model), gamma =
//   (D + 16) * 2^-24 covers the float32 rounding of ||b||^2, of the epilogue fma and of warp_sqdist itself.
// Any row whose v exceeds v_min + 2E therefore cannot be the float32 nearest neighbour (not even through a tie).  Each
// producer CTA kept its two smallest v; if every CTA's SECOND value is above the threshold, all rows inside the band
// are first values -> they are ALL re-checked exactly and the result is certified identical to a full exact scan.
// A producer whose second value is inside the band may hide further rows: the (query, producer) pair is queued and
// the producer's ~R/producers rows are rescanned exactly (rescan_kernel) -- or, when a call queues so many pairs that
// this would cost more than a GEMM (fallback_use_rescan; banks full of near-duplicates), the uncertified queries are
// redone with the FP32-equivalent 3-term GEMM.  Either way min_val / min_idx equal those of an exact scan of the whole bank.
// ---------------------------------------------------------------------------------------------------------------
// One block per QB consecutive queries (launched with QB = 8), three phases:
//   (1) the producers' lists are read with the QUERY index along the lanes (a warp-wide load is 32 / QB contiguous runs of
//       QB x 16 bytes of cand[c][q0 ...]; round 1 read them one query per warp, 32 sectors of 32 producers per request,
//       which was two thirds of the kernel's time); every thread keeps its share in registers; smallest first value per
//       query through shared memory -> threshold;
//   (2) from the registers: every kept value inside a query's band goes to that query's row list in shared memory;
//       producers whose SECOND value is inside the band -- or whose row no longer fits the list -- are queued for the rescan;
//   (3) the listed rows are re-checked exactly, one warp per query, four rows at a time (warp_sqdist4).
// The last block of the grid to finish also takes the tier decision for the launches behind it (ctl[2..4]).
constexpr int kCertThreads = 256;
constexpr int kCertRows = 24;    // rows per query list; a query with more in-band first values hands the surplus to the rescan

// v_ref + 2E(q) with slack for the float32 evaluation of E itself, rounded up; +inf where that is not orderable (NaN,
// overflow): nothing is certified then
__device__ __forceinline__ float cert_threshold(float v_ref, float qn, float qe, float bmax, float eb_max, float acc_model, int dim) {
    const float bh = __fadd_ru(bmax, eb_max);
    float E = __fmul_ru(qe, bh);
    E = __fmaf_ru(qn, eb_max, E);
    E = __fmaf_ru(__fmul_ru(acc_model, __fadd_ru(qn, qe)), bh, E);
    E = __fmul_ru(2.f, E);
    const float span = __fadd_ru(qn, bmax);
    E = __fmaf_ru(__fmul_ru((float)(dim + 16) * 5.9604645e-8f, span), span, E);
    const float t = __fadd_ru(v_ref, __fmul_ru(2.0625f, E));
    return v_ref < INFINITY && t < INFINITY ? t : INFINITY;
}

// exact re-check of a query's listed rows (the smallest (d^2, row) wins: the order of the list does not matter)
__device__ __forceinline__ void cert_recheck(const int *list, int n_list, const float *__restrict__ qrow, const float *__restrict__ bank,
                                             int dim, int lane, float &best, int &best_i) {
    const int dim4 = dim >> 2;
    for (int j = 0; j < n_list; j += 4) {
        const int r0 = list[j], r1 = list[min(j + 1, n_list - 1)], r2 = list[min(j + 2, n_list - 1)], r3 = list[min(j + 3, n_list - 1)];
        float d[4];
        if (j + 1 < n_list) {
            warp_sqdist4(qrow, bank + (size_t)r0 * dim, bank + (size_t)r1 * dim, bank + (size_t)r2 * dim, bank + (size_t)r3 * dim,
                         dim4, lane, d);
        } else {
            d[0] = warp_sqdist(qrow, bank + (size_t)r0 * dim, dim4, lane);
            d[1] = d[2] = d[3] = d[0];
        }
        const int rr[4] = {r0, r1, r2, r3};
#pragma unroll
        for (int k = 0; k < 4; ++k)  // duplicates of the last row (padding of the group) change nothing
            if (best_i < 0 || d[k] < best || (d[k] == best && rr[k] < best_i)) best = d[k], best_i = rr[k];
    }
}

template <int QB>  // queries per block: 8, 16 or 32 (8: more blocks, one query per warp in phase 3)
__global__ void __launch_bounds__(kCertThreads) refine_cert_kernel(const float4 *__restrict__ cand, int n_cand, int cand_stride,
                                                          const float *__restrict__ q, const float *__restrict__ bank, int dim,
                                                          int P, int P_img, long long row_offset,
                                                          const float *__restrict__ q_norm, const float *__restrict__ q_eps,
                                                          float bmax, float eb_max, float acc_model,
                                                          float *__restrict__ min_val,
                                                          long long *__restrict__ min_idx, unsigned long long *s_key,
                                                          int *__restrict__ fail_list, int *__restrict__ ctl,
                                                          int2 *__restrict__ work_list, unsigned long long *__restrict__ best_key) {
    constexpr int kWarps = kCertThreads / 32;
    constexpr int PL = 32 / QB;            // producers covered by one warp-wide load
    constexpr int CSTEP = kWarps * PL;     // producers covered by one block-wide load
    __shared__ float part_s[CSTEP][QB];    // per (producer class, query) minima of phase 1
    __shared__ float thr_s[QB];
    __shared__ int cnt_s[QB], bad_s[QB], list_s[QB][kCertRows];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int ql = lane % QB;              // query of this thread inside the block (phases 1 and 2)
    const int q0 = blockIdx.x * QB, qi = q0 + ql;
    const int cls = warp * PL + lane / QB; // producers cls, cls + CSTEP, ...
    const bool live = qi < P;
    const float4 *col = cand + (live ? qi : q0);
    if (threadIdx.x < QB) cnt_s[threadIdx.x] = 0, bad_s[threadIdx.x] = 0;
    // ---- phase 1: smallest first value (a producer without any row for this query has idx < 0).  The thread's share of
    //      the lists stays in registers for phase 2 (kHold loads in flight together, ONE memory round trip for both
    //      phases; producers beyond kHold * CSTEP -- none on a 148-SM part -- are read again in phase 2) ----
    constexpr int kHold = QB <= 16 ? 320 / CSTEP : 8;
    const float4 empty = make_float4(INFINITY, __int_as_float(-1), INFINITY, __int_as_float(-1));
    float4 held[kHold];
    float v1 = INFINITY;
#pragma unroll
    for (int k = 0; k < kHold; ++k) {
        const int c = cls + k * CSTEP;
        held[k] = c < n_cand ? col[(size_t)c * cand_stride] : empty;
    }
#pragma unroll
    for (int k = 0; k < kHold; ++k)
        if (__float_as_int(held[k].y) >= 0) v1 = fminf(v1, held[k].x);
#pragma unroll 4
    for (int c = cls + kHold * CSTEP; c < n_cand; c += CSTEP) {
        const float4 t = col[(size_t)c * cand_stride];
        if (__float_as_int(t.y) >= 0) v1 = fminf(v1, t.x);
    }
    part_s[cls][ql] = v1;
    __syncthreads();
    if (threadIdx.x < QB) {
        float v1min = part_s[0][threadIdx.x];
#pragma unroll
        for (int k = 1; k < CSTEP; ++k) v1min = fminf(v1min, part_s[k][threadIdx.x]);
        const int qq = q0 + threadIdx.x;
        float thr = INFINITY;  // +inf: everything is inside the band
        if (qq < P) thr = cert_threshold(v1min, q_norm[qq], q_eps[qq], bmax, eb_max, acc_model, dim);
        thr_s[threadIdx.x] = thr;
    }
    __syncthreads();
    // ---- phase 2: band membership; rows to the query's list, (query, producer) pairs to the rescan queue ----
    {
        const float thr = thr_s[ql];
        const bool all_in = !(thr < INFINITY);
        auto band = [&](const float4 t, int c) {
            const int i1 = __float_as_int(t.y), i2 = __float_as_int(t.w);
            const bool in1 = i1 >= 0 && (t.x <= thr || all_in), in2 = i2 >= 0 && (t.z <= thr || all_in);
            bool queue = in2;   // a producer whose SECOND value is inside the band may hide more rows
            if (in1) {
                const int slot = atomicAdd(&cnt_s[ql], 1);
                if (slot < kCertRows) list_s[ql][slot] = i1;
                else queue = true;   // the row is covered by the exact rescan of its producer instead
            }
            if (in2) {
                const int slot = atomicAdd(&cnt_s[ql], 1);
                if (slot < kCertRows) list_s[ql][slot] = i2;
            }
            if (queue) {
                atomicAdd(&bad_s[ql], 1);
                const int slot = atomicAdd(ctl + 1, 1);
                if (slot < kWorkCap) work_list[slot] = make_int2(qi, c);
            }
        };
        if (live) {
#pragma unroll
            for (int k = 0; k < kHold; ++k) band(held[k], cls + k * CSTEP);   // empty entries (idx < 0) are never inside
#pragma unroll 4
            for (int c = cls + kHold * CSTEP; c < n_cand; c += CSTEP) band(col[(size_t)c * cand_stride], c);
        }
    }
    __syncthreads();
    // ---- phase 3: exact re-checks, one warp per query ----
    for (int k = warp; k < QB; k += kWarps) {
        const int qq = q0 + k;
        if (qq >= P) break;
        float best = INFINITY;
        int best_i = -1;
        cert_recheck(list_s[k], min(cnt_s[k], kCertRows), q + (size_t)qq * dim, bank, dim, lane, best, best_i);
        if (lane == 0) {
            if (bad_s[k] == 0 && best_i >= 0) {
                const float dv = sqrtf(best);
                min_val[qq] = dv;
                min_idx[qq] = (long long)best_i + row_offset;
                argmax_publish(s_key, qq, P_img, dv);
            } else {
                fail_list[atomicAdd(ctl + 0, 1)] = qq;
                best_key[qq] = best_i < 0 ? ~0ULL : pack_min_key(best, (unsigned int)best_i);
            }
        }
    }
    // the last block of the grid decides the tier: [2] rows of the GEMM fallback, [3] pairs of the rescan, [4] queries the
    // rescan path finishes (the launches behind this kernel size themselves from these)
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(ctl + 5, 1) == (int)gridDim.x - 1) {
            __threadfence();
            const int fails = atomicAdd(ctl + 0, 0), pairs = atomicAdd(ctl + 1, 0);
            const bool rescan = fallback_use_rescan(fails, pairs);
            ctl[2] = rescan ? 0 : fails;
            ctl[3] = rescan ? pairs : 0;
            ctl[4] = rescan ? fails : 0;
        }
    }
}

// exact rescan: work item = (query, producer); the producer (CTA c, column group g) saw, for the query's M tile, the N
// tiles rescan_tile names and of each the columns [g, g+1) * 256 / EG.  Unit = (item, tile slot, 32-row slice): the
// exact distances of its rows, the smallest (d^2 bits, row) folded into best_key[query] (atomicMin).  The first-pass
// GEMM launches are single CTAs (certified mode runs the 1-term GEMM), checked by score_rescan.
__global__ void __launch_bounds__(256) rescan_kernel(const int2 *__restrict__ work, const int *__restrict__ n_items_ptr,
                                                     const float *__restrict__ q, const float *__restrict__ bank, int dim,
                                                     long long rows, GemmSched full, GemmSched last, int chunk_tiles,
                                                     int mt_total, unsigned long long *best_key,
                                                     const int *__restrict__ fail_list, int *__restrict__ ctl, int P_img,
                                                     long long row_offset, float *__restrict__ min_val,
                                                     long long *__restrict__ min_idx, unsigned long long *s_key) {
    __shared__ int last_block;
    const int n_items = min(*n_items_ptr, kWorkCap);
    const int tiles_per = producer_slots(full, last);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int cols = kScoreBN / kGemmEpiGroups;
    // warp unit = (item, tile slot of the producer, 32-row slice of the tile's column group, warp slot): four exact
    // distances (rows r, r + 8, r + 16, r + 24) with all loads in flight together, one atomicMin per warp; no block barrier
    constexpr int kUnitRows = 32;
    const int units_per_tile = cols / kUnitRows;
    const long long n_work = (long long)n_items * tiles_per * units_per_tile * 8;
    for (long long wu = (long long)blockIdx.x * 8 + warp; wu < n_work; wu += (long long)gridDim.x * 8) {
        const int wsub = (int)(wu & 7);
        const long long u = wu >> 3;
        // item varies fastest: a producer's tile slots beyond its real tiles (about half of them: tiles_per covers the
        // longest producer) are empty, and this way every block meets its share of them instead of whole blocks idling
        const int item = (int)(u % n_items);
        const int rem = (int)(u / n_items);
        const int kt = rem / units_per_tile, sub = rem % units_per_tile;
        const int2 w = work[item];
        const int qi = w.x, c = w.y / kGemmEpiGroups, g = w.y % kGemmEpiGroups;
        const int n = rescan_tile(full, last, chunk_tiles, mt_total, qi / kScoreBM, c, kt);
        if (n < full.nt) {
            const long long r0 = (long long)n * kScoreBN + g * cols + sub * kUnitRows + wsub;
            if (r0 < rows) {
                const long long rl = rows - 1;
                const float *qrow = q + (size_t)qi * dim;
                float d[4];
                warp_sqdist4(qrow, bank + (size_t)r0 * dim, bank + (size_t)min(r0 + 8, rl) * dim, bank + (size_t)min(r0 + 16, rl) * dim,
                             bank + (size_t)min(r0 + 24, rl) * dim, dim >> 2, lane, d);
                unsigned long long key = ~0ULL;
#pragma unroll
                for (int kk4 = 0; kk4 < 4; ++kk4) {  // rows clamped to the last one repeat its key: harmless for a minimum
                    const unsigned long long kk = pack_min_key(d[kk4], (unsigned int)min(r0 + 8 * kk4, rl));
                    key = kk < key ? kk : key;
                }
                if (lane == 0) atomicMin(best_key + qi, key);
            }
        }
    }
    __syncthreads();
    // the last block to finish publishes min_val / min_idx / the argmax keys of the rescanned queries
    if (threadIdx.x == 0) {
        __threadfence();
        last_block = atomicAdd(ctl + 6, 1) == (int)gridDim.x - 1;
    }
    __syncthreads();
    if (!last_block) return;
    __threadfence();
    const int n_fin = ctl[4];
    for (int i = threadIdx.x; i < n_fin; i += blockDim.x) {
        const int qi = fail_list[i];
        const unsigned long long key = __ldcg(best_key + qi);
        const float dv = sqrtf(key_value(key));
        min_val[qi] = dv;
        min_idx[qi] = key == ~0ULL ? -1 : key_row(key) + row_offset;
        argmax_publish(s_key, qi, P_img, dv);
    }
}

// test hook: the exact scan the certificate promises equality with -- every (query, bank row) distance by warp_sqdist, smallest
// (d^2 bits, row) key per query.  grid (row chunks, query groups of 8); one warp per query.
__global__ void __launch_bounds__(256) exact_scan_kernel(const float *__restrict__ q, int P, const float *__restrict__ bank,
                                                         long long rows, int dim, long long chunk,
                                                         unsigned long long *__restrict__ best_key) {
    const int lane = threadIdx.x & 31, qi = blockIdx.y * 8 + (threadIdx.x >> 5);
    if (qi >= P) return;
    const long long r0 = (long long)blockIdx.x * chunk, r1 = min(rows, r0 + chunk);
    unsigned long long key = ~0ULL;
    for (long long r = r0; r < r1; ++r) {
        const float d2 = warp_sqdist(q + (size_t)qi * dim, bank + (size_t)r * dim, dim >> 2, lane);
        const unsigned long long kk = pack_min_key(d2, (unsigned int)r);
        key = kk < key ? kk : key;
    }
    if (lane == 0 && key != ~0ULL) atomicMin(best_key + qi, key);
}

int score_exact_scan(cmdb_bank *b, const float *q_dev, int P, unsigned long long *keys_dev) {
    const long long chunk = std::max<long long>(64, (b->fin_rows + 4 * b->num_sms - 1) / (4 * b->num_sms));
    const int gx = (int)((b->fin_rows + chunk - 1) / chunk);
    exact_scan_kernel<<<dim3(gx, (P + 7) / 8), 256, 0, b->handle_stream()>>>(q_dev, P, b->data, b->fin_rows, b->dim, chunk, keys_dev);
    CMDB_CUDA(cudaGetLastError());
    return CMDB_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// diagnostics scorer: exact direct-form float32 distances on CUDA cores, same candidate format as the GEMM epilogue.
// grid (query tiles of 64, bank slices); block 256 = 16x16 threads, 4x4 outputs each, K chunks of 32 through smem.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) simt_min_kernel(const float *__restrict__ q, int P, const float *__restrict__ bank,
                                                       long long R, int dim, float4 *__restrict__ cand, int cand_stride) {
    __shared__ float qs[64][33], bs[64][33];
    __shared__ float rv[64][16][2];
    __shared__ int ri[64][16][2];
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
    const int q0 = blockIdx.x * 64;
    const long long rows_per_slice = ((R + gridDim.y - 1) / gridDim.y + 63) / 64 * 64;
    const long long r_begin = (long long)blockIdx.y * rows_per_slice, r_end = min(R, r_begin + rows_per_slice);
    float b1[4], b2[4];
    int i1[4], i2[4];
#pragma unroll
    for (int a = 0; a < 4; ++a) b1[a] = b2[a] = INFINITY, i1[a] = i2[a] = -1;
    for (long long r0 = r_begin; r0 < r_end; r0 += 64) {
        float acc[4][4] = {};
        for (int k0 = 0; k0 < dim; k0 += 32) {
            __syncthreads();
            for (int i = threadIdx.x; i < 64 * 32; i += 256) {
                const int r = i >> 5, c = i & 31;
                qs[r][c] = (q0 + r < P) ? q[(size_t)(q0 + r) * dim + k0 + c] : 0.f;
                bs[r][c] = (r0 + r < r_end) ? bank[(size_t)(r0 + r) * dim + k0 + c] : 0.f;
            }
            __syncthreads();
#pragma unroll 8
            for (int k = 0; k < 32; ++k) {
                float qa[4], ba[4];
#pragma unroll
                for (int a = 0; a < 4; ++a) qa[a] = qs[ty * 4 + a][k], ba[a] = bs[tx * 4 + a][k];
#pragma unroll
                for (int a = 0; a < 4; ++a)
#pragma unroll
                    for (int c = 0; c < 4; ++c) {
                        const float d = qa[a] - ba[c];
                        acc[a][c] = fmaf(d, d, acc[a][c]);
                    }
            }
        }
#pragma unroll
        for (int a = 0; a < 4; ++a)
#pragma unroll
            for (int c = 0; c < 4; ++c) {
                const long long r = r0 + tx * 4 + c;
                if (r >= r_end) continue;
                const float v = acc[a][c];
                const int ri_ = (int)r;
                if (v < b1[a] || (v == b1[a] && ri_ < i1[a]) || i1[a] < 0) {
                    b2[a] = b1[a], i2[a] = i1[a], b1[a] = v, i1[a] = ri_;
                } else if (v < b2[a] || (v == b2[a] && ri_ < i2[a]) || i2[a] < 0) {
                    b2[a] = v, i2[a] = ri_;
                }
            }
    }
    __syncthreads();
#pragma unroll
    for (int a = 0; a < 4; ++a) {
        rv[ty * 4 + a][tx][0] = b1[a], rv[ty * 4 + a][tx][1] = b2[a];
        ri[ty * 4 + a][tx][0] = i1[a], ri[ty * 4 + a][tx][1] = i2[a];
    }
    __syncthreads();
    if (threadIdx.x < 64 && q0 + threadIdx.x < P) {
        float c1 = INFINITY, c2 = INFINITY;
        int j1 = -1, j2 = -1;
        for (int t = 0; t < 16; ++t)
            for (int u = 0; u < 2; ++u) {
                const float v = rv[threadIdx.x][t][u];
                const int i = ri[threadIdx.x][t][u];
                if (i < 0) continue;
                if (j1 < 0 || v < c1 || (v == c1 && i < j1)) c2 = c1, j2 = j1, c1 = v, j1 = i;
                else if (j2 < 0 || v < c2 || (v == c2 && i < j2)) c2 = v, j2 = i;
            }
        cand[(size_t)blockIdx.y * cand_stride + q0 + threadIdx.x] = make_float4(c1, __int_as_float(j1), c2, __int_as_float(j2));
    }
}

int score_simt_candidates(const ScoreCall &c, int P, int *n_cand_out) {
    const cmdb_bank *b = c.b;
    const int q_tiles = (P + 63) / 64;
    int slices = std::max(1, std::min(b->num_sms, (2 * b->num_sms + q_tiles - 1) / q_tiles));
    slices = (int)std::min<long long>(slices, (b->fin_rows + 63) / 64);
    simt_min_kernel<<<dim3(q_tiles, slices), 256, 0, c.stream>>>(c.slot->q_f32, P, b->data, b->fin_rows, b->dim, c.lane->cand,
                                                                b->layout.cap_p);
    CMDB_CUDA(cudaGetLastError());
    *n_cand_out = slices;
    return CMDB_OK;
}

int score_refine(const ScoreCall &c, cudaStream_t st, int B, int P_img, int n_cand, bool compact) {
    const cmdb_bank *b = c.b;
    const Lane &l = *c.lane;
    const int P = B * P_img;
    // compact mode follows score_certify, which already reset s_key and published the certified queries
    if (!compact) CMDB_CUDA(cudaMemsetAsync(l.s_key, 0, sizeof(unsigned long long) * B, st));
    refine_kernel<<<(P + 7) / 8, 256, 0, st>>>(l.cand, n_cand, b->layout.cap_p, c.slot->q_f32, b->data, b->dim, P, P_img,
                                               b->row_offset, c.min_val, c.min_idx, l.s_key, compact ? l.fail_list : nullptr,
                                               compact ? l.fail_ctl + 2 : nullptr);
    CMDB_CUDA(cudaGetLastError());
    return CMDB_OK;
}

static int score_certify(const ScoreCall &c, int B, int P_img, int n_cand) {
    const cmdb_bank *b = c.b;
    const Lane &s = *c.lane;
    const int P = B * P_img;
    cudaStream_t st = c.stream;
    CMDB_CUDA(cudaMemsetAsync(s.fail_ctl, 0, 8 * sizeof(int) + sizeof(unsigned long long) * B, st));  // control block + s_key
    const float acc_model = cert_acc_model(b->dim);
    if (b->timing == 2) CMDB_CUDA(cudaEventRecord(s.ev_dbg[0], st));
    // queries per block: 8 = one query per warp in phase 3 and 10 list entries per thread held in registers (measured best)
    constexpr int QB = 8;
    refine_cert_kernel<QB><<<(P + QB - 1) / QB, kCertThreads, 0, st>>>(s.cand, n_cand, b->layout.cap_p, c.slot->q_f32, b->data, b->dim,
                                                                       P, P_img, b->row_offset, s.q_norm, s.q_eps, b->cert_bmax,
                                                                       b->cert_eb_max, acc_model, c.min_val, c.min_idx, s.s_key,
                                                                       s.fail_list, s.fail_ctl, s.work_list, s.best_key);
    if (b->timing == 2) CMDB_CUDA(cudaEventRecord(s.ev_dbg[1], st));
    CMDB_CUDA(cudaGetLastError());
    return CMDB_OK;
}

static int score_rescan(const ScoreCall &c, int P_img) {
    const cmdb_bank *b = c.b;
    const Lane &s = *c.lane;
    cudaStream_t st = c.stream;
    CMDB_CUDA(cudaGetLastError());
    // tier 1: few uncertified (query, producer) pairs -> exact rescan of those producers' rows, along the first-pass schedule
    CMDB_REQUIRE(!c.first.pair && !c.last.pair, CMDB_ERR_UNSUPPORTED, "scoring: the exact rescan cannot walk a CTA-pair GEMM schedule");
    rescan_kernel<<<b->num_sms * 8, 256, 0, st>>>(s.work_list, s.fail_ctl + 3, c.slot->q_f32, b->data, b->dim, b->fin_rows, c.first,
                                                  c.last, c.chunk_tiles, c.mt_total, s.best_key, s.fail_list, s.fail_ctl, P_img,
                                                  b->row_offset, c.min_val, c.min_idx, s.s_key);
    CMDB_CUDA(cudaGetLastError());
    if (b->timing == 2) CMDB_CUDA(cudaEventRecord(s.ev_dbg[2], st));
    return CMDB_OK;
}

// min_val / min_idx / s_key of a sub-batch in the bank's GEMM mode: stages the queries into the slot's q_f32, builds the
// candidate lists, refines.  ev_gemm / ev_refine: timing event slots recorded before the (first) GEMM and before the
// (first) refine, or -1.
// Host queries are staged in up to kMaxStageChunks chunks on a copy stream; chunk c is split and multiplied while chunk
// c + 1 is still crossing PCIe.  (One GEMM launch per chunk: each streams the fp16 bank once more, which is cheap next to
// the host link.)  Device-resident queries use one chunk.
int score_local_min(ScoreCall &c, const float *src, int src_is_device, int B, int P_img, int ev_gemm, int ev_refine,
                    cudaEvent_t stage_after) {
    cmdb_bank *b = c.b;
    const Lane &l = *c.lane;
    float *q_f32 = c.slot->q_f32;
    cudaStream_t st = c.stream;
    const int P = B * P_img;
    const size_t D = b->dim;
    int n_cand = 0;
    const int64_t prev_queries = b->last_queries;
    b->last_queries = P;
    if (b->score_impl != CMDB_SCORE_TCGEN05) {
        b->last_mode = 3;
        CMDB_CUDA(cudaMemcpyAsync(q_f32, src, sizeof(float) * P * D, src_is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
        if (b->q_norm_enabled) launch_normalize(st, b->num_sms, q_f32, (int64_t)P * D, b->q_mean, b->q_std);
        CMDB_CHECK(score_mark(c, ev_gemm, st));
        CMDB_CHECK(score_simt_candidates(c, P, &n_cand));
        CMDB_CHECK(score_mark(c, ev_refine, st));
        return score_refine(c, st, B, P_img, n_cand, false);
    }
    int mode = b->prefilter_terms;
    if (mode == 0) {
        // adaptive: when most queries of the previous certified call needed the GEMM fallback (dense near-duplicate
        // banks), run the FP32-equivalent GEMM directly for a while, then probe the pre-filter again
        // (the counters of the previous certified call; if their copy has not landed yet -- pipelined submits -- look again
        // next time instead of stalling the host)
        if (b->fail_pending && b->last_fail_host && cudaEventQuery(b->ev_fail) == cudaSuccess) {
            b->fail_pending = false;
            if (prev_queries > 0 && !fallback_use_rescan(b->last_fail_host[0], b->last_fail_host[1]) &&
                (double)b->last_fail_host[0] > 0.5 * (double)prev_queries)
                b->direct_calls_left = 32;
        }
        if (b->direct_calls_left > 0) {
            --b->direct_calls_left;
            mode = 3;
        }
    }
    b->last_mode = mode;
    const int mt_total = (P + kScoreBM - 1) / kScoreBM;
    // another batch in flight on this handle (submit / wait pipeline): the whole copy already overlaps that batch's
    // kernels, so one chunk -- and one GEMM launch -- is best
    const bool overlapped = b->any_pending();
    const bool via_copy_stream = !src_is_device && (overlapped || mt_total >= 16);
    int n_chunks = 1;
    if (via_copy_stream && !overlapped) n_chunks = mt_total >= 64 ? 4 : 2;
    n_chunks = std::max(1, std::min(std::min(n_chunks, kMaxStageChunks), mt_total));
    const int chunk_tiles = (mt_total + n_chunks - 1) / n_chunks;
    n_chunks = (mt_total + chunk_tiles - 1) / chunk_tiles;
    c.chunk_tiles = chunk_tiles, c.mt_total = mt_total;
    if (via_copy_stream) {
        // the copy stream may only overwrite q_f32 once its previous readers are done: the event the caller names, or
        // everything queued on the compute stream so far
        if (!stage_after) {
            CMDB_CUDA(cudaEventRecord(b->ev_chunk[0], st));
            stage_after = b->ev_chunk[0];
        }
        CMDB_CUDA(cudaStreamWaitEvent(b->copy_stream, stage_after, 0));
    }
    for (int k = 0; k < n_chunks; ++k) {
        const int row0 = k * chunk_tiles * kScoreBM, rows = std::min(P, (k + 1) * chunk_tiles * kScoreBM) - row0;
        const size_t o = (size_t)row0 * D;
        if (!via_copy_stream) {
            CMDB_CUDA(cudaMemcpyAsync(q_f32, src, sizeof(float) * P * D, src_is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, st));
        } else {
            CMDB_CUDA(cudaMemcpyAsync(q_f32 + o, src + o, sizeof(float) * rows * D, cudaMemcpyHostToDevice, b->copy_stream));
            CMDB_CUDA(cudaEventRecord(b->ev_chunk[k], b->copy_stream));
        }
    }
    GemmSched sched{};
    for (int k = 0; k < n_chunks; ++k) {
        const int row0 = k * chunk_tiles * kScoreBM, rows = std::min(P, (k + 1) * chunk_tiles * kScoreBM) - row0;
        if (via_copy_stream) CMDB_CUDA(cudaStreamWaitEvent(st, b->ev_chunk[k], 0));
        // (patch - mean) / std on the device (multiple_features.py:90): without chunking the one copy above covers all rows
        if (b->q_norm_enabled)
            launch_normalize(st, b->num_sms, q_f32 + (size_t)row0 * D, (int64_t)(via_copy_stream ? rows : P) * D, b->q_mean, b->q_std);
        CMDB_CHECK(score_query_prep(c, st, rows, false, row0));
        if (k == 0) CMDB_CHECK(score_mark(c, ev_gemm, st));
        CMDB_CHECK(score_gemm_candidates(c, st, rows, mode == 3 ? 3 : 1, false, &sched, row0));
        if (k == 0) c.first = sched;
    }
    c.last = sched;
    n_cand = sched.producers;
    CMDB_CHECK(score_mark(c, ev_refine, st));
    if (mode != 0) return score_refine(c, st, B, P_img, n_cand, false);
    // certificate kernel (takes the tier decision), then the two tiers side by side: the exact rescan on the lane's stream,
    // the counters copy and the tier-2 launches on the lane's side stream.  The tiers are exclusive (the control block
    // enables one of them) and touch disjoint buffers, so nothing orders them against each other; the side stream's launches
    // are empty in the common case and their launch latencies (27 us in a row) disappear behind the rescan.
    cudaStream_t aux = l.aux;
    CMDB_CHECK(score_certify(c, B, P_img, n_cand));
    CMDB_CUDA(cudaEventRecord(l.ev_fork, st));
    CMDB_CUDA(cudaStreamWaitEvent(aux, l.ev_fork, 0));
    CMDB_CHECK(score_rescan(c, P_img));
    int rc = CMDB_OK;
    if (cudaMemcpyAsync(l.fail_count_host, l.fail_ctl, 2 * sizeof(int), cudaMemcpyDeviceToHost, aux) != cudaSuccess ||
        cudaEventRecord(b->ev_fail, aux) != cudaSuccess)
        rc = CMDB_ERR_CUDA;
    b->fail_pending = true;
    b->last_fail_host = l.fail_count_host;   // this lane's pinned counters
    // tier 2 (many uncertified pairs): FP32-equivalent GEMM over the compacted uncertified queries; every launch sizes
    // itself from the device-side control block and returns at once in the common case
    if (rc == CMDB_OK) rc = score_query_prep(c, aux, P, true);
    if (rc == CMDB_OK) rc = score_gemm_candidates(c, aux, P, 3, true, &sched);
    if (rc == CMDB_OK) rc = score_refine(c, aux, B, P_img, sched.producers, true);
    if (rc != CMDB_OK) {
        if (rc == CMDB_ERR_CUDA) set_error("scoring: CUDA error while enqueuing the fallback tier: %s", cudaGetErrorString(cudaGetLastError()));
        return rc;
    }
    CMDB_CUDA(cudaEventRecord(l.ev_join, aux));
    CMDB_CUDA(cudaStreamWaitEvent(st, l.ev_join, 0));
    if (b->timing == 2) CMDB_CUDA(cudaEventRecord(l.ev_dbg[3], st));
    return CMDB_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// select (sharded mode): image b = blockIdx.x: decode the argmax key, stage m_test and (if owned locally) m_star
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) select_kernel(const unsigned long long *s_key, const long long *min_idx, int P_img,
                                                     const float *__restrict__ q, const float *__restrict__ bank, int dim,
                                                     long long row_offset, long long rows, float *m_test, float *m_star,
                                                     TailResult *res) {
    const int b = blockIdx.x;
    const unsigned long long key = s_key[b];
    const int s_idx = argmax_query(key);
    const long long g = min_idx[(size_t)b * P_img + s_idx];
    for (int c = threadIdx.x; c < dim; c += blockDim.x) {
        m_test[(size_t)b * dim + c] = q[((size_t)b * P_img + s_idx) * dim + c];
        const long long l = g - row_offset;
        if (m_star) m_star[(size_t)b * dim + c] = (l >= 0 && l < rows) ? bank[(size_t)l * dim + c] : 0.f;
    }
    if (threadIdx.x == 0) {
        res[b].s_idx = s_idx;
        res[b].s_star = key_value(key);
        res[b].m_star_row = g;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// reweight: exact ||m_star_b - bank_r||^2 for every local bank row and every image b of the batch, 3 smallest per image
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void top3_insert(unsigned long long (&t)[3], unsigned long long k) {
    if (k < t[2]) {
        if (k < t[1]) {
            t[2] = t[1];
            if (k < t[0]) t[1] = t[0], t[0] = k;
            else t[1] = k;
        } else {
            t[2] = k;
        }
    }
}
__device__ __forceinline__ void top3_insert_sh(unsigned long long *t, unsigned long long k) {  // t[3] in shared memory
    unsigned long long r[3] = {t[0], t[1], t[2]};
    top3_insert(r, k);
    t[0] = r[0], t[1] = r[1], t[2] = r[2];
}
// warp-wide 3 smallest of per-lane sorted triples (keys unique): "everyone offers its head, the winner pops" x3
__device__ __forceinline__ void warp_top3(unsigned long long (&t)[3], unsigned long long (&out)[3]) {
#pragma unroll
    for (int r = 0; r < 3; ++r) {
        unsigned long long v = t[0];
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            const unsigned long long ov = __shfl_xor_sync(0xffffffffu, v, o);
            v = ov < v ? ov : v;
        }
        out[r] = v;
        if (v != ~0ULL && t[0] == v) t[0] = t[1], t[1] = t[2], t[2] = ~0ULL;
    }
}

// m_star_knn, w and s of an image (features.py:275-290) from s* and the distances to m_star's two nearest other rows
__device__ __forceinline__ void reweight_final(TailResult *res, float s_star, float knn0, float knn1, int dim) {
    const float Dn = sqrtf((float)dim);  // torch.sqrt(torch.tensor(patch.shape[1]))  (features.py:285)
    const float den = expf(knn0 / Dn) + expf(knn1 / Dn);
    const float w = 1.f - expf(s_star / Dn) / den;  // features.py:287
    res->w = w;
    res->s = w * s_star;  // features.py:290
    res->knn0 = knn0, res->knn1 = knn1;
}

struct ReweightParams {
    const float *bank;               // [rows, dim] float32 (local shard)
    long long rows, row_offset;
    int dim, B, P_img;
    const float *q;                  // [B*P_img, dim] normalised patches
    const unsigned long long *s_key; // [B] packed argmax of min_val
    const long long *min_idx;        // [B*P_img] global rows
    unsigned long long *block_keys;  // [B][gridDim.x * 3]
    unsigned long long *top3;        // [B][3] merged result
    unsigned int *done_counter;      // last-block-done counter (self resetting)
    TailResult *res;                 // [B]
};

// w_dist pass (features.py:239-254) for a batch of B images in ONE sweep over the bank: every warp keeps a bank row in
// registers and evaluates its exact squared distance to all B m_star rows (shared memory), so the bank is read once
// per batch (rows*dim*4 bytes).  Prologue = "select" (decode s*, s_idx, locate m_star); epilogue = last-block-done
// merge + final re-weighting, so the whole re-weighting stage is one launch.
template <int DV>  // float4 vectors per lane: ceil(dim / 128)
__global__ void __launch_bounds__(256) reweight_kernel(ReweightParams p) {
    extern __shared__ __align__(16) float ms[];  // [B][dim] m_star rows, then wtop [8][B][3]
    const int dim = p.dim, B = p.B;
    unsigned long long *wtop = reinterpret_cast<unsigned long long *>(ms + (size_t)B * dim);
    __shared__ int s_idx_sh[32];
    __shared__ long long g_sh[32];
    __shared__ bool is_last;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    if (threadIdx.x < B) {
        const unsigned long long skey = p.s_key[threadIdx.x];
        const int s_idx = argmax_query(skey);
        s_idx_sh[threadIdx.x] = s_idx;
        g_sh[threadIdx.x] = p.min_idx[(size_t)threadIdx.x * p.P_img + s_idx];
    }
    for (int i = threadIdx.x; i < 8 * B * 3; i += blockDim.x) wtop[i] = ~0ULL;
    __syncthreads();
    for (int i = threadIdx.x; i < B * dim; i += blockDim.x) {
        const int b = i / dim, c = i - b * dim;
        ms[i] = p.bank[(size_t)(g_sh[b] - p.row_offset) * dim + c];
    }
    __syncthreads();
    const float4 *ms4 = reinterpret_cast<const float4 *>(ms);
    const int dim4 = dim >> 2;
    unsigned long long *my_top = wtop + (size_t)warp * B * 3;
    const long long warps = (long long)gridDim.x * 8;
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
    bool valid[DV];  // dim is a multiple of 64: the last vector may cover only lanes 0..15
#pragma unroll
    for (int j = 0; j < DV; ++j) valid[j] = lane + 32 * j < dim4;
    // two bank rows per iteration share every shared-memory read of the B targets; the next pair is prefetched while
    // the current one is compared
    float4 x0[DV], x1[DV], n0[DV], n1[DV];
    auto load_pair = [&](long long r, float4(&a)[DV], float4(&c)[DV]) {
        const long long r2 = r + warps;
#pragma unroll
        for (int j = 0; j < DV; ++j) {
            a[j] = (valid[j] && r < p.rows) ? __ldg(reinterpret_cast<const float4 *>(p.bank + (size_t)r * dim) + lane + 32 * j) : zero4;
            c[j] = (valid[j] && r2 < p.rows) ? __ldg(reinterpret_cast<const float4 *>(p.bank + (size_t)r2 * dim) + lane + 32 * j) : zero4;
        }
    };
    long long r = (long long)blockIdx.x * 8 + warp;
    load_pair(r, x0, x1);
    for (; r < p.rows; r += 2 * warps) {
        load_pair(r + 2 * warps, n0, n1);
        const long long r2 = r + warps;
        const unsigned int grow0 = (unsigned int)(r + p.row_offset), grow1 = (unsigned int)(r2 + p.row_offset);
        for (int b = 0; b < B; ++b) {
            float acc0 = 0.f, acc1 = 0.f;
#pragma unroll
            for (int j = 0; j < DV; ++j) {
                const float4 y = valid[j] ? ms4[b * dim4 + lane + 32 * j] : zero4;
                float d;
                d = x0[j].x - y.x, acc0 = fmaf(d, d, acc0);
                d = x0[j].y - y.y, acc0 = fmaf(d, d, acc0);
                d = x0[j].z - y.z, acc0 = fmaf(d, d, acc0);
                d = x0[j].w - y.w, acc0 = fmaf(d, d, acc0);
                d = x1[j].x - y.x, acc1 = fmaf(d, d, acc1);
                d = x1[j].y - y.y, acc1 = fmaf(d, d, acc1);
                d = x1[j].z - y.z, acc1 = fmaf(d, d, acc1);
                d = x1[j].w - y.w, acc1 = fmaf(d, d, acc1);
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                acc0 += __shfl_xor_sync(0xffffffffu, acc0, o);
                acc1 += __shfl_xor_sync(0xffffffffu, acc1, o);
            }
            if (lane == 0) {
                const unsigned long long k0 = pack_min_key(acc0, grow0);
                if (k0 < my_top[b * 3 + 2]) top3_insert_sh(my_top + b * 3, k0);
                if (r2 < p.rows) {
                    const unsigned long long k1 = pack_min_key(acc1, grow1);
                    if (k1 < my_top[b * 3 + 2]) top3_insert_sh(my_top + b * 3, k1);
                }
            }
        }
#pragma unroll
        for (int j = 0; j < DV; ++j) x0[j] = n0[j], x1[j] = n1[j];
    }
    __syncthreads();
    // block result per image: merge the 8 warps' triples
    if (threadIdx.x < B) {
        unsigned long long f[3] = {~0ULL, ~0ULL, ~0ULL};
        for (int w = 0; w < 8; ++w)
            for (int k = 0; k < 3; ++k) top3_insert(f, wtop[((size_t)w * B + threadIdx.x) * 3 + k]);
        unsigned long long *dst = p.block_keys + ((size_t)threadIdx.x * gridDim.x + blockIdx.x) * 3;
        dst[0] = f[0], dst[1] = f[1], dst[2] = f[2];
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) is_last = atomicAdd(p.done_counter, 1u) == gridDim.x - 1;
    __syncthreads();
    if (!is_last) return;
    // ---- last block: one warp per image merges every block's keys, then finishes the re-weighting ----
    __threadfence();
    if (threadIdx.x == 0) *p.done_counter = 0;
    for (int b = warp; b < B; b += 8) {
        unsigned long long t[3] = {~0ULL, ~0ULL, ~0ULL}, f[3];
        const unsigned long long *src = p.block_keys + (size_t)b * gridDim.x * 3;
        for (int i = lane; i < (int)gridDim.x * 3; i += 32) top3_insert(t, __ldcg(src + i));
        warp_top3(t, f);
        const float s_star = key_value(p.s_key[b]);
        const int s_idx = s_idx_sh[b];
        float knn[2] = {NAN, NAN};  // features.py:275-283: m_star_knn = ||m_test - bank[nn_idx[1:]]||, m_test = patch[s_idx]
#pragma unroll
        for (int k = 0; k < 2; ++k)
            if (f[1 + k] != ~0ULL)
                knn[k] = sqrtf(warp_sqdist(p.q + ((size_t)b * p.P_img + s_idx) * dim,
                                           p.bank + (size_t)(key_row(f[1 + k]) - p.row_offset) * dim, dim4, lane));
        if (lane == 0) {
            TailResult *res = p.res + b;
            p.top3[b * 3 + 0] = f[0], p.top3[b * 3 + 1] = f[1], p.top3[b * 3 + 2] = f[2];
            res->s_idx = s_idx;
            res->s_star = s_star;
            res->m_star_row = g_sh[b];
            for (int k = 0; k < 3; ++k) res->nn_idx[k] = f[k] == ~0ULL ? -1 : key_row(f[k]);
            reweight_final(res, s_star, knn[0], knn[1], dim);
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// re-weighting on the tensor cores: the B m_star rows go through the same hi.hi distance GEMM (one M tile), and this
// kernel -- one block per image -- turns the producers' top-2 lists into the EXACT three nearest bank rows:
//   thr = (third smallest kept value) + 2E, E as in refine_cert_kernel.  Three kept rows lie at or below v3, so any
//   row above thr is strictly farther (in float32) than three other rows and cannot be in the top-3.  Every kept value
//   <= thr is re-checked exactly; a producer whose SECOND value is <= thr may hide more rows, so its ~R/producers rows
//   are scanned exactly by the block.  Keys are (d^2 bits << 32 | global row) with d^2 from warp_sqdist -- the same
//   arithmetic as reweight_kernel, hence identical keys, order and ties.
// ---------------------------------------------------------------------------------------------------------------
struct ReweightCertParams {
    const float4 *cand;
    int n_cand, cand_stride;
    const float *m_star;             // [B, dim]
    const float *m_test;             // [B, dim] (with res only)
    const float *bank;
    long long rows, row_offset;
    int dim;
    const float *q_norm, *q_eps;     // of the m_star rows (q_split_kernel)
    float bmax, eb_max, acc_model;
    GemmSched sched;                 // of the GEMM launch (single CTAs)
    const unsigned long long *s_key;
    unsigned long long *top3;
    TailResult *res;                 // nullptr: only the keys (table build)
};

__device__ __forceinline__ unsigned int float_order_bits(float v) {  // monotone float -> uint (handles negatives)
    const unsigned int b = __float_as_uint(v);
    return b ^ ((b >> 31) ? 0xffffffffu : 0x80000000u);
}
__device__ __forceinline__ float float_from_order_bits(unsigned int u) {
    return __uint_as_float(u ^ ((u >> 31) ? 0x80000000u : 0xffffffffu));
}

__global__ void __launch_bounds__(256) reweight_cert_kernel(ReweightCertParams p) {
    constexpr int kMaxProd = 2 * 160;            // producers (CTAs x epilogue groups) this kernel supports
    __shared__ unsigned long long wkeys[8][3];
    __shared__ int cand_rows[kMaxProd];
    __shared__ int bad_prod[kMaxProd];
    __shared__ int n_rows_sh, n_bad_sh;
    __shared__ float thr_sh;
    const int b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int dim = p.dim, dim4 = dim >> 2;
    const float *ms = p.m_star + (size_t)b * dim;
    if (threadIdx.x == 0) n_rows_sh = 0, n_bad_sh = 0;
    // ---- third smallest kept approximate value ----
    unsigned long long t3[3] = {~0ULL, ~0ULL, ~0ULL}, f3[3];
    for (int c = threadIdx.x; c < p.n_cand; c += blockDim.x) {
        const float4 t = p.cand[(size_t)c * p.cand_stride + b];
        const int i1 = __float_as_int(t.y), i2 = __float_as_int(t.w);
        if (i1 >= 0) top3_insert(t3, ((unsigned long long)float_order_bits(t.x) << 32) | (unsigned int)i1);
        if (i2 >= 0) top3_insert(t3, ((unsigned long long)float_order_bits(t.z) << 32) | (unsigned int)i2);
    }
    warp_top3(t3, f3);
    if (lane == 0) wkeys[warp][0] = f3[0], wkeys[warp][1] = f3[1], wkeys[warp][2] = f3[2];
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long g3[3] = {~0ULL, ~0ULL, ~0ULL};
        for (int w = 0; w < 8; ++w)
            for (int k = 0; k < 3; ++k) top3_insert(g3, wkeys[w][k]);
        float thr = INFINITY;  // fewer than three real rows: everything is a candidate
        if (g3[2] != ~0ULL)
            thr = cert_threshold(float_from_order_bits((unsigned int)(g3[2] >> 32)), p.q_norm[b], p.q_eps[b], p.bmax, p.eb_max,
                                 p.acc_model, dim);
        thr_sh = thr;
    }
    __syncthreads();
    const float thr = thr_sh;
    // ---- candidate rows (kept values inside the band) and producers that may hide more ----
    for (int c = threadIdx.x; c < p.n_cand; c += blockDim.x) {
        const float4 t = p.cand[(size_t)c * p.cand_stride + b];
        const int i1 = __float_as_int(t.y), i2 = __float_as_int(t.w);
        // second value inside the band: the whole producer is rescanned (that covers its two kept rows as well)
        if (i2 >= 0 && !(t.z > thr)) bad_prod[atomicAdd(&n_bad_sh, 1)] = c;
        else if (i1 >= 0 && !(t.x > thr)) cand_rows[atomicAdd(&n_rows_sh, 1)] = i1;
    }
    __syncthreads();
    // ---- exact keys: candidates, then every row of the producers that could not be certified ----
    unsigned long long w3[3] = {~0ULL, ~0ULL, ~0ULL};  // identical in all lanes of the warp
    auto visit = [&](long long r) {
        const float d2 = warp_sqdist(ms, p.bank + (size_t)r * dim, dim4, lane);
        const unsigned long long key = pack_min_key(d2, (unsigned int)(r + p.row_offset));
        if (key != w3[0] && key != w3[1] && key != w3[2]) top3_insert(w3, key);
    };
    const int n_rows = n_rows_sh, n_bad = n_bad_sh;
    for (int i = warp; i < n_rows; i += 8) visit(cand_rows[i]);
    const int cols = kScoreBN / kGemmEpiGroups, slots = producer_slots(p.sched, p.sched);
    for (int i = 0; i < n_bad; ++i) {
        const int c = bad_prod[i] / kGemmEpiGroups, g = bad_prod[i] % kGemmEpiGroups;
        // the query row's M tile inside the GEMM launch: 0 for the re-weighting of a batch, the table build has many
        for (int j = warp; j < slots * cols; j += 8) {
            const int n = producer_tile(p.sched, p.sched.run, c, b / kScoreBM, j / cols);
            const long long r = (long long)n * kScoreBN + g * cols + j % cols;
            if (n < p.sched.nt && r < p.rows) visit(r);
        }
    }
    if (lane == 0) wkeys[warp][0] = w3[0], wkeys[warp][1] = w3[1], wkeys[warp][2] = w3[2];
    __syncthreads();
    if (warp != 0) return;
    unsigned long long f[3] = {~0ULL, ~0ULL, ~0ULL};
    for (int w = 0; w < 8; ++w)
        for (int k = 0; k < 3; ++k) {
            const unsigned long long key = wkeys[w][k];
            if (key != f[0] && key != f[1] && key != f[2]) top3_insert(f, key);
        }
    float s_star = 0.f;
    float knn[2] = {NAN, NAN};
    if (p.res) {  // features.py:275-283: m_star_knn = ||m_test - bank[nn_idx[1:]]||, m_test = patch[s_idx]
        s_star = key_value(p.s_key[b]);
#pragma unroll
        for (int k = 0; k < 2; ++k)
            if (f[1 + k] != ~0ULL)
                knn[k] = sqrtf(warp_sqdist(p.m_test + (size_t)b * dim,
                                           p.bank + (size_t)(key_row(f[1 + k]) - p.row_offset) * dim, dim4, lane));
    }
    if (lane == 0) {
        p.top3[(size_t)b * 3 + 0] = f[0], p.top3[(size_t)b * 3 + 1] = f[1], p.top3[(size_t)b * 3 + 2] = f[2];
        if (!p.res) return;  // table build: only the keys
        TailResult *res = p.res + b;
        for (int k = 0; k < 3; ++k) res->nn_idx[k] = f[k] == ~0ULL ? -1 : key_row(f[k]);
        reweight_final(res, s_star, knn[0], knn[1], dim);
    }
}

// re-weighting with the bank's precomputed neighbour table (cmdb_bank_build_knn): image b = blockIdx.x, 2 warps.
// m_star is bank row res[b].m_star_row (select_kernel), so its three nearest rows are table[m_star_row]; what is left of
// features.py:239-290 is m_star_knn = ||m_test - bank[nn_idx[1:]]||, w and s.
__global__ void __launch_bounds__(64) reweight_lookup_kernel(const unsigned long long *__restrict__ table, const float *__restrict__ m_test,
                                                            const float *__restrict__ bank, int dim,
                                                            const unsigned long long *__restrict__ s_key, unsigned long long *top3,
                                                            TailResult *res_all) {
    const int b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    __shared__ float knn[2];
    TailResult *res = res_all + b;
    const unsigned long long *keys3 = table + (size_t)res->m_star_row * 3;
    const unsigned long long key = keys3[1 + warp];
    float v = NAN;
    if (key != ~0ULL) v = sqrtf(warp_sqdist(m_test + (size_t)b * dim, bank + (size_t)key_row(key) * dim, dim >> 2, lane));
    if (lane == 0) knn[warp] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        const float s_star = key_value(s_key[b]);
        for (int k = 0; k < 3; ++k) {
            top3[b * 3 + k] = keys3[k];
            res->nn_idx[k] = keys3[k] == ~0ULL ? -1 : key_row(keys3[k]);
        }
        reweight_final(res, s_star, knn[0], knn[1], dim);
    }
}

// sharded mode with the REPLICATED neighbour table (every rank holds the keys of all global rows; the bank rows themselves
// stay sharded): image b = blockIdx.x, 2 warps.  m_star's three nearest rows are table[m_star_row]; this rank contributes
// the exact squared distance ||m_test - bank[nn_k]||^2 (k = 1, 2) for the neighbour rows it owns and 0 for the others, so
// that a float SUM all-reduce over the ranks reproduces warp_sqdist's value bit for bit (x + 0 + ... + 0).
__global__ void __launch_bounds__(64) shard_lookup_kernel(const unsigned long long *__restrict__ table, const float *__restrict__ m_test,
                                                         const float *__restrict__ bank, long long rows, long long row_offset,
                                                         int dim, unsigned long long *top3, TailResult *res_all,
                                                         float *__restrict__ contrib) {
    const int b = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    TailResult *res = res_all + b;
    const unsigned long long *keys3 = table + (size_t)res->m_star_row * 3;
    const unsigned long long key = keys3[1 + warp];
    const long long l = key_row(key) - row_offset;
    float v = 0.f;
    if (key != ~0ULL && l >= 0 && l < rows) v = warp_sqdist(m_test + (size_t)b * dim, bank + (size_t)l * dim, dim >> 2, lane);
    if (lane == 0) contrib[b * 2 + warp] = v;
    if (threadIdx.x == 0)
        for (int k = 0; k < 3; ++k) {
            top3[b * 3 + k] = keys3[k];
            res->nn_idx[k] = keys3[k] == ~0ULL ? -1 : key_row(keys3[k]);
        }
}

// ... and after the SUM all-reduce: m_star_knn, w, s (features.py:275-290) from the summed squared distances
__global__ void shard_final_kernel(const unsigned long long *__restrict__ top3, const float *__restrict__ d2_sum, int dim, int B,
                                   TailResult *res_all) {
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    TailResult *res = res_all + b;
    float knn[2];
    for (int k = 0; k < 2; ++k) knn[k] = top3[b * 3 + 1 + k] == ~0ULL ? NAN : sqrtf(d2_sum[b * 2 + k]);
    reweight_final(res, res->s_star, knn[0], knn[1], dim);
}

// ---------------------------------------------------------------------------------------------------------------
// NCCL-free exchanges of a sharded round over peer-mapped memory (CUDA IPC / NVLink, cmdb_comm): the collective is fused
// into the kernels on both sides of it.
//   push   every rank packs its local (min distance, global row) keys and stores them straight into the round's slot
//          [slot][rank][query] of EVERY rank's buffer (coalesced 8-byte NVLink stores); the last block to finish raises
//          the rank's flag (the round's epoch) in every buffer: threadfence_system by all writers, then a release store
//   reduce every rank waits for the world flags in its LOCAL buffer, takes the MIN over the world key arrays (non-negative
//          distance bits << 32 | global row: integer MIN == argmin with lowest-row tie-break) and decodes min_val / min_idx /
//          the per-image argmax key -- what ncclAllReduce(MIN) + unpack did in two launches and ~60 us at 8 ranks.
// Slots alternate by round parity; a rank can be at most one round ahead of the slowest rank (it needs everybody's flag
// of round r + 1 before it can finish that round), so a slot is never overwritten while someone still reads it.
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void st_release_sys_u64(unsigned long long *p, unsigned long long v) {
    asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys_u64(const unsigned long long *p) {
    unsigned long long v;
    asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}

__global__ void __launch_bounds__(256) shard_push_keys_kernel(const float *__restrict__ min_val, const long long *__restrict__ min_idx,
                                                              int n, PeerPtrs peers, int world, int rank, size_t keys_off,
                                                              size_t flag_off, unsigned long long epoch, unsigned int *ctr) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const long long key = exchange_key(min_val[i], min_idx[i]);
        for (int r = 0; r < world; ++r)
            reinterpret_cast<long long *>(peers.p[r] + keys_off)[(size_t)rank * kShardKeysCap + i] = key;
    }
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        if (atomicAdd(ctr, 1u) == gridDim.x - 1) {   // every block's stores are fenced: publish
            __threadfence_system();
            *ctr = 0u;
            for (int r = 0; r < world; ++r)
                st_release_sys_u64(reinterpret_cast<unsigned long long *>(peers.p[r] + flag_off) + rank, epoch);
        }
    }
}

// returns false on timeout (a peer never arrived): the abort word is set and the caller's results are invalid
__device__ __forceinline__ bool wait_flags(const unsigned char *local, size_t flag_off, int world, unsigned long long epoch,
                                           unsigned int *abort_word) {
    __shared__ int ok_sh;
    if (threadIdx.x == 0) ok_sh = 1;
    __syncthreads();
    if (threadIdx.x < world) {
        const unsigned long long *f = reinterpret_cast<const unsigned long long *>(local + flag_off) + threadIdx.x;
        const long long t0 = clock64();
        while (ld_acquire_sys_u64(f) < epoch) {
            if (clock64() - t0 > 40LL * 1000 * 1000 * 1000) {  // ~20 s
                ok_sh = 0;
                *abort_word = 1u;
                break;
            }
        }
    }
    __syncthreads();
    return ok_sh != 0;
}

__global__ void __launch_bounds__(256) shard_reduce_keys_kernel(const unsigned char *__restrict__ local, size_t keys_off,
                                                                size_t flag_off, int world, unsigned long long epoch, int n,
                                                                int P_img, float *__restrict__ min_val,
                                                                long long *__restrict__ min_idx, unsigned long long *s_key,
                                                                unsigned int *abort_word) {
    if (!wait_flags(local, flag_off, world, epoch, abort_word)) return;
    const long long *keys = reinterpret_cast<const long long *>(local + keys_off);
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        long long k = 0x7fffffffffffffffLL;
        for (int r = 0; r < world; ++r) {
            const long long v = __ldcg(keys + (size_t)r * kShardKeysCap + i);
            k = v < k ? v : k;
        }
        const float v = key_value((unsigned long long)k);
        min_val[i] = v;
        min_idx[i] = key_row((unsigned long long)k);
        argmax_publish(s_key, i, P_img, v);
    }
}

// the second exchange: 2 squared neighbour distances per image, one non-zero contribution among the ranks
__global__ void __launch_bounds__(64) shard_push_d2_kernel(const float *__restrict__ contrib, int n, PeerPtrs peers, int world, int rank,
                                                          size_t d2_off, size_t flag_off, unsigned long long epoch) {
    for (int i = threadIdx.x; i < n; i += blockDim.x)
        for (int r = 0; r < world; ++r) reinterpret_cast<float *>(peers.p[r] + d2_off)[rank * kShardD2Cap + i] = contrib[i];
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0)
        for (int r = 0; r < world; ++r) st_release_sys_u64(reinterpret_cast<unsigned long long *>(peers.p[r] + flag_off) + rank, epoch);
}

__global__ void __launch_bounds__(64) shard_sum_d2_kernel(const unsigned char *__restrict__ local, size_t d2_off, size_t flag_off,
                                                         int world, unsigned long long epoch, int n, float *__restrict__ d2_sum,
                                                         unsigned int *abort_word) {
    if (!wait_flags(local, flag_off, world, epoch, abort_word)) return;
    const float *d = reinterpret_cast<const float *>(local + d2_off);
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        float acc = 0.f;  // one owner contributes the value, the others 0: x + 0 + ... + 0 is exact in any order
        for (int r = 0; r < world; ++r) acc += __ldcg(d + r * kShardD2Cap + i);
        d2_sum[i] = acc;
    }
}

static size_t shard_flag_off(int slot, int kind) { return kCommScoreFlagsOff + (size_t)((slot * 2 + kind) * kMaxRanks) * 8; }
static_assert(kCommScoreFlagsOff + kShardSlots * 2 * kMaxRanks * 8 <= kCommScoreD2Off, "flags overlap the d2 slots");
static_assert(kCommScoreD2Off + (size_t)kShardSlots * kMaxRanks * kShardD2Cap * 4 <= kCommScoreKeysOff, "d2 slots overlap the key slots");
static_assert(kCommScoreKeysOff + (size_t)kShardSlots * kMaxRanks * kShardKeysCap * 8 <= kCommHeaderBytes, "key slots exceed the header");

int score_shard_exchange_keys(const ScoreCall &c, int B, int P_img, const PeerPtrs &peers, int world, int rank, int slot,
                              unsigned long long epoch) {
    const cmdb_bank *b = c.b;
    cudaStream_t st = c.stream;
    const int n = B * P_img;
    CMDB_REQUIRE(n <= kShardKeysCap, CMDB_ERR_UNSUPPORTED, "sharded round: %d queries exceed the exchange slot (%d)", n, kShardKeysCap);
    const size_t keys_off = kCommScoreKeysOff + (size_t)slot * kMaxRanks * kShardKeysCap * 8;
    const int blocks = std::min((n + 255) / 256, 2 * b->num_sms);
    shard_push_keys_kernel<<<blocks, 256, 0, st>>>(c.min_val, c.min_idx, n, peers, world, rank, keys_off, shard_flag_off(slot, 0), epoch,
                                                   b->shard_ctr + (slot & 1));  // consecutive rounds (= the two lanes) use different counters
    CMDB_CUDA(cudaMemsetAsync(c.lane->s_key, 0, sizeof(unsigned long long) * B, st));
    shard_reduce_keys_kernel<<<blocks, 256, 0, st>>>(peers.p[rank], keys_off, shard_flag_off(slot, 0), world, epoch, n, P_img, c.min_val,
                                                     c.min_idx, c.lane->s_key, b->shard_abort_dev);
    CMDB_CUDA(cudaGetLastError());
    return CMDB_OK;
}

int score_shard_exchange_d2(const ScoreCall &c, int B, const PeerPtrs &peers, int world, int rank, int slot,
                            unsigned long long epoch, const float *contrib_dev, float *d2_sum_dev) {
    const cmdb_bank *b = c.b;
    cudaStream_t st = c.stream;
    CMDB_REQUIRE(2 * B <= kShardD2Cap, CMDB_ERR_UNSUPPORTED, "sharded round: batch %d exceeds the exchange slot", B);
    const size_t d2_off = kCommScoreD2Off + (size_t)slot * kMaxRanks * kShardD2Cap * 4;
    shard_push_d2_kernel<<<1, 64, 0, st>>>(contrib_dev, 2 * B, peers, world, rank, d2_off, shard_flag_off(slot, 1), epoch);
    shard_sum_d2_kernel<<<1, 64, 0, st>>>(peers.p[rank], d2_off, shard_flag_off(slot, 1), world, epoch, 2 * B, d2_sum_dev, b->shard_abort_dev);
    CMDB_CUDA(cudaGetLastError());
    return CMDB_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// upsample + blur in two small multi-CTA kernels (the image is split into 16 row bands, then 16 column bands):
//   K0  every CTA takes the max of its row band of the upsampled map (the global max is needed before the 8-bit
//       quantisation; round 1 recomputed all 50k pixels in every CTA of K1, which was two thirds of K1's time);
//   K1  folds the 16 band maxima, upsamples + quantises its row band and runs the 3 horizontal box passes in shared memory;
//   K2  every CTA loads its column band of K1's result and runs the 3 vertical passes (Pillow transposes instead), then
//       applies ToTensor (/255) and * max.
// ---------------------------------------------------------------------------------------------------------------
constexpr int kBlurThreads = 512;
constexpr int kBlurBands = 16;

__device__ __forceinline__ void bilinear_coeff(int dst, float scale, int n_in, int &i0, int &i1, float &w0, float &w1) {
    // ATen area_pixel_compute_source_index (align_corners=False) + HelperInterpLinear weights
    float real = fmaxf(__fsub_rn(__fmul_rn(scale, (float)dst + 0.5f), 0.5f), 0.f);
    i0 = (int)real;
    i1 = min(i0 + 1, n_in - 1);
    w1 = __fsub_rn(real, (float)i0);
    w0 = __fsub_rn(1.f, w1);
}

__device__ __forceinline__ float bilinear_at(const float *__restrict__ in_s, int fh, int fw_, float sh, float sw, int y, int x) {
    int y0, y1, x0, x1;
    float wy0, wy1, wx0, wx1;
    bilinear_coeff(y, sh, fh, y0, y1, wy0, wy1);
    bilinear_coeff(x, sw, fw_, x0, x1, wx0, wx1);
    // ATen Interpolate<2,...,interp_size 2>: t0*w0 + t1*w1 contracted as fma(t0, w0, t1*w1), W inside H
    const float t0 = __fmaf_rn(in_s[y0 * fw_ + x0], wx0, __fmul_rn(in_s[y0 * fw_ + x1], wx1));
    const float t1 = __fmaf_rn(in_s[y1 * fw_ + x0], wx0, __fmul_rn(in_s[y1 * fw_ + x1], wx1));
    return __fmaf_rn(t0, wy0, __fmul_rn(t1, wy1));
}

// one box pass along the `n`-long axis of an [n_lines][n] (x_stride == 1) or [n][n_lines] (x_stride == n_lines) tile;
// Pillow ImagingLineBoxBlur8 as a clamped 9-tap integer FIR with 32-bit fixed-point weights
__device__ __forceinline__ void box_pass(const unsigned char *__restrict__ src, unsigned char *__restrict__ dst, int n_lines,
                                         int n, int line_stride, int x_stride, int radius, unsigned int ww, unsigned int fw) {
    for (int i = threadIdx.x; i < n_lines * n; i += kBlurThreads) {
        // consecutive threads walk the contiguous tile dimension in both orientations (bank-conflict free)
        int line, x;
        if (x_stride == 1) line = i / n, x = i - line * n;
        else x = i / n_lines, line = i - x * n_lines;
        const unsigned char *ln = src + line * line_stride;
        unsigned int acc = 0;
        for (int k = -radius; k <= radius; ++k) acc += ln[min(max(x + k, 0), n - 1) * x_stride];
        const unsigned int far = ln[max(x - radius - 1, 0) * x_stride] + ln[min(x + radius + 1, n - 1) * x_stride];
        const unsigned int bulk = acc * ww + far * fw;
        dst[line * line_stride + x * x_stride] = (unsigned char)((bulk + (1u << 23)) >> 24);
    }
}

constexpr int kMaxThreads = 256;
__global__ void __launch_bounds__(kMaxThreads) upsample_max_kernel(const float *__restrict__ map_in, int fh, int fw_, int out_hw,
                                                                   int band, float *__restrict__ mx_part, int img_first, int img_step) {
    extern __shared__ __align__(16) unsigned char sm[];
    const size_t img = img_first + (size_t)blockIdx.y * img_step;
    map_in += img * fh * fw_;
    float *in_s = reinterpret_cast<float *>(sm);
    __shared__ float red[kMaxThreads / 32];
    // only the input rows this band interpolates from
    const float sh = (float)fh / (float)out_hw, sw = (float)fw_ / (float)out_hw;
    const int y0 = blockIdx.x * band, rows = min(band, out_hw - y0);
    float mx = -INFINITY;  // fmaxf ignores NaN and is order independent: the fold of the band maxima equals one global pass
    if (rows > 0) {
        int r_lo, r_hi, t0, t1;
        float w0, w1;
        bilinear_coeff(y0, sh, fh, r_lo, t1, w0, w1);
        bilinear_coeff(y0 + rows - 1, sh, fh, t0, r_hi, w0, w1);
        for (int i = threadIdx.x + r_lo * fw_; i < (r_hi + 1) * fw_; i += kMaxThreads) in_s[i] = map_in[i];
        __syncthreads();
        for (int i = threadIdx.x; i < rows * out_hw; i += kMaxThreads)
            mx = fmaxf(mx, bilinear_at(in_s, fh, fw_, sh, sw, y0 + i / out_hw, i % out_hw));
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
    __syncthreads();
    if (threadIdx.x == 0) {
#pragma unroll
        for (int w = 1; w < kMaxThreads / 32; ++w) mx = fmaxf(mx, red[w]);
        mx_part[img * kBlurBands + blockIdx.x] = mx;
    }
}

__global__ void __launch_bounds__(kBlurThreads) upsample_hblur_kernel(const float *__restrict__ map_in, int fh, int fw_,
                                                                      int out_hw, int band, float *__restrict__ pre,
                                                                      unsigned char *__restrict__ u8_out,
                                                                      unsigned char *__restrict__ tmp, float *__restrict__ mx_out,
                                                                      const float *__restrict__ mx_part,
                                                                      int radius, unsigned int ww, unsigned int fwt, int img_first,
                                                                      int img_step, size_t map_stride) {
    extern __shared__ __align__(16) unsigned char sm[];
    {  // image of the batch handled by this CTA
        const size_t img = img_first + (size_t)blockIdx.y * img_step;
        map_in += img * fh * fw_, tmp += img * map_stride, mx_out += img, mx_part += img * kBlurBands;
        if (pre) pre += img * map_stride;
        if (u8_out) u8_out += img * map_stride;
    }
    float *in_s = reinterpret_cast<float *>(sm);                    // [fh*fw]
    unsigned char *A = sm + sizeof(float) * ((fh * fw_ + 3) & ~3);  // [band][out_hw]
    unsigned char *B = A + ((band * out_hw + 15) & ~15);
    for (int i = threadIdx.x; i < fh * fw_; i += kBlurThreads) in_s[i] = map_in[i];
    __syncthreads();
    const float sh = (float)fh / (float)out_hw, sw = (float)fw_ / (float)out_hw;
    float mx = mx_part[0];  // map_max = img.max() over the WHOLE upsampled image (utils/utils.py:81): fold of K0's band maxima
#pragma unroll
    for (int w = 1; w < kBlurBands; ++w) mx = fmaxf(mx, mx_part[w]);
    if (blockIdx.x == 0 && threadIdx.x == 0) *mx_out = mx;
    const int y0 = blockIdx.x * band, rows = min(band, out_hw - y0);
    if (rows <= 0) return;
    // KNNGaussianBlur: img / max -> ToPILImage: mul(255).byte() (truncation)
    for (int i = threadIdx.x; i < rows * out_hw; i += kBlurThreads) {
        const int y = y0 + i / out_hw, x = i % out_hw;
        const float v = bilinear_at(in_s, fh, fw_, sh, sw, y, x);
        if (pre) pre[y * out_hw + x] = v;
        const unsigned char u = (unsigned char)(int)__fmul_rn(__fdiv_rn(v, mx), 255.f);
        A[i] = u;
        if (u8_out) u8_out[y * out_hw + x] = u;
    }
    __syncthreads();
    box_pass(A, B, rows, out_hw, out_hw, 1, radius, ww, fwt);
    __syncthreads();
    box_pass(B, A, rows, out_hw, out_hw, 1, radius, ww, fwt);
    __syncthreads();
    box_pass(A, B, rows, out_hw, out_hw, 1, radius, ww, fwt);
    __syncthreads();
    for (int i = threadIdx.x; i < rows * out_hw; i += kBlurThreads) tmp[y0 * out_hw + i] = B[i];
}

__global__ void __launch_bounds__(kBlurThreads) vblur_kernel(const unsigned char *__restrict__ tmp, int out_hw, int band,
                                                             const float *__restrict__ mx_in, float *__restrict__ out,
                                                             int radius, unsigned int ww, unsigned int fwt, int img_first,
                                                             int img_step, size_t map_stride) {
    extern __shared__ __align__(16) unsigned char sm[];
    {
        const size_t img = img_first + (size_t)blockIdx.y * img_step;
        tmp += img * map_stride, out += img * map_stride, mx_in += img;
    }
    const int x0 = blockIdx.x * band, cols = min(band, out_hw - x0);
    if (cols <= 0) return;
    unsigned char *A = sm;  // [out_hw][cols]: column band, lines = columns (stride 1), pass axis = rows (stride cols)
    unsigned char *B = A + ((out_hw * band + 15) & ~15);
    for (int i = threadIdx.x; i < out_hw * cols; i += kBlurThreads) {
        const int y = i / cols, c = i - y * cols;
        A[i] = tmp[y * out_hw + x0 + c];
    }
    __syncthreads();
    box_pass(A, B, cols, out_hw, 1, cols, radius, ww, fwt);
    __syncthreads();
    box_pass(B, A, cols, out_hw, 1, cols, radius, ww, fwt);
    __syncthreads();
    box_pass(A, B, cols, out_hw, 1, cols, radius, ww, fwt);
    __syncthreads();
    const float mx = *mx_in;
    // ToTensor (/255) then * map_max
    for (int i = threadIdx.x; i < out_hw * cols; i += kBlurThreads) {
        const int y = i / cols, c = i - y * cols;
        out[y * out_hw + x0 + c] = __fmul_rn(__fdiv_rn((float)B[i], 255.f), mx);
    }
}

int score_select(const ScoreCall &c, int B, int P_img, bool local_m_star) {
    const cmdb_bank *b = c.b;
    const Lane &l = *c.lane;
    select_kernel<<<B, 256, 0, c.stream>>>(l.s_key, c.min_idx, P_img, c.slot->q_f32, b->data, b->dim, b->row_offset, b->fin_rows,
                                           l.m_test, local_m_star ? l.m_star : nullptr, c.tail);
    CMDB_CUDA(cudaGetLastError());
    return CMDB_OK;
}

// reweight_cert_kernel over the n m_star rows of the GEMM launch `sched` on the call's lane, one block per row: the three
// nearest rows as keys into top3 and, with res, the final re-weighting (m_test, s_key) into res
static int launch_reweight_cert(const ScoreCall &c, const GemmSched &sched, int n, const float *m_star, long long row_offset,
                                unsigned long long *top3, TailResult *res) {
    const cmdb_bank *b = c.b;
    const Lane &s = *c.lane;
    CMDB_REQUIRE(!sched.pair, CMDB_ERR_UNSUPPORTED, "scoring: the re-weighting certificate cannot walk a CTA-pair GEMM schedule");
    CMDB_REQUIRE(sched.producers <= 320, CMDB_ERR_UNSUPPORTED, "scoring: %d GEMM producers exceed reweight_cert_kernel's limit",
                 sched.producers);
    ReweightCertParams p{};
    p.cand = s.cand, p.n_cand = sched.producers, p.cand_stride = b->layout.cap_p;
    p.m_star = m_star, p.m_test = res ? s.m_test : nullptr, p.bank = b->data, p.rows = b->fin_rows, p.row_offset = row_offset;
    p.dim = b->dim, p.q_norm = s.q_norm, p.q_eps = s.q_eps;
    p.bmax = b->cert_bmax, p.eb_max = b->cert_eb_max, p.acc_model = cert_acc_model(b->dim);
    p.sched = sched;
    p.s_key = res ? s.s_key : nullptr, p.top3 = top3, p.res = res;
    reweight_cert_kernel<<<n, 256, 0, c.stream>>>(p);
    CMDB_CUDA(cudaGetLastError());
    return CMDB_OK;
}

// tensor-core variant: select -> fp16 split of the m_star rows -> hi.hi GEMM with one M tile -> reweight_cert_kernel
static int score_reweight_tensor(const ScoreCall &c, int B, int P_img) {
    const Lane &s = *c.lane;
    CMDB_CHECK(score_select(c, B, P_img, true));  // m_test, m_star, s*, s_idx, m_star_row
    // the min/argmin phase is complete: its query operand buffers and candidate lists are free again
    q_split_rows(c, s.m_star, B);
    CMDB_CUDA(cudaGetLastError());
    GemmSched sched{};
    CMDB_CHECK(score_gemm_candidates(c, c.stream, B, 1, false, &sched));
    return launch_reweight_cert(c, sched, B, s.m_star, c.b->row_offset, s.top3, c.tail);
}

// SURVEY 8f-1: three nearest bank rows of every bank row.  The bank is its own query set: chunks of rows go through the
// fp16 split, the certified pre-filter GEMM and reweight_cert_kernel (one block per row, keys only).
int score_build_knn_table(cmdb_bank *b, long long row_first, long long row_count) {
    const int chunk = 64 * kScoreBM;  // 8192 rows: 64 M tiles per GEMM launch
    // scratch for `chunk` query rows; sized like a 32-image batch so that later scoring calls do not have to grow it
    const size_t map_stride = b->layout.map_stride;
    CMDB_CHECK(score_scratch_alloc(b, 32, chunk / 32, map_stride ? (int)lround(sqrt((double)map_stride)) : 224));
    const ScoreCall c = score_call(b, 0, 0);   // lane 0; the result slot is not used
    cudaStream_t st = c.stream;
    if (!b->knn_table || b->knn_rows != b->fin_rows) {
        cudaFree(b->knn_table);
        b->knn_table = nullptr;
        CMDB_CUDA(cudaMalloc(&b->knn_table, sizeof(unsigned long long) * 3 * (size_t)b->fin_rows));
        CMDB_CUDA(cudaMemsetAsync(b->knn_table, 0xff, sizeof(unsigned long long) * 3 * (size_t)b->fin_rows, st));
        b->knn_rows = b->fin_rows;
    }
    const long long row_end = row_first + row_count;
    for (long long r0 = row_first; r0 < row_end; r0 += chunk) {
        const int n = (int)std::min<long long>(chunk, row_end - r0);
        const float *rows = b->data + (size_t)r0 * b->dim;
        q_split_rows(c, rows, n);
        CMDB_CUDA(cudaGetLastError());
        GemmSched sched{};
        CMDB_CHECK(score_gemm_candidates(c, st, n, 1, false, &sched));
        CMDB_CHECK(launch_reweight_cert(c, sched, n, rows, 0, b->knn_table + (size_t)r0 * 3, nullptr));
    }
    CMDB_CUDA(cudaStreamSynchronize(st));
    return CMDB_OK;
}

int score_reweight(const ScoreCall &c, int B, int P_img) {
    const cmdb_bank *b = c.b;
    const Lane &l = *c.lane;
    if (b->knn_table && b->row_offset == 0 && b->knn_rows == b->fin_rows) {  // the bank's neighbour table: the w_dist pass is a lookup
        CMDB_CHECK(score_select(c, B, P_img, true));
        reweight_lookup_kernel<<<B, 64, 0, c.stream>>>(b->knn_table, l.m_test, b->data, b->dim, l.s_key, l.top3, c.tail);
        CMDB_CUDA(cudaGetLastError());
        return CMDB_OK;
    }
    // a single image: the one-launch CUDA-core sweep is as fast as a one-tile GEMM over the whole bank; batches go to the
    // tensor cores, whose cost does not grow with B (identical keys either way).
    if (b->score_impl == CMDB_SCORE_TCGEN05 && b->prefilter_terms == 0 && B >= 2 && B <= kScoreBM)
        return score_reweight_tensor(c, B, P_img);
    ReweightParams p{};
    p.bank = b->data, p.rows = b->fin_rows, p.row_offset = b->row_offset, p.dim = b->dim, p.B = B, p.P_img = P_img;
    p.q = c.slot->q_f32, p.s_key = l.s_key, p.min_idx = c.min_idx;
    p.block_keys = l.topk_keys, p.top3 = l.top3, p.done_counter = l.done_counter;
    p.res = c.tail;
    const size_t smem = sizeof(float) * (size_t)B * b->dim + sizeof(unsigned long long) * 8 * B * 3;
    const int blocks = b->layout.n_topk_blocks;
#define CMDB_RW(DVV)                                                                                              \
    case DVV:                                                                                                     \
        CMDB_CUDA(cudaFuncSetAttribute(reweight_kernel<DVV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)); \
        reweight_kernel<DVV><<<blocks, 256, smem, c.stream>>>(p);                                                 \
        break;
    switch ((b->dim / 4 + 31) / 32) {
        CMDB_RW(1) CMDB_RW(2) CMDB_RW(3) CMDB_RW(4) CMDB_RW(5) CMDB_RW(6) CMDB_RW(7) CMDB_RW(8) CMDB_RW(9) CMDB_RW(10)
        CMDB_RW(11) CMDB_RW(12) CMDB_RW(13) CMDB_RW(14) CMDB_RW(15) CMDB_RW(16)
        default:
            set_error("scoring: dim=%d exceeds the supported 2048", b->dim);
            return CMDB_ERR_UNSUPPORTED;
    }
#undef CMDB_RW
    CMDB_CUDA(cudaGetLastError());
    return CMDB_OK;
}

int score_shard_lookup(const ScoreCall &c, int B, float *contrib_dev) {
    const cmdb_bank *b = c.b;
    shard_lookup_kernel<<<B, 64, 0, c.stream>>>(b->knn_table, c.lane->m_test, b->data, b->fin_rows, b->row_offset, b->dim,
                                                c.lane->top3, c.tail, contrib_dev);
    CMDB_CUDA(cudaGetLastError());
    return CMDB_OK;
}

int score_shard_final(const ScoreCall &c, int B, const float *d2_sum_dev) {
    shard_final_kernel<<<1, 64, 0, c.stream>>>(c.lane->top3, d2_sum_dev, c.b->dim, B, c.tail);
    CMDB_CUDA(cudaGetLastError());
    return CMDB_OK;
}

void tail_prefer_carveout() {
    CMDB_PREFER_MAX_SMEM(refine_kernel);
    CMDB_PREFER_MAX_SMEM(refine_cert_kernel<8>);
    CMDB_PREFER_MAX_SMEM(rescan_kernel);
    CMDB_PREFER_MAX_SMEM(select_kernel);
    CMDB_PREFER_MAX_SMEM(reweight_cert_kernel);
    CMDB_PREFER_MAX_SMEM(reweight_lookup_kernel);
    CMDB_PREFER_MAX_SMEM(shard_lookup_kernel);
    CMDB_PREFER_MAX_SMEM(shard_final_kernel);
    CMDB_PREFER_MAX_SMEM(shard_push_keys_kernel);
    CMDB_PREFER_MAX_SMEM(shard_reduce_keys_kernel);
    CMDB_PREFER_MAX_SMEM(shard_push_d2_kernel);
    CMDB_PREFER_MAX_SMEM(shard_sum_d2_kernel);
    CMDB_PREFER_MAX_SMEM(upsample_max_kernel);
    CMDB_PREFER_MAX_SMEM(upsample_hblur_kernel);
    CMDB_PREFER_MAX_SMEM(vblur_kernel);
    (void)cudaGetLastError();
}

// images img_first, img_first + img_step, ... (n_img of them); per-image stride of the map buffers = map_stride pixels
int upsample_blur_launch(cudaStream_t stream, int n_img, int img_first, int img_step, size_t map_stride, const float *map_dev,
                         int fh, int fw, int out_hw, float *pre_dev, float *out_dev, unsigned char *u8_dev,
                         unsigned char *tmp_dev, float *mx_dev, float *mx_part_dev) {
    if (n_img <= 0) return CMDB_OK;
    CMDB_REQUIRE(fh > 0 && fw > 0 && out_hw >= 8 && out_hw <= 256, CMDB_ERR_INVALID,
                 "upsample_blur: need out_hw in [8,256] (got %d) and positive map dims", out_hw);
    // Pillow _gaussian_blur_radius(radius=4, passes=3) evaluated like BoxBlur.c (float sigma2 = 16/3, the rest double)
    const float sigma2 = 4.f * 4.f / 3.f;
    const double L = sqrt(12.0 * (double)sigma2 + 1.0);
    const double l = floor((L - 1.0) / 2.0);
    double a = (2 * l + 1) * (l * (l + 1) - 3 * (double)sigma2);
    a /= 6 * ((double)sigma2 - (l + 1) * (l + 1));
    const float fr = (float)(l + a);
    const int radius = (int)fr;
    const unsigned int ww = (unsigned int)((float)(1 << 24) / (fr * 2 + 1));
    const unsigned int fwt = ((1u << 24) - (unsigned int)(radius * 2 + 1) * ww) / 2;
    CMDB_REQUIRE(out_hw > radius + 1, CMDB_ERR_INVALID, "upsample_blur: image smaller than the blur radius");
    const int band = (out_hw + kBlurBands - 1) / kBlurBands;
    const size_t tile = (size_t)((band * out_hw + 15) & ~15);
    const size_t smem1 = sizeof(float) * ((fh * fw + 3) & ~3) + 2 * tile;
    CMDB_REQUIRE(smem1 <= 200 * 1024, CMDB_ERR_UNSUPPORTED, "upsample_blur: map too large for shared memory");
    CMDB_CUDA(cudaFuncSetAttribute(upsample_hblur_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem1));
    CMDB_CUDA(cudaFuncSetAttribute(upsample_max_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(sizeof(float) * fh * fw)));
    upsample_max_kernel<<<dim3(kBlurBands, n_img), kMaxThreads, sizeof(float) * fh * fw, stream>>>(map_dev, fh, fw, out_hw, band,
                                                                                                   mx_part_dev, img_first, img_step);
    upsample_hblur_kernel<<<dim3(kBlurBands, n_img), kBlurThreads, smem1, stream>>>(
        map_dev, fh, fw, out_hw, band, pre_dev, u8_dev, tmp_dev, mx_dev, mx_part_dev, radius, ww, fwt, img_first, img_step, map_stride);
    vblur_kernel<<<dim3(kBlurBands, n_img), kBlurThreads, 2 * tile, stream>>>(tmp_dev, out_hw, band, mx_dev, out_dev, radius, ww,
                                                                             fwt, img_first, img_step, map_stride);
    CMDB_CUDA(cudaGetLastError());
    return CMDB_OK;
}

}  // namespace cmdb
