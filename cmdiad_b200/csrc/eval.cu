// Evaluation on the device-side result store (SURVEY 8f-3): what calculate_metrics (reference features.py:302-324) does
// with sklearn / numpy on 50 176 Python scalars per image, computed where the fused maps already are.
//
//   pixel AUROC  roc_auc_score(pixel_labels, pixel_preds) == U / (n_pos * n_neg) with the Mann-Whitney U statistic
//                (ties count one half): returned as the exact integer 2U, the host does one division;
//   AU-PRO       utils/au_pro_util.py:104-224: thresholds at equidistant ranks of the sorted anomaly-free scores, per
//                ground-truth component the number of its scores <= threshold.  Returned as exact integer counts; the
//                host turns them into the curve with the reference's own float64 operations (cmdiad_b200/metrics.py),
//                so the values are bit-identical to the reference.
//
// All of it hangs off ONE stable LSD radix sort of (score, label) pairs over all pixels of the test set -- HBM-bound
// integer work: 8 passes x (read 12 B + write 12 B) per pixel.  Every warp owns a contiguous slice of the input, counts
// its digits (warp match), a single-block scan turns the digit-major [256][warps] table into output offsets, and the
// same warp scatters its slice in order, which keeps the sort stable without any local sorting.
// Connected components of the masks are labelled on the host (scipy.ndimage.label, exactly as the reference: the masks
// are host inputs of predict()); labels travel as one int32 per pixel.
#include <vector>

#include "common.cuh"

namespace cmdb {

constexpr int kSortThreads = 256;
constexpr int kSortWarps = kSortThreads / 32;

__device__ __forceinline__ unsigned long long order_key(double v) {  // monotone double -> uint64
    const unsigned long long b = (unsigned long long)__double_as_longlong(v);
    return (b >> 63) ? ~b : (b | 0x8000000000000000ULL);
}
__device__ __forceinline__ double key_to_double(unsigned long long k) {
    const unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffULL) : ~k;
    return __longlong_as_double((long long)b);
}

__global__ void __launch_bounds__(256) eval_make_keys_kernel(const double *__restrict__ scores, long long n,
                                                             unsigned long long *__restrict__ keys) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        keys[i] = order_key(scores[i]);
}

// slice of warp w: [w * per_warp, min(n, (w + 1) * per_warp)), per_warp a multiple of 32
__global__ void __launch_bounds__(kSortThreads) radix_hist_kernel(const unsigned long long *__restrict__ keys, long long n,
                                                                  long long per_warp, int shift, unsigned int *__restrict__ hist,
                                                                  int n_warps_total) {
    __shared__ unsigned int cnt[kSortWarps][256];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    for (int i = lane; i < 256; i += 32) cnt[warp][i] = 0;
    __syncwarp();
    const long long w = (long long)blockIdx.x * kSortWarps + warp;
    const long long lo = w * per_warp, hi = min(n, lo + per_warp);
    for (long long base = lo; base < hi; base += 32) {
        const long long i = base + lane;
        const bool valid = i < hi;
        const unsigned int active = __ballot_sync(0xffffffffu, valid);
        if (valid) {
            const unsigned int d = (unsigned int)(keys[i] >> shift) & 255u;
            const unsigned int m = __match_any_sync(active, d);
            if (lane == __ffs(m) - 1) cnt[warp][d] += __popc(m);
        }
        __syncwarp();
    }
    __syncwarp();
    if (w < n_warps_total)
        for (int i = lane; i < 256; i += 32) hist[(size_t)i * n_warps_total + w] = cnt[warp][i];
}

// exclusive scan of `count` unsigned ints in place, one block
__global__ void __launch_bounds__(1024) scan_u32_kernel(unsigned int *__restrict__ a, long long count) {
    __shared__ unsigned long long part[1024];
    const long long per = (count + 1023) / 1024;
    const long long lo = min(count, (long long)threadIdx.x * per), hi = min(count, lo + per);
    unsigned long long s = 0;
    for (long long i = lo; i < hi; ++i) s += a[i];
    part[threadIdx.x] = s;
    __syncthreads();
    for (int off = 1; off < 1024; off <<= 1) {  // Hillis-Steele inclusive scan of the 1024 partial sums
        unsigned long long v = threadIdx.x >= off ? part[threadIdx.x - off] : 0ULL;
        __syncthreads();
        part[threadIdx.x] += v;
        __syncthreads();
    }
    unsigned long long run = threadIdx.x ? part[threadIdx.x - 1] : 0ULL;
    for (long long i = lo; i < hi; ++i) {
        const unsigned int v = a[i];
        a[i] = (unsigned int)run;
        run += v;
    }
}

__global__ void __launch_bounds__(kSortThreads) radix_scatter_kernel(const unsigned long long *__restrict__ keys,
                                                                     const unsigned int *__restrict__ vals, long long n,
                                                                     long long per_warp, int shift,
                                                                     const unsigned int *__restrict__ offs, int n_warps_total,
                                                                     unsigned long long *__restrict__ keys_out,
                                                                     unsigned int *__restrict__ vals_out) {
    __shared__ unsigned int off[kSortWarps][256];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long long w = (long long)blockIdx.x * kSortWarps + warp;
    if (w >= n_warps_total) return;
    for (int i = lane; i < 256; i += 32) off[warp][i] = offs[(size_t)i * n_warps_total + w];
    __syncwarp();
    const long long lo = w * per_warp, hi = min(n, lo + per_warp);
    for (long long base = lo; base < hi; base += 32) {
        const long long i = base + lane;
        const bool valid = i < hi;
        const unsigned int active = __ballot_sync(0xffffffffu, valid);
        unsigned long long k = 0;
        unsigned int v = 0, d = 0, m = 0, dst = 0;
        if (valid) {
            k = keys[i], v = vals[i];
            d = (unsigned int)(k >> shift) & 255u;
            m = __match_any_sync(active, d);
            dst = off[warp][d] + __popc(m & ((1u << lane) - 1u));  // lanes in index order: stable
        }
        __syncwarp();
        if (valid) {
            keys_out[dst] = k, vals_out[dst] = v;
            if (lane == __ffs(m) - 1) off[warp][d] += __popc(m);
        }
        __syncwarp();
    }
}

// ---- exclusive prefix count of anomaly-free pixels (label == 0) over the sorted order: 3 kernels ----
constexpr int kScanTile = 4096;  // elements per block

__global__ void __launch_bounds__(256) neg_block_count_kernel(const unsigned int *__restrict__ labels, long long n,
                                                              unsigned int *__restrict__ block_cnt) {
    __shared__ unsigned int red[8];
    const long long lo = (long long)blockIdx.x * kScanTile;
    unsigned int c = 0;
    for (int j = threadIdx.x; j < kScanTile; j += 256)
        if (lo + j < n && labels[lo + j] == 0u) ++c;
    for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = c;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned int s = 0;
        for (int i = 0; i < 8; ++i) s += red[i];
        block_cnt[blockIdx.x] = s;
    }
}

__global__ void __launch_bounds__(256) neg_prefix_kernel(const unsigned int *__restrict__ labels, long long n,
                                                         const unsigned int *__restrict__ block_off,
                                                         unsigned int *__restrict__ negprefix) {
    // thread t owns 16 consecutive elements of the tile
    __shared__ unsigned int part[256];
    const long long lo = (long long)blockIdx.x * kScanTile + (long long)threadIdx.x * 16;
    unsigned int c = 0;
    for (int j = 0; j < 16; ++j)
        if (lo + j < n && labels[lo + j] == 0u) ++c;
    part[threadIdx.x] = c;
    __syncthreads();
    for (int off = 1; off < 256; off <<= 1) {
        unsigned int v = threadIdx.x >= off ? part[threadIdx.x - off] : 0u;
        __syncthreads();
        part[threadIdx.x] += v;
        __syncthreads();
    }
    unsigned int run = block_off[blockIdx.x] + (threadIdx.x ? part[threadIdx.x - 1] : 0u);
    for (int j = 0; j < 16; ++j)
        if (lo + j < n) {
            negprefix[lo + j] = run;
            if (labels[lo + j] == 0u) ++run;
        }
}

// thresholds: thr[t] = score of the anomaly-free pixel with rank pos[t] (au_pro_util.py:179-183); pos ascending
__global__ void __launch_bounds__(256) pick_thresholds_kernel(const unsigned long long *__restrict__ keys,
                                                              const unsigned int *__restrict__ labels,
                                                              const unsigned int *__restrict__ negprefix, long long n,
                                                              const long long *__restrict__ pos, int n_thr,
                                                              unsigned long long *__restrict__ thr_keys) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        if (labels[i] != 0u) continue;
        const long long r = negprefix[i];
        int a = 0, b = n_thr;  // first t with pos[t] >= r
        while (a < b) {
            const int mid = (a + b) >> 1;
            if (pos[mid] < r) a = mid + 1;
            else b = mid;
        }
        for (int t = a; t < n_thr && pos[t] == r; ++t) thr_keys[t] = keys[i];
    }
}

// per ground-truth component: histogram of "first threshold >= score" (bin n_thr = above every threshold), and
// the pixel AUROC's 2U = sum over anomalous pixels of #{ok < x} + #{ok <= x} (group bounds by binary search in the sorted keys)
__global__ void __launch_bounds__(256) eval_count_kernel(const unsigned long long *__restrict__ keys,
                                                         const unsigned int *__restrict__ labels,
                                                         const unsigned int *__restrict__ negprefix, long long n,
                                                         unsigned int n_neg, const unsigned long long *__restrict__ thr_keys,
                                                         int n_thr, unsigned long long *__restrict__ comp_hist,
                                                         unsigned long long *__restrict__ u2) {
    extern __shared__ unsigned long long thr_s[];
    for (int t = threadIdx.x; t < n_thr; t += blockDim.x) thr_s[t] = thr_keys[t];
    __syncthreads();
    unsigned long long acc = 0;
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
        const unsigned int lab = labels[i];
        if (lab == 0u) continue;
        const unsigned long long k = keys[i];
        int a = 0, b = n_thr;  // first t with thr[t] >= k  (the component pixel is "<= threshold" from there on)
        while (a < b) {
            const int mid = (a + b) >> 1;
            if (thr_s[mid] < k) a = mid + 1;
            else b = mid;
        }
        atomicAdd(comp_hist + (size_t)(lab - 1) * (n_thr + 1) + a, 1ULL);
        long long lo = 0, hi = i;  // first index with key == k
        while (lo < hi) {
            const long long mid = (lo + hi) >> 1;
            if (keys[mid] < k) lo = mid + 1;
            else hi = mid;
        }
        const long long gs = lo;
        lo = i + 1, hi = n;        // first index with key > k
        while (lo < hi) {
            const long long mid = (lo + hi) >> 1;
            if (keys[mid] <= k) lo = mid + 1;
            else hi = mid;
        }
        acc += (unsigned long long)negprefix[gs] + (unsigned long long)(lo < n ? negprefix[lo] : n_neg);
    }
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0 && acc) atomicAdd(u2, acc);
}

__global__ void keys_to_double_kernel(const unsigned long long *__restrict__ k, int n, double *__restrict__ out) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = key_to_double(k[i]);
}

}  // namespace cmdb

using namespace cmdb;

extern "C" {

// test hook (not in the public header): appends n_images maps of acc_npix float64 values to the device-side result store
// under the checks of the fused submit (store reserved, room for the images, no batch outstanding), so that the metrics
// can be driven with chosen values -- ties, sign mixes, 10 M-pixel stores -- instead of whatever scoring produces.  The
// image scores of the loaded images are set to 0.
int cmdb_debug_eval_load(cmdb_bank *b, const double *maps_host, int64_t n_images) {
    CMDB_REQUIRE(b && maps_host && n_images >= 1, CMDB_ERR_INVALID, "cmdb_debug_eval_load: bad arguments");
    cmdb_bank::Fused &f = b->fused;
    CMDB_REQUIRE(!f.active[0] && !f.active[1], CMDB_ERR_STATE, "cmdb_debug_eval_load: a submitted batch is outstanding");
    CMDB_REQUIRE(f.acc_maps && f.acc_n + n_images <= f.acc_cap, CMDB_ERR_CAPACITY,
                 "cmdb_debug_eval_load: device-side result store missing or full (%lld + %lld > %lld); call cmdb_eval_reserve",
                 f.acc_n, (long long)n_images, f.acc_cap);
    CMDB_CUDA(cudaSetDevice(b->device));
    CMDB_CUDA(cudaMemcpyAsync(f.acc_maps + (size_t)f.acc_n * f.acc_npix, maps_host, sizeof(double) * (size_t)n_images * f.acc_npix,
                              cudaMemcpyHostToDevice, b->handle_stream()));
    CMDB_CUDA(cudaMemsetAsync(f.acc_scores + f.acc_n, 0, sizeof(double) * (size_t)n_images, b->handle_stream()));
    CMDB_CUDA(cudaStreamSynchronize(b->handle_stream()));
    f.acc_n += n_images;
    return CMDB_OK;
}

int cmdb_eval_pixel_metrics(cmdb_bank *b, const int32_t *labels_host, int64_t n_components, const int64_t *ok_rank_pos_host,
                            int n_thresholds, double *out_thresholds, int64_t *out_component_le_counts,
                            int64_t *out_component_sizes, uint64_t *out_two_u, int64_t *out_n_pos, int64_t *out_n_neg) {
    CMDB_REQUIRE(b && labels_host && ok_rank_pos_host && out_thresholds && out_component_le_counts && out_component_sizes &&
                     out_two_u && out_n_pos && out_n_neg,
                 CMDB_ERR_INVALID, "cmdb_eval_pixel_metrics: NULL argument");
    cmdb_bank::Fused &f = b->fused;
    CMDB_REQUIRE(f.acc_n > 0 && f.acc_maps, CMDB_ERR_STATE, "cmdb_eval_pixel_metrics: the device-side result store is empty");
    CMDB_REQUIRE(!f.active[0] && !f.active[1], CMDB_ERR_STATE, "cmdb_eval_pixel_metrics: a submitted batch is outstanding");
    CMDB_REQUIRE(n_components >= 0 && n_thresholds >= 1 && n_thresholds <= 4096, CMDB_ERR_INVALID,
                 "cmdb_eval_pixel_metrics: n_components=%lld / n_thresholds=%d out of range", (long long)n_components, n_thresholds);
    const long long n = f.acc_n * (long long)f.acc_npix;
    CMDB_REQUIRE(n < (1LL << 32), CMDB_ERR_UNSUPPORTED, "cmdb_eval_pixel_metrics: more than 2^32 pixels");
    long long n_neg = 0;
    for (long long i = 0; i < n; ++i) {
        CMDB_REQUIRE(labels_host[i] >= 0 && labels_host[i] <= n_components, CMDB_ERR_INVALID,
                     "cmdb_eval_pixel_metrics: label %d at pixel %lld outside [0, %lld]", labels_host[i], i, (long long)n_components);
        n_neg += labels_host[i] == 0;
    }
    for (int t = 0; t < n_thresholds; ++t)
        CMDB_REQUIRE(ok_rank_pos_host[t] >= 0 && ok_rank_pos_host[t] < n_neg && (t == 0 || ok_rank_pos_host[t] >= ok_rank_pos_host[t - 1]),
                     CMDB_ERR_INVALID, "cmdb_eval_pixel_metrics: threshold ranks must be ascending and inside [0, %lld)", n_neg);
    CMDB_CUDA(cudaSetDevice(b->device));
    cudaStream_t st = b->handle_stream();
    const int n_blocks = (int)std::min<long long>((n + kSortThreads * 32 - 1) / (kSortThreads * 32), (long long)b->num_sms * 8);
    const int n_warps = n_blocks * kSortWarps;
    const long long per_warp = ((n + n_warps - 1) / n_warps + 31) / 32 * 32;
    const int scan_blocks = (int)((n + kScanTile - 1) / kScanTile);
    const size_t hist_cols = (size_t)n_components * (n_thresholds + 1);
    unsigned long long *keys[2] = {nullptr, nullptr}, *thr_keys = nullptr, *comp_hist = nullptr, *u2 = nullptr;
    unsigned int *vals[2] = {nullptr, nullptr}, *hist = nullptr, *block_cnt = nullptr, *negprefix = nullptr;
    long long *pos_dev = nullptr;
    double *thr_dev = nullptr;
    int rc = CMDB_OK;
    auto cleanup = [&]() {
        cudaFree(keys[0]), cudaFree(keys[1]), cudaFree(vals[0]), cudaFree(vals[1]), cudaFree(hist), cudaFree(block_cnt);
        cudaFree(negprefix), cudaFree(thr_keys), cudaFree(comp_hist), cudaFree(u2), cudaFree(pos_dev), cudaFree(thr_dev);
    };
#define EV_TRY(expr)                                                                          \
    do {                                                                                      \
        cudaError_t _e = (expr);                                                              \
        if (_e != cudaSuccess) {                                                              \
            set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e));   \
            (void)cudaGetLastError();                                                         \
            cleanup();                                                                        \
            return CMDB_ERR_CUDA;                                                             \
        }                                                                                     \
    } while (0)
    for (int i = 0; i < 2; ++i) {
        EV_TRY(cudaMalloc(&keys[i], sizeof(unsigned long long) * (size_t)n));
        EV_TRY(cudaMalloc(&vals[i], sizeof(unsigned int) * (size_t)n));
    }
    EV_TRY(cudaMalloc(&hist, sizeof(unsigned int) * 256 * (size_t)n_warps));
    EV_TRY(cudaMalloc(&block_cnt, sizeof(unsigned int) * (size_t)(scan_blocks + 1)));
    EV_TRY(cudaMalloc(&negprefix, sizeof(unsigned int) * (size_t)n));
    EV_TRY(cudaMalloc(&thr_keys, sizeof(unsigned long long) * n_thresholds));
    EV_TRY(cudaMalloc(&thr_dev, sizeof(double) * n_thresholds));
    EV_TRY(cudaMalloc(&comp_hist, sizeof(unsigned long long) * std::max<size_t>(1, hist_cols)));
    EV_TRY(cudaMalloc(&u2, sizeof(unsigned long long)));
    EV_TRY(cudaMalloc(&pos_dev, sizeof(long long) * n_thresholds));
    EV_TRY(cudaMemsetAsync(comp_hist, 0, sizeof(unsigned long long) * std::max<size_t>(1, hist_cols), st));
    EV_TRY(cudaMemsetAsync(u2, 0, sizeof(unsigned long long), st));
    EV_TRY(cudaMemcpyAsync(vals[0], labels_host, sizeof(unsigned int) * (size_t)n, cudaMemcpyHostToDevice, st));
    EV_TRY(cudaMemcpyAsync(pos_dev, ok_rank_pos_host, sizeof(long long) * n_thresholds, cudaMemcpyHostToDevice, st));
    eval_make_keys_kernel<<<b->num_sms * 8, 256, 0, st>>>(f.acc_maps, n, keys[0]);
    EV_TRY(cudaGetLastError());
    int cur = 0;
    for (int pass = 0; pass < 8; ++pass) {  // stable LSD radix sort, 8 bits per pass
        radix_hist_kernel<<<n_blocks, kSortThreads, 0, st>>>(keys[cur], n, per_warp, 8 * pass, hist, n_warps);
        scan_u32_kernel<<<1, 1024, 0, st>>>(hist, 256LL * n_warps);
        radix_scatter_kernel<<<n_blocks, kSortThreads, 0, st>>>(keys[cur], vals[cur], n, per_warp, 8 * pass, hist, n_warps,
                                                                keys[cur ^ 1], vals[cur ^ 1]);
        EV_TRY(cudaGetLastError());
        cur ^= 1;
    }
    neg_block_count_kernel<<<scan_blocks, 256, 0, st>>>(vals[cur], n, block_cnt);
    scan_u32_kernel<<<1, 1024, 0, st>>>(block_cnt, scan_blocks);
    neg_prefix_kernel<<<scan_blocks, 256, 0, st>>>(vals[cur], n, block_cnt, negprefix);
    pick_thresholds_kernel<<<b->num_sms * 8, 256, 0, st>>>(keys[cur], vals[cur], negprefix, n, pos_dev, n_thresholds, thr_keys);
    eval_count_kernel<<<b->num_sms * 8, 256, sizeof(unsigned long long) * n_thresholds, st>>>(
        keys[cur], vals[cur], negprefix, n, (unsigned int)n_neg, thr_keys, n_thresholds, comp_hist, u2);
    keys_to_double_kernel<<<(n_thresholds + 255) / 256, 256, 0, st>>>(thr_keys, n_thresholds, thr_dev);
    EV_TRY(cudaGetLastError());
    std::vector<unsigned long long> h_hist(std::max<size_t>(1, hist_cols));
    unsigned long long h_u2 = 0;
    EV_TRY(cudaMemcpyAsync(h_hist.data(), comp_hist, sizeof(unsigned long long) * std::max<size_t>(1, hist_cols), cudaMemcpyDeviceToHost, st));
    EV_TRY(cudaMemcpyAsync(&h_u2, u2, sizeof(h_u2), cudaMemcpyDeviceToHost, st));
    EV_TRY(cudaMemcpyAsync(out_thresholds, thr_dev, sizeof(double) * n_thresholds, cudaMemcpyDeviceToHost, st));
    EV_TRY(cudaStreamSynchronize(st));
#undef EV_TRY
    cleanup();
    // cumulative counts: #{scores of component c <= thr[t]}  (GroundTruthComponent.compute_overlap, au_pro_util.py:44-49)
    for (int64_t c = 0; c < n_components; ++c) {
        unsigned long long run = 0;
        for (int t = 0; t < n_thresholds; ++t) {
            run += h_hist[(size_t)c * (n_thresholds + 1) + t];
            out_component_le_counts[c * n_thresholds + t] = (int64_t)run;
        }
        out_component_sizes[c] = (int64_t)(run + h_hist[(size_t)c * (n_thresholds + 1) + n_thresholds]);
    }
    *out_two_u = h_u2;
    *out_n_neg = n_neg;
    *out_n_pos = n - n_neg;
    return rc;
}

}  // extern "C"
