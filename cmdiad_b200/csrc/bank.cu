// Memory-bank storage: pre-allocated row-major float32 bank in HBM, statistics, normalisation, gather and the
// split-fp16 scoring layout.  Replaces the Python-list banks + torch.cat + mean/std/normalise/index-select of
// run_coreset (reference multiple_features.py:37-48 and the five other variants).
#include <math.h>

#include <cstdlib>

#include "common.cuh"

namespace cmdb {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}

// ---------------------------------------------------------------------------------------------------------------
// statistics in float64, two passes over the bank (float4 loads, grid sized to the SM count): pass 1 sums x, pass 2
// sums (x - mean)^2 with mean = sum / n, so the variance does not cancel when |mean| >> std.  Every block writes one
// partial and a single block adds the partials in index order: no atomics, the result does not depend on the order
// in which blocks finish, and repeated calls are bit-identical.
// ---------------------------------------------------------------------------------------------------------------
template <bool kSqDev>
__global__ void __launch_bounds__(512) stats_pass_kernel(const float *__restrict__ x, int64_t n, const double *__restrict__ sum,
                                                         double *__restrict__ partial) {
    const double mean = kSqDev ? *sum / (double)n : 0.0;
    double s = 0.0;
    const int64_t n4 = n >> 2;
    const float4 *x4 = reinterpret_cast<const float4 *>(x);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        float4 v = __ldg(x4 + i);
        // per-vector partial in float64 keeps the dependent chain short
        if (kSqDev) {
            const double a = v.x - mean, b = v.y - mean, c = v.z - mean, d = v.w - mean;
            s += a * a + b * b + c * c + d * d;
        } else {
            s += (double)v.x + (double)v.y + (double)v.z + (double)v.w;
        }
    }
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
        const double v = (double)x[(n4 << 2) + threadIdx.x] - mean;
        s += kSqDev ? v * v : v;
    }
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    __shared__ double sh[16];
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) sh[w] = s;
    __syncthreads();
    if (w == 0) {
        s = l < (blockDim.x >> 5) ? sh[l] : 0.0;
        for (int o = 8; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (l == 0) partial[blockIdx.x] = s;
    }
}

// one block: *out = sum of partial[0 .. n_part) in a fixed order
__global__ void __launch_bounds__(256) stats_reduce_kernel(const double *__restrict__ partial, int n_part, double *__restrict__ out) {
    double s = 0.0;
    for (int i = threadIdx.x; i < n_part; i += blockDim.x) s += partial[i];
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    __shared__ double sh[8];
    if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        s = 0.0;
        for (int w = 0; w < (int)(blockDim.x >> 5); ++w) s += sh[w];
        *out = s;
    }
}

// (x - mean) / std with one IEEE subtract and one IEEE divide per element == torch's float32 CPU result
__global__ void __launch_bounds__(512) normalize_kernel(float *__restrict__ x, int64_t n, float mean, float stdv) {
    const int64_t n4 = n >> 2;
    float4 *x4 = reinterpret_cast<float4 *>(x);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        float4 v = x4[i];
        v.x = __fdiv_rn(__fsub_rn(v.x, mean), stdv);
        v.y = __fdiv_rn(__fsub_rn(v.y, mean), stdv);
        v.z = __fdiv_rn(__fsub_rn(v.z, mean), stdv);
        v.w = __fdiv_rn(__fsub_rn(v.w, mean), stdv);
        x4[i] = v;
    }
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) {
        int64_t i = (n4 << 2) + threadIdx.x;
        x[i] = __fdiv_rn(__fsub_rn(x[i], mean), stdv);
    }
}

__global__ void __launch_bounds__(256) gather_rows_kernel(const float *__restrict__ src, float *__restrict__ dst,
                                                          const long long *__restrict__ idx, int64_t n, int dim4) {
    // one warp per destination row, float4 copies
    const int warps_per_block = blockDim.x >> 5;
    const int lane = threadIdx.x & 31;
    for (int64_t r = (int64_t)blockIdx.x * warps_per_block + (threadIdx.x >> 5); r < n;
         r += (int64_t)gridDim.x * warps_per_block) {
        const float4 *s = reinterpret_cast<const float4 *>(src) + idx[r] * dim4;
        float4 *d = reinterpret_cast<float4 *>(dst) + r * dim4;
        for (int c = lane; c < dim4; c += 32) d[c] = __ldg(s + c);
    }
}

__global__ void __launch_bounds__(512) absmax_kernel(const float *__restrict__ x, int64_t n, unsigned int *out) {
    float m = 0.f;
    const int64_t n4 = n >> 2;
    const float4 *x4 = reinterpret_cast<const float4 *>(x);
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        float4 v = __ldg(x4 + i);
        m = fmaxf(fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
    }
    if (blockIdx.x == 0 && threadIdx.x < (n & 3)) m = fmaxf(m, fabsf(x[(n4 << 2) + threadIdx.x]));
    for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(out, __float_as_uint(m));  // non-negative floats order like uints
}

// Split x*2^e into fp16 hi + fp16 lo (hi + lo carries ~22 significand bits) and compute ||x||^2 (true units) per row.
// One warp per row; rows >= n_rows (padding up to the GEMM tile) are zero with norm = +inf so they never win a min.
__global__ void __launch_bounds__(256) split_rows_kernel_impl(const float *__restrict__ x, int64_t n_rows, int64_t n_pad,
                                                         int dim, float scale, __half *__restrict__ hi,
                                                         __half *__restrict__ lo, float *__restrict__ norm,
                                                         float pad_norm, unsigned int *cert_buf) {
    const int warps_per_block = blockDim.x >> 5;
    const int lane = threadIdx.x & 31;
    const int dim4 = dim >> 2;
    for (int64_t r = (int64_t)blockIdx.x * warps_per_block + (threadIdx.x >> 5); r < n_pad;
         r += (int64_t)gridDim.x * warps_per_block) {
        uint2 *h = reinterpret_cast<uint2 *>(hi + r * dim);
        uint2 *l = reinterpret_cast<uint2 *>(lo + r * dim);
        if (r >= n_rows) {
            for (int c = lane; c < dim4; c += 32) {
                h[c] = make_uint2(0u, 0u);
                l[c] = make_uint2(0u, 0u);
            }
            if (lane == 0) norm[r] = pad_norm;
            continue;
        }
        const float4 *s = reinterpret_cast<const float4 *>(x + r * dim);
        double acc = 0.0, err = 0.0;  // ||x||^2 (true units), ||x*scale - hi||^2 (scaled units; the residuals are exact)
        for (int c = lane; c < dim4; c += 32) {
            float4 v = __ldg(s + c);
            acc += (double)v.x * v.x + (double)v.y * v.y + (double)v.z * v.z + (double)v.w * v.w;  // true units
            v.x *= scale, v.y *= scale, v.z *= scale, v.w *= scale;  // power of two: exact
            __half2 h0 = __floats2half2_rn(v.x, v.y), h1 = __floats2half2_rn(v.z, v.w);
            float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
            const float r0 = v.x - f0.x, r1 = v.y - f0.y, r2 = v.z - f1.x, r3 = v.w - f1.y;
            err += (double)r0 * r0 + (double)r1 * r1 + (double)r2 * r2 + (double)r3 * r3;
            __half2 l0 = __floats2half2_rn(r0, r1), l1 = __floats2half2_rn(r2, r3);
            h[c] = make_uint2(*reinterpret_cast<unsigned int *>(&h0), *reinterpret_cast<unsigned int *>(&h1));
            l[c] = make_uint2(*reinterpret_cast<unsigned int *>(&l0), *reinterpret_cast<unsigned int *>(&l1));
        }
        for (int o = 16; o > 0; o >>= 1) {
            acc += __shfl_xor_sync(0xffffffffu, acc, o);
            err += __shfl_xor_sync(0xffffffffu, err, o);
        }
        if (lane == 0) {
            norm[r] = (float)acc;
            if (cert_buf) {  // maxima of ||b|| and ||b - b_hi|| in true units, rounded up (non-negative floats order as uints)
                atomicMax(cert_buf + 0, __float_as_uint(__double2float_ru(sqrt(acc) * (1.0 + 1e-6))));
                atomicMax(cert_buf + 1, __float_as_uint(__double2float_ru(sqrt(err) / (double)scale * (1.0 + 1e-6))));
            }
        }
    }
}

void bank_prefer_carveout() {
    CMDB_PREFER_MAX_SMEM(normalize_kernel);
    (void)cudaGetLastError();
}

void launch_normalize(cudaStream_t stream, int num_sms, float *x, int64_t n, float mean, float stdv) {
    if (n <= 0) return;
    int grid = (int)std::min<int64_t>((n / 4 + 511) / 512 + 1, (int64_t)num_sms * 4);
    normalize_kernel<<<grid, 512, 0, stream>>>(x, n, mean, stdv);
}

void launch_split_rows(cudaStream_t stream, int num_sms, const float *x, int64_t n_rows, int64_t n_pad, int dim,
                       int scale_exp, __half *hi, __half *lo, float *norm, float pad_norm, unsigned int *cert_buf) {
    int grid = (int)std::min<int64_t>((n_pad + 7) / 8, (int64_t)num_sms * 8);
    split_rows_kernel_impl<<<grid, 256, 0, stream>>>(x, n_rows, n_pad, dim, ldexpf(1.f, scale_exp), hi, lo, norm, pad_norm,
                                                     cert_buf);
}

int bank_max_abs(cmdb_bank *b, const float *x, int64_t n, float *out_host) {
    CMDB_CUDA(cudaMemsetAsync(b->absmax_buf, 0, sizeof(unsigned int), b->handle_stream()));
    int grid = (int)std::min<int64_t>((n / 4 + 511) / 512 + 1, (int64_t)b->num_sms * 4);
    absmax_kernel<<<grid, 512, 0, b->handle_stream()>>>(x, n, b->absmax_buf);
    CMDB_CUDA(cudaGetLastError());
    unsigned int bits = 0;
    CMDB_CUDA(cudaMemcpyAsync(&bits, b->absmax_buf, sizeof(bits), cudaMemcpyDeviceToHost, b->handle_stream()));
    CMDB_CUDA(cudaStreamSynchronize(b->handle_stream()));
    memcpy(out_host, &bits, sizeof(float));
    return CMDB_OK;
}

// scale exponent e such that max|x| * 2^e lands in [2^12, 2^13): far from fp16 overflow (65504) after the
// query-side scaling is applied too, and keeps the lo parts of all but negligible elements in fp16's normal range
int pick_scale_exp(float absmax) {
    if (!(absmax > 0.f) || !isfinite(absmax)) return 0;
    int e;
    frexpf(absmax, &e);  // absmax = m * 2^e, m in [0.5, 1)
    return 13 - e;
}

}  // namespace cmdb

using namespace cmdb;

extern "C" {

int cmdb_version(void) { return 100; }

const char *cmdb_last_error(void) { return cmdb::g_err; }

int cmdb_device_count(int *out_n) {
    CMDB_REQUIRE(out_n != nullptr, CMDB_ERR_INVALID, "cmdb_device_count: out_n is NULL");
    int n = 0;
    *out_n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        (void)cudaGetLastError();
        return CMDB_OK;  // no driver / no device: zero devices, not an error
    }
    int ok = 0;
    for (int d = 0; d < n; ++d) {
        int major = 0;
        if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, d) == cudaSuccess && major == 10) ++ok;
    }
    *out_n = ok;
    return CMDB_OK;
}

int cmdb_bank_create(int device, int dim, int64_t capacity_rows, cmdb_bank **out) {
    CMDB_REQUIRE(out != nullptr, CMDB_ERR_INVALID, "cmdb_bank_create: out is NULL");
    *out = nullptr;
    CMDB_REQUIRE(dim > 0 && dim % 64 == 0, CMDB_ERR_INVALID, "cmdb_bank_create: dim=%d must be a positive multiple of 64",
                 dim);
    CMDB_REQUIRE(capacity_rows > 0, CMDB_ERR_INVALID, "cmdb_bank_create: capacity_rows=%lld must be positive",
                 (long long)capacity_rows);
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        (void)cudaGetLastError();
        set_error("cmdb_bank_create: no CUDA device (%s); this library has no CPU fallback",
                  e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        return CMDB_ERR_CUDA;
    }
    CMDB_REQUIRE(device >= 0 && device < ndev, CMDB_ERR_INVALID, "cmdb_bank_create: device %d out of range [0,%d)", device,
                 ndev);
    int major = 0;
    CMDB_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
    CMDB_REQUIRE(major == 10, CMDB_ERR_CUDA, "cmdb_bank_create: device %d is sm_%d0, this library is sm_100a only", device,
                 major);
    CMDB_CUDA(cudaSetDevice(device));
    cmdb_bank *b = new cmdb_bank();
    b->device = device;
    b->dim = dim;
    b->capacity = capacity_rows;
    cudaDeviceGetAttribute(&b->num_sms, cudaDevAttrMultiProcessorCount, device);
    cudaError_t err = cudaStreamCreateWithFlags(&b->copy_stream, cudaStreamNonBlocking);
    if (err == cudaSuccess) err = cudaStreamCreateWithFlags(&b->d2h_stream, cudaStreamNonBlocking);
    for (Lane &l : b->lane) {
        if (err == cudaSuccess) err = cudaStreamCreateWithFlags(&l.stream, cudaStreamNonBlocking);
        if (err == cudaSuccess) err = cudaStreamCreateWithFlags(&l.aux, cudaStreamNonBlocking);
        if (err == cudaSuccess) err = cudaEventCreateWithFlags(&l.ev_fork, cudaEventDisableTiming);
        if (err == cudaSuccess) err = cudaEventCreateWithFlags(&l.ev_join, cudaEventDisableTiming);
    }
    for (ResultSlot &s : b->slot) {
        if (err == cudaSuccess) err = cudaEventCreateWithFlags(&s.ev_done, cudaEventDisableTiming);
        if (err == cudaSuccess) err = cudaEventCreateWithFlags(&s.ev_compute, cudaEventDisableTiming);
    }
    if (err == cudaSuccess) err = cudaEventCreateWithFlags(&b->ev_fail, cudaEventDisableTiming);
    for (auto &e : b->ev_chunk)
        if (err == cudaSuccess) err = cudaEventCreateWithFlags(&e, cudaEventDisableTiming);
    if (err == cudaSuccess) err = cudaMalloc(&b->data, sizeof(float) * (size_t)capacity_rows * dim);
    if (err == cudaSuccess) err = cudaMalloc(&b->stats_buf, sizeof(double) * (2 + (size_t)b->num_sms * 4));
    if (err == cudaSuccess) err = cudaMalloc(&b->absmax_buf, sizeof(unsigned int));
    if (err != cudaSuccess) {
        set_error("cmdb_bank_create: allocation of %lld x %d floats failed: %s", (long long)capacity_rows, dim,
                  cudaGetErrorString(err));
        (void)cudaGetLastError();
        cmdb_bank_destroy(b);
        return CMDB_ERR_CUDA;
    }
    *out = b;
    return CMDB_OK;
}

static void free_scoring_layout(cmdb_bank *b) {
    cudaFree(b->hi);
    cudaFree(b->lo);
    cudaFree(b->norm);
    cudaFree(b->knn_table);
    b->knn_table = nullptr, b->knn_rows = 0;
    b->hi = b->lo = nullptr;
    b->norm = nullptr;
    free(b->tmap_hi);
    free(b->tmap_lo);
    free(b->tmap_hi2);
    free(b->tmap_lo2);
    b->tmap_hi = b->tmap_lo = b->tmap_hi2 = b->tmap_lo2 = nullptr;
    score_scratch_free(b);
    b->finalized = false;
}

void cmdb_bank_destroy(cmdb_bank *b) {
    if (!b) return;
    cudaSetDevice(b->device);
    free_scoring_layout(b);   // synchronises every stream of the handle first
    for (int i = 0; i < 2; ++i) {
        cudaFree(b->fused.dev[i]);
        if (b->fused.host[i]) cudaFreeHost(b->fused.host[i]);
        if (b->fused.ev_done[i]) cudaEventDestroy(b->fused.ev_done[i]);
    }
    cudaFree(b->fused.acc_maps), cudaFree(b->fused.acc_scores);
    cudaFree(b->shard_ctr), cudaFree(b->shard_d2);
    if (b->shard_abort_host) cudaFreeHost(b->shard_abort_host);
    cudaFree(b->data);
    cudaFree(b->stats_buf);
    cudaFree(b->absmax_buf);
    cudaFree(b->cert_buf);
    for (auto &e : b->ev)
        if (e) cudaEventDestroy(e);
    if (b->ev_base) cudaEventDestroy(b->ev_base);
    for (Lane &l : b->lane) {
        for (auto &e : l.ev_tl)
            if (e) cudaEventDestroy(e);
        for (auto &e : l.ev_dbg)
            if (e) cudaEventDestroy(e);
        if (l.stream) cudaStreamDestroy(l.stream);
        if (l.aux) cudaStreamDestroy(l.aux);
        if (l.ev_fork) cudaEventDestroy(l.ev_fork);
        if (l.ev_join) cudaEventDestroy(l.ev_join);
    }
    if (b->copy_stream) cudaStreamDestroy(b->copy_stream);
    if (b->d2h_stream) cudaStreamDestroy(b->d2h_stream);
    for (ResultSlot &s : b->slot) {
        if (s.ev_done) cudaEventDestroy(s.ev_done);
        if (s.ev_compute) cudaEventDestroy(s.ev_compute);
    }
    if (b->ev_fail) cudaEventDestroy(b->ev_fail);
    for (auto &e : b->ev_chunk)
        if (e) cudaEventDestroy(e);
    delete b;
}

int cmdb_bank_append(cmdb_bank *b, const float *rows, int64_t n_rows, int rows_is_device) {
    CMDB_REQUIRE(b && rows && n_rows >= 0, CMDB_ERR_INVALID, "cmdb_bank_append: bad arguments");
    CMDB_REQUIRE(b->rows + n_rows <= b->capacity, CMDB_ERR_CAPACITY, "cmdb_bank_append: %lld + %lld rows exceed capacity %lld",
                 (long long)b->rows, (long long)n_rows, (long long)b->capacity);
    if (n_rows == 0) return CMDB_OK;
    CMDB_CUDA(cudaSetDevice(b->device));
    CMDB_CUDA(cudaMemcpyAsync(b->data + b->rows * b->dim, rows, sizeof(float) * (size_t)n_rows * b->dim,
                              rows_is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, b->handle_stream()));
    // the caller may reuse / free its buffer as soon as we return (pageable host memory is staged synchronously anyway)
    CMDB_CUDA(cudaStreamSynchronize(b->handle_stream()));
    b->rows += n_rows;
    b->finalized = false;
    return CMDB_OK;
}

int cmdb_bank_rows(const cmdb_bank *b, int64_t *out_rows) {
    CMDB_REQUIRE(b && out_rows, CMDB_ERR_INVALID, "cmdb_bank_rows: bad arguments");
    *out_rows = b->rows;
    return CMDB_OK;
}

int cmdb_bank_dim(const cmdb_bank *b, int *out_dim) {
    CMDB_REQUIRE(b && out_dim, CMDB_ERR_INVALID, "cmdb_bank_dim: bad arguments");
    *out_dim = b->dim;
    return CMDB_OK;
}

int cmdb_bank_set_row_offset(cmdb_bank *b, int64_t row_offset) {
    CMDB_REQUIRE(b && row_offset >= 0, CMDB_ERR_INVALID, "cmdb_bank_set_row_offset: bad arguments");
    b->row_offset = row_offset;
    return CMDB_OK;
}

int cmdb_bank_set_option(cmdb_bank *b, int option, int value) {
    CMDB_REQUIRE(b, CMDB_ERR_INVALID, "cmdb_bank_set_option: bank is NULL");
    if (option == CMDB_OPT_SCORE_IMPL) {
        CMDB_REQUIRE(value == CMDB_SCORE_TCGEN05 || value == CMDB_SCORE_SIMT, CMDB_ERR_INVALID,
                     "cmdb_bank_set_option: unknown scoring implementation %d", value);
        b->score_impl = value;
        return CMDB_OK;
    }
    if (option == CMDB_OPT_PREFILTER_TERMS) {
        CMDB_REQUIRE(value == 0 || value == 1 || value == 3, CMDB_ERR_INVALID,
                     "cmdb_bank_set_option: prefilter terms must be 0 (certified), 1 or 3");
        b->prefilter_terms = value;
        b->direct_calls_left = 0;
        b->fail_pending = false;
        return CMDB_OK;
    }
    if (option == CMDB_OPT_TIMING) {
        b->timing = value == 2 ? 2 : (value != 0);
        if (b->timing && !b->ev[0]) {
            CMDB_CUDA(cudaSetDevice(b->device));
            for (auto &e : b->ev) CMDB_CUDA(cudaEventCreate(&e));
        }
        if (b->timing == 2) {  // lane timeline (diagnostics): per-lane events against a common base
            CMDB_CUDA(cudaSetDevice(b->device));
            if (!b->ev_base) {
                CMDB_CUDA(cudaEventCreate(&b->ev_base));
                for (Lane &l : b->lane) {
                    for (auto &e : l.ev_tl) CMDB_CUDA(cudaEventCreate(&e));
                    for (auto &e : l.ev_dbg) CMDB_CUDA(cudaEventCreate(&e));
                }
            }
            CMDB_CUDA(cudaDeviceSynchronize());
            CMDB_CUDA(cudaEventRecord(b->ev_base, b->lane[0].stream));
        }
        b->ev_valid = false;
        return CMDB_OK;
    }
    set_error("cmdb_bank_set_option: unknown option %d", option);
    return CMDB_ERR_INVALID;
}

int cmdb_bank_set_query_norm(cmdb_bank *b, float mean, float stdv, int enabled) {
    CMDB_REQUIRE(b, CMDB_ERR_INVALID, "cmdb_bank_set_query_norm: bank is NULL");
    CMDB_REQUIRE(!enabled || (isfinite(mean) && isfinite(stdv) && stdv != 0.f), CMDB_ERR_INVALID,
                 "cmdb_bank_set_query_norm: need finite mean and a finite non-zero std");
    b->q_norm_enabled = enabled != 0;
    b->q_mean = mean, b->q_std = stdv;
    return CMDB_OK;
}

int cmdb_bank_stream(cmdb_bank *b, void **out_stream) {
    CMDB_REQUIRE(b && out_stream, CMDB_ERR_INVALID, "cmdb_bank_stream: bad arguments");
    // the lane of the open sharded round (its collectives), else the lane the NEXT scoring call of this handle runs on
    *out_stream = (void *)b->lane[b->round.open ? b->round.lane : b->next_lane].stream;
    return CMDB_OK;
}

int cmdb_bank_lane_streams(cmdb_bank *b, void **out_streams2) {
    CMDB_REQUIRE(b && out_streams2, CMDB_ERR_INVALID, "cmdb_bank_lane_streams: bad arguments");
    out_streams2[0] = (void *)b->lane[0].stream, out_streams2[1] = (void *)b->lane[1].stream;
    return CMDB_OK;
}

int cmdb_bank_get_timings(cmdb_bank *b, float *out_ms) {
    CMDB_REQUIRE(b && out_ms, CMDB_ERR_INVALID, "cmdb_bank_get_timings: bad arguments");
    CMDB_REQUIRE(b->timing && b->ev_valid, CMDB_ERR_STATE, "cmdb_bank_get_timings: enable CMDB_OPT_TIMING and call cmdb_score first");
    CMDB_CUDA(cudaEventSynchronize(b->ev[CMDB_T_COUNT]));  // recorded right behind the event the wait call synchronised on
    for (int i = 0; i < CMDB_T_COUNT; ++i) CMDB_CUDA(cudaEventElapsedTime(out_ms + i, b->ev[i], b->ev[i + 1]));
    return CMDB_OK;
}

static int build_knn_checks(cmdb_bank *b, const char *fn) {
    CMDB_REQUIRE(b, CMDB_ERR_INVALID, "%s: bank is NULL", fn);
    CMDB_REQUIRE(b->finalized, CMDB_ERR_STATE, "%s: call cmdb_bank_finalize first", fn);
    CMDB_REQUIRE(b->row_offset == 0, CMDB_ERR_UNSUPPORTED,
                 "%s: the table is computed on a handle that holds every bank row (row-sharded handles install a replicated "
                 "table with cmdb_bank_set_knn_table)", fn);
    CMDB_REQUIRE(!b->any_pending(), CMDB_ERR_STATE, "%s: a submitted batch is outstanding", fn);
    CMDB_CUDA(cudaSetDevice(b->device));
    return CMDB_OK;
}

int cmdb_bank_build_knn(cmdb_bank *b) {
    CMDB_CHECK(build_knn_checks(b, "cmdb_bank_build_knn"));
    return score_build_knn_table(b, 0, b->fin_rows);
}

int cmdb_bank_build_knn_rows(cmdb_bank *b, int64_t row_first, int64_t n_rows) {
    CMDB_CHECK(build_knn_checks(b, "cmdb_bank_build_knn_rows"));
    CMDB_REQUIRE(row_first >= 0 && n_rows >= 0 && row_first + n_rows <= b->fin_rows, CMDB_ERR_INVALID,
                 "cmdb_bank_build_knn_rows: rows [%lld,%lld) outside [0,%lld)", (long long)row_first,
                 (long long)(row_first + n_rows), (long long)b->fin_rows);
    return score_build_knn_table(b, row_first, n_rows);
}

int cmdb_bank_read_knn(cmdb_bank *b, int64_t row_first, int64_t n_rows, uint64_t *out_keys, int out_is_device) {
    CMDB_REQUIRE(b && out_keys && b->knn_table && row_first >= 0 && n_rows >= 0 && row_first + n_rows <= b->knn_rows,
                 CMDB_ERR_INVALID, "cmdb_bank_read_knn: no table, or rows outside it");
    if (n_rows == 0) return CMDB_OK;
    CMDB_CUDA(cudaSetDevice(b->device));
    CMDB_CUDA(cudaMemcpyAsync(out_keys, b->knn_table + (size_t)row_first * 3, sizeof(uint64_t) * 3 * (size_t)n_rows,
                              out_is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost, b->handle_stream()));
    CMDB_CUDA(cudaStreamSynchronize(b->handle_stream()));
    return CMDB_OK;
}

int cmdb_bank_set_knn_table(cmdb_bank *b, const uint64_t *keys, int64_t n_rows_total, int keys_is_device) {
    CMDB_REQUIRE(b && keys && n_rows_total >= 1, CMDB_ERR_INVALID, "cmdb_bank_set_knn_table: bad arguments");
    CMDB_REQUIRE(b->finalized, CMDB_ERR_STATE, "cmdb_bank_set_knn_table: call cmdb_bank_finalize first");
    CMDB_REQUIRE(b->row_offset + b->fin_rows <= n_rows_total, CMDB_ERR_INVALID,
                 "cmdb_bank_set_knn_table: the table must cover all GLOBAL rows (this shard ends at %lld, table has %lld)",
                 (long long)(b->row_offset + b->fin_rows), (long long)n_rows_total);
    CMDB_REQUIRE(!b->any_pending(), CMDB_ERR_STATE, "cmdb_bank_set_knn_table: a submitted batch is outstanding");
    CMDB_CUDA(cudaSetDevice(b->device));
    CMDB_CUDA(cudaStreamSynchronize(b->handle_stream()));
    cudaFree(b->knn_table);
    b->knn_table = nullptr, b->knn_rows = 0;
    CMDB_CUDA(cudaMalloc(&b->knn_table, sizeof(uint64_t) * 3 * (size_t)n_rows_total));
    CMDB_CUDA(cudaMemcpyAsync(b->knn_table, keys, sizeof(uint64_t) * 3 * (size_t)n_rows_total,
                              keys_is_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, b->handle_stream()));
    CMDB_CUDA(cudaStreamSynchronize(b->handle_stream()));
    b->knn_rows = n_rows_total;
    return CMDB_OK;
}

int cmdb_bank_score_stats(cmdb_bank *b, int64_t *out6) {
    CMDB_REQUIRE(b && out6, CMDB_ERR_INVALID, "cmdb_bank_score_stats: bad arguments");
    CMDB_CUDA(cudaSetDevice(b->device));
    for (const Lane &l : b->lane) CMDB_CUDA(cudaStreamSynchronize(l.stream));
    const bool cert = b->last_mode == 0 && b->last_fail_host;
    out6[0] = b->last_queries;
    out6[1] = b->last_mode;
    out6[2] = cert ? (int64_t)b->last_fail_host[0] : 0;
    out6[3] = cert ? (int64_t)b->last_fail_host[1] : 0;
    out6[4] = cert && !cmdb::fallback_use_rescan(b->last_fail_host[0], b->last_fail_host[1]);
    out6[5] = b->direct_calls_left;
    return CMDB_OK;
}

int cmdb_bank_stats(cmdb_bank *b, double *out_mean, double *out_std, double *out_sum, double *out_sumsq) {
    CMDB_REQUIRE(b, CMDB_ERR_INVALID, "cmdb_bank_stats: bank is NULL");
    CMDB_REQUIRE(b->rows > 0, CMDB_ERR_STATE, "cmdb_bank_stats: bank is empty");
    CMDB_CUDA(cudaSetDevice(b->device));
    const int64_t n = b->rows * b->dim;
    // stats_buf: [0] sum, [1] sum of squared deviations, [2 ..) one partial per block (sized for num_sms * 4 blocks)
    const int grid = (int)std::min<int64_t>((n / 4 + 511) / 512 + 1, (int64_t)b->num_sms * 4);
    double *part = b->stats_buf + 2;
    stats_pass_kernel<false><<<grid, 512, 0, b->handle_stream()>>>(b->data, n, nullptr, part);
    stats_reduce_kernel<<<1, 256, 0, b->handle_stream()>>>(part, grid, b->stats_buf);
    stats_pass_kernel<true><<<grid, 512, 0, b->handle_stream()>>>(b->data, n, b->stats_buf, part);
    stats_reduce_kernel<<<1, 256, 0, b->handle_stream()>>>(part, grid, b->stats_buf + 1);
    CMDB_CUDA(cudaGetLastError());
    double h[2];
    CMDB_CUDA(cudaMemcpyAsync(h, b->stats_buf, sizeof(h), cudaMemcpyDeviceToHost, b->handle_stream()));
    CMDB_CUDA(cudaStreamSynchronize(b->handle_stream()));
    const double mean = h[0] / (double)n;
    const double var = n > 1 ? h[1] / (double)(n - 1) : NAN;  // unbiased, like torch.std
    if (out_mean) *out_mean = mean;
    if (out_std) *out_std = sqrt(var);
    if (out_sum) *out_sum = h[0];
    if (out_sumsq) *out_sumsq = h[1] + h[0] * mean;  // sum of squares, rebuilt from the deviations
    return CMDB_OK;
}

int cmdb_bank_normalize(cmdb_bank *b, float mean, float stdv) {
    CMDB_REQUIRE(b, CMDB_ERR_INVALID, "cmdb_bank_normalize: bank is NULL");
    CMDB_REQUIRE(!b->any_pending(), CMDB_ERR_STATE, "cmdb_bank_normalize: a submitted call still reads the rows; wait for it first");
    if (b->rows == 0) return CMDB_OK;
    CMDB_CUDA(cudaSetDevice(b->device));
    const int64_t n = b->rows * b->dim;
    int grid = (int)std::min<int64_t>((n / 4 + 511) / 512 + 1, (int64_t)b->num_sms * 4);
    normalize_kernel<<<grid, 512, 0, b->handle_stream()>>>(b->data, n, mean, stdv);
    CMDB_CUDA(cudaGetLastError());
    CMDB_CUDA(cudaStreamSynchronize(b->handle_stream()));
    b->finalized = false;
    return CMDB_OK;
}

int cmdb_bank_gather(cmdb_bank *b, const int64_t *idx_host, int64_t n) {
    CMDB_REQUIRE(b && idx_host && n > 0, CMDB_ERR_INVALID, "cmdb_bank_gather: bad arguments");
    CMDB_REQUIRE(n <= b->capacity, CMDB_ERR_CAPACITY, "cmdb_bank_gather: n exceeds capacity");
    for (int64_t i = 0; i < n; ++i)
        CMDB_REQUIRE(idx_host[i] >= 0 && idx_host[i] < b->rows, CMDB_ERR_INVALID,
                     "cmdb_bank_gather: idx[%lld]=%lld out of range [0,%lld)", (long long)i, (long long)idx_host[i],
                     (long long)b->rows);
    CMDB_REQUIRE(!b->any_pending(), CMDB_ERR_STATE, "cmdb_bank_gather: a submitted call still reads the rows; wait for it first");
    CMDB_CUDA(cudaSetDevice(b->device));
    long long *idx_dev = nullptr;
    float *tmp = nullptr;
    CMDB_CUDA(cudaMalloc(&idx_dev, sizeof(long long) * (size_t)n));
    cudaError_t e = cudaMalloc(&tmp, sizeof(float) * (size_t)n * b->dim);
    if (e != cudaSuccess) {
        cudaFree(idx_dev);
        CMDB_CUDA(e);
    }
    e = cudaMemcpyAsync(idx_dev, idx_host, sizeof(long long) * (size_t)n, cudaMemcpyHostToDevice, b->handle_stream());
    if (e == cudaSuccess) {
        int grid = (int)std::min<int64_t>((n + 7) / 8, (int64_t)b->num_sms * 8);
        gather_rows_kernel<<<grid, 256, 0, b->handle_stream()>>>(b->data, tmp, idx_dev, n, b->dim / 4);
        e = cudaGetLastError();
    }
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(b->data, tmp, sizeof(float) * (size_t)n * b->dim, cudaMemcpyDeviceToDevice, b->handle_stream());
    if (e == cudaSuccess) e = cudaStreamSynchronize(b->handle_stream());
    cudaFree(idx_dev);
    cudaFree(tmp);
    CMDB_CUDA(e);
    b->rows = n;
    b->finalized = false;
    return CMDB_OK;
}

int cmdb_bank_read(cmdb_bank *b, int64_t row0, int64_t n_rows, float *out_host) {
    CMDB_REQUIRE(b && out_host && row0 >= 0 && n_rows >= 0 && row0 + n_rows <= b->rows, CMDB_ERR_INVALID,
                 "cmdb_bank_read: rows [%lld,%lld) outside [0,%lld)", (long long)row0, (long long)(row0 + n_rows),
                 b ? (long long)b->rows : 0LL);
    if (n_rows == 0) return CMDB_OK;
    CMDB_CUDA(cudaSetDevice(b->device));
    CMDB_CUDA(cudaMemcpyAsync(out_host, b->data + row0 * b->dim, sizeof(float) * (size_t)n_rows * b->dim,
                              cudaMemcpyDeviceToHost, b->handle_stream()));
    CMDB_CUDA(cudaStreamSynchronize(b->handle_stream()));
    return CMDB_OK;
}

int cmdb_bank_finalize(cmdb_bank *b) {
    CMDB_REQUIRE(b, CMDB_ERR_INVALID, "cmdb_bank_finalize: bank is NULL");
    CMDB_REQUIRE(b->rows > 0, CMDB_ERR_STATE, "cmdb_bank_finalize: bank is empty");
    CMDB_REQUIRE(b->rows + b->row_offset < (1LL << 31), CMDB_ERR_UNSUPPORTED,
                 "cmdb_bank_finalize: global row numbers must fit 31 bits for the packed (distance,row) keys");
    CMDB_REQUIRE(!b->any_pending(), CMDB_ERR_STATE,
                 "cmdb_bank_finalize: a submitted call still uses the scoring layout; wait for it first");
    CMDB_CUDA(cudaSetDevice(b->device));
    free_scoring_layout(b);
    const int64_t pad = (b->rows + kScoreBN - 1) / kScoreBN * kScoreBN;
    CMDB_CUDA(cudaMalloc(&b->hi, sizeof(__half) * (size_t)pad * b->dim));
    CMDB_CUDA(cudaMalloc(&b->lo, sizeof(__half) * (size_t)pad * b->dim));
    CMDB_CUDA(cudaMalloc(&b->norm, sizeof(float) * (size_t)pad));
    float absmax = 0.f;
    CMDB_CHECK(bank_max_abs(b, b->data, b->rows * b->dim, &absmax));
    CMDB_REQUIRE(isfinite(absmax), CMDB_ERR_INVALID, "cmdb_bank_finalize: bank contains non-finite values");
    b->scale_exp = pick_scale_exp(absmax);
    if (!b->cert_buf) CMDB_CUDA(cudaMalloc(&b->cert_buf, 2 * sizeof(unsigned int)));
    CMDB_CUDA(cudaMemsetAsync(b->cert_buf, 0, 2 * sizeof(unsigned int), b->handle_stream()));
    launch_split_rows(b->handle_stream(), b->num_sms, b->data, b->rows, pad, b->dim, b->scale_exp, b->hi, b->lo, b->norm, INFINITY,
                      b->cert_buf);
    CMDB_CUDA(cudaGetLastError());
    float cert[2] = {0.f, 0.f};
    CMDB_CUDA(cudaMemcpyAsync(cert, b->cert_buf, sizeof(cert), cudaMemcpyDeviceToHost, b->handle_stream()));
    CMDB_CUDA(cudaStreamSynchronize(b->handle_stream()));
    b->cert_bmax = cert[0], b->cert_eb_max = cert[1];
    b->direct_calls_left = 0, b->fail_pending = false;
    b->fin_rows = b->rows;
    b->fin_rows_pad = pad;
    CMDB_CHECK(score_make_tensor_maps(b));
    b->finalized = true;
    return CMDB_OK;
}

}  // extern "C"
