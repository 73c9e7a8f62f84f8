// Sparse random projection z = X @ C^T, bit-exact with sklearn's SparseRandomProjection.transform
// (reference features.py:365-366): X float32 is up-cast to float64; for every output (i, j) the products
// data[k] * x[i, indices[k]] are added in the CSR row's STORED order with separate IEEE multiply and add
// (scipy csr_matvecs: y[i,:] += a * x[j,:] per non-zero, no fma) -- see oracle/coreset_oracle.c:oracle_sparse_project.
//
// HBM-bound by design: each bank row (D*4 bytes) is read once into shared memory and reused for all d' outputs.
// Layout: a CTA stages RT rows with row stride D+1 floats, so the 32 lanes of a warp (= 32 different rows, same output
// column j, hence the same CSR index) hit 32 different banks; the CSR (indptr + 16-bit index|sign) sits in shared
// memory and is read as a warp broadcast.
#include "common.cuh"

namespace cmdb {

template <int RT>
__global__ void __launch_bounds__(256)
project_kernel(const float *__restrict__ x, int64_t n_rows, int D, const int *__restrict__ indptr,
               const unsigned short *__restrict__ packed, const double *__restrict__ data, double mag, int d_proj,
               int nnz, double *__restrict__ z) {
    extern __shared__ unsigned char smem_raw[];
    float *xs = reinterpret_cast<float *>(smem_raw);                       // [RT][D+1]
    int *s_indptr = reinterpret_cast<int *>(xs + (size_t)RT * (D + 1));     // [d_proj+1]
    unsigned short *s_packed = reinterpret_cast<unsigned short *>(s_indptr + d_proj + 1);  // [nnz] (uniform magnitude)
    const bool uniform = packed != nullptr;
    for (int i = threadIdx.x; i <= d_proj; i += blockDim.x) s_indptr[i] = indptr[i];
    if (uniform)
        for (int i = threadIdx.x; i < nnz; i += blockDim.x) s_packed[i] = packed[i];
    constexpr int JG = 256 / RT;
    const int row = threadIdx.x % RT, jg = threadIdx.x / RT;
    const int64_t n_tiles = (n_rows + RT - 1) / RT;
    for (int64_t tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
        const int64_t row0 = tile * RT;
        __syncthreads();
        // coalesced float4 loads of RT consecutive rows, scalar stores into the padded tile
        const int D4 = D >> 2;
        for (int i = threadIdx.x; i < RT * D4; i += blockDim.x) {
            const int r = i / D4, c = i - r * D4;
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (row0 + r < n_rows) v = __ldg(reinterpret_cast<const float4 *>(x + (row0 + r) * D) + c);
            float *dst = xs + (size_t)r * (D + 1) + 4 * c;
            dst[0] = v.x, dst[1] = v.y, dst[2] = v.z, dst[3] = v.w;
        }
        __syncthreads();
        const float *xr = xs + (size_t)row * (D + 1);
        if (row0 + row < n_rows) {
            for (int j = jg; j < d_proj; j += JG) {
                double y = 0.0;
                const int k0 = s_indptr[j], k1 = s_indptr[j + 1];
                if (uniform) {
                    for (int k = k0; k < k1; ++k) {
                        const unsigned int p = s_packed[k];
                        const double a = (p & 0x8000u) ? -mag : mag;
                        y = __dadd_rn(y, __dmul_rn(a, (double)xr[p & 0x7fffu]));
                    }
                } else {
                    for (int k = k0; k < k1; ++k) {
                        const int col = __ldg(reinterpret_cast<const int *>(data + nnz) + k);
                        y = __dadd_rn(y, __dmul_rn(__ldg(data + k), (double)xr[col]));
                    }
                }
                z[(row0 + row) * d_proj + j] = y;
            }
        }
    }
}

// Uploads the CSR matrix.  If every |data| is the same value (sklearn's matrix: +-sqrt(1/density)/sqrt(d')) and
// D < 32768 the kernel uses a 16-bit index|sign stream in shared memory; otherwise it reads float64 data + int32
// indices (stored behind the data array) through L1.
int project_rows(cmdb_bank *b, const float *x_dev, int64_t n_rows, int D, const int32_t *indptr_h,
                 const int32_t *indices_h, const double *data_h, int d_proj, double *z_dev) {
    CMDB_REQUIRE(indptr_h && indices_h && data_h && d_proj > 0, CMDB_ERR_INVALID, "projection: CSR arrays missing");
    CMDB_REQUIRE(indptr_h[0] == 0, CMDB_ERR_INVALID, "projection: csr_indptr[0] must be 0");
    const int nnz = indptr_h[d_proj];
    CMDB_REQUIRE(nnz >= 0, CMDB_ERR_INVALID, "projection: negative nnz");
    bool uniform = D < 32768 && nnz > 0;
    const double mag = nnz > 0 ? fabs(data_h[0]) : 0.0;
    for (int j = 0; j < d_proj; ++j)
        CMDB_REQUIRE(indptr_h[j + 1] >= indptr_h[j], CMDB_ERR_INVALID, "projection: csr_indptr not monotone");
    for (int k = 0; k < nnz; ++k) {
        CMDB_REQUIRE(indices_h[k] >= 0 && indices_h[k] < D, CMDB_ERR_INVALID, "projection: csr index %d out of [0,%d)",
                     indices_h[k], D);
        if (fabs(data_h[k]) != mag) uniform = false;
    }
    int *indptr_d = nullptr;
    unsigned short *packed_d = nullptr;
    double *data_d = nullptr;  // [nnz] doubles followed by [nnz] int32 indices (generic path)
    cudaError_t e = cudaMalloc(&indptr_d, sizeof(int) * (d_proj + 1));
    if (e == cudaSuccess)
        e = cudaMemcpyAsync(indptr_d, indptr_h, sizeof(int) * (d_proj + 1), cudaMemcpyHostToDevice, b->handle_stream());
    unsigned short *packed_h = nullptr;
    if (e == cudaSuccess && uniform) {
        packed_h = (unsigned short *)malloc(sizeof(unsigned short) * (size_t)nnz);
        for (int k = 0; k < nnz; ++k)
            packed_h[k] = (unsigned short)(indices_h[k] | (data_h[k] < 0 ? 0x8000 : 0));
        e = cudaMalloc(&packed_d, sizeof(unsigned short) * (size_t)nnz);
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(packed_d, packed_h, sizeof(unsigned short) * (size_t)nnz, cudaMemcpyHostToDevice,
                                b->handle_stream());
    } else if (e == cudaSuccess) {
        e = cudaMalloc(&data_d, (sizeof(double) + sizeof(int)) * (size_t)(nnz > 0 ? nnz : 1));
        if (e == cudaSuccess && nnz > 0)
            e = cudaMemcpyAsync(data_d, data_h, sizeof(double) * (size_t)nnz, cudaMemcpyHostToDevice, b->handle_stream());
        if (e == cudaSuccess && nnz > 0)
            e = cudaMemcpyAsync(reinterpret_cast<int *>(data_d + nnz), indices_h, sizeof(int) * (size_t)nnz,
                                cudaMemcpyHostToDevice, b->handle_stream());
    }
    if (e == cudaSuccess) {
        const size_t csr_bytes = sizeof(int) * (d_proj + 1) + (uniform ? sizeof(unsigned short) * (size_t)nnz : 0) + 16;
        const size_t budget = 220 * 1024;
        int rt = 32;
        while (rt > 8 && sizeof(float) * (size_t)rt * (D + 1) + csr_bytes > budget) rt >>= 1;
        const size_t smem = sizeof(float) * (size_t)rt * (D + 1) + csr_bytes;
        if (smem > budget) {
            set_error("projection: dim=%d with %d non-zeros does not fit shared memory", D, nnz);
            e = cudaErrorInvalidValue;
        } else {
            const int64_t n_tiles = (n_rows + rt - 1) / rt;
            const int grid = (int)std::min<int64_t>(n_tiles, (int64_t)b->num_sms);
            auto launch = [&](auto kern) {
                cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
                kern<<<grid, 256, smem, b->handle_stream()>>>(x_dev, n_rows, D, indptr_d, packed_d, data_d, mag, d_proj, nnz, z_dev);
            };
            if (rt == 32) launch(project_kernel<32>);
            else if (rt == 16) launch(project_kernel<16>);
            else launch(project_kernel<8>);
            e = cudaGetLastError();
        }
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(b->handle_stream());
    free(packed_h);
    cudaFree(indptr_d);
    cudaFree(packed_d);
    cudaFree(data_d);
    if (e != cudaSuccess && e != cudaErrorInvalidValue) CMDB_CUDA(e);
    return e == cudaSuccess ? CMDB_OK : CMDB_ERR_INVALID;
}

}  // namespace cmdb
