// extern "C" entry points that orchestrate the kernels: coreset selection, projection, scoring (single GPU and the
// row-sharded phases), stand-alone upsample+blur.  Declarations and reference citations: include/cmdiad_b200.h.
#include <math.h>

#include <vector>

#include "common.cuh"

namespace cmdb {

__global__ void __launch_bounds__(512) f32_to_f64_kernel(const float *__restrict__ x, long long n, double *__restrict__ z) {
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
        z[i] = (double)x[i];
}

// keys[p] = exchange_key(local min d^2, global row) -- a round's local min_val holds d^2 (ScoreCall::sq_min); and the
// inverse, which takes the root: min_val = sqrtf(d^2) as a single bank computes it
__global__ void pack_keys_kernel(const float *__restrict__ min_d2, const long long *__restrict__ min_idx, int P,
                                 long long *__restrict__ keys) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < P) keys[i] = exchange_key(min_d2[i], min_idx[i]);
}
__global__ void unpack_keys_kernel(const long long *__restrict__ keys, int P, int P_img, float *__restrict__ min_val,
                                   long long *__restrict__ min_idx, unsigned long long *s_key) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < P) {
        const unsigned long long k = (unsigned long long)keys[i];
        const float v = sqrtf(key_value(k));
        min_val[i] = v;
        min_idx[i] = key_row(k);
        argmax_publish(s_key, i, P_img, v);
    }
}

void api_prefer_carveout_fuse();
void api_prefer_carveout() {
    api_prefer_carveout_fuse();
    CMDB_PREFER_MAX_SMEM(pack_keys_kernel);
    CMDB_PREFER_MAX_SMEM(unpack_keys_kernel);
    (void)cudaGetLastError();
}

static int check_score_args(cmdb_bank *b, const void *patch, int B, int P, const char *fn) {
    CMDB_REQUIRE(b && patch, CMDB_ERR_INVALID, "%s: NULL argument", fn);
    CMDB_REQUIRE(b->finalized, CMDB_ERR_STATE, "%s: call cmdb_bank_finalize first", fn);
    CMDB_REQUIRE(P >= 1 && P <= (1 << 20), CMDB_ERR_INVALID, "%s: P=%d out of range", fn, P);
    CMDB_REQUIRE(B >= 1 && B <= 4096, CMDB_ERR_INVALID, "%s: batch=%d out of range", fn, B);
    return CMDB_OK;
}

// Opens a scoring call on b: takes the next compute lane and result slot and sizes the scratch for B images (at most
// score_max_batch) of P patches with out_hw x out_hw maps.  The map stride is fixed per scratch: another out_hw frees the
// scratch first, which needs every submitted call waited for.
static int begin_call(cmdb_bank *b, int B, int P, int out_hw, const char *fn, ScoreCall *c) {
    CMDB_REQUIRE(B <= score_max_batch(b), CMDB_ERR_INVALID, "%s: batch=%d exceeds the per-call limit %d", fn, B, score_max_batch(b));
    CMDB_CUDA(cudaSetDevice(b->device));
    if (b->layout.map_stride && (size_t)out_hw * out_hw != b->layout.map_stride) {
        CMDB_REQUIRE(!b->any_pending(), CMDB_ERR_STATE, "%s: out_hw changes while a submitted call is outstanding; wait for it first",
                     fn);
        score_scratch_free(b);
    }
    CMDB_REQUIRE(!b->slot[b->next_slot].pending.active, CMDB_ERR_STATE,
                 "%s: all %d result slots hold submitted calls; wait for one first", fn, kResultSlots);
    CMDB_CHECK(score_scratch_alloc(b, B, P, out_hw));  // fails with CMDB_ERR_STATE if the scratch would have to grow
    *c = score_call(b, b->next_lane, b->next_slot);
    b->next_lane ^= 1;
    b->next_slot = (b->next_slot + 1) % kResultSlots;
    return CMDB_OK;
}

// Hands a call to the caller once its result copies are enqueued on the d2h stream: the slot holds the results of B images
// (maps of images img_first, img_first + img_step, ...) until the caller waits for the call's ticket.
static int publish_call(const ScoreCall &c, int B, int P, int out_hw, unsigned want, bool host_maps, int img_first, int img_step) {
    cmdb_bank *b = c.b;
    CMDB_CUDA(cudaEventRecord(c.slot->ev_done, b->d2h_stream));
    c.slot->pending = ResultSlot::Pending{true, B, P, out_hw, want, host_maps, img_first, img_step, ++b->ticket_counter};
    return CMDB_OK;
}

// bytes of the result block that a full-batch copy has to move (want: bit 0 = pre-blur maps, bit 1 = 8-bit maps)
static size_t out_block_extent(const cmdb_bank *b, int B, unsigned want) {
    const ScoreLayout &s = b->layout;
    size_t bytes = s.off_map_out + sizeof(float) * s.map_stride * B;
    if (want & 1u) bytes = s.off_map_pre + sizeof(float) * s.map_stride * B;
    if (want & 2u) bytes = s.off_map_u8 + s.map_stride * B;
    return bytes;
}
static unsigned want_mask_of(const cmdb_score_out *outs, int B) {
    unsigned w = 0;
    for (int i = 0; i < B; ++i) w |= (outs[i].s_map_pre ? 1u : 0u) | (outs[i].s_map_u8 ? 2u : 0u);
    return w;
}

// host block of a slot -> the caller's buffers (maps = false: only the scalars and per-patch arrays of image i)
static void scatter_one(const cmdb_bank *b, const unsigned char *h, int i, int P, int out_hw, cmdb_score_out *out, bool maps) {
    const ScoreLayout &s = b->layout;
    const size_t npix = (size_t)out_hw * out_hw;
    TailResult tr;
    memcpy(&tr, h + sizeof(TailResult) * i, sizeof(tr));
    if (out->min_val) memcpy(out->min_val, h + s.off_min_val + sizeof(float) * (size_t)i * P, sizeof(float) * P);
    if (out->min_idx) memcpy(out->min_idx, h + s.off_min_idx + sizeof(long long) * (size_t)i * P, sizeof(long long) * P);
    if (maps) {
        if (out->s_map) memcpy(out->s_map, h + s.off_map_out + sizeof(float) * s.map_stride * i, sizeof(float) * npix);
        if (out->s_map_pre) memcpy(out->s_map_pre, h + s.off_map_pre + sizeof(float) * s.map_stride * i, sizeof(float) * npix);
        if (out->s_map_u8) memcpy(out->s_map_u8, h + s.off_map_u8 + s.map_stride * i, npix);
    }
    if (out->s) *out->s = tr.s;
    if (out->s_star) *out->s_star = tr.s_star;
    if (out->s_idx) *out->s_idx = tr.s_idx;
    if (out->w) *out->w = tr.w;
    if (out->m_star_knn) out->m_star_knn[0] = tr.knn0, out->m_star_knn[1] = tr.knn1;
    if (out->nn_idx)
        for (int k = 0; k < 3; ++k) out->nn_idx[k] = tr.nn_idx[k];
}

static int blur_batch(const ScoreCall &c, int B, int fh, int fw, int out_hw, int img_first = 0, int img_step = 1) {
    const ScoreLayout &s = c.b->layout;
    const Lane &l = *c.lane;
    CMDB_REQUIRE((size_t)out_hw * out_hw <= s.map_stride, CMDB_ERR_INVALID, "scoring: out_hw=%d larger than the scratch maps", out_hw);
    const int n_img = img_first < B ? (B - img_first + img_step - 1) / img_step : 0;
    return upsample_blur_launch(c.stream, n_img, img_first, img_step, s.map_stride, c.min_val, fh, fw, out_hw, c.map_pre,
                                c.map_out, c.map_u8, l.map_tmp, l.map_max, l.map_max + s.cap_b);
}

// ---------------------------------------------------------------------------------------------------------------
// late-fusion head (multiple_features.py:986-994): lambda scaling in float32, SGDOneClassSVM.score_samples in float64
//   X @ coef_: dgemv evaluates fma(x0, c0, x1 * c1) for the [npix, 2] map matrix and fma(x2, c2, fma(x0, c0, x1 * c1))
//   for [npix, 3]; the ddot of a single row is a sequential fma over the columns, fma(x1, c1, x0 * c0) and
//   fma(x2, c2, fma(x1, c1, x0 * c0)) (OpenBLAS as shipped with numpy/scipy; pinned by tests against sklearn).
// grid (pixel blocks, images)
// ---------------------------------------------------------------------------------------------------------------
struct FuseParams {
    int n_modal, B, npix;
    const float *maps[3];
    size_t map_stride[3];
    const TailResult *tails[3];
    float s_lambda[3], smap_lambda[3];
    double det_coef[3], det_off, seg_coef[3], seg_off;
    double *out_s;        // [B]
    float *out_s_modal;   // [B][3]
    double *out_map;      // [B][npix] or nullptr
    double *acc_map;      // [B][npix] slice of the device-side result store, or nullptr
    double *acc_s;        // [B] or nullptr
};

__global__ void __launch_bounds__(256) fuse_head_kernel(FuseParams p) {
    const int b = blockIdx.y;
    const float *m0 = p.maps[0] + (size_t)b * p.map_stride[0];
    const float *m1 = p.n_modal > 1 ? p.maps[1] + (size_t)b * p.map_stride[1] : nullptr;
    const float *m2 = p.n_modal > 2 ? p.maps[2] + (size_t)b * p.map_stride[2] : nullptr;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < p.npix; i += gridDim.x * blockDim.x) {
        // lambda * s_map in float32 (python float * float32 tensor), then sklearn's float64 copy
        const double x0 = (double)__fmul_rn(p.smap_lambda[0], m0[i]);
        double v;
        if (p.n_modal == 1) {
            v = __dmul_rn(x0, p.seg_coef[0]);
        } else {
            const double x1 = (double)__fmul_rn(p.smap_lambda[1], m1[i]);
            if (p.n_modal == 2) {
                v = __fma_rn(x0, p.seg_coef[0], __dmul_rn(x1, p.seg_coef[1]));
            } else {
                const double x2 = (double)__fmul_rn(p.smap_lambda[2], m2[i]);
                v = __fma_rn(x2, p.seg_coef[2], __fma_rn(x0, p.seg_coef[0], __dmul_rn(x1, p.seg_coef[1])));
            }
        }
        v = __dadd_rn(__dsub_rn(v, p.seg_off), p.seg_off);  // decision_function(X) + offset_
        if (p.out_map) p.out_map[(size_t)b * p.npix + i] = v;
        if (p.acc_map) p.acc_map[(size_t)b * p.npix + i] = v;
    }
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        double x[3] = {0.0, 0.0, 0.0};
        for (int m = 0; m < p.n_modal; ++m) {
            const float sm = __fmul_rn(p.s_lambda[m], p.tails[m][b].s);
            p.out_s_modal[b * 3 + m] = sm;
            x[m] = (double)sm;
        }
        double v = __dmul_rn(x[0], p.det_coef[0]);  // a single row goes through ddot: sequential fma over the columns
        for (int m = 1; m < p.n_modal; ++m) v = __fma_rn(x[m], p.det_coef[m], v);
        v = __dadd_rn(__dsub_rn(v, p.det_off), p.det_off);
        p.out_s[b] = v;
        if (p.acc_s) p.acc_s[b] = v;
    }
}

void api_prefer_carveout_fuse() { CMDB_PREFER_MAX_SMEM(fuse_head_kernel); }

}  // namespace cmdb

using namespace cmdb;

extern "C" {

int cmdb_project(cmdb_bank *b, const int32_t *indptr, const int32_t *indices, const double *data, int d_proj, int64_t row0,
                 int64_t n_rows, double *out_host) {
    CMDB_REQUIRE(b && out_host && row0 >= 0 && n_rows > 0 && row0 + n_rows <= b->rows, CMDB_ERR_INVALID,
                 "cmdb_project: bad row range");
    CMDB_REQUIRE(d_proj > 0, CMDB_ERR_INVALID, "cmdb_project: d_proj must be positive");
    CMDB_CUDA(cudaSetDevice(b->device));
    Buffer<double> z;
    CMDB_CUDA(z.alloc((size_t)n_rows * d_proj));
    CMDB_CHECK(project_rows(b, b->data + row0 * b->dim, n_rows, b->dim, indptr, indices, data, d_proj, z));
    CMDB_CUDA(cudaMemcpy(out_host, z, sizeof(double) * (size_t)n_rows * d_proj, cudaMemcpyDeviceToHost));
    return CMDB_OK;
}

static int coreset_impl(cmdb_bank *b, int64_t n_select, const int32_t *indptr, const int32_t *indices, const double *data,
                        int d_proj, int dtype_mode, int64_t *out_idx_host, const int64_t *force_idx, void *out_min_last,
                        ShardCtx *sh = nullptr, bool force_mind_global = false) {
    CMDB_REQUIRE(b && out_idx_host, CMDB_ERR_INVALID, "cmdb_coreset_select: NULL argument");
    CMDB_REQUIRE(b->rows > 0, CMDB_ERR_STATE, "cmdb_coreset_select: bank is empty");
    const int64_t n_total = sh ? sh->n_total : b->rows;
    CMDB_REQUIRE(n_select >= 1 && n_select <= n_total, CMDB_ERR_INVALID, "cmdb_coreset_select: n_select=%lld not in [1,%lld]",
                 (long long)n_select, (long long)n_total);
    CMDB_REQUIRE(d_proj >= 0 && d_proj <= b->dim, CMDB_ERR_INVALID,
                 "cmdb_coreset_select: d_proj=%d exceeds dim=%d (sklearn raises ValueError here; pass 0 to skip the projection)",
                 d_proj, b->dim);
    CMDB_CUDA(cudaSetDevice(b->device));
    const int d = d_proj > 0 ? d_proj : b->dim;
    // The kernels' 16-byte vector loads assume that address alignment follows the alignment class they compute for a
    // row.  The row-sharded loop (world > 1) computes it from the GLOBAL row, so the shard's projected rows start
    // (row_offset*d) & 3 elements past a 32-byte boundary (see coreset_greedy_dev).  Every other call runs with
    // row_offset 0 -- also on a handle whose row_offset is set -- and its rows start on the boundary.
    const bool sharded = sh && sh->world > 1;
    const int pad = sharded ? (int)((b->row_offset * d) & 3) : 0;
    Buffer<double> z_alloc;
    CMDB_CUDA(z_alloc.alloc((size_t)b->rows * d + 4));
    double *z = z_alloc + pad;
    if (d_proj > 0) {
        CMDB_CHECK(project_rows(b, b->data, b->rows, b->dim, indptr, indices, data, d_proj, z));
    } else {
        // features.py:369-370: projection skipped, the float32 bank itself is used
        f32_to_f64_kernel<<<b->num_sms * 4, 512, 0, b->handle_stream()>>>(b->data, (long long)b->rows * d, z);
        CMDB_CUDA(cudaGetLastError());
    }
    return coreset_greedy_dev(b, z, b->rows, d, n_select, dtype_mode, out_idx_host, force_idx, out_min_last, sh,
                              force_mind_global);
}

int cmdb_coreset_select(cmdb_bank *b, int64_t n_select, const int32_t *indptr, const int32_t *indices, const double *data,
                        int d_proj, int dtype_mode, int64_t *out_idx_host) {
    return coreset_impl(b, n_select, indptr, indices, data, d_proj, dtype_mode, out_idx_host, nullptr, nullptr);
}

// test hook (not in the public header): teacher forcing, the final min-distance vector, and (mind_global != 0) the
// min-distance vector kept in global memory at any bank size
int cmdb_coreset_select_debug(cmdb_bank *b, int64_t n_select, const int32_t *indptr, const int32_t *indices,
                              const double *data, int d_proj, int dtype_mode, int64_t *out_idx_host,
                              const int64_t *force_idx_host, void *out_min_last_host, int mind_global) {
    return coreset_impl(b, n_select, indptr, indices, data, d_proj, dtype_mode, out_idx_host, force_idx_host,
                        out_min_last_host, nullptr, mind_global != 0);
}

// host-only test hook (not in the public header): the coreset kernel's rows per CTA on num_sms SMs and whether their
// min-distances live in shared memory (1) or global memory (0) -- the rule launch_coreset applies
int cmdb_debug_coreset_plan(int num_sms, int64_t N, int d, int dtype_mode, int64_t *rows_per_cta, int *mind_in_smem) {
    return coreset_plan_info(num_sms, N, d, dtype_mode, rows_per_cta, mind_in_smem);
}

size_t cmdb_coreset_mailbox_bytes(int world, int d_proj_max) {
    (void)world, (void)d_proj_max;
    return kCommHeaderBytes;  // flags + key slots; the replica of the projected bank follows (cmdb_coreset_comm_bytes)
}

size_t cmdb_coreset_comm_bytes(int world, int d_proj, int64_t n_total_rows, int dtype_mode) {
    (void)world;
    const size_t es = dtype_mode == CMDB_CORESET_FP16 ? sizeof(__half) : sizeof(double);
    return kCommHeaderBytes + es * (size_t)std::max<int64_t>(n_total_rows, 1) * (size_t)std::max(d_proj, 1) + 256;
}

int cmdb_coreset_select_sharded(cmdb_bank *b, cmdb_comm *comm, int64_t n_total_rows, int64_t n_select, const int32_t *indptr,
                                const int32_t *indices, const double *data, int d_proj, int dtype_mode, const double *z0_host,
                                int64_t *out_idx_host) {
    CMDB_REQUIRE(b && comm && z0_host && out_idx_host, CMDB_ERR_INVALID, "cmdb_coreset_select_sharded: NULL argument");
    CMDB_REQUIRE(d_proj > 0, CMDB_ERR_UNSUPPORTED, "cmdb_coreset_select_sharded: needs a projection (d_proj > 0)");
    ShardCtx sh{};
    size_t mb_bytes = 0;
    unsigned char *local = nullptr;
    CMDB_CHECK(comm_info(comm, &sh.rank, &sh.world, &local, sh.peers, &mb_bytes));
    sh.row_offset = b->row_offset, sh.n_total = n_total_rows, sh.z0_host = z0_host;
    sh.comm_bytes = mb_bytes;
    CMDB_REQUIRE(mb_bytes >= cmdb_coreset_comm_bytes(sh.world, d_proj, n_total_rows, dtype_mode), CMDB_ERR_INVALID,
                 "cmdb_coreset_select_sharded: the peer buffer has %zu bytes, need %zu (cmdb_coreset_comm_bytes)", mb_bytes,
                 cmdb_coreset_comm_bytes(sh.world, d_proj, n_total_rows, dtype_mode));
    CMDB_REQUIRE(b->row_offset + b->rows <= n_total_rows, CMDB_ERR_INVALID, "cmdb_coreset_select_sharded: shard exceeds n_total_rows");
    CMDB_CUDA(cudaSetDevice(b->device));
    return coreset_impl(b, n_select, indptr, indices, data, d_proj, dtype_mode, out_idx_host, nullptr, nullptr, &sh);
}

int cmdb_coreset_rownorms(int device, const void *z_host, const void *last_host, int64_t n_rows, int d, int dtype_mode,
                          void *out_host) {
    return coreset_rownorms(device, z_host, last_host, n_rows, d, dtype_mode, out_host);
}

// Enqueue one sub-batch (<= score_max_batch images) of an opened call: staging, GEMM + certificate, maps, re-weighting and
// the device->host copies of the results (on the d2h stream, the maps as soon as the blur is done), then publish it.  No
// host sync.
static int submit_sub_batch(ScoreCall &c, const float *src, int is_device, int bc, int P, int fh, int fw, int out_hw,
                            unsigned want, bool host_maps = true) {
    cmdb_bank *b = c.b;
    const ScoreLayout &L = b->layout;
    ResultSlot &s = *c.slot;
    cudaStream_t st = c.stream;
    CMDB_CHECK(score_mark(c, CMDB_T_STAGE_IN, st));
    // this slot's q_f32 was last read by the batch submitted three calls ago
    CMDB_CHECK(score_local_min(c, src, is_device, bc, P, CMDB_T_GEMM, CMDB_T_REFINE, s.ev_compute));
    CMDB_CHECK(score_mark(c, CMDB_T_MAP, st));
    CMDB_CHECK(blur_batch(c, bc, fh, fw, out_hw));
    // min_val / min_idx / maps do not depend on the re-weighting: their copy overlaps it
    CMDB_CUDA(cudaEventRecord(b->ev_chunk[0], st));
    CMDB_CUDA(cudaStreamWaitEvent(b->d2h_stream, b->ev_chunk[0], 0));
    CMDB_CUDA(cudaMemcpyAsync(s.out_block_host + L.off_min_val, s.out_block + L.off_min_val,
                              (host_maps ? out_block_extent(b, bc, want) : L.off_map_out) - L.off_min_val, cudaMemcpyDeviceToHost,
                              b->d2h_stream));
    CMDB_CHECK(score_mark(c, CMDB_T_REWEIGHT, st));
    CMDB_CHECK(score_reweight(c, bc, P));
    CMDB_CHECK(score_mark(c, CMDB_T_OUT, st));
    CMDB_CUDA(cudaEventRecord(s.ev_compute, st));
    CMDB_CUDA(cudaStreamWaitEvent(b->d2h_stream, s.ev_compute, 0));
    CMDB_CUDA(cudaMemcpyAsync(s.out_block_host, s.out_block, L.off_min_val, cudaMemcpyDeviceToHost, b->d2h_stream));
    CMDB_CHECK(publish_call(c, bc, P, out_hw, want, host_maps, 0, 1));
    CMDB_CHECK(score_mark(c, CMDB_T_COUNT, b->d2h_stream));
    if (b->timing) b->ev_valid = true;  // only batches record the stage events, sharded rounds do not
    return CMDB_OK;
}

// Waits for a submitted batch or sharded round and fills outs[0 .. B): the scalars and per-patch arrays of every image,
// the maps of images img_first, img_first + img_step, ... (all of them for a batch; a sharded round only finished those).
static int wait_slot(cmdb_bank *b, int slot, cmdb_score_out *outs) {
    ResultSlot &s = b->slot[slot];
    ResultSlot::Pending &pd = s.pending;
    CMDB_CUDA(cudaEventSynchronize(s.ev_done));
    pd.active = false;
    if (b->shard_abort_host && *b->shard_abort_host) {
        set_error("a peer rank did not arrive at the exchange of a sharded round within the timeout (all ranks must submit "
                  "the same rounds in the same order)");
        return CMDB_ERR_CUDA;
    }
    for (int i = 0; i < pd.B; ++i) {
        const bool maps = i >= pd.img_first && (i - pd.img_first) % pd.img_step == 0;
        scatter_one(b, s.out_block_host, i, pd.P, pd.out_hw, outs + i, maps);
    }
    return CMDB_OK;
}

static int check_batch_args(cmdb_bank *b, const float *patches, int B, int P, int fh, int fw, int out_hw, const char *fn) {
    CMDB_CHECK(check_score_args(b, patches, B, P, fn));
    CMDB_REQUIRE(fh > 0 && fw > 0 && fh * fw == P, CMDB_ERR_INVALID, "%s: feature_map_dims %dx%d != P=%d", fn, fh, fw, P);
    CMDB_REQUIRE(out_hw >= 8 && out_hw <= 256, CMDB_ERR_INVALID, "%s: out_hw=%d not in [8,256]", fn, out_hw);
    return CMDB_OK;
}

int cmdb_score_batch(cmdb_bank *b, const float *patches, int B, int P, int fh, int fw, int out_hw, int patch_is_device,
                     cmdb_score_out *outs) {
    CMDB_REQUIRE(outs, CMDB_ERR_INVALID, "cmdb_score_batch: outs is NULL");
    CMDB_CHECK(check_batch_args(b, patches, B, P, fh, fw, out_hw, "cmdb_score_batch"));
    const int bc_max = score_max_batch(b);
    // sub-batches alternate between the two lanes: sub-batch k + 1 is enqueued before the host waits for sub-batch k
    int prev_slot = -1, prev_b0 = 0;
    for (int b0 = 0; b0 < B; b0 += bc_max) {
        const int bc = std::min(bc_max, B - b0);
        ScoreCall c{};
        CMDB_CHECK(begin_call(b, bc, P, out_hw, "cmdb_score_batch", &c));
        CMDB_CHECK(submit_sub_batch(c, patches + (size_t)b0 * P * b->dim, patch_is_device, bc, P, fh, fw, out_hw,
                                    want_mask_of(outs + b0, bc)));
        if (prev_slot >= 0) CMDB_CHECK(wait_slot(b, prev_slot, outs + prev_b0));
        prev_slot = c.slot_idx, prev_b0 = b0;
    }
    if (prev_slot >= 0) CMDB_CHECK(wait_slot(b, prev_slot, outs + prev_b0));
    return CMDB_OK;
}

int cmdb_score_batch_submit(cmdb_bank *b, const float *patches, int B, int P, int fh, int fw, int out_hw, int patch_is_device,
                            unsigned want_maps, int64_t *out_ticket) {
    CMDB_REQUIRE(out_ticket, CMDB_ERR_INVALID, "cmdb_score_batch_submit: out_ticket is NULL");
    CMDB_CHECK(check_batch_args(b, patches, B, P, fh, fw, out_hw, "cmdb_score_batch_submit"));
    ScoreCall c{};
    CMDB_CHECK(begin_call(b, B, P, out_hw, "cmdb_score_batch_submit", &c));
    CMDB_CHECK(submit_sub_batch(c, patches, patch_is_device, B, P, fh, fw, out_hw, want_maps & 3u));
    *out_ticket = c.slot->pending.ticket;
    return CMDB_OK;
}

static int wait_ticket(cmdb_bank *b, int64_t ticket, cmdb_score_out *outs, const char *fn) {
    CMDB_REQUIRE(b && outs, CMDB_ERR_INVALID, "%s: NULL argument", fn);
    for (int slot = 0; slot < kResultSlots; ++slot)
        if (b->slot[slot].pending.active && b->slot[slot].pending.ticket == ticket) {
            CMDB_CUDA(cudaSetDevice(b->device));
            return wait_slot(b, slot, outs);
        }
    set_error("%s: ticket %lld is not outstanding", fn, (long long)ticket);
    return CMDB_ERR_STATE;
}

int cmdb_score_batch_wait(cmdb_bank *b, int64_t ticket, cmdb_score_out *outs) {
    return wait_ticket(b, ticket, outs, "cmdb_score_batch_wait");
}

int cmdb_score(cmdb_bank *b, const float *patch, int P, int fh, int fw, int out_hw, int patch_is_device,
               cmdb_score_out *out) {
    return cmdb_score_batch(b, patch, 1, P, fh, fw, out_hw, patch_is_device, out);
}

// Last phase of a sharded round (both forms): final scores from the summed neighbour distances, the maps of this rank's
// images, the result copies; publishes the round.
static int finish_round(const ScoreCall &c, const float *knn_d2_sum_device, int B, int P, int fh, int fw, int out_hw,
                        int img_first, int img_step, unsigned want_maps, int64_t *out_ticket) {
    cmdb_bank *b = c.b;
    const ScoreLayout &L = b->layout;
    ResultSlot &s = *c.slot;
    CMDB_CHECK(score_shard_final(c, B, knn_d2_sum_device));
    CMDB_CHECK(blur_batch(c, B, fh, fw, out_hw, img_first, img_step));
    CMDB_CUDA(cudaEventRecord(s.ev_compute, c.stream));
    CMDB_CUDA(cudaStreamWaitEvent(b->d2h_stream, s.ev_compute, 0));
    // scalar / per-patch prefix of ALL images in one copy, then the maps of the images this rank finished
    const size_t npix = (size_t)out_hw * out_hw;
    want_maps &= 3u;
    if (img_first == 0 && img_step == 1) {
        CMDB_CUDA(cudaMemcpyAsync(s.out_block_host, s.out_block, out_block_extent(b, B, want_maps), cudaMemcpyDeviceToHost, b->d2h_stream));
    } else {
        CMDB_CUDA(cudaMemcpyAsync(s.out_block_host, s.out_block, L.off_map_out, cudaMemcpyDeviceToHost, b->d2h_stream));
        for (int i = img_first; i < B; i += img_step) {
            const size_t o1 = L.off_map_out + sizeof(float) * L.map_stride * i, o2 = L.off_map_pre + sizeof(float) * L.map_stride * i;
            const size_t o3 = L.off_map_u8 + L.map_stride * i;
            CMDB_CUDA(cudaMemcpyAsync(s.out_block_host + o1, s.out_block + o1, sizeof(float) * npix, cudaMemcpyDeviceToHost, b->d2h_stream));
            if (want_maps & 1u) CMDB_CUDA(cudaMemcpyAsync(s.out_block_host + o2, s.out_block + o2, sizeof(float) * npix, cudaMemcpyDeviceToHost, b->d2h_stream));
            if (want_maps & 2u) CMDB_CUDA(cudaMemcpyAsync(s.out_block_host + o3, s.out_block + o3, npix, cudaMemcpyDeviceToHost, b->d2h_stream));
        }
    }
    CMDB_CHECK(publish_call(c, B, P, out_hw, want_maps, true, img_first, img_step));
    *out_ticket = s.pending.ticket;
    return CMDB_OK;
}

int cmdb_score_shard_min(cmdb_bank *b, const float *patches, int B, int P, int patch_is_device, int out_hw,
                         int64_t *keys_device) {
    CMDB_CHECK(check_score_args(b, patches, B, P, "cmdb_score_shard_min"));
    CMDB_REQUIRE(keys_device, CMDB_ERR_INVALID, "cmdb_score_shard_min: keys_device is NULL");
    CMDB_REQUIRE(out_hw >= 8 && out_hw <= 256, CMDB_ERR_INVALID, "cmdb_score_shard_min: out_hw=%d not in [8,256]", out_hw);
    // the round runs on the lane that cmdb_bank_stream returns before this call; with the submit / wait finish up to three
    // rounds may be outstanding (three result slots on the two lanes)
    ScoreCall c{};
    CMDB_CHECK(begin_call(b, B, P, out_hw, "cmdb_score_shard_min", &c));
    c.sq_min = true;   // the keys carry d^2
    CMDB_CHECK(score_local_min(c, patches, patch_is_device, B, P, -1, -1, c.slot->ev_compute));
    pack_keys_kernel<<<(B * P + 255) / 256, 256, 0, c.stream>>>(c.min_val, c.min_idx, B * P, (long long *)keys_device);
    CMDB_CUDA(cudaGetLastError());
    b->round = cmdb_bank::Round{true, c.lane_idx, c.slot_idx};
    return CMDB_OK;  // stream-ordered on the round's lane (cmdb_bank_stream): run the collective there
}

int cmdb_score_shard_lookup(cmdb_bank *b, const int64_t *reduced_keys_device, int B, int P, float *knn_d2_contrib_device) {
    CMDB_CHECK(check_score_args(b, reduced_keys_device, B, P, "cmdb_score_shard_lookup"));
    CMDB_REQUIRE(b->round.open, CMDB_ERR_STATE, "cmdb_score_shard_lookup: no open round (call cmdb_score_shard_min first)");
    CMDB_REQUIRE(knn_d2_contrib_device && B * P <= b->layout.cap_p && B <= b->layout.cap_b, CMDB_ERR_INVALID,
                 "cmdb_score_shard_lookup: bad arguments");
    CMDB_REQUIRE(b->knn_table && b->knn_rows >= b->row_offset + b->fin_rows, CMDB_ERR_STATE,
                 "cmdb_score_shard_lookup: install the replicated neighbour table first (cmdb_bank_set_knn_table)");
    CMDB_CUDA(cudaSetDevice(b->device));
    const ScoreCall c = score_call(b, b->round.lane, b->round.slot);
    CMDB_CUDA(cudaMemsetAsync(c.lane->s_key, 0, sizeof(unsigned long long) * B, c.stream));
    unpack_keys_kernel<<<(B * P + 255) / 256, 256, 0, c.stream>>>((const long long *)reduced_keys_device, B * P, P, c.min_val,
                                                                  c.min_idx, c.lane->s_key);
    CMDB_CHECK(score_select(c, B, P, false));  // m_test, s*, s_idx, m_star_row (a global row: no bank access needed)
    return score_shard_lookup(c, B, knn_d2_contrib_device);
}

int cmdb_score_shard_finish_submit(cmdb_bank *b, const float *knn_d2_sum_device, int B, int P, int fh, int fw, int out_hw,
                                   int img_first, int img_step, unsigned want_maps, int64_t *out_ticket) {
    CMDB_CHECK(check_score_args(b, knn_d2_sum_device, B, P, "cmdb_score_shard_finish_submit"));
    CMDB_REQUIRE(b->round.open, CMDB_ERR_STATE, "cmdb_score_shard_finish_submit: no open round (call cmdb_score_shard_min first)");
    CMDB_REQUIRE(out_ticket && fh > 0 && fw > 0 && fh * fw == P && B * P <= b->layout.cap_p && B <= b->layout.cap_b, CMDB_ERR_INVALID,
                 "cmdb_score_shard_finish_submit: bad arguments");
    CMDB_REQUIRE((size_t)out_hw * out_hw == b->layout.map_stride, CMDB_ERR_INVALID,
                 "cmdb_score_shard_finish_submit: out_hw differs from cmdb_score_shard_min");
    CMDB_REQUIRE(img_first >= 0 && img_step >= 1, CMDB_ERR_INVALID, "cmdb_score_shard_finish_submit: bad image subset");
    CMDB_REQUIRE(!b->slot[b->round.slot].pending.active, CMDB_ERR_STATE,
                 "cmdb_score_shard_finish_submit: this round's slot is still outstanding");
    CMDB_CUDA(cudaSetDevice(b->device));
    CMDB_CHECK(finish_round(score_call(b, b->round.lane, b->round.slot), knn_d2_sum_device, B, P, fh, fw, out_hw, img_first,
                            img_step, want_maps, out_ticket));
    b->round.open = false;
    return CMDB_OK;
}

// ---- NCCL-free sharded rounds: the two exchanges go through peer-mapped memory (cmdb_comm), fused into the kernels ----

int cmdb_bank_attach_comm(cmdb_bank *b, cmdb_comm *comm) {
    CMDB_REQUIRE(b, CMDB_ERR_INVALID, "cmdb_bank_attach_comm: bank is NULL");
    CMDB_REQUIRE(!b->any_pending(), CMDB_ERR_STATE, "cmdb_bank_attach_comm: a submitted round is outstanding");
    if (!comm) {
        b->comm = nullptr;
        return CMDB_OK;
    }
    int rank = 0, world = 1;
    size_t bytes = 0;
    unsigned char *local = nullptr, *peers[kMaxRanks];
    CMDB_CHECK(comm_info(comm, &rank, &world, &local, peers, &bytes));
    CMDB_REQUIRE(bytes >= kCommHeaderBytes, CMDB_ERR_INVALID, "cmdb_bank_attach_comm: the peer buffer has %zu bytes, need >= %zu", bytes,
                 (size_t)kCommHeaderBytes);
    CMDB_CUDA(cudaSetDevice(b->device));
    if (!b->shard_ctr) {   // the exchange buffers go to the handle only once all of them exist
        Buffer<unsigned int> ctr;
        Buffer<float> d2;
        Buffer<unsigned int, Mem::Mapped> abort_host;
        unsigned int *abort_dev = nullptr;
        CMDB_CUDA(ctr.alloc(4));
        CMDB_CUDA(cudaMemset(ctr, 0, 4 * sizeof(unsigned int)));
        CMDB_CUDA(d2.alloc(2 * kShardSlots * kShardD2Cap));
        CMDB_CUDA(abort_host.alloc(1));
        *abort_host = 0u;
        CMDB_CUDA(cudaHostGetDevicePointer(&abort_dev, abort_host, 0));
        b->shard_ctr = std::move(ctr), b->shard_d2 = std::move(d2), b->shard_abort_host = std::move(abort_host);
        b->shard_abort_dev = abort_dev;
    }
    b->comm = comm;   // last: a failed attach leaves the handle as it was
    return CMDB_OK;
}

int cmdb_score_shard_round_submit(cmdb_bank *b, const float *patches, int B, int P, int fh, int fw, int out_hw, int patch_is_device,
                                  int img_first, int img_step, unsigned want_maps, int64_t *out_ticket) {
    CMDB_CHECK(check_score_args(b, patches, B, P, "cmdb_score_shard_round_submit"));
    CMDB_REQUIRE(b->comm, CMDB_ERR_STATE, "cmdb_score_shard_round_submit: attach the peer buffers first (cmdb_bank_attach_comm)");
    CMDB_REQUIRE(b->knn_table && b->knn_rows >= b->row_offset + b->fin_rows, CMDB_ERR_STATE,
                 "cmdb_score_shard_round_submit: install the replicated neighbour table first (cmdb_bank_set_knn_table)");
    CMDB_REQUIRE(out_ticket && fh > 0 && fw > 0 && fh * fw == P && out_hw >= 8 && out_hw <= 256 && img_first >= 0 && img_step >= 1,
                 CMDB_ERR_INVALID, "cmdb_score_shard_round_submit: bad arguments");
    int rank = 0, world = 1;
    size_t bytes = 0;
    unsigned char *local = nullptr;
    PeerPtrs peers{};
    CMDB_CHECK(comm_info(b->comm, &rank, &world, &local, peers.p, &bytes));
    ScoreCall c{};
    CMDB_CHECK(begin_call(b, B, P, out_hw, "cmdb_score_shard_round_submit", &c));
    c.sq_min = true;   // the keys carry d^2
    CMDB_CHECK(score_local_min(c, patches, patch_is_device, B, P, -1, -1, c.slot->ev_compute));
    const unsigned long long epoch = comm_next_score_epoch(b->comm);  // per buffer, not per bank: several banks may share it
    const int xslot = (int)(epoch % kShardSlots);
    CMDB_CHECK(score_shard_exchange_keys(c, B, P, peers, world, rank, xslot, epoch));
    CMDB_CHECK(score_select(c, B, P, false));
    float *contrib = b->shard_d2 + xslot * kShardD2Cap, *d2_sum = b->shard_d2 + (kShardSlots + xslot) * kShardD2Cap;
    CMDB_CHECK(score_shard_lookup(c, B, contrib));
    CMDB_CHECK(score_shard_exchange_d2(c, B, peers, world, rank, xslot, epoch, contrib, d2_sum));
    return finish_round(c, d2_sum, B, P, fh, fw, out_hw, img_first, img_step, want_maps, out_ticket);
}

int cmdb_score_shard_wait(cmdb_bank *b, int64_t ticket, cmdb_score_out *outs) {
    return wait_ticket(b, ticket, outs, "cmdb_score_shard_wait");
}

int cmdb_bank_read_device(cmdb_bank *b, int64_t row0, int64_t n_rows, float *out_device) {
    CMDB_REQUIRE(b && out_device && row0 >= 0 && n_rows >= 0 && row0 + n_rows <= b->rows, CMDB_ERR_INVALID,
                 "cmdb_bank_read_device: rows [%lld,%lld) outside [0,%lld)", (long long)row0, (long long)(row0 + n_rows),
                 b ? (long long)b->rows : 0LL);
    if (n_rows == 0) return CMDB_OK;
    CMDB_CUDA(cudaSetDevice(b->device));
    CMDB_CUDA(cudaMemcpyAsync(out_device, b->data + row0 * b->dim, sizeof(float) * (size_t)n_rows * b->dim, cudaMemcpyDeviceToDevice,
                              b->handle_stream()));
    CMDB_CUDA(cudaStreamSynchronize(b->handle_stream()));
    return CMDB_OK;
}

// test hook (not in the public header): the GEMM epilogue's per-CTA top-2 lists of the last call, [n_cta][n_q][4] floats
int cmdb_debug_read_candidates(cmdb_bank *b, float *out_host, int n_cta, int n_q) {
    CMDB_REQUIRE(b && out_host && n_cta >= 1 && n_cta <= 2 * b->num_sms && n_q >= 1 && n_q <= b->layout.cap_p, CMDB_ERR_INVALID,
                 "cmdb_debug_read_candidates: bad arguments");
    const Lane &l = b->lane[b->last_lane];   // the lists of the most recent call
    CMDB_CUDA(cudaSetDevice(b->device));
    CMDB_CUDA(cudaStreamSynchronize(l.stream));
    CMDB_CUDA(cudaMemcpy2D(out_host, sizeof(float4) * n_q, l.cand, sizeof(float4) * b->layout.cap_p, sizeof(float4) * n_q, n_cta,
                           cudaMemcpyDeviceToHost));
    return CMDB_OK;
}

// test hook (not in the public header): exact float32 scan of the whole bank with the arithmetic of the re-check kernels
// (warp_sqdist, lowest row on ties) -- what the certified pre-filter must reproduce bit for bit
int cmdb_debug_exact_min(cmdb_bank *b, const float *patch_host, int P, float *min_val_out, int64_t *min_idx_out) {
    CMDB_REQUIRE(b && patch_host && min_val_out && min_idx_out && P >= 1 && b->finalized, CMDB_ERR_INVALID, "cmdb_debug_exact_min: bad arguments");
    CMDB_CUDA(cudaSetDevice(b->device));
    Buffer<float> q;
    Buffer<unsigned long long> keys;
    std::vector<unsigned long long> h((size_t)P);
    CMDB_CUDA(q.alloc((size_t)P * b->dim));
    CMDB_CUDA(keys.alloc(P));
    cudaStream_t st = b->handle_stream();
    CMDB_CUDA(cudaMemcpyAsync(q, patch_host, sizeof(float) * (size_t)P * b->dim, cudaMemcpyHostToDevice, st));
    CMDB_CHECK(score_exact_scan(b, st, q, P, keys));
    CMDB_CUDA(cudaMemcpyAsync(h.data(), keys, sizeof(unsigned long long) * (size_t)P, cudaMemcpyDeviceToHost, st));
    CMDB_CUDA(cudaStreamSynchronize(st));
    for (int i = 0; i < P; ++i) {
        const unsigned int bits = (unsigned int)(h[i] >> 32);
        float d2;
        memcpy(&d2, &bits, sizeof(d2));
        min_val_out[i] = sqrtf(d2);
        min_idx_out[i] = (int64_t)(h[i] & 0xffffffffULL) + b->row_offset;
    }
    return CMDB_OK;
}

// host-only test hooks (not in the public header): the GEMM's tile-schedule stride and the fallback-tier rule
int cmdb_debug_tile_stride(int mt, int G) { return tile_stride(mt, G); }

// host-only test hook (not in the public header): the N tiles the exact rescan visits for (M tile mtile of a batch whose
// first-pass GEMM ran in launches of chunk_tiles out of mt_total M tiles on num_sms CTAs, producer CTA c), in slot order --
// the schedules gemm_sched records, walked by rescan_tile.  One chunk (chunk_tiles == mt_total) is the walk of the
// re-weighting certificate over a launch of mt_total M tiles.
int cmdb_debug_producer_tiles(int num_sms, int nt, int chunk_tiles, int mt_total, int mtile, int c, int32_t *tiles, int cap,
                              int *n_out) {
    CMDB_REQUIRE(num_sms >= 1 && nt >= 1 && chunk_tiles >= 1 && chunk_tiles <= mt_total && mtile >= 0 && mtile < mt_total && c >= 0 &&
                     c < num_sms && tiles && n_out,
                 CMDB_ERR_INVALID, "cmdb_debug_producer_tiles: bad arguments");
    const int last_tiles = mt_total - (mt_total - 1) / chunk_tiles * chunk_tiles;
    const GemmSched full = gemm_sched(nt, chunk_tiles, num_sms, false);
    const GemmSched last = gemm_sched(nt, last_tiles, num_sms, false);
    int n = 0;
    for (int kt = 0; kt < producer_slots(full, last); ++kt) {
        const int t = rescan_tile(full, last, chunk_tiles, mt_total, mtile, c, kt);
        if (t >= nt) continue;
        CMDB_REQUIRE(n < cap, CMDB_ERR_CAPACITY, "cmdb_debug_producer_tiles: more than %d tiles", cap);
        tiles[n++] = t;
    }
    *n_out = n;
    return CMDB_OK;
}
int cmdb_debug_fallback_use_rescan(int fails, int pairs) { return fallback_use_rescan(fails, pairs) ? 1 : 0; }

// test hook (not in the public header): rows [r0, r0 + n) of the neighbour table as packed (d^2 bits << 32 | row) keys
int cmdb_debug_read_knn(cmdb_bank *b, unsigned long long *out_host, long long r0, long long n) {
    CMDB_REQUIRE(b && out_host && b->knn_table && r0 >= 0 && n >= 1 && r0 + n <= b->fin_rows, CMDB_ERR_INVALID,
                 "cmdb_debug_read_knn: bad arguments");
    CMDB_CUDA(cudaSetDevice(b->device));
    CMDB_CUDA(cudaMemcpy(out_host, b->knn_table + (size_t)r0 * 3, sizeof(unsigned long long) * 3 * (size_t)n, cudaMemcpyDeviceToHost));
    return CMDB_OK;
}


// ---- late-fusion head on the device -------------------------------------------------------------------------------

static size_t fused_off_modal(int cap_b) { return (sizeof(double) * cap_b + 255) & ~size_t(255); }
static size_t fused_off_map(int cap_b) { return fused_off_modal(cap_b) + ((sizeof(float) * 3 * cap_b + 255) & ~size_t(255)); }
constexpr int kFusedCapB = 32;

static int fused_alloc(cmdb_bank *b0, int out_hw) {
    cmdb_bank::Fused &f = b0->fused;
    const size_t need = fused_off_map(kFusedCapB) + sizeof(double) * (size_t)out_hw * out_hw * kFusedCapB;
    if (f.cap_bytes >= need) return CMDB_OK;
    CMDB_REQUIRE(!f.active[0] && !f.active[1], CMDB_ERR_STATE, "fused scoring: out_hw grows while a submitted batch is outstanding");
    for (int i = 0; i < 2; ++i) {
        CMDB_CUDA(f.dev[i].alloc(need));
        CMDB_CUDA(f.host[i].alloc(need));
        if (!f.ev_done[i]) CMDB_CUDA(f.ev_done[i].create());
    }
    f.cap_bytes = need;
    return CMDB_OK;
}

int cmdb_score_fused_batch_submit(cmdb_bank *const *banks, const float *const *patches, const int *P, const int *fh,
                                  const int *fw, int B, int out_hw, int patch_is_device, const cmdb_fusion_head *head,
                                  unsigned flags, int64_t *out_ticket) {
    CMDB_REQUIRE(banks && patches && P && fh && fw && head && out_ticket, CMDB_ERR_INVALID, "cmdb_score_fused_batch_submit: NULL argument");
    const int M = head->n_modal;
    CMDB_REQUIRE(M >= 1 && M <= 3, CMDB_ERR_INVALID, "cmdb_score_fused_batch_submit: n_modal=%d not in [1,3]", M);
    for (int m = 0; m < M; ++m) {
        CMDB_REQUIRE(banks[m], CMDB_ERR_INVALID, "cmdb_score_fused_batch_submit: banks[%d] is NULL", m);
        CMDB_REQUIRE(banks[m]->device == banks[0]->device, CMDB_ERR_INVALID, "cmdb_score_fused_batch_submit: all banks must live on one GPU");
        for (int k = 0; k < m; ++k)
            CMDB_REQUIRE(banks[k] != banks[m], CMDB_ERR_INVALID, "cmdb_score_fused_batch_submit: one handle per modality");
        CMDB_CHECK(check_batch_args(banks[m], patches[m], B, P[m], fh[m], fw[m], out_hw, "cmdb_score_fused_batch_submit"));
        CMDB_REQUIRE(B <= score_max_batch(banks[m]) && B <= kFusedCapB, CMDB_ERR_INVALID,
                     "cmdb_score_fused_batch_submit: batch=%d exceeds the per-call limit %d", B, std::min(kFusedCapB, score_max_batch(banks[m])));
    }
    cmdb_bank *b0 = banks[0];
    cmdb_bank::Fused &f = b0->fused;
    CMDB_CUDA(cudaSetDevice(b0->device));
    CMDB_CHECK(fused_alloc(b0, out_hw));
    const int fs = f.next_fs;   // two fused blocks: at most two fused batches are outstanding
    CMDB_REQUIRE(!f.active[fs], CMDB_ERR_STATE, "cmdb_score_fused_batch_submit: two fused batches are already outstanding; wait for one first");
    const int npix = out_hw * out_hw;
    const bool keep = (flags & CMDB_FUSED_KEEP_ON_DEVICE) != 0, host_maps = (flags & CMDB_FUSED_NO_HOST_MAPS) == 0;
    if (keep) {
        CMDB_REQUIRE(f.acc_maps && f.acc_npix == npix && f.acc_n + B <= f.acc_cap, CMDB_ERR_CAPACITY,
                     "cmdb_score_fused_batch_submit: device-side result store missing or full (%lld + %d > %lld); call cmdb_eval_reserve",
                     f.acc_n, B, f.acc_cap);
    }
    // every modality's lane and result slot first, so that a refused one leaves nothing enqueued
    ScoreCall calls[3] = {};
    for (int m = 0; m < M; ++m) CMDB_CHECK(begin_call(banks[m], B, P[m], out_hw, "cmdb_score_fused_batch_submit", &calls[m]));
    cudaStream_t st = calls[0].stream;   // the head runs on modality 0's lane
    FuseParams fp{};
    fp.n_modal = M, fp.B = B, fp.npix = npix;
    for (int m = 0; m < M; ++m) {
        ScoreCall &c = calls[m];
        CMDB_CHECK(submit_sub_batch(c, patches[m], patch_is_device, B, P[m], fh[m], fw[m], out_hw, 0u, false));
        f.banks[fs][m] = banks[m], f.slots[fs][m] = c.slot_idx;
        fp.maps[m] = c.map_out;
        fp.map_stride[m] = banks[m]->layout.map_stride;
        fp.tails[m] = c.tail;
        fp.s_lambda[m] = head->s_lambda[m], fp.smap_lambda[m] = head->smap_lambda[m];
        fp.det_coef[m] = head->detect_coef[m], fp.seg_coef[m] = head->seg_coef[m];
        if (m > 0) CMDB_CUDA(cudaStreamWaitEvent(st, c.slot->ev_compute, 0));
    }
    fp.det_off = head->detect_offset, fp.seg_off = head->seg_offset;
    unsigned char *blk = f.dev[fs];
    fp.out_s = reinterpret_cast<double *>(blk);
    fp.out_s_modal = reinterpret_cast<float *>(blk + fused_off_modal(kFusedCapB));
    fp.out_map = host_maps ? reinterpret_cast<double *>(blk + fused_off_map(kFusedCapB)) : nullptr;
    if (keep) {
        fp.acc_map = f.acc_maps + (size_t)f.acc_n * npix;
        fp.acc_s = f.acc_scores + f.acc_n;
        f.acc_n += B;
    }
    fuse_head_kernel<<<dim3((npix + 1023) / 1024, B), 256, 0, st>>>(fp);
    CMDB_CUDA(cudaGetLastError());
    // results of this slot: scalars (+ maps) on the d2h stream; the next batch's kernels may already run meanwhile
    CMDB_CUDA(cudaEventRecord(b0->ev_chunk[1], st));
    CMDB_CUDA(cudaStreamWaitEvent(b0->d2h_stream, b0->ev_chunk[1], 0));
    const size_t bytes = host_maps ? fused_off_map(kFusedCapB) + sizeof(double) * (size_t)npix * B : fused_off_map(kFusedCapB);
    CMDB_CUDA(cudaMemcpyAsync(f.host[fs], blk, bytes, cudaMemcpyDeviceToHost, b0->d2h_stream));
    CMDB_CUDA(cudaEventRecord(f.ev_done[fs], b0->d2h_stream));
    // the fuse kernel read the other banks' result blocks: their slots may only be reused after it (they wait on it through
    // the ticket: a slot is busy until cmdb_score_fused_batch_wait returned)
    f.active[fs] = true, f.n_modal[fs] = M, f.B[fs] = B, f.out_hw[fs] = out_hw;
    f.next_fs ^= 1;
    f.ticket[fs] = calls[0].slot->pending.ticket;
    *out_ticket = f.ticket[fs];
    return CMDB_OK;
}

int cmdb_score_fused_batch_wait(cmdb_bank *b0, int64_t ticket, cmdb_fused_out *outs) {
    CMDB_REQUIRE(b0 && outs, CMDB_ERR_INVALID, "cmdb_score_fused_batch_wait: NULL argument");
    cmdb_bank::Fused &f = b0->fused;
    for (int fs = 0; fs < 2; ++fs) {
        if (!f.active[fs] || f.ticket[fs] != ticket) continue;
        CMDB_CUDA(cudaSetDevice(b0->device));
        CMDB_CUDA(cudaEventSynchronize(f.ev_done[fs]));
        const int B = f.B[fs], M = f.n_modal[fs], npix = f.out_hw[fs] * f.out_hw[fs];
        std::vector<cmdb_score_out> tmp((size_t)B);
        for (int m = 0; m < M; ++m) {
            for (int i = 0; i < B; ++i) {
                tmp[i] = cmdb_score_out{};
                tmp[i].min_val = outs[i].min_val[m], tmp[i].min_idx = outs[i].min_idx[m];
            }
            CMDB_CHECK(wait_slot(f.banks[fs][m], f.slots[fs][m], tmp.data()));
        }
        const unsigned char *h = f.host[fs];
        const double *hs = reinterpret_cast<const double *>(h);
        const float *hm = reinterpret_cast<const float *>(h + fused_off_modal(kFusedCapB));
        const double *hmap = reinterpret_cast<const double *>(h + fused_off_map(kFusedCapB));
        for (int i = 0; i < B; ++i) {
            if (outs[i].s) *outs[i].s = hs[i];
            if (outs[i].s_modal)
                for (int m = 0; m < M; ++m) outs[i].s_modal[m] = hm[i * 3 + m];
            if (outs[i].s_map) memcpy(outs[i].s_map, hmap + (size_t)i * npix, sizeof(double) * npix);
        }
        f.active[fs] = false;
        return CMDB_OK;
    }
    set_error("cmdb_score_fused_batch_wait: ticket %lld is not outstanding", (long long)ticket);
    return CMDB_ERR_STATE;
}

int cmdb_score_fused_batch(cmdb_bank *const *banks, const float *const *patches, const int *P, const int *fh, const int *fw,
                           int B, int out_hw, int patch_is_device, const cmdb_fusion_head *head, unsigned flags,
                           cmdb_fused_out *outs) {
    CMDB_REQUIRE(banks && patches && P && head && outs && B >= 1, CMDB_ERR_INVALID, "cmdb_score_fused_batch: bad arguments");
    const int M = head->n_modal;
    CMDB_REQUIRE(M >= 1 && M <= 3, CMDB_ERR_INVALID, "cmdb_score_fused_batch: n_modal=%d not in [1,3]", M);
    int bc_max = kFusedCapB;
    for (int m = 0; m < M; ++m) {
        CMDB_REQUIRE(banks[m] && patches[m], CMDB_ERR_INVALID, "cmdb_score_fused_batch: NULL bank / patches");
        bc_max = std::min(bc_max, score_max_batch(banks[m]));
    }
    // sub-batches are pipelined: batch k + 1 is submitted before the host waits for batch k
    int64_t prev_ticket = 0;
    int prev_b0 = -1;
    for (int b0 = 0; b0 < B; b0 += bc_max) {
        const int bc = std::min(bc_max, B - b0);
        const float *pp[3] = {nullptr, nullptr, nullptr};
        for (int m = 0; m < M; ++m) pp[m] = patches[m] + (size_t)b0 * P[m] * banks[m]->dim;
        int64_t t = 0;
        CMDB_CHECK(cmdb_score_fused_batch_submit(banks, pp, P, fh, fw, bc, out_hw, patch_is_device, head, flags, &t));
        if (prev_b0 >= 0) CMDB_CHECK(cmdb_score_fused_batch_wait(banks[0], prev_ticket, outs + prev_b0));
        prev_ticket = t, prev_b0 = b0;
    }
    return cmdb_score_fused_batch_wait(banks[0], prev_ticket, outs + prev_b0);
}


// ---- device-side result store (SURVEY 8f-3): replaces pixel_preds.extend / predictions.append of 50 176 scalars per image
//      (multiple_features.py:996-1001); the fused maps stay in HBM until cmdb_eval_* consumes them ----

int cmdb_eval_reserve(cmdb_bank *b, int64_t n_images, int out_hw) {
    CMDB_REQUIRE(b && n_images >= 1 && out_hw >= 8 && out_hw <= 256, CMDB_ERR_INVALID, "cmdb_eval_reserve: bad arguments");
    cmdb_bank::Fused &f = b->fused;
    CMDB_REQUIRE(!f.active[0] && !f.active[1], CMDB_ERR_STATE, "cmdb_eval_reserve: a submitted batch is outstanding");
    CMDB_CUDA(cudaSetDevice(b->device));
    CMDB_CUDA(cudaStreamSynchronize(b->handle_stream()));
    f.acc_cap = f.acc_n = 0, f.acc_npix = out_hw * out_hw;
    CMDB_CUDA(f.acc_maps.alloc((size_t)n_images * f.acc_npix));
    CMDB_CUDA(f.acc_scores.alloc(n_images));
    f.acc_cap = n_images;
    return CMDB_OK;
}

int cmdb_eval_count(cmdb_bank *b, int64_t *out_n) {
    CMDB_REQUIRE(b && out_n, CMDB_ERR_INVALID, "cmdb_eval_count: bad arguments");
    *out_n = b->fused.acc_n;
    return CMDB_OK;
}

int cmdb_eval_reset(cmdb_bank *b) {
    CMDB_REQUIRE(b, CMDB_ERR_INVALID, "cmdb_eval_reset: bank is NULL");
    CMDB_REQUIRE(!b->fused.active[0] && !b->fused.active[1], CMDB_ERR_STATE, "cmdb_eval_reset: a submitted batch is outstanding");
    b->fused.acc_n = 0;
    return CMDB_OK;
}

int cmdb_eval_read(cmdb_bank *b, int64_t first, int64_t n, double *maps_host, double *scores_host) {
    cmdb_bank::Fused &f = b->fused;
    CMDB_REQUIRE(b && first >= 0 && n >= 0 && first + n <= f.acc_n, CMDB_ERR_INVALID, "cmdb_eval_read: images [%lld,%lld) outside [0,%lld)",
                 (long long)first, (long long)(first + n), (long long)f.acc_n);
    if (n == 0) return CMDB_OK;
    CMDB_CUDA(cudaSetDevice(b->device));
    if (maps_host)
        CMDB_CUDA(cudaMemcpyAsync(maps_host, f.acc_maps + (size_t)first * f.acc_npix, sizeof(double) * (size_t)n * f.acc_npix,
                                  cudaMemcpyDeviceToHost, b->handle_stream()));
    if (scores_host)
        CMDB_CUDA(cudaMemcpyAsync(scores_host, f.acc_scores + first, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost,
                                  b->handle_stream()));
    CMDB_CUDA(cudaStreamSynchronize(b->handle_stream()));
    return CMDB_OK;
}

int cmdb_upsample_blur(int device, const float *map_host, int fh, int fw, int out_hw, float *out_host, float *out_pre_host,
                       uint8_t *out_u8_host) {
    CMDB_REQUIRE(map_host && out_host && fh > 0 && fw > 0, CMDB_ERR_INVALID, "cmdb_upsample_blur: bad arguments");
    CMDB_REQUIRE(out_hw >= 8 && out_hw <= 256, CMDB_ERR_INVALID, "cmdb_upsample_blur: out_hw=%d not in [8,256]", out_hw);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        (void)cudaGetLastError();
        set_error("cmdb_upsample_blur: no CUDA device; this library has no CPU fallback");
        return CMDB_ERR_CUDA;
    }
    CMDB_CUDA(cudaSetDevice(device));
    const size_t npix = (size_t)out_hw * out_hw;
    Buffer<float> in, pre, o, mx;
    Buffer<unsigned char> u8, tmp;
    CMDB_CUDA(in.alloc(fh * fw));
    CMDB_CUDA(tmp.alloc(npix));
    CMDB_CUDA(mx.alloc(17));
    CMDB_CUDA(pre.alloc(npix));
    CMDB_CUDA(o.alloc(npix));
    CMDB_CUDA(u8.alloc(npix));
    CMDB_CUDA(cudaMemcpy(in, map_host, sizeof(float) * fh * fw, cudaMemcpyHostToDevice));
    CMDB_CHECK(upsample_blur_launch(nullptr, 1, 0, 1, npix, in, fh, fw, out_hw, pre, o, u8, tmp, mx, mx + 1));
    CMDB_CUDA(cudaMemcpy(out_host, o, sizeof(float) * npix, cudaMemcpyDeviceToHost));
    if (out_pre_host) CMDB_CUDA(cudaMemcpy(out_pre_host, pre, sizeof(float) * npix, cudaMemcpyDeviceToHost));
    if (out_u8_host) CMDB_CUDA(cudaMemcpy(out_u8_host, u8, npix, cudaMemcpyDeviceToHost));
    return CMDB_OK;
}

}  // extern "C"
