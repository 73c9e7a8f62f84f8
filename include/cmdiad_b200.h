/*
 * cmdiad_b200 -- C ABI of the B200-native (sm_100a) memory-bank anomaly-scoring path of evenrose/CMDIAD.
 *
 * The reference has no plugin/operator registry: the seam is a handful of Python methods on the `Features` classes
 * (feature_extractors/features.py, feature_extractors/multiple_features.py).  Each entry point below names the
 * reference lines it replaces; INTEGRATION.md shows the ctypes binding a maintainer adds on the reference side.
 *
 * Conventions
 *   - plain C, no torch types: pointers + sizes.  The caller owns every input/output buffer; the library owns only the
 *     opaque bank handle and the device memory behind it.
 *   - every function returns 0 on success or a negative cmdb_status; nothing throws across the ABI.
 *     cmdb_last_error() returns a thread-local, NUL-terminated description of the last failure on this thread.
 *   - `*_is_device` flags: 0 = the pointer is host memory (pageable or pinned), 1 = device memory on the bank's GPU.
 *     ORDERING CONTRACT for device pointers: the library reads them on the handle's own non-blocking stream
 *     (cmdb_bank_stream), which does NOT implicitly follow the caller's streams.  Before the call, the work that
 *     produces the buffer must either be complete or be ordered before that stream (record an event on the producer
 *     stream and cudaStreamWaitEvent it on cmdb_bank_stream; the Python wrapper does this with
 *     stream.wait_stream(torch.cuda.current_stream()) and by holding the tensor until the call has consumed it).  The buffer must stay valid until the
 *     call -- or, for submit / wait pairs, the matching wait -- has returned.
 *   - calls on one handle are serialised by the caller (the reference is single-threaded per method object); distinct
 *     handles may be used from different threads.  Each handle owns one CUDA stream; host-visible results are complete
 *     when the call returns.
 *   - there is no CPU fallback: on a machine without an sm_100 GPU every compute call fails with CMDB_ERR_CUDA.
 *   - indices are int64 and GLOBAL row numbers (shard row offset + local row) so that "ties -> lowest index" survives
 *     row-sharding across GPUs.
 */
#ifndef CMDIAD_B200_H
#define CMDIAD_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct cmdb_comm cmdb_comm; /* peer mailboxes of one rank for the row-sharded coreset loop (one process per GPU) */
typedef struct cmdb_bank cmdb_bank; /* one memory bank (patch_rgb_lib / patch_xyz_lib / patch_fusion_lib) on one GPU */

typedef enum cmdb_status {
    CMDB_OK = 0,
    CMDB_ERR_INVALID = -1,  /* bad argument (NULL, negative size, d_proj > dim, ...) */
    CMDB_ERR_CUDA = -2,     /* CUDA runtime/driver failure, or no sm_100 device */
    CMDB_ERR_STATE = -3,    /* call not valid in the bank's current state (e.g. score before finalize) */
    CMDB_ERR_CAPACITY = -4, /* append beyond capacity_rows */
    CMDB_ERR_UNSUPPORTED = -5
} cmdb_status;

/* coreset_dtype of the reference (main.py:151, features.py:388-395) */
#define CMDB_CORESET_FP16 0 /* 'FP16': half data, float accumulate (reference default) */
#define CMDB_CORESET_FP64 1 /* 'TF32': the reference only flips a matmul flag, the data stays float64 */

/* scoring implementation selector (cmdb_bank_set_option(CMDB_OPT_SCORE_IMPL)) */
#define CMDB_SCORE_TCGEN05 0 /* tcgen05/TMEM split-fp16 distance GEMM (default, the product path) */
#define CMDB_SCORE_SIMT 1    /* exact float32 scan of the whole bank on CUDA cores (warp_sqdist, lowest row on ties);
                                diagnostics and test reference */

#define CMDB_OPT_SCORE_IMPL 1
/* Mode of the distance GEMM behind calculate_dist (features.py:186-190):
 *  0 (default) CERTIFIED PRE-FILTER: one hi.hi MMA per K step (11-bit operands) finds candidates; a per-query error bound
 *              (Cauchy-Schwarz on the operand rounding + a model of the tensor-core accumulation) proves for each query
 *              that every bank row outside the re-checked candidate set is strictly farther in float32 than the row
 *              returned.  Where the certificate fails, the rows it could not exclude are rescanned exactly inside the same
 *              call: min_val / min_idx then equal an exact float32 scan of the whole bank, lowest row on ties.  Only when
 *              a call queues more than 16 384 unresolved (query, producer) pairs (banks dominated by rows float32 cannot
 *              tell apart) are the uncertified queries redone with mode 3 instead; cmdb_bank_score_stats reports the
 *              counts, and a bank where most queries end up there switches itself to mode 3 for the next 32 calls.
 *  3           FP32-equivalent split for every query: hi.hi + hi.lo + lo.hi, three MMAs per K step, exact re-check of the
 *              4 best candidates (no certificate: among more than 4 rows within float32 noise of the minimum it may return
 *              another one of them -- equal up to the resolution of a float32 |a|^2 + |b|^2 - 2ab evaluation, not necessarily the lowest row).
 *  1           uncertified hi.hi pre-filter + exact re-check of the 4 best candidates (diagnostics). */
#define CMDB_OPT_PREFILTER_TERMS 3
#define CMDB_OPT_TIMING 2 /* non-zero = record CUDA events between the stages of cmdb_score (see cmdb_bank_get_timings) */

/* stage indices of cmdb_bank_get_timings */
#define CMDB_T_STAGE_IN 0   /* patch copy + fp16 split of the queries */
#define CMDB_T_GEMM 1       /* tcgen05 distance GEMM + fused top-2 epilogue (or the exact CUDA-core scan) */
#define CMDB_T_REFINE 2     /* exact re-check -> min_val / min_idx / s_star */
#define CMDB_T_MAP 3        /* bilinear upsample + Gaussian blur (then the maps start their device -> host copy) */
#define CMDB_T_REWEIGHT 4   /* m_star selection, w_dist top-3 over the bank, w and s (overlaps the copy of the maps) */
#define CMDB_T_OUT 5        /* rest of the device -> host copies of the results */
#define CMDB_T_COUNT 6

int cmdb_version(void);
const char *cmdb_last_error(void);
/* number of visible sm_100 devices (0 and CMDB_OK when there is none) */
int cmdb_device_count(int *out_n);

/* ---- bank storage: replaces the Python-list banks and torch.cat (multiple_features.py:35,38; features.py:49-51) ---- */

/* Pre-allocates a row-major float32 [capacity_rows, dim] bank in HBM on `device`. dim must be a multiple of 64. */
int cmdb_bank_create(int device, int dim, int64_t capacity_rows, cmdb_bank **out);
void cmdb_bank_destroy(cmdb_bank *bank);
/* self.patch_*_lib.append(patch)  (multiple_features.py:35, 131, 217, 363-365, 607-609, 870-871) */
int cmdb_bank_append(cmdb_bank *bank, const float *rows, int64_t n_rows, int rows_is_device);
int cmdb_bank_rows(const cmdb_bank *bank, int64_t *out_rows);
int cmdb_bank_dim(const cmdb_bank *bank, int *out_dim);
/* Row-sharding (SURVEY 8e): this handle holds global rows [row_offset, row_offset + rows). Default offset 0. */
int cmdb_bank_set_row_offset(cmdb_bank *bank, int64_t row_offset);
int cmdb_bank_set_option(cmdb_bank *bank, int option, int value);
/* torch.mean / torch.std (unbiased) over ALL elements (multiple_features.py:39-40): float64 accumulation on the GPU, two
 * passes (sum, then sum of squared deviations from the mean) reduced in a fixed order, so repeated calls are bit-identical.
 * out_sum / out_sumsq (optional) return the float64 sum and sum of squares (the latter rebuilt as
 * sum((x - mean)^2) + sum * mean) so that shards can be combined on the host. */
int cmdb_bank_stats(cmdb_bank *bank, double *out_mean, double *out_std_unbiased, double *out_sum, double *out_sumsq);
/* lib = (lib - mean) / std in float32, in place (multiple_features.py:41); one IEEE subtract and one IEEE divide.
 * normalize, gather and finalize return CMDB_ERR_STATE while a submitted call (batch, round, fused batch) is outstanding. */
int cmdb_bank_normalize(cmdb_bank *bank, float mean, float std);
/* lib = lib[idx] (multiple_features.py:48): keeps n rows in the given order; idx are LOCAL row numbers. */
int cmdb_bank_gather(cmdb_bank *bank, const int64_t *idx_host, int64_t n);
/* copies rows [row0, row0+n_rows) back to the host (to refill self.patch_*_lib, which features.py:238-283 index) */
int cmdb_bank_read(cmdb_bank *bank, int64_t row0, int64_t n_rows, float *out_host);
/* the same into DEVICE memory on the bank's GPU (e.g. to all-gather the shards of a row-sharded bank over NCCL) */
int cmdb_bank_read_device(cmdb_bank *bank, int64_t row0, int64_t n_rows, float *out_device);
/* Builds the scoring layout (fp16 hi/lo split, row norms) for the current rows. Must precede cmdb_score*. */
int cmdb_bank_finalize(cmdb_bank *bank);
/* A handle has two compute lanes (stream + private scratch each); scoring calls alternate between them so that the tail of
 * one batch / round overlaps the distance GEMM of the next.  Everything else runs on lane 0.  cmdb_bank_stream: the
 * cudaStream_t the NEXT scoring call on this handle will run on, or during a sharded round the round's (order producer work /
 * collectives against it); cmdb_bank_lane_streams: both of them. */
int cmdb_bank_stream(cmdb_bank *bank, void **out_stream);
int cmdb_bank_lane_streams(cmdb_bank *bank, void **out_streams2);
/* milliseconds of each stage (CMDB_T_*) of the last cmdb_score call on this handle; needs CMDB_OPT_TIMING on.
 * out_ms: float [CMDB_T_COUNT].  Measured with CUDA events on the handle's stream. */
int cmdb_bank_get_timings(cmdb_bank *bank, float *out_ms);
/* Optional (SURVEY 8f-1): the three nearest bank rows of EVERY bank row, computed once after cmdb_bank_finalize with the
 * certified pre-filter GEMM of the bank against itself (exact keys, same order and ties as the per-image w_dist top-3 of
 * features.py:239-254, whose query m_star is always a bank row).  With the table the re-weighting of cmdb_score /
 * cmdb_score_batch is a lookup instead of a pass over the bank; results are unchanged.  Un-sharded banks only (the table
 * needs all rows on one GPU); freed by the next cmdb_bank_finalize. */
int cmdb_bank_build_knn(cmdb_bank *bank);
/* Row-sharded banks: the table itself is small (24 B per row: 4.8 MB at 200k rows, 96 MB at 4M), so every rank keeps a
 * REPLICATED copy covering all global rows while the bank rows stay sharded.  Building it: gather the shards into a
 * temporary un-sharded handle on every rank, cmdb_bank_build_knn_rows for the rows this rank owns (the R x R work is
 * split evenly over the ranks), cmdb_bank_read_knn, all-gather the slices (any transport), cmdb_bank_set_knn_table on
 * the sharded handle (Bank.build_knn_sharded does exactly this over NCCL).  Keys hold GLOBAL rows. */
int cmdb_bank_build_knn_rows(cmdb_bank *bank, int64_t row_first, int64_t n_rows);
int cmdb_bank_read_knn(cmdb_bank *bank, int64_t row_first, int64_t n_rows, uint64_t *out_keys /* [n_rows][3] */,
                       int out_is_device);
int cmdb_bank_set_knn_table(cmdb_bank *bank, const uint64_t *keys /* [n_rows_total][3] */, int64_t n_rows_total,
                            int keys_is_device);
/* statistics of the last scoring call on this handle (waits for the handle's stream): out6[0] = query rows, out6[1] = GEMM
 * mode that ran (0 / 1 / 3, see CMDB_OPT_PREFILTER_TERMS); mode 0 only: out6[2] = query rows the pre-filter could not
 * certify, out6[3] = (query, producer) pairs queued for the exact rescan, out6[4] = 1 if there were too many pairs and
 * the uncertified queries went through the 3-term GEMM instead; out6[5] = calls the adaptive mode will still run
 * directly in mode 3. */
int cmdb_bank_score_stats(cmdb_bank *bank, int64_t *out6);

/* ---- coreset: replaces Features.get_coreset_idx_randomp (features.py:360-425) ---- */

/*
 * Sparse random projection (features.py:365-366) followed by the greedy k-center loop (features.py:372-420), all on
 * the GPU in one persistent kernel.  The CSR matrix [d_proj, dim] is sklearn's SparseRandomProjection.components_
 * (float64 data, per-row indices in STORED order), generated on the host by the caller exactly as the reference does;
 * d_proj == 0 means "no projection" (the reference's ValueError branch, features.py:369-370).
 * out_idx_host: int64 [n_select], out_idx_host[0] == 0 always (features.py:372).  Indices are local rows.
 */
int cmdb_coreset_select(cmdb_bank *bank, int64_t n_select, const int32_t *csr_indptr, const int32_t *csr_indices,
                        const double *csr_data, int d_proj, int dtype_mode, int64_t *out_idx_host);

/*
 * Row-sharded coreset selection over the GPUs of one NVSwitch box (one process per GPU, SURVEY 8e).  Every rank holds a
 * contiguous block of bank rows (cmdb_bank_set_row_offset) and runs the same persistent kernel on its shard.  The ranks
 * share through peer-mapped buffers (CUDA IPC over NVLink, one per rank):
 *   - a REPLICA of the whole projected bank in the loop's storage type (half: 2 * n_total * d' bytes -- 120 MB at
 *     200k x 301, 3 GB at 4M x 375), filled once per call: every rank copies its projected slice into all peers' replicas;
 *   - key slots [parity][rank][CTA]: per pick every CTA of every GPU stores its candidate (value, global row) as
 *     self-flagged 8-byte words straight into all ranks' slots and polls the world x CTAs keys of its LOCAL buffer -- one
 *     NVLink hop per pick, no system-scope fence, no NCCL call, no host round trip; the winning row is then read from the
 *     local replica.
 * Setup, once:  cmdb_comm_create on every rank -> cmdb_comm_export -> all-gather the handles (any host transport) ->
 * cmdb_comm_import.  mailbox_bytes >= cmdb_coreset_comm_bytes(world, d_proj, n_total_rows, dtype_mode).
 * cmdb_coreset_select_sharded: z0_host = the float64 projection of GLOBAL row 0 (cmdb_project on the owning rank,
 * broadcast by the caller); n_total_rows = rows of all shards; out_idx_host gets the same n_select GLOBAL rows on every
 * rank, bit-identical to the single-GPU cmdb_coreset_select on the un-sharded bank, in both dtype modes.
 * All ranks must call it together (it waits for its peers inside the kernel, with a timeout).
 */
int cmdb_comm_create(int device, int rank, int world, size_t mailbox_bytes, cmdb_comm **out);
int cmdb_comm_handle_bytes(void);
int cmdb_comm_export(cmdb_comm *comm, void *handle_out);
int cmdb_comm_import(cmdb_comm *comm, const void *handles /* [world][cmdb_comm_handle_bytes()] */);
/* clears the local mailbox; every rank calls it, then the ranks barrier, before each cmdb_coreset_select_sharded */
int cmdb_comm_reset(cmdb_comm *comm);
void cmdb_comm_destroy(cmdb_comm *comm);
size_t cmdb_coreset_mailbox_bytes(int world, int d_proj_max); /* header: coreset key slots + the scoring exchange slots */
size_t cmdb_coreset_comm_bytes(int world, int d_proj, int64_t n_total_rows, int dtype_mode); /* + the replica */
int cmdb_coreset_select_sharded(cmdb_bank *bank, cmdb_comm *comm, int64_t n_total_rows, int64_t n_select,
                                const int32_t *csr_indptr, const int32_t *csr_indices, const double *csr_data, int d_proj,
                                int dtype_mode, const double *z0_host, int64_t *out_idx_host);

/* Projection only: out_host float64 [n_rows, d_proj] for rows [row0, row0+n_rows) (bit-exact with sklearn). */
int cmdb_project(cmdb_bank *bank, const int32_t *csr_indptr, const int32_t *csr_indices, const double *csr_data,
                 int d_proj, int64_t row0, int64_t n_rows, double *out_host);

/* One distance pass of the greedy loop (features.py:405) in the canonical reduction order, for parity pinning:
 * z [n_rows, d] and last [d] are half bits (dtype_mode FP16) or float64 (FP64); out has the same type, [n_rows]. */
int cmdb_coreset_rownorms(int device, const void *z_host, const void *last_host, int64_t n_rows, int d, int dtype_mode,
                          void *out_host);

/* ---- scoring: replaces Features.calculate_dist + compute_single_s_s_map (features.py:186-190, 225-297) ---- */

typedef struct cmdb_score_out {
    /* all pointers are HOST buffers owned by the caller; NULL = not wanted */
    float *s;            /* [1]  w * s_star                                   (features.py:290) */
    float *s_star;       /* [1]  max_p min_r dist                             (features.py:231) */
    int64_t *s_idx;      /* [1]  argmax_p, ties -> lowest p                   (features.py:228) */
    float *min_val;      /* [P]  min_r ||patch_p - bank_r||_2                 (features.py:227) */
    int64_t *min_idx;    /* [P]  argmin_r (global rows), ties -> lowest r     (features.py:227) */
    int64_t *nn_idx;     /* [3]  3 nearest bank rows of m_star, ascending     (features.py:254) */
    float *m_star_knn;   /* [2]  ||m_test - bank[nn_idx[1:]]||_2              (features.py:275-283) */
    float *w;            /* [1]  re-weighting factor                          (features.py:287) */
    float *s_map;        /* [out_hw*out_hw] upsampled + blurred map           (features.py:293-295) */
    float *s_map_pre;    /* [out_hw*out_hw] bilinear map before the blur      (features.py:294) */
    uint8_t *s_map_u8;   /* [out_hw*out_hw] the 8-bit image handed to the blur (utils/utils.py:82 ToPILImage) */
} cmdb_score_out;

/*
 * Scores one image's patches against the bank: dist = cdist(patch, bank), min/argmin, s*, m*, top-3 re-weighting,
 * bilinear upsample to out_hw x out_hw and the PIL-exact Gaussian blur (radius 4).  patch: float32 [P, dim], already
 * normalised by the caller ((patch - mean) / std, multiple_features.py:90); P == fh*fw (feature_map_dims).
 * The [P, R] distance matrix is never materialised.
 */
int cmdb_score(cmdb_bank *bank, const float *patch, int P, int fh, int fw, int out_hw, int patch_is_device,
               cmdb_score_out *out);

/* Pipelined form of cmdb_score_batch.  submit enqueues everything for one batch (B <= 32 images, <= 160 KB of m_star rows:
 * the limit cmdb_score_batch splits larger batches by) -- host->device staging, scoring, device->host copies into an
 * internal pinned block -- and returns without waiting; wait blocks until that batch is complete and fills outs[B].
 * Up to three batches may be outstanding per handle (three result blocks, two compute lanes with their own query blocks
 * and scratch): the result copy of batch k and the staging of batch k+1 overlap the kernels of the other lane, and with two
 * calls queued behind the running one the host's enqueue time never delays the next distance GEMM.  `patches` must stay valid until the
 * matching wait returns.  want_maps: bit 0 = outs[].s_map_pre will be requested, bit 1 = outs[].s_map_u8.
 * Results are identical to cmdb_score_batch.  Not combined with the sharded phases on the same handle. */
int cmdb_score_batch_submit(cmdb_bank *bank, const float *patches, int batch, int P, int fh, int fw, int out_hw,
                            int patch_is_device, unsigned want_maps, int64_t *out_ticket);
int cmdb_score_batch_wait(cmdb_bank *bank, int64_t ticket, cmdb_score_out *outs);

/*
 * Batch form: B images of P patches each, patches float32 [B, P, dim], outs[B].  One sweep of the distance GEMM and ONE
 * sweep of the bank for the re-weighting serve the whole batch (the reference scores train and test images one by one,
 * cmdiad_runner.py:58-65, 80-85; per-image results are identical to B calls of cmdb_score).  Large batches are
 * processed in internal sub-batches.
 */
int cmdb_score_batch(cmdb_bank *bank, const float *patches, int B, int P, int fh, int fw, int out_hw, int patch_is_device,
                     cmdb_score_out *outs);

/*
 * Query normalisation on the device: with enabled != 0 every scoring entry point of this handle takes RAW patches and
 * applies (patch - mean) / std in float32 (one IEEE subtract, one IEEE divide == torch's CPU result) right after staging
 * them, i.e. the first line of compute_s_s_map (multiple_features.py:90, 976-977) moves behind the ABI.
 */
int cmdb_bank_set_query_norm(cmdb_bank *bank, float mean, float std, int enabled);

/*
 * Late-fusion head on the device (SURVEY 8f-2): what compute_s_s_map does after compute_single_s_s_map
 * (multiple_features.py:986-994 and the five sibling classes) for up to 3 modalities:
 *     s      = detect_fuser.score_samples([[lambda_s[0] * s_0, lambda_s[1] * s_1, ...]])
 *     s_map  = seg_fuser.score_samples(stack_m(lambda_map[m] * s_map_m))            [out_hw^2], float64
 * with SGDOneClassSVM.score_samples(X) = (X @ coef_ - offset_) + offset_ evaluated in float64 on the float32 products
 * lambda * value exactly as sklearn does on the reference's float32 tensors (features.py:114-115, 352-358).
 */
typedef struct cmdb_fusion_head {
    int n_modal;             /* columns of s / s_map = number of bank handles of the call (1..3), in column order */
    float s_lambda[3];       /* args.{xyz,rgb,fusion}_s_lambda    (main.py:114-125) */
    float smap_lambda[3];    /* args.{xyz,rgb,fusion}_smap_lambda */
    double detect_coef[3];   /* detect_fuser.coef_ */
    double detect_offset;    /* detect_fuser.offset_ */
    double seg_coef[3];      /* seg_fuser.coef_ */
    double seg_offset;       /* seg_fuser.offset_ */
} cmdb_fusion_head;

typedef struct cmdb_fused_out {
    /* HOST buffers owned by the caller; NULL = not wanted */
    double *s;        /* [1]        fused image score  (multiple_features.py:990) */
    double *s_map;    /* [out_hw^2] fused pixel map    (multiple_features.py:992-994) */
    float *s_modal;   /* [n_modal]  lambda_s[m] * s_m: the row add_sample_to_late_fusion_mem_bank appends to s_lib */
    /* per-modality per-patch results, as in cmdb_score_out (optional) */
    float *min_val[3];
    int64_t *min_idx[3];
} cmdb_fused_out;

#define CMDB_FUSED_KEEP_ON_DEVICE 1u /* append the fused maps / scores to the handle's device-side result store (cmdb_eval_*) */
#define CMDB_FUSED_NO_HOST_MAPS 2u   /* do not copy the fused maps to the host (outs[].s_map is ignored) */

/*
 * Scores B images against n_modal banks (one handle per modality, all on the same GPU; patches[m]: float32
 * [B, P[m], dim_m]) and applies the late-fusion head.  The per-modality maps never leave HBM; per image one float64 map
 * and one float64 score travel to the host.  submit / wait follow cmdb_score_batch_submit / _wait (two FUSED batches may be
 * outstanding; B <= the per-call limit of every bank); cmdb_score_fused_batch = submit + wait, any B.
 * The ticket belongs to banks[0].
 */
int cmdb_score_fused_batch_submit(cmdb_bank *const *banks, const float *const *patches, const int *P, const int *fh,
                                  const int *fw, int B, int out_hw, int patch_is_device, const cmdb_fusion_head *head,
                                  unsigned flags, int64_t *out_ticket);
int cmdb_score_fused_batch_wait(cmdb_bank *bank0, int64_t ticket, cmdb_fused_out *outs);
int cmdb_score_fused_batch(cmdb_bank *const *banks, const float *const *patches, const int *P, const int *fh, const int *fw,
                           int B, int out_hw, int patch_is_device, const cmdb_fusion_head *head, unsigned flags,
                           cmdb_fused_out *outs);

/*
 * Device-side result store (SURVEY 8f-3).  The reference extends Python lists by 50 176 scalars per test image
 * (pixel_preds / predictions, multiple_features.py:996-1001) and evaluates them with sklearn / numpy on the host
 * (features.py:321-324, utils/au_pro_util.py:157-224).  With CMDB_FUSED_KEEP_ON_DEVICE the fused float64 maps and image
 * scores of every cmdb_score_fused_batch* call are appended, in call order, to a pre-allocated store on banks[0]'s GPU.
 */
int cmdb_eval_reserve(cmdb_bank *bank, int64_t n_images, int out_hw); /* (re)allocates and empties the store */
int cmdb_eval_reset(cmdb_bank *bank);                                 /* empties it */
int cmdb_eval_count(cmdb_bank *bank, int64_t *out_n_images);
int cmdb_eval_read(cmdb_bank *bank, int64_t first, int64_t n, double *maps_host /* [n, out_hw^2] or NULL */,
                   double *scores_host /* [n] or NULL */);

/*
 * Row-sharded scoring (one process per GPU, SURVEY 8e).  Every rank holds a contiguous block of bank rows
 * (cmdb_bank_set_row_offset), the REPLICATED neighbour table of all global rows (cmdb_bank_set_knn_table) and the full
 * batch of patches.  All buffers named *_device are device memory on the bank's GPU, owned by the caller (torch tensors),
 * so the collectives between the phases run on them directly.  A round scores B images (B <= 32 and B*dim*4 <= 160 KB)
 * in three phases with TWO small collectives; all phases of one round use the same B, P, out_hw:
 *   1. cmdb_score_shard_min            keys[b*P+p] = (float_bits(local min SQUARED distance) << 32) | global_row
 *      (non-negative, so integer MIN == argmin with lowest-global-row tie-break; squared, because sqrtf maps neighbouring
 *      float32 d^2 to one distance and the single bank's argmin is that of d^2)              -> all-reduce MIN (int64[B*P])
 *   2. cmdb_score_shard_lookup         decodes the reduced keys (min_val = sqrtf(d^2), min_idx, s*, s_idx, m_star row), reads the three
 *      nearest rows of m_star from the table and writes, per image, the exact SQUARED distances ||m_test - bank[nn_k]||^2
 *      (k = 1, 2; features.py:275-283) for the neighbour rows this rank owns, 0 for the others     -> all-reduce SUM (float[B*2])
 *   3. cmdb_score_shard_finish_submit  m_star_knn = sqrt(sum), w, s for all images; upsample + blur + device->host copy of
 *      the maps of images img_first, img_first + img_step, ... (0, 1 = all images; rank, world = each rank finishes only
 *      its share); returns a ticket without waiting.
 *      cmdb_score_shard_wait(ticket, outs[B]) blocks until the round is complete: every outs[i] gets the scalars and
 *      per-patch arrays (replicated on all ranks), the maps are filled for the images this rank finished (the map buffers
 *      of the other outs[] entries are left untouched).
 * Phases 1 and 2 only enqueue work on the handle's stream (cmdb_bank_stream) and return; run the collectives on that same
 * stream.  Nothing synchronises the host between the phases, and three rounds can be outstanding per handle (the result
 * copy of round k and the host work for the next rounds overlap the kernels of the other lane).  cmdb_score_shard_min opens
 * the round and cmdb_score_shard_finish_submit closes it; phases 2 and 3 return CMDB_ERR_STATE when no round is open.
 * Results are bit-identical to cmdb_score_batch on the un-sharded bank.
 */
int cmdb_score_shard_min(cmdb_bank *bank, const float *patches, int B, int P, int patch_is_device, int out_hw,
                         int64_t *keys_device);
int cmdb_score_shard_lookup(cmdb_bank *bank, const int64_t *reduced_keys_device, int B, int P, float *knn_d2_contrib_device);
int cmdb_score_shard_finish_submit(cmdb_bank *bank, const float *knn_d2_sum_device, int B, int P, int fh, int fw, int out_hw,
                                   int img_first, int img_step, unsigned want_maps, int64_t *out_ticket);
int cmdb_score_shard_wait(cmdb_bank *bank, int64_t ticket, cmdb_score_out *outs);
/*
 * The same round WITHOUT NCCL: with a cmdb_comm attached (the peer-mapped buffers the sharded coreset loop uses; needs
 * >= cmdb_coreset_mailbox_bytes bytes) one call enqueues the whole round -- local min, exchange, lookup, exchange, finish --
 * and both exchanges are fused into the kernels around them: the pack kernel stores every rank's keys straight into the
 * round's slot of ALL ranks' buffers over NVLink and raises a flag (threadfence_system + release store by its last
 * block); the decode kernel waits for the world flags in its local buffer and takes the MIN while unpacking.  ~10 us per
 * exchange instead of two launches + an NCCL all-reduce (60 us at 8 ranks for the 98 KB of keys).  Collective: every
 * rank submits the same rounds in the same order; if a peer never arrived, cmdb_score_shard_wait and every later wait on
 * the handle return CMDB_ERR_CUDA.
 */
int cmdb_bank_attach_comm(cmdb_bank *bank, cmdb_comm *comm);
int cmdb_score_shard_round_submit(cmdb_bank *bank, const float *patches, int B, int P, int fh, int fw, int out_hw,
                                  int patch_is_device, int img_first, int img_step, unsigned want_maps, int64_t *out_ticket);

/*
 * Pixel-level evaluation of everything in the result store, on the device (features.py:321-324: pixel AUROC and the two
 * AU-PRO values of utils/au_pro_util.py:104-224).  One stable radix sort of all (score, label) pairs, then:
 *   out_two_u        exact integer 2U of the Mann-Whitney statistic (ties count 1/2): pixel AUROC = 2U / (2 n_pos n_neg),
 *                    what sklearn's roc_auc_score computes by trapezoids;
 *   out_thresholds   [n_thresholds] the anomaly-free scores at ranks ok_rank_pos_host[t] of their sorted order
 *                    (np.linspace(0, n_ok - 1, num, dtype=int), au_pro_util.py:176);
 *   out_component_le_counts [n_components][n_thresholds]  #{scores of ground-truth component c <= threshold t}
 *                    (GroundTruthComponent.compute_overlap, :44-49), out_component_sizes [n_components].
 * The counts are exact integers; the host finishes the PRO curve and its integral with the reference's own float64
 * operations (cmdiad_b200/metrics.py), so au_pro / au_pro_001 are bit-identical to the reference.
 * labels_host: int32 [n_images * out_hw^2], 0 = anomaly-free pixel, c in 1..n_components = pixel of ground-truth component
 * c (scipy.ndimage.label per mask with the 8-connectivity structure of au_pro_util.py:129, numbered through the set in
 * image order; the masks are host inputs of predict(), so labelling them stays on the host).
 */
int cmdb_eval_pixel_metrics(cmdb_bank *bank, const int32_t *labels_host, int64_t n_components, const int64_t *ok_rank_pos_host,
                            int n_thresholds, double *out_thresholds, int64_t *out_component_le_counts,
                            int64_t *out_component_sizes, uint64_t *out_two_u, int64_t *out_n_pos, int64_t *out_n_neg);

/* Stand-alone score-map post-processing (features.py:293-295, utils/utils.py:71-83): map [fh*fw] -> [out_hw^2]. */
int cmdb_upsample_blur(int device, const float *map_host, int fh, int fw, int out_hw, float *out_host,
                       float *out_pre_host, uint8_t *out_u8_host);

#ifdef __cplusplus
}
#endif
#endif /* CMDIAD_B200_H */
