// Shared declarations of the cmdiad_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include <cstdarg>
#include <cstdio>
#include <cstring>

#include "../../include/cmdiad_b200.h"

namespace cmdb {

void set_error(const char *fmt, ...);

#define CMDB_CUDA(expr)                                                                              \
    do {                                                                                             \
        cudaError_t _e = (expr);                                                                     \
        if (_e != cudaSuccess) {                                                                     \
            cmdb::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e));    \
            (void)cudaGetLastError();                                                                \
            return CMDB_ERR_CUDA;                                                                    \
        }                                                                                            \
    } while (0)

#define CMDB_CHECK(expr)           \
    do {                           \
        int _s = (expr);           \
        if (_s != CMDB_OK) return _s; \
    } while (0)

#define CMDB_REQUIRE(cond, status, ...)   \
    do {                                  \
        if (!(cond)) {                    \
            cmdb::set_error(__VA_ARGS__); \
            return status;                \
        }                                 \
    } while (0)

constexpr int kNumSMsDefault = 148;
constexpr int kMaxRanks = 8;         // GPUs of one NVSwitch box
constexpr int kScoreBN = 256;        // bank rows per GEMM tile
constexpr int kScoreBM = 128;        // query rows per GEMM tile
constexpr int kGemmEpiGroups = 2;    // epilogue warp groups per GEMM CTA: producers = groups * CTAs
constexpr int kResultSlots = 3;      // result blocks / outstanding submitted calls per handle (the compute lanes stay two)
constexpr int kMaxStageChunks = 4;   // host query batches are staged and multiplied in up to this many chunks
constexpr int kWorkCap = 16384;      // capacity of Lane::work_list
// Fallback tiers of the certified pre-filter.  Tier 1, exact rescan: ~R/296 rows x D x 4 B per (query, producer) pair, HBM
// bound (~0.32 us per pair at 200k x 768) -- RIGOROUS: the result equals the exact float32 scan, lowest row on ties.
// Tier 2, 3-term GEMM over the compacted uncertified queries + exact re-check of the 4 best candidates: at least one sweep
// of the hi + lo bank (~0.25 ms), then ~0.55 us per query -- cheaper when a call queues very many pairs, but NOT certified:
// among more than 4 rows within the float32 resolution of |a|^2 + |b|^2 - 2ab it may return another one of them (not
// necessarily the exact minimum / lowest row).  Round 1 picked the cheaper tier; round 2 keeps the contract instead: tier 1 whenever the
// pairs fit the work list (<= 5 ms of rescans in the worst case), tier 2 only beyond it (banks dominated by rows that
// float32 cannot tell apart, where the reference's own mm-form argmin is arbitrary as well).
__host__ __device__ inline bool fallback_use_rescan(int fails, int pairs) {
    (void)fails;
    return pairs <= kWorkCap;
}
constexpr int kScoreBK = 64;         // fp16 K elements per pipeline stage (one 128-byte swizzle row)

// Sizes of the scoring scratch of a handle (score_scratch_alloc), common to both lanes and all result slots.  The results
// of a call live in ONE device block (tail | min_val | min_idx | map_out | map_pre | map_u8) mirrored by a pinned host
// block, so a scoring call ends with a single device->host copy; the offsets below locate the sections.
struct ScoreLayout {
    int cap_p = 0;          // padded query-row capacity of a sub-batch (multiple of 128)
    int cap_b = 0;          // image capacity of a sub-batch
    size_t map_stride = 0;  // pixels reserved per image in the map sections
    size_t off_min_val = 0, off_min_idx = 0, off_map_out = 0, off_map_pre = 0, off_map_u8 = 0, out_block_bytes = 0;
    int n_topk_blocks = 0;  // blocks of reweight_kernel
};

// A compute lane: the streams a call runs on and every device buffer that lives only while a call computes.  Call k runs on
// lane k & 1, so the tail of a batch / round -- certificate, rescans, exchanges, re-weighting, maps -- overlaps the
// distance GEMM of the next one (the GEMM is one persistent CTA per SM; the small tail kernels fit beside it).
struct Lane {
    cudaStream_t stream = nullptr;
    cudaStream_t aux = nullptr;     // side stream of the (normally empty) tier-2 launches and the counters copy, beside the rescan
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    // CMDB_OPT_TIMING = 2 (diagnostics): this lane's stage marks and the four marks inside the refine stage (before / after
    // the certificate kernel, after the rescan, after the tier-2 launches), read by cmdb_debug_lane_timeline
    cudaEvent_t ev_tl[CMDB_T_COUNT + 1] = {};
    cudaEvent_t ev_dbg[4] = {};
    __half *q_hi = nullptr;         // [cap_p, D]  split-fp16 query operand
    __half *q_lo = nullptr;
    int *q_scale_exp = nullptr;     // device [cap_p]: per-row exponent e_q with q_hi + q_lo = q * 2^e_q
    float *q_norm = nullptr;        // [cap_p] ||q|| (rounded up)            -- certified pre-filter, score_tail.cu
    float *q_eps = nullptr;         // [cap_p] ||q - q_hi * 2^-e_q|| (rounded up)
    int *fail_list = nullptr;       // [cap_p] query rows whose pre-filter result could not be certified
    // device control block of the fallback: [0] uncertified queries, [1] (query, producer) pairs to rescan,
    // [2] rows of the 3-term GEMM fallback, [3] pairs of the exact rescan, [4] queries the rescan finishes
    // ([2..4] are derived from [0..1] by the last block of refine_cert_kernel: pairs that fit the work list -> rescan, more ->
    // GEMM), [5] / [6] last-block tickets of the certificate / rescan kernels; the per-image argmax keys (s_key) follow at
    // fail_ctl + 8 in the same allocation so that one memset clears both
    int *fail_ctl = nullptr;
    unsigned long long *s_key = nullptr;    // [cap_b] packed argmax key of min_val
    int *fail_count_host = nullptr; // pinned copy of [0..1] (statistics / adaptive mode)
    int2 *work_list = nullptr;      // [kWorkCap] (query row, producer) pairs whose producer may hide rows inside the band
    unsigned long long *best_key = nullptr;  // [cap_p] running exact (d^2 bits << 32 | row) of the uncertified queries
    unsigned int *done_counter = nullptr;  // last-block-done counter of reweight_kernel
    float4 *cand = nullptr;         // [n_ctas, cap_p] per-CTA running top-2 (val1, idx1, val2, idx2) of the GEMM epilogue
    unsigned char *map_tmp = nullptr;  // horizontally blurred 8-bit images between the two blur kernels
    float *map_max = nullptr;       // [cap_b] map maxima, then [cap_b][16] band maxima
    unsigned long long *topk_keys = nullptr;  // [n_blocks*3] per-block w_dist top-3 packed keys
    unsigned long long *top3 = nullptr;  // merged 3 smallest w_dist keys
    float *m_test = nullptr;        // [cap_b, D] patch[s_idx]
    float *m_star = nullptr;        // [cap_b, D] bank[min_idx[s_idx]]
    void *tmap_qhi = nullptr;       // host CUtensorMap objects for q_hi / q_lo
    void *tmap_qlo = nullptr;
};

// A result slot: what a submitted call holds until the caller has waited for it.  The slots cycle independently of the
// lanes (call k uses slot k % kResultSlots), so the results of calls k - 1 and k travel to the host / wait for the caller
// while call k + 1 is already enqueued, and its queries are staged while call k is still scored.
struct ResultSlot {
    float *q_f32 = nullptr;                 // [cap_p, D] normalised query patches
    unsigned char *out_block = nullptr;     // device result block (ScoreLayout)
    unsigned char *out_block_host = nullptr;  // its pinned mirror
    cudaEvent_t ev_done = nullptr;          // the block is in the pinned host memory
    cudaEvent_t ev_compute = nullptr;       // the kernels of the call that used the slot are done (q_f32 may be overwritten)
    struct Pending {
        bool active = false;
        int B = 0, P = 0, out_hw = 0;
        unsigned want = 0;
        bool host_maps = true;   // false: the per-modality maps stay in HBM (fused late-fusion head), only scalars travel
        int img_first = 0, img_step = 1;  // images whose maps were finished (a sharded round's rank: its share; a batch: all)
        long long ticket = 0;
    } pending;
};

}  // namespace cmdb

struct cmdb_bank {
    int device = 0;
    int dim = 0;
    int num_sms = cmdb::kNumSMsDefault;
    int64_t capacity = 0;
    int64_t rows = 0;
    int64_t row_offset = 0;
    int score_impl = CMDB_SCORE_TCGEN05;
    // distance GEMM mode: 0 = certified hi.hi pre-filter with FP32-equivalent fallback for uncertified queries (default),
    // 3 = FP32-equivalent split for every query, 1 = uncertified hi.hi pre-filter (diagnostics)
    int prefilter_terms = 0;
    // error-bound inputs of the certificate, true units, rounded up (cmdb_bank_finalize)
    float cert_bmax = 0.f;    // max ||b||
    float cert_eb_max = 0.f;  // max ||b - b_hi * 2^-scale_exp||
    unsigned int *cert_buf = nullptr;  // device [2]: the two maxima as float bits
    // optional table of the three nearest bank rows of every bank row, as packed (d^2 bits << 32 | row) keys
    // (cmdb_bank_build_knn; SURVEY 8f-1): turns the per-image w_dist pass into a lookup
    unsigned long long *knn_table = nullptr;  // [knn_rows][3]
    // rows the table covers: fin_rows for a table built on this handle (cmdb_bank_build_knn); the GLOBAL row count for a
    // replicated table installed on a row-sharded handle (cmdb_bank_set_knn_table)
    long long knn_rows = 0;
    // statistics of the last scoring call / adaptive fallback to the direct 3-term GEMM
    int64_t last_queries = 0;
    int last_mode = 0;           // GEMM mode the last call actually ran
    bool fail_pending = false;   // fail_count_host holds the count of a finished-or-in-flight call
    int direct_calls_left = 0;   // certified mode: calls to run directly with 3 terms before probing the pre-filter again
    // Scoring calls take the next of the two compute lanes and the next of the kResultSlots result slots (cmdb::ScoreCall,
    // api.cu).  Everything else -- append, read, statistics, normalize, gather, finalize, coreset, projection, evaluation --
    // runs on lane 0's stream (handle_stream()).
    cmdb::ScoreLayout layout;
    cmdb::Lane lane[2];
    cmdb::ResultSlot slot[cmdb::kResultSlots];
    int next_lane = 0;    // compute lane of the next scoring call (alternates)
    int next_slot = 0;    // result slot of the next scoring call (cycles through kResultSlots)
    int last_lane = 0;    // lane of the most recent scoring call or table build (cmdb_debug_read_candidates)
    // the sharded round opened by cmdb_score_shard_min and closed by cmdb_score_shard_finish_submit
    struct Round { bool open = false; int lane = 0, slot = 0; } round;
    int *last_fail_host = nullptr;   // pinned certificate counters of the most recent certified call (either lane)
    cudaStream_t copy_stream = nullptr;   // host -> device staging of query chunks, overlapped with the GEMM of earlier chunks
    cudaEvent_t ev_chunk[cmdb::kMaxStageChunks] = {};
    cudaStream_t d2h_stream = nullptr;    // device -> host copies of the results
    cudaEvent_t ev_fail = nullptr;        // the certificate counters of the last certified call are on the host
    cudaStream_t handle_stream() const { return lane[0].stream; }
    bool any_pending() const {  // a submitted call (batch, round, fused batch) still uses the handle's buffers
        for (const auto &s : slot)
            if (s.pending.active) return true;
        return fused.active[0] || fused.active[1];
    }
    // queries are normalised on the device right after staging: (q - q_mean) / q_std, one IEEE subtract + one IEEE divide
    // like the reference's torch expression (multiple_features.py:90, 976-977); cmdb_bank_set_query_norm
    bool q_norm_enabled = false;
    float q_mean = 0.f, q_std = 1.f;
    // late-fusion head on the device (cmdb_score_fused_batch*; this handle is modality 0 of the fused call): per slot the
    // fused float64 maps / image scores / lambda-scaled per-modality s in one device block mirrored by a pinned host block
    struct Fused {
        unsigned char *dev[2] = {nullptr, nullptr};
        unsigned char *host[2] = {nullptr, nullptr};
        size_t cap_bytes = 0;
        cudaEvent_t ev_done[2] = {};
        bool active[2] = {false, false};
        int next_fs = 0;   // fused block of the next fused call (two fused batches may be outstanding)
        int n_modal[2] = {0, 0}, B[2] = {0, 0}, out_hw[2] = {0, 0};
        cmdb_bank *banks[2][3] = {};
        int slots[2][3] = {};
        long long ticket[2] = {0, 0};
        // device-resident accumulation of the fused maps over predict calls (cmdb_eval_*; SURVEY 8f-3)
        double *acc_maps = nullptr;     // [acc_cap][npix]
        double *acc_scores = nullptr;   // [acc_cap]
        long long acc_cap = 0, acc_n = 0;
        int acc_npix = 0;
    } fused;
    long long ticket_counter = 0;
    cmdb_comm *comm = nullptr;             // peer buffers for NCCL-free sharded rounds (cmdb_bank_attach_comm; not owned)
    unsigned int *shard_ctr = nullptr;     // [0] device: last-block counter of the push kernels
    unsigned int *shard_abort_host = nullptr;  // pinned + mapped: set by a kernel whose peers never arrived
    unsigned int *shard_abort_dev = nullptr;   // device alias of shard_abort_host
    float *shard_d2 = nullptr;             // device [2][kShardD2Cap]: local contributions / sums of the neighbour distances
    float *data = nullptr;  // [capacity, dim] float32 row-major
    // scoring layout (cmdb_bank_finalize)
    bool finalized = false;
    int64_t fin_rows = 0;
    int64_t fin_rows_pad = 0;  // multiple of kScoreBN
    __half *hi = nullptr;      // [fin_rows_pad, dim] fp16(x * 2^scale_exp)
    __half *lo = nullptr;      // [fin_rows_pad, dim] fp16(x * 2^scale_exp - hi)
    float *norm = nullptr;     // [fin_rows_pad] ||x * 2^scale_exp||^2 ; +inf on padding rows
    int scale_exp = 0;
    void *tmap_hi = nullptr;  // host copies of the CUtensorMap objects (128 B each)
    void *tmap_lo = nullptr;
    void *tmap_hi2 = nullptr;  // box of 128 bank rows (CTA-pair kernels)
    void *tmap_lo2 = nullptr;
    int timing = 0;
    cudaEvent_t ev[CMDB_T_COUNT + 1] = {};
    bool ev_valid = false;
    // CMDB_OPT_TIMING = 2 (diagnostics): common time base of the lanes' stage events (Lane::ev_tl), so that the overlap of
    // the two lanes can be read (cmdb_debug_lane_timeline)
    cudaEvent_t ev_base = nullptr;
    double *stats_buf = nullptr;  // 2 + num_sms * 4 doubles on device (cmdb_bank_stats)
    unsigned int *absmax_buf = nullptr;
};

namespace cmdb {

// bank.cu
int bank_max_abs(cmdb_bank *b, const float *x, int64_t n, float *out_host);
int pick_scale_exp(float absmax);
void launch_normalize(cudaStream_t stream, int num_sms, float *x, int64_t n, float mean, float stdv);
void launch_split_rows(cudaStream_t stream, int num_sms, const float *x, int64_t n_rows, int64_t n_pad, int dim,
                       int scale_exp, __half *hi, __half *lo, float *norm, float pad_norm, unsigned int *cert_buf);

// project.cu
int project_rows(cmdb_bank *b, const float *x_dev, int64_t n_rows, int D, const int32_t *indptr_h,
                 const int32_t *indices_h, const double *data_h, int d_proj, double *z_dev);

// comm.cu
int comm_info(cmdb_comm *c, int *rank, int *world, unsigned char **local, unsigned char **peers, size_t *bytes);
unsigned long long comm_next_score_epoch(cmdb_comm *c);

// coreset.cu
// layout of a rank's peer-mapped buffer (cmdb_comm): [0, 256) per-rank "shard arrived" flags | key slots
// [parity][rank][CTA] x 32 B | at kCommHeaderBytes: replica of the whole projected bank in storage type
constexpr unsigned int kCommReadyOff = 0;
constexpr unsigned int kCommKeysOff = 256;
constexpr unsigned int kCommMaxCtas = 192;
constexpr size_t kCommCoresetBytes = 256 * 1024;  // coreset flags + key slots (>= 256 + 2 * kMaxRanks * kCommMaxCtas * 32); cleared by cmdb_comm_reset
// row-sharded SCORING rounds exchange through the same buffer (never cleared: every word is rewritten with the round's epoch):
//   flags  [4 slots][2 kinds][kMaxRanks] u64 at kCommScoreFlagsOff
//   d2     [4 slots][kMaxRanks][kShardD2Cap] float at kCommScoreD2Off        (squared neighbour distances, 2 per image)
//   keys   [4 slots][kMaxRanks][kShardKeysCap] int64 at kCommScoreKeysOff    (packed (min distance, global row) per query)
// (4 slots, round r uses slot r & 3: with two lanes per rank a rank may start round r + 2 while a peer still reads round r)
constexpr size_t kCommScoreFlagsOff = kCommCoresetBytes;
constexpr size_t kCommScoreD2Off = kCommScoreFlagsOff + 4096;
constexpr int kShardD2Cap = 64;
constexpr size_t kCommScoreKeysOff = kCommScoreD2Off + 16384;
constexpr int kShardKeysCap = 128 * 1024;   // queries per round (32 images x 3136 patches = 100 352)
constexpr int kShardSlots = 4;
constexpr size_t kCommHeaderBytes = 34 * 1024 * 1024;  // >= kCommScoreKeysOff + kShardSlots * kMaxRanks * kShardKeysCap * 8; the replica follows
struct ShardCtx {  // row-sharded coreset loop
    int world, rank;
    long long row_offset, n_total;
    unsigned char *peers[kMaxRanks];
    size_t comm_bytes;
    const double *z0_host;  // float64 projection of global row 0
};
int coreset_greedy_dev(cmdb_bank *b, const double *z_dev, int64_t N, int d, int64_t n_select, int dtype_mode,
                       int64_t *out_idx_host, const int64_t *force_idx_host, void *out_min_last_host, const ShardCtx *sh,
                       bool force_mind_global);
// host only: rows per CTA of the persistent kernel on num_sms SMs and whether their min-distances fit shared memory
int coreset_plan_info(int num_sms, int64_t N, int d, int dtype_mode, int64_t *rows_per_cta, int *mind_in_smem);
int coreset_greedy(cmdb_bank *b, const double *z_dev, int64_t N, int d, int64_t n_select, int dtype_mode,
                   int64_t *out_idx_host);
int coreset_rownorms(int device, const void *z_host, const void *last_host, int64_t n_rows, int d, int dtype_mode,
                     void *out_host);

struct TailResult {  // head of a result block (ScoreCall::tail), one per image
    float s, s_star, w, knn0, knn1;
    int s_idx;
    long long nn_idx[3];
    long long m_star_row;  // global row of m_star
};

// Launch schedule of one distance-GEMM launch, decided by score_gemm_candidates alone (gemm_sched).  N tiles go in order,
// dealt as runs of `run` consecutive tiles: run j of M tile m (M tile pair when pair) goes to unit (j * stride + m) % units.
struct GemmSched {
    int producers;  // (CTA, column group) candidate lists
    bool pair;      // CTA pairs (cta_group::2)
    int units;      // scheduling units G: CTAs, or CTA pairs
    int stride;     // tile_stride(M tiles per unit, G); 0 for a compact launch, which sizes itself on the device
    int inv;        // stride^-1 mod G
    int run;        // N tiles per visit of an M tile (score_gemm_run)
    int nt;         // N tiles of the launch
};

// Smallest s >= mt with gcd(s mod G, G) == 1: the stride of the GEMM's tile schedule (score_gemm.cu, TileIter).
__host__ __device__ __forceinline__ int tile_stride(int mt, int G) {
    for (int s = mt;; ++s) {
        int a = s % G, b = G;
        if (a == 0) a = G;
        while (b) {
            const int t = a % b;
            a = b, b = t;
        }
        if (a == 1 || G == 1) return s;
    }
}

// Which rows a producer (unit c, column group) saw for M tile m of a launch with schedule s: the runs j, j + G, j + 2G,
// ... with j * stride = c - m (mod G), i.e. j = (c - m) * stride^-1 mod G.  The certificate consumers walk them in tile
// slots `width` >= s.run tiles wide: slot kt is the (kt % width)-th tile of the (kt / width)-th run.  Returns the N tile,
// or >= s.nt for an empty slot.
__host__ __device__ __forceinline__ int producer_tile(const GemmSched &s, int width, int c, int m, int kt) {
    const int G = s.units, k = kt / width, t = kt % width;
    const int want = ((c - m % G) % G + G) % G;
    const int jrun = (int)(((long long)want * s.inv) % G) + k * G;
    return t < s.run ? jrun * s.run + t : s.nt;
}
// Slots that cover the longest producer of two launches over the same N tiles (of one launch: a == b): runs counted at
// the shorter run length, slots as wide as the longer one.
__host__ __device__ __forceinline__ int producer_slots(const GemmSched &a, const GemmSched &b) {
    const int run_min = a.run < b.run ? a.run : b.run, run_max = a.run < b.run ? b.run : a.run;
    return ((a.nt + run_min - 1) / run_min + a.units - 1) / a.units * run_max;
}
// Slot kt of the exact rescan of (M tile mtile of a batch, unit c): the batch's first-pass GEMM ran in chunks of
// chunk_tiles M tiles with schedule `full`; the last chunk, which may be shorter, with schedule `last`.
__host__ __device__ __forceinline__ int rescan_tile(const GemmSched &full, const GemmSched &last, int chunk_tiles, int mt_total,
                                                    int mtile, int c, int kt) {
    const int chunk = mtile / chunk_tiles;
    const bool is_last = (chunk + 1) * chunk_tiles >= mt_total;
    return producer_tile(is_last ? last : full, full.run < last.run ? last.run : full.run, c, mtile - chunk * chunk_tiles, kt);
}

// Packed 64-bit keys: a non-negative float's bits above an index, so that the integer order is the (value, index) order.
// The value of any of them:
__device__ __forceinline__ float key_value(unsigned long long k) { return __uint_as_float((unsigned int)(k >> 32)); }
// (d^2 or distance, row): the minimum is the nearest row, the lowest row on ties; ~0ULL = no row
__device__ __forceinline__ unsigned long long pack_min_key(float v, unsigned int row) {
    return ((unsigned long long)__float_as_uint(v) << 32) | row;
}
__device__ __forceinline__ long long key_row(unsigned long long k) { return (long long)(k & 0xffffffffULL); }
// exchange key of a sharded round: (min distance, global row) as a signed integer, INT64_MAX where there is no row, so
// that a MIN over the ranks is the global argmin (decoded with key_value / key_row)
__device__ __forceinline__ long long exchange_key(float v, long long row) {
    return row < 0 ? 0x7fffffffffffffffLL : (long long)(((unsigned long long)__float_as_uint(v) << 32) | (unsigned long long)row);
}
// argmax key of an image: an atomicMax over (min_val bits, ~query) keeps the largest value, the lowest query on ties
__device__ __forceinline__ void argmax_publish(unsigned long long *s_key, int qi, int P_img, float v) {
    atomicMax(s_key + qi / P_img, ((unsigned long long)__float_as_uint(v) << 32) | (0xffffffffu - (unsigned int)(qi % P_img)));
}
__device__ __forceinline__ int argmax_query(unsigned long long k) { return (int)(0xffffffffu - (unsigned int)(k & 0xffffffffu)); }

// alpha of the certificate's error bound: the tensor core's accumulation of D/16 MMAs of 16 exact fp16 products
inline float cert_acc_model(int dim) { return (float)(dim / 16 + 1) * 17.f * 1.1920929e-7f; }

// One scoring call: the handle, the compute lane and result slot it uses, and where in the slot's result block its
// results go.  The submit paths take the next lane and slot (api.cu); the neighbour-table build uses lane 0.
struct ScoreCall {
    cmdb_bank *b;
    int lane_idx, slot_idx;
    Lane *lane;
    ResultSlot *slot;
    cudaStream_t stream;   // the lane's stream
    TailResult *tail;      // [cap_b]
    float *min_val;        // [cap_p]
    long long *min_idx;    // [cap_p]
    float *map_out, *map_pre;   // [cap_b][map_stride]
    unsigned char *map_u8;
    // first-pass GEMM of score_local_min, which the exact rescan walks: M tiles, chunks of chunk_tiles tiles, and the
    // schedules of the first and the last chunk launch
    int mt_total = 0, chunk_tiles = 0;
    GemmSched first{}, last{};
};

// score_gemm.cu
int score_scratch_alloc(cmdb_bank *b, int B, int P_img, int out_hw);
ScoreCall score_call(cmdb_bank *b, int lane, int slot);  // call on that lane with its results in that slot's block
int score_mark(const ScoreCall &c, int stage, cudaStream_t st);  // timing event of `stage` (< 0: none) on st
int score_max_batch(const cmdb_bank *b);  // images per internal sub-batch (shared-memory bound of reweight_kernel)
void score_scratch_free(cmdb_bank *b);
int score_make_tensor_maps(cmdb_bank *b);
// q_f32 -> q_hi / q_lo (device-side scale selection) on st.  compact = true: only the rows of fail_list (count on the
// device), written to rows 0..count-1
int score_query_prep(const ScoreCall &c, cudaStream_t st, int P, bool compact, int row0 = 0);  // rows [row0, row0 + P) (row0 % 128 == 0)
// q_hi / q_lo -> cand via the tcgen05 distance GEMM with `terms` MMAs per K step on st; compact = true: the M extent is
// the device-side fail count
int score_gemm_candidates(const ScoreCall &c, cudaStream_t st, int P, int terms, bool compact, GemmSched *sched, int row0 = 0);
void q_split_rows(const ScoreCall &c, const float *rows_dev, int n);
GemmSched gemm_sched(int nt, int mt, int num_sms, bool pair);  // schedule of a non-compact launch over mt M tiles
// stage the queries (src: host or device, [B*P_img, dim]) + candidates + refine, all modes
// stage_after: event the copy stream waits for before it overwrites q_f32 (nullptr: everything queued so far)
int score_local_min(ScoreCall &c, const float *src, int src_is_device, int B, int P_img, int ev_gemm, int ev_refine,
                    cudaEvent_t stage_after = nullptr);

// The distance GEMM keeps one persistent CTA per SM with ~200 KB of dynamic shared memory, i.e. the SM runs in its largest
// shared-memory carve-out.  For the other lane's small kernels to become co-resident with it they must ask for the SAME
// carve-out (an SM is only re-configured when it is idle); one function per translation unit sets that preference once.
#define CMDB_PREFER_MAX_SMEM(kernel) \
    (void)cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared)
void tail_prefer_carveout();   // score_tail.cu
void gemm_prefer_carveout();   // score_gemm.cu
void api_prefer_carveout();    // api.cu
void bank_prefer_carveout();   // bank.cu

// score_tail.cu
int score_simt_candidates(const ScoreCall &c, int P, int *n_cand_out);
int score_refine(const ScoreCall &c, cudaStream_t st, int B, int P_img, int n_cand, bool compact);
int score_select(const ScoreCall &c, int B, int P_img, bool local_m_star);
int score_reweight(const ScoreCall &c, int B, int P_img);
int score_build_knn_table(cmdb_bank *b, long long row_first, long long row_count);
int score_exact_scan(cmdb_bank *b, const float *q_dev, int P, unsigned long long *keys_dev);
int score_shard_lookup(const ScoreCall &c, int B, float *contrib_dev);
int score_shard_final(const ScoreCall &c, int B, const float *d2_sum_dev);
// peer-memory form of the two exchanges of a sharded round (no NCCL): see score_tail.cu
struct PeerPtrs {
    unsigned char *p[kMaxRanks];
};
int score_shard_exchange_keys(const ScoreCall &c, int B, int P_img, const PeerPtrs &peers, int world, int rank, int slot, unsigned long long epoch);
int score_shard_exchange_d2(const ScoreCall &c, int B, const PeerPtrs &peers, int world, int rank, int slot, unsigned long long epoch,
                            const float *contrib_dev, float *d2_sum_dev);
int upsample_blur_launch(cudaStream_t stream, int n_img, int img_first, int img_step, size_t map_stride, const float *map_dev,
                         int fh, int fw, int out_hw, float *pre_dev, float *out_dev, unsigned char *u8_dev,
                         unsigned char *tmp_dev, float *mx_dev, float *mx_part_dev /* [n images][16] band maxima */);

}  // namespace cmdb
