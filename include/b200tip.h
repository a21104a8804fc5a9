/*
 * b200tip.h — C ABI of libb200tip.so, the B200 (sm_100a) scoring engine behind the
 * reference's `src.core` prioritizer API (testingautomated-usi/simple-tip).
 *
 * The reference has no FFI layer: its boundary is the Python class API of src/core
 * (SURVEY.md §8b).  The host mirror in simple_tip_b200/core keeps those classes and calls
 * the entry points below through ctypes.  Every array argument is a DEVICE pointer to a
 * contiguous row-major buffer owned by the caller (PyTorch on the Python side); the library
 * never frees caller memory and keeps no state between calls.  `stream` is a cudaStream_t
 * passed as void*; launches are asynchronous on it.  Every function returns 0 on success or
 * a negative tip_status; tip_last_error() returns a thread-local message.
 *
 * Which reference arithmetic each entry point replaces (paths relative to the reference):
 *   tip_deepgini        src/core/deepgini.py:31-35     argmax + 1 - sum(p*p)
 *   tip_kmnc            src/core/neuron_coverage.py:82-94 (+ sum_score :8-22)
 *   tip_cam_buckets     src/core/prioritizers.py:16-45 (greedy loop of cam) on compact KMNC profiles
 *   tip_pair_prep       (new) operand packing for the tensor-core pass
 *   tip_nn_filter       src/core/surprise.py:638-647   the B x M x D difference/norm/min, as a
 *                       tcgen05 pass that yields a per-query candidate set provably containing
 *                       NumPy's argmin
 *   tip_nn_rerank       src/core/surprise.py:640-648   exact np.linalg.norm / np.min / np.argmin
 *                       on the candidates, in NumPy's summation order (bit-identical)
 *   tip_gather_rows     src/core/surprise.py:648       to_ats[closest_position]
 *   tip_whiten          scipy==1.4.1 gaussian_kernel_estimate: points . cholesky(inv_cov)
 *   tip_kde_lse         scipy==1.4.1 gaussian_kernel_estimate pair loop (called from
 *                       src/core/stable_kde.py:101), in the log domain
 *   tip_kde_combine     merge of per-column-chunk (max, sum) partials
 */
#ifndef B200TIP_H
#define B200TIP_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TIP_VERSION 200

typedef enum tip_status {
  TIP_OK = 0,
  TIP_ERR_INVALID = -1,    /* bad argument (shape, dtype, alignment) */
  TIP_ERR_CUDA = -2,       /* CUDA runtime / driver error, see tip_last_error() */
  TIP_ERR_UNSUPPORTED = -3 /* not an sm_100 device */
} tip_status;

typedef enum tip_dtype {
  TIP_F32 = 0,
  TIP_F64 = 1,
  TIP_BF16 = 2,
  TIP_I16 = 3,
  TIP_I32 = 4
} tip_dtype;

/* operand roles / packing modes for tip_pair_prep */
#define TIP_ROLE_QUERY 0 /* rows become TMEM lanes (test traces / stage-2 winners)    */
#define TIP_ROLE_TRAIN 1 /* rows become accumulator columns (training traces)         */

/* row selection for tip_nn_rerank */
#define TIP_RANGE_SAME_CLASS 0   /* columns [off[c], off[c+1])                      */
#define TIP_RANGE_OTHER_CLASSES 1 /* columns [0, off[c]) U [off[c+1], off[C])       */

/* One unit of work of the tensor-core pass: a tile of query rows (128, or 256 for
 * tip_nn_filter on short traces, see tip_nn_filter_tile) x a span of train rows. */
typedef struct tip_work_item {
  int32_t q_row0;  /* first query row of the tile                                   */
  int32_t q_rows;  /* valid rows in the tile (1..tile); others are computed, not stored */
  int32_t col0;    /* first train row of the span                                   */
  int32_t col1;    /* one past the last train row of the span                       */
  int32_t slot;    /* tip_kde_lse: partial-result slot of this span; unused otherwise */
  int32_t reserved; /* flags: bit 0 = every query ignores the train rows of its own class
                     * (tip_nn_filter with q_class / class_off) */
} tip_work_item;

int tip_version(void);
const char* tip_last_error(void);
/* sm count and compute capability of the current device */
int tip_device_info(int* sm_count, int* cc_major, int* cc_minor);
/* number of kernels this library has launched in this process (bench.py: gpu_launches) */
uint64_t tip_launch_count(void);

/* ---- DeepGini (deepgini.py:31-35) ----------------------------------------------------
 * probs: n x c (TIP_F32 or TIP_F64).  pred[n] = first argmax, gini[n] = 1 - sum(p*p) in the
 * input dtype, summed in NumPy's pairwise order (bit-identical to np.sum(p*p, axis=1)). */
int tip_deepgini(const void* probs, int dtype, int64_t n, int64_t c, int32_t* pred, void* gini,
                 void* stream);

/* ---- KMNC (neuron_coverage.py:65-94) -------------------------------------------------
 * act: n x d (TIP_F32/TIP_F64); mins, jumps: d values of stat_dtype, jumps = (max-min)/k
 * computed by the caller with the reference's NumPy expression.  Thresholds are
 * t_i = min + jumps*i evaluated on the fly in stat_dtype (same rounding as NumPy).
 * bucket[n*d] (TIP_I16 or TIP_I32) = the i with t_i <= a < t_{i+1}, or -1; score[n] = number of
 * neurons with a bucket (== sum of the reference's dense profile). bucket may be NULL. */
int tip_kmnc(const void* act, int act_dtype, int64_t n, int64_t d, const void* mins,
             const void* jumps, int stat_dtype, int32_t sections, void* bucket, int bucket_dtype,
             int32_t* score, void* stream);

/* ---- Coverage-Additional Method over compact coverage profiles (prioritizers.py:16-59) ----
 * bucket: n x d section ids as tip_kmnc writes them (TIP_I16 / TIP_I32, -1 = none): the one-hot-per-
 * neuron profile of neuron_coverage.py:82-94 without its dense n x d x sections form.  Runs up to
 * `rounds` rounds of the reference's greedy loop — pick = first index of the largest gain (np.argmax),
 * mark the cells the pick newly covers, subtract from every sample the number of those cells it shares
 * — and stops for good when the best gain is 0.  Caller-owned state, all on the device:
 *   gain[n]      in: number of valid cells per sample (= KMNC score); updated in place
 *   covered      ceil(d*sections/32) words, zero before the first call
 *   newlist      2*d int32 scratch
 *   order[n]     out: the picks in order; state[0] = how many (zero before the first call)
 *   state[4]     {picks, done flag, scratch, scratch}, zero before the first call; call again with the
 *                same buffers while state[1] == 0 && state[0] < n.
 * The tail of the reference's generator (not-yet-picked samples by np.argsort(-scores), :47-59) is host
 * NumPy, so ties fall exactly as in the reference. */
int tip_cam_buckets(const void* bucket, int bucket_dtype, int64_t n, int64_t d, int32_t sections,
                    int32_t* gain, uint32_t* covered, int32_t* newlist, int32_t* order, int32_t* state,
                    int32_t rounds, void* stream);

/* ---- sibling coverage criteria and their fit step (neuron_coverage.py:52-62,97-173;
 * aggregate_statistics.py:37-67 + welford==0.2.5) ------------------------------------------
 * tip_cover_threshold: act n x d (TIP_F32/TIP_F64); mode
 *   TIP_COVER_NAC   profile[n,d]   = act >  threshold                      (lo = hi = NULL)
 *   TIP_COVER_SNAC  profile[n,d]   = act >= hi[d]
 *   TIP_COVER_NBC   profile[n,d,2] = (act <= lo[d], act >= hi[d])
 * lo / hi: d boundaries of stat_dtype, computed by the caller with the reference's NumPy expressions
 * (min - s*std, max + s*std); comparisons run in NumPy's promoted dtype of (act, boundary), so the
 * profile is bit-identical.  profile_u8 (one byte per entry: the reference's dense bool array) and
 * bits (the same profile bit-packed for tip_cam_bits, tip_cover_packed_words(d) words per row and
 * plane, NBC: 2 planes; layout in csrc/coverage.cu) are both optional; score[n] = number of set
 * entries per sample (== sum_score, neuron_coverage.py:8-22). */
#define TIP_COVER_NAC 0
#define TIP_COVER_SNAC 1
#define TIP_COVER_NBC 2
int64_t tip_cover_packed_words(int64_t d);
int tip_cover_threshold(const void* act, int act_dtype, int64_t n, int64_t d, const void* lo,
                        const void* hi, int stat_dtype, double threshold, int mode, void* profile_u8,
                        uint32_t* bits, int32_t* score, void* stream);
/* Top-k neuron coverage of ONE layer (neuron_coverage.py:160-168): for every sample the k largest of its
 * d_layer activations are marked in profile_u8[r * row_stride + col_off + i] (all entries of the layer's
 * columns are written) and/or OR-ed into the packed words of neuron col_off + i (bits must be zero-filled
 * by the caller; bit_words = words per row).  Equal values: the higher index wins (NumPy's unstable
 * argsort leaves that case implementation-defined). */
int tip_tknc(const void* act, int dtype, int64_t n, int64_t d_layer, int32_t k, void* profile_u8,
             int64_t row_stride, int64_t col_off, uint32_t* bits, int64_t bit_words, void* stream);
/* Streaming per-neuron statistics over a batch of n samples x d neurons: mins/maxs and welford==0.2.5's
 * `add` applied sample by sample in the activation dtype (mean, m2 = sum of squared deviations; the caller
 * keeps the integer count: count_before = samples folded in so far).  State arrays hold d values of
 * `dtype`; initial state: mean = m2 = 0, mins = +inf, maxs = -inf. */
int tip_stats_update(const void* act, int dtype, int64_t n, int64_t d, int64_t count_before, void* mean,
                     void* m2, void* mins, void* maxs, void* stream);

/* ---- Coverage-Additional Method over dense boolean profiles, bit-packed (prioritizers.py:16-45) ----
 * tip_pack_bool: byte profile n x f (non-zero = covered) -> ceil(f/32) words per row.
 * tip_cam_bits: bits n x words (any packing, the order of the picks does not depend on it).  One
 * persistent cooperative kernel runs up to max_rounds greedy rounds: pick = first index of the largest
 * gain, new = profile[pick] & ~covered, gain[i] -= popcount(profile[i] & new); it stops for good when
 * the best gain is 0.  Caller-owned device state: gain[n] (init_gain != 0: initialised here to the row
 * popcounts), covered2[2*words] zero-filled, cand_scratch[4*TIP_CAM_MAX_BLOCKS] int32, order[n],
 * state[4] = {picks, done, -, -} zero-filled before the first call; call again with the same buffers
 * (init_gain = 0) while state[1] == 0 && state[0] < n.  max_rounds must be even when more calls follow
 * (the covered set is double-buffered by round parity). */
#define TIP_CAM_MAX_BLOCKS 1024
int tip_pack_bool(const void* profile_u8, int64_t n, int64_t f, uint32_t* bits, void* stream);
int tip_cam_bits(const uint32_t* bits, int64_t n, int64_t words, int32_t* gain, uint32_t* covered2,
                 int32_t* cand_scratch, int32_t* order, int32_t* state, int32_t max_rounds,
                 int32_t init_gain, void* stream);

/* ---- operand packing for the tensor-core pass ----------------------------------------
 * Packed row (bf16), D16 = round_up(d,16), one 16-wide tail block:
 *   segments == 1:  [ s*h(v) | tail ]                 v = fl32(x - center)
 *   segments == 3:  query: [ h | l | h | tail ]       h = bf16(v), l = bf16(v - h)
 *                   train: [ s*h | s*h | s*l | tail ]
 *   tail(query) = [1,1,1,0...]; tail(train) = bf16 3-way split of norm_coef*|v|^2
 * so that one K-loop accumulates  norm_coef*|y|^2 + s * <x, y>  in fp32 TMEM.
 * sqnorm[rows] receives |h(v)|^2 (segments==1) or |v|^2 (segments==3) as fp32.
 * rounderr[rows] (may be NULL) receives the Euclidean norm of what the packed operand drops,
 * |v - h(v)| (segments==1) or |v - h - l| (segments==3), rounded up: the per-row input-rounding
 * term of tip_nn_filter's error window.
 * tip_pair_pitch returns the packed row pitch in elements (multiple of 64). */
int64_t tip_pair_pitch(int64_t d, int segments);
int tip_pair_prep(const void* src, int dtype, int64_t rows, int64_t d, const float* center,
                  int role, int segments, float scale, float norm_coef, void* dst_bf16,
                  float* sqnorm, float* rounderr, void* stream);

/* Query side of tip_nn_filter in one launch: packs the queries (segments = 1, no scaling) and
 * resets the per-query filter state (row_min_bits = +inf, cand_cnt = 0).  q_idx (may be NULL): packed row r is
 * taken from q + q_idx[r]*d — the class-sorting gather of DSA.__call__ (surprise.py:580-587) fused into the pack. */
int tip_nn_query_prep(const void* q, int dtype, int64_t m, int64_t d, const float* center,
                      void* q_pack, float* q_sqnorm, float* q_rounderr, uint32_t* row_min_bits,
                      int32_t* cand_cnt, const int32_t* q_idx, void* stream);

/* ---- nearest-neighbour candidate filter (tcgen05 + TMA) ------------------------------
 * q_pack: m x pitch, t_pack: n x pitch (tip_pair_prep, scale=-2, norm_coef=1).
 * For every query row and every work item covering it, scans the item's train span and
 * appends one entry per 32-row chunk of train rows that contains a row whose approximate squared
 * distance is within the proven error window of the running minimum (see DESIGN.md §4):
 * cand_idx[(row*cap + k)*2] = first train row of the chunk, cand_idx[(row*cap + k)*2 + 1] = 32-bit
 * mask of the rows of the chunk that pass (cand_idx holds 2*cap int32 per query); cand_cnt[row]
 * counts appends (may exceed cap: overflow -> tip_nn_rerank falls back to an exact scan).
 * row_min_bits[m] (uint32 float bits, initialised to +inf = 0x7f800000 by the caller) carries
 * the running minimum across items/CTAs.  t_rmax = max_j |h(y_j)| over the train rows.
 * q_rounderr[m] / t_errmax = max_j rounderr(y_j) (tip_pair_prep) give the window its measured
 * input-rounding term |d_bf16 - d| <= rounderr(x) + rounderr(y); with q_rounderr == NULL the
 * a-priori bound 2^-9 (|h(x)| + |h(y)|) is used instead (about twice as wide).
 * Scheduling: CTA b of the G = min(n_items, #SMs) persistent CTAs runs items b, b + G, ... below
 * n_static; items [n_static, n_items) are a shared pool that CTAs drain through sched_counter
 * once their static share is done — the pool evens out CTAs whose
 * tiles turn out slower.  sched_counter points to TWO int32 that are zero on entry; the kernel
 * leaves them zero (one call at a time per counter pair).  n_static == n_items (sched_counter may
 * be NULL) is a purely static run;
 * pools need the resident-query kernel (d <= 128).  Items with col0 == col1 are skipped.
 * q_class[m] / class_off[C+1] (may be NULL if no item sets flag bit 0): for flagged items a query of
 * class c ignores train rows [class_off[c], class_off[c+1]) — DSA's other-class search over
 * query tiles that mix classes (surprise.py:622-629). */
int tip_nn_filter(const void* q_pack, const float* q_sqnorm, int64_t m, const void* t_pack,
                  int64_t n, int64_t d, int64_t pitch, const tip_work_item* items,
                  int32_t n_items, const int32_t* q_class, const int32_t* class_off, float t_rmax,
                  const float* q_rounderr, float t_errmax, uint32_t* row_min_bits, int32_t* cand_idx,
                  int32_t* cand_cnt, int32_t cap, int32_t n_static, int32_t* sched_counter,
                  void* stream);

/* Tile geometry tip_nn_filter uses for traces of width d: work items must start on query rows
 * that are multiples of nothing in particular but cover at most *q_rows rows (128, or 256 for
 * the resident-query kernel used when the packed row has <= 9 K-steps, i.e. d <= 128); *t_rows
 * is the train-tile height (256 or 128), useful for sizing spans. */
int tip_nn_filter_tile(int64_t d, int32_t* q_rows, int32_t* t_rows);
/* which tensor-core kernel tip_nn_filter runs for traces of width d: 1 = resident-query (d <= 128, 256 x 192
 * tiles), 0 = streaming (128 x 256 tiles).  tip_kde_tile_rows: query rows per work item of tip_kde_lse*. */
int tip_nn_filter_kind(int64_t d);
int tip_kde_tile_rows(void);
int tip_kde_slot_parts(void);   /* partial (max, sum) pairs per work-item slot: part_max / part_sum hold slots x this x m */

/* ---- exact re-rank (NumPy-order distances, first-occurrence argmin) -------------------
 * q, t: original-dtype (TIP_F32/TIP_F64) matrices m x d and n x d; train rows are grouped by
 * class (class_off[C+1]); q_class[m] gives each query's class, mode the column range.
 * Rows with 1..cap candidate entries (tip_nn_filter's chunk + mask pairs, rows clipped to the
 * class range) are re-ranked over the flagged rows; rows with 0 or > cap
 * candidates (or cand_cnt == NULL) are scanned exhaustively over their range.
 * out_dist[m] (dtype) = sqrt(pairwise_sum((x-y)^2)) of the winner, out_pos[m] = its train row
 * (ties: lowest t_gid); optional out_gid[m] = t_gid of the winner (-1 if none) and
 * out_rows[m x d] = a copy of the winning train rows (DSA's stage-2 queries, surprise.py:648).
 * work: scratch of tip_nn_rerank_work_bytes(m, dtype) bytes (queue of queries that need the
 * exhaustive scan + the per-slice partial winners of that scan).  The caller zero-fills it once;
 * every call leaves the two words it relies on (queue length work[0], completion counter
 * work[1 + m]) at zero again, so the buffer can be reused by the next call on the same stream.
 * stats[0] += rows that took the exhaustive scan (stats[1] is reserved; candidate counts are in
 * cand_cnt).
 * next_*: optional (all NULL, or pack + sqnorm + row_min_bits + cand_cnt given): the winning rows are
 * also emitted as the packed queries and reset filter state of a following tip_nn_filter call —
 * exactly what tip_nn_query_prep(out_rows, center = next_center) would write — so DSA's second
 * stage (whose queries are stage 1's winners, surprise.py:627-629) needs no pack launch.
 * extras (optional, host struct read at launch time):
 * q_idx: the queries are rows q_idx[r] of q (no separately gathered copy needed); fin_*: fused result scatter.
 * next_seed_ub (optional, with next_rounderr): n floats, for every train row an upper bound on its exact
 * distance to SOME row the next search will scan for it (e.g. its nearest other-class row inside a fixed sample
 * of the training set, computed once at fit time; +inf = none).  The winner's bound, widened by the filter's own
 * error terms (next_t_rmax / next_t_errmax = the t_rmax / t_errmax of the next tip_nn_filter call), becomes the
 * initial next_row_min_bits instead of +inf: the next filter collects no far-away candidates while its running
 * minima warm up.  A seed never narrows the proven window below the final one (DESIGN.md §4). */
typedef struct tip_rerank_extras {
  const int32_t* q_idx;       /* query row r is q + q_idx[r]*d (e.g. class-sorted order over the caller's buffer) */
  const float* next_seed_ub;  /* see above */
  float next_t_rmax;
  float next_t_errmax;
  const void* fin_dist_a;     /* fused result scatter: with fin_out != NULL this search's distance is taken as dist_b */
  const int32_t* fin_gid;     /* and out[0..3][fin_idx[r]] = dist_a, dist_b, gid, dist_a / dist_b as tip_dsa_pack_out */
  const int32_t* fin_idx;     /* writes them (fin_idx == NULL: r itself); fin_dist_a in `dtype`, fin_out 4*fin_n_total */
  int64_t fin_n_total;        /* doubles */
  double* fin_out;
  int32_t count_overflow_only; /* != 0 (filtered searches only): queries whose candidate list is empty or overflowed are */
  int32_t reserved;            /* only COUNTED in work[0] — no queue, no exhaustive-scan launch, their outputs are not    */
                               /* written; the caller checks work[0] after the call, resets it and repeats without this   */
                               /* flag if it is non-zero (speculative execution of the normal, fallback-free case)        */
} tip_rerank_extras;
int32_t tip_sizeof_rerank_extras(void);   /* bindings check their struct layout against this */
int64_t tip_nn_rerank_work_bytes(int64_t m, int dtype);
int tip_nn_rerank(const void* q, const void* t, int dtype, int64_t m, int64_t n, int64_t d,
                  const int32_t* cand_idx, const int32_t* cand_cnt, int32_t cap,
                  const int32_t* q_class, const int32_t* class_off, int32_t n_classes, int mode,
                  const int32_t* t_gid, void* out_dist, int32_t* out_pos, int32_t* out_gid,
                  void* out_rows, int32_t* work, int64_t* stats, const float* next_center,
                  void* next_pack, float* next_sqnorm, float* next_rounderr,
                  uint32_t* next_row_min_bits, int32_t* next_cand_cnt, const tip_rerank_extras* extras,
                  void* stream);

/* DSA result packing (surprise.py:576-611 scatter by index): for i < m,
 *   out[0*n_total + j] = dist_a[i], out[1*n_total + j] = dist_b[i], out[2*n_total + j] = gid[i],
 *   out[3*n_total + j] = dist_a[i] / dist_b[i]  (IEEE division in `dtype`, surprise.py:595)
 * with j = idx[i] (idx == NULL: j = i); values in `dtype` (TIP_F32/TIP_F64) are widened to double
 * exactly, gid (int32) likewise.  out holds 4*n_total doubles; columns not named by idx are left
 * untouched. */
int tip_dsa_pack_out(const void* dist_a, const void* dist_b, int dtype, const int32_t* gid,
                     const int32_t* idx, int64_t m, int64_t n_total, double* out, void* stream);

/* dst[i,:] = src[pos[i],:]  (rows of `row_bytes` bytes; pos < 0 -> zero row) */
int tip_gather_rows(const void* src, int64_t row_bytes, const int32_t* pos, int64_t m, void* dst,
                    void* stream);

/* ---- N_train sharded over the GPUs of one NVSwitch box (SURVEY.md 8e; no counterpart in the
 * reference — the dependency that forces the exchange is src/core/surprise.py:615-631: stage 2's
 * queries are the GLOBAL stage-1 winners) -------------------------------------------------------
 * A tip_comm is a set of symmetric receive buffers, one per rank (one process per GPU), opened
 * across processes through CUDA IPC.  An exchange is: every rank pushes m 16-byte records into the
 * slots of all peers with plain NVLink stores and raises a flag (tip_comm_push_*); the consumer
 * kernel (tip_shard_winner_queries / tip_comm_min / tip_comm_lse) waits for all flags and reduces the
 * `world` records per query from local memory in its prologue.  Exchanges must be issued in the same
 * order on every rank; at most `cap_records` records per exchange.  Set-up (host side, once):
 *   tip_comm_alloc      cudaMalloc + zero the local buffer, return its 64-byte IPC handle
 *   (all-gather the handles with torch.distributed)
 *   tip_comm_open       map the peers' buffers; all_handles = world x 64 bytes in rank order
 *   tip_comm_close      unmap the peers;  tip_comm_free_local frees the local buffer. */
#define TIP_COMM_MAX_WORLD 16
#define TIP_COMM_HANDLE_BYTES 64
typedef struct tip_comm tip_comm;
int64_t tip_comm_bytes(int32_t world, int64_t cap_records);
int tip_comm_alloc(int32_t world, int64_t cap_records, void** local_buf, void* ipc_handle);
int tip_comm_open(int32_t rank, int32_t world, void* local_buf, const void* all_handles,
                  int64_t cap_records, tip_comm** out);
int tip_comm_close(tip_comm* comm);
int tip_comm_free_local(void* local_buf);
/* record i = (bit pattern of dist[i] (NaN = no row on this shard), gid[i] or 0): the per-shard result
 * of tip_nn_rerank for query i; dtype TIP_F32 / TIP_F64 */
int tip_comm_push_nn(tip_comm* comm, const void* dist, int dtype, const int32_t* gid, int64_t m,
                     void* stream);
/* record i = this shard's partial KDE sum (running max, sum of exp(. - max)) of tip_kde_combine */
int tip_comm_push_lse(tip_comm* comm, const float* part_max, const float* part_sum, int64_t m,
                      void* stream);
/* out_dist[i] = min over the ranks of the pushed distances (NaN if no shard had a row) */
int tip_comm_min(tip_comm* comm, int dtype, int64_t m, void* out_dist, void* stream);
/* merged log-sum-exp partials, in rank order, identical on every rank: out_max = max_r max_r,
 * out_sum = sum_r sum_r * exp(max_r - out_max) (double) */
int tip_comm_lse(tip_comm* comm, int64_t m, float* out_max, double* out_sum, void* stream);
/* Global stage-1 winners -> stage-2 queries.  comm != NULL: waits for the exchange started by the
 * last tip_comm_push_nn and takes, per query, the lexicographic minimum of (distance, original
 * index) over the shards; comm == NULL: gdist[m] / ggid[m] hold that minimum already (reduced by
 * torch.distributed).  train_full: the whole (post-subsample) training set, n_full x d in the trace
 * dtype, rows in ORIGINAL order, replicated on every rank (C5: 10.5 GB of 180).  Writes the global
 * dist_a (NaN if the class has no training row anywhere), the winner's original index (-1), a copy
 * of the winning rows (out_rows, m x d: the exact re-rank's queries) and the packed bf16 queries +
 * reset filter state of the following tip_nn_filter call (see tip_nn_rerank's next_* outputs). */
int tip_shard_winner_queries(tip_comm* comm, const void* gdist, const int32_t* ggid, int dtype,
                             int64_t m, int64_t d, const void* train_full, int64_t n_full,
                             const float* center, void* out_dist, int32_t* out_gid, void* out_rows,
                             void* next_pack, float* next_sqnorm, float* next_rounderr,
                             uint32_t* next_row_min_bits, int32_t* next_cand_cnt, void* stream);

/* ---- LSA: whitening and the fused Gaussian-KDE log-sum-exp ---------------------------
 * out[m x d_out] (fp32) = (x[:, cols] - mu) . w, x: m x d_in (TIP_F32/TIP_F64), cols[d_out] the kept
 * columns (NULL = all), mu: d_out doubles, w: d_out x d_out fp32 row-major. */
int tip_whiten(const void* x, int dtype, int64_t m, int64_t d_in, const int32_t* cols,
               int64_t d_out, const double* mu, const float* w, float* out, void* stream);

/* out[m] (double) = sum_k y[row,k]^2 of a whitened matrix y (m x d fp32, from tip_whiten): the squared
 * Mahalanobis distance to one centre (MDSA, surprise.py:374-393: sklearn EmpiricalCovariance.mahalanobis) or
 * the quadratic form of one mixture component (MLSA, surprise.py:498-520: sklearn
 * _estimate_log_gaussian_prob, y = (x - mu_k) . precisions_cholesky_k). */
int tip_row_sqnorm(const float* y, int64_t m, int64_t d, double* out, void* stream);

/* q_pack / t_pack from tip_pair_prep(segments=3, scale=1, norm_coef=-0.5 on the train side).
 * For every work item writes the partial (max_i a_ij, sum_i exp(a_ij - max)) of
 * a_ij = <p_i, q_j> - |p_i|^2/2 over the item's span into part_max/part_sum[(P*slot+h)*m + row],
 * P = tip_kde_slot_parts(), h = 0..P-1 for the column parts of the 256-wide tiles each group of four epilogue
 * warps reduces (so P*slots*m floats each, which the caller initialises to -inf / 0). */
int tip_kde_lse(const void* q_pack, int64_t m, const void* t_pack, int64_t n, int64_t d,
                int64_t pitch, const tip_work_item* items, int32_t n_items, float* part_max,
                float* part_sum, void* stream);
/* The same pass with ONE fp16 segment (a third of the tensor work): operands from tip_pair_prep_f16, i.e.
 * a_ij = <h(p_i), h(q_j)> - |p_i|^2/2 with h = fp16 rounding (11-bit significands: |error| ~ 2^-12 per product,
 * against ~2^-17 for the three-segment bf16 form).  Whether that is accurate enough for rtol 1e-4 on the
 * log-density depends on the data; the caller verifies it against tip_kde_lse on a sample of the queries and
 * falls back (simple_tip_b200/core/stable_kde.py).  Same outputs as tip_kde_lse; pitch = tip_pair_pitch(d, 1). */
int tip_kde_lse_f16(const void* q_pack, int64_t m, const void* t_pack, int64_t n, int64_t d,
                    int64_t pitch, const tip_work_item* items, int32_t n_items, float* part_max,
                    float* part_sum, void* stream);
/* fp16 operand packing for tip_kde_lse_f16: row = [ h(fl32(x - center)) | tail ], tail(query) = [S,S,S,0..],
 * tail(train) = 3-way fp16 split of norm_coef*|v|^2/S with S = norm_scale (a power of two; keeps the norm
 * term in fp16's range).  sqnorm[rows] = |v|^2 (fp32, may be NULL); flags[0] |= 1 if anything left fp16's finite
 * range (flags may be NULL). */
int tip_pair_prep_f16(const void* src, int dtype, int64_t rows, int64_t d, const float* center, int role,
                      float norm_coef, float norm_scale, void* dst_f16, float* sqnorm, int32_t* flags,
                      void* stream);
/* merges `slots` partials per row in ascending slot order: out_max, out_sum (fp32) */
int tip_kde_combine(const float* part_max, const float* part_sum, int64_t m, int32_t slots,
                    float* out_max, float* out_sum, void* stream);

/* ---- bring-up / validation: plain accumulator dump ------------------------------------
 * out[256*256] (fp32, row-major, leading dimension 256) = tail-augmented dot products of q rows
 * [0,128) (streaming kernel) or [0,256) (resident-query kernel) with t rows [0,256).
 * variant: 0 = the kernel tip_nn_filter would pick, 1 = streaming, 2 = resident-query. */
int tip_pair_probe(const void* q_pack, int64_t m, const void* t_pack, int64_t n, int64_t d,
                   int segments, int64_t pitch, int variant, float* out, void* stream);

/* bring-up: while buf != NULL, block 0 of the resident-query filter kernel records clock64()
 * stamps (16 int64 slots per train tile, up to `tiles` tiles): MMA warp 0/1 before/after the
 * train-tile wait, 2/3 and 11/12 start/end of the issue of query half 0 and 1; 4..7 one epilogue
 * thread (before/after the accumulator wait, at TMEM release, at tile end), 8..10 TMA producer. */
int tip_debug_timeline(long long* buf, int32_t tiles);
/* bring-up: while buf != NULL, every CTA of the resident-query filter kernel writes
 * {globaltimer ns at start, at end, train tiles, work items} to buf[4*blockIdx.x ...]. */
int tip_debug_cta_clock(long long* buf);

#ifdef __cplusplus
}
#endif
#endif /* B200TIP_H */
