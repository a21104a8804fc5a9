// rerank.cu — exact stage of the nearest-neighbour search (surprise.py:633-651).
//
// For every query row the tensor-core filter (pair_tc.cu) leaves a candidate set that provably
// contains NumPy's argmin.  Here each candidate's distance is recomputed exactly as
//   np.linalg.norm(from[:, None] - to, axis=2)   (surprise.py:638-640)
// does it: difference, square, NumPy's pairwise summation order, correctly rounded sqrt — all in
// the input dtype with no FMA contraction — and the winner is the lexicographic minimum of
// (distance, original train index), i.e. np.argmin's first occurrence (surprise.py:645-647).
//
// Two kernels: (1) one WARP per query walks its short candidate list (the work per query is a
// handful of rows, so the kernel is a chain of dependent memory latencies: many queries in
// flight matter, not threads per query); queries without a usable list (0 or > cap entries, or
// no filter at all) are appended to a work list; (2) the listed queries' class ranges are scanned
// exhaustively — the reference-grade fallback, normally empty, in which case every block of the
// second kernel returns at once.  The last block to finish merges the per-slice winners and
// re-arms the queue (work[0] and the completion counter are 0 on entry and on exit).
// Both also emit the winner's original index and (optionally) copy the winning train row, which
// is the query of DSA's second stage (surprise.py:627-629, 648).
#include <algorithm>
#include <map>
#include <mutex>
#include <vector>
#include "common.cuh"

namespace tip {

constexpr int kScanThreads = 128;

template <typename T>
struct Best {
  T dist;
  int gid;
  int pos;
};

template <typename T>
__device__ __forceinline__ void consider(Best<T>& b, T dist, int gid, int pos) {
  // NaN distances never win (np.min would propagate NaN; documented as unsupported input)
  if (dist < b.dist || (dist == b.dist && gid < b.gid)) {
    b.dist = dist;
    b.gid = gid;
    b.pos = pos;
  }
}

template <typename T>
__device__ __forceinline__ Best<T> merge(Best<T> a, T dist, int gid, int pos) {
  if (pos >= 0) {
    if (a.pos < 0) { a.dist = dist; a.gid = gid; a.pos = pos; }
    else consider(a, dist, gid, pos);
  }
  return a;
}

template <typename T>
struct RerankArgs {
  const T* q;
  const T* t;
  int64_t m, n;
  int d;
  const int32_t* cand_idx;
  const int32_t* cand_cnt;
  int cap;
  const int32_t* q_class;
  const int32_t* class_off;
  int n_classes;
  int mode;
  const int32_t* t_gid;
  T* out_dist;
  int32_t* out_pos;
  int32_t* out_gid;   // nullable
  T* out_rows;        // nullable: m x d copy of the winning train rows
  int32_t* work;      // work[0] = number of queued queries, work[1..] = their rows
  unsigned long long* stats;
  // optional: the winning rows packed as the queries of the next tip_nn_filter call (what
  // tip_nn_query_prep would produce from out_rows), so DSA's second stage needs no pack launch
  const float* next_center;
  __nv_bfloat16* next_pack;
  int64_t next_pitch;
  float* next_sqnorm;
  float* next_rounderr;
  uint32_t* next_row_min;
  int32_t* next_cand_cnt;
  SeedParams seed;    // optional: per-train-row upper bounds that seed the next stage's running minima
  const int32_t* q_idx;   // optional: query row r lives at q + q_idx[r] * d (class-sorted order over the caller's buffer)
  // optional fused result scatter (what tip_dsa_pack_out does): this search's distance is dist_b
  const T* fin_dist_a;
  const int32_t* fin_gid;
  const int32_t* fin_idx;
  int64_t fin_n_total;
  double* fin_out;
  // long traces: NumPy's pairwise-sum schedule for this trace width, flattened on the host (common.cuh)
  const uint32_t* sum_prog;
  int sum_leaves;
  int count_only;     // speculative call: overflowed / empty lists are only counted in work[0] (tip_rerank_extras)
};

template <typename T>
__device__ __forceinline__ const T* query_row(const RerankArgs<T>& a, int64_t row) {
  return a.q + (a.q_idx ? (int64_t)a.q_idx[row] : row) * (int64_t)a.d;
}

template <typename T>
__device__ __forceinline__ void write_result(const RerankArgs<T>& a, int64_t row, const Best<T>& b, int lane) {
  // all 32 lanes of the calling warp hold the same `b`
  if (lane == 0) {
    const T dist = b.pos >= 0 ? b.dist : (T)NAN;   // empty range -> NaN / -1
    a.out_dist[row] = dist;
    a.out_pos[row] = b.pos;
    if (a.out_gid) a.out_gid[row] = b.pos >= 0 ? (a.t_gid ? a.t_gid[b.pos] : b.pos) : -1;
    if (a.fin_out) {   // dist_a, dist_b, winner index, dist_a / dist_b in the caller's row order (surprise.py:595,611)
      const int64_t j = a.fin_idx ? a.fin_idx[row] : row;
      if (j >= 0 && j < a.fin_n_total) {
        const T da = a.fin_dist_a[row];
        a.fin_out[j] = (double)da;
        a.fin_out[a.fin_n_total + j] = (double)dist;
        a.fin_out[2 * a.fin_n_total + j] = (double)a.fin_gid[row];
        a.fin_out[3 * a.fin_n_total + j] = (double)Rn<T>::div(da, dist);
      }
    }
  }
  const T* src = a.t + (int64_t)(b.pos < 0 ? 0 : b.pos) * a.d;
  if (a.out_rows) {
    T* dst = a.out_rows + row * (int64_t)a.d;
    for (int i = lane; i < a.d; i += 32) dst[i] = b.pos >= 0 ? src[i] : (T)0;
  }
  if (a.next_pack)
    warp_pack_query<T>(b.pos >= 0 ? src : nullptr, a.d, a.next_center, a.next_pack + row * a.next_pitch, a.next_pitch,
                       a.next_sqnorm + row, a.next_rounderr ? a.next_rounderr + row : nullptr, a.next_row_min + row,
                       a.next_cand_cnt + row, lane,
                       (a.seed.ub && b.pos >= 0) ? a.seed.ub[b.pos] : __int_as_float(0x7f800000), &a.seed);
}

// ---- kernel 1: one warp per query, candidate lists ----------------------------------------------
// SMALL = traces of at most 128 elements (one leaf of NumPy's pairwise sum): every lane keeps the
// query elements of the stride-8 accumulator it owns in registers — loaded once, in the same
// round trip as the candidate count — and a candidate row costs 16 loads + 47 flops per lane.
// WPB = warps (queries) per block.  The warps of a block never talk to each other; a block's slot on the SM is
// only handed to the next block when its SLOWEST query is done, and candidate lists differ in length, so small
// blocks let the hardware scheduler balance the ~2 queries per resident warp slot (10 000 queries at C2).
// FULL = the trace length is exactly 128 (one whole leaf, no tail): every bounds predicate of the SMALL path folds away.
template <typename T, bool SMALL, int WPB, bool FULL = false>
__global__ void __launch_bounds__(32 * WPB, (sizeof(T) == 4 ? (SMALL ? 32 : 16) : 8) / WPB)
rerank_list_kernel(const RerankArgs<T> a) {
  using R = Rn<T>;
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * WPB + (threadIdx.x >> 5);
  if (row >= a.m) return;
  const int sub = lane & 7, grp = lane >> 3;
  // The work per query is a chain of dependent loads; issue everything that does not depend on
  // another load at once: the count, the class, the query row and (speculatively — the slots
  // exist whatever the count) the first four candidate entries, one per 8-lane group.
  const int cnt = a.cand_cnt ? a.cand_cnt[row] : 0;
  const int cls = a.q_class ? a.q_class[row] : 0;
  const bool spec = a.cand_cnt != nullptr && a.cap >= 4;
  int2 first = make_int2(0, 0);
  if (spec) first = *reinterpret_cast<const int2*>(a.cand_idx + (row * (int64_t)a.cap + grp) * 2);
  const T* x = query_row(a, row);
  const int n = FULL ? 128 : a.d;
  const int lim = FULL ? 128 : n - (n % 8);
  T xr[SMALL ? 16 : 1], xt[SMALL ? 7 : 1];
  if (SMALL) {
#pragma unroll
    for (int u = 0; u < 16; u++) xr[u] = 8 * u + sub < lim ? x[8 * u + sub] : (T)0;
#pragma unroll
    for (int u = 0; u < 7; u++) xt[u] = lim + u < n ? x[lim + u] : (T)0;
  }
  if (cls < 0 || cls >= a.n_classes) {   // never scored by the reference either
    Best<T> none{Rn<T>::inf(), 0x7fffffff, -1};
    write_result(a, row, none, lane);
    return;
  }
  if (a.cand_cnt == nullptr || cnt < 1 || cnt > a.cap) {
    if (lane == 0) {
      if (a.count_only) atomicAdd(a.work, 1);
      else a.work[1 + atomicAdd(a.work, 1)] = (int32_t)row;
    }
    return;
  }
  const int c0 = a.class_off[cls], c1 = a.class_off[cls + 1], cn = a.class_off[a.n_classes];
  const unsigned gmask = 0xFFu << (lane & 24);
  Best<T> best{Rn<T>::inf(), 0x7fffffff, -1};
  // entries are (first train row of a 32-row chunk, 32-bit mask of the rows inside the window);
  // the four 8-lane groups of the warp take entries round-robin and walk their mask bits
  for (int e0 = 0; e0 < cnt; e0 += 4) {
    const int e = e0 + grp;
    if (e < cnt) {
      int2 ent = first;
      if (!(spec && e0 == 0)) ent = *reinterpret_cast<const int2*>(a.cand_idx + (row * (int64_t)a.cap + e) * 2);
      const int start = ent.x;
      unsigned cmask = (unsigned)ent.y;
      while (cmask) {
        const int bit = __ffs(cmask) - 1;
        cmask &= cmask - 1;
        const int j = start + bit;
        if (j < 0 || j >= a.n) continue;
        // the filter only flags rows of the item's span, so the class-range test (which waits for
        // class_off) practically never rejects: it is applied after the row has been fetched
        const int gid = a.t_gid ? a.t_gid[j] : j;
        const T* y = a.t + (int64_t)j * a.d;
        T s;
        if (SMALL) {
          // NumPy's leaf (n <= 128): n < 8 sequential from 0; else the stride-8 accumulator of this
          // lane, the tree ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)) by xor-shuffles, then the tail
          T yr[16], yt[7];
#pragma unroll
          for (int u = 0; u < 16; u++) yr[u] = 8 * u + sub < lim ? y[8 * u + sub] : (T)0;
#pragma unroll
          for (int u = 0; u < 7; u++) yt[u] = lim + u < n ? y[lim + u] : (T)0;
          T r = (T)0;
          if (lim > 0) {
            T d0 = R::sub(xr[0], yr[0]);
            r = R::mul(d0, d0);
#pragma unroll
            for (int u = 1; u < 16; u++) {
              if (8 * u < lim) {          // uniform: lim is a multiple of 8
                const T du = R::sub(xr[u], yr[u]);
                r = R::add(r, R::mul(du, du));
              }
            }
            r = R::add(r, __shfl_xor_sync(gmask, r, 1));
            r = R::add(r, __shfl_xor_sync(gmask, r, 2));
            r = R::add(r, __shfl_xor_sync(gmask, r, 4));
          }
#pragma unroll
          for (int u = 0; u < 7; u++) {
            if (lim + u < n) {
              const T du = R::sub(xt[u], yt[u]);
              r = R::add(r, R::mul(du, du));
            }
          }
          s = r;
        } else {
          s = a.sum_prog ? np_sumsq_prog_g8<T>(x, y, a.sum_prog, a.sum_leaves, sub, gmask)
                         : np_sumsq_g8<T>(x, y, a.d, sub, gmask);
        }
        const bool in_range = a.mode == TIP_RANGE_SAME_CLASS ? (j >= c0 && j < c1) : (j < cn && (j < c0 || j >= c1));
        if (in_range) consider(best, Rn<T>::sqrt(s), gid, j);   // all 8 lanes agree
      }
    }
  }
  __syncwarp();
  for (int o = 8; o < 32; o <<= 1) {
    const T od = __shfl_xor_sync(0xffffffffu, best.dist, o);
    const int og = __shfl_xor_sync(0xffffffffu, best.gid, o);
    const int op = __shfl_xor_sync(0xffffffffu, best.pos, o);
    best = merge(best, od, og, op);
  }
  // (no global statistics here: one same-address atomic per query serialises in L2; candidate
  // counts can be read from cand_cnt)
  write_result(a, row, best, lane);
}

// ---- kernels 2+3: exhaustive scan of the class range for queued queries ---------------------------
// The queue is normally empty or a handful of queries, each needing up to N x D work, so every
// queued query is split into S column slices ("units") spread over the whole grid; a unit writes
// its local winner to scratch and a merge kernel picks the lexicographic minimum per query.
constexpr int kScanUnitTarget = 4096;

__device__ __forceinline__ int scan_slices(int queued) {
  const int s = kScanUnitTarget / max(queued, 1);
  return s < 1 ? 1 : (s > 64 ? 64 : s);
}

template <typename T>
struct ScanScratch {
  T* dist;
  int32_t* gid;
  int32_t* pos;
};

template <typename T>
__device__ __forceinline__ ScanScratch<T> scan_scratch(const RerankArgs<T>& a) {
  // layout after the queue (1 + m ints) and the completion counter (1 int):
  // [cap] T dist (8-byte aligned), [cap] gid, [cap] pos
  const int64_t cap = a.m + kScanUnitTarget;
  uintptr_t base = reinterpret_cast<uintptr_t>(a.work + 2 + a.m);
  base = (base + 7) & ~(uintptr_t)7;
  ScanScratch<T> sc;
  sc.dist = reinterpret_cast<T*>(base);
  sc.gid = reinterpret_cast<int32_t*>(sc.dist + cap);
  sc.pos = sc.gid + cap;
  return sc;
}

template <typename T>
__device__ __forceinline__ void rerank_merge(const RerankArgs<T>& a, int queued) {
  // executed by the last block of rerank_scan_kernel (kScanThreads threads)
  const int S = scan_slices(queued);
  const ScanScratch<T> sc = scan_scratch(a);
  const int lane = threadIdx.x & 31;
  constexpr int kWarps = kScanThreads / 32;
  for (int w = threadIdx.x >> 5; w < queued; w += kWarps) {
    Best<T> best{Rn<T>::inf(), 0x7fffffff, -1};
    for (int sl = lane; sl < S; sl += 32) {
      const int64_t u = (int64_t)w * S + sl;
      best = merge(best, sc.dist[u], sc.gid[u], sc.pos[u]);
    }
    for (int o = 1; o < 32; o <<= 1) {
      const T od = __shfl_xor_sync(0xffffffffu, best.dist, o);
      const int og = __shfl_xor_sync(0xffffffffu, best.gid, o);
      const int op = __shfl_xor_sync(0xffffffffu, best.pos, o);
      best = merge(best, od, og, op);
    }
    if (lane == 0 && a.stats) atomicAdd(a.stats + 0, 1ULL);
    write_result(a, a.work[1 + w], best, lane);
  }
}

template <typename T>
__global__ void __launch_bounds__(kScanThreads) rerank_scan_kernel(const RerankArgs<T> a) {
  __shared__ T s_dist[kScanThreads / 8];
  __shared__ int s_gid[kScanThreads / 8];
  __shared__ int s_pos[kScanThreads / 8];
  const int queued = a.work[0];
  if (queued == 0) return;
  const int S = scan_slices(queued);
  const ScanScratch<T> sc = scan_scratch(a);
  const int sub = threadIdx.x & 7, grp = threadIdx.x >> 3;
  constexpr int kGroups = kScanThreads / 8;
  const unsigned gmask = 0xFFu << (threadIdx.x & 24);
  const int64_t units = (int64_t)queued * S;
  for (int64_t u = blockIdx.x; u < units; u += gridDim.x) {
    const int w = (int)(u / S), sl = (int)(u % S);
    const int64_t row = a.work[1 + w];
    const int cls = a.q_class ? a.q_class[row] : 0;
    const T* x = query_row(a, row);
    Best<T> best{Rn<T>::inf(), 0x7fffffff, -1};
    const int c0 = a.class_off[cls], c1 = a.class_off[cls + 1], cn = a.class_off[a.n_classes];
    // SAME_CLASS: [c0, c1);  OTHER_CLASSES: [0, c0) U [c1, cn) — as one linear index space
    const int len0 = a.mode == TIP_RANGE_SAME_CLASS ? c1 - c0 : c0;
    const int len1 = a.mode == TIP_RANGE_SAME_CLASS ? 0 : cn - c1;
    const int base0 = a.mode == TIP_RANGE_SAME_CLASS ? c0 : 0;
    const int64_t total = (int64_t)len0 + len1;
    const int64_t lo = total * sl / S, hi = total * (sl + 1) / S;
    for (int64_t li = lo + grp; li < hi; li += kGroups) {
      const int j = li < len0 ? base0 + (int)li : c1 + (int)(li - len0);
      const T s = a.sum_prog ? np_sumsq_prog_g8<T>(x, a.t + (int64_t)j * a.d, a.sum_prog, a.sum_leaves, sub, gmask)
                             : np_sumsq_g8<T>(x, a.t + (int64_t)j * a.d, a.d, sub, gmask);
      consider(best, Rn<T>::sqrt(s), a.t_gid ? a.t_gid[j] : j, j);
    }
    if (sub == 0) { s_dist[grp] = best.dist; s_gid[grp] = best.gid; s_pos[grp] = best.pos; }
    __syncthreads();
    if (threadIdx.x == 0) {
      Best<T> b{Rn<T>::inf(), 0x7fffffff, -1};
      for (int g = 0; g < kGroups; g++) b = merge(b, s_dist[g], s_gid[g], s_pos[g]);
      sc.dist[u] = b.dist; sc.gid[u] = b.gid; sc.pos[u] = b.pos;
    }
    __syncthreads();
  }
  // completion: the last block merges the slices of every queued query and re-arms the queue
  __shared__ int s_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(a.work + 1 + a.m, 1) == (int)gridDim.x - 1);
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  rerank_merge(a, queued);
  __syncthreads();
  if (threadIdx.x == 0) {
    a.work[0] = 0;
    a.work[1 + a.m] = 0;
  }
}

template <typename T>
static int launch_rerank(const RerankArgs<T>& a, cudaStream_t st) {
  // precondition (and postcondition): work[0] == 0 and work[1 + m] == 0
  // queries (warps) per block, measured with 8 / 2 / 1 (one box): C2 0.1943 / 0.1926 / 0.1928 ms per step, long traces
  // (C5 slice) 40.4 / 40.6 / 40.9.  One 8-lane group per query instead of a warp was slower at C2 (0.216 vs 0.199 ms).
  if (a.d == 128) rerank_list_kernel<T, true, 2, true><<<(unsigned)((a.m + 1) / 2), 64, 0, st>>>(a);
  else if (a.d < 128) rerank_list_kernel<T, true, 2><<<(unsigned)((a.m + 1) / 2), 64, 0, st>>>(a);
  else rerank_list_kernel<T, false, 8><<<(unsigned)((a.m + 7) / 8), 256, 0, st>>>(a);
  TIP_LAUNCH_CHECK();
  if (a.count_only) return TIP_OK;   // speculative call: no exhaustive-scan launch, the caller inspects work[0]
  // normally an empty queue: every block returns at once, so keep the grid small (the fallback itself is rare)
  rerank_scan_kernel<T><<<sm_count() * 2, kScanThreads, 0, st>>>(a);
  TIP_LAUNCH_CHECK();
  return TIP_OK;
}

}  // namespace tip

using namespace tip;

static int next_pitch_k16(int64_t d) {     // K=16 steps of the one-segment packed row (pair_tc.cu: k16_of(d, 1))
  const int64_t d16 = (d + 15) & ~(int64_t)15;
  return (int)((d16 + 16) / 16);
}

// NumPy's pairwise schedule for width d as one word per leaf (common.cuh: np_sumsq_prog_g8), cached per
// (device, d) in device memory.  Built outside stream capture: the first search of an engine is eager.
static void build_sum_prog(int off, int n, std::vector<uint32_t>& prog) {
  if (n <= 128) {
    prog.push_back((uint32_t)(off / 8) | ((uint32_t)(n - 1) << 20));
    return;
  }
  int n2 = n / 2;
  n2 -= n2 % 8;
  build_sum_prog(off, n2, prog);
  build_sum_prog(off + n2, n - n2, prog);
  prog.back() += 1u << 27;          // after the right subtree: merge it with the left one
}

static int get_sum_prog(int64_t d, const uint32_t** dev_prog, int* n_leaves) {
  static std::mutex mu;
  static std::map<std::pair<int, int64_t>, std::pair<uint32_t*, int>> cache;
  *dev_prog = nullptr;
  *n_leaves = 0;
  if (d <= 128 || d > (8LL << 20)) return TIP_OK;      // short traces: register-resident leaf; absurd widths: generic routine
  int dev = 0;
  TIP_CHECK_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(mu);
  auto it = cache.find({dev, d});
  if (it == cache.end()) {
    std::vector<uint32_t> prog;
    build_sum_prog(0, (int)d, prog);
    for (uint32_t w : prog)
      if ((w >> 27) >= 31) return TIP_OK;               // cannot happen below 2^31 elements; fall back if it does
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    uint32_t* p = nullptr;
    TIP_CHECK_CUDA(cudaMalloc(&p, prog.size() * sizeof(uint32_t)));
    TIP_CHECK_CUDA(cudaMemcpy(p, prog.data(), prog.size() * sizeof(uint32_t), cudaMemcpyHostToDevice));
    (void)cap;
    it = cache.emplace(std::make_pair(dev, d), std::make_pair(p, (int)prog.size())).first;
  }
  *dev_prog = it->second.first;
  *n_leaves = it->second.second;
  return TIP_OK;
}

extern "C" int32_t tip_sizeof_rerank_extras(void) { return (int32_t)sizeof(tip_rerank_extras); }

extern "C" int64_t tip_nn_rerank_work_bytes(int64_t m, int dtype) {
  if (m < 0) return -1;
  const int64_t cap = m + kScanUnitTarget;
  return (2 + m) * 4 + 8 + cap * ((dtype == TIP_F64 ? 8 : 4) + 8);
}

extern "C" int tip_nn_rerank(const void* q, const void* t, int dtype, int64_t m, int64_t n, int64_t d,
                             const int32_t* cand_idx, const int32_t* cand_cnt, int32_t cap, const int32_t* q_class,
                             const int32_t* class_off, int32_t n_classes, int mode, const int32_t* t_gid,
                             void* out_dist, int32_t* out_pos, int32_t* out_gid, void* out_rows, int32_t* work,
                             int64_t* stats, const float* next_center, void* next_pack, float* next_sqnorm,
                             float* next_rounderr, uint32_t* next_row_min_bits, int32_t* next_cand_cnt,
                             const tip_rerank_extras* extras, void* stream) {
  TIP_REQUIRE(q && t && out_dist && out_pos && work, "null pointer");
  const tip_rerank_extras ex = extras ? *extras : tip_rerank_extras{};
  const float* next_seed_ub = ex.next_seed_ub;
  const float next_t_rmax = ex.next_t_rmax, next_t_errmax = ex.next_t_errmax;
  TIP_REQUIRE(next_seed_ub == nullptr || (next_pack && next_rounderr), "seeds need the next-stage query state incl. rounderr");
  TIP_REQUIRE(ex.fin_out == nullptr || (ex.fin_dist_a && ex.fin_gid && ex.fin_n_total >= 0), "fused result scatter: dist_a, gid, n_total");
  TIP_REQUIRE(class_off && n_classes >= 1, "class offsets");
  TIP_REQUIRE(m >= 0 && m < (1LL << 31) - 8 && n >= 0 && n < (1LL << 31) && d >= 1 && d < (1LL << 31), "shape");
  TIP_REQUIRE(mode == TIP_RANGE_SAME_CLASS || mode == TIP_RANGE_OTHER_CLASSES, "mode");
  TIP_REQUIRE(cand_cnt == nullptr || (cand_idx != nullptr && cap >= 1), "candidate buffers");
  TIP_REQUIRE(next_pack == nullptr || (next_sqnorm && next_row_min_bits && next_cand_cnt),
              "next-stage query state: pack, sqnorm, row_min_bits and cand_cnt go together");
  TIP_REQUIRE(!ex.count_overflow_only || cand_cnt != nullptr, "count_overflow_only needs candidate lists");
  if (m == 0) return TIP_OK;
  const int count_only = ex.count_overflow_only != 0;
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t next_pitch = tip_pair_pitch(d, 1);
  const uint32_t* sum_prog = nullptr;
  int sum_leaves = 0;
  {
    const int rc = get_sum_prog(d, &sum_prog, &sum_leaves);
    if (rc != TIP_OK) return rc;
  }
  // gamma of tip_nn_filter for this trace width (packed width + 16 fp32 accumulation steps)
  const SeedParams seed{next_seed_ub, next_t_rmax, next_t_errmax, (float)(next_pitch_k16(d) * 16 + 16) * 1.1920929e-7f};
  if (dtype == TIP_F32) {
    RerankArgs<float> a{(const float*)q, (const float*)t, m, n, (int)d, cand_idx, cand_cnt, cap, q_class, class_off,
                        n_classes, mode, t_gid, (float*)out_dist, out_pos, out_gid, (float*)out_rows, work,
                        (unsigned long long*)stats, next_center, (__nv_bfloat16*)next_pack, next_pitch, next_sqnorm,
                        next_rounderr, next_row_min_bits, next_cand_cnt, seed, ex.q_idx, (const float*)ex.fin_dist_a,
                        ex.fin_gid, ex.fin_idx, ex.fin_n_total, ex.fin_out, sum_prog, sum_leaves, count_only};
    return launch_rerank<float>(a, st);
  }
  if (dtype == TIP_F64) {
    RerankArgs<double> a{(const double*)q, (const double*)t, m, n, (int)d, cand_idx, cand_cnt, cap, q_class,
                         class_off, n_classes, mode, t_gid, (double*)out_dist, out_pos, out_gid, (double*)out_rows,
                         work, (unsigned long long*)stats, next_center, (__nv_bfloat16*)next_pack, next_pitch,
                         next_sqnorm, next_rounderr, next_row_min_bits, next_cand_cnt, seed, ex.q_idx, (const double*)ex.fin_dist_a,
                         ex.fin_gid, ex.fin_idx, ex.fin_n_total, ex.fin_out, sum_prog, sum_leaves, count_only};
    return launch_rerank<double>(a, st);
  }
  TIP_REQUIRE(false, "dtype must be TIP_F32 or TIP_F64");
}
