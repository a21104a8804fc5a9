// simple.cu — bandwidth-bound kernels and small utilities of libb200tip.so:
//   DeepGini (deepgini.py:31-35), KMNC (neuron_coverage.py:65-94), operand packing for the
//   tensor-core pass, row gather, LSA whitening, LSE partial merge, and the C-ABI basics.
#include <stdarg.h>
#include <algorithm>

#include <atomic>
#include <map>
#include <mutex>
#include <vector>

#include <cuda_fp16.h>
#include "common.cuh"

namespace tip {

static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }

int sm_count() {
  static int cached = 0;
  if (!cached) {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) == cudaSuccess &&
        cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0)
      cached = n;
    else
      return 148;
  }
  return cached;
}

// =============================================================================================
// DeepGini
// =============================================================================================
// Narrow rows (c <= kGiniSmallC): a block stages 128 rows in shared memory with coalesced
// 16-byte-agnostic loads, then one thread per row walks its row in NumPy's pairwise order.
constexpr int kGiniRows = 128;

template <typename T>
__global__ void __launch_bounds__(kGiniRows) gini_small_kernel(const T* __restrict__ p, int64_t n, int c,
                                                               int32_t* __restrict__ pred,
                                                               T* __restrict__ gini) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  T* tile = reinterpret_cast<T*>(smem_raw);
  const int stride = c + 1;  // +1 padding: thread r reads tile[r*stride + k], conflict-free for odd strides
  for (int64_t row0 = (int64_t)blockIdx.x * kGiniRows; row0 < n; row0 += (int64_t)gridDim.x * kGiniRows) {
    const int rows = (int)min((int64_t)kGiniRows, n - row0);
    const T* src = p + row0 * c;
    const int total = rows * c;
    for (int i = threadIdx.x; i < total; i += kGiniRows) {
      const int r = i / c, k = i - r * c;
      tile[r * stride + k] = src[i];
    }
    __syncthreads();
    if (threadIdx.x < rows) {
      const T* row = tile + threadIdx.x * stride;
      int best = 0;
      T bv = row[0];
      for (int k = 1; k < c; k++) {
        const T v = row[k];
        if (v > bv) { bv = v; best = k; }
      }
      const T ss = np_sumsq<T>(row, nullptr, c);
      pred[row0 + threadIdx.x] = best;
      gini[row0 + threadIdx.x] = Rn<T>::sub((T)1, ss);
    }
    __syncthreads();
  }
}

// Wide rows: one warp per row.  NumPy's pairwise tree for a row of c elements is fixed, so the
// host builds it once per width: the list of <=128-element leaves and a post-order combine
// program.  The row is staged in shared memory with coalesced loads; the four 8-lane groups of
// the warp evaluate leaves cooperatively (lane j owns NumPy's stride-8 accumulator j), lane 0 then
// runs the combine program over the leaf sums.
constexpr int kGiniMaxLeaves = 1024;
constexpr int kGiniStageElems = 4096;   // rows up to this width are staged in shared memory

struct GiniTree {
  int n_leaves = 0, n_prog = 0;
  int* leaf_off = nullptr;   // device: [n_leaves]
  int* leaf_len = nullptr;   // device: [n_leaves]
  short* prog = nullptr;     // device: [n_prog], >= 0: push leaf, -1: pop two, push their sum
};

static void gini_build(int off, int n, std::vector<int>& lo, std::vector<int>& ll, std::vector<short>& prog) {
  if (n <= 128) {
    prog.push_back((short)lo.size());
    lo.push_back(off);
    ll.push_back(n);
    return;
  }
  int n2 = n / 2;
  n2 -= n2 % 8;
  gini_build(off, n2, lo, ll, prog);
  gini_build(off + n2, n - n2, lo, ll, prog);
  prog.push_back(-1);
}

static int gini_tree_for(int c, GiniTree* out) {
  static std::mutex mu;
  static std::map<int, GiniTree> cache;
  std::lock_guard<std::mutex> lock(mu);
  auto it = cache.find(c);
  if (it == cache.end()) {
    std::vector<int> lo, ll;
    std::vector<short> prog;
    gini_build(0, c, lo, ll, prog);
    GiniTree t;
    t.n_leaves = (int)lo.size();
    t.n_prog = (int)prog.size();
    TIP_CHECK_CUDA(cudaMalloc(&t.leaf_off, lo.size() * sizeof(int)));
    TIP_CHECK_CUDA(cudaMalloc(&t.leaf_len, ll.size() * sizeof(int)));
    TIP_CHECK_CUDA(cudaMalloc(&t.prog, prog.size() * sizeof(short)));
    TIP_CHECK_CUDA(cudaMemcpy(t.leaf_off, lo.data(), lo.size() * sizeof(int), cudaMemcpyHostToDevice));
    TIP_CHECK_CUDA(cudaMemcpy(t.leaf_len, ll.data(), ll.size() * sizeof(int), cudaMemcpyHostToDevice));
    TIP_CHECK_CUDA(cudaMemcpy(t.prog, prog.data(), prog.size() * sizeof(short), cudaMemcpyHostToDevice));
    it = cache.emplace(c, t).first;
  }
  *out = it->second;
  return TIP_OK;
}

template <typename T>
__global__ void __launch_bounds__(128) gini_wide_kernel(const T* __restrict__ p, int64_t n, int c, GiniTree tree,
                                                        bool staged, int32_t* __restrict__ pred,
                                                        T* __restrict__ gini) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int sub = lane & 7, grp = lane >> 3;
  const unsigned gmask = 0xFFu << (lane & 24);
  // per-warp scratch sized by the actual tree / row width (occupancy: smem is what limits it)
  T* leaf_sums = reinterpret_cast<T*>(smem_raw) + warp * tree.n_leaves;
  T* stage = reinterpret_cast<T*>(smem_raw) + 4 * tree.n_leaves + warp * c;
  for (int64_t row = (int64_t)blockIdx.x * 4 + warp; row < n; row += (int64_t)gridDim.x * 4) {
    const T* src = p + row * c;
    // coalesced pass: argmax (first occurrence) and, if the row fits, a copy into shared memory
    T bv = src[0];
    int bi = 0;
    for (int k = lane; k < c; k += 32) {
      const T v = src[k];
      if (staged) stage[k] = v;
      if (v > bv || (v == bv && k < bi)) { bv = v; bi = k; }
    }
    for (int o = 16; o > 0; o >>= 1) {
      const T ov = __shfl_xor_sync(0xffffffffu, bv, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (ov > bv || (ov == bv && oi < bi)) { bv = ov; bi = oi; }
    }
    __syncwarp();
    const T* x = staged ? stage : src;
    for (int l0 = 0; l0 < tree.n_leaves; l0 += 4) {
      const int l = l0 + grp;
      if (l < tree.n_leaves) {
        const T s = np_leaf_sumsq_g8<T>(x + tree.leaf_off[l], nullptr, tree.leaf_len[l], sub, gmask);
        if (sub == 0) leaf_sums[l] = s;
      }
    }
    __syncwarp();
    if (lane == 0) {
      T stack[32];
      int sp = 0;
      for (int i = 0; i < tree.n_prog; i++) {
        const int op = tree.prog[i];
        if (op >= 0) stack[sp++] = leaf_sums[op];
        else { const T r = stack[--sp]; const T a = stack[--sp]; stack[sp++] = Rn<T>::add(a, r); }
      }
      pred[row] = bi;
      gini[row] = Rn<T>::sub((T)1, stack[0]);
    }
    __syncwarp();
  }
}

template <typename T>
static int launch_gini(const T* p, int64_t n, int64_t c, int32_t* pred, T* gini, cudaStream_t st) {
  const int sms = sm_count();
  const size_t small_bytes = (size_t)kGiniRows * (size_t)(c + 1) * sizeof(T);
  if (small_bytes <= 96 * 1024) {
    TIP_CHECK_CUDA(cudaFuncSetAttribute(gini_small_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)small_bytes));
    const int64_t blocks = (n + kGiniRows - 1) / kGiniRows;
    const int grid = (int)std::min<int64_t>(blocks, (int64_t)sms * 8);
    gini_small_kernel<T><<<grid, kGiniRows, small_bytes, st>>>(p, n, (int)c, pred, gini);
  } else {
    TIP_REQUIRE(c <= (int64_t)kGiniMaxLeaves * 64, "row too wide");
    GiniTree tree;
    int rc = gini_tree_for((int)c, &tree);
    if (rc != TIP_OK) return rc;
    TIP_REQUIRE(tree.n_leaves <= kGiniMaxLeaves, "row too wide");
    const bool staged = c <= kGiniStageElems;
    const size_t bytes = 4 * (size_t)tree.n_leaves * sizeof(T) + (staged ? 4 * (size_t)c * sizeof(T) : 0);
    TIP_CHECK_CUDA(cudaFuncSetAttribute(gini_wide_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)(4 * (kGiniMaxLeaves + kGiniStageElems) * sizeof(T))));
    const int grid = (int)std::min<int64_t>((n + 3) / 4, (int64_t)sms * 16);
    gini_wide_kernel<T><<<grid, 128, bytes, st>>>(p, n, (int)c, tree, staged, pred, gini);
  }
  TIP_LAUNCH_CHECK();
  return TIP_OK;
}

// =============================================================================================
// KMNC
// =============================================================================================
template <typename TA, typename TS> struct CmpType { using type = double; };
template <> struct CmpType<float, float> { using type = float; };

template <typename TA, typename TS>
__device__ __forceinline__ int kmnc_bucket(TA a_in, TS lo, TS jump, int k) {
  using TC = typename CmpType<TA, TS>::type;
  using R = Rn<TS>;
  if (!(jump > (TS)0)) return -1;  // constant / inverted / NaN range: never covered
  const TC a = (TC)a_in;
  auto t = [&](int i) -> TC { return (TC)R::add(lo, R::mul(jump, (TS)i)); };  // NumPy: min + jumps*i
  // cheap estimate of the section, then exact fix-up against the NumPy-rounded thresholds
  int i;
  if (sizeof(TA) == 4 && sizeof(TS) == 4) {
    const float est = __fdividef((float)a_in - (float)lo, (float)jump);
    i = est >= (float)(k - 1) ? k - 1 : (est > 0.f ? (int)est : 0);
  } else {
    const double est = ((double)a_in - (double)lo) / (double)jump;
    i = est >= (double)(k - 1) ? k - 1 : (est > 0.0 ? (int)est : 0);
  }
  // common case: the estimate is already the section (one exact check); otherwise walk
  if (a >= t(i) && a < t(i + 1)) return i;
  while (i > 0 && a < t(i)) i--;
  while (i < k - 1 && a >= t(i + 1)) i++;
  // i is now the only possible section; NaN / out-of-range values fail this test
  return (a >= t(i) && a < t(i + 1)) ? i : -1;
}

// float traces + float statistics: the hot configuration.  ~16 instructions on the common path
// (estimate, clamp, the two NumPy-rounded thresholds around it, one exact check); anything unusual
// (section edge, constant neuron, out of range, NaN) takes the generic routine.
__device__ __noinline__ int kmnc_bucket_slow(float a, float lo, float jump, int k) {
  return kmnc_bucket<float, float>(a, lo, jump, k);
}

__device__ __forceinline__ int kmnc_bucket_ff(float a, float lo, float jump, int k) {
  const float est = __fdividef(__fsub_rn(a, lo), jump);
  int i = __float2int_rd(est);
  i = min(max(i, 0), k - 1);
  const float fi = (float)i;
  const float t0 = __fadd_rn(lo, __fmul_rn(jump, fi));
  const float t1 = __fadd_rn(lo, __fmul_rn(jump, fi + 1.0f));   // (float)(i+1) == fi + 1 exactly for i < 2^24
  if (a >= t0 && a < t1 && jump > 0.f) return i;
  return kmnc_bucket_slow(a, lo, jump, k);
}

template <typename TA, typename TS, typename TB>
__global__ void __launch_bounds__(256) kmnc_kernel(const TA* __restrict__ act, int64_t n, int64_t d,
                                                   const TS* __restrict__ mins, const TS* __restrict__ jumps,
                                                   int k, TB* __restrict__ bucket, int32_t* __restrict__ score) {
  __shared__ int warp_cnt[8];
  for (int64_t row = blockIdx.x; row < n; row += gridDim.x) {
    const TA* a = act + row * d;
    TB* b = bucket ? bucket + row * d : nullptr;
    int cnt = 0;
    for (int64_t j = threadIdx.x; j < d; j += 256) {
      const int i = kmnc_bucket<TA, TS>(a[j], mins[j], jumps[j], k);
      cnt += (i >= 0);
      if (b) b[j] = (TB)i;
    }
    cnt = warp_sum(cnt);
    if ((threadIdx.x & 31) == 0) warp_cnt[threadIdx.x >> 5] = cnt;
    __syncthreads();
    if (threadIdx.x == 0) {
      int s = 0;
      for (int w = 0; w < 8; w++) s += warp_cnt[w];
      score[row] = s;
    }
    __syncthreads();
  }
}

// float traces, float statistics, d % 4 == 0, 16-byte aligned: 128-bit loads, 64-bit stores.
// One warp owns 128 consecutive neurons of one sample at a time (grid-stride over such chunks);
// per-sample counts are accumulated with one atomic per chunk into a zeroed score array.
template <typename TB>
__global__ void __launch_bounds__(256) kmnc_vec4_kernel(const float* __restrict__ act, int64_t n, int64_t d,
                                                        const float* __restrict__ mins,
                                                        const float* __restrict__ jumps, int k,
                                                        TB* __restrict__ bucket, int32_t* __restrict__ score) {
  const int lane = threadIdx.x & 31;
  const int64_t d4 = d >> 2;
  const int64_t cpr = (d4 + 31) >> 5;  // chunks per row
  const int64_t total = n * cpr;
  const bool small = total < (1LL << 31);
  const int64_t nwarps = (int64_t)gridDim.x * 8;
  constexpr int kUnroll = 4;   // four independent 16-byte loads in flight per thread
  for (int64_t chunk0 = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); chunk0 < total; chunk0 += nwarps * kUnroll) {
    float4 v[kUnroll];
    int64_t row[kUnroll], j[kUnroll];
    bool ok[kUnroll];
#pragma unroll
    for (int u = 0; u < kUnroll; u++) {
      const int64_t chunk = chunk0 + (int64_t)u * nwarps;
      // 64-bit division is emulated (~70 instructions); chunk indices fit 32 bits in practice
      row[u] = small ? (int64_t)((uint32_t)chunk / (uint32_t)cpr) : chunk / cpr;
      j[u] = (chunk - row[u] * cpr) * 32 + lane;
      ok[u] = chunk < total && j[u] < d4;
      if (ok[u]) {
        asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
                     : "=f"(v[u].x), "=f"(v[u].y), "=f"(v[u].z), "=f"(v[u].w)
                     : "l"(reinterpret_cast<const float4*>(act + row[u] * d) + j[u]));
      }
    }
#pragma unroll
    for (int u = 0; u < kUnroll; u++) {
      int cnt = 0;
      if (ok[u]) {
        const float4 lo = __ldg(reinterpret_cast<const float4*>(mins) + j[u]);
        const float4 jp = __ldg(reinterpret_cast<const float4*>(jumps) + j[u]);
        const int i0 = kmnc_bucket_ff(v[u].x, lo.x, jp.x, k);
        const int i1 = kmnc_bucket_ff(v[u].y, lo.y, jp.y, k);
        const int i2 = kmnc_bucket_ff(v[u].z, lo.z, jp.z, k);
        const int i3 = kmnc_bucket_ff(v[u].w, lo.w, jp.w, k);
        cnt = (i0 >= 0) + (i1 >= 0) + (i2 >= 0) + (i3 >= 0);
        if (bucket) {
          TB* bp = bucket + row[u] * d + (j[u] << 2);
          if (sizeof(TB) == 2) {
            *reinterpret_cast<short4*>(bp) = make_short4((short)i0, (short)i1, (short)i2, (short)i3);
          } else {
            *reinterpret_cast<int4*>(bp) = make_int4(i0, i1, i2, i3);
          }
        }
      }
      if (chunk0 + (int64_t)u * nwarps < total) {   // warp-uniform
        cnt = warp_sum(cnt);
        if (lane == 0 && cnt) atomicAdd(score + row[u], cnt);
      }
    }
  }
}

// Column-strip variant of the above for the hot configuration (many samples): a block owns a strip
// of 1024 neurons and a contiguous share of the samples; every thread keeps the fast-path constants of its
// four neurons in registers and walks down its samples with kStripRows independent 16-byte loads in flight,
// so the inner loop is load -> ~12 ALU instructions per value -> 8-byte store with no index arithmetic and
// no statistics traffic.  Per-sample counts: REDUX over the warp -> one `red` per (sample, warp).  The grid is
// one resident wave (occupancy x SMs, rounded down to a multiple of the strip count) and the samples are split
// evenly over the blocks of a strip, so there is no partial last wave.
constexpr int kStripRows = 8;

// Section index without threshold arithmetic on the common path.  e = (a - lo) / jump is estimated as
// fma(a - lo, 1/jump, -1/2) and rounded to an integer by adding 1.5 * 2^23 (no F2I / I2F: those run on the
// quarter-rate XU pipe); the low mantissa bits of the biased float ARE the integer.  The estimate is accepted
// without looking at a threshold when e - 1/2 lies within `lim` = 1/2 - delta of that integer, i.e. when a is
// at least delta sections away from both neighbouring thresholds, where delta bounds everything that separates
// the estimate from NumPy's comparison against its rounded thresholds  T_i = fl(min + fl(jumps * i))
// (neuron_coverage.py:73-79, 87-91), in units of one section, u = 2^-24:
//     |T_i - (min + jumps*i)| / jumps  <=  u (2 i + |min| / jumps)(1 + u)            (two roundings)
//     |e_computed - e_exact|           <=  3.1 u (|e| + 1)                           (a - lo, 1/jump, product)
//   delta = 1.01 u (5.1 (k + 1) + |min| / jumps + 2)      — 3e-4 at k = 1000: 0.06 % of the values take the exact path
// (kmnc_bucket_slow: the two NumPy-rounded thresholds around the estimate, then a walk).  Below the range the
// sign of a - lo is exact (T_0 = min), above it e >= k + delta puts a beyond T_k: both yield -1 without a test.
//
// a == min exactly (every zero of a ReLU layer whose minimum is 0) sits ON the edge T_0 and would fail the margin
// test, but e = 0 there with no rounding anywhere: section 0 is certain as long as T_1 = fl(min + jump) > min, and
// the rounded estimate is 0 as well (-1/2 + 1.5 * 2^23 ties to even).  Neurons for which that does not hold, or
// whose delta exceeds 1/2 or is not a number, get lo = NaN on the fast path: then neither a - lo == 0 nor the margin test can
// pass and every value of that neuron takes the exact path (which reads the true statistics from memory).
// A neuron that can never be covered (jump <= 0 or NaN: constant / inverted range) costs nothing extra: its
// inv is 0 and its lim +inf, so every finite activation passes the test, and its section count kk = 0 (k for the
// others) turns the result into -1.
struct KmncLane {
  float lo, inv, lim;
  int kk;
};

__device__ __forceinline__ KmncLane kmnc_lane(float lo, float jp, int k) {
  KmncLane s;
  const bool dead = !(jp > 0.f);
  s.inv = dead ? 0.f : 1.0f / jp;
  const float delta = 1.01f * 5.9604645e-8f * (5.1f * (float)(k + 1) + fabsf(lo) * fabsf(s.inv) * 1.0001f + 2.0f);
  // (delta > 1/2 or NaN: jump underflows, 1/jump overflows, |min| / jump is huge — nothing can pass the margin test)
  const bool exact_only = !dead && (!(delta <= 0.5f) || !(__fadd_rn(lo, __fmul_rn(jp, 1.0f)) > lo));
  s.lim = dead ? __int_as_float(0x7f800000) : 0.5f - delta;   // negative: only a == min passes
  s.lo = exact_only ? __int_as_float(0x7fc00000) : lo;
  s.kk = dead ? 0 : k;
  asm volatile("" : "+r"(s.kk));   // keep it a register: recomputing it from jump costs two instructions per value
  return s;
}

__device__ __forceinline__ int kmnc_fast(float a, const KmncLane& s, bool& ok) {
  constexpr float kMagic = 12582912.0f;   // 1.5 * 2^23
  const float x = __fsub_rn(a, s.lo);
  const float eh = __fmaf_rn(x, s.inv, -0.5f);
  const float m = __fadd_rn(eh, kMagic);
  const float fr = __fsub_rn(eh, __fsub_rn(m, kMagic));       // distance of e - 1/2 to the nearest integer
  ok = (fabsf(fr) <= s.lim) || (x == 0.f);                    // NaN / inf / huge values fail -> exact path
  const int i = __float_as_int(m) - 0x4B400000;
  return (unsigned)i < (unsigned)s.kk ? i : -1;
}

__device__ __forceinline__ void red_add_s32_if(int32_t* p, int v, bool on) {   // predicated, no branch
  asm volatile("{ .reg .pred p; setp.ne.b32 p, %2, 0; @p red.global.add.s32 [%0], %1; }" ::"l"(p), "r"(v), "r"((int)on)
               : "memory");
}

// one sample row x four neurons of this thread: sections, optional store, number of covered neurons
template <typename TB, bool STORE>
__device__ __forceinline__ int kmnc_strip_row(const float4 v, const KmncLane& s0, const KmncLane& s1,
                                              const KmncLane& s2, const KmncLane& s3, int k,
                                              const float* __restrict__ lo_g, const float* __restrict__ jp_g,
                                              TB* __restrict__ bp) {
  bool ok0, ok1, ok2, ok3;
  int i0 = kmnc_fast(v.x, s0, ok0);
  int i1 = kmnc_fast(v.y, s1, ok1);
  int i2 = kmnc_fast(v.z, s2, ok2);
  int i3 = kmnc_fast(v.w, s3, ok3);
  if (!(ok0 && ok1 && ok2 && ok3)) {   // within delta of a section edge, NaN, inf: NumPy's thresholds decide
    if (!ok0) i0 = kmnc_bucket_slow(v.x, __ldg(lo_g + 0), __ldg(jp_g + 0), k);
    if (!ok1) i1 = kmnc_bucket_slow(v.y, __ldg(lo_g + 1), __ldg(jp_g + 1), k);
    if (!ok2) i2 = kmnc_bucket_slow(v.z, __ldg(lo_g + 2), __ldg(jp_g + 2), k);
    if (!ok3) i3 = kmnc_bucket_slow(v.w, __ldg(lo_g + 3), __ldg(jp_g + 3), k);
  }
  if (STORE) {
    if (sizeof(TB) == 2) {
      *reinterpret_cast<short4*>(bp) = make_short4((short)i0, (short)i1, (short)i2, (short)i3);
    } else {
      *reinterpret_cast<int4*>(bp) = make_int4(i0, i1, i2, i3);
    }
  }
  return 4 + (i0 >> 31) + (i1 >> 31) + (i2 >> 31) + (i3 >> 31);   // sections are -1 or >= 0
}

__device__ __forceinline__ float4 ld_stream_f4(const float4* p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p));
  return v;
}

template <typename TB, bool STORE, int ROWS>
__device__ __forceinline__ void kmnc_strip_batch(const float4* __restrict__ src, int64_t d4, int64_t d,
                                                 const KmncLane& s0, const KmncLane& s1, const KmncLane& s2,
                                                 const KmncLane& s3, int k, const float* __restrict__ lo_g,
                                                 const float* __restrict__ jp_g, TB* __restrict__ dst,
                                                 int32_t* __restrict__ sc, unsigned live, bool leader) {
  float4 v[ROWS];
#pragma unroll
  for (int u = 0; u < ROWS; u++) v[u] = ld_stream_f4(src + u * d4);
#pragma unroll
  for (int u = 0; u < ROWS; u++) {
    int cnt = kmnc_strip_row<TB, STORE>(v[u], s0, s1, s2, s3, k, lo_g, jp_g, STORE ? dst + u * d : nullptr);
    cnt = __reduce_add_sync(live, cnt);
    red_add_s32_if(sc + u, cnt, leader);
  }
}

// grid = nstrips * lanes; block b: strip b % nstrips, samples [n * l / lanes, n * (l + 1) / lanes) with l = b / nstrips
template <typename TB, bool STORE>
__global__ void __launch_bounds__(256) kmnc_strip_kernel(const float* __restrict__ act, int64_t n, int64_t d,
                                                         const float* __restrict__ mins,
                                                         const float* __restrict__ jumps, int k,
                                                         TB* __restrict__ bucket, int32_t* __restrict__ score,
                                                         int nstrips, int lanes) {
  const int lane = threadIdx.x & 31;
  const int strip = blockIdx.x % nstrips;
  const int64_t l = blockIdx.x / nstrips;
  const int64_t d4 = d >> 2;
  const int64_t j = (int64_t)strip * 256 + threadIdx.x;   // float4 column
  const unsigned live = __ballot_sync(0xffffffffu, j < d4);   // lanes of this warp that own columns
  if (j >= d4) return;                                         // no block-wide barriers below
  const bool leader = lane == __ffs(live) - 1;
  const float* lo_g = mins + (j << 2);
  const float* jp_g = jumps + (j << 2);
  const float4 lo = __ldg(reinterpret_cast<const float4*>(lo_g));
  const float4 jp = __ldg(reinterpret_cast<const float4*>(jp_g));
  const KmncLane s0 = kmnc_lane(lo.x, jp.x, k), s1 = kmnc_lane(lo.y, jp.y, k);
  const KmncLane s2 = kmnc_lane(lo.z, jp.z, k), s3 = kmnc_lane(lo.w, jp.w, k);
  const int64_t row0 = n * l / lanes;
  const int64_t row1 = n * (l + 1) / lanes;
  const float4* src = reinterpret_cast<const float4*>(act) + row0 * d4 + j;
  TB* dst = STORE ? bucket + row0 * d + (j << 2) : nullptr;
  int32_t* sc = score + row0;
  int64_t r = row0;
  for (; r + kStripRows <= row1; r += kStripRows) {
    kmnc_strip_batch<TB, STORE, kStripRows>(src, d4, d, s0, s1, s2, s3, k, lo_g, jp_g, dst, sc, live, leader);
    src += kStripRows * d4;
    if (STORE) dst += kStripRows * d;
    sc += kStripRows;
  }
  if (r + 4 <= row1) {
    kmnc_strip_batch<TB, STORE, 4>(src, d4, d, s0, s1, s2, s3, k, lo_g, jp_g, dst, sc, live, leader);
    src += 4 * d4;
    if (STORE) dst += 4 * d;
    sc += 4;
    r += 4;
  }
  for (; r < row1; r++) {
    kmnc_strip_batch<TB, STORE, 1>(src, d4, d, s0, s1, s2, s3, k, lo_g, jp_g, dst, sc, live, leader);
    src += d4;
    if (STORE) dst += d;
    sc++;
  }
}

template <typename TA, typename TS>
static int launch_kmnc(const void* act, int64_t n, int64_t d, const void* mins, const void* jumps, int k,
                       void* bucket, int bucket_dtype, int32_t* score, cudaStream_t st) {
  const int grid = (int)std::min<int64_t>(n, (int64_t)sm_count() * 8);
  if (bucket == nullptr || bucket_dtype == TIP_I16) {
    kmnc_kernel<TA, TS, int16_t><<<grid, 256, 0, st>>>((const TA*)act, n, d, (const TS*)mins, (const TS*)jumps,
                                                       k, (int16_t*)bucket, score);
  } else {
    kmnc_kernel<TA, TS, int32_t><<<grid, 256, 0, st>>>((const TA*)act, n, d, (const TS*)mins, (const TS*)jumps,
                                                       k, (int32_t*)bucket, score);
  }
  TIP_LAUNCH_CHECK();
  return TIP_OK;
}

// =============================================================================================
// Operand packing for the tensor-core pass (layout documented in b200tip.h)
// =============================================================================================
template <typename T>
__global__ void __launch_bounds__(256) pair_prep_kernel(const T* __restrict__ src, int64_t rows, int d,
                                                        const float* __restrict__ center, int role,
                                                        int segments, float scale, float norm_coef,
                                                        __nv_bfloat16* __restrict__ dst, int64_t pitch,
                                                        float* __restrict__ sqnorm, float* __restrict__ rounderr,
                                                        uint32_t* __restrict__ row_min, int32_t* __restrict__ cand_cnt,
                                                        const int32_t* __restrict__ src_idx) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int d16 = (d + 15) & ~15;
  const T* x = src + (src_idx ? (int64_t)src_idx[row] : row) * (int64_t)d;
  __nv_bfloat16* out = dst + row * pitch;
  double acc = 0.0, err = 0.0;   // err: squared norm of what the bf16 operand drops (v - h, exact in fp32)
  for (int c = lane; c < d16; c += 32) {
    float v = 0.f;
    if (c < d) {
      const float ctr = center ? center[c] : 0.f;
      v = sizeof(T) == 8 ? (float)((double)x[c] - (double)ctr) : __fsub_rn((float)x[c], ctr);
    }
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    const float hf = __bfloat162float(h);
    if (segments == 1) {
      acc += (double)hf * (double)hf;
      const float res = __fsub_rn(v, hf);
      err += (double)res * (double)res;
      out[c] = role == TIP_ROLE_TRAIN ? __float2bfloat16_rn(scale * hf) : h;
    } else {
      const __nv_bfloat16 l = __float2bfloat16_rn(__fsub_rn(v, hf));
      const float res = __fsub_rn(__fsub_rn(v, hf), __bfloat162float(l));
      err += (double)res * (double)res;
      acc += (double)v * (double)v;
      if (role == TIP_ROLE_TRAIN) {
        const __nv_bfloat16 sh = __float2bfloat16_rn(scale * hf);
        out[c] = sh;
        out[d16 + c] = sh;
        out[2 * d16 + c] = __float2bfloat16_rn(scale * __bfloat162float(l));
      } else {
        out[c] = h;
        out[d16 + c] = l;
        out[2 * d16 + c] = h;
      }
    }
  }
  acc = warp_sum(acc);
  if (rounderr) err = warp_sum(err);
  const float nrm = (float)acc;
  const int tail = segments * d16;
  // tail block + zero padding up to the pitch
  for (int c = tail + lane; c < pitch; c += 32) {
    float v = 0.f;
    const int t = c - tail;
    if (t < 3) {
      if (role == TIP_ROLE_TRAIN) {
        const float cv = norm_coef * nrm;
        const float c0 = __bfloat162float(__float2bfloat16_rn(cv));
        const float c1 = __bfloat162float(__float2bfloat16_rn(cv - c0));
        const float c2 = __bfloat162float(__float2bfloat16_rn(cv - c0 - c1));
        v = t == 0 ? c0 : (t == 1 ? c1 : c2);
      } else {
        v = 1.f;
      }
    }
    out[c] = __float2bfloat16_rn(v);
  }
  if (lane == 0) {
    if (sqnorm) sqnorm[row] = nrm;
    if (rounderr) rounderr[row] = (float)sqrt(err) * 1.000001f;   // rounded up
    if (row_min) row_min[row] = 0x7f800000u;   // +inf: no distance seen yet (tip_nn_filter)
    if (cand_cnt) cand_cnt[row] = 0;
  }
}

// One-segment fp16 operand of the fast LSA pass: [ h(v) | tail ], h = round-to-nearest fp16 of v = fl32(x - center);
// tail(query) = [S, S, S, 0..], tail(train) = 3-way fp16 split of norm_coef*|v|^2 / S (S = norm_scale, a power of two
// that keeps the norm term inside fp16's range), so one K-loop accumulates norm_coef*|y|^2 + <h(x), h(y)> in fp32.
// sqnorm = exact |v|^2 (fp32).  flags[0] |= 1 when a value or the scaled norm term leaves fp16's finite range.
template <typename T>
__global__ void __launch_bounds__(256) pair_prep_f16_kernel(const T* __restrict__ src, int64_t rows, int d,
                                                            const float* __restrict__ center, int role, float norm_coef,
                                                            float norm_scale, __half* __restrict__ dst, int64_t pitch,
                                                            float* __restrict__ sqnorm, int32_t* __restrict__ flags) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int d16 = (d + 15) & ~15;
  const T* x = src + row * (int64_t)d;
  __half* out = dst + row * pitch;
  double acc = 0.0;
  bool bad = false;
  for (int c = lane; c < d16; c += 32) {
    float v = 0.f;
    if (c < d) {
      const float ctr = center ? center[c] : 0.f;
      v = sizeof(T) == 8 ? (float)((double)x[c] - (double)ctr) : __fsub_rn((float)x[c], ctr);
    }
    acc += (double)v * (double)v;
    bad |= !(fabsf(v) <= 65504.f);
    out[c] = __float2half_rn(v);
  }
  acc = warp_sum(acc);
  const float nrm = (float)acc;
  for (int c = d16 + lane; c < pitch; c += 32) {
    float v = 0.f;
    const int t = c - d16;
    if (t < 3) {
      if (role == TIP_ROLE_TRAIN) {
        const float cv = norm_coef * nrm / norm_scale;
        bad |= !(fabsf(cv) <= 65504.f);
        const float c0 = __half2float(__float2half_rn(cv));
        const float c1 = __half2float(__float2half_rn(cv - c0));
        const float c2 = __half2float(__float2half_rn(cv - c0 - c1));
        v = t == 0 ? c0 : (t == 1 ? c1 : c2);
      } else {
        v = norm_scale;
      }
    }
    out[c] = __float2half_rn(v);
  }
  if (__any_sync(0xffffffffu, bad) && lane == 0 && flags) atomicOr(flags, 1);
  if (lane == 0 && sqnorm) sqnorm[row] = nrm;
}

// =============================================================================================
// gather / whiten / combine
// =============================================================================================
__global__ void __launch_bounds__(256) gather_rows_kernel(const unsigned char* __restrict__ src,
                                                          int64_t row_bytes, const int32_t* __restrict__ pos,
                                                          int64_t m, unsigned char* __restrict__ dst) {
  if ((row_bytes & 15) == 0 && ((uintptr_t)src & 15) == 0 && ((uintptr_t)dst & 15) == 0) {
    // flat index space over 16-byte pieces: every thread busy whatever the row length
    const int64_t n16 = row_bytes >> 4;
    const int64_t total = m * n16;
    const uint4* s4 = reinterpret_cast<const uint4*>(src);
    uint4* o4 = reinterpret_cast<uint4*>(dst);
    for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < total; i += (int64_t)gridDim.x * 256) {
      const int64_t row = i / n16, col = i - row * n16;
      const int32_t p = pos[row];
      o4[i] = p < 0 ? make_uint4(0, 0, 0, 0) : s4[(int64_t)p * n16 + col];
    }
    return;
  }
  for (int64_t row = blockIdx.x; row < m; row += gridDim.x) {
    const int32_t p = pos[row];
    unsigned char* o = dst + row * row_bytes;
    {
      const unsigned char* s = src + (int64_t)(p < 0 ? 0 : p) * row_bytes;
      for (int64_t i = threadIdx.x; i < row_bytes; i += 256) o[i] = p < 0 ? 0 : s[i];
    }
  }
}

// out[m x dn] = (x[:, cols] - mu) . w   (fp32 FFMA; 128 x 64 tiles, 8 x 4 outputs per thread, K in steps of 32).
// The centring happens in double on the way into shared memory (one rounding to float, as a float64 host expression
// would give); a warp reads 32 consecutive K of one row per load (128 B), the inner loop is 3 x LDS.128 per 32 FFMA.
constexpr int kWhBM = 128, kWhBN = 64, kWhBK = 32;
template <typename T>
__global__ void __launch_bounds__(256) whiten_kernel(const T* __restrict__ x, int64_t m, int64_t d_in,
                                                     const int32_t* __restrict__ cols, int dn,
                                                     const double* __restrict__ mu, const float* __restrict__ w,
                                                     float* __restrict__ out) {
  __shared__ __align__(16) float As[kWhBK][kWhBM + 4];
  __shared__ __align__(16) float Bs[kWhBK][kWhBN + 4];
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;       // 16 column groups of 4, 16 row groups of 8
  const int64_t row0 = (int64_t)blockIdx.y * kWhBM;
  const int col0 = blockIdx.x * kWhBN;
  float acc[8][4] = {};
  for (int k0 = 0; k0 < dn; k0 += kWhBK) {
#pragma unroll 4
    for (int i = threadIdx.x; i < kWhBM * kWhBK; i += 256) {
      const int r = i >> 5, k = i & 31;
      float v = 0.f;
      if (row0 + r < m && k0 + k < dn) {
        const int src_col = cols ? cols[k0 + k] : (k0 + k);
        v = (float)((double)x[(row0 + r) * d_in + src_col] - mu[k0 + k]);
      }
      As[k][r] = v;
    }
#pragma unroll 4
    for (int i = threadIdx.x; i < kWhBK * kWhBN; i += 256) {
      const int k = i >> 6, c = i & 63;
      Bs[k][c] = (k0 + k < dn && col0 + c < dn) ? w[(int64_t)(k0 + k) * dn + col0 + c] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < kWhBK; k++) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[k][ty * 8]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[k][ty * 8 + 4]);
      const float4 b = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float bb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
      for (int i = 0; i < 8; i++)
#pragma unroll
        for (int j = 0; j < 4; j++) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 8; i++) {
    const int64_t r = row0 + ty * 8 + i;
    if (r >= m) continue;
    const int c = col0 + tx * 4;
    if (c + 3 < dn && (dn & 3) == 0) {
      *reinterpret_cast<float4*>(out + r * dn + c) = make_float4(acc[i][0], acc[i][1], acc[i][2], acc[i][3]);
    } else {
#pragma unroll
      for (int j = 0; j < 4; j++)
        if (c + j < dn) out[r * dn + c + j] = acc[i][j];
    }
  }
}

// merge of the per-slot (max, sum exp(. - max)) partials of every query: 32 queries x 8 slot groups per block
__global__ void __launch_bounds__(256) kde_combine_kernel(const float* __restrict__ pm, const float* __restrict__ ps,
                                                          int64_t m, int slots, float* __restrict__ om,
                                                          float* __restrict__ os) {
  __shared__ float s_mx[8][32];
  __shared__ float s_sum[8][32];
  const int lane = threadIdx.x & 31, g = threadIdx.x >> 5;
  const int64_t row = (int64_t)blockIdx.x * 32 + lane;
  float mx = -INFINITY, sum = 0.f;
  if (row < m) {
    for (int s = g; s < slots; s += 8) {               // online merge: one pass over this group's slots
      const float v = pm[(int64_t)s * m + row];
      if (v > -INFINITY) {
        const float p = ps[(int64_t)s * m + row];
        if (v > mx) { sum = sum * expf(mx - v) + p; mx = v; }   // mx = -inf: sum is 0, expf(-inf) = 0
        else sum += p * expf(v - mx);
      }
    }
  }
  s_mx[g][lane] = mx;
  s_sum[g][lane] = sum;
  __syncthreads();
  if (g == 0 && row < m) {
    float M = -INFINITY;
#pragma unroll
    for (int q = 0; q < 8; q++) M = fmaxf(M, s_mx[q][lane]);
    float S = 0.f;
    if (M > -INFINITY) {
#pragma unroll
      for (int q = 0; q < 8; q++)
        if (s_mx[q][lane] > -INFINITY) S += s_sum[q][lane] * expf(s_mx[q][lane] - M);
    }
    om[row] = M;
    os[row] = S;
  }
}

// out[row] = sum_k y[row, k]^2 accumulated in double (one warp per row): the squared Mahalanobis distance /
// the Gaussian quadratic form of a whitened row (MDSA, MLSA)
__global__ void __launch_bounds__(256) row_sqnorm_kernel(const float* __restrict__ y, int64_t m, int64_t d,
                                                         double* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= m) return;
  const float* r = y + row * d;
  double acc = 0.0;
  for (int64_t k = lane; k < d; k += 32) acc += (double)r[k] * (double)r[k];
  acc = warp_sum(acc);
  if (lane == 0) out[row] = acc;
}

}  // namespace tip

// =============================================================================================
// C ABI
// =============================================================================================
using namespace tip;

extern "C" int tip_version(void) { return TIP_VERSION; }
extern "C" const char* tip_last_error(void) { return g_err; }
extern "C" uint64_t tip_launch_count(void) { return g_launches.load(); }

extern "C" int tip_device_info(int* sms, int* major, int* minor) {
  int dev = 0;
  TIP_CHECK_CUDA(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  TIP_CHECK_CUDA(cudaGetDeviceProperties(&prop, dev));
  if (sms) *sms = prop.multiProcessorCount;
  if (major) *major = prop.major;
  if (minor) *minor = prop.minor;
  return TIP_OK;
}

extern "C" int tip_deepgini(const void* probs, int dtype, int64_t n, int64_t c, int32_t* pred, void* gini,
                            void* stream) {
  TIP_REQUIRE(probs && pred && gini, "null pointer");
  TIP_REQUIRE(n >= 0 && c >= 1 && c < (1 << 30), "shape");
  if (n == 0) return TIP_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == TIP_F32) return launch_gini<float>((const float*)probs, n, c, pred, (float*)gini, st);
  if (dtype == TIP_F64) return launch_gini<double>((const double*)probs, n, c, pred, (double*)gini, st);
  TIP_REQUIRE(false, "dtype must be TIP_F32 or TIP_F64");
}

extern "C" int tip_kmnc(const void* act, int act_dtype, int64_t n, int64_t d, const void* mins, const void* jumps,
                        int stat_dtype, int32_t sections, void* bucket, int bucket_dtype, int32_t* score,
                        void* stream) {
  TIP_REQUIRE(act && mins && jumps && score, "null pointer");
  TIP_REQUIRE(n >= 0 && d >= 1, "shape");
  TIP_REQUIRE(sections >= 1, "sections");
  TIP_REQUIRE(bucket == nullptr || bucket_dtype == TIP_I16 || bucket_dtype == TIP_I32, "bucket dtype");
  TIP_REQUIRE(!(bucket && bucket_dtype == TIP_I16) || sections <= 32767, "sections exceed int16 bucket ids");
  if (n == 0) return TIP_OK;
  cudaStream_t st = (cudaStream_t)stream;
  if (act_dtype == TIP_F32 && stat_dtype == TIP_F32) {
    const bool aligned = (d % 4 == 0) && (((uintptr_t)act | (uintptr_t)mins | (uintptr_t)jumps) & 15) == 0 &&
                         (bucket == nullptr || ((uintptr_t)bucket & 15) == 0);
    if (aligned) {
      TIP_CHECK_CUDA(cudaMemsetAsync(score, 0, (size_t)n * sizeof(int32_t), st));
      const int64_t nstrips = ((d >> 2) + 255) / 256;
      if (n >= 4 * kStripRows && nstrips <= 65535 && sections <= (1 << 22)) {
        // enough samples to amortise the per-block statistics load: column-strip kernel, one resident wave
        const bool i16 = bucket == nullptr || bucket_dtype == TIP_I16;
        const void* fn = bucket == nullptr ? (const void*)kmnc_strip_kernel<int16_t, false>
                         : i16             ? (const void*)kmnc_strip_kernel<int16_t, true>
                                           : (const void*)kmnc_strip_kernel<int32_t, true>;
        const int which = bucket == nullptr ? 0 : (i16 ? 1 : 2);
        static int per_sm_of[3] = {0, 0, 0};   // occupancy of each instance (same on every device of a box)
        if (per_sm_of[which] == 0) {
          int v = 0;
          TIP_CHECK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&v, fn, 256, 0));
          per_sm_of[which] = std::max(v, 1);
        }
        const int64_t resident = (int64_t)sm_count() * per_sm_of[which];
        const int64_t lanes = std::max<int64_t>(1, std::min<int64_t>(resident / nstrips, n / (2 * kStripRows)));
        const int ns = (int)nstrips, ln = (int)lanes;
        const float* a = (const float*)act;
        const float* lo = (const float*)mins;
        const float* jp = (const float*)jumps;
        void* args[] = {&a, &n, &d, &lo, &jp, &sections, &bucket, &score, (void*)&ns, (void*)&ln};
        TIP_CHECK_CUDA(cudaLaunchKernel(fn, dim3((unsigned)(nstrips * lanes)), dim3(256), args, 0, st));
        TIP_LAUNCH_CHECK();
        return TIP_OK;
      }
      const int64_t chunks = n * (((d >> 2) + 31) >> 5);
      const int grid = (int)std::min<int64_t>((chunks + 7) / 8, (int64_t)sm_count() * 8);
      if (bucket == nullptr || bucket_dtype == TIP_I16)
        kmnc_vec4_kernel<int16_t><<<grid, 256, 0, st>>>((const float*)act, n, d, (const float*)mins,
                                                        (const float*)jumps, sections, (int16_t*)bucket, score);
      else
        kmnc_vec4_kernel<int32_t><<<grid, 256, 0, st>>>((const float*)act, n, d, (const float*)mins,
                                                        (const float*)jumps, sections, (int32_t*)bucket, score);
      TIP_LAUNCH_CHECK();
      return TIP_OK;
    }
    return launch_kmnc<float, float>(act, n, d, mins, jumps, sections, bucket, bucket_dtype, score, st);
  }
  if (act_dtype == TIP_F32 && stat_dtype == TIP_F64)
    return launch_kmnc<float, double>(act, n, d, mins, jumps, sections, bucket, bucket_dtype, score, st);
  if (act_dtype == TIP_F64 && stat_dtype == TIP_F32)
    return launch_kmnc<double, float>(act, n, d, mins, jumps, sections, bucket, bucket_dtype, score, st);
  if (act_dtype == TIP_F64 && stat_dtype == TIP_F64)
    return launch_kmnc<double, double>(act, n, d, mins, jumps, sections, bucket, bucket_dtype, score, st);
  TIP_REQUIRE(false, "dtypes must be TIP_F32 / TIP_F64");
}

extern "C" int64_t tip_pair_pitch(int64_t d, int segments) {
  if (d < 1 || (segments != 1 && segments != 3)) return -1;
  const int64_t d16 = (d + 15) & ~(int64_t)15;
  return (segments * d16 + 16 + 63) & ~(int64_t)63;
}

static int pair_prep_impl(const void* src, int dtype, int64_t rows, int64_t d, const float* center, int role,
                          int segments, float scale, float norm_coef, void* dst, float* sqnorm, float* rounderr,
                          uint32_t* row_min, int32_t* cand_cnt, const int32_t* src_idx, void* stream) {
  TIP_REQUIRE(src && dst, "null pointer");
  TIP_REQUIRE(segments == 1 || segments == 3, "segments must be 1 or 3");
  TIP_REQUIRE(role == TIP_ROLE_QUERY || role == TIP_ROLE_TRAIN, "role");
  TIP_REQUIRE(d >= 1 && d <= (1 << 20), "d");
  TIP_REQUIRE(rows >= 0, "rows");
  if (rows == 0) return TIP_OK;
  const int64_t pitch = tip_pair_pitch(d, segments);
  const int64_t blocks = (rows + 7) / 8;
  TIP_REQUIRE(blocks < (1LL << 31), "too many rows");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == TIP_F32)
    pair_prep_kernel<float><<<(unsigned)blocks, 256, 0, st>>>((const float*)src, rows, (int)d, center, role, segments,
                                                             scale, norm_coef, (__nv_bfloat16*)dst, pitch, sqnorm,
                                                             rounderr, row_min, cand_cnt, src_idx);
  else if (dtype == TIP_F64)
    pair_prep_kernel<double><<<(unsigned)blocks, 256, 0, st>>>((const double*)src, rows, (int)d, center, role,
                                                              segments, scale, norm_coef, (__nv_bfloat16*)dst, pitch,
                                                              sqnorm, rounderr, row_min, cand_cnt, src_idx);
  else
    TIP_REQUIRE(false, "dtype must be TIP_F32 or TIP_F64");
  TIP_LAUNCH_CHECK();
  return TIP_OK;
}

extern "C" int tip_pair_prep(const void* src, int dtype, int64_t rows, int64_t d, const float* center, int role,
                             int segments, float scale, float norm_coef, void* dst, float* sqnorm, float* rounderr,
                             void* stream) {
  return pair_prep_impl(src, dtype, rows, d, center, role, segments, scale, norm_coef, dst, sqnorm, rounderr, nullptr,
                        nullptr, nullptr, stream);
}

extern "C" int tip_pair_prep_f16(const void* src, int dtype, int64_t rows, int64_t d, const float* center, int role,
                                 float norm_coef, float norm_scale, void* dst_f16, float* sqnorm, int32_t* flags,
                                 void* stream) {
  TIP_REQUIRE(src && dst_f16, "null pointer");
  TIP_REQUIRE(role == TIP_ROLE_QUERY || role == TIP_ROLE_TRAIN, "role");
  TIP_REQUIRE(d >= 1 && d <= (1 << 20) && rows >= 0, "shape");
  TIP_REQUIRE(norm_scale >= 1.f && norm_scale <= 32768.f, "norm_scale");
  if (rows == 0) return TIP_OK;
  const int64_t pitch = tip_pair_pitch(d, 1);
  const int64_t blocks = (rows + 7) / 8;
  TIP_REQUIRE(blocks < (1LL << 31), "too many rows");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == TIP_F32)
    pair_prep_f16_kernel<float><<<(unsigned)blocks, 256, 0, st>>>((const float*)src, rows, (int)d, center, role, norm_coef,
                                                                 norm_scale, (__half*)dst_f16, pitch, sqnorm, flags);
  else if (dtype == TIP_F64)
    pair_prep_f16_kernel<double><<<(unsigned)blocks, 256, 0, st>>>((const double*)src, rows, (int)d, center, role,
                                                                  norm_coef, norm_scale, (__half*)dst_f16, pitch, sqnorm,
                                                                  flags);
  else
    TIP_REQUIRE(false, "dtype must be TIP_F32 or TIP_F64");
  TIP_LAUNCH_CHECK();
  return TIP_OK;
}

extern "C" int tip_nn_query_prep(const void* q, int dtype, int64_t m, int64_t d, const float* center, void* q_pack,
                                 float* q_sqnorm, float* q_rounderr, uint32_t* row_min_bits, int32_t* cand_cnt,
                                 const int32_t* q_idx, void* stream) {
  TIP_REQUIRE(q_sqnorm && row_min_bits && cand_cnt, "null pointer");
  return pair_prep_impl(q, dtype, m, d, center, TIP_ROLE_QUERY, 1, 1.0f, 0.0f, q_pack, q_sqnorm, q_rounderr,
                        row_min_bits, cand_cnt, q_idx, stream);
}

template <typename T>
__global__ void __launch_bounds__(256) dsa_pack_out_kernel(const T* __restrict__ da, const T* __restrict__ db,
                                                           const int32_t* __restrict__ gid,
                                                           const int32_t* __restrict__ idx, int64_t m,
                                                           int64_t n_total, double* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x;
  if (i >= m) return;
  const int64_t j = idx ? idx[i] : i;
  if (j < 0 || j >= n_total) return;
  const T a = da[i], b = db[i];
  out[j] = (double)a;
  out[n_total + j] = (double)b;
  out[2 * n_total + j] = (double)gid[i];
  out[3 * n_total + j] = (double)Rn<T>::div(a, b);   // dist_a / dist_b in the input dtype (surprise.py:595), IEEE RN
}

extern "C" int tip_dsa_pack_out(const void* dist_a, const void* dist_b, int dtype, const int32_t* gid,
                                const int32_t* idx, int64_t m, int64_t n_total, double* out, void* stream) {
  TIP_REQUIRE(dist_a && dist_b && gid && out, "null pointer");
  TIP_REQUIRE(m >= 0 && n_total >= 0, "shape");
  if (m == 0) return TIP_OK;
  const unsigned blocks = (unsigned)((m + 255) / 256);
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == TIP_F32)
    dsa_pack_out_kernel<float><<<blocks, 256, 0, st>>>((const float*)dist_a, (const float*)dist_b, gid, idx, m, n_total, out);
  else if (dtype == TIP_F64)
    dsa_pack_out_kernel<double><<<blocks, 256, 0, st>>>((const double*)dist_a, (const double*)dist_b, gid, idx, m, n_total, out);
  else
    TIP_REQUIRE(false, "dtype must be TIP_F32 or TIP_F64");
  TIP_LAUNCH_CHECK();
  return TIP_OK;
}

extern "C" int tip_gather_rows(const void* src, int64_t row_bytes, const int32_t* pos, int64_t m, void* dst,
                               void* stream) {
  TIP_REQUIRE(src && pos && dst, "null pointer");
  TIP_REQUIRE(row_bytes > 0 && m >= 0, "shape");
  if (m == 0) return TIP_OK;
  const int64_t pieces = (row_bytes & 15) == 0 ? m * (row_bytes >> 4) : m * 256;
  const int grid = (int)std::max<int64_t>(1, std::min<int64_t>((pieces + 255) / 256, (int64_t)sm_count() * 16));
  gather_rows_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const unsigned char*)src, row_bytes, pos, m,
                                                            (unsigned char*)dst);
  TIP_LAUNCH_CHECK();
  return TIP_OK;
}

extern "C" int tip_whiten(const void* x, int dtype, int64_t m, int64_t d_in, const int32_t* cols, int64_t d_out,
                          const double* mu, const float* w, float* out, void* stream) {
  TIP_REQUIRE(x && mu && w && out, "null pointer");
  TIP_REQUIRE(m >= 0 && d_in >= 1 && d_out >= 1 && d_out <= 65535 * 64, "shape");
  TIP_REQUIRE(cols != nullptr || d_in >= d_out, "without a column list the input must be at least d_out wide");
  if (m == 0) return TIP_OK;
  dim3 grid((unsigned)((d_out + kWhBN - 1) / kWhBN), (unsigned)((m + kWhBM - 1) / kWhBM));
  TIP_REQUIRE((m + kWhBM - 1) / kWhBM <= 65535, "too many rows for one launch");
  cudaStream_t st = (cudaStream_t)stream;
  if (dtype == TIP_F32)
    whiten_kernel<float><<<grid, 256, 0, st>>>((const float*)x, m, d_in, cols, (int)d_out, mu, w, out);
  else if (dtype == TIP_F64)
    whiten_kernel<double><<<grid, 256, 0, st>>>((const double*)x, m, d_in, cols, (int)d_out, mu, w, out);
  else
    TIP_REQUIRE(false, "dtype must be TIP_F32 or TIP_F64");
  TIP_LAUNCH_CHECK();
  return TIP_OK;
}

extern "C" int tip_row_sqnorm(const float* y, int64_t m, int64_t d, double* out, void* stream) {
  TIP_REQUIRE(y && out, "null pointer");
  TIP_REQUIRE(m >= 0 && d >= 1, "shape");
  if (m == 0) return TIP_OK;
  row_sqnorm_kernel<<<(unsigned)((m + 7) / 8), 256, 0, (cudaStream_t)stream>>>(y, m, d, out);
  TIP_LAUNCH_CHECK();
  return TIP_OK;
}

extern "C" int tip_kde_combine(const float* pm, const float* ps, int64_t m, int32_t slots, float* om, float* os,
                               void* stream) {
  TIP_REQUIRE(pm && ps && om && os, "null pointer");
  TIP_REQUIRE(m >= 0 && slots >= 1, "shape");
  if (m == 0) return TIP_OK;
  kde_combine_kernel<<<(unsigned)((m + 31) / 32), 256, 0, (cudaStream_t)stream>>>(pm, ps, m, slots, om, os);
  TIP_LAUNCH_CHECK();
  return TIP_OK;
}
