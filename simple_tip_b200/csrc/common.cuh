// common.cuh — shared helpers for libb200tip.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/b200tip.h"

namespace tip {

// ---- error plumbing ---------------------------------------------------------------------
void set_error(const char* fmt, ...);
void count_launch(int n = 1);

#define TIP_CHECK_CUDA(expr)                                                              \
  do {                                                                                    \
    cudaError_t _e = (expr);                                                              \
    if (_e != cudaSuccess) {                                                              \
      tip::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return TIP_ERR_CUDA;                                                                \
    }                                                                                     \
  } while (0)

#define TIP_REQUIRE(cond, msg)                                                            \
  do {                                                                                    \
    if (!(cond)) {                                                                        \
      tip::set_error("%s:%d invalid argument: %s (%s)", __FILE__, __LINE__, msg, #cond);  \
      return TIP_ERR_INVALID;                                                             \
    }                                                                                     \
  } while (0)

#define TIP_LAUNCH_CHECK()                                                                \
  do {                                                                                    \
    tip::count_launch();                                                                  \
    TIP_CHECK_CUDA(cudaGetLastError());                                                   \
  } while (0)

int sm_count();

// ---- IEEE arithmetic without FMA contraction (NumPy never fuses) --------------------------
template <typename T> struct Rn;
template <> struct Rn<float> {
  static __device__ __forceinline__ float sub(float a, float b) { return __fsub_rn(a, b); }
  static __device__ __forceinline__ float add(float a, float b) { return __fadd_rn(a, b); }
  static __device__ __forceinline__ float mul(float a, float b) { return __fmul_rn(a, b); }
  static __device__ __forceinline__ float sqrt(float a) { return __fsqrt_rn(a); }
  static __device__ __forceinline__ float div(float a, float b) { return __fdiv_rn(a, b); }
  static __device__ __forceinline__ float inf() { return __int_as_float(0x7f800000); }
};
template <> struct Rn<double> {
  static __device__ __forceinline__ double sub(double a, double b) { return __dsub_rn(a, b); }
  static __device__ __forceinline__ double add(double a, double b) { return __dadd_rn(a, b); }
  static __device__ __forceinline__ double mul(double a, double b) { return __dmul_rn(a, b); }
  static __device__ __forceinline__ double sqrt(double a) { return __dsqrt_rn(a); }
  static __device__ __forceinline__ double div(double a, double b) { return __ddiv_rn(a, b); }
  static __device__ __forceinline__ double inf() { return __longlong_as_double(0x7ff0000000000000LL); }
};

// One leaf (n <= 128) of NumPy's pairwise summation applied to (x-y)^2 (or x^2 if y == nullptr):
// n < 8 sequential from 0; else eight stride-8 accumulators, tree-combined, tail sequential.
template <typename T>
__device__ __forceinline__ T np_leaf_sumsq(const T* __restrict__ x, const T* __restrict__ y, int n) {
  using R = Rn<T>;
  auto term = [&](int i) -> T {
    T d = y ? R::sub(x[i], y[i]) : x[i];
    return R::mul(d, d);
  };
  if (n < 8) {
    T res = (T)0;
    for (int i = 0; i < n; i++) res = R::add(res, term(i));
    return res;
  }
  T r0 = term(0), r1 = term(1), r2 = term(2), r3 = term(3);
  T r4 = term(4), r5 = term(5), r6 = term(6), r7 = term(7);
  int i = 8;
  const int lim = n - (n % 8);
  for (; i < lim; i += 8) {
    r0 = R::add(r0, term(i + 0));
    r1 = R::add(r1, term(i + 1));
    r2 = R::add(r2, term(i + 2));
    r3 = R::add(r3, term(i + 3));
    r4 = R::add(r4, term(i + 4));
    r5 = R::add(r5, term(i + 5));
    r6 = R::add(r6, term(i + 6));
    r7 = R::add(r7, term(i + 7));
  }
  T res = R::add(R::add(R::add(r0, r1), R::add(r2, r3)), R::add(R::add(r4, r5), R::add(r6, r7)));
  for (; i < n; i++) res = R::add(res, term(i));
  return res;
}

// Full NumPy pairwise sum of (x-y)^2 over n elements: blocks > 128 are split at
// n2 = n/2 - (n/2)%8 recursively; done here with an explicit stack (depth <= 32).
template <typename T>
__device__ T np_sumsq(const T* __restrict__ x, const T* __restrict__ y, int n) {
  if (n <= 128) return np_leaf_sumsq<T>(x, y, n);
  int off[32], len[32];
  unsigned char phase[32];
  T vals[32];
  int sp = 0, vp = 0;
  off[0] = 0; len[0] = n; phase[0] = 0; sp = 1;
  while (sp > 0) {
    const int top = sp - 1;
    const int o = off[top], l = len[top];
    if (l <= 128) {
      vals[vp++] = np_leaf_sumsq<T>(x + o, y ? y + o : nullptr, l);
      sp--;
    } else {
      int n2 = l / 2;
      n2 -= n2 % 8;
      if (phase[top] == 0) {
        phase[top] = 1;
        off[sp] = o; len[sp] = n2; phase[sp] = 0; sp++;
      } else if (phase[top] == 1) {
        phase[top] = 2;
        off[sp] = o + n2; len[sp] = l - n2; phase[sp] = 0; sp++;
      } else {
        const T r = vals[--vp];
        const T lft = vals[--vp];
        vals[vp++] = Rn<T>::add(lft, r);
        sp--;
      }
    }
  }
  return vals[0];
}

// ---- the same sums, computed cooperatively by a group of 8 consecutive lanes ----------------
// Lane `sub` (0..7) owns NumPy's stride-8 accumulator r[sub]; the tree
// ((r0+r1)+(r2+r3))+((r4+r5)+(r6+r7)) is three xor-shuffles (IEEE addition is commutative, so
// every lane of the group ends with the same bits).  gmask names the 8 lanes of the calling
// group, so the four groups of a warp may diverge (skip work independently).
template <typename T>
__device__ __forceinline__ T np_leaf_sumsq_g8(const T* __restrict__ x, const T* __restrict__ y, int n, int sub,
                                              unsigned gmask) {
  using R = Rn<T>;
  auto term = [&](int i) -> T {
    T d = y ? R::sub(x[i], y[i]) : x[i];
    return R::mul(d, d);
  };
  if (n < 8) {
    T res = (T)0;
    for (int i = 0; i < n; i++) res = R::add(res, term(i));
    return res;
  }
  // A leaf has at most 128 elements = 16 steps of the stride-8 accumulator this lane owns.  All
  // loads/squares are issued up front (one memory round trip), then added in NumPy's order: this
  // code sits at the end of a chain of dependent loads, latency is all that matters.
  const int lim = n - (n % 8);
  T t[16];
#pragma unroll
  for (int u = 0; u < 16; u++) {
    const int idx = 8 * u + sub;
    t[u] = idx < lim ? term(idx) : (T)0;
  }
  T tail[7];
#pragma unroll
  for (int u = 0; u < 7; u++) tail[u] = lim + u < n ? term(lim + u) : (T)0;
  T r = t[0];
#pragma unroll
  for (int u = 1; u < 16; u++)
    if (8 * u < lim) r = R::add(r, t[u]);          // uniform condition: lim is a multiple of 8
  r = R::add(r, __shfl_xor_sync(gmask, r, 1));
  r = R::add(r, __shfl_xor_sync(gmask, r, 2));
  r = R::add(r, __shfl_xor_sync(gmask, r, 4));
#pragma unroll
  for (int u = 0; u < 7; u++)
    if (lim + u < n) r = R::add(r, tail[u]);
  return r;
}

template <typename T>
__device__ T np_sumsq_g8(const T* __restrict__ x, const T* __restrict__ y, int n, int sub, unsigned gmask) {
  if (n <= 128) return np_leaf_sumsq_g8<T>(x, y, n, sub, gmask);
  int off[32], len[32];
  unsigned char phase[32];
  T vals[32];
  int sp = 1, vp = 0;
  off[0] = 0; len[0] = n; phase[0] = 0;
  while (sp > 0) {
    const int top = sp - 1;
    const int o = off[top], l = len[top];
    if (l <= 128) {
      vals[vp++] = np_leaf_sumsq_g8<T>(x + o, y ? y + o : nullptr, l, sub, gmask);
      sp--;
    } else {
      int n2 = l / 2;
      n2 -= n2 % 8;
      if (phase[top] == 0) { phase[top] = 1; off[sp] = o; len[sp] = n2; phase[sp] = 0; sp++; }
      else if (phase[top] == 1) { phase[top] = 2; off[sp] = o + n2; len[sp] = l - n2; phase[sp] = 0; sp++; }
      else { const T r = vals[--vp]; const T a = vals[--vp]; vals[vp++] = Rn<T>::add(a, r); sp--; }
    }
  }
  return vals[0];
}

// ---- the same pairwise sum driven by a precomputed leaf program (long traces) ------------------
// NumPy's recursion (blocks > 128 split at n/2 - (n/2)%8) visits its leaves left to right and combines
// the partial sums as a binary tree in post-order.  For a given trace width that schedule is fixed, so the
// host flattens it once into one word per leaf — offset/8 (20 bits) | len-1 (7 bits) | number of tree
// merges to perform after this leaf (5 bits) — and the device walks it with a value stack held in
// REGISTERS (static indexing: a push / merge shifts the whole stack) instead of the recursion's
// dynamically indexed arrays, which live in local memory (measured: the re-rank of 10 000 queries at
// D = 2048 took 0.85-1.0 ms with the generic routine).  The next leaf's operands are fetched while the
// current one is reduced.
constexpr int kSumStack = 24;

template <typename T>
struct LeafRegs {
  T t[16];
  T tail[7];
};

template <typename T>
__device__ __forceinline__ void leaf_load_g8(LeafRegs<T>& r, const T* __restrict__ x, const T* __restrict__ y, int n,
                                             int sub) {
  using R = Rn<T>;
  const int lim = n - (n % 8);
#pragma unroll
  for (int u = 0; u < 16; u++) {
    const int idx = 8 * u + sub;
    T d = (T)0;
    if (n >= 8 ? idx < lim : false) d = R::sub(x[idx], y[idx]);
    r.t[u] = R::mul(d, d);
  }
#pragma unroll
  for (int u = 0; u < 7; u++) {
    const int idx = (n >= 8 ? lim : 0) + u;
    T d = (T)0;
    if (idx < n) d = R::sub(x[idx], y[idx]);
    r.tail[u] = R::mul(d, d);
  }
}

template <typename T>
__device__ __forceinline__ T leaf_reduce_g8(const LeafRegs<T>& r, int n, unsigned gmask) {
  using R = Rn<T>;
  const int lim = n - (n % 8);
  T acc = (T)0;
  if (n >= 8) {
    acc = r.t[0];
#pragma unroll
    for (int u = 1; u < 16; u++)
      if (8 * u < lim) acc = R::add(acc, r.t[u]);          // uniform: lim is a multiple of 8
    acc = R::add(acc, __shfl_xor_sync(gmask, acc, 1));
    acc = R::add(acc, __shfl_xor_sync(gmask, acc, 2));
    acc = R::add(acc, __shfl_xor_sync(gmask, acc, 4));
  }
  // n < 8: sequential from 0 (the "tail" registers hold elements 0..n-1); else the tail after the tree
#pragma unroll
  for (int u = 0; u < 7; u++)
    if ((n >= 8 ? lim : 0) + u < n) acc = R::add(acc, r.tail[u]);
  return acc;
}

template <typename T>
__device__ __forceinline__ T np_sumsq_prog_g8(const T* __restrict__ x, const T* __restrict__ y,
                                              const uint32_t* __restrict__ prog, int n_leaves, int sub, unsigned gmask) {
  T st[kSumStack];
#pragma unroll
  for (int i = 0; i < kSumStack; i++) st[i] = (T)0;
  LeafRegs<T> cur, nxt;
  uint32_t w = prog[0];
  leaf_load_g8<T>(cur, x + (int64_t)(w & 0xFFFFFu) * 8, y + (int64_t)(w & 0xFFFFFu) * 8, (int)((w >> 20) & 127u) + 1, sub);
  for (int li = 0; li < n_leaves; li++) {
    const int len = (int)((w >> 20) & 127u) + 1;
    const int merges = (int)(w >> 27);
    uint32_t wn = 0;
    if (li + 1 < n_leaves) {
      wn = prog[li + 1];
      const int64_t off = (int64_t)(wn & 0xFFFFFu) * 8;
      leaf_load_g8<T>(nxt, x + off, y + off, (int)((wn >> 20) & 127u) + 1, sub);
    }
    const T v = leaf_reduce_g8<T>(cur, len, gmask);
#pragma unroll
    for (int i = kSumStack - 1; i > 0; i--) st[i] = st[i - 1];     // push
    st[0] = v;
    for (int m = 0; m < merges; m++) {                              // post-order merges: left + right
      st[0] = Rn<T>::add(st[1], st[0]);
#pragma unroll
      for (int i = 1; i < kSumStack - 1; i++) st[i] = st[i + 1];
    }
    cur = nxt;
    w = wn;
  }
  return st[0];
}

__device__ __forceinline__ float warp_min(float v) {
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
__device__ __forceinline__ int warp_sum(int v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Seed of a query's running minimum in tip_nn_filter's "approximate squared distance" space from an upper
// bound `ub` on the exact distance to SOME row of the range it is about to scan (DESIGN.md §4): that row's
// accumulator value s satisfies s <= (d + e)^2 + g with e the summed input-rounding norms and g the accumulation
// slack, so every threshold derived from the seed is at least as wide as the one the scan would reach on its
// own — the candidate set still contains NumPy's argmin, it just stops collecting far-away rows from tile one.
struct SeedParams {
  const float* ub;     // per train row (by position), +inf = no bound; nullptr = no seeding
  float t_rmax, t_err, gamma;
};

__device__ __forceinline__ uint32_t seed_row_min_bits(float ub, float nx, float q_err, const SeedParams& sp) {
  if (!(ub < __int_as_float(0x7f800000))) return 0x7f800000u;
  const float r = sqrtf(nx) + sp.t_rmax;
  const float e = (q_err + sp.t_err + 1.2e-7f * r) * 1.00001f;
  const float g = sp.gamma * r * r;
  const float d = ub * 1.000004f + e;
  const float s = (d * d + g) * 1.000002f;
  return s < __int_as_float(0x7f800000) ? __float_as_uint(s) : 0x7f800000u;
}

// One query row -> packed bf16 operand of tip_nn_filter (one segment) + reset filter state, by a full
// warp: the arithmetic of pair_prep_kernel (query role): centre in fp32, round to bf16, |h|^2 and
// the dropped part's norm accumulated in double.  src == nullptr packs a zero row.
template <typename T>
__device__ __forceinline__ void warp_pack_query(const T* __restrict__ src, int d, const float* __restrict__ center,
                                                __nv_bfloat16* __restrict__ out, int64_t pitch, float* sqnorm,
                                                float* rounderr, uint32_t* row_min, int32_t* cand_cnt, int lane,
                                                float seed_ub = 3.4e38f, const SeedParams* sp = nullptr) {
  const int d16 = (d + 15) & ~15;
  double acc = 0.0, err = 0.0;
  for (int c = lane; c < d16; c += 32) {
    float v = 0.f;
    if (c < d) {
      const T xv = src ? src[c] : (T)0;
      const float ctr = center ? center[c] : 0.f;
      v = sizeof(T) == 8 ? (float)((double)xv - (double)ctr) : __fsub_rn((float)xv, ctr);
    }
    const __nv_bfloat16 h = __float2bfloat16_rn(v);
    const float hf = __bfloat162float(h);
    const float res = __fsub_rn(v, hf);
    acc += (double)hf * (double)hf;
    err += (double)res * (double)res;
    out[c] = h;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    acc += __shfl_xor_sync(0xffffffffu, acc, o);
    err += __shfl_xor_sync(0xffffffffu, err, o);
  }
  for (int c = d16 + lane; c < pitch; c += 32) out[c] = __float2bfloat16_rn(c - d16 < 3 ? 1.f : 0.f);
  if (lane == 0) {
    const float nx = (float)acc;
    const float qe = (float)sqrt(err) * 1.000001f;
    *sqnorm = nx;
    if (rounderr) *rounderr = qe;
    // the seed needs the measured rounding norm; without it (a-priori window) no seeding
    *row_min = (sp && sp->ub && rounderr) ? seed_row_min_bits(seed_ub, nx, qe, *sp) : 0x7f800000u;
    *cand_cnt = 0;
  }
}

}  // namespace tip
