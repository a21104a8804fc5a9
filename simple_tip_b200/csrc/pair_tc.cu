// pair_tc.cu — the tensor-core pass over (query, train) activation-trace pairs (sm_100a).
//
// One persistent, warp-specialised kernel computes, for 128 query rows x 256 train rows at a
// time, the fp32 accumulator
//        acc[i][j] = norm_coef*|y_j|^2 + scale*<x_i, y_j>
// (both terms come out of the same tcgen05.mma K-loop: the packed operands carry a 16-wide tail
// block with a 3-way bf16 split of the norm on the train side and ones on the query side, see
// tip_pair_prep) and reduces it on the fly — no N_test x N_train intermediate ever leaves the SM:
//   MODE_NN   per-row running minimum + candidate emission (DSA, surprise.py:638-647)
//   MODE_LSE  per-row online log-sum-exp (LSA / Gaussian KDE, scipy 1.4.1 gaussian_kernel_estimate)
//   MODE_DUMP raw accumulator tile (bring-up / validation)
//
// Roles (320 threads): warp 0 = TMA producer (one lane), warp 1 = TMEM owner + MMA issuer (one
// lane), warps 2..9 = epilogue (TMEM lane quadrant = warp % 4, column half = (warp-2)/4; one
// query row x 128 columns per thread, TMEM loads software-pipelined against the reduction).
// Pipelines: 4-stage smem ring (full/empty mbarriers, TMA -> MMA) and a 2-deep TMEM accumulator
// ring (2 x 256 columns, MMA -> epilogue).
#include <cuda.h>
#include <cudaTypedefs.h>

#include <algorithm>
#include "common.cuh"

namespace tip {

constexpr int BM = 128;
constexpr int BN = 256;
constexpr int BK = 64;  // bf16 elements per smem row = one 128-byte swizzle atom
constexpr int kStages = 4;
constexpr int kABytes = BM * BK * 2;
constexpr int kBBytes = BN * BK * 2;
constexpr int kStageBytes = kABytes + kBBytes;
constexpr int kResAChunks = 5;               // resident-A variant (RESA): query tiles of up to 5 x 64 K elements
constexpr int kEpiThreads = 256;             // 8 epilogue warps
// epilogue warps of the streaming kernel in log-sum-exp mode (8 or 16, see pair_kernel).  16 was measured at C3 and
// changes nothing (0.338 ms either way): the K = 272 pass is bound by shared-memory bandwidth — both operands stream
// through shared memory for every tile (TMA writes 94 B/clk + MMA reads 96 B/clk against a 128 B/clk port = the
// measured 3400 cycles per 2176-cycle tile), not by the ex2 pipe's latency.
constexpr int kLseEpiWarps = 8;
constexpr int kCandSlots = 8;   // per-query staging slots for candidates (MODE_NN)
constexpr int kCandBytes = kCandSlots * 256 * 12;   // value, chunk start, 32-bit column mask
constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*align slack*/ + 256 /*barriers*/ + kCandBytes;
constexpr uint32_t kTmemCols = 512;

enum { MODE_NN = 0, MODE_LSE = 1, MODE_DUMP = 2 };

struct PairArgs {
  const tip_work_item* items;
  int n_items;
  // resident kernel: items [0, n_static) are scheduled statically (CTA b runs b, b + G, ...), items
  // [n_static, n_items) form a pool that CTAs drain through the atomic counter once they run dry
  int n_static;
  int* sched_counter;
  int k16;  // number of K=16 MMA steps per tile (packed width / 16)
  uint32_t idesc;   // streaming kernel: instruction descriptor (bf16 x bf16 or fp16 x fp16 operands); 0 = bf16 default
  int64_t m;
  // MODE_NN
  const int32_t* q_class;     // with class_off: per-query excluded train range (items flagged 1)
  const int32_t* class_off;
  const float* q_sqnorm;
  float rmax, eps2, gamma;  // error-window constants (DESIGN.md §4)
  const float* q_err;       // measured input-rounding norms |x~ - bf16(x~)| per query (or nullptr: a-priori bound)
  float t_err;              // max over the train rows of the same
  uint32_t* row_min_bits;
  int32_t* cand_idx;
  int32_t* cand_cnt;
  int cap;
  // MODE_LSE
  float* part_max;
  float* part_sum;
  // MODE_DUMP
  float* dump;
  // bring-up: per-tile clock64 stamps of block 0 (16 slots per tile), or nullptr
  long long* timeline;
  int timeline_tiles;
  // bring-up: per-CTA {globaltimer at start, at end, tiles, items} of the resident kernel, or nullptr
  long long* cta_clock;
};

// ---- PTX wrappers --------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded spin: a protocol bug must surface as a trapped kernel, never as a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if (++spins > 200000000u) __trap();
  }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_acc(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.eq.u32 p, 1, 1;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_first(uint32_t d_tmem, uint64_t adesc, uint64_t bdesc, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.eq.u32 p, 1, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(adesc), "l"(bdesc), "r"(idesc)
      : "memory");
}
// A operand from tensor memory (lane = row, one 32-bit column = two consecutive K elements): shared memory is then
// read for B only.  tcgen05.cp copies 128 rows x 256 bits (one K = 16 step of a K-major operand, described like an
// MMA operand) into 8 columns; cp and mma of one thread execute in issue order, so no barrier is needed between them.
__device__ __forceinline__ void tmem_cp_128x256b(uint32_t taddr, uint64_t sdesc) {
  asm volatile("tcgen05.cp.cta_group::1.128x256b [%0], %1;" ::"r"(taddr), "l"(sdesc) : "memory");
}
__device__ __forceinline__ void umma_bf16_ts_acc(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.eq.u32 p, 1, 1;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc)
      : "memory");
}
__device__ __forceinline__ void umma_bf16_ts_first(uint32_t d_tmem, uint32_t a_tmem, uint64_t bdesc, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.eq.u32 p, 1, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(bdesc), "r"(idesc)
      : "memory");
}
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, 128-byte-swizzled operand tile: rows of 128 B, 8-row groups 1024 B apart
// (cute::UMMA::SmemDescriptor: start>>4 | LBO=1<<16 | SBO=64<<32 | version=1<<46 | SWIZZLE_128B=2<<61).
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr) {
  return (uint64_t)((addr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}
// cute::UMMA::InstrDescriptor: D=f32 (1<<4), A=B=bf16 (1<<7, 1<<10), K-major both, N>>3 @17, M>>4 @24.
constexpr uint32_t kIdesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
// the same shape with fp16 operands (format code 0 for A and B): 11-bit significands, used by the one-segment
// LSA pass (tip_kde_lse_f16)
constexpr uint32_t kIdescF16 = (1u << 4) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);

// Acceptance threshold (accumulator space) for a query whose smallest approximate squared
// distance so far is s: every train row whose exact NumPy distance could still be the minimum
// has acc <= thr.  r = |x_b| + max|y_b|, e2 = 2*eps'*r, g = gamma*r^2 (DESIGN.md §4).
__device__ __forceinline__ float nn_threshold(float s, float nx, float e2, float g) {
  float root;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(root) : "f"(s + g));   // <= 2 ulp; covered by the slack below
  float r = root + e2;
  r *= 1.00004f;
  float thr = fmaf(r, r, g) - nx;
  return thr + fabsf(thr) * 1e-6f + 1e-30f;
}

struct EpiState {
  bool valid_row;
  int64_t row;
  int col1;
  int ex_lo, ex_hi;                    // train rows this query must ignore (its own class), or empty
  float nx, e2, g, best, thr, s_ref;   // MODE_NN
  int n_staged;
  float run_max, run_sum;              // MODE_LSE
};
struct EpiShared {
  float* cand_val;
  int* cand_col;
  uint32_t* cand_mask;
  int etid;
};

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

__device__ __forceinline__ uint32_t ld_volatile_u32(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.volatile.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// Reduce 32 accumulator columns [cbase, cbase+32) of one query row.
// (Keeping the rare paths out of line was tried and is far slower: taking the address of the
// register tile demotes it to local memory.  Code size is what matters here: the four unrolled
// chunk bodies of a tile have to stay inside the instruction cache.)
template <int MODE, bool EXCL, int SLOTS = kCandSlots, int STRIDE = kEpiThreads>
__device__ __forceinline__ void epi_chunk(const PairArgs& args, EpiState& st, const EpiShared& sh, uint32_t (&r)[32],
                                          int cbase, bool partial, bool dump_tile, int dump_row, int dump_col) {
  const float kInf = __int_as_float(0x7f800000);
  if (MODE == MODE_DUMP) {
    if (dump_tile) {
#pragma unroll
      for (int j = 0; j < 32; j++)
        if (dump_col + j < 256) args.dump[(int64_t)dump_row * 256 + dump_col + j] = __uint_as_float(r[j]);
    }
  } else if (MODE == MODE_NN) {
    if (partial || (EXCL && cbase < st.ex_hi && cbase + 32 > st.ex_lo)) {
      // rare: the chunk runs past the span, or overlaps the train rows this query must ignore
#pragma unroll
      for (int j = 0; j < 32; j++) {
        const int c = cbase + j;
        if (c >= st.col1 || (EXCL && c >= st.ex_lo && c < st.ex_hi)) r[j] = 0x7f800000u;
      }
    }
    float gmin[4];
#pragma unroll
    for (int gi = 0; gi < 4; gi++) {
      const float a0 = fminf(__uint_as_float(r[8 * gi + 0]), __uint_as_float(r[8 * gi + 1]));
      const float a1 = fminf(__uint_as_float(r[8 * gi + 2]), __uint_as_float(r[8 * gi + 3]));
      const float a2 = fminf(__uint_as_float(r[8 * gi + 4]), __uint_as_float(r[8 * gi + 5]));
      const float a3 = fminf(__uint_as_float(r[8 * gi + 6]), __uint_as_float(r[8 * gi + 7]));
      gmin[gi] = fminf(fminf(a0, a1), fminf(a2, a3));
    }
    const float mn = fminf(fminf(gmin[0], gmin[1]), fminf(gmin[2], gmin[3]));
    if (st.valid_row && mn <= st.thr && mn < kInf) {
      // event: this chunk holds a value inside the acceptance window of this query.  Kept short
      // and branch-light — with 32 independent queries per warp, events are frequent until the
      // running minima have warmed up.
      if (mn < st.best) {
        st.best = mn;
        st.s_ref = fminf(st.s_ref, fmaxf(st.best + st.nx, 0.f));
        st.thr = nn_threshold(st.s_ref, st.nx, st.e2, st.g);
      }
      // exact per-column mask of the chunk: the re-rank then touches only rows inside the window
      uint32_t mask = 0;
#pragma unroll
      for (int gi = 0; gi < 4; gi++) {
        if (gmin[gi] <= st.thr) {        // usually one group of 8 columns holds the value(s) inside the window
          uint32_t mg = 0;
#pragma unroll
          for (int j = 0; j < 8; j++) mg |= (__uint_as_float(r[8 * gi + j]) <= st.thr) ? (1u << j) : 0u;
          mask |= mg << (8 * gi);
        }
      }
      if (st.n_staged == SLOTS) {              // compact against the (tighter) current threshold
        int keep = 0;
        for (int k = 0; k < SLOTS; k++) {
          const float sv = sh.cand_val[k * STRIDE + sh.etid];
          if (sv <= st.thr) {
            sh.cand_val[keep * STRIDE + sh.etid] = sv;
            sh.cand_col[keep * STRIDE + sh.etid] = sh.cand_col[k * STRIDE + sh.etid];
            sh.cand_mask[keep * STRIDE + sh.etid] = sh.cand_mask[k * STRIDE + sh.etid];
            keep++;
          }
        }
        st.n_staged = keep;
      }
      if (st.n_staged < SLOTS) {
        sh.cand_val[st.n_staged * STRIDE + sh.etid] = mn;
        sh.cand_col[st.n_staged * STRIDE + sh.etid] = cbase;
        sh.cand_mask[st.n_staged * STRIDE + sh.etid] = mask;
        st.n_staged++;
      } else {                                 // staging full of live chunks: emit directly
        const int pos = atomicAdd(args.cand_cnt + st.row, 1);
        if (pos < args.cap) {
          args.cand_idx[(st.row * args.cap + pos) * 2] = cbase;
          args.cand_idx[(st.row * args.cap + pos) * 2 + 1] = (int)mask;
        }
      }
    }
  } else {  // MODE_LSE
    constexpr float kL2e = 1.4426950408889634f;
    float mx = -kInf;
    if (partial) {
#pragma unroll
      for (int j = 0; j < 32; j++) {
        const float v = (cbase + j < st.col1) ? __uint_as_float(r[j]) : -kInf;
        r[j] = __float_as_uint(v);
        mx = fmaxf(mx, v);
      }
    } else {
#pragma unroll
      for (int j = 0; j < 32; j += 2) mx = fmaxf(mx, fmaxf(__uint_as_float(r[j]), __uint_as_float(r[j + 1])));
    }
    if (mx > st.run_max) {
      st.run_sum *= fast_exp2((st.run_max - mx) * kL2e);  // run_max = -inf -> factor 0
      st.run_max = mx;
    }
    if (st.run_max > -kInf) {
      const float off = -st.run_max * kL2e;
      float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
      for (int j = 0; j < 32; j += 4) {
        s0 += fast_exp2(fmaf(__uint_as_float(r[j + 0]), kL2e, off));
        s1 += fast_exp2(fmaf(__uint_as_float(r[j + 1]), kL2e, off));
        s2 += fast_exp2(fmaf(__uint_as_float(r[j + 2]), kL2e, off));
        s3 += fast_exp2(fmaf(__uint_as_float(r[j + 3]), kL2e, off));
      }
      st.run_sum += (s0 + s1) + (s2 + s3);
    }
  }
}

template <int MODE, bool EXCL, int EW = 8, bool RESA = false>
__global__ void __launch_bounds__(64 + 32 * EW, 1)
pair_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const PairArgs args) {
  // EW epilogue warps: 8 = one query row x 128 columns per thread, 16 = one row x 64 columns (kLseEpiWarps)
  constexpr int PARTS = EW / 4;          // column parts of a tile, one per group of four epilogue warps
  constexpr int CPT = BN / PARTS;        // columns per thread and tile
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw);
  // RESA (short K, tip_kde_lse*): the query tile's K chunks stay RESIDENT in shared memory for the whole work item
  // (kResAChunks x 16 KB at `base`, loaded once per item) and the ring carries train chunks only (kStages x 32 KB
  // behind it) — re-streaming A for every train tile cost a third of the TMA write traffic of a bandwidth-bound pass.
  const uint32_t b_ring = base + (RESA ? kResAChunks * kABytes : 0);
  const uint32_t bar0 = RESA ? b_ring + kStages * kBBytes : base + kStages * kStageBytes;
  auto full_bar = [&](int s) { return bar0 + 8u * s; };
  auto empty_bar = [&](int s) { return bar0 + 8u * (kStages + s); };
  auto tfull_bar = [&](int a) { return bar0 + 8u * (2 * kStages + a); };
  auto tempty_bar = [&](int a) { return bar0 + 8u * (2 * kStages + 2 + a); };
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + (bar0 - base) + 8 * (2 * kStages + 4));
  const uint32_t a_full = bar0 + 8u * (2 * kStages + 6), a_empty = bar0 + 8u * (2 * kStages + 7);   // RESA

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA);
    tma_prefetch_desc(&tmB);
    for (int s = 0; s < kStages; s++) { mbar_init(full_bar(s), 1); mbar_init(empty_bar(s), 1); }
    for (int a = 0; a < 2; a++) { mbar_init(tfull_bar(a), 1); mbar_init(tempty_bar(a), EW); }
    if (RESA) { mbar_init(a_full, 1); mbar_init(a_empty, 1); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)),
                 "r"(kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const int k16 = args.k16;
  const int nchunks = (k16 + 3) >> 2;

  if (warp == 0) {
    // ================= TMA producer =================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      uint32_t a_phase = 0;
      for (int w = blockIdx.x; w < args.n_items; w += gridDim.x) {
        const tip_work_item it = args.items[w];
        const int ntiles = (it.col1 - it.col0 + BN - 1) / BN;
        if (RESA && ntiles > 0) {
          mbar_wait(a_empty, a_phase ^ 1u);      // the previous item's MMAs have retired (first item: passes at once)
          mbar_expect_tx(a_full, (uint32_t)nchunks * kABytes);
          for (int c = 0; c < nchunks; c++) tma_load_2d(base + (uint32_t)c * kABytes, &tmA, a_full, c * BK, it.q_row0);
          a_phase ^= 1u;
        }
        for (int t = 0; t < ntiles; t++) {
          for (int c = 0; c < nchunks; c++) {
            mbar_wait(empty_bar(stage), phase ^ 1u);
            if (RESA) {
              mbar_expect_tx(full_bar(stage), kBBytes);
              tma_load_2d(b_ring + (uint32_t)stage * kBBytes, &tmB, full_bar(stage), c * BK, it.col0 + t * BN);
            } else {
              mbar_expect_tx(full_bar(stage), kStageBytes);
              const uint32_t a_dst = base + stage * kStageBytes;
              tma_load_2d(a_dst, &tmA, full_bar(stage), c * BK, it.q_row0);
              tma_load_2d(a_dst + kABytes, &tmB, full_bar(stage), c * BK, it.col0 + t * BN);
            }
            if (++stage == kStages) { stage = 0; phase ^= 1u; }
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ================= MMA issuer =================
    // Whole warp runs the loop (uniform control flow -> descriptors live in uniform registers),
    // one elected lane issues; full chunks are four straight-line MMAs.
    const bool leader = elect_one();
    const uint32_t idesc = args.idesc ? args.idesc : kIdesc;
    int stage = 0, acc = 0;
    uint32_t phase = 0, acc_phase = 0, a_phase = 0;
    for (int w = blockIdx.x; w < args.n_items; w += gridDim.x) {
      const tip_work_item it = args.items[w];
      const int ntiles = (it.col1 - it.col0 + BN - 1) / BN;
      if (RESA && ntiles > 0) {
        mbar_wait(a_full, a_phase);
        a_phase ^= 1u;
        tc_fence_after();
      }
      for (int t = 0; t < ntiles; t++) {
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u);
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)acc * BN;
        for (int c = 0; c < nchunks; c++) {
          mbar_wait(full_bar(stage), phase);
          tc_fence_after();
          const uint32_t a_addr = base + stage * kStageBytes;
          const uint64_t adesc = smem_desc(RESA ? base + (uint32_t)c * kABytes : a_addr);
          const uint64_t bdesc = smem_desc(RESA ? b_ring + (uint32_t)stage * kBBytes : a_addr + kABytes);
          const int nm = min(4, k16 - 4 * c);
          if (leader) {
            // +32 bytes (one K=16 slice) inside the 128-byte swizzle row = +2 in the >>4 field
            if (c == 0) umma_bf16_first(d_tmem, adesc, bdesc, idesc);
            else umma_bf16_acc(d_tmem, adesc, bdesc, idesc);
            if (nm == 4) {
              umma_bf16_acc(d_tmem, adesc + 2u, bdesc + 2u, idesc);
              umma_bf16_acc(d_tmem, adesc + 4u, bdesc + 4u, idesc);
              umma_bf16_acc(d_tmem, adesc + 6u, bdesc + 6u, idesc);
            } else {
              for (int k = 1; k < nm; k++) umma_bf16_acc(d_tmem, adesc + 2u * k, bdesc + 2u * k, idesc);
            }
            umma_commit(empty_bar(stage));
            if (c == nchunks - 1) umma_commit(tfull_bar(acc));
          }
          __syncwarp();
          if (++stage == kStages) { stage = 0; phase ^= 1u; }
        }
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1u;
      }
      if (RESA && ntiles > 0) {
        if (leader) umma_commit(a_empty);      // the resident query tile is free once this item's MMAs have retired
        __syncwarp();
      }
    }
  } else {
    // ================= epilogue =================
    // EW warps: TMEM lane quadrant = warp % 4 (hardware rule), column part = (warp - 2) / 4.
    // One thread = one query row x one CPT-column part of every tile; the parts of a row
    // never talk to each other except through row_min_bits (like CTAs on different spans do).
    const int quad = warp & 3;
    const int half = (warp - 2) >> 2;    // column part index, 0 .. PARTS-1
    const int row_local = quad * 32 + lane;
    const uint32_t lane_addr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(half * CPT);
    const int etid = threadIdx.x - 64;   // index among the epilogue threads
    EpiShared sh;
    sh.cand_val = reinterpret_cast<float*>(smem + kStages * kStageBytes + 256);
    sh.cand_col = reinterpret_cast<int*>(sh.cand_val + kCandSlots * kEpiThreads);
    sh.cand_mask = reinterpret_cast<uint32_t*>(sh.cand_col + kCandSlots * kEpiThreads);
    sh.etid = etid;
    int acc = 0;
    uint32_t acc_phase = 0;
    const float kInf = __int_as_float(0x7f800000);
    for (int w = blockIdx.x; w < args.n_items; w += gridDim.x) {
      const tip_work_item it = args.items[w];
      const int ntiles = (it.col1 - it.col0 + BN - 1) / BN;
      EpiState st;
      st.valid_row = row_local < it.q_rows;
      st.row = (int64_t)it.q_row0 + row_local;
      st.nx = 0.f; st.e2 = 0.f; st.g = 0.f; st.best = kInf; st.thr = kInf; st.s_ref = kInf; st.n_staged = 0;
      st.run_max = -kInf; st.run_sum = 0.f;
      st.col1 = it.col1;
      st.ex_lo = 0; st.ex_hi = 0;
      if (MODE == MODE_NN && st.valid_row) {
        if (EXCL && (it.reserved & 1) && args.q_class) {
          const int cls = args.q_class[st.row];
          st.ex_lo = args.class_off[cls];
          st.ex_hi = args.class_off[cls + 1];
        }
        st.nx = args.q_sqnorm[st.row];
        const float r = sqrtf(st.nx) + args.rmax;
        st.e2 = args.q_err ? 2.f * (args.q_err[st.row] + args.t_err + 1.2e-7f * r) * 1.00001f : args.eps2 * r;
        st.g = args.gamma * r * r;
        st.s_ref = __uint_as_float(ld_volatile_u32(args.row_min_bits + st.row));
        st.thr = nn_threshold(st.s_ref, st.nx, st.e2, st.g);
      }

      for (int t = 0; t < ntiles; t++) {
        mbar_wait(tfull_bar(acc), acc_phase);
        tc_fence_after();
        const int col_base = it.col0 + t * BN + half * CPT;
        const bool partial = col_base + CPT > it.col1;
        uint32_t seen_bits = 0x7f800000u;
        if (MODE == MODE_NN && st.valid_row) seen_bits = ld_volatile_u32(args.row_min_bits + st.row);
        const uint32_t taddr = lane_addr + (uint32_t)(acc * BN);
        // software pipeline over the 4 x 32 columns of this half: the TMEM load of chunk q+1 is in
        // flight while chunk q is reduced
        uint32_t ra[32], rb[32];
        tmem_ld32(taddr, ra);
#pragma unroll 1
        for (int h = 0; h < CPT / 64; h++) {   // rolled on purpose: the epilogue has to stay inside the I-cache
          tmem_wait_ld();
          tmem_ld32(taddr + 64 * h + 32, rb);
          epi_chunk<MODE, EXCL>(args, st, sh, ra, col_base + 64 * h, partial, w == 0 && t == 0, row_local,
                          half * CPT + 64 * h);
          tmem_wait_ld();
          if (h + 1 < CPT / 64) {
            tmem_ld32(taddr + 64 * (h + 1), ra);
          } else {
            // accumulator drained into registers: hand the TMEM stage back to the MMA warp early
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(tempty_bar(acc));
          }
          epi_chunk<MODE, EXCL>(args, st, sh, rb, col_base + 64 * h + 32, partial, w == 0 && t == 0, row_local,
                          half * CPT + 64 * h + 32);
        }

        if (MODE == MODE_NN && st.valid_row) {
          // share the running minimum across everybody scanning other columns for the same query
          const float mine = fmaxf(st.best + st.nx, 0.f);
          const float seen = __uint_as_float(seen_bits);
          if (mine < seen) atomicMin(args.row_min_bits + st.row, __float_as_uint(mine));
          if (seen < st.s_ref) {
            st.s_ref = seen;
            st.thr = nn_threshold(st.s_ref, st.nx, st.e2, st.g);
          }
        }
        acc ^= 1;
        if (acc == 0) acc_phase ^= 1u;
      }

      if (MODE == MODE_NN) {
        if (st.valid_row) {
          // other CTAs / halves have been scanning other columns of this query meanwhile: only
          // flush the groups that survive the best bound known by now
          const float seen = __uint_as_float(ld_volatile_u32(args.row_min_bits + st.row));
          if (seen < st.s_ref) {
            st.s_ref = seen;
            st.thr = nn_threshold(st.s_ref, st.nx, st.e2, st.g);
          }
          for (int k = 0; k < st.n_staged; k++) {
            if (sh.cand_val[k * kEpiThreads + etid] <= st.thr) {
              const int pos = atomicAdd(args.cand_cnt + st.row, 1);
              if (pos < args.cap) {
                args.cand_idx[(st.row * args.cap + pos) * 2] = sh.cand_col[k * kEpiThreads + etid];
                args.cand_idx[(st.row * args.cap + pos) * 2 + 1] = (int)sh.cand_mask[k * kEpiThreads + etid];
              }
            }
          }
        }
      } else if (MODE == MODE_LSE) {
        if (st.valid_row) {
          args.part_max[(int64_t)(it.slot * PARTS + half) * args.m + st.row] = st.run_max;
          args.part_sum[(int64_t)(it.slot * PARTS + half) * args.m + st.row] = st.run_sum;
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

// =============================================================================================
// Resident-query variant for short traces (packed width <= 9 K-steps, e.g. D = 128):
// 256 query rows stay in shared memory for a whole work item and 192-row train tiles are
// streamed (2-stage ring), so the L2 -> SM traffic per 256 x 192 output tile is the train tile
// alone (55.3 KB at D = 128).  The packed row is consumed as full 64-element chunks (128-byte
// swizzle) plus 16-element panels (32-byte swizzle) so no padding is fetched.
// MMA shape M128 x N192 x K16: per instruction the tensor pipe reads 4 KB of A and 6 KB of B from
// shared memory for 96 cycles of work (107 B/clk, under the 128 B/clk shared-memory bandwidth that
// the earlier M128 x N128 version sat on), and the single issuing thread (~45 cycles per
// instruction) needs a third fewer instructions per flop.
// TMEM: query half h accumulates in columns [256 h, 256 h + 192); the halves ping-pong — while the
// tensor pipe fills half h of tile t, the epilogue warps of half 1-h drain their accumulator.
// Epilogue: 16 warps = 4 lane quadrants x 2 query halves x 2 column halves; one query row x 96
// columns per thread (3 chunks of 32, TMEM loads double-buffered).  (N = 256 with 8 epilogue warps
// was measured epilogue-bound: a lone warp per scheduler cannot hide the tcgen05.ld latency.)
// =============================================================================================
constexpr int RS_BM = 256;
constexpr int RS_BN = 192;
constexpr int kRsMaxK16 = 9;
constexpr int kRsEpiThreads = 512;            // 16 epilogue warps
constexpr int kRsThreads = 64 + kRsEpiThreads + 32;   // TMA warp, MMA warp (query half 0), 16 epilogue warps, MMA warp (half 1)
constexpr int kRsMmaWarp1 = 2 + kRsEpiThreads / 32;     // the second issuing warp sits behind the epilogue warps
constexpr int kRsStages = 2;
// MMA shape M128 x N96 x K16: every (query half, column half) QUARTER of the tile is its own accumulator with its own
// full / empty barriers, so a quarter is handed back to the tensor pipe as soon as ITS four epilogue warps have
// drained it (accumulator round trip 432 + ~830 cycles of latency against a 1728-cycle tile, instead of 864 + ~830
// with halves — the round trip, not the pipe, was the tile period).
constexpr int RS_QN = RS_BN / 2;
constexpr uint32_t kIdescRs = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(RS_QN >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);

struct RsGeom {
  int nfull, rem;
  uint32_t a_bytes, b_bytes;
};

__host__ __device__ constexpr RsGeom rs_geom(int k16) {
  return RsGeom{k16 / 4, k16 % 4, (uint32_t)((k16 / 4) * RS_BM * 128 + (k16 % 4) * RS_BM * 32),
                (uint32_t)((k16 / 4) * RS_BN * 128 + (k16 % 4) * RS_BN * 32)};
}
constexpr int kRsBarBytes = 256;
// second buffer for the K tail of the query tile (the tail is read from shared memory for the whole item, so the next
// query tile's tail needs its own place when the tile is prefetched early; the full chunks live in tensor memory)
__host__ __device__ constexpr int rs_tail_bytes(int k16) { return (k16 % 4) * RS_BM * 32; }
constexpr int kSmemMax = 232448;   // 227 KB per CTA on sm_100
// candidate staging slots per query that still fit next to the operand buffers (3 at K16 = 9)
__host__ __device__ constexpr int rs_slots(int k16) {
  const int left = kSmemMax - 1024 - kRsBarBytes - (int)(rs_geom(k16).a_bytes + kRsStages * rs_geom(k16).b_bytes) - rs_tail_bytes(k16);
  const int s = left / (kRsEpiThreads * 12);
  return s > kCandSlots ? kCandSlots : s;
}
__host__ __device__ constexpr int rs_smem_bytes(int k16) {
  return (int)(rs_geom(k16).a_bytes + kRsStages * rs_geom(k16).b_bytes) + rs_tail_bytes(k16) + 1024 + kRsBarBytes +
         rs_slots(k16) * kRsEpiThreads * 12;
}
static_assert(rs_slots(kRsMaxK16) >= 2 && rs_smem_bytes(kRsMaxK16) <= kSmemMax, "resident kernel does not fit");

__device__ __forceinline__ uint64_t smem_desc_sw32(uint32_t addr) {
  // K-major, 32-byte swizzle: rows of 32 B, 8-row groups 256 B apart
  return (uint64_t)((addr & 0x3FFFFu) >> 4) | (1ull << 16) | (16ull << 32) | (1ull << 46) | (6ull << 61);
}

template <int MODE, int K16, bool EXCL>
__global__ void __launch_bounds__(kRsThreads, 1)
pair_rs_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmAt,
               const __grid_constant__ CUtensorMap tmB, const __grid_constant__ CUtensorMap tmBt, const PairArgs args) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  const uint32_t base = (raw + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (base - raw);
  constexpr int NFULL = K16 / 4, REM = K16 % 4;
  constexpr RsGeom geo = rs_geom(K16);
  constexpr int SLOTS = rs_slots(K16);
  int tl_tile = 0;
#define TL(slot)                                                                              \
  do {                                                                                        \
    if (args.timeline && blockIdx.x == 0 && tl_tile < args.timeline_tiles)                    \
      args.timeline[(int64_t)tl_tile * 16 + (slot)] = clock64();                              \
  } while (0)
  const uint32_t a_base = base;
  const uint32_t a_rem = a_base + (uint32_t)NFULL * RS_BM * 128;
  const uint32_t b_base = a_base + geo.a_bytes;
  const uint32_t a_rem2 = b_base + (uint32_t)kRsStages * geo.b_bytes;     // see rs_tail_bytes
  constexpr uint32_t tiles_bytes = geo.a_bytes + (uint32_t)kRsStages * geo.b_bytes + (uint32_t)rs_tail_bytes(K16);
  // A from tensor memory: the query tile's full 64-element K chunks are copied into the free TMEM columns [192, 256)
  // of each accumulator half once per query tile and the MMAs read A from there (the K tail stays in shared memory;
  // measured at C2: 0.186 -> 0.183 ms per step).  With no full chunk (d < 64) A is read from shared memory.
  constexpr bool ta = NFULL > 0;
  const uint32_t bar0 = base + tiles_bytes;
  // barriers: 0 a_full, 1 a_empty, 2..3 b_full, 4..5 b_empty, 20..23 tfull[quarter], 24..27 tempty[quarter],
  // 10..11 sched_full[slot], 12..13 sched_empty[slot]; then the TMEM base and the 2-slot item ring
  auto bar = [&](int i) { return bar0 + 8u * i; };
  volatile uint32_t* tmem_slot = reinterpret_cast<volatile uint32_t*>(smem + tiles_bytes + 8 * 16);
  volatile int* sched_ring = reinterpret_cast<volatile int*>(smem + tiles_bytes + 8 * 17);
  // Item hand-out: the TMA thread decides which item comes next (static stride first, then the
  // shared pool) and publishes its index; the MMA warp and the 16 epilogue warps consume it.
  auto next_item = [&](int k) -> int {     // consumers: k-th item of this CTA, or -1
    const int slot = k & 1;
    mbar_wait(bar(10 + slot), (uint32_t)(k >> 1) & 1u);
    const int idx = sched_ring[slot];
    __syncwarp();
    if ((threadIdx.x & 31) == 0) mbar_arrive(bar(12 + slot));
    return idx;
  };
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  long long t_entry = 0;
  if (args.cta_clock && threadIdx.x == 0) asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t_entry));

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmA); tma_prefetch_desc(&tmAt); tma_prefetch_desc(&tmB); tma_prefetch_desc(&tmBt);
    mbar_init(bar(0), 1); mbar_init(bar(1), 2);            // a_empty, b_empty: one commit per issuing warp
    for (int s = 0; s < kRsStages; s++) { mbar_init(bar(2 + s), 1); mbar_init(bar(4 + s), 2); }
    for (int q = 0; q < 4; q++) { mbar_init(bar(20 + q), 1); mbar_init(bar(24 + q), kRsEpiThreads / 128); }   // tfull / tempty
    for (int s = 0; s < 2; s++) { mbar_init(bar(10 + s), 1); mbar_init(bar(12 + s), 2 + kRsEpiThreads / 32); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32((const void*)tmem_slot)),
                 "r"(kTmemCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  auto global_ns = [] { long long t; asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t)); return t; };
  if (args.cta_clock && threadIdx.x == 0) {
    args.cta_clock[blockIdx.x * 4] = global_ns();
    args.cta_clock[1024 + blockIdx.x] = t_entry;      // kernel entry, before barrier init / TMEM allocation
  }

  if (warp == 0) {
    // ================= TMA producer =================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0, a_phase = 0;
      long long n_tiles_done = 0, n_items_done = 0;
      int w_static = blockIdx.x;
      int prev_q0 = -1, prev_qn = -1;   // query tile currently resident (consecutive items may share it)
      int a_loads = 0;                  // query tiles loaded so far (parity selects the tail buffer)
      for (int k = 0;; k++) {
        int w;
        if (w_static < args.n_static) { w = w_static; w_static += gridDim.x; }
        else if (args.sched_counter) {
          w = args.n_static + atomicAdd(args.sched_counter, 1);
          if (w >= args.n_items) w = -1;
        } else w = -1;
        const int slot = k & 1;
        mbar_wait(bar(12 + slot), ((uint32_t)(k >> 1) & 1u) ^ 1u);
        sched_ring[slot] = w;
        mbar_arrive(bar(10 + slot));
        if (w < 0) break;
        const tip_work_item it = args.items[w];
        const int ntiles = (it.col1 - it.col0 + RS_BN - 1) / RS_BN;
        if (ntiles <= 0) continue;   // padding entry of a balanced work list
        n_tiles_done += ntiles; n_items_done++;
        const bool new_a = it.q_row0 != prev_q0 || it.q_rows != prev_qn;
        prev_q0 = it.q_row0; prev_qn = it.q_rows;
        // the first train tile of the new item is prefetched while the previous item still owns
        // the query buffer; the queries follow as soon as the MMA warp releases it
        const int a_at = min(kRsStages - 1, ntiles);
        for (int t = 0; t <= ntiles; t++) {
          if (t == a_at && new_a) {
            mbar_wait(bar(1), a_phase ^ 1u);
            mbar_expect_tx(bar(0), geo.a_bytes);
            for (int c = 0; c < NFULL; c++) tma_load_2d(a_base + (uint32_t)c * RS_BM * 128, &tmA, bar(0), c * 64, it.q_row0);
            const uint32_t rem_dst = (ta && (a_loads & 1)) ? a_rem2 : a_rem;
            for (int p = 0; p < REM; p++)
              tma_load_2d(rem_dst + (uint32_t)p * RS_BM * 32, &tmAt, bar(0), NFULL * 64 + p * 16, it.q_row0);
            a_phase ^= 1u;
            a_loads++;
          }
          if (t == ntiles) break;
          TL(8);
          mbar_wait(bar(4 + stage), phase ^ 1u);
          TL(9);
          mbar_expect_tx(bar(2 + stage), geo.b_bytes);
          const uint32_t b_dst = b_base + (uint32_t)stage * geo.b_bytes;
          const int row = it.col0 + t * RS_BN;
          for (int c = 0; c < NFULL; c++) tma_load_2d(b_dst + (uint32_t)c * RS_BN * 128, &tmB, bar(2 + stage), c * 64, row);
          for (int p = 0; p < REM; p++)
            tma_load_2d(b_dst + (uint32_t)(NFULL * RS_BN * 128 + p * RS_BN * 32), &tmBt, bar(2 + stage),
                        NFULL * 64 + p * 16, row);
          TL(10);
          tl_tile++;
          if (++stage == kRsStages) { stage = 0; phase ^= 1u; }
        }
      }
      if (args.cta_clock) {
        args.cta_clock[blockIdx.x * 4 + 2] = n_tiles_done;
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        args.cta_clock[blockIdx.x * 4 + 3] = n_items_done | ((long long)smid << 32);
      }
    }
    __syncwarp();
  } else if (warp == 1 || warp == kRsMmaWarp1) {
    // ================= MMA issuers: one warp per query half =================
    // Each warp runs this loop for ITS accumulator half h (warp-uniform control flow keeps descriptors and barrier
    // addresses in uniform registers); one elected lane issues tcgen05.mma / commit.  The K16 MMAs of a half tile are
    // straight-line code: a single thread's dependent instruction stream costs ~45 cycles per issue, against 96 cycles
    // of tensor work per M128 x N192 x K16 instruction.  Two issuing warps instead of one: a half's next tile is
    // issued as soon as ITS accumulator has been drained, not after the other half's nine MMAs have been pushed
    // through the (back-pressured) issue queue — the accumulator round trip was the tile period (timeline: 2083 of
    // 2122 cycles against 1728 of tensor work).
    const int h = (warp == 1) ? 0 : 1;
    const bool leader = elect_one();
    int stage = 0;
    uint32_t phase = 0, t_phase = 0, a_phase = 0;
    int prev_q0 = -1, prev_qn = -1;
    int a_tiles = -1;                    // index of the resident query tile (parity selects its tail buffer)
    for (int k = 0;; k++) {
      const int w = next_item(k);
      if (w < 0) break;
      const tip_work_item it = args.items[w];
      const int ntiles = (it.col1 - it.col0 + RS_BN - 1) / RS_BN;
      if (ntiles <= 0) continue;
      if (it.q_row0 != prev_q0 || it.q_rows != prev_qn) {
        // a different query tile.  A from shared memory: release the resident one (free once the MMAs issued so
        // far retire), then wait for the new one.  A from tensor memory: the shared-memory copy was released right
        // after it had been copied (below), so the new tile has normally landed long ago.
        if (!ta && prev_qn >= 0 && leader) umma_commit(bar(1));
        __syncwarp();
        prev_q0 = it.q_row0; prev_qn = it.q_rows;
        mbar_wait(bar(0), a_phase);
        a_phase ^= 1u;
        a_tiles++;
        if (ta) {
          tc_fence_after();
          if (leader) {
#pragma unroll
            for (int c = 0; c < NFULL; c++) {
              const uint64_t adesc = smem_desc(a_base + (uint32_t)c * RS_BM * 128 + (uint32_t)h * 128 * 128);
#pragma unroll
              for (int k = 0; k < 4; k++)
                tmem_cp_128x256b(tmem_base + (uint32_t)(h * 256 + RS_BN + (c * 4 + k) * 8), adesc + 2u * k);
            }
            // the copies (and every MMA before them) done -> the producer may fetch the NEXT query tile into the
            // same shared memory while this one is still being used from tensor memory
            umma_commit(bar(1));
          }
          __syncwarp();
        }
      }
      const uint32_t a_rem_cur = (ta && (a_tiles & 1)) ? a_rem2 : a_rem;
      for (int t = 0; t < ntiles; t++) {
        if (leader && h == 0) TL(0);
        mbar_wait(bar(2 + stage), phase);
        if (leader && h == 0) TL(1);
        const uint32_t b_src = b_base + (uint32_t)stage * geo.b_bytes;
#pragma unroll
        for (int cq = 0; cq < 2; cq++) {
          const int q = h * 2 + cq;
          mbar_wait(bar(24 + q), t_phase ^ 1u);   // the epilogue has drained this quarter of the previous tile
          tc_fence_after();
          if (leader) {
            if (cq == 0) TL(2 + 9 * h);   // slots 2 and 11
            const uint32_t d_tmem = tmem_base + (uint32_t)(h * 256 + cq * RS_QN);
            const uint32_t b_q = b_src + (uint32_t)(cq * RS_QN * 128);            // train rows [96 cq, 96 cq + 96) of a chunk
            if (ta) {
              const uint32_t a_t = tmem_base + (uint32_t)(h * 256 + RS_BN);
#pragma unroll
              for (int c = 0; c < NFULL; c++) {
                const uint64_t bdesc = smem_desc(b_q + (uint32_t)c * RS_BN * 128);
#pragma unroll
                for (int k = 0; k < 4; k++) {
                  if (c == 0 && k == 0) umma_bf16_ts_first(d_tmem, a_t, bdesc, kIdescRs);
                  else umma_bf16_ts_acc(d_tmem, a_t + (uint32_t)((c * 4 + k) * 8), bdesc + 2u * k, kIdescRs);
                }
              }
            } else {
#pragma unroll
              for (int c = 0; c < NFULL; c++) {
                const uint64_t adesc = smem_desc(a_base + (uint32_t)c * RS_BM * 128 + (uint32_t)h * 128 * 128);
                const uint64_t bdesc = smem_desc(b_q + (uint32_t)c * RS_BN * 128);
#pragma unroll
                for (int k = 0; k < 4; k++) {
                  if (c == 0 && k == 0) umma_bf16_first(d_tmem, adesc, bdesc, kIdescRs);
                  else umma_bf16_acc(d_tmem, adesc + 2u * k, bdesc + 2u * k, kIdescRs);
                }
              }
            }
#pragma unroll
            for (int p = 0; p < REM; p++) {
              const uint64_t adesc = smem_desc_sw32(a_rem_cur + (uint32_t)p * RS_BM * 32 + (uint32_t)h * 128 * 32);
              const uint64_t bdesc = smem_desc_sw32(b_src + (uint32_t)(NFULL * RS_BN * 128 + p * RS_BN * 32 + cq * RS_QN * 32));
              if (NFULL == 0 && p == 0) umma_bf16_first(d_tmem, adesc, bdesc, kIdescRs);
              else umma_bf16_acc(d_tmem, adesc, bdesc, kIdescRs);
            }
            umma_commit(bar(20 + q));
            if (cq == 1) {
              umma_commit(bar(4 + stage));       // the train tile is free once BOTH halves' MMAs have retired
              TL(3 + 9 * h);   // slots 3 and 12
            }
          }
          __syncwarp();
        }
        tl_tile++;
        if (++stage == kRsStages) { stage = 0; phase ^= 1u; }
        t_phase ^= 1u;
      }
    }
  } else {
    // ===== epilogue: warps 2..17; lane quadrant = warp % 4 (hardware rule), query half and column
    // half from the warp's index among the epilogue warps =====
    const int e = warp - 2;
    const int quad = warp & 3;
    const int mhalf = (e >> 2) & 1;
    const int chalf = e >> 3;
    constexpr int CW = RS_BN / 2;          // columns per thread and tile
    const int row_local = mhalf * 128 + quad * 32 + lane;
    const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(mhalf * 256 + chalf * CW);
    const bool tl_thread = (threadIdx.x == 64);   // first epilogue thread of (half 0, columns 0..95)
    EpiShared sh;
    sh.cand_val = reinterpret_cast<float*>(smem + tiles_bytes + kRsBarBytes);
    sh.cand_col = reinterpret_cast<int*>(sh.cand_val + SLOTS * kRsEpiThreads);
    sh.cand_mask = reinterpret_cast<uint32_t*>(sh.cand_col + SLOTS * kRsEpiThreads);
    sh.etid = threadIdx.x - 64;
    uint32_t t_phase = 0;
    const float kInf = __int_as_float(0x7f800000);
    bool first_item = true;
    for (int k = 0;; k++) {
      const int w = next_item(k);
      if (w < 0) break;
      const tip_work_item it = args.items[w];
      const int ntiles = (it.col1 - it.col0 + RS_BN - 1) / RS_BN;
      if (ntiles <= 0) continue;
      EpiState st;
      st.valid_row = row_local < it.q_rows;
      st.row = (int64_t)it.q_row0 + row_local;
      st.nx = 0.f; st.e2 = 0.f; st.g = 0.f; st.best = kInf; st.thr = kInf; st.s_ref = kInf; st.n_staged = 0;
      st.run_max = -kInf; st.run_sum = 0.f;
      st.col1 = it.col1;
      st.ex_lo = 0; st.ex_hi = 0;
      if (MODE == MODE_NN && st.valid_row) {
        if (EXCL && (it.reserved & 1) && args.q_class) {
          const int cls = args.q_class[st.row];
          st.ex_lo = args.class_off[cls];
          st.ex_hi = args.class_off[cls + 1];
        }
        st.nx = args.q_sqnorm[st.row];
        const float r = sqrtf(st.nx) + args.rmax;
        st.e2 = args.q_err ? 2.f * (args.q_err[st.row] + args.t_err + 1.2e-7f * r) * 1.00001f : args.eps2 * r;
        st.g = args.gamma * r * r;
        st.s_ref = __uint_as_float(ld_volatile_u32(args.row_min_bits + st.row));
        st.thr = nn_threshold(st.s_ref, st.nx, st.e2, st.g);
      }
      const bool dump_item = first_item;
      first_item = false;
      for (int t = 0; t < ntiles; t++) {
        if (tl_thread) TL(4);
        mbar_wait(bar(20 + mhalf * 2 + chalf), t_phase);
        if (tl_thread) TL(5);
        tc_fence_after();
        const int tcol = t * RS_BN + chalf * CW;          // first column of this thread, item-relative
        const int col_base = it.col0 + tcol;
        const bool partial = col_base + CW > it.col1;
        const bool dump = (dump_item && blockIdx.x == 0 && t < 2);
        uint32_t seen_bits = 0x7f800000u;
        if (MODE == MODE_NN && st.valid_row) seen_bits = ld_volatile_u32(args.row_min_bits + st.row);
        uint32_t ra[32], rb[32];
        tmem_ld32(taddr, ra);
        tmem_wait_ld();
        tmem_ld32(taddr + 32, rb);
        epi_chunk<MODE, EXCL, SLOTS, kRsEpiThreads>(args, st, sh, ra, col_base, partial, dump, row_local, tcol);
        tmem_wait_ld();
        tmem_ld32(taddr + 64, ra);
        epi_chunk<MODE, EXCL, SLOTS, kRsEpiThreads>(args, st, sh, rb, col_base + 32, partial, dump, row_local, tcol + 32);
        tmem_wait_ld();
        // accumulator columns of this warp are in registers: hand them back to the MMA warp
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar(24 + mhalf * 2 + chalf));
        if (tl_thread) TL(6);
        epi_chunk<MODE, EXCL, SLOTS, kRsEpiThreads>(args, st, sh, ra, col_base + 64, partial, dump, row_local, tcol + 64);
        if (MODE == MODE_NN && st.valid_row) {
          const float mine = fmaxf(st.best + st.nx, 0.f);
          const float seen = __uint_as_float(seen_bits);
          if (mine < seen) atomicMin(args.row_min_bits + st.row, __float_as_uint(mine));
          if (seen < st.s_ref) {
            st.s_ref = seen;
            st.thr = nn_threshold(st.s_ref, st.nx, st.e2, st.g);
          }
        }
        if (tl_thread) { TL(7); tl_tile++; }
        t_phase ^= 1u;
      }
      if (MODE == MODE_NN && st.valid_row) {
        const float seen = __uint_as_float(ld_volatile_u32(args.row_min_bits + st.row));
        if (seen < st.s_ref) {
          st.s_ref = seen;
          st.thr = nn_threshold(st.s_ref, st.nx, st.e2, st.g);
        }
        for (int k = 0; k < st.n_staged; k++) {
          if (sh.cand_val[k * kRsEpiThreads + sh.etid] <= st.thr) {
            const int pos = atomicAdd(args.cand_cnt + st.row, 1);
            if (pos < args.cap) {
              args.cand_idx[(st.row * args.cap + pos) * 2] = sh.cand_col[k * kRsEpiThreads + sh.etid];
              args.cand_idx[(st.row * args.cap + pos) * 2 + 1] = (int)sh.cand_mask[k * kRsEpiThreads + sh.etid];
            }
          }
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (args.cta_clock && threadIdx.x == 0) args.cta_clock[blockIdx.x * 4 + 1] = global_ns();
  if (args.sched_counter && threadIdx.x == 0) {
    // every CTA has drawn its last pool index by now: the last one out re-arms the counters
    if (atomicAdd(args.sched_counter + 1, 1) == (int)gridDim.x - 1) {
      args.sched_counter[0] = 0;
      args.sched_counter[1] = 0;
    }
  }
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(kTmemCols) : "memory");
  }
}

// ---- host side -----------------------------------------------------------------------------
static PFN_cuTensorMapEncodeTiled_v12000 get_encode() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = (PFN_cuTensorMapEncodeTiled_v12000)p;
  }
  return fn;
}

static int make_map(CUtensorMap* map, const void* basep, int64_t rows, int64_t pitch, int box_rows, int box_cols = BK) {
  auto fn = get_encode();
  if (!fn) { set_error("cuTensorMapEncodeTiled not available from the driver"); return TIP_ERR_CUDA; }
  cuuint64_t gdim[2] = {(cuuint64_t)pitch, (cuuint64_t)rows};
  cuuint64_t gstride[1] = {(cuuint64_t)pitch * 2};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapSwizzle sw = box_cols == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_32B;
  CUresult r = fn(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(basep), gdim, gstride, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed with CUresult %d", (int)r); return TIP_ERR_CUDA; }
  return TIP_OK;
}

static int check_device() {
  static int ok = -1;
  if (ok < 0) {
    int dev = 0, major = 0;
    if (cudaGetDevice(&dev) != cudaSuccess ||
        cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) {
      set_error("no CUDA device");
      return TIP_ERR_CUDA;
    }
    ok = (major == 10) ? 1 : 0;
  }
  if (!ok) { set_error("libb200tip tensor-core kernels need an sm_100 device"); return TIP_ERR_UNSUPPORTED; }
  return TIP_OK;
}

static_assert(kResAChunks * kABytes + kStages * kBBytes + 256 + 1024 <= kSmemBytes, "resident-A layout does not fit");

template <int MODE, bool EXCL = false>
static int launch_pair(const void* q_pack, int64_t m, const void* t_pack, int64_t n, int64_t pitch, PairArgs args,
                       cudaStream_t st) {
  int rc = check_device();
  if (rc != TIP_OK) return rc;
  TIP_REQUIRE(((uintptr_t)q_pack & 127) == 0 && ((uintptr_t)t_pack & 127) == 0, "packed operands must be 128-byte aligned");
  TIP_REQUIRE(pitch % 64 == 0 && args.k16 * 16 <= pitch, "pitch");
  TIP_REQUIRE(m >= 1 && n >= 1 && m < (1LL << 31) && n < (1LL << 31), "shape");
  CUtensorMap ma, mb;
  rc = make_map(&ma, q_pack, m, pitch, BM);
  if (rc != TIP_OK) return rc;
  rc = make_map(&mb, t_pack, n, pitch, BN);
  if (rc != TIP_OK) return rc;
  constexpr int EW = MODE == MODE_LSE ? kLseEpiWarps : 8;
  static bool attr_set = false;   // one flag per template instantiation
  if (!attr_set) {
    TIP_CHECK_CUDA(cudaFuncSetAttribute(pair_kernel<MODE, EXCL, EW>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    if (MODE == MODE_LSE)
      TIP_CHECK_CUDA(cudaFuncSetAttribute(pair_kernel<MODE, EXCL, EW, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmemBytes));
    attr_set = true;
  }
  const int grid = min(args.n_items, sm_count());
  // a query tile that fits stays resident in the log-sum-exp pass (measured at C3: 0.3406 -> 0.3320 ms per step)
  if (MODE == MODE_LSE && (args.k16 + 3) / 4 <= kResAChunks)
    pair_kernel<MODE, EXCL, EW, MODE == MODE_LSE><<<grid, 64 + 32 * EW, kSmemBytes, st>>>(ma, mb, args);
  else
    pair_kernel<MODE, EXCL, EW><<<grid, 64 + 32 * EW, kSmemBytes, st>>>(ma, mb, args);
  TIP_LAUNCH_CHECK();
  return TIP_OK;
}

template <int MODE, bool EXCL = false>
static int launch_pair_rs(const void* q_pack, int64_t m, const void* t_pack, int64_t n, int64_t pitch, PairArgs args,
                          cudaStream_t st) {
  int rc = check_device();
  if (rc != TIP_OK) return rc;
  TIP_REQUIRE(((uintptr_t)q_pack & 127) == 0 && ((uintptr_t)t_pack & 127) == 0, "packed operands must be 128-byte aligned");
  TIP_REQUIRE(args.k16 >= 1 && args.k16 <= kRsMaxK16 && args.k16 * 16 <= pitch, "packed width too large for the resident kernel");
  TIP_REQUIRE(m >= 1 && n >= 1 && m < (1LL << 31) && n < (1LL << 31), "shape");
  CUtensorMap ma, mat, mb, mbt;
  if ((rc = make_map(&ma, q_pack, m, pitch, RS_BM, 64)) != TIP_OK) return rc;
  if ((rc = make_map(&mat, q_pack, m, pitch, RS_BM, 16)) != TIP_OK) return rc;
  if ((rc = make_map(&mb, t_pack, n, pitch, RS_BN, 64)) != TIP_OK) return rc;
  if ((rc = make_map(&mbt, t_pack, n, pitch, RS_BN, 16)) != TIP_OK) return rc;
  static bool attr_set[kRsMaxK16 + 1] = {};   // per template instantiation
  if (!attr_set[args.k16]) {
#define TIP_RS_ATTR(K)                                                                                   \
  case K:                                                                                                \
    TIP_CHECK_CUDA(cudaFuncSetAttribute(pair_rs_kernel<MODE, K, EXCL>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                        rs_smem_bytes(K)));                                              \
    break;
    switch (args.k16) {
      TIP_RS_ATTR(1) TIP_RS_ATTR(2) TIP_RS_ATTR(3) TIP_RS_ATTR(4) TIP_RS_ATTR(5)
      TIP_RS_ATTR(6) TIP_RS_ATTR(7) TIP_RS_ATTR(8) TIP_RS_ATTR(9)
      default: TIP_REQUIRE(false, "k16");
    }
#undef TIP_RS_ATTR
    attr_set[args.k16] = true;
  }
  const int grid = std::min(args.n_items, sm_count());
  const int smem_k = rs_smem_bytes(args.k16);
#define TIP_RS_CASE(K)                                                                                   \
  case K:                                                                                                \
    pair_rs_kernel<MODE, K, EXCL><<<grid, kRsThreads, smem_k, st>>>(ma, mat, mb, mbt, args);               \
    break;
  switch (args.k16) {
    TIP_RS_CASE(1) TIP_RS_CASE(2) TIP_RS_CASE(3) TIP_RS_CASE(4) TIP_RS_CASE(5)
    TIP_RS_CASE(6) TIP_RS_CASE(7) TIP_RS_CASE(8) TIP_RS_CASE(9)
    default: TIP_REQUIRE(false, "k16");
  }
#undef TIP_RS_CASE
  TIP_LAUNCH_CHECK();
  return TIP_OK;
}

static int k16_of(int64_t d, int segments) {
  const int64_t d16 = (d + 15) & ~(int64_t)15;
  return (int)((segments * d16 + 16) / 16);
}

}  // namespace tip

using namespace tip;

static long long* g_timeline = nullptr;
static int g_timeline_tiles = 0;
static long long* g_cta_clock = nullptr;
extern "C" int tip_debug_timeline(long long* buf, int32_t tiles) {
  g_timeline = buf;
  g_timeline_tiles = tiles;
  return TIP_OK;
}
extern "C" int tip_debug_cta_clock(long long* buf) {
  g_cta_clock = buf;
  return TIP_OK;
}

extern "C" int tip_nn_filter(const void* q_pack, const float* q_sqnorm, int64_t m, const void* t_pack, int64_t n,
                             int64_t d, int64_t pitch, const tip_work_item* items, int32_t n_items,
                             const int32_t* q_class, const int32_t* class_off, float t_rmax,
                             const float* q_rounderr, float t_errmax, uint32_t* row_min_bits, int32_t* cand_idx,
                             int32_t* cand_cnt, int32_t cap, int32_t n_static, int32_t* sched_counter,
                             void* stream) {
  TIP_REQUIRE(q_pack && q_sqnorm && t_pack && items && row_min_bits && cand_idx && cand_cnt, "null pointer");
  TIP_REQUIRE(cap >= 1 && n_items >= 0, "cap / n_items");
  TIP_REQUIRE(pitch == tip_pair_pitch(d, 1), "pitch does not match tip_pair_pitch(d, 1)");
  if (n_items == 0) return TIP_OK;
  PairArgs a{};
  a.items = items; a.n_items = n_items; a.k16 = k16_of(d, 1); a.m = m;
  TIP_REQUIRE(n_static >= 0 && n_static <= n_items, "n_static");
  TIP_REQUIRE(sched_counter != nullptr || n_static == n_items, "a pool of dynamic items needs sched_counter");
  a.n_static = n_static; a.sched_counter = n_static < n_items ? sched_counter : nullptr;
  TIP_REQUIRE(a.k16 <= kRsMaxK16 || n_static == n_items, "dynamic items need the resident-query kernel (d <= 128)");
  a.q_sqnorm = q_sqnorm; a.rmax = t_rmax;
  a.q_err = q_rounderr; a.t_err = t_errmax;
  TIP_REQUIRE(!q_rounderr || t_errmax >= 0.f, "t_errmax");
  a.q_class = q_class; a.class_off = class_off;
  // eps' = (2^-9 + 2^-23)/(1 - that): bf16 rounding of the centred traces (triangle inequality);
  // gamma: fp32 accumulation over K products + norm rounding, assuming nothing better than
  // truncating adds inside the tensor core.
  a.eps2 = 2.0f * 1.96e-3f;
  a.gamma = (float)(a.k16 * 16 + 16) * 1.1920929e-7f;
  a.row_min_bits = row_min_bits; a.cand_idx = cand_idx; a.cand_cnt = cand_cnt; a.cap = cap;
  a.timeline = g_timeline; a.timeline_tiles = g_timeline_tiles;
  a.cta_clock = g_cta_clock;
  const bool excl = q_class != nullptr && class_off != nullptr;   // per-query own-class masking compiled in only then
  if (a.k16 <= kRsMaxK16)
    return excl ? launch_pair_rs<MODE_NN, true>(q_pack, m, t_pack, n, pitch, a, (cudaStream_t)stream)
                : launch_pair_rs<MODE_NN, false>(q_pack, m, t_pack, n, pitch, a, (cudaStream_t)stream);
  return excl ? launch_pair<MODE_NN, true>(q_pack, m, t_pack, n, pitch, a, (cudaStream_t)stream)
              : launch_pair<MODE_NN, false>(q_pack, m, t_pack, n, pitch, a, (cudaStream_t)stream);
}

extern "C" int tip_nn_filter_tile(int64_t d, int32_t* q_rows, int32_t* t_rows) {
  TIP_REQUIRE(d >= 1 && q_rows && t_rows, "arguments");
  const bool rs = k16_of(d, 1) <= kRsMaxK16;
  *q_rows = rs ? RS_BM : BM;
  *t_rows = rs ? RS_BN : BN;
  return TIP_OK;
}

extern "C" int tip_nn_filter_kind(int64_t d) {
  if (d < 1) return -1;
  return k16_of(d, 1) <= kRsMaxK16 ? 1 : 0;
}

extern "C" int tip_kde_tile_rows(void) { return BM; }
extern "C" int tip_kde_slot_parts(void) { return kLseEpiWarps / 4; }

extern "C" int tip_kde_lse(const void* q_pack, int64_t m, const void* t_pack, int64_t n, int64_t d, int64_t pitch,
                           const tip_work_item* items, int32_t n_items, float* part_max, float* part_sum,
                           void* stream) {
  TIP_REQUIRE(q_pack && t_pack && items && part_max && part_sum, "null pointer");
  TIP_REQUIRE(pitch == tip_pair_pitch(d, 3), "pitch does not match tip_pair_pitch(d, 3)");
  if (n_items == 0) return TIP_OK;
  PairArgs a{};
  a.items = items; a.n_items = n_items; a.n_static = n_items; a.k16 = k16_of(d, 3); a.m = m;
  a.part_max = part_max; a.part_sum = part_sum;
  return launch_pair<MODE_LSE>(q_pack, m, t_pack, n, pitch, a, (cudaStream_t)stream);
}

extern "C" int tip_kde_lse_f16(const void* q_pack, int64_t m, const void* t_pack, int64_t n, int64_t d, int64_t pitch,
                               const tip_work_item* items, int32_t n_items, float* part_max, float* part_sum,
                               void* stream) {
  TIP_REQUIRE(q_pack && t_pack && items && part_max && part_sum, "null pointer");
  TIP_REQUIRE(pitch == tip_pair_pitch(d, 1), "pitch does not match tip_pair_pitch(d, 1)");
  if (n_items == 0) return TIP_OK;
  PairArgs a{};
  a.items = items; a.n_items = n_items; a.n_static = n_items; a.k16 = k16_of(d, 1); a.m = m;
  a.part_max = part_max; a.part_sum = part_sum;
  a.idesc = kIdescF16;
  return launch_pair<MODE_LSE>(q_pack, m, t_pack, n, pitch, a, (cudaStream_t)stream);
}

extern "C" int tip_pair_probe(const void* q_pack, int64_t m, const void* t_pack, int64_t n, int64_t d, int segments,
                              int64_t pitch, int variant, float* out, void* stream) {
  TIP_REQUIRE(q_pack && t_pack && out, "null pointer");
  TIP_REQUIRE(pitch == tip_pair_pitch(d, segments), "pitch does not match tip_pair_pitch");
  TIP_REQUIRE(variant >= 0 && variant <= 2, "variant: 0 auto, 1 streaming, 2 resident");
  static tip_work_item* d_item = nullptr;
  if (!d_item) TIP_CHECK_CUDA(cudaMalloc(&d_item, sizeof(tip_work_item)));
  const int k16 = k16_of(d, segments);
  const bool rs = variant == 2 || (variant == 0 && k16 <= kRsMaxK16);
  tip_work_item h{0, (int32_t)std::min<int64_t>(m, rs ? RS_BM : BM), 0, (int32_t)std::min<int64_t>(n, 256), 0, 0};
  TIP_CHECK_CUDA(cudaMemcpyAsync(d_item, &h, sizeof(h), cudaMemcpyHostToDevice, (cudaStream_t)stream));
  PairArgs a{};
  a.items = d_item; a.n_items = 1; a.n_static = 1; a.k16 = k16; a.m = m; a.dump = out;
  if (rs) return launch_pair_rs<MODE_DUMP>(q_pack, m, t_pack, n, pitch, a, (cudaStream_t)stream);
  return launch_pair<MODE_DUMP>(q_pack, m, t_pack, n, pitch, a, (cudaStream_t)stream);
}
