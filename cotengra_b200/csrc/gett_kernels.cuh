// gett_kernels.cuh -- permutation-fused pairwise tensor contraction for sm_100a.
//
// Replaces cotengra/contract.py:364-411 (`_do_contraction_via_bmm`: transpose ->
// reshape(copy) -> matmul -> reshape/transpose) by ONE kernel:
//   * operands are read where they lie: every tile element is fetched with a
//     cp.async (LDGSTS) from  base(tile) + kbase(k-step) + delta(element),
//     the three terms being sums of digit*stride over the GRID, K-GRID and TILE
//     dims of the descriptor (gett_desc.h);  no permuted copy of A, B or C is
//     ever materialised in HBM;
//   * a 3-4 stage shared-memory ring hides HBM/L2 latency;
//   * the compute policy is pluggable: FMA register tiles (any dtype), per-thread
//     k partial sums (dot-product-like nodes), or fp64 tensor-core mma.sync
//     (DMMA m8n8k4) for float64 / complex128;
//   * results are stored straight into the parent's index order (strided C),
//     optionally accumulated (slice sums, core.py:3842-3844) or atomically
//     added (split-K).
#pragma once
#include <cuda_runtime.h>
#include <math_constants.h>
#include <stdint.h>

#include "gett_desc.h"

namespace ctgb {

// ------------------------------------------------------------------ elements
__device__ __forceinline__ void mac(float& c, float a, float b) { c = fmaf(a, b, c); }
__device__ __forceinline__ void mac(double& c, double a, double b) { c = fma(a, b, c); }
__device__ __forceinline__ void mac(float2& c, float2 a, float2 b) {
  c.x = fmaf(a.x, b.x, c.x);
  c.x = fmaf(-a.y, b.y, c.x);
  c.y = fmaf(a.x, b.y, c.y);
  c.y = fmaf(a.y, b.x, c.y);
}
__device__ __forceinline__ void mac(double2& c, double2 a, double2 b) {
  c.x = fma(a.x, b.x, c.x);
  c.x = fma(-a.y, b.y, c.x);
  c.y = fma(a.x, b.y, c.y);
  c.y = fma(a.y, b.x, c.y);
}
template <typename T> __device__ __forceinline__ T zero_of();
template <> __device__ __forceinline__ float zero_of<float>() { return 0.f; }
template <> __device__ __forceinline__ double zero_of<double>() { return 0.0; }
template <> __device__ __forceinline__ float2 zero_of<float2>() { return make_float2(0.f, 0.f); }
template <> __device__ __forceinline__ double2 zero_of<double2>() { return make_double2(0.0, 0.0); }

__device__ __forceinline__ float add_of(float a, float b) { return a + b; }
__device__ __forceinline__ double add_of(double a, double b) { return a + b; }
__device__ __forceinline__ float2 add_of(float2 a, float2 b) { return make_float2(a.x + b.x, a.y + b.y); }
__device__ __forceinline__ double2 add_of(double2 a, double2 b) { return make_double2(a.x + b.x, a.y + b.y); }

__device__ __forceinline__ void atomic_add_of(float* p, float v) { atomicAdd(p, v); }
__device__ __forceinline__ void atomic_add_of(double* p, double v) { atomicAdd(p, v); }
__device__ __forceinline__ void atomic_add_of(float2* p, float2 v) {
  atomicAdd(&p->x, v.x);
  atomicAdd(&p->y, v.y);
}
__device__ __forceinline__ void atomic_add_of(double2* p, double2 v) {
  atomicAdd(&p->x, v.x);
  atomicAdd(&p->y, v.y);
}

// two adjacent elements with one store; 256-bit (STG.E.ENL2.256) for complex128
template <typename T>
__device__ __forceinline__ void store_pair_of(T* p, T v0, T v1) {
  p[0] = v0;
  p[1] = v1;
}
template <>
__device__ __forceinline__ void store_pair_of<double2>(double2* p, double2 v0, double2 v1) {
  asm volatile("st.global.v4.f64 [%0], {%1,%2,%3,%4};" ::"l"(p), "d"(v0.x), "d"(v0.y), "d"(v1.x), "d"(v1.y)
               : "memory");
}

__device__ __forceinline__ float shfl_down_of(float v, int d) { return __shfl_down_sync(0xffffffffu, v, d); }
__device__ __forceinline__ double shfl_down_of(double v, int d) { return __shfl_down_sync(0xffffffffu, v, d); }
__device__ __forceinline__ float2 shfl_down_of(float2 v, int d) {
  return make_float2(__shfl_down_sync(0xffffffffu, v.x, d), __shfl_down_sync(0xffffffffu, v.y, d));
}
__device__ __forceinline__ double2 shfl_down_of(double2 v, int d) {
  return make_double2(__shfl_down_sync(0xffffffffu, v.x, d), __shfl_down_sync(0xffffffffu, v.y, d));
}

// ------------------------------------------------------------------ fused strip_exponent
// contract.py:816-829 normalises every pairwise result by its largest magnitude and adds the
// log10 of that factor to a running exponent.  Done literally that is two extra passes over
// every intermediate (max, then divide).  Here the division is LAZY: a node stores its raw
// product and records factor = max|C| in a slot; whoever consumes C multiplies its own
// accumulators by 1/(factor_A * factor_B) in the epilogue -- the same numbers the reference
// forms, (A/fA)(B/fB), since the product is bilinear -- and the exponent is the sum of
// log10(factor) over the nodes, formed once per slice.
struct StripMax {
  double run2;              // largest |value|^2 this thread has stored (the common path)
  double runh;              // largest |value| among values whose square leaves the double range
  int thr, thrf;            // integer filters: high word of (max/sqrt 2) as a double / its bits as a float
};
struct StripCtx {
  double s;                 // 1/(fA fB): one multiply per component (0 when an operand is identically
                            // zero: check_zero); unused when the host pre-scaled the small operand
  double sb;                // second factor, only used when the product 1/fA * 1/fB leaves the double range
  float sf;                 // s as a float when it is a normal float (single precision kernels), else 0
  StripMax m;
  unsigned long long* fc;   // factor slot of C (nullptr: the caller measures C separately)
  bool on, scale, two;
};
__device__ __forceinline__ StripCtx strip_begin(const int64_t* __restrict__ D) {
  StripCtx c;
  const double* pa = reinterpret_cast<const double*>(D[W_SCALE_A]);
  const double* pb = reinterpret_cast<const double*>(D[W_SCALE_B]);
  c.scale = pa != nullptr;
  c.fc = reinterpret_cast<unsigned long long*>(D[W_FACTOR_C]);
  c.on = c.scale || c.fc != nullptr;
  c.m.run2 = c.m.runh = 0.0;
  c.m.thr = c.m.thrf = 0;
  c.s = c.sb = 1.0;
  c.sf = 1.f;
  c.two = false;
  if (c.scale) {
    const double fa = *pa, fb = *pb;
    const double sa = fa != 0.0 ? 1.0 / fa : 0.0, sb = fb != 0.0 ? 1.0 / fb : 0.0;
    const double prod = sa * sb;
    // (1/fA)(1/fB) overflows or underflows only for factors near the ends of the double range; a
    // subnormal product has lost significant bits already (1e-160 * 1e-160: 11 of 53)
    c.two = (sa != 0.0 && sb != 0.0) && (prod < 2.2250738585072014e-308 || prod > 1.7e308);
    c.s = c.two ? sa : prod;
    c.sb = c.two ? sb : 1.0;
    const double ap = fabs(prod);
    // (sf == 0 with s != 0: single precision kernels fall back to the double multiply)
    c.sf = (!c.two && (ap == 0.0 || (ap > 1e-30 && ap < 1e30))) ? (float)prod : 0.f;
  }
  return c;
}
// max |v|: INLINE there is only an integer filter -- non-negative floating-point numbers order like
// their bit patterns, so an element whose larger component lies below (current maximum)/sqrt(2) is
// dismissed with four ALU instructions and touches neither the fp64 pipe the DMMAs run on nor the
// instruction cache (with the arithmetic inlined at each of the 32-64 store sites of an unrolled
// epilogue the DMMA nodes lost 18 %, the tcgen05 nodes 60 %: instruction fetch).  The rare candidates
// call ONE out-of-line routine: re^2 + im^2 against the running maximum of squares (square root taken
// once at the end); squares that would leave the double range, and NaNs, take a hypot path with its own
// maximum, so that magnitudes down to the denormals survive.
__device__ __noinline__ StripMax strip_track_slow(StripMax m, double re, double im) {
  const double q = fma(re, re, im * im);
  if (q >= 1e-280 && q <= 1e300) {
    if (!(q > m.run2)) return m;
    m.run2 = q;
  } else if (!(re == 0.0 && im == 0.0)) {
    const double hy = hypot(re, im);                         // tiny, huge or NaN
    m.runh = (hy != hy || m.runh != m.runh) ? __longlong_as_double(0x7ff8000000000000LL) : fmax(m.runh, hy);
  } else {
    return m;
  }
  // high word of max/sqrt(2), rounded down: everything strictly below it cannot raise the maximum
  const double t = fmax(sqrt(m.run2), m.runh) * 0.70710678118654746;
  m.thr = (t == t) ? __double2hiint(t) : 0;
  m.thrf = (t == t && t < 3e38) ? __float_as_int((float)t * 0.999999f) : 0;
  return m;
}
__device__ __forceinline__ void strip_track(StripCtx& c, double re, double im) {
  const int h = max(__double2hiint(re) & 0x7fffffff, __double2hiint(im) & 0x7fffffff);
  if (h >= c.m.thr) c.m = strip_track_slow(c.m, re, im);
}
__device__ __forceinline__ void strip_track_f(StripCtx& c, float re, float im) {
  const int h = max(__float_as_int(re) & 0x7fffffff, __float_as_int(im) & 0x7fffffff);
  if (h >= c.m.thrf) c.m = strip_track_slow(c.m, (double)re, (double)im);
}
// branch-free part of the filter, for a scan over a whole tile of accumulators before they are
// stored: the bit pattern of the largest component, sign stripped (two integer ops per component)
__device__ __forceinline__ int strip_hi(float v) { return __float_as_int(v) & 0x7fffffff; }
__device__ __forceinline__ int strip_hi(double v) { return __double2hiint(v) & 0x7fffffff; }
__device__ __forceinline__ int strip_hi(float2 v) { return max(strip_hi(v.x), strip_hi(v.y)); }
__device__ __forceinline__ int strip_hi(double2 v) { return max(strip_hi(v.x), strip_hi(v.y)); }
template <typename T> struct StripSingle { static constexpr bool value = false; };
template <> struct StripSingle<float> { static constexpr bool value = true; };
template <> struct StripSingle<float2> { static constexpr bool value = true; };
// can anything with this (sign-stripped) leading bit pattern raise the running maximum?
template <typename T>
__device__ __forceinline__ bool strip_hot(const StripCtx& c, int hmax) {
  return hmax >= (StripSingle<T>::value ? c.m.thrf : c.m.thr);
}
__device__ __forceinline__ void strip_note(StripCtx& c, float v) { strip_track_f(c, v, 0.f); }
__device__ __forceinline__ void strip_note(StripCtx& c, double v) { strip_track(c, v, 0.0); }
__device__ __forceinline__ void strip_note(StripCtx& c, float2 v) { strip_track_f(c, v.x, v.y); }
__device__ __forceinline__ void strip_note(StripCtx& c, double2 v) { strip_track(c, v.x, v.y); }
__device__ __forceinline__ double strip_mul(const StripCtx& c, double v) { return c.two ? v * c.s * c.sb : v * c.s; }
__device__ __forceinline__ float strip_mul(const StripCtx& c, float v) {
  return (c.sf != 0.f || c.s == 0.0) ? v * c.sf : (float)strip_mul(c, (double)v);
}
__device__ __forceinline__ float strip_apply(StripCtx& c, float v) {
  const float r = c.scale ? strip_mul(c, v) : v;
  strip_track_f(c, r, 0.f);
  return r;
}
__device__ __forceinline__ double strip_apply(StripCtx& c, double v) {
  const double r = c.scale ? strip_mul(c, v) : v;
  strip_track(c, r, 0.0);
  return r;
}
__device__ __forceinline__ float2 strip_apply(StripCtx& c, float2 v) {
  const float2 r = c.scale ? make_float2(strip_mul(c, v.x), strip_mul(c, v.y)) : v;
  strip_track_f(c, r.x, r.y);
  return r;
}
__device__ __forceinline__ double2 strip_apply(StripCtx& c, double2 v) {
  const double2 r = c.scale ? make_double2(strip_mul(c, v.x), strip_mul(c, v.y)) : v;
  strip_track(c, r.x, r.y);
  return r;
}
// all threads of the (converged) warp: one atomicMax per warp; non-negative doubles order like
// their bit patterns, NaN (sign clear) above everything -- it propagates like the reference's
__device__ __forceinline__ void strip_end(const StripCtx& c) {
  if (c.fc == nullptr) return;
  const double m = fmax(sqrt(c.m.run2), c.m.runh);
  const bool nan = c.m.run2 != c.m.run2 || c.m.runh != c.m.runh;
  unsigned long long bits = (unsigned long long)__double_as_longlong(nan ? __longlong_as_double(0x7ff8000000000000LL) : m);
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    const unsigned long long o = __shfl_xor_sync(0xffffffffu, bits, d);
    bits = o > bits ? o : bits;
  }
  if ((threadIdx.x & 31) == 0 && bits != 0ull) atomicMax(c.fc, bits);
}

// ------------------------------------------------------------------ cp.async
template <int BYTES>
__device__ __forceinline__ void cp_async_zfill(void* smem_dst, const void* gsrc, bool valid) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  int src_bytes = valid ? BYTES : 0;
  if constexpr (BYTES == 16) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(s), "l"(gsrc), "r"(src_bytes) : "memory");
  } else {
    asm volatile("cp.async.ca.shared.global [%0], [%1], %2, %3;\n" ::"r"(s), "l"(gsrc), "n"(BYTES), "r"(src_bytes)
                 : "memory");
  }
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory");
}

// sum of NON-NEGATIVE 64-bit offsets over the warp with three redux.sync
// (24-bit chunks cannot overflow 32 bits when added over 32 lanes)
__device__ __forceinline__ long long warp_sum_ll(long long v) {
  const unsigned long long u = (unsigned long long)v;
  const unsigned lo = __reduce_add_sync(0xffffffffu, (unsigned)(u & 0xFFFFFFull));
  const unsigned mid = __reduce_add_sync(0xffffffffu, (unsigned)((u >> 24) & 0xFFFFFFull));
  const unsigned hi = __reduce_add_sync(0xffffffffu, (unsigned)(u >> 48));
  return (long long)((unsigned long long)lo + ((unsigned long long)mid << 24) + ((unsigned long long)hi << 48));
}
__device__ __forceinline__ int warp_sum_i(int v) { return (int)__reduce_add_sync(0xffffffffu, (unsigned)v); }

// ------------------------------------------------------------------ policies
// A policy fixes the CTA tile (MT x NT x KT), the pipeline depth, the shared
// memory layout of the operand tiles and how the tile product is computed.

// Generic FMA register-tile policy: works for every dtype and every extent.
template <typename T, int MT_, int NT_, int KT_, int STAGES_>
struct SimtPolicy {
  static constexpr int MT = MT_, NT = NT_, KT = KT_, STAGES = STAGES_;
  static constexpr int THREADS = 256;
  static constexpr int TM = MT / 16, TN = NT / 16;
  static constexpr int A_ELEMS = MT * KT, B_ELEMS = NT * KT;
  static constexpr int SCRATCH_ELEMS = 0;
  static constexpr int CONSUMER_REGS = 0, PRODUCER_REGS = 0;
  static constexpr bool HAS_BCACHE = false;
  static constexpr int MIN_BLOCKS = sizeof(T) == 16 ? 1 : 2;
  // strip_exponent: may the epilogue be traversed more than once (scan for max|C|, then store)?
  static constexpr bool SCAN_OK = true;
  struct Acc {
    T v[TM][TN];
  };
  __device__ static __forceinline__ int idxA(int r, int kk) { return kk * MT + r; }
  __device__ static __forceinline__ int idxB(int c, int kk) { return kk * NT + c; }
  __device__ static __forceinline__ void clear(Acc& acc) {
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
      for (int j = 0; j < TN; ++j) acc.v[i][j] = zero_of<T>();
  }
  __device__ static __forceinline__ void compute(const T* __restrict__ sA, const T* __restrict__ sB, Acc& acc,
                                                 int kvalid, int ncols) {
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
#pragma unroll
    for (int kk = 0; kk < KT; ++kk) {
      T a[TM], b[TN];
#pragma unroll
      for (int i = 0; i < TM; ++i) a[i] = sA[kk * MT + ty + 16 * i];
#pragma unroll
      for (int j = 0; j < TN; ++j) b[j] = sB[kk * NT + tx + 16 * j];
#pragma unroll
      for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < TN; ++j) mac(acc.v[i][j], a[i], b[j]);
    }
  }
  __device__ static __forceinline__ void finalize(Acc&) {}
  template <typename F, typename F2>
  __device__ static __forceinline__ void epilogue(Acc& acc, T* scratch, F&& store, F2&& store_pair, bool pair_ok,
                                                  int ncols) {
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
      for (int j = 0; j < TN; ++j) store(ty + 16 * i, tx + 16 * j, acc.v[i][j]);
  }
};

// Tiny M x N with a huge contracted space (the final inner product of an
// amplitude network is M = N = 1, K = 2^30): every thread owns a strided set
// of k and all (r, c) pairs; partial sums are reduced across the block once.
template <typename T, int MT_, int NT_, int KT_, int STAGES_>
struct KredPolicy {
  static constexpr int MT = MT_, NT = NT_, KT = KT_, STAGES = STAGES_;
  static constexpr int THREADS = 256;
  static constexpr int A_ELEMS = MT * KT, B_ELEMS = NT * KT;
  static constexpr int SCRATCH_ELEMS = MT * NT * (THREADS / 32);
  static constexpr int CONSUMER_REGS = 0, PRODUCER_REGS = 0;
  static constexpr bool HAS_BCACHE = false;
  static constexpr int MIN_BLOCKS = 2;
  // strip_exponent: may the epilogue be traversed more than once (scan for max|C|, then store)?
  static constexpr bool SCAN_OK = false;
  struct Acc {
    T v[MT][NT];
  };
  __device__ static __forceinline__ int idxA(int r, int kk) { return r * KT + kk; }
  __device__ static __forceinline__ int idxB(int c, int kk) { return c * KT + kk; }
  __device__ static __forceinline__ void clear(Acc& acc) {
#pragma unroll
    for (int i = 0; i < MT; ++i)
#pragma unroll
      for (int j = 0; j < NT; ++j) acc.v[i][j] = zero_of<T>();
  }
  __device__ static __forceinline__ void compute(const T* __restrict__ sA, const T* __restrict__ sB, Acc& acc,
                                                 int kvalid, int ncols) {
#pragma unroll
    for (int kk = threadIdx.x; kk < KT; kk += THREADS) {
      T a[MT], b[NT];
#pragma unroll
      for (int i = 0; i < MT; ++i) a[i] = sA[i * KT + kk];
#pragma unroll
      for (int j = 0; j < NT; ++j) b[j] = sB[j * KT + kk];
#pragma unroll
      for (int i = 0; i < MT; ++i)
#pragma unroll
        for (int j = 0; j < NT; ++j) mac(acc.v[i][j], a[i], b[j]);
    }
  }
  __device__ static __forceinline__ void finalize(Acc&) {}
  template <typename F, typename F2>
  __device__ static __forceinline__ void epilogue(Acc& acc, T* scratch, F&& store, F2&& store_pair, bool pair_ok,
                                                  int ncols) {
    // block reduction of every (r, c) partial sum: shuffles, then 8 warps via smem
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
    for (int i = 0; i < MT; ++i)
#pragma unroll
      for (int j = 0; j < NT; ++j) {
        T v = acc.v[i][j];
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) v = add_of(v, shfl_down_of(v, d));
        if (lane == 0) scratch[(i * NT + j) * (THREADS / 32) + warp] = v;
      }
    asm volatile("bar.sync 2, %0;\n" ::"n"(THREADS) : "memory");  // consumers only
    if (threadIdx.x < MT * NT) {
      T v = zero_of<T>();
#pragma unroll
      for (int w = 0; w < THREADS / 32; ++w) v = add_of(v, scratch[threadIdx.x * (THREADS / 32) + w]);
      store(threadIdx.x / NT, threadIdx.x % NT, v);
    }
    asm volatile("bar.sync 2, %0;\n" ::"n"(THREADS) : "memory");
  }
};

// Skinny nodes (few kept indices on the small operand: N <= 8) are HBM-bound.
// 128 consumer threads, two output rows per thread; the small operand is
// broadcast from shared memory, or -- when its tile is the same for every work
// item (all of K and N inside the tile, no batch) -- read ONCE into registers
// (broadcast LDS.128 of B were 60% of the shared-memory wavefronts under ncu).
template <typename T, int MT_, int NT_, int KT_, int STAGES_>
struct RowPolicy {
  static constexpr int MT = MT_, NT = NT_, KT = KT_, STAGES = STAGES_;
  static constexpr int THREADS = MT / 2;
  static constexpr int A_ELEMS = MT * KT, B_ELEMS = NT * KT;
  static constexpr int SCRATCH_ELEMS = 0;
  // (no setmaxnreg here: the CTA's register pool is regs-per-thread as chosen by
  // ptxas times the block size, and an .inc beyond that pool would block forever)
  static constexpr int CONSUMER_REGS = 0, PRODUCER_REGS = 0;
  static constexpr int MIN_BLOCKS = 2;
  static constexpr bool HAS_BCACHE = sizeof(T) * KT * NT <= 256;
  struct BCache {
    T v[KT][NT];
  };
  // strip_exponent: may the epilogue be traversed more than once (scan for max|C|, then store)?
  static constexpr bool SCAN_OK = true;
  struct Acc {
    T v[2][NT];
  };
  __device__ static __forceinline__ int idxA(int r, int kk) { return kk * MT + r; }
  __device__ static __forceinline__ int idxB(int c, int kk) { return kk * NT + c; }
  __device__ static __forceinline__ void clear(Acc& acc) {
#pragma unroll
    for (int j = 0; j < NT; ++j) acc.v[0][j] = acc.v[1][j] = zero_of<T>();
  }
  __device__ static __forceinline__ void load_b(const T* __restrict__ sB, BCache& bc) {
#pragma unroll
    for (int kk = 0; kk < KT; ++kk)
#pragma unroll
      for (int j = 0; j < NT; ++j) bc.v[kk][j] = sB[kk * NT + j];
  }
  __device__ static __forceinline__ void compute_cached(const T* __restrict__ sA, const BCache& bc, Acc& acc,
                                                        int kvalid, int ncols) {
#pragma unroll
    for (int kk = 0; kk < KT; ++kk) {
      if (kk < kvalid) {
        const T a0 = sA[kk * MT + threadIdx.x], a1 = sA[kk * MT + threadIdx.x + THREADS];
#pragma unroll
        for (int j = 0; j < NT; ++j)
          if (j < ncols) {
            mac(acc.v[0][j], a0, bc.v[kk][j]);
            mac(acc.v[1][j], a1, bc.v[kk][j]);
          }
      }
    }
  }
  __device__ static __forceinline__ void compute(const T* __restrict__ sA, const T* __restrict__ sB, Acc& acc,
                                                 int kvalid, int ncols) {
#pragma unroll 1
    for (int kk = 0; kk < KT; ++kk) {
      if (kk >= kvalid) break;
      const T a0 = sA[kk * MT + threadIdx.x], a1 = sA[kk * MT + threadIdx.x + THREADS];
#pragma unroll
      for (int j = 0; j < NT; ++j) {
        if (j >= ncols) break;
        const T b = sB[kk * NT + j];
        mac(acc.v[0][j], a0, b);
        mac(acc.v[1][j], a1, b);
      }
    }
  }
  __device__ static __forceinline__ void finalize(Acc&) {}
  template <typename F, typename F2>
  __device__ static __forceinline__ void epilogue(Acc& acc, T* scratch, F&& store, F2&& store_pair, bool pair_ok,
                                                  int ncols) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int r = (int)threadIdx.x + h * THREADS;
      if (pair_ok) {
        // the row's columns are adjacent in C: 32-byte (256-bit) stores, full sectors
#pragma unroll
        for (int j = 0; j < NT; j += 2) {
          if (j >= ncols) break;
          store_pair(r, j, acc.v[h][j], acc.v[h][j + 1]);
        }
      } else {
#pragma unroll
        for (int j = 0; j < NT; ++j) {
          if (j >= ncols) break;
          store(r, j, acc.v[h][j]);
        }
      }
    }
  }
};

// fp64 tensor-core policy: mma.sync.aligned.m8n8k4 (DMMA).  tcgen05 has no f64
// kind (cute/arch/mma_sm100_umma.hpp exposes f16/tf32/f8f6f4/i8/mx* only), so
// the double-precision tensor path on sm_100a is the warp-level DMMA.
// Complex products are four real DMMAs per (A-frag, B-frag) pair:
//   Cr += Ar*Br;  Cr += (-Ai)*Bi;  Ci += Ar*Bi;  Ci += Ai*Br
// or, with M3 ("3M", the ZGEMM3M identity), three:
//   P1 += Ar*Br;  P2 += Ai*Bi;  P3 += (Ar+Ai)*(Br+Bi);   Cr = P1 - P2,  Ci = P3 - P1 - P2
// -- 25 % fewer tensor-pipe cycles for 50 % more accumulator registers (hence the
// narrower warp tiles of the 3M variants) and a normwise (not componentwise) error
// bound of the same order, K*eps*|A||B|.
__device__ __forceinline__ void dmma8x8x4(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(c0), "+d"(c1)
               : "d"(a), "d"(b));
}

template <typename T, int WARPS_M, int WARPS_N, int FM, int FN, int KT_, int STAGES_, bool M3_ = false>
struct DmmaPolicy {
  // T is double (real) or double2 (complex)
  static constexpr bool CPLX = sizeof(T) == 16;
  static constexpr bool M3 = M3_ && CPLX;
  static constexpr int MT = WARPS_M * FM * 8, NT = WARPS_N * FN * 8, KT = KT_, STAGES = STAGES_;
  static constexpr int THREADS = WARPS_M * WARPS_N * 32;
  static constexpr int A_ELEMS = MT * KT, B_ELEMS = NT * KT;
  static constexpr int SCRATCH_ELEMS = 0;
  // 8 consumer warps x 232 + 4 producer warps x 40 registers = 64512 <= 65536
  static constexpr int CONSUMER_REGS = (THREADS == 256) ? 232 : 0, PRODUCER_REGS = 40;
  static constexpr bool HAS_BCACHE = false;
  static constexpr int MIN_BLOCKS = THREADS <= 128 ? 2 : 1;  // the 32 x 32 split-K policy: two CTAs per SM
  static_assert(KT % 4 == 0, "KT must be a multiple of the DMMA k");
  static constexpr bool SCAN_OK = true;
  struct Acc {
    double re[FM][FN][2];
    double im[CPLX ? FM : 1][CPLX ? FN : 1][2];
    double p3[M3 ? FM : 1][M3 ? FN : 1][2];  // 3M: re = P1, im = P2 until the epilogue
  };
  // [k/4][row][k%4]: the 4 k of one fragment row are contiguous (64 B complex),
  // fragment rows contiguous -> conflict-free LDS.128 / LDS.64 fragment loads.
  __device__ static __forceinline__ int idxA(int r, int kk) { return ((kk >> 2) * MT + r) * 4 + (kk & 3); }
  __device__ static __forceinline__ int idxB(int c, int kk) { return ((kk >> 2) * NT + c) * 4 + (kk & 3); }
  __device__ static __forceinline__ void clear(Acc& acc) {
#pragma unroll
    for (int i = 0; i < FM; ++i)
#pragma unroll
      for (int j = 0; j < FN; ++j) {
        acc.re[i][j][0] = acc.re[i][j][1] = 0.0;
        if constexpr (CPLX) acc.im[i][j][0] = acc.im[i][j][1] = 0.0;
        if constexpr (M3) acc.p3[i][j][0] = acc.p3[i][j][1] = 0.0;
      }
  }
  __device__ static __forceinline__ void compute(const T* __restrict__ sA, const T* __restrict__ sB, Acc& acc,
                                                 int kvalid, int ncols) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int wm = warp % WARPS_M, wn = warp / WARPS_M;
    const int frow = lane >> 2, fk = lane & 3;
    const T* pa = sA + ((wm * FM * 8 + frow) * 4 + fk);
    const T* pb = sB + ((wn * FN * 8 + frow) * 4 + fk);
#pragma unroll
    for (int k4 = 0; k4 < KT / 4; ++k4) {
      if (k4 * 4 >= kvalid) break;  // uniform: trailing k of a ragged step are zero
      T a[FM], b[FN];
#pragma unroll
      for (int i = 0; i < FM; ++i) a[i] = pa[(k4 * MT + i * 8) * 4];
#pragma unroll
      for (int j = 0; j < FN; ++j) b[j] = pb[(k4 * NT + j * 8) * 4];
      if constexpr (M3) {
        // three passes of FM*FN independent DMMAs
        double as[FM], bs[FN];
#pragma unroll
        for (int i = 0; i < FM; ++i) as[i] = a[i].x + a[i].y;
#pragma unroll
        for (int j = 0; j < FN; ++j) bs[j] = b[j].x + b[j].y;
#pragma unroll
        for (int i = 0; i < FM; ++i)
#pragma unroll
          for (int j = 0; j < FN; ++j) dmma8x8x4(acc.re[i][j][0], acc.re[i][j][1], a[i].x, b[j].x);
#pragma unroll
        for (int i = 0; i < FM; ++i)
#pragma unroll
          for (int j = 0; j < FN; ++j) dmma8x8x4(acc.im[i][j][0], acc.im[i][j][1], a[i].y, b[j].y);
#pragma unroll
        for (int i = 0; i < FM; ++i)
#pragma unroll
          for (int j = 0; j < FN; ++j) dmma8x8x4(acc.p3[i][j][0], acc.p3[i][j][1], as[i], bs[j]);
      } else if constexpr (CPLX) {
        // four passes of FM*FN independent DMMAs: the two updates of one
        // accumulator are FM*FN*2 instructions apart, so the tensor pipe never
        // waits on its own result
        double nai[FM];
#pragma unroll
        for (int i = 0; i < FM; ++i) nai[i] = -a[i].y;
#pragma unroll
        for (int i = 0; i < FM; ++i)
#pragma unroll
          for (int j = 0; j < FN; ++j) dmma8x8x4(acc.re[i][j][0], acc.re[i][j][1], a[i].x, b[j].x);
#pragma unroll
        for (int i = 0; i < FM; ++i)
#pragma unroll
          for (int j = 0; j < FN; ++j) dmma8x8x4(acc.im[i][j][0], acc.im[i][j][1], a[i].x, b[j].y);
#pragma unroll
        for (int i = 0; i < FM; ++i)
#pragma unroll
          for (int j = 0; j < FN; ++j) dmma8x8x4(acc.re[i][j][0], acc.re[i][j][1], nai[i], b[j].y);
#pragma unroll
        for (int i = 0; i < FM; ++i)
#pragma unroll
          for (int j = 0; j < FN; ++j) dmma8x8x4(acc.im[i][j][0], acc.im[i][j][1], a[i].y, b[j].x);
      } else {
#pragma unroll
        for (int i = 0; i < FM; ++i)
#pragma unroll
          for (int j = 0; j < FN; ++j) dmma8x8x4(acc.re[i][j][0], acc.re[i][j][1], a[i], b[j]);
      }
    }
  }
  // once per tile, before the epilogue passes: 3M turns (P1, P2, P3) into (re, im)
  __device__ static __forceinline__ void finalize(Acc& acc) {
    if constexpr (M3) {
#pragma unroll
      for (int i = 0; i < FM; ++i)
#pragma unroll
        for (int j = 0; j < FN; ++j)
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const double p1 = acc.re[i][j][e], p2 = acc.im[i][j][e];
            acc.re[i][j][e] = p1 - p2;
            acc.im[i][j][e] = acc.p3[i][j][e] - p1 - p2;
          }
    }
  }
  template <typename F, typename F2>
  __device__ static __forceinline__ void epilogue(Acc& acc, T* scratch, F&& store, F2&& store_pair, bool pair_ok,
                                                  int ncols) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int wm = warp % WARPS_M, wn = warp / WARPS_M;
    const int frow = lane >> 2, fc = (lane & 3) * 2;
#pragma unroll
    for (int i = 0; i < FM; ++i)
#pragma unroll
      for (int j = 0; j < FN; ++j) {
        const int r = (wm * FM + i) * 8 + frow;
        const int c = (wn * FN + j) * 8 + fc;
        if constexpr (CPLX) {
          // a lane owns two adjacent columns of the fragment: one 256-bit store
          if (pair_ok) {
            store_pair(r, c, make_double2(acc.re[i][j][0], acc.im[i][j][0]),
                       make_double2(acc.re[i][j][1], acc.im[i][j][1]));
          } else {
            store(r, c, make_double2(acc.re[i][j][0], acc.im[i][j][0]));
            store(r, c + 1, make_double2(acc.re[i][j][1], acc.im[i][j][1]));
          }
        } else {
          store(r, c, acc.re[i][j][0]);
          store(r, c + 1, acc.re[i][j][1]);
        }
      }
  }
};

#include "tf32_policy.cuh"
#include "rowstream.cuh"
#include "dmmastream.cuh"
#include "dotstream.cuh"
#include "tc05_policy.cuh"
#include "gett_ws.cuh"
#include "tc05_kernel.cuh"

// ------------------------------------------------------------------ single operand
// out[o] = sum_s X[off_o(o) + off_s(s)]  (diag via summed strides; contract.py:332-361)
template <typename T>
__global__ void single_kernel(const int64_t* __restrict__ D, const T* __restrict__ X, T* __restrict__ out) {
  const int n_o = (int)D[S_NO], n_s = (int)D[S_NS];
  const long long out_elems = D[S_OUT_ELEMS], sum_elems = D[S_SUM_ELEMS];
  const bool accumulate = (D[S_FLAGS] & 1) != 0;
  for (long long o = blockIdx.x * (long long)blockDim.x + threadIdx.x; o < out_elems;
       o += (long long)gridDim.x * blockDim.x) {
    long long e = o, xo = 0, oo = 0;
    for (int d = 0; d < n_o; ++d) {
      const int64_t* L = D + OFF_SO + d * 3;
      long long dig = e % L[0];
      e /= L[0];
      xo += dig * L[1];
      oo += dig * L[2];
    }
    T acc = zero_of<T>();
    for (long long s = 0; s < sum_elems; ++s) {
      long long e2 = s, xs = 0;
      for (int d = 0; d < n_s; ++d) {
        const int64_t* L = D + OFF_SS + d * 2;
        xs += (e2 % L[0]) * L[1];
        e2 /= L[0];
      }
      acc = add_of(acc, X[xo + xs]);
    }
    out[oo] = accumulate ? add_of(out[oo], acc) : acc;
  }
}

// the same with a block per output element: few outputs, a long summed range (a full trace or a
// reduction of a large preprocessing operand) -- the thread-per-output kernel above would walk the
// summed range serially
template <typename T>
__global__ void __launch_bounds__(256) single_reduce_kernel(const int64_t* __restrict__ D, const T* __restrict__ X,
                                                            T* __restrict__ out) {
  __shared__ T s_part[8];
  const int n_o = (int)D[S_NO], n_s = (int)D[S_NS];
  const long long out_elems = D[S_OUT_ELEMS], sum_elems = D[S_SUM_ELEMS];
  const bool accumulate = (D[S_FLAGS] & 1) != 0;
  for (long long o = blockIdx.x; o < out_elems; o += gridDim.x) {
    long long e = o, xo = 0, oo = 0;
    for (int d = 0; d < n_o; ++d) {
      const int64_t* L = D + OFF_SO + d * 3;
      const long long dig = e % L[0];
      e /= L[0];
      xo += dig * L[1];
      oo += dig * L[2];
    }
    T acc = zero_of<T>();
    for (long long s = threadIdx.x; s < sum_elems; s += blockDim.x) {
      long long e2 = s, xs = 0;
      for (int d = 0; d < n_s; ++d) {
        const int64_t* L = D + OFF_SS + d * 2;
        xs += (e2 % L[0]) * L[1];
        e2 /= L[0];
      }
      acc = add_of(acc, X[xo + xs]);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) acc = add_of(acc, shfl_down_of(acc, d));
    if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
      T v = s_part[0];
      for (int w = 1; w < 8; ++w) v = add_of(v, s_part[w]);
      out[oo] = accumulate ? add_of(out[oo], v) : v;
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------ strip_exponent helpers
// contract.py:816-829: factor = max|p|; exponent += log10(factor); p /= factor  (fused into the
// kernels' epilogues, StripCtx above; absmax_kernel serves the nodes that add partial sums atomically)
__device__ __forceinline__ double abs_of(float v) { return fabs((double)v); }
__device__ __forceinline__ double abs_of(double v) { return fabs(v); }
__device__ __forceinline__ double abs_of(float2 v) { return hypot((double)v.x, (double)v.y); }
__device__ __forceinline__ double abs_of(double2 v) { return hypot(v.x, v.y); }

template <typename T>
__global__ void absmax_kernel(const T* __restrict__ p, long long n, unsigned long long* __restrict__ slot) {
  double m = 0.0;
  bool nan = false;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    double a = abs_of(p[i]);
    if (a != a) nan = true;
    m = fmax(m, a);
  }
  if (nan) m = __longlong_as_double(0x7ff8000000000000LL);
  // non-negative doubles (and +NaN) order like their bit patterns
  unsigned long long bits = (unsigned long long)__double_as_longlong(m);
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    unsigned long long o = __shfl_xor_sync(0xffffffffu, bits, d);
    bits = o > bits ? o : bits;
  }
  if ((threadIdx.x & 31) == 0) atomicMax(slot, bits);
}

__device__ __forceinline__ float mulr_of(float v, double s) { return (float)(v * s); }
__device__ __forceinline__ double mulr_of(double v, double s) { return v * s; }
__device__ __forceinline__ float2 mulr_of(float2 v, double s) { return make_float2((float)(v.x * s), (float)(v.y * s)); }
__device__ __forceinline__ double2 mulr_of(double2 v, double s) { return make_double2(v.x * s, v.y * s); }

// Exponent-aware slice accumulation (core.py:163-170):
//   e = max(E, es);  out = out * 10^(E - e) (+ chunk: m * 10^(es - e));  E = e
// Phase 0 rescales the whole output (early-out when the scale is exactly 1),
// phase 1 adds the slice mantissa into its chunk, phase 2 commits E.
template <typename T>
__global__ void rescale_out_kernel(T* __restrict__ out, long long n, const double* __restrict__ E,
                                   const double* __restrict__ es) {
  const double e = fmax(*E, *es);
  const double so = (*E == e) ? 1.0 : pow(10.0, *E - e);
  if (so == 1.0) return;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = mulr_of(out[i], so);
}
template <typename T>
__global__ void add_chunk_kernel(const int64_t* __restrict__ D, T* __restrict__ out, const T* __restrict__ m,
                                 const double* __restrict__ E, const double* __restrict__ es,
                                 const double* __restrict__ froot) {
  // D: single-operand descriptor mapping the dense slice result onto the chunk
  // froot: the root's own factor max|m| -- the stored root is not normalised yet (lazy scaling)
  const double e = fmax(*E, *es);
  double sn = (*es == e) ? 1.0 : pow(10.0, *es - e);
  if (froot != nullptr) sn = (*froot != 0.0) ? sn / *froot : 0.0;
  const int n_o = (int)D[S_NO];
  const long long n = D[S_OUT_ELEMS];
  for (long long o = blockIdx.x * (long long)blockDim.x + threadIdx.x; o < n; o += (long long)gridDim.x * blockDim.x) {
    long long t = o, xo = 0, oo = 0;
    for (int d = 0; d < n_o; ++d) {
      const int64_t* L = D + OFF_SO + d * 3;
      long long dig = t % L[0];
      t /= L[0];
      xo += dig * L[1];
      oo += dig * L[2];
    }
    out[oo] = add_of(out[oo], mulr_of(m[xo], sn));
  }
}
__global__ void commit_exponent_kernel(double* __restrict__ E, const double* __restrict__ es) {
  *E = fmax(*E, *es);
}
// strip_exponent, small operand pre-scaled: dst = src / (fA fB) over the whole underlying buffer of
// the node's small operand (a few KB on a contraction stem), so that the big kernel's epilogue
// only has to track max|C| -- two multiplies per output element of a 16 GiB result are not free
// on the fp64 pipe the DMMAs run on.
// v * sa * sb with the intermediate kept in double (sa alone may leave the float range)
__device__ __forceinline__ float scale2_of(float v, double sa, double sb) { return (float)((double)v * sa * sb); }
__device__ __forceinline__ double scale2_of(double v, double sa, double sb) { return v * sa * sb; }
__device__ __forceinline__ float2 scale2_of(float2 v, double sa, double sb) {
  return make_float2((float)((double)v.x * sa * sb), (float)((double)v.y * sa * sb));
}
__device__ __forceinline__ double2 scale2_of(double2 v, double sa, double sb) {
  return make_double2(v.x * sa * sb, v.y * sa * sb);
}
template <typename T>
__global__ void scale_copy_kernel(const T* __restrict__ src, T* __restrict__ dst, long long n,
                                  const double* __restrict__ fa, const double* __restrict__ fb) {
  const double a = *fa, b = *fb;
  const double sa = a != 0.0 ? 1.0 / a : 0.0, sb = b != 0.0 ? 1.0 / b : 0.0;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    dst[i] = scale2_of(src[i], sa, sb);
}

// strip_exponent range guard.  An operand of an epilogue-scaled node is stored raw, so its consumer
// accumulates up to fA * fB * K before the epilogue multiplies by 1/(fA fB); the reference's operands
// are normalised (magnitude <= 1) at that point.  A factor outside [lo, hi] would let that product
// leave the range of T, so the operand is divided by its factor in place and the consumer scales by
// 1 instead (*eff).  The exponent still sums log10(f): the factor slot itself is left alone.  In
// range, this is one read of the slot and one store -- no pass over the operand.
__device__ __forceinline__ float div_of(float v, double f) { return (float)((double)v / f); }
__device__ __forceinline__ double div_of(double v, double f) { return v / f; }
__device__ __forceinline__ float2 div_of(float2 v, double f) { return make_float2(div_of(v.x, f), div_of(v.y, f)); }
__device__ __forceinline__ double2 div_of(double2 v, double f) { return make_double2(v.x / f, v.y / f); }
template <typename T>
__global__ void strip_band_kernel(T* __restrict__ x, long long n, const double* __restrict__ f,
                                  double* __restrict__ eff, double lo, double hi) {
  const double v = *f;
  // (0, NaN and inf are passed on unchanged: zero / NaN / overflowed operands stay what they are)
  const bool norm = (v > 0.0 && v < lo) || (v > hi && v <= 1.7976931348623157e308);
  if (blockIdx.x == 0 && threadIdx.x == 0) *eff = norm ? 1.0 : v;
  if (!norm) return;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    x[i] = div_of(x[i], v);
}

// fused strip_exponent bookkeeping: factor slots of the listed tensors back to zero
__global__ void reset_slots_kernel(double* __restrict__ f, const int* __restrict__ list, int n) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) f[list[i]] = 0.0;
}
// exponent = base + sum_i log10(factor[list[i]])   (-inf as soon as one factor is zero; one block)
__global__ void sum_log_kernel(const double* __restrict__ f, const int* __restrict__ list, int n,
                               double* __restrict__ exponent, const double* __restrict__ base) {
  __shared__ double part[8];
  double acc = 0.0;
  for (int i = threadIdx.x; i < n; i += blockDim.x) {
    const double v = f[list[i]];
    acc += (v != 0.0) ? log10(v) : -CUDART_INF;
  }
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, d);
  if ((threadIdx.x & 31) == 0) part[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = base ? *base : 0.0;
    for (int w = 0; w < (int)(blockDim.x >> 5); ++w) t += part[w];
    *exponent = t;
  }
}
__global__ void set_double_kernel(double* p, double v) { *p = v; }

}  // namespace ctgb
