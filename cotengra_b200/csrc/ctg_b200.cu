// ctg_b200.cu -- C-ABI implementation (include/ctg_b200.h): kernel dispatch, the
// per-slice node loop and the slice loop, all on the device stream.
//
// Reference path replaced:
//   Contractor.__call__ node loop ........ cotengra/contract.py:791-832
//   ContractionTree.contract slice loop .. cotengra/core.py:4015-4030
//   slice_key / slice_arrays ............. cotengra/core.py:3775-3819
//   gather_slices (sum and stack) ........ cotengra/core.py:3825-3882
//   contract_mpi round robin ............. cotengra/core.py:4070
#include <cuda.h>  // CUtensorMap (types only: the encoder is fetched through cudaGetDriverEntryPoint)
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <atomic>
#include <type_traits>
#include <string>
#include <vector>

#include "../../include/ctg_b200.h"
#include "gett_desc.h"
#include "gett_kernels.cuh"
#include "probe.cuh"

using namespace ctgb;

namespace {

thread_local std::string g_err;
std::atomic<int64_t> g_launches{0};

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
#define CUDA_TRY(expr)                                                                       \
  do {                                                                                       \
    cudaError_t _e = (expr);                                                                 \
    if (_e != cudaSuccess)                                                                   \
      return fail(CTGB_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(_e));          \
  } while (0)

struct DevInfo {
  bool ok = false;
  int sms = 0, major = 0, minor = 0;
  size_t smem_optin = 0;
};
DevInfo& devinfo() {
  static thread_local DevInfo d;
  static thread_local int cached_dev = -1;
  int dev = -1;
  if (cudaGetDevice(&dev) != cudaSuccess) {
    d.ok = false;
    return d;
  }
  if (dev != cached_dev) {
    cudaDeviceProp p;
    if (cudaGetDeviceProperties(&p, dev) == cudaSuccess) {
      d.ok = true;
      d.sms = p.multiProcessorCount;
      d.major = p.major;
      d.minor = p.minor;
      d.smem_optin = p.sharedMemPerBlockOptin;
      cached_dev = dev;
      // the tcgen05 launches take their B' scratch from the stream-ordered pool: keep freed
      // blocks cached across synchronisation points instead of returning them to the driver
      cudaMemPool_t pool;
      if (cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
        uint64_t keep = UINT64_MAX;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
      }
    } else {
      d.ok = false;
    }
  }
  return d;
}

size_t elem_size(int dtype) {
  switch (dtype) {
    case CTGB_F32: return 4;
    case CTGB_F64: return 8;
    case CTGB_C64: return 8;
    case CTGB_C128: return 16;
  }
  return 0;
}

// ---------------------------------------------------------------- dispatch
template <typename T, class P>
int launch_gett_policy(const int64_t* h, const int64_t* d, const void* A, const void* B, void* C, cudaStream_t st) {
  DevInfo& di = devinfo();
  if (!di.ok) return fail(CTGB_E_CUDA, "no CUDA device");
  constexpr size_t smem = GettSmem<P>::template bytes<T>();
  if (smem > di.smem_optin) return fail(CTGB_E_CUDA, "kernel variant needs more shared memory than the device offers");
  static thread_local int attr_dev = -1;
  int dev;
  cudaGetDevice(&dev);
  if (attr_dev != dev) {
    CUDA_TRY(cudaFuncSetAttribute(gett_kernel<T, P>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    attr_dev = dev;
  }
  if constexpr (P::CONSUMER_REGS > 0) {
    // setmaxnreg safety: the re-partitioned registers must fit the pool the CTA
    // was launched with (regs/thread chosen by ptxas x block size), otherwise
    // setmaxnreg.inc would block forever
    static thread_local int checked = 0;
    if (!checked) {
      cudaFuncAttributes fa;
      CUDA_TRY(cudaFuncGetAttributes(&fa, gett_kernel<T, P>));
      const long pool = (long)fa.numRegs * (P::THREADS + PRODUCER_THREADS);
      const long want = (long)P::CONSUMER_REGS * P::THREADS + (long)P::PRODUCER_REGS * PRODUCER_THREADS;
      if (want > pool) return fail(CTGB_E_CUDA, "setmaxnreg budget exceeds the launch register pool");
      checked = 1;
    }
  }
  static thread_local int occ = 0;
  if (occ == 0) {
    CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, gett_kernel<T, P>, P::THREADS + PRODUCER_THREADS, smem));
    if (occ < 1) occ = 1;
  }
  const uint64_t work = (uint64_t)h[W_TILES_M] * (uint64_t)h[W_TILES_N] * (uint64_t)h[W_TILES_B] * (uint64_t)h[W_SPLITK];
  if (work == 0) return CTGB_OK;
  if (work >= (1ull << 31)) return fail(CTGB_E_VALUE, "too many tiles for one launch");
  uint64_t grid = (uint64_t)di.sms * occ;
  if (grid > work) grid = work;
  if (h[W_SPLITK] > 1 && !(h[W_FLAGS] & 1)) {
    if (h[W_CELEMS] <= 0) return fail(CTGB_E_VALUE, "split-K into a strided C needs accumulate");
    CUDA_TRY(cudaMemsetAsync(C, 0, (size_t)h[W_CELEMS] * sizeof(T), st));
  }
  gett_kernel<T, P><<<(unsigned)grid, P::THREADS + PRODUCER_THREADS, smem, st>>>(d, (const T*)A, (const T*)B, (T*)C);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  CUDA_TRY(cudaGetLastError());
  return CTGB_OK;
}

template <typename T>
int launch_rowstream(const int64_t* h, const int64_t* d, const void* A, const void* B, void* C, cudaStream_t st) {
  DevInfo& di = devinfo();
  if (!di.ok) return fail(CTGB_E_CUDA, "no CUDA device");
  const int N = (int)h[W_NTA], K = (int)h[W_KTA];
  if (N > 8 || K > 8 || h[W_TILES_N] != 1 || h[W_TILES_B] != 1 || h[W_STEPS_K] != 1 || h[W_SPLITK] != 1 ||
      h[W_PGM] >= 0 && (h[W_MFULL] % h[W_MTEXT]) != 0 || h[W_PGN] >= 0 || h[W_PGK] >= 0)
    return fail(CTGB_E_VALUE, "descriptor does not fit the row-stream kernel");
  const unsigned long long M = (unsigned long long)h[W_MTA] * (unsigned long long)h[W_TILES_M];
  if (M >= (1ull << 32)) return fail(CTGB_E_VALUE, "too many rows for the row-stream kernel");
  unsigned long long blocks = (M + 255) / 256;
  const unsigned long long cap = (unsigned long long)di.sms * 8;
  if (blocks > cap) blocks = cap;
  if (blocks == 0) return CTGB_OK;
  const T* a = (const T*)A;
  const T* b = (const T*)B;
  T* c = (T*)C;
  const bool strip = h[W_SCALE_A] != 0 || h[W_FACTOR_C] != 0;  // fused strip_exponent: separate instantiations
  if (N <= 4 && K <= 4) {
    if (strip) rowstream_kernel<T, 4, 4, true, true><<<(unsigned)blocks, 256, 0, st>>>(d, a, b, c);
    else rowstream_kernel<T, 4, 4, true><<<(unsigned)blocks, 256, 0, st>>>(d, a, b, c);
  } else if (N <= 2) {  // (B from shared memory: in registers it costs 154 registers = one block / SM)
    if (strip) rowstream_kernel<T, 2, 8, sizeof(T) < 16, true><<<(unsigned)blocks, 256, 0, st>>>(d, a, b, c);
    else rowstream_kernel<T, 2, 8, sizeof(T) < 16><<<(unsigned)blocks, 256, 0, st>>>(d, a, b, c);
  } else {
    if (strip) rowstream_kernel<T, 8, 8, false, true><<<(unsigned)blocks, 256, 0, st>>>(d, a, b, c);
    else rowstream_kernel<T, 8, 8, false><<<(unsigned)blocks, 256, 0, st>>>(d, a, b, c);
  }
  g_launches.fetch_add(1, std::memory_order_relaxed);
  CUDA_TRY(cudaGetLastError());
  return CTGB_OK;
}

template <typename T>
int launch_rowstream_longk(const int64_t* h, const int64_t* d, const void* A, const void* B, void* C, cudaStream_t st) {
  DevInfo& di = devinfo();
  if (!di.ok) return fail(CTGB_E_CUDA, "no CUDA device");
  if constexpr (sizeof(T) > 8) {
    return fail(CTGB_E_VALUE, "the long-k row stream takes 8-byte and narrower element types");
  } else {
    const int N = (int)h[W_NTA], K = (int)h[W_KTA];
    if (N > RSK_NMAX || K > RSK_KMAX || h[W_TILES_N] != 1 || h[W_TILES_B] != 1 || h[W_STEPS_K] != 1 ||
        h[W_SPLITK] != 1 || h[W_PGM] >= 0 && (h[W_MFULL] % h[W_MTEXT]) != 0 || h[W_PGN] >= 0 || h[W_PGK] >= 0)
      return fail(CTGB_E_VALUE, "descriptor does not fit the long-k row-stream kernel");
    // offset(k) must decompose as chunk_base[k / 8] + in_chunk[k % 8]
    auto koff = [&](long long e) {
      long long o = 0;
      for (int i = 0; i < (int)h[W_NTK]; ++i) {
        o += (e % h[OFF_TK + 3 * i]) * h[OFF_TK + 3 * i + 1];
        e /= h[OFF_TK + 3 * i];
      }
      return o;
    };
    for (long long e = 0; e < K; ++e)
      if (koff(e) != koff(e - e % 8) + koff(e % 8)) return fail(CTGB_E_VALUE, "k offsets do not split into chunks of 8");
    const unsigned long long M = (unsigned long long)h[W_MTA] * (unsigned long long)h[W_TILES_M];
    if (M >= (1ull << 32)) return fail(CTGB_E_VALUE, "too many rows for the row-stream kernel");
    unsigned long long blocks = (M + 511) / 512;
    const unsigned long long cap = (unsigned long long)di.sms * 6;
    if (blocks > cap) blocks = cap;
    if (blocks == 0) return CTGB_OK;
    if (h[W_SCALE_A] != 0 || h[W_FACTOR_C] != 0)
      rowstream_longk_kernel<T, true><<<(unsigned)blocks, 256, 0, st>>>(d, (const T*)A, (const T*)B, (T*)C);
    else
      rowstream_longk_kernel<T><<<(unsigned)blocks, 256, 0, st>>>(d, (const T*)A, (const T*)B, (T*)C);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    CUDA_TRY(cudaGetLastError());
    return CTGB_OK;
  }
}

template <typename T>
int launch_dotstream(const int64_t* h, const int64_t* d, const void* A, const void* B, void* C, cudaStream_t st) {
  DevInfo& di = devinfo();
  if (!di.ok) return fail(CTGB_E_CUDA, "no CUDA device");
  const bool mn = h[W_VARIANT] == VAR_DOTSTREAM4;
  const int lim = mn ? DOT4_MN : 1, kt = mn ? dot4_kt<T>() : DOT_KT;
  if (h[W_MTA] > lim || h[W_NTA] > lim || h[W_TILES_M] != 1 || h[W_TILES_N] != 1 || h[W_TILES_B] != 1 ||
      h[W_KTA] > kt || h[W_NGK] > 64 || h[W_STEPS_K] >= (1ll << 31) || h[W_PGM] >= 0 || h[W_PGN] >= 0 ||
      (h[W_PGK] >= 0 && (h[W_KFULL] % h[W_KTEXT]) != 0))
    return fail(CTGB_E_VALUE, "descriptor does not fit the dot-stream kernel");
  if (h[W_STEPS_K] == 0) return CTGB_OK;
  if (!(h[W_FLAGS] & 1)) {
    // block partial sums are added atomically: a dense result is zeroed first
    const long long celems = h[W_MTA] * h[W_NTA];
    if (celems > 1 && h[W_CELEMS] != celems) return fail(CTGB_E_VALUE, "dot-stream into a strided C needs accumulate");
    CUDA_TRY(cudaMemsetAsync(C, 0, (size_t)celems * sizeof(T), st));
  }
  unsigned long long blocks = (unsigned long long)h[W_STEPS_K];
  // one wave: two resident blocks per SM (one for the 16-accumulator variant)
  const unsigned long long cap = (unsigned long long)di.sms * (mn ? 1 : 2);
  if (blocks > cap) blocks = cap;
  if (mn)
    dotstream_kernel<T, DOT4_MN, DOT4_MN, dot4_u<T>()><<<(unsigned)blocks, DOT_THREADS, 0, st>>>(d, (const T*)A, (const T*)B, (T*)C);
  else
    dotstream_kernel<T, 1, 1, DOT_U><<<(unsigned)blocks, DOT_THREADS, 0, st>>>(d, (const T*)A, (const T*)B, (T*)C);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  CUDA_TRY(cudaGetLastError());
  return CTGB_OK;
}

int launch_dmmastream(const int64_t* h, const int64_t* d, const void* A, const void* B, void* C, cudaStream_t st) {
  DevInfo& di = devinfo();
  if (!di.ok) return fail(CTGB_E_CUDA, "no CUDA device");
  const int N = (int)h[W_NTA], K = (int)h[W_KTA];
  if (h[W_DTYPE] != CTGB_C128 || N > 32 || K > DS_KMAX || h[W_TILES_N] != 1 || h[W_TILES_B] != 1 ||
      h[W_STEPS_K] != 1 || h[W_SPLITK] != 1 || h[W_PGM] >= 0 && (h[W_MFULL] % h[W_MTEXT]) != 0 || h[W_PGN] >= 0 ||
      h[W_PGK] >= 0)
    return fail(CTGB_E_VALUE, "descriptor does not fit the DMMA stream kernel");
  const unsigned long long M = (unsigned long long)h[W_MTA] * (unsigned long long)h[W_TILES_M];
  if (M >= (1ull << 32)) return fail(CTGB_E_VALUE, "too many rows for the DMMA stream kernel");
  if (M == 0) return CTGB_OK;
  unsigned long long blocks = (M + 127) / 128;  // 4 warps x 32 rows per block and pass
  const unsigned long long cap = (unsigned long long)di.sms * 12;
  if (blocks > cap) blocks = cap;
  const bool strip = h[W_SCALE_A] != 0 || h[W_FACTOR_C] != 0;  // fused strip_exponent: separate instantiations
  const double2 *a = (const double2*)A, *b = (const double2*)B;
  if (N <= 8) {
    if (strip) dmmastream_kernel<1, true><<<(unsigned)blocks, 128, 0, st>>>(d, a, b, (double2*)C);
    else dmmastream_kernel<1><<<(unsigned)blocks, 128, 0, st>>>(d, a, b, (double2*)C);
  } else if (N <= 16) {
    if (strip) dmmastream_kernel<2, true><<<(unsigned)blocks, 128, 0, st>>>(d, a, b, (double2*)C);
    else dmmastream_kernel<2><<<(unsigned)blocks, 128, 0, st>>>(d, a, b, (double2*)C);
  } else {
    if (strip) dmmastream_kernel<4, true><<<(unsigned)blocks, 128, 0, st>>>(d, a, b, (double2*)C);
    else dmmastream_kernel<4><<<(unsigned)blocks, 128, 0, st>>>(d, a, b, (double2*)C);
  }
  g_launches.fetch_add(1, std::memory_order_relaxed);
  CUDA_TRY(cudaGetLastError());
  return CTGB_OK;
}

std::atomic<int64_t> g_tmap_launches{0};

// Tensor map for the A tile of the tcgen05 kernel.  The tile is described in A's memory order by
// the descriptor's load list (ext, stride), smallest stride first; adjacent entries that continue
// each other coalesce into box dims.  If at most four box dims remain, the innermost is contiguous
// and everything is 16-byte granular, ONE cp.async.bulk.tensor fetches the tile: dims 0..n-1 are
// the box (coordinates 0), and one more dim of stride 16 bytes carries the tile's base offset as
// its coordinate (tensor-map strides need not nest).  Returns the rank (2..5) or 0.
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
int tc05_make_tensor_map(const int64_t* h, const void* A, CUtensorMap* tm) {
  static EncodeTiledFn encode = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      encode = (EncodeTiledFn)fn;
    else
      cudaGetLastError();
  }
  if (!encode || ((uintptr_t)A & 15u)) return 0;
  struct Dim { uint64_t ext, stride; } box[8];
  int nb = 0;
  const int n_lda = (int)h[W_NLDA];
  for (int i = 0; i < n_lda; ++i) {
    const uint64_t ext = (uint64_t)h[OFF_LDA + 4 * i], st = (uint64_t)h[OFF_LDA + 4 * i + 1];
    if (h[OFF_LDA + 4 * i + 1] <= 0) return 0;
    if (nb && st == box[nb - 1].stride * box[nb - 1].ext) {
      box[nb - 1].ext *= ext;
    } else {
      if (nb == 4) return 0;
      box[nb].ext = ext;
      box[nb].stride = st;
      ++nb;
    }
  }
  // a box dim holds at most 256 elements: split longer (contiguous) ones
  for (int i = 0; i < nb; ++i) {
    while (box[i].ext > 256) {
      uint64_t f = 256;
      while (f > 1 && box[i].ext % f) --f;
      if (f < 2 || nb == 4) return 0;
      for (int j = nb; j > i + 1; --j) box[j] = box[j - 1];
      box[i + 1].ext = box[i].ext / f;
      box[i + 1].stride = box[i].stride * f;
      box[i].ext = f;
      ++nb;
    }
  }
  if (nb == 0 || box[0].stride != 1 || (box[0].ext & 1)) return 0;
  uint64_t prod = 1;
  for (int i = 0; i < nb; ++i) {
    if (box[i].ext > 256 || (i && (box[i].stride & 1))) return 0;
    prod *= box[i].ext;
  }
  if (prod != (uint64_t)(h[W_MTA] * h[W_KTA])) return 0;
  // base offsets of the tiles: sums of grid-dim digits times even strides, below 2^32 elements
  uint64_t reach = 0;
  auto grid = [&](int off, int n, int width, int col) -> bool {
    for (int i = 0; i < n; ++i) {
      const int64_t e = h[off + i * width], st = h[off + i * width + col];
      if (st < 0 || (st & 1)) return false;
      reach += (uint64_t)(e - 1) * (uint64_t)st;
    }
    return true;
  };
  if (!grid(OFF_GM, (int)h[W_NGM], 4, 2) || !grid(OFF_GK, (int)h[W_NGK], 4, 2) || !grid(OFF_GB, (int)h[W_NGB], 5, 2))
    return 0;
  if (reach >= (1ull << 32)) return 0;
  cuuint64_t gdim[5], gstr[4];
  cuuint32_t bdim[5], estr[5];
  for (int i = 0; i < nb; ++i) {
    gdim[i] = box[i].ext;
    bdim[i] = (cuuint32_t)box[i].ext;
    estr[i] = 1;
    if (i) gstr[i - 1] = box[i].stride * 8;
  }
  gdim[nb] = 1ull << 31;  // offset dim: coordinate = base offset in 16-byte units
  bdim[nb] = 1;
  estr[nb] = 1;
  gstr[nb - 1] = 16;
  const CUresult rc = encode(tm, CU_TENSOR_MAP_DATA_TYPE_UINT64, (cuuint32_t)(nb + 1), const_cast<void*>(A), gdim, gstr,
                             bdim, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE,
                             CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return rc == CUDA_SUCCESS ? nb + 1 : 0;
}

// complex64 on tcgen05: prepare B' (hi/lo, tile order) once, then the warp-specialised kernel
template <int NT>
int launch_tc05(const int64_t* h, const int64_t* d, const void* A, const void* B, void* C, cudaStream_t st) {
  using Cfg = Tc05Cfg<NT>;
  DevInfo& di = devinfo();
  if (!di.ok) return fail(CTGB_E_CUDA, "no CUDA device");
  auto exact = [&](int pg, int full, int text) { return h[pg] < 0 || (h[full] % h[text]) == 0; };
  // every tile has the same shape: the full 128 x NT x 16, or exact divisors of the index extents
  // (MTa <= 128 rows, NTa <= NT columns, KTa a multiple of 4 up to 16)
  if (h[W_DTYPE] != CTGB_C64 || h[W_MTA] < 1 || h[W_MTA] > 128 || h[W_NTA] < 1 || h[W_NTA] > NT || h[W_KTA] < 4 ||
      h[W_KTA] > 16 || (h[W_KTA] & 3) ||
      !exact(W_PGM, W_MFULL, W_MTEXT) || !exact(W_PGN, W_NFULL, W_NTEXT) || !exact(W_PGK, W_KFULL, W_KTEXT) ||
      h[W_STEPS_K] > TC05_KTAB || h[W_LBOPAD] < 0 || h[W_LBOPAD] > 4 ||
      ((h[W_FLAGS] & 64) && (h[W_RUNA] < 16 || (h[W_MTA] * h[W_KTA]) % h[W_RUNA] != 0)))
    return fail(CTGB_E_VALUE, "descriptor does not fit the tcgen05 kernel");
  const uint64_t work = (uint64_t)h[W_TILES_M] * (uint64_t)h[W_TILES_N] * (uint64_t)h[W_TILES_B] * (uint64_t)h[W_SPLITK];
  if (work == 0) return CTGB_OK;
  if (work >= (1ull << 31)) return fail(CTGB_E_VALUE, "too many tiles for one launch");
  static thread_local int attr_dev = -1;
  int dev;
  cudaGetDevice(&dev);
  if (attr_dev != dev) {
    CUDA_TRY(cudaFuncSetAttribute(tc05_kernel<NT, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)di.smem_optin - 1024));
    CUDA_TRY(cudaFuncSetAttribute(tc05_kernel<NT, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)di.smem_optin - 1024));
    attr_dev = dev;
  }
  // ring depths: B' resident (one slot per k-step) when this CTA's B' tiles never change and
  // still leave room for >= 3 A stages; otherwise a 3-slot B' ring.  A gets the rest.
  const long long pool = (long long)di.smem_optin - 1024 /* static + slack */ - (long long)Cfg::fixed_bytes();
  const long long steps_k = h[W_STEPS_K], tiles_n = h[W_TILES_N];
  uint64_t grid = (uint64_t)di.sms;
  int b_stat = 0;
  long long nb = 3;
  if (h[W_TILES_B] == 1 && h[W_SPLITK] == 1 && steps_k <= Cfg::NB_MAX && tiles_n <= (long long)di.sms &&
      pool - steps_k * Cfg::PAIR_BYTES >= 3ll * Cfg::A_TILE * 8) {
    b_stat = 1;
    nb = steps_k;
    grid = (grid / (uint64_t)tiles_n) * (uint64_t)tiles_n;  // t % tiles_n is the same for every work item of a CTA
  }
  long long sa = (pool - nb * Cfg::PAIR_BYTES) / ((long long)Cfg::A_TILE * 8);
  if (sa > Cfg::SA_MAX) sa = Cfg::SA_MAX;
  if (sa < 2) return fail(CTGB_E_CUDA, "tcgen05 kernel needs more shared memory than the device offers");
  if (grid > work) {
    grid = work;
    if (b_stat && grid % (uint64_t)tiles_n != 0) b_stat = 0, nb = nb < 3 ? 3 : nb;  // tiny launch: plain ring
  }
  const size_t smem = Cfg::smem_bytes((int)sa, (int)nb);
  if (smem + 1024 > di.smem_optin)
    return fail(CTGB_E_CUDA, "tcgen05 kernel needs more shared memory than the device offers");

  const unsigned long long tiles = (unsigned long long)h[W_TILES_B] * h[W_TILES_N] * h[W_STEPS_K];
  const size_t bytes = (size_t)tiles * Cfg::PAIR_BYTES;
  float* Bp = nullptr;
  CUDA_TRY(cudaMallocAsync((void**)&Bp, bytes, st));
  const unsigned long long total = tiles * Cfg::TILE_FLOATS;
  unsigned long long blocks = (total + 255) / 256;
  if (blocks > (unsigned long long)di.sms * 8) blocks = (unsigned long long)di.sms * 8;
  bprime_kernel<NT><<<(unsigned)blocks, 256, 0, st>>>(d, (const float2*)B, Bp);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  if (h[W_SPLITK] > 1 && !(h[W_FLAGS] & 1)) {
    if (h[W_CELEMS] <= 0) {
      cudaFreeAsync(Bp, st);
      return fail(CTGB_E_VALUE, "split-K into a strided C needs accumulate");
    }
    CUDA_TRY(cudaMemsetAsync(C, 0, (size_t)h[W_CELEMS] * sizeof(float2), st));
  }
  CUtensorMap tm;
  memset(&tm, 0, sizeof(tm));
  // (CTGB_NO_TENSOR_MAP=1 is a measurement knob: bulk-copy / gather staging only)
  static const bool tm_off = getenv("CTGB_NO_TENSOR_MAP") != nullptr;
  const int tm_rank = tm_off ? 0 : tc05_make_tensor_map(h, A, &tm);
  if (tm_rank) g_tmap_launches.fetch_add(1, std::memory_order_relaxed);
  // the lean epilogue: 32-byte quads of a dense, aligned C, no accumulation (see tc05_kernel.cuh)
  const bool lean = (h[W_FLAGS] & 16) && !(h[W_FLAGS] & 1) && h[W_SPLITK] == 1 &&
                    (reinterpret_cast<unsigned long long>(C) & 31ull) == 0;
  if (lean)
    tc05_kernel<NT, 0><<<(unsigned)grid, Cfg::THREADS, smem, st>>>(d, (const float2*)A, Bp, (float2*)C, (unsigned)sa,
                                                                    (unsigned)nb, b_stat, tm, tm_rank);
  else
    tc05_kernel<NT, 1><<<(unsigned)grid, Cfg::THREADS, smem, st>>>(d, (const float2*)A, Bp, (float2*)C, (unsigned)sa,
                                                                    (unsigned)nb, b_stat, tm, tm_rank);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  cudaError_t e = cudaGetLastError();
  cudaFreeAsync(Bp, st);
  if (e != cudaSuccess) return fail(CTGB_E_CUDA, cudaGetErrorString(e));
  return CTGB_OK;
}

template <typename T>
int launch_gett_typed(const int64_t* h, const int64_t* d, const void* A, const void* B, void* C, cudaStream_t st) {
  const int variant = (int)h[W_VARIANT];
  if (variant == VAR_ROWSTREAM) return launch_rowstream<T>(h, d, A, B, C, st);
  if (variant == VAR_ROWSTREAM_K) return launch_rowstream_longk<T>(h, d, A, B, C, st);
  if (variant == VAR_DMMASTREAM) return launch_dmmastream(h, d, A, B, C, st);
  if (variant == VAR_DOTSTREAM || variant == VAR_DOTSTREAM4) return launch_dotstream<T>(h, d, A, B, C, st);
  if constexpr (std::is_same<T, float2>::value) {
    if (variant == VAR_TC05_128x64) return launch_tc05<64>(h, d, A, B, C, st);
    if (variant == VAR_TC05_128x32) return launch_tc05<32>(h, d, A, B, C, st);
    if (variant == VAR_TC05_128x16) return launch_tc05<16>(h, d, A, B, C, st);
  }
  switch (variant) {
    case VAR_SIMT_64x64: return launch_gett_policy<T, SimtPolicy<T, 64, 64, 8, 3>>(h, d, A, B, C, st);
    case VAR_KRED: return launch_gett_policy<T, KredPolicy<T, 1, 1, 512, 6>>(h, d, A, B, C, st);
    case VAR_ROW_128x8: return launch_gett_policy<T, RowPolicy<T, 256, 8, 4, 3>>(h, d, A, B, C, st);
    case VAR_ROW_256x4: return launch_gett_policy<T, RowPolicy<T, 256, 4, 4, 3>>(h, d, A, B, C, st);
    default: break;
  }
  if constexpr (sizeof(T) == 16 || (sizeof(T) == 8 && std::is_same<T, double>::value)) {
    switch (variant) {
      case VAR_DMMA_128x64: return launch_gett_policy<T, DmmaPolicy<T, 4, 2, 4, 4, 16, 3>>(h, d, A, B, C, st);
      case VAR_DMMA_64x128: return launch_gett_policy<T, DmmaPolicy<T, 2, 4, 4, 4, 16, 3>>(h, d, A, B, C, st);
      case VAR_DMMA_256x32: return launch_gett_policy<T, DmmaPolicy<T, 8, 1, 4, 4, 8, 4>>(h, d, A, B, C, st);
      case VAR_DMMA_256x16: return launch_gett_policy<T, DmmaPolicy<T, 8, 1, 4, 2, 8, 5>>(h, d, A, B, C, st);
      // (K 16 x 4 stages = 80 KB per CTA: with K 32 x 3 stages -- 122 KB -- only ONE CTA fitted an SM,
      // four consumer warps, tensor pipe 72 % under ncu)
      case VAR_DMMA_32x32: return launch_gett_policy<T, DmmaPolicy<T, 2, 2, 2, 2, 16, 4>>(h, d, A, B, C, st);
      default: break;
    }
  }
  if constexpr (sizeof(T) == 16) {
    switch (variant) {
      case VAR_DMMA3M_128x32: return launch_gett_policy<T, DmmaPolicy<T, 4, 2, 4, 2, 16, 4, true>>(h, d, A, B, C, st);
      case VAR_DMMA3M_256x16: return launch_gett_policy<T, DmmaPolicy<T, 8, 1, 4, 2, 8, 5, true>>(h, d, A, B, C, st);
      default: break;
    }
  }
  if constexpr (std::is_same<T, float>::value || std::is_same<T, float2>::value) {
    // single precision on the tensor pipe: 3xTF32 mma.sync, same tile shapes
    switch (variant) {
      case VAR_DMMA_128x64: return launch_gett_policy<T, Tf32Policy<T, 4, 2, 2, 4, 16, 3>>(h, d, A, B, C, st);
      case VAR_DMMA_64x128: return launch_gett_policy<T, Tf32Policy<T, 2, 4, 2, 4, 16, 3>>(h, d, A, B, C, st);
      case VAR_DMMA_256x32: return launch_gett_policy<T, Tf32Policy<T, 8, 1, 2, 4, 8, 3>>(h, d, A, B, C, st);
      case VAR_DMMA_256x16: return launch_gett_policy<T, Tf32Policy<T, 8, 1, 2, 2, 8, 3>>(h, d, A, B, C, st);
      default: break;
    }
  }
  return fail(CTGB_E_VALUE, "unknown kernel variant for this dtype");
}

int launch_gett(const int64_t* h, const int64_t* d, const void* A, const void* B, void* C, cudaStream_t st) {
  if (h[W_MAGIC] != DESC_MAGIC) return fail(CTGB_E_VALUE, "bad pair descriptor magic");
  switch ((int)h[W_DTYPE]) {
    case CTGB_F32: return launch_gett_typed<float>(h, d, A, B, C, st);
    case CTGB_F64: return launch_gett_typed<double>(h, d, A, B, C, st);
    case CTGB_C64: return launch_gett_typed<float2>(h, d, A, B, C, st);
    case CTGB_C128: return launch_gett_typed<double2>(h, d, A, B, C, st);
  }
  return fail(CTGB_E_VALUE, "bad dtype");
}

template <typename T>
int launch_single_typed(const int64_t* h, const int64_t* d, const void* X, void* out, cudaStream_t st) {
  long long n = h[S_OUT_ELEMS];
  if (n <= 0) return CTGB_OK;
  long long blocks = (n + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  if (h[S_SUM_ELEMS] >= 1024 && n <= 148 * 16) {
    // few outputs over a long summed range: one block per output element
    single_reduce_kernel<T><<<(unsigned)n, 256, 0, st>>>(d, (const T*)X, (T*)out);
  } else {
    single_kernel<T><<<(unsigned)blocks, 256, 0, st>>>(d, (const T*)X, (T*)out);
  }
  g_launches.fetch_add(1, std::memory_order_relaxed);
  CUDA_TRY(cudaGetLastError());
  return CTGB_OK;
}
int launch_single(const int64_t* h, const int64_t* d, const void* X, void* out, cudaStream_t st) {
  if (h[S_MAGIC] != SDESC_MAGIC) return fail(CTGB_E_VALUE, "bad single descriptor magic");
  switch ((int)h[S_DTYPE]) {
    case CTGB_F32: return launch_single_typed<float>(h, d, X, out, st);
    case CTGB_F64: return launch_single_typed<double>(h, d, X, out, st);
    case CTGB_C64: return launch_single_typed<float2>(h, d, X, out, st);
    case CTGB_C128: return launch_single_typed<double2>(h, d, X, out, st);
  }
  return fail(CTGB_E_VALUE, "bad dtype");
}

unsigned flat_grid(long long n) {
  long long b = (n + 255) / 256;
  if (b > 148 * 8) b = 148 * 8;
  if (b < 1) b = 1;
  return (unsigned)b;
}

template <typename T>
int scale_copy_typed(const void* src, void* dst, long long n, const double* fa, const double* fb, cudaStream_t st) {
  scale_copy_kernel<T><<<flat_grid(n), 256, 0, st>>>((const T*)src, (T*)dst, n, fa, fb);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  CUDA_TRY(cudaGetLastError());
  return CTGB_OK;
}
int scale_copy(int dtype, const void* src, void* dst, long long n, const double* fa, const double* fb, cudaStream_t st) {
  switch (dtype) {
    case CTGB_F32: return scale_copy_typed<float>(src, dst, n, fa, fb, st);
    case CTGB_F64: return scale_copy_typed<double>(src, dst, n, fa, fb, st);
    case CTGB_C64: return scale_copy_typed<float2>(src, dst, n, fa, fb, st);
    case CTGB_C128: return scale_copy_typed<double2>(src, dst, n, fa, fb, st);
  }
  return fail(CTGB_E_VALUE, "bad dtype");
}

// max|C| of a node whose own epilogue cannot measure it (split-K / block partial sums)
template <typename T>
int absmax_typed(const void* p, long long n, unsigned long long* slot, cudaStream_t st) {
  absmax_kernel<T><<<flat_grid(n), 256, 0, st>>>((const T*)p, n, slot);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  CUDA_TRY(cudaGetLastError());
  return CTGB_OK;
}
int absmax_into(int dtype, const void* p, long long n, unsigned long long* slot, cudaStream_t st) {
  switch (dtype) {
    case CTGB_F32: return absmax_typed<float>(p, n, slot, st);
    case CTGB_F64: return absmax_typed<double>(p, n, slot, st);
    case CTGB_C64: return absmax_typed<float2>(p, n, slot, st);
    case CTGB_C128: return absmax_typed<double2>(p, n, slot, st);
  }
  return fail(CTGB_E_VALUE, "bad dtype");
}

// the range guard of an operand of an epilogue-scaled node (strip_band_kernel): the band keeps
// fA * fB * K inside the range of the element type for any K below 2^33
template <typename T>
int band_typed(void* p, long long n, const double* f, double* eff, cudaStream_t st) {
  const bool single = sizeof(T) == 4 || std::is_same<T, float2>::value;
  const double lim = single ? 1e12 : 1e120;
  strip_band_kernel<T><<<flat_grid(n), 256, 0, st>>>((T*)p, n, f, eff, 1.0 / lim, lim);
  g_launches.fetch_add(1, std::memory_order_relaxed);
  CUDA_TRY(cudaGetLastError());
  return CTGB_OK;
}
int band_into(int dtype, void* p, long long n, const double* f, double* eff, cudaStream_t st) {
  switch (dtype) {
    case CTGB_F32: return band_typed<float>(p, n, f, eff, st);
    case CTGB_F64: return band_typed<double>(p, n, f, eff, st);
    case CTGB_C64: return band_typed<float2>(p, n, f, eff, st);
    case CTGB_C128: return band_typed<double2>(p, n, f, eff, st);
  }
  return fail(CTGB_E_VALUE, "bad dtype");
}

template <typename T>
int accum_stripped_typed(const int64_t* dchunk, const int64_t* hchunk, void* out, void* chunk, long long out_elems,
                         const void* m, double* E, const double* es, const double* froot, cudaStream_t st) {
  rescale_out_kernel<T><<<flat_grid(out_elems), 256, 0, st>>>((T*)out, out_elems, E, es);
  add_chunk_kernel<T><<<flat_grid(hchunk[S_OUT_ELEMS]), 256, 0, st>>>(dchunk, (T*)chunk, (const T*)m, E, es, froot);
  commit_exponent_kernel<<<1, 1, 0, st>>>(E, es);
  g_launches.fetch_add(3, std::memory_order_relaxed);
  CUDA_TRY(cudaGetLastError());
  return CTGB_OK;
}
int accum_stripped(int dtype, const int64_t* dchunk, const int64_t* hchunk, void* out, void* chunk,
                   long long out_elems, const void* m, double* E, const double* es, const double* froot,
                   cudaStream_t st) {
  switch (dtype) {
    case CTGB_F32: return accum_stripped_typed<float>(dchunk, hchunk, out, chunk, out_elems, m, E, es, froot, st);
    case CTGB_F64: return accum_stripped_typed<double>(dchunk, hchunk, out, chunk, out_elems, m, E, es, froot, st);
    case CTGB_C64: return accum_stripped_typed<float2>(dchunk, hchunk, out, chunk, out_elems, m, E, es, froot, st);
    case CTGB_C128: return accum_stripped_typed<double2>(dchunk, hchunk, out, chunk, out_elems, m, E, es, froot, st);
  }
  return fail(CTGB_E_VALUE, "bad dtype");
}

}  // namespace

// ================================================================== plans
struct ctgb_plan {
  int dtype = 0;
  int n_inputs = 0;
  struct Tensor {
    int kind, input_index;
    int64_t offset, nbytes;
    std::vector<int32_t> slice_pos;
    std::vector<int64_t> slice_stride;
  };
  struct Node {
    int kind, a, b, c, invariant, is_root;
    size_t desc_off;  // word offset into descs
    int64_t c_elems;  // dense elements of the result (strip_exponent)
    int measure_after = 0;  // strip_exponent: max|C| needs its own pass (split-K / block partial sums)
    int prescale_b = 0;     // strip_exponent: the small operand is copied, scaled by 1/(fA fB), first
    int band = 0;           // strip_exponent: C feeds an epilogue-scaled node -- range guard after it
  };
  std::vector<Tensor> tensors;
  std::vector<Node> nodes;
  std::vector<int64_t> descs;  // host copy of every descriptor, concatenated
  int64_t* d_descs = nullptr;
  std::vector<int64_t> radix, project, out_stride;
  int64_t out_elements = 0, workspace_bytes = 0, persistent_bytes = 0;
  int strip_exponent = 0;
  int64_t launches_per_slice = 0;
  // strip_exponent scratch (device): [1] slice exponent, [2] invariant exponent
  double* d_scalars = nullptr;
  // fused strip_exponent: one factor slot per tensor (1.0 for inputs and single-operand results,
  // max|C| for pairwise results) and the slots to reset / sum per pass
  double* d_factors = nullptr;
  // what the consumer divides a range-guarded operand by: its factor, or 1 once it was normalised
  double* d_eff = nullptr;
  char* d_bscale = nullptr;     // scaled copy of the current node's small operand
  size_t bscale_bytes = 0;
  int* d_slot_lists = nullptr;  // [variant slots..., invariant slots...]
  int n_var_slots = 0, n_inv_slots = 0;
  // chunk descriptor for stripped accumulation (host + device), built at create
  std::vector<int64_t> chunk_desc;
  int64_t* d_chunk_desc = nullptr;
  int device = -1;
  // optional per-node timing (bench.py roofline): events around every node launch
  bool profile = false;
  std::vector<cudaEvent_t> ev0, ev1;
  // pinned staging block of ctgb_plan_execute_host (all inputs in one H2D copy)
  char* h_stage = nullptr;
  size_t h_stage_bytes = 0;
};

extern "C" {

int ctgb_abi_version(void) { return CTGB_ABI_VERSION; }
int ctgb_desc_words(void) { return DESC_WORDS; }
int ctgb_single_desc_words(void) { return SDESC_WORDS; }
const char* ctgb_last_error(void) { return g_err.c_str(); }
int64_t ctgb_launch_count(void) { return g_launches.load(); }
int64_t ctgb_tensor_map_launches(void) { return g_tmap_launches.load(); }

int ctgb_device_info(int* sm_count, int* cc_major, int* cc_minor, size_t* smem_optin_bytes) {
  DevInfo& d = devinfo();
  if (!d.ok) return fail(CTGB_E_CUDA, "no CUDA device");
  if (sm_count) *sm_count = d.sms;
  if (cc_major) *cc_major = d.major;
  if (cc_minor) *cc_minor = d.minor;
  if (smem_optin_bytes) *smem_optin_bytes = d.smem_optin;
  return CTGB_OK;
}

int ctgb_probe_fp64_peaks(double* dmma_tflops, double* dfma_tflops, void* stream) {
  DevInfo& di = devinfo();
  if (!di.ok) return fail(CTGB_E_CUDA, "no CUDA device");
  cudaStream_t st = (cudaStream_t)stream;
  double* sink = nullptr;
  CUDA_TRY(cudaMalloc((void**)&sink, 64));
  cudaEvent_t e0, e1;
  CUDA_TRY(cudaEventCreate(&e0));
  CUDA_TRY(cudaEventCreate(&e1));
  const int blocks = di.sms * 8, iters = 4096;
  auto timed = [&](int which, double flop_per_thread_iter, double* out) -> int {
    float best = 1e30f;
    for (int rep = 0; rep < 4; ++rep) {
      CUDA_TRY(cudaEventRecord(e0, st));
      if (which == 0) probe_dmma_kernel<<<blocks, 256, 0, st>>>(sink, iters);
      else probe_dfma_kernel<<<blocks, 256, 0, st>>>(sink, iters);
      CUDA_TRY(cudaEventRecord(e1, st));
      CUDA_TRY(cudaEventSynchronize(e1));
      float ms = 0.f;
      CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
      if (rep > 0 && ms < best) best = ms;
    }
    g_launches.fetch_add(4, std::memory_order_relaxed);
    *out = flop_per_thread_iter * iters * 256.0 * blocks / (best * 1e-3) / 1e12;
    return CTGB_OK;
  };
  int rc = CTGB_OK;
  // one DMMA = 8*8*4 MACs per warp = 512 flop / 32 lanes; 8 per iteration
  if (dmma_tflops) rc = timed(0, 8 * 512.0 / 32.0, dmma_tflops);
  if (!rc && dfma_tflops) rc = timed(1, 8 * 2.0, dfma_tflops);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(sink);
  return rc;
}

int ctgb_contract_pair(const int64_t* desc, const void* A, const void* B, void* C, void* stream) {
  if (!desc) return fail(CTGB_E_VALUE, "null descriptor");
  cudaStream_t st = (cudaStream_t)stream;
  int64_t* d = nullptr;
  CUDA_TRY(cudaMallocAsync((void**)&d, DESC_WORDS * sizeof(int64_t), st));
  CUDA_TRY(cudaMemcpyAsync(d, desc, DESC_WORDS * sizeof(int64_t), cudaMemcpyHostToDevice, st));
  int rc = launch_gett(desc, d, A, B, C, st);
  cudaFreeAsync(d, st);
  return rc;
}

int ctgb_reduce_single(const int64_t* desc, const void* X, void* out, void* stream) {
  if (!desc) return fail(CTGB_E_VALUE, "null descriptor");
  cudaStream_t st = (cudaStream_t)stream;
  int64_t* d = nullptr;
  CUDA_TRY(cudaMallocAsync((void**)&d, SDESC_WORDS * sizeof(int64_t), st));
  CUDA_TRY(cudaMemcpyAsync(d, desc, SDESC_WORDS * sizeof(int64_t), cudaMemcpyHostToDevice, st));
  int rc = launch_single(desc, d, X, out, st);
  cudaFreeAsync(d, st);
  return rc;
}

int ctgb_plan_create(const ctgb_plan_desc* pd, ctgb_plan** out) {
  if (!pd || !out) return fail(CTGB_E_VALUE, "null argument");
  if (elem_size(pd->dtype) == 0) return fail(CTGB_E_VALUE, "bad dtype");
  ctgb_plan* p = new ctgb_plan();
  p->dtype = pd->dtype;
  p->n_inputs = pd->n_inputs;
  p->tensors.resize(pd->n_tensors);
  for (int i = 0; i < pd->n_tensors; ++i) {
    const ctgb_tensor& t = pd->tensors[i];
    auto& q = p->tensors[i];
    q.kind = t.kind;
    q.input_index = t.input_index;
    q.offset = t.offset;
    q.nbytes = t.nbytes;
    if (t.kind == 0 && (t.input_index < 0 || t.input_index >= pd->n_inputs)) {
      delete p;
      return fail(CTGB_E_VALUE, "tensor refers to a missing input");
    }
    for (int j = 0; j < t.n_sliced; ++j) {
      if (t.slice_pos[j] < 0 || t.slice_pos[j] >= pd->n_sliced) {
        delete p;
        return fail(CTGB_E_VALUE, "slice position out of range");
      }
      q.slice_pos.push_back(t.slice_pos[j]);
      q.slice_stride.push_back(t.slice_stride[j]);
    }
  }
  p->nodes.resize(pd->n_nodes);
  int64_t per_slice = 0;
  for (int i = 0; i < pd->n_nodes; ++i) {
    const ctgb_node& n = pd->nodes[i];
    auto& q = p->nodes[i];
    q.kind = n.kind;
    q.a = n.a;
    q.b = n.b;
    q.c = n.c;
    q.invariant = n.invariant;
    q.is_root = n.is_root;
    const int words = n.kind == 0 ? (int)DESC_WORDS : (int)SDESC_WORDS;
    const int64_t magic = n.kind == 0 ? DESC_MAGIC : SDESC_MAGIC;
    if (!n.desc || n.desc[0] != magic) {
      delete p;
      return fail(CTGB_E_VALUE, "bad node descriptor");
    }
    auto bad = [&](int t) { return t < 0 || t >= pd->n_tensors; };
    if (bad(n.a) || bad(n.c) || (n.kind == 0 && bad(n.b))) {
      delete p;
      return fail(CTGB_E_VALUE, "node refers to a missing tensor");
    }
    q.desc_off = p->descs.size();
    p->descs.insert(p->descs.end(), n.desc, n.desc + words);
    q.c_elems = p->tensors[n.c].nbytes / (int64_t)elem_size(pd->dtype);
    if (pd->strip_exponent && n.kind == 0) {
      const int64_t* w = n.desc;
      q.measure_after = w[W_SPLITK] > 1 || w[W_VARIANT] == VAR_DOTSTREAM || w[W_VARIANT] == VAR_DOTSTREAM4;
      // (the block-reduction epilogue of KRED runs once: its result is measured afterwards as well;
      // so is a tcgen05 node whose contracted range is folded into C chunk by chunk)
      q.measure_after |= w[W_VARIANT] == VAR_KRED;
      q.measure_after |= (w[W_VARIANT] == VAR_TC05_128x64 || w[W_VARIANT] == VAR_TC05_128x32 ||
                          w[W_VARIANT] == VAR_TC05_128x16) &&
                         tc05_chunk_steps((unsigned)((w[W_STEPS_K] + w[W_SPLITK] - 1) / w[W_SPLITK]),
                                          (unsigned)(w[W_KTA] >> 2)) < (unsigned)w[W_STEPS_K];
    }
    if (!n.invariant) per_slice += 1 + q.measure_after + (pd->strip_exponent && n.kind == 0 ? 1 : 0);
  }
  if (pd->strip_exponent) per_slice += 5;  // reset slots, sum of logs, rescale/add/commit
  p->launches_per_slice = per_slice;
  p->radix.assign(pd->slice_radix, pd->slice_radix + pd->n_sliced);
  p->project.assign(pd->slice_project, pd->slice_project + pd->n_sliced);
  p->out_stride.assign(pd->slice_out_stride, pd->slice_out_stride + pd->n_sliced);
  p->out_elements = pd->out_elements;
  p->workspace_bytes = pd->workspace_bytes;
  p->persistent_bytes = pd->persistent_bytes;
  p->strip_exponent = pd->strip_exponent;

  if (cudaGetDevice(&p->device) != cudaSuccess) {
    delete p;
    return fail(CTGB_E_CUDA, "no CUDA device");
  }
  cudaError_t e = cudaMalloc((void**)&p->d_descs, p->descs.size() * sizeof(int64_t) + 8);
  if (e == cudaSuccess)
    e = cudaMemcpy(p->d_descs, p->descs.data(), p->descs.size() * sizeof(int64_t), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMalloc((void**)&p->d_scalars, 8 * sizeof(double));
  if (e == cudaSuccess) e = cudaMemset(p->d_scalars, 0, 8 * sizeof(double));
  if (e == cudaSuccess && p->strip_exponent) {
    // factor slots + the per-node pointers into them (patched into the plan's descriptors)
    const size_t nt = p->tensors.size();
    std::vector<double> ones(nt + 1, 1.0);
    e = cudaMalloc((void**)&p->d_factors, (nt + 1) * sizeof(double));
    if (e == cudaSuccess) e = cudaMemcpy(p->d_factors, ones.data(), (nt + 1) * sizeof(double), cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMalloc((void**)&p->d_eff, (nt + 1) * sizeof(double));
    if (e == cudaSuccess) e = cudaMemcpy(p->d_eff, ones.data(), (nt + 1) * sizeof(double), cudaMemcpyHostToDevice);
    std::vector<int> var_slots, inv_slots;
    std::vector<char> guarded(nt, 0);
    for (auto& n : p->nodes) {
      if (n.kind != 0) continue;
      // small second operand (the usual case on a stem): scale a copy of it instead of every
      // output element; otherwise the epilogue multiplies by 1/(fA fB), and the pairwise results
      // among the operands get a range guard
      const int64_t bbytes = p->tensors[n.b].nbytes;
      n.prescale_b = bbytes > 0 && bbytes <= (16ll << 20) && p->tensors[n.b].kind != 3;
      if (!n.prescale_b) guarded[n.a] = guarded[n.b] = 1;
    }
    for (auto& n : p->nodes) {
      if (n.kind != 0) continue;
      n.band = guarded[n.c] != 0;
      if (n.band) guarded[n.c] = 2;  // a guarded pairwise result
      if (n.band && !n.invariant) ++p->launches_per_slice;
    }
    for (auto& n : p->nodes) {
      if (n.kind != 0) continue;
      int64_t* w = p->descs.data() + n.desc_off;
      if (n.prescale_b) {
        const size_t bbytes = (size_t)p->tensors[n.b].nbytes;
        if (bbytes > p->bscale_bytes) p->bscale_bytes = bbytes;
      } else {
        // (inputs and single-operand results: factor 1, never normalised)
        auto scale_of = [&](int t) { return (int64_t)(uintptr_t)((guarded[t] == 2 ? p->d_eff : p->d_factors) + t); };
        w[W_SCALE_A] = scale_of(n.a);
        w[W_SCALE_B] = scale_of(n.b);
      }
      w[W_FACTOR_C] = n.measure_after ? 0 : (int64_t)(uintptr_t)(p->d_factors + n.c);
      (n.invariant ? inv_slots : var_slots).push_back(n.c);
    }
    p->n_var_slots = (int)var_slots.size();
    p->n_inv_slots = (int)inv_slots.size();
    var_slots.insert(var_slots.end(), inv_slots.begin(), inv_slots.end());
    if (e == cudaSuccess && p->bscale_bytes) e = cudaMalloc((void**)&p->d_bscale, p->bscale_bytes + 256);
    if (e == cudaSuccess) e = cudaMalloc((void**)&p->d_slot_lists, (var_slots.size() + 1) * sizeof(int));
    if (e == cudaSuccess && !var_slots.empty())
      e = cudaMemcpy(p->d_slot_lists, var_slots.data(), var_slots.size() * sizeof(int), cudaMemcpyHostToDevice);
    if (e == cudaSuccess)
      e = cudaMemcpy(p->d_descs, p->descs.data(), p->descs.size() * sizeof(int64_t), cudaMemcpyHostToDevice);
  }
  if (e != cudaSuccess) {
    std::string msg = cudaGetErrorString(e);
    ctgb_plan_destroy(p);
    return fail(CTGB_E_CUDA, "plan upload: " + msg);
  }
  *out = p;
  return CTGB_OK;
}

int ctgb_plan_profile(ctgb_plan* p, int enable) {
  if (!p) return fail(CTGB_E_VALUE, "null plan");
  if (enable && p->ev0.empty()) {
    p->ev0.resize(p->nodes.size());
    p->ev1.resize(p->nodes.size());
    for (size_t i = 0; i < p->nodes.size(); ++i) {
      CUDA_TRY(cudaEventCreate(&p->ev0[i]));
      CUDA_TRY(cudaEventCreate(&p->ev1[i]));
    }
  }
  p->profile = enable != 0;
  return CTGB_OK;
}

int ctgb_plan_profile_read(ctgb_plan* p, float* ms, int n_nodes) {
  if (!p || !ms) return fail(CTGB_E_VALUE, "null argument");
  if (p->ev0.empty()) return fail(CTGB_E_VALUE, "profiling was never enabled");
  if (n_nodes != (int)p->nodes.size()) return fail(CTGB_E_VALUE, "node count mismatch");
  for (int i = 0; i < n_nodes; ++i) {
    ms[i] = -1.f;
    if (cudaEventQuery(p->ev1[i]) == cudaErrorInvalidResourceHandle) continue;
    cudaError_t e = cudaEventSynchronize(p->ev1[i]);
    if (e != cudaSuccess) { cudaGetLastError(); continue; }
    float t = 0.f;
    if (cudaEventElapsedTime(&t, p->ev0[i], p->ev1[i]) == cudaSuccess) ms[i] = t; else cudaGetLastError();
  }
  return CTGB_OK;
}

void ctgb_plan_destroy(ctgb_plan* p) {
  if (!p) return;
  for (auto e : p->ev0) cudaEventDestroy(e);
  for (auto e : p->ev1) cudaEventDestroy(e);
  if (p->d_descs) cudaFree(p->d_descs);
  if (p->d_scalars) cudaFree(p->d_scalars);
  if (p->d_factors) cudaFree(p->d_factors);
  if (p->d_eff) cudaFree(p->d_eff);
  if (p->d_bscale) cudaFree(p->d_bscale);
  if (p->d_slot_lists) cudaFree(p->d_slot_lists);
  if (p->d_chunk_desc) cudaFree(p->d_chunk_desc);
  if (p->h_stage) cudaFreeHost(p->h_stage);
  delete p;
}

size_t ctgb_plan_workspace_bytes(const ctgb_plan* p) {
  return p ? (size_t)(p->workspace_bytes + p->persistent_bytes) : 0;
}
int64_t ctgb_plan_launches_per_slice(const ctgb_plan* p) { return p ? p->launches_per_slice : 0; }

// Install the (single-operand style) descriptor that maps the dense root result
// of one slice onto its chunk of the full output; only used with strip_exponent.
int ctgb_plan_set_chunk_desc(ctgb_plan* p, const int64_t* desc) {
  if (!p || !desc || desc[0] != SDESC_MAGIC) return fail(CTGB_E_VALUE, "bad chunk descriptor");
  p->chunk_desc.assign(desc, desc + SDESC_WORDS);
  if (!p->d_chunk_desc) CUDA_TRY(cudaMalloc((void**)&p->d_chunk_desc, SDESC_WORDS * sizeof(int64_t)));
  CUDA_TRY(cudaMemcpy(p->d_chunk_desc, desc, SDESC_WORDS * sizeof(int64_t), cudaMemcpyHostToDevice));
  return CTGB_OK;
}

int ctgb_plan_execute(ctgb_plan* p, const void* const* inputs, void* out, double* exponent_dev, void* workspace,
                      size_t workspace_bytes, int64_t slice_begin, int64_t slice_step, int64_t slice_count,
                      void* stream) {
  if (!p) return fail(CTGB_E_VALUE, "null plan");
  if (workspace_bytes < (size_t)(p->workspace_bytes + p->persistent_bytes))
    return fail(CTGB_E_MEMORY, "workspace too small");
  if (p->strip_exponent && (!exponent_dev || p->chunk_desc.empty()))
    return fail(CTGB_E_VALUE, "strip_exponent needs an exponent buffer and a chunk descriptor");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t es = elem_size(p->dtype);
  char* persistent = (char*)workspace;
  char* scratch = persistent + p->persistent_bytes;
  const int ns = (int)p->radix.size();
  std::vector<int64_t> digits(ns, 0);

  double* d_slice_exp = p->d_scalars + 1;
  double* d_inv_exp = p->d_scalars + 2;

  auto resolve = [&](int t, int64_t out_off) -> char* {
    const ctgb_plan::Tensor& q = p->tensors[t];
    switch (q.kind) {
      case 0: {
        int64_t off = 0;
        for (size_t j = 0; j < q.slice_pos.size(); ++j) off += digits[q.slice_pos[j]] * q.slice_stride[j];
        return (char*)inputs[q.input_index] + off * (int64_t)es;
      }
      case 1: return scratch + q.offset;
      case 2: return persistent + q.offset;
      default: return (char*)out + out_off * (int64_t)es;
    }
  };

  auto run_nodes = [&](bool invariant_pass, int64_t out_off) -> int {
    for (size_t ni = 0; ni < p->nodes.size(); ++ni) {
      const auto& n = p->nodes[ni];
      if ((n.invariant != 0) != invariant_pass) continue;
      if (p->profile) cudaEventRecord(p->ev0[ni], st);
      const int64_t* h = p->descs.data() + n.desc_off;
      const int64_t* d = p->d_descs + n.desc_off;
      char* A = resolve(n.a, out_off);
      char* C = resolve(n.c, out_off);
      int rc;
      if (n.kind == 0) {
        char* B = resolve(n.b, out_off);
        if (n.prescale_b) {
          // the whole underlying buffer of the small operand (a sliced input keeps its base
          // offset into the copy), scaled by 1/(fA fB) read from the factor slots on the device
          const ctgb_plan::Tensor& tb = p->tensors[n.b];
          char* under = tb.kind == 0 ? (char*)inputs[tb.input_index] : (tb.kind == 1 ? scratch : persistent) + tb.offset;
          rc = scale_copy(p->dtype, under, p->d_bscale, tb.nbytes / (int64_t)es, p->d_factors + n.a,
                          p->d_factors + n.b, st);
          if (rc) return rc;
          B = p->d_bscale + (B - under);
        }
        rc = launch_gett(h, d, A, B, C, st);
      } else {
        rc = launch_single(h, d, A, C, st);
      }
      if (rc) return rc;
      // contract.py:816-829 strips after every *pairwise* node (single-operand preprocessing
      // steps `continue` before reaching it, :792-796).  The kernels do it in their epilogues
      // (scale by the operands' factors, record max|C|: gett_kernels.cuh StripCtx); only nodes
      // that add partial sums atomically need max|C| measured in a pass of its own.
      if (p->strip_exponent && n.kind == 0 && n.measure_after) {
        rc = absmax_into(p->dtype, C, n.c_elems, (unsigned long long*)(p->d_factors + n.c), st);
        if (rc) return rc;
      }
      if (p->strip_exponent && n.band) {
        rc = band_into(p->dtype, C, n.c_elems, p->d_factors + n.c, p->d_eff + n.c, st);
        if (rc) return rc;
      }
      if (p->profile) cudaEventRecord(p->ev1[ni], st);
    }
    return CTGB_OK;
  };

  // slice-invariant subtrees: once per execute call, kept in the persistent arena
  bool any_inv = false;
  for (const auto& n : p->nodes) any_inv |= n.invariant != 0;
  if (p->strip_exponent && p->n_inv_slots > 0) {
    reset_slots_kernel<<<1, 256, 0, st>>>(p->d_factors, p->d_slot_lists + p->n_var_slots, p->n_inv_slots);
    g_launches.fetch_add(1, std::memory_order_relaxed);
  }
  if (any_inv) {
    int rc = run_nodes(true, 0);
    if (rc) return rc;
  }
  if (p->strip_exponent) {
    // exponent of the slice-invariant part: sum of log10(factor) over the hoisted pairwise nodes
    sum_log_kernel<<<1, 256, 0, st>>>(p->d_factors, p->d_slot_lists + p->n_var_slots, p->n_inv_slots, d_inv_exp,
                                      nullptr);
    g_launches.fetch_add(1, std::memory_order_relaxed);
  }

  for (int64_t k = 0; k < slice_count; ++k) {
    // slice id -> digits, most significant first (core.py:3775-3800)
    int64_t i = slice_begin + k * slice_step;
    {
      // least-significant digit first: the same digits as i // stride_j % radix_j,
      // without forming the strides (their product overflows 64 bits for trees
      // with more than 63 binary sliced indices; ids themselves are < 2^63)
      int64_t rem = i;
      for (int j = ns - 1; j >= 0; --j) {
        if (p->project[j] >= 0) {
          digits[j] = p->project[j];
        } else {
          digits[j] = rem % p->radix[j];
          rem /= p->radix[j];
        }
      }
    }
    int64_t out_off = 0;
    for (int j = 0; j < ns; ++j) out_off += digits[j] * p->out_stride[j];
    if (p->strip_exponent && p->n_var_slots > 0) {
      reset_slots_kernel<<<1, 256, 0, st>>>(p->d_factors, p->d_slot_lists, p->n_var_slots);
      g_launches.fetch_add(1, std::memory_order_relaxed);
    }
    int rc = run_nodes(false, out_off);
    if (rc) return rc;
    if (p->strip_exponent) {
      sum_log_kernel<<<1, 256, 0, st>>>(p->d_factors, p->d_slot_lists, p->n_var_slots, d_slice_exp, d_inv_exp);
      g_launches.fetch_add(1, std::memory_order_relaxed);
      // the root wrote a dense mantissa into its workspace slot; fold it into the
      // output against the running exponent (core.py:163-170, 3856-3861)
      const ctgb_plan::Node* root = nullptr;
      for (const auto& n : p->nodes)
        if (n.is_root) root = &n;
      if (!root) return fail(CTGB_E_VALUE, "plan has no root node");
      char* m = resolve(root->c, 0);
      // (the stored root is the raw product: its own factor divides it here)
      const double* froot = root->kind == 0 ? p->d_factors + root->c : nullptr;
      rc = accum_stripped(p->dtype, p->d_chunk_desc, p->chunk_desc.data(), out, (char*)out + out_off * (int64_t)es,
                          p->out_elements, m, exponent_dev, d_slice_exp, froot, st);
      if (rc) return rc;
    }
  }
  return CTGB_OK;
}

int ctgb_plan_execute_host(ctgb_plan* p, const void* const* host_inputs, const int64_t* input_nbytes, void* host_out,
                           double* host_exponent, void* workspace, size_t workspace_bytes, int64_t slice_begin,
                           int64_t slice_step, int64_t slice_count, void* stream) {
  if (!p) return fail(CTGB_E_VALUE, "null plan");
  cudaStream_t st = (cudaStream_t)stream;
  const size_t es = elem_size(p->dtype);
  const size_t core = (size_t)(p->workspace_bytes + p->persistent_bytes);
  // staging area at the tail of the workspace: inputs, output, exponent
  size_t need = core;
  auto align = [](size_t x) { return (x + 255) & ~(size_t)255; };
  need = align(need);
  std::vector<size_t> in_off(p->n_inputs);
  for (int i = 0; i < p->n_inputs; ++i) {
    in_off[i] = need;
    need = align(need + (size_t)input_nbytes[i]);
  }
  const size_t out_off = need;
  need = align(need + (size_t)p->out_elements * es);
  const size_t exp_off = need;
  need += 256;
  if (workspace_bytes < need) return fail(CTGB_E_MEMORY, "workspace too small for host staging");
  char* ws = (char*)workspace;
  std::vector<const void*> dev_inputs(p->n_inputs);
  // ONE host->device copy for all inputs (a Sycamore network has 381 tensors of 16-256 bytes:
  // 381 separate copies cost more than the bytes): pack them into the plan's pinned staging
  // block at their device offsets, then copy the block
  const size_t in_base = p->n_inputs ? in_off[0] : out_off, in_span = out_off - in_base;
  if (in_span <= ((size_t)64 << 20)) {
    if (p->h_stage_bytes < in_span) {
      if (p->h_stage) cudaFreeHost(p->h_stage);
      p->h_stage = nullptr;
      p->h_stage_bytes = 0;
      CUDA_TRY(cudaHostAlloc((void**)&p->h_stage, in_span ? in_span : 1, cudaHostAllocDefault));
      p->h_stage_bytes = in_span;
    } else {
      // the previous call's copy out of this block has completed (each call ends synchronised)
    }
    for (int i = 0; i < p->n_inputs; ++i) {
      memcpy(p->h_stage + (in_off[i] - in_base), host_inputs[i], (size_t)input_nbytes[i]);
      dev_inputs[i] = ws + in_off[i];
    }
    if (in_span) CUDA_TRY(cudaMemcpyAsync(ws + in_base, p->h_stage, in_span, cudaMemcpyHostToDevice, st));
  } else {
    for (int i = 0; i < p->n_inputs; ++i) {
      CUDA_TRY(cudaMemcpyAsync(ws + in_off[i], host_inputs[i], (size_t)input_nbytes[i], cudaMemcpyHostToDevice, st));
      dev_inputs[i] = ws + in_off[i];
    }
  }
  CUDA_TRY(cudaMemsetAsync(ws + out_off, 0, (size_t)p->out_elements * es, st));
  double* d_exp = (double*)(ws + exp_off);
  if (p->strip_exponent) {
    // running exponent starts at -inf so that the first slice sets it
    const double ninf = -__builtin_huge_val();
    CUDA_TRY(cudaMemcpyAsync(d_exp, &ninf, sizeof(double), cudaMemcpyHostToDevice, st));
  }
  int rc = ctgb_plan_execute(p, dev_inputs.data(), ws + out_off, d_exp, workspace, core, slice_begin, slice_step,
                             slice_count, stream);
  if (rc) return rc;
  CUDA_TRY(cudaMemcpyAsync(host_out, ws + out_off, (size_t)p->out_elements * es, cudaMemcpyDeviceToHost, st));
  if (p->strip_exponent && host_exponent)
    CUDA_TRY(cudaMemcpyAsync(host_exponent, d_exp, sizeof(double), cudaMemcpyDeviceToHost, st));
  CUDA_TRY(cudaStreamSynchronize(st));
  return CTGB_OK;
}

}  // extern "C"
