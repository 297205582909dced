// K1 / K2: fused Philox sampling -> perturbation write -> objective row-reduction, and the stand-alone
// evaluation kernel.  HBM-bound design: one warp owns one direction (a +/- row pair) or one row; every
// lane produces 4 consecutive columns per step from ONE Philox4x32-10 call, writes them with 128-bit
// streaming stores (512 contiguous bytes per warp-row) and folds them into the objective accumulators
// while they are still in registers, so the population is written once and never re-read for evaluation.
#include "evok_common.cuh"

namespace evok {

static int g_sm_count = 0;
static int sm_count() {
  if (g_sm_count == 0) {
    int dev = 0, n = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = kNumSMs;
    g_sm_count = n;
  }
  return g_sm_count;
}

// tunables (profiles/ records the sweep that chose the defaults)
#ifndef EVOK_SAMPLE_THREADS
#define EVOK_SAMPLE_THREADS 256
#endif
#ifndef EVOK_SAMPLE_MINB
#define EVOK_SAMPLE_MINB 3
#endif
#ifndef EVOK_SAMPLE_UNR
#define EVOK_SAMPLE_UNR 2
#endif
#ifndef EVOK_SAMPLEONLY_MINB
#define EVOK_SAMPLEONLY_MINB 5
#endif
#ifndef EVOK_SAMPLEONLY_UNR
#define EVOK_SAMPLEONLY_UNR 1
#endif
constexpr int kSampleThreads = EVOK_SAMPLE_THREADS;
// the fused kernels are issue/XU bound (two independent Philox chains per lane help); the sample-only kernel is store
// bound and prefers occupancy (kbench sweep in profiles/)
template <int OBJ>
struct SampleTune {
  static constexpr int kUnroll = OBJ == EVOK_OBJ_NONE ? EVOK_SAMPLEONLY_UNR : EVOK_SAMPLE_UNR;
  static constexpr int kMinBlocks = OBJ == EVOK_OBJ_NONE ? EVOK_SAMPLEONLY_MINB : EVOK_SAMPLE_MINB;
};

// one column group (4 columns) of one unit: sample, store, accumulate
template <int OBJ, bool SYM, bool STORE, bool VEC>
__device__ __forceinline__ void sample_group(const PhiloxKey& key, uint32_t sw, uint64_t unit, uint32_t q, int64_t D,
                                             const float* __restrict__ mu, const float* __restrict__ sigma, float* xp, float* xm,
                                             ObjAcc<OBJ>& accp, ObjAcc<OBJ>& accm) {
  float z[4];
  normals4(key, sw, unit, q, z);
  const int64_t j = (int64_t)q << 2;
  if (VEC) {
    const float4 m = __ldg(reinterpret_cast<const float4*>(mu + j));
    const float4 s = __ldg(reinterpret_cast<const float4*>(sigma + j));
    const float p0 = fmaf(s.x, z[0], m.x), p1 = fmaf(s.y, z[1], m.y), p2 = fmaf(s.z, z[2], m.z), p3 = fmaf(s.w, z[3], m.w);
    if (STORE) st_stream4(xp + j, p0, p1, p2, p3);
    accp.add(p0); accp.add(p1); accp.add(p2); accp.add(p3);
    if (SYM) {
      const float n0 = fmaf(-s.x, z[0], m.x), n1 = fmaf(-s.y, z[1], m.y), n2 = fmaf(-s.z, z[2], m.z), n3 = fmaf(-s.w, z[3], m.w);
      if (STORE) st_stream4(xm + j, n0, n1, n2, n3);
      accm.add(n0); accm.add(n1); accm.add(n2); accm.add(n3);
    }
  } else {
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      if (j + c < D) {
        const float m = __ldg(mu + j + c), s = __ldg(sigma + j + c);
        const float p = fmaf(s, z[c], m);
        if (STORE) st_stream1(xp + j + c, p);
        accp.add(p);
        if (SYM) {
          const float n = fmaf(-s, z[c], m);
          if (STORE) st_stream1(xm + j + c, n);
          accm.add(n);
        }
      }
    }
  }
}

template <int OBJ, bool SYM, bool STORE, bool VEC>
__global__ void __launch_bounds__(kSampleThreads, SampleTune<OBJ>::kMinBlocks)
    sample_eval_kernel(float* __restrict__ X, int64_t ldx, const float* __restrict__ mu, const float* __restrict__ sigma,
                       int64_t row0, int64_t n_units, int64_t D, const __grid_constant__ PhiloxKey key, const uint32_t* __restrict__ stream_off,
                       float* __restrict__ f) {
  const int lane = threadIdx.x & 31;
  const uint32_t sw = key.stream_lo + (stream_off ? __ldg(stream_off) : 0u);
  const int64_t warps_total = (int64_t)gridDim.x * (kSampleThreads / 32);
  const int64_t gw = (int64_t)blockIdx.x * (kSampleThreads / 32) + (threadIdx.x >> 5);
  const uint32_t nq = (uint32_t)((D + 3) >> 2);
  const uint64_t unit0 = (uint64_t)(SYM ? (row0 >> 1) : row0);

  for (int64_t u = gw; u < n_units; u += warps_total) {
    ObjAcc<OBJ> accp, accm;
    const int64_t r = SYM ? 2 * u : u;
    float* xp = STORE ? X + r * ldx : nullptr;
    float* xm = STORE ? xp + ldx : nullptr;
    const uint64_t unit = unit0 + (uint64_t)u;
    constexpr int kSampleUnroll = SampleTune<OBJ>::kUnroll;
    uint32_t q = lane;
    if (kSampleUnroll > 1) {
      // independent Philox chains in flight per lane
      for (; q + 32u * (kSampleUnroll - 1) < nq; q += 32u * kSampleUnroll) {
#pragma unroll
        for (int uu = 0; uu < kSampleUnroll; ++uu)
          sample_group<OBJ, SYM, STORE, VEC>(key, sw, unit, q + 32u * uu, D, mu, sigma, xp, xm, accp, accm);
      }
    }
    for (; q < nq; q += 32) sample_group<OBJ, SYM, STORE, VEC>(key, sw, unit, q, D, mu, sigma, xp, xm, accp, accm);
    if (OBJ != EVOK_OBJ_NONE) {
      const float fp = accp.finish(D);
      float fm = 0.f;
      if (SYM) fm = accm.finish(D);
      if (lane == 0) {
        f[r] = fp;
        if (SYM) f[r + 1] = fm;
      }
    }
  }
}

// Batched searches (functional ask/tell API with leading batch dimensions, funcpgpe.py:301-327): blockIdx.y = batch item, every
// item has its own centre / stdev row (item stride 0 = shared) and its own Philox stream (stream word + item), so one launch
// draws the populations of all items -- bit-identical to one evok_sample_eval call per item with stream_id = item.
template <bool SYM, bool VEC>
__global__ void __launch_bounds__(kSampleThreads, SampleTune<EVOK_OBJ_NONE>::kMinBlocks)
    sample_batched_kernel(float* __restrict__ X, int64_t item_stride_x, int64_t ldx, const float* __restrict__ mu, int64_t item_stride_mu,
                          const float* __restrict__ sigma, int64_t item_stride_sigma, int64_t n_units, int64_t D, const __grid_constant__ PhiloxKey key) {
  const int lane = threadIdx.x & 31;
  const int64_t item = blockIdx.y;
  X += item * item_stride_x;
  mu += item * item_stride_mu;
  sigma += item * item_stride_sigma;
  const uint32_t sw = key.stream_lo + (uint32_t)item;
  const int64_t warps_total = (int64_t)gridDim.x * (kSampleThreads / 32);
  const int64_t gw = (int64_t)blockIdx.x * (kSampleThreads / 32) + (threadIdx.x >> 5);
  const uint32_t nq = (uint32_t)((D + 3) >> 2);
  for (int64_t u = gw; u < n_units; u += warps_total) {
    ObjAcc<EVOK_OBJ_NONE> accp, accm;
    float* xp = X + (SYM ? 2 * u : u) * ldx;
    float* xm = xp + ldx;
    for (uint32_t q = lane; q < nq; q += 32) sample_group<EVOK_OBJ_NONE, SYM, true, VEC>(key, sw, (uint64_t)u, q, D, mu, sigma, xp, xm, accp, accm);
  }
}

constexpr int kEvalThreads = 256;

template <int OBJ, bool VEC>
__global__ void __launch_bounds__(kEvalThreads)
    eval_kernel(const float* __restrict__ X, int64_t ldx, int64_t n_rows, int64_t D, float* __restrict__ f) {
  const int lane = threadIdx.x & 31;
  const int64_t warps_total = (int64_t)gridDim.x * (kEvalThreads / 32);
  const int64_t gw = (int64_t)blockIdx.x * (kEvalThreads / 32) + (threadIdx.x >> 5);
  for (int64_t r = gw; r < n_rows; r += warps_total) {
    ObjAcc<OBJ> acc;
    const float* x = X + r * ldx;
    if (VEC) {
      const int64_t nq = D >> 2;
      int64_t q = lane;
      // 4 independent 128-bit loads in flight per lane
      for (; q + 96 < nq; q += 128) {
        const float4 a = ld_stream4(x + 4 * q), b = ld_stream4(x + 4 * (q + 32)), c = ld_stream4(x + 4 * (q + 64)),
                     d = ld_stream4(x + 4 * (q + 96));
        acc.add(a.x); acc.add(a.y); acc.add(a.z); acc.add(a.w);
        acc.add(b.x); acc.add(b.y); acc.add(b.z); acc.add(b.w);
        acc.add(c.x); acc.add(c.y); acc.add(c.z); acc.add(c.w);
        acc.add(d.x); acc.add(d.y); acc.add(d.z); acc.add(d.w);
      }
      for (; q < nq; q += 32) {
        const float4 a = ld_stream4(x + 4 * q);
        acc.add(a.x); acc.add(a.y); acc.add(a.z); acc.add(a.w);
      }
    } else {
      for (int64_t j = lane; j < D; j += 32) acc.add(ld_stream1(x + j));
    }
    const float v = acc.finish(D);
    if (lane == 0) f[r] = v;
  }
}

template <typename K>
static int resident_grid(K kernel, int threads, int64_t units_per_cta_needed) {
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, threads, 0) != cudaSuccess || per_sm <= 0) per_sm = 4;
  int64_t g = (int64_t)per_sm * sm_count();
  if (g > units_per_cta_needed) g = units_per_cta_needed;
  if (g < 1) g = 1;
  return (int)g;
}

template <int OBJ, bool SYM, bool STORE>
static int launch_sample(float* X, int64_t ldx, const float* mu, const float* sigma, int64_t row0, int64_t n_rows, int64_t D,
                         uint64_t seed, uint64_t stream_id, const uint32_t* stream_off, float* f, cudaStream_t st) {
  const int64_t n_units = SYM ? n_rows / 2 : n_rows;
  const bool vec = (D % 4 == 0) && aligned16(mu) && aligned16(sigma) && (!STORE || (aligned16(X) && ldx % 4 == 0));
  const int64_t ctas_needed = (n_units + (kSampleThreads / 32) - 1) / (kSampleThreads / 32);
  const PhiloxKey key = make_philox_key(seed, stream_id);
  if (vec) {
    auto k = sample_eval_kernel<OBJ, SYM, STORE, true>;
    k<<<resident_grid(k, kSampleThreads, ctas_needed), kSampleThreads, 0, st>>>(X, ldx, mu, sigma, row0, n_units, D, key, stream_off, f);
  } else {
    auto k = sample_eval_kernel<OBJ, SYM, STORE, false>;
    k<<<resident_grid(k, kSampleThreads, ctas_needed), kSampleThreads, 0, st>>>(X, ldx, mu, sigma, row0, n_units, D, key, stream_off, f);
  }
  EVOK_CHECK_LAUNCH();
  return 0;
}

template <int OBJ>
static int dispatch_sample(float* X, int64_t ldx, const float* mu, const float* sigma, int64_t row0, int64_t n_rows, int64_t D,
                           int symmetric, uint64_t seed, uint64_t stream_id, const uint32_t* stream_off, float* f, cudaStream_t st) {
  if (symmetric) {
    return X ? launch_sample<OBJ, true, true>(X, ldx, mu, sigma, row0, n_rows, D, seed, stream_id, stream_off, f, st)
             : launch_sample<OBJ, true, false>(X, ldx, mu, sigma, row0, n_rows, D, seed, stream_id, stream_off, f, st);
  }
  return X ? launch_sample<OBJ, false, true>(X, ldx, mu, sigma, row0, n_rows, D, seed, stream_id, stream_off, f, st)
           : launch_sample<OBJ, false, false>(X, ldx, mu, sigma, row0, n_rows, D, seed, stream_id, stream_off, f, st);
}

template <int OBJ>
static int launch_eval(const float* X, int64_t ldx, int64_t n_rows, int64_t D, float* f, cudaStream_t st) {
  const bool vec = (D % 4 == 0) && aligned16(X) && (ldx % 4 == 0);
  const int64_t ctas_needed = (n_rows + (kEvalThreads / 32) - 1) / (kEvalThreads / 32);
  if (vec) {
    auto k = eval_kernel<OBJ, true>;
    k<<<resident_grid(k, kEvalThreads, ctas_needed), kEvalThreads, 0, st>>>(X, ldx, n_rows, D, f);
  } else {
    auto k = eval_kernel<OBJ, false>;
    k<<<resident_grid(k, kEvalThreads, ctas_needed), kEvalThreads, 0, st>>>(X, ldx, n_rows, D, f);
  }
  EVOK_CHECK_LAUNCH();
  return 0;
}

}  // namespace evok

using namespace evok;

extern "C" EVOK_API int evok_sample_eval(int objective, float* X, int64_t ldx, const float* mu, const float* sigma, int64_t row0,
                                int64_t n_rows, int64_t D, int symmetric, uint64_t seed, uint64_t stream_id,
                                const uint32_t* stream_offset_dev, float* f, void* stream) {
  const uint32_t* stream_off = stream_offset_dev;
  if (!mu || !sigma) return EVOK_E_NULLPTR;
  if (objective < 0 || objective >= EVOK_OBJ_COUNT) return EVOK_E_BADENUM;
  if (objective == EVOK_OBJ_NONE && !X) return EVOK_E_NULLPTR;
  if (objective != EVOK_OBJ_NONE && !f) return EVOK_E_NULLPTR;
  if (n_rows < 0 || D <= 0 || row0 < 0 || (X && ldx < D)) return EVOK_E_BADSIZE;
  if (symmetric && ((n_rows & 1) || (row0 & 1))) return EVOK_E_ODDROWS;
  if (n_rows == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  switch (objective) {
    case EVOK_OBJ_NONE: return dispatch_sample<EVOK_OBJ_NONE>(X, ldx, mu, sigma, row0, n_rows, D, symmetric, seed, stream_id, stream_off, f, st);
    case EVOK_OBJ_SPHERE: return dispatch_sample<EVOK_OBJ_SPHERE>(X, ldx, mu, sigma, row0, n_rows, D, symmetric, seed, stream_id, stream_off, f, st);
    case EVOK_OBJ_RASTRIGIN: return dispatch_sample<EVOK_OBJ_RASTRIGIN>(X, ldx, mu, sigma, row0, n_rows, D, symmetric, seed, stream_id, stream_off, f, st);
    case EVOK_OBJ_ACKLEY: return dispatch_sample<EVOK_OBJ_ACKLEY>(X, ldx, mu, sigma, row0, n_rows, D, symmetric, seed, stream_id, stream_off, f, st);
  }
  return EVOK_E_BADENUM;
}

extern "C" EVOK_API int evok_eval(int objective, const float* X, int64_t ldx, int64_t n_rows, int64_t D, float* f, void* stream) {
  if (!X || !f) return EVOK_E_NULLPTR;
  if (objective <= EVOK_OBJ_NONE || objective >= EVOK_OBJ_COUNT) return EVOK_E_BADENUM;
  if (n_rows < 0 || D <= 0 || ldx < D) return EVOK_E_BADSIZE;
  if (n_rows == 0) return 0;
  cudaStream_t st = (cudaStream_t)stream;
  switch (objective) {
    case EVOK_OBJ_SPHERE: return launch_eval<EVOK_OBJ_SPHERE>(X, ldx, n_rows, D, f, st);
    case EVOK_OBJ_RASTRIGIN: return launch_eval<EVOK_OBJ_RASTRIGIN>(X, ldx, n_rows, D, f, st);
    case EVOK_OBJ_ACKLEY: return launch_eval<EVOK_OBJ_ACKLEY>(X, ldx, n_rows, D, f, st);
  }
  return EVOK_E_BADENUM;
}

extern "C" EVOK_API int evok_sample_batched(float* X, int64_t item_stride_x, int64_t ldx, const float* mu, int64_t item_stride_mu, const float* sigma,
                                            int64_t item_stride_sigma, int64_t n_items, int64_t n_rows, int64_t D, int symmetric, uint64_t seed,
                                            uint64_t stream_id0, void* stream) {
  if (!X || !mu || !sigma) return EVOK_E_NULLPTR;
  if (n_items < 0 || n_items > 65535 || n_rows < 0 || D <= 0 || ldx < D || item_stride_x < 0 || item_stride_mu < 0 || item_stride_sigma < 0)
    return EVOK_E_BADSIZE;
  if (symmetric && (n_rows & 1)) return EVOK_E_ODDROWS;
  if (n_items == 0 || n_rows == 0) return 0;
  const int64_t n_units = symmetric ? n_rows / 2 : n_rows;
  const bool vec = (D % 4 == 0) && aligned16(mu) && aligned16(sigma) && aligned16(X) && ldx % 4 == 0 && item_stride_x % 4 == 0 &&
                   item_stride_mu % 4 == 0 && item_stride_sigma % 4 == 0;
  int64_t ctas = (n_units + (kSampleThreads / 32) - 1) / (kSampleThreads / 32);
  const int64_t cap = ((int64_t)sm_count() * 8 + n_items - 1) / n_items;  // about 8 CTAs per SM over all items
  if (ctas > cap) ctas = cap < 1 ? 1 : cap;
  const PhiloxKey key = make_philox_key(seed, stream_id0);
  dim3 grid((unsigned)ctas, (unsigned)n_items);
  cudaStream_t st = (cudaStream_t)stream;
#define EVOK_LAUNCH_SB(SYMV, VECV)                                                                                                    \
  sample_batched_kernel<SYMV, VECV><<<grid, kSampleThreads, 0, st>>>(X, item_stride_x, ldx, mu, item_stride_mu, sigma, item_stride_sigma, \
                                                                     n_units, D, key)
  if (symmetric) {
    if (vec) EVOK_LAUNCH_SB(true, true);
    else EVOK_LAUNCH_SB(true, false);
  } else {
    if (vec) EVOK_LAUNCH_SB(false, true);
    else EVOK_LAUNCH_SB(false, false);
  }
#undef EVOK_LAUNCH_SB
  EVOK_CHECK_LAUNCH();
  return 0;
}
