// Shared device helpers for libevok (sm_100a).  See include/evok.h for the ABI.
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/evok.h"

#define EVOK_CHECK_LAUNCH_N(n)                       \
  do {                                               \
    cudaError_t e__ = cudaPeekAtLastError();         \
    if (e__ != cudaSuccess) return (int)e__;         \
    evok::count_launches(n);                         \
  } while (0)
#define EVOK_CHECK_LAUNCH() EVOK_CHECK_LAUNCH_N(1)

namespace evok {

// number of kernels this library has launched (exposed as evok_launch_count(); bench.py reports it)
extern unsigned long long g_launch_count;
inline void count_launches(int n) { __atomic_fetch_add(&g_launch_count, (unsigned long long)n, __ATOMIC_RELAXED); }

constexpr int kWarp = 32;
constexpr int kNumSMs = 148;  // B200

// ------------------------------------------------------------------------------------------------
// Peer exchange over NVLink (evok_peer.cu): where a producing kernel's result is needed by every GPU, the kernel itself
// stores it into every peer's buffer and the LAST CTA to finish raises this rank's flag in every peer's flag array.
// ------------------------------------------------------------------------------------------------
struct PeerSink {
  void* data[EVOK_MAX_PEERS];                 // peer p's destination buffer (this rank's own buffer at p == rank)
  unsigned long long* flags[EVOK_MAX_PEERS];  // peer p's flag array (one 64-bit epoch per source rank)
  int world, rank;
};

__device__ __forceinline__ void st_release_sys(unsigned long long* p, unsigned long long v) {
  asm volatile("st.release.sys.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
__device__ __forceinline__ unsigned long long ld_acquire_sys(const unsigned long long* p) {
  unsigned long long v;
  asm volatile("ld.acquire.sys.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
  return v;
}

// Call from ALL threads of EVERY CTA of a 1-D grid after the CTA's last peer store.  `epoch` (local) holds the number of
// completed exchanges; the flag value raised is epoch + 1 (the waiting kernel advances `epoch`).  `done` is a local counter
// that returns to 0 for the next launch.
static __device__ __noinline__ void peer_signal_tail(const PeerSink& s, const unsigned long long* epoch, unsigned int* done) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();  // this CTA's peer stores are visible system-wide before the counter moves
    const unsigned int prev = atomicAdd(done, 1u);
    if (prev == gridDim.x - 1) {
      *done = 0;
      __threadfence_system();
      const unsigned long long e = *epoch + 1ull;
      for (int p = 0; p < s.world; ++p) st_release_sys(s.flags[p] + s.rank, e);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al., SC'11).  One call -> 4 x 32 random bits.
// ------------------------------------------------------------------------------------------------
struct U4 {
  uint32_t x, y, z, w;
};

// The 10 round keys of one (seed, stream) pair, precomputed on the host and passed to the kernels BY VALUE: they live in
// the constant bank, so each round's key XOR takes its operand straight from c[][] (no per-thread key-schedule adds).
struct PhiloxKey {
  uint32_t k0[10], k1[10];
  uint32_t stream_lo;
};

inline PhiloxKey make_philox_key(uint64_t seed, uint64_t stream_id) {
  PhiloxKey k;
  uint32_t a = (uint32_t)seed, b = (uint32_t)(seed >> 32) ^ (uint32_t)(stream_id >> 32);
  for (int r = 0; r < 10; ++r) {
    k.k0[r] = a;
    k.k1[r] = b;
    a += 0x9E3779B9u;
    b += 0xBB67AE85u;
  }
  k.stream_lo = (uint32_t)stream_id;
  return k;
}

// EVOK_PHILOX_ROUNDS exists for MEASUREMENT builds only (scripts/build_variants.py: what would fewer rounds buy?); the
// product is Philox4x32-10, the variant cuRAND / torch use, and the oracle restates exactly that.
#ifndef EVOK_PHILOX_ROUNDS
#define EVOK_PHILOX_ROUNDS 10
#endif
__device__ __forceinline__ U4 philox4x32_10(U4 c, const PhiloxKey& key) {
  constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
#pragma unroll
  for (int r = 0; r < EVOK_PHILOX_ROUNDS; ++r) {
    const uint32_t hi0 = __umulhi(M0, c.x), lo0 = M0 * c.x;
    const uint32_t hi1 = __umulhi(M1, c.z), lo1 = M1 * c.z;
    U4 n;
    n.x = hi1 ^ c.y ^ key.k0[r];
    n.y = lo1;
    n.z = hi0 ^ c.w ^ key.k1[r];
    n.w = lo0;
    c = n;
  }
  return c;
}

__device__ __forceinline__ float sqrt_approx(float x) {
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

__device__ __forceinline__ float lg2_approx(float x) {
  float r;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// Box-Muller on 32+32 random bits -> two standard normals.
//   u1 = 2^-33 + a * 2^-32 in (0, 1]  (never 0, so the log is finite);  r = sqrt(-2 ln u1) = sqrt(lg2(u1) * (-2 ln 2))
//   theta = 2 pi (2^-33 + b * 2^-32): the 2 pi is folded into the conversion constants.
__device__ __forceinline__ void box_muller(uint32_t a, uint32_t b, float& z0, float& z1) {
  const float u1 = fmaf((float)a, 2.3283064365386963e-10f, 1.1641532182693481e-10f);
  const float th = fmaf((float)b, 1.4629180792671596e-09f, 7.314590396335798e-10f);
  const float r = sqrt_approx(lg2_approx(u1) * -1.3862943611198906f);
  float s, c;
  __sincosf(th, &s, &c);
  z0 = r * c;
  z1 = r * s;
}

// The four standard normals of (unit, column group q): `unit` is the GLOBAL direction index (symmetric
// sampling: rows 2*unit and 2*unit+1) or the global row index (non-symmetric); columns 4q .. 4q+3.
// `stream_word` = low 32 bits of the stream id (key.stream_lo plus an optional device-side generation offset, which lets a
// CUDA graph that was captured once draw a fresh population on every replay)
__device__ __forceinline__ void normals4(const PhiloxKey& key, uint32_t stream_word, uint64_t unit, uint32_t q, float z[4]) {
  U4 c;
  c.x = q;
  c.y = (uint32_t)unit;
  c.z = (uint32_t)(unit >> 32);
  c.w = stream_word;
  const U4 r = philox4x32_10(c, key);
  box_muller(r.x, r.y, z[0], z[1]);
  box_muller(r.z, r.w, z[2], z[3]);
}

// ------------------------------------------------------------------------------------------------
// Warp / block reductions
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Sum over a whole CTA (blockDim.x multiple of 32, <= 1024).  Result valid in every thread.
template <typename T>
__device__ __forceinline__ T block_sum(T v, T* smem /* >= 33 entries */) {
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();  // protect smem reuse across consecutive calls
  if (lane == 0) smem[wid] = v;
  __syncthreads();
  if (wid == 0) {
    T t = lane < nw ? smem[lane] : T(0);
    t = warp_sum(t);
    if (lane == 0) smem[32] = t;
  }
  __syncthreads();
  return smem[32];
}

// streaming 128-bit accesses: the population is touched once per kernel, keep it out of L1
__device__ __forceinline__ float4 ld_stream4(const float* p) {
  float4 v;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p));
  return v;
}
__device__ __forceinline__ float ld_stream1(const float* p) {
  float v;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ void st_stream4(float* p, float a, float b, float c, float d) {
  asm volatile("st.global.cs.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}
__device__ __forceinline__ void st_stream1(float* p, float a) {
  asm volatile("st.global.cs.f32 [%0], %1;" ::"l"(p), "f"(a) : "memory");
}

// ------------------------------------------------------------------------------------------------
// Objective accumulators: add(x) per element, then the per-lane partials are warp-reduced and finished.
// ------------------------------------------------------------------------------------------------
template <int OBJ>
struct ObjAcc;

template <>
struct ObjAcc<EVOK_OBJ_NONE> {
  __device__ __forceinline__ void add(float) {}
  __device__ __forceinline__ float finish(int64_t) { return 0.f; }
};
template <>
struct ObjAcc<EVOK_OBJ_SPHERE> {
  float s2 = 0.f;
  __device__ __forceinline__ void add(float x) { s2 = fmaf(x, x, s2); }
  __device__ __forceinline__ float finish(int64_t) { return warp_sum(s2); }
};
template <>
struct ObjAcc<EVOK_OBJ_RASTRIGIN> {
  float s2 = 0.f, sc = 0.f;
  __device__ __forceinline__ void add(float x) {
    s2 = fmaf(x, x, s2);
    sc += __cosf(6.2831853071795865f * x);
  }
  __device__ __forceinline__ float finish(int64_t D) {
    const float a = warp_sum(s2), c = warp_sum(sc);
    return fmaf(-10.f, c, a) + 10.f * (float)D;
  }
};
template <>
struct ObjAcc<EVOK_OBJ_ACKLEY> {
  float s2 = 0.f, sc = 0.f;
  __device__ __forceinline__ void add(float x) {
    s2 = fmaf(x, x, s2);
    sc += __cosf(6.2831853071795865f * x);
  }
  __device__ __forceinline__ float finish(int64_t D) {
    const float a = warp_sum(s2), c = warp_sum(sc);
    const float invD = 1.0f / (float)D;
    return -20.f * expf(-0.2f * sqrtf(a * invD)) - expf(c * invD) + 20.f + 2.718281828459045f;
  }
};

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }
__device__ __forceinline__ bool aligned16_dev(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// activations of the policy-forward kernels (tanh to ~1e-6 absolute: a 4-term odd polynomial below 0.25, (1 - e) / (1 + e) above)
__device__ __forceinline__ float tanh_1e6(float x) {
  const float ax = fabsf(x);
  float r;
  if (ax < 0.25f) {
    const float t = ax * ax;
    r = ax * fmaf(t, fmaf(t, fmaf(t, fmaf(t, 0.021869488f, -0.053968254f), 0.13333334f), -0.33333334f), 1.0f);
  } else {
    const float e = __expf(-2.0f * ax);
    r = __fdividef(1.0f - e, 1.0f + e);
  }
  return copysignf(r, x);
}
// branch-free tanh = (1 - e) / (1 + e), e = exp(-2 |x|), with the hardware ex2 / rcp: 7 instructions, absolute error ~1e-7 (the RELATIVE
// error grows towards x = 0, where 1 - e cancels: use tanh_1e6 where that matters).  For the GEMM epilogue of the policy forward, where
// 128 activations per thread sit on the critical path of every tile.
__device__ __forceinline__ float tanh_abs1e7(float x) {
  const float e = __expf(-2.0f * fabsf(x));
  return copysignf(__fdividef(1.0f - e, 1.0f + e), x);
}
__device__ __forceinline__ float activate_fast(float v, int act) {
  switch (act) {
    case EVOK_ACT_TANH: return tanh_1e6(v);
    case EVOK_ACT_RELU: return fmaxf(v, 0.0f);
    case EVOK_ACT_SIGMOID: return __fdividef(1.0f, 1.0f + __expf(-v));
    default: return v;
  }
}

// Stacked-rows GEMM of the shared-minibatch policy forward (evok_gemm.cu, used by evok_mlp.cu):
//   C[(i * n_cols + b) * rows_per_batch + h] = act( sum_k W_i[h, k] * X[b, k] + bias_i[h] )
// W_i = params + i * batch_stride + w_offset (rows_per_batch x K, row-major, any 4-byte alignment), bias_i = params + i * batch_stride +
// bias_offset (bias_offset < 0: none); X is n_cols x K at pitch ldx.  ws: gemm_gather_rows_workspace_bytes(n_cols, K) bytes.
size_t gemm_gather_rows_workspace_bytes(int64_t n_cols, int64_t K);
int gemm_gather_rows_ws(const float* params, int64_t batch_stride, int64_t w_offset, int64_t rows_per_batch, int64_t n_batches, const float* X,
                        int64_t ldx, int64_t n_cols, int64_t K, int64_t bias_offset, int act, float* C, void* ws, size_t ws_bytes, void* stream);

}  // namespace evok
