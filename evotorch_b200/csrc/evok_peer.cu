// Peer exchange over NVLink / NVSwitch: buffer sharing between the per-GPU processes (CUDA IPC) and the two consumer-side
// kernels -- the flag wait and the slot reduction -- plus the fitness push.  The gradient's producer side lives in the kernel that
// produces it (grad_finalize_push_kernel); see PeerSink / peer_signal_tail in evok_common.cuh.
//
// Protocol per exchange point (fitness gather, gradient reduce), all counters 64-bit and monotone:
//   producer rank r, generation g : stores its data into every peer's buffer, fence.sys, flag[p][r] = g + 1 (st.release.sys)
//   consumer rank p               : spins until flag[p][r] >= g + 1 for all r (ld.acquire.sys), then epoch = g + 1
// A buffer is rewritten for generation g + 1 only after the writer has consumed the OTHER exchange point of generation g,
// which every rank raises after it has finished reading this one -- so no double buffering is needed (DESIGN.md section 5).
#include <string.h>

#include "evok_common.cuh"

namespace evok {

__device__ __forceinline__ unsigned long long global_timer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

// true when every flag reached `want` before the deadline
__device__ __forceinline__ bool spin_until(const unsigned long long* flag, unsigned long long want, unsigned long long timeout_ns) {
  const unsigned long long t0 = global_timer_ns();
  while (ld_acquire_sys(flag) < want) {
    if (global_timer_ns() - t0 > timeout_ns) return false;
    __nanosleep(64);
  }
  return true;
}

__global__ void __launch_bounds__(32) peer_wait_kernel(const unsigned long long* flags, int world, unsigned long long* epoch, unsigned int* err,
                                                       unsigned long long timeout_ns) {
  const unsigned long long want = *epoch + 1ull;
  bool ok = true;
  if ((int)threadIdx.x < world) ok = spin_until(flags + threadIdx.x, want, timeout_ns);
  __syncwarp();
  if (!ok) atomicExch(err, 1u);
  if (threadIdx.x == 0) *epoch = want;
}

// One CTA per destination GPU: copy this rank's slice into that peer's buffer with 16-byte stores, then ONE system fence and the
// flag.  Pushing the fitnesses from inside the sampler costs every one of its 444 CTAs a system-scope fence behind scattered 4-byte
// remote stores (+68 us on a 0.86 ms kernel at 8 GPUs, measured); a dedicated 8-CTA kernel right behind the sampler moves the same
// 500 KB per peer as coalesced vectors and fences 8 times.
constexpr int kPushThreads = 1024;

__global__ void __launch_bounds__(kPushThreads)
    peer_push_kernel(const unsigned char* __restrict__ src, int64_t n_bytes, int64_t dst_offset, const __grid_constant__ PeerSink sink,
                     const unsigned long long* epoch) {
  const int p = (sink.rank + 1 + blockIdx.x) % sink.world;  // rotated: the GPUs do not all start on the same link
  unsigned char* dst = static_cast<unsigned char*>(sink.data[p]) + dst_offset;
  if (dst != src) {
    const bool vec = ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15u) == 0;
    if (vec) {
      const int64_t nq = n_bytes >> 4;
      for (int64_t q = threadIdx.x; q < nq; q += kPushThreads) reinterpret_cast<uint4*>(dst)[q] = reinterpret_cast<const uint4*>(src)[q];
      for (int64_t i = (nq << 4) + threadIdx.x; i < n_bytes; i += kPushThreads) dst[i] = src[i];
    } else {
      const int64_t nw = n_bytes >> 2;  // slices are made of 4-byte elements
      for (int64_t q = threadIdx.x; q < nw; q += kPushThreads) reinterpret_cast<uint32_t*>(dst)[q] = reinterpret_cast<const uint32_t*>(src)[q];
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence_system();
    st_release_sys(sink.flags[p] + sink.rank, *epoch + 1ull);
  }
}

constexpr int kReduceThreads = 256;

__global__ void __launch_bounds__(kReduceThreads)
    peer_reduce_kernel(const float* slots, int world, int64_t n, const unsigned long long* flags, unsigned long long* epoch, unsigned int* done,
                       unsigned int* err, unsigned long long timeout_ns, float* __restrict__ out) {
  const unsigned long long want = *epoch + 1ull;
  if ((int)threadIdx.x < world && !spin_until(flags + threadIdx.x, want, timeout_ns)) atomicExch(err, 1u);
  __syncthreads();
  const int64_t j = (int64_t)blockIdx.x * kReduceThreads + threadIdx.x;
  if (j < n) {
    float t = 0.0f;
    for (int r = 0; r < world; ++r) t += __ldcg(slots + (int64_t)r * n + j);  // L2 loads: the slots were written by peers while this kernel may have been spinning
    out[j] = t;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    // every CTA has read `epoch` before it arrives here, so the last one may advance it
    const unsigned int prev = atomicAdd(done, 1u);
    if (prev == gridDim.x - 1) {
      *done = 0;
      *epoch = want;
    }
  }
}

}  // namespace evok

using namespace evok;

extern "C" EVOK_API int evok_peer_alloc(size_t bytes, void** dev_ptr, void* handle_out) {
  if (!dev_ptr || !handle_out) return EVOK_E_NULLPTR;
  if (bytes == 0) return EVOK_E_BADSIZE;
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, bytes);
  if (e != cudaSuccess) return (int)e;
  e = cudaMemset(p, 0, bytes);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e == cudaSuccess) e = cudaIpcGetMemHandle(reinterpret_cast<cudaIpcMemHandle_t*>(handle_out), p);
  if (e != cudaSuccess) {
    cudaFree(p);
    return (int)e;
  }
  *dev_ptr = p;
  return 0;
}

extern "C" EVOK_API int evok_peer_open(const void* handle, void** dev_ptr) {
  if (!handle || !dev_ptr) return EVOK_E_NULLPTR;
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  return (int)cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess);
}

extern "C" EVOK_API int evok_peer_close(void* dev_ptr) { return dev_ptr ? (int)cudaIpcCloseMemHandle(dev_ptr) : EVOK_E_NULLPTR; }
extern "C" EVOK_API int evok_peer_free(void* dev_ptr) { return dev_ptr ? (int)cudaFree(dev_ptr) : EVOK_E_NULLPTR; }

extern "C" EVOK_API int evok_peer_wait(const uint64_t* flags_local, int world, uint64_t* epoch_dev, uint32_t* err_dev, uint64_t timeout_ns, void* stream) {
  if (!flags_local || !epoch_dev || !err_dev) return EVOK_E_NULLPTR;
  if (world < 1 || world > EVOK_MAX_PEERS) return EVOK_E_BADSIZE;
  peer_wait_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(reinterpret_cast<const unsigned long long*>(flags_local), world,
                                                      reinterpret_cast<unsigned long long*>(epoch_dev), err_dev, timeout_ns);
  EVOK_CHECK_LAUNCH();
  return 0;
}

extern "C" EVOK_API int evok_peer_reduce(const float* slots_local, int world, int64_t n, const uint64_t* flags_local, uint64_t* epoch_dev,
                                         uint32_t* done_dev, uint32_t* err_dev, uint64_t timeout_ns, float* out, void* stream) {
  if (!slots_local || !flags_local || !epoch_dev || !done_dev || !err_dev || !out) return EVOK_E_NULLPTR;
  if (world < 1 || world > EVOK_MAX_PEERS || n < 1) return EVOK_E_BADSIZE;
  peer_reduce_kernel<<<(unsigned)((n + kReduceThreads - 1) / kReduceThreads), kReduceThreads, 0, (cudaStream_t)stream>>>(
      slots_local, world, n, reinterpret_cast<const unsigned long long*>(flags_local), reinterpret_cast<unsigned long long*>(epoch_dev), done_dev,
      err_dev, timeout_ns, out);
  EVOK_CHECK_LAUNCH();
  return 0;
}

extern "C" EVOK_API int evok_peer_push(const void* src_local, int64_t n_bytes, int64_t dst_offset_bytes, int world, int rank, void* const* peer_base_host,
                                       void* const* peer_flags_host, const uint64_t* epoch_dev, void* stream) {
  if (!src_local || !peer_base_host || !peer_flags_host || !epoch_dev) return EVOK_E_NULLPTR;
  if (world < 1 || world > EVOK_MAX_PEERS || rank < 0 || rank >= world || n_bytes < 0 || dst_offset_bytes < 0 || (n_bytes & 3)) return EVOK_E_BADSIZE;
  PeerSink sink{};
  sink.world = world;
  sink.rank = rank;
  for (int p = 0; p < world; ++p) {
    if (!peer_base_host[p] || !peer_flags_host[p]) return EVOK_E_NULLPTR;
    sink.data[p] = peer_base_host[p];
    sink.flags[p] = static_cast<unsigned long long*>(peer_flags_host[p]);
  }
  peer_push_kernel<<<world, kPushThreads, 0, (cudaStream_t)stream>>>(static_cast<const unsigned char*>(src_local), n_bytes, dst_offset_bytes, sink,
                                                                    reinterpret_cast<const unsigned long long*>(epoch_dev));
  EVOK_CHECK_LAUNCH();
  return 0;
}
