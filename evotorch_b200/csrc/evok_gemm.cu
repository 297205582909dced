// K6 / K7: fp32-accurate GEMM on the 5th-generation tensor cores (tcgen05 + TMEM + TMA), for the dense contractions of
// CMA-ES (cmaes.py:427 `Y = Z A^T`, :548 rank-mu update `Y^T diag(w) Y`) and XNES.
//
//   C[M x N] = A[M x K] * B[N x K]^T            (A, B row-major with K contiguous: "K-major"; fp32 in, fp32 out)
//
// Accuracy: every fp32 operand x is split as x = hi + lo with hi = x rounded down to TF32 (13 low mantissa bits cleared)
// and lo = x - hi (exact); the kernel accumulates hi*hi + hi*lo + lo*hi in the fp32 TMEM accumulator with
// tcgen05.mma.kind::tf32 ("3xTF32"), which restores ~2^-21 relative accuracy per product -- plain single-pass TF32 (2^-10)
// would break the 1e-5 parity bar of the searchers' state.
//
// Structure (one CTA per 128 x 256 output tile, optional split-K over blockIdx.z):
//   warp 0      TMA producer, 2-stage mbarrier ring.  CONVERT = true (operands 16-byte aligned, the normal case): TWO raw fp32
//               tile loads per K-block (A, B; 128-byte swizzle) -- the tensor core ignores the 13 low mantissa bits of a tf32
//               operand, so the raw tile IS the hi operand, and two converter warps derive the lo tiles (x - trunc(x), same
//               swizzled positions, element-wise) in shared memory while earlier MMAs run: the operands are read from HBM exactly
//               once and no split copies exist.  CONVERT = false (unaligned operands): 4 loads of tiles pre-split by a pre-pass
//   warp 1      TMEM allocation + single-thread tcgen05.mma issue (12 MMAs of 128 x 256 x 8 per K-block),
//               tcgen05.commit releases the stage / signals the epilogue
//   warps 2-3   converters (CONVERT only, see warp 0)
//   warps 4-11  epilogue: the K loop is accumulated in TMEM in chunks of 4 K-blocks (two ping-pong accumulators); each finished
//               chunk is folded into per-thread fp32 REGISTER accumulators (round-to-nearest) via tcgen05.ld, the final tile is
//               written through a shared-memory transpose; optional second output C2 = alpha * acc + bias[col]
#include <cuda.h>

#include <cstdlib>

#include "evok_common.cuh"

namespace evok {

constexpr int kGemmBM = 128;
constexpr int kGemmBN = 256;
constexpr int kGemmBK = 32;  // floats = 128 bytes = one swizzle span
constexpr int kGemmStages = 2;
constexpr int kGemmThreads = 384;  // TMA warp, MMA warp, 2 converter warps, 8 epilogue warps (two aligned warpgroups: warp % 4 = TMEM lane quadrant)
constexpr int kUmmaK = 8;  // tf32: 32 bytes of K per MMA
constexpr uint32_t kTileABytes = kGemmBM * kGemmBK * 4;  // 16 KB
constexpr uint32_t kTileBBytes = kGemmBN * kGemmBK * 4;  // 32 KB
constexpr uint32_t kStageBytes = 2 * kTileABytes + 2 * kTileBBytes;  // 96 KB
constexpr int kEpiPitch = 36;  // floats per row of the epilogue transpose tile (144 B: keeps float4 alignment, spreads banks)
constexpr size_t kGemmSmemBytes = (size_t)kGemmStages * kStageBytes + 1024 /*align slack*/ + 256 /*barriers*/;

// ---- PTX wrappers ---------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t s32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void bar_init(uint64_t* b, uint32_t n) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(s32(b)), "r"(n) : "memory"); }
__device__ __forceinline__ void bar_expect_tx(uint64_t* b, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(s32(b)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bar_wait(uint64_t* b, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}" ::"r"(s32(b)), "r"(parity) : "memory");
}
// The same wait for warps that are NOT on the critical path (the epilogue warps waiting for an accumulator chunk): sleep between polls.  A tight try_wait loop issues continuously, and eight spinning epilogue warps share
// the four schedulers with the two converter warps -- ncu showed the converters issue-starved at 0.13 IPC while the spin loops
// executed more instructions than the rest of the kernel.
__device__ __forceinline__ void bar_wait_relaxed(uint64_t* b, uint32_t parity) {
  for (;;) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n"
        "selp.u32 %0, 1, 0, P1;\n"
        "}"
        : "=r"(ok)
        : "r"(s32(b)), "r"(parity)
        : "memory");
    if (ok) return;
    __nanosleep(200);
  }
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int x, int y, uint64_t* bar) {
  asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::"r"(s32(dst)),
               "l"(reinterpret_cast<uint64_t>(map)), "r"(x), "r"(y), "r"(s32(bar))
               : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s32(dst_smem)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t addr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(s32(bar)) : "memory");
}
// D[tmem] (+)= A[smem desc] * B[smem desc]^T, tf32 inputs, fp32 accumulate
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}" ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, "
      "%28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
        "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
        "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]),
        "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
        "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// shared-memory matrix descriptor of a K-major tile stored as rows of 128 bytes with the 128-byte swizzle
// (cute::UMMA::SmemDescriptor: start>>4 | LBO<<16 | SBO<<32 | version(1)<<46 | layout(SWIZZLE_128B = 2)<<61)
__device__ __forceinline__ uint64_t make_sw128_desc(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;            // leading byte offset (unused for swizzled K-major), canonical value 1
  d |= (uint64_t)(1024 >> 4) << 32;  // stride byte offset: 8 rows x 128 B between core-matrix groups
  d |= (uint64_t)1 << 46;            // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;            // SWIZZLE_128B
  return d;
}
// instruction descriptor (cute::UMMA::InstrDescriptor): D = F32, A = B = TF32, both K-major, M = 128, N = 256
constexpr uint32_t kIdesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(kGemmBN >> 3) << 17) | ((uint32_t)(kGemmBM >> 4) << 24);

// lo = x - trunc_tf32(x) of a whole tile, by 64 threads: thread ct handles the float4 at byte ct * 16 + j * 1024 (addresses in the shared
// window); 16 loads are issued before the first use
template <uint32_t BYTES>
__device__ __forceinline__ void split_lo_tile(uint32_t src, uint32_t dst) {
#pragma unroll
  for (uint32_t b = 0; b < BYTES / 1024u; b += 16) {
    float4 v[16];
#pragma unroll
    for (int j = 0; j < 16; ++j)
      asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v[j].x), "=f"(v[j].y), "=f"(v[j].z), "=f"(v[j].w) : "r"(src + (b + j) * 1024u));
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const float lx = v[j].x - __uint_as_float(__float_as_uint(v[j].x) & 0xFFFFE000u);
      const float ly = v[j].y - __uint_as_float(__float_as_uint(v[j].y) & 0xFFFFE000u);
      const float lz = v[j].z - __uint_as_float(__float_as_uint(v[j].z) & 0xFFFFE000u);
      const float lw = v[j].w - __uint_as_float(__float_as_uint(v[j].w) & 0xFFFFE000u);
      asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(dst + (b + j) * 1024u), "f"(lx), "f"(ly), "f"(lz), "f"(lw) : "memory");
    }
  }
}

// parameters of the generic kernel (gemm_tf32x3_kernel)
struct GemmParams {
  int M, N, K;
  int kblocks_per_split;
  float* C;
  int64_t ldc;
  int64_t split_stride;  // elements between the partial outputs of consecutive K splits
  float* C2;             // optional second output alpha * acc + bias[col]
  int64_t ldc2;
  const float* alpha_dev;
  const float* bias;
  // optional in-place style update  C = k[0] * acc + k[1] * E[i][j] + k[2] * u[i] * u[j]   (k: 3 device floats; CMA-ES covariance
  // update cmaes.py:519-553 with acc = Y^T diag(w) Y, E = old C, u = p_c).  Applied by the epilogue, or by the split-K reduction.
  const float* affine_k;
  const float* affine_E;
  int64_t lde;
  const float* affine_u;
  long long* trace;  // -DEVOK_GEMM_TRACE builds only: clock64() stamps of CTA 0's roles per K-block (scripts/gemm_trace.py)
};

// parameters of the persistent gather kernel (gemm_gather_persistent_kernel, batched policy forward, stacked weight rows): row m of
// the A operand lives at
//   gather_a + (m / ga_rows_per_batch) * ga_batch_stride + (m % ga_rows_per_batch) * ga_row_stride     (any 4-byte alignment)
// and the epilogue applies  act(acc + row_bias[(m / rows_per_batch) * rb_batch_stride + m % rows_per_batch])  and stores it unit-fastest:
//   C[(batch * N + col) * rows_per_batch + row_in_batch]     (one cache line per store instruction)
struct GatherParams {
  int M, N, K;
  float* C;
  const float* gather_a;
  int64_t ga_rows_per_batch, ga_batch_stride, ga_row_stride;
  const float* row_bias;
  int64_t rb_batch_stride;
  int row_act;
  long long* trace;  // -DEVOK_GEMM_TRACE builds only: clock64() stamps of CTA 0's roles per K-block (scripts/gather_trace.py)
};

#ifdef EVOK_GEMM_TRACE
#define EVOK_TRACE(slot, idx)                                                                                      \
  do {                                                                                                             \
    if (p.trace && blockIdx.x == 0 && blockIdx.y == 0 && blockIdx.z == 0 && (idx) < 512u) p.trace[(size_t)(idx) * 16 + (slot)] = clock64();               \
  } while (0)
#else
#define EVOK_TRACE(slot, idx) \
  do {                        \
  } while (0)
#endif

// The tensor core adds every MMA into the TMEM accumulator with round-toward-zero; over hundreds of MMAs that is a
// systematic shrink of ~2e-8 per MMA (measured: -7e-6 relative after 384 MMAs).  The accumulation is therefore CHUNKED:
// kGemmChunk K-blocks (48 MMAs) go into one of two TMEM accumulators, then the epilogue warps fold that partial into
// register accumulators with ordinary round-to-nearest fp32 adds while the MMA warp fills the other TMEM accumulator.
constexpr int kGemmChunk = 4;

template <bool CONVERT>
__global__ void __launch_bounds__(kGemmThreads, 1)
    gemm_tf32x3_kernel(const __grid_constant__ CUtensorMap map_a_hi, const __grid_constant__ CUtensorMap map_a_lo,
                       const __grid_constant__ CUtensorMap map_b_hi, const __grid_constant__ CUtensorMap map_b_lo, const GemmParams p) {
  extern __shared__ unsigned char gemm_smem_raw[];
  // tiles need 1024-byte alignment (swizzle atom)
  unsigned char* base = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(gemm_smem_raw) + 1023) & ~(uintptr_t)1023);
  uint64_t* full = reinterpret_cast<uint64_t*>(base + (size_t)kGemmStages * kStageBytes);
  uint64_t* empty = full + kGemmStages;
  uint64_t* tmem_full = empty + kGemmStages;  // [2]
  uint64_t* tmem_empty = tmem_full + 2;       // [2]
  uint64_t* conv = tmem_empty + 2;            // [kGemmStages] lo tiles of the stage derived (CONVERT)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(conv + kGemmStages);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int m0 = blockIdx.x * kGemmBM, n0 = blockIdx.y * kGemmBN;
  const int total_kb = (p.K + kGemmBK - 1) / kGemmBK;
  const int kb_begin = blockIdx.z * p.kblocks_per_split;
  const int kb_end = min(total_kb, kb_begin + p.kblocks_per_split);
  const int num_kb = max(kb_end - kb_begin, 0);
  const int num_chunks = (num_kb + kGemmChunk - 1) / kGemmChunk;
  if (threadIdx.x == 0) EVOK_TRACE(13, 0u);  // kernel start

  if (threadIdx.x == 0) {
    for (int s = 0; s < kGemmStages; ++s) {
      bar_init(&full[s], 1);
      bar_init(&empty[s], 1);
      bar_init(&conv[s], 2);  // one arrival per converter warp
    }
    for (int t = 0; t < 2; ++t) {
      bar_init(&tmem_full[t], 1);
      bar_init(&tmem_empty[t], 8);  // one arrival per epilogue warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(tmem_slot, 2 * kGemmBN);  // two accumulators of 256 fp32 columns x 128 lanes = all 512 columns
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    if (lane == 0) {
      for (int i = 0; i < num_kb; ++i) {
        const int s = i % kGemmStages;
        const uint32_t use = i / kGemmStages;
        bar_wait(&empty[s], (use & 1) ^ 1);  // first use of a stage passes immediately (tight poll: with two stages the wake-up is on the critical path)
        EVOK_TRACE(9, (uint32_t)i);
        unsigned char* st = base + (size_t)s * kStageBytes;
        bar_expect_tx(&full[s], CONVERT ? kTileABytes + kTileBBytes : kStageBytes);
        const int kx = (kb_begin + i) * kGemmBK;
        tma_load_2d(st, &map_a_hi, kx, m0, &full[s]);
        if (!CONVERT) tma_load_2d(st + kTileABytes, &map_a_lo, kx, m0, &full[s]);
        tma_load_2d(st + 2 * kTileABytes, &map_b_hi, kx, n0, &full[s]);
        if (!CONVERT) tma_load_2d(st + 2 * kTileABytes + kTileBBytes, &map_b_lo, kx, n0, &full[s]);
      }
    }
  } else if (warp == 1) {
    if (lane == 0) {
      for (int i = 0; i < num_kb; ++i) {
        const int s = i % kGemmStages;
        const uint32_t use = i / kGemmStages;
        const int ch = i / kGemmChunk, in_chunk = i % kGemmChunk;
        const int buf = ch & 1;
        if (in_chunk == 0 && ch >= 2) {  // the epilogue must have drained this accumulator (chunk ch - 2)
          bar_wait(&tmem_empty[buf], ((ch >> 1) - 1) & 1);
          tc_fence_after();
        }
        bar_wait(CONVERT ? &conv[s] : &full[s], use & 1);  // CONVERT: the converter warps have derived the lo tiles of this stage
        EVOK_TRACE(6, (uint32_t)i);
        tc_fence_after();
        const uint32_t acc = tmem_base + (uint32_t)(buf * kGemmBN);
        const uint32_t st = s32(base + (size_t)s * kStageBytes);
        const uint64_t a_hi = make_sw128_desc(st), a_lo = make_sw128_desc(st + kTileABytes);
        const uint64_t b_hi = make_sw128_desc(st + 2 * kTileABytes), b_lo = make_sw128_desc(st + 2 * kTileABytes + kTileBBytes);
#pragma unroll
        for (int k = 0; k < kGemmBK / kUmmaK; ++k) {
          const uint64_t adv = (uint64_t)((k * kUmmaK * 4) >> 4);  // advance the start address by 32 bytes per MMA along K
          // small terms first, the dominant hi*hi product last
          umma_tf32(acc, a_hi + adv, b_lo + adv, kIdesc, (in_chunk | k) != 0);
          umma_tf32(acc, a_lo + adv, b_hi + adv, kIdesc, 1);
          umma_tf32(acc, a_hi + adv, b_hi + adv, kIdesc, 1);
        }
        umma_commit(&empty[s]);  // stage reusable once these MMAs have consumed it
        if (in_chunk == kGemmChunk - 1 || i == num_kb - 1) umma_commit(&tmem_full[buf]);  // chunk accumulator complete
        EVOK_TRACE(8, (uint32_t)i);
      }
    }
  } else if (warp < 4) {
    // ===== 2 converter warps (CONVERT): per K-block wait for the raw tiles, derive lo = x - trunc_tf32(x) for both operands
    // (element-wise, so every element simply keeps its swizzled position: 3072 float4 per stage, 48 per thread), publish them to
    // the tensor core (async proxy) and signal the MMA warp.  Runs one or two K-blocks ahead of the MMAs.
    if (CONVERT) {
      const int ct = threadIdx.x - 64;  // 0 .. 63
      for (int i = 0; i < num_kb; ++i) {
        const int s = i % kGemmStages;
        const uint32_t use = i / kGemmStages;
        unsigned char* st = base + (size_t)s * kStageBytes;
        if (threadIdx.x == 64) EVOK_TRACE(0, (uint32_t)i);
        bar_wait(&full[s], use & 1);
        if (threadIdx.x == 64) EVOK_TRACE(1, (uint32_t)i);
        const float4* a_raw = reinterpret_cast<const float4*>(st);
        float4* a_lo = reinterpret_cast<float4*>(st + kTileABytes);
        const float4* b_raw = reinterpret_cast<const float4*>(st + 2 * kTileABytes);
        float4* b_lo = reinterpret_cast<float4*>(st + 2 * kTileABytes + kTileBBytes);
        // (a single warp runs this dependent stream at ~0.2 IPC, so the instruction count per K-block is what matters: shared-space
        // 16-byte loads / stores with immediate offsets, 16 loads in flight)
        split_lo_tile<kTileABytes>(s32(a_raw) + (uint32_t)ct * 16u, s32(a_lo) + (uint32_t)ct * 16u);
        split_lo_tile<kTileBBytes>(s32(b_raw) + (uint32_t)ct * 16u, s32(b_lo) + (uint32_t)ct * 16u);
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy stores -> visible to the tensor core's reads
        __syncwarp();
        if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(s32(&conv[s])) : "memory");
        if (threadIdx.x == 64) EVOK_TRACE(3, (uint32_t)i);
      }
    }
  } else {
    // ===== 8 epilogue warps: TMEM lane quadrant = warp % 4, column half = (warp - 4) / 4 =====
    // Every thread keeps its row's 128 partial sums in REGISTERS and folds each finished TMEM chunk into them with
    // round-to-nearest fp32 adds (no memory traffic); the final tile goes out through a padded shared-memory transpose so that a
    // warp writes 4 rows x 128 contiguous bytes per instruction.
    const int quad = warp & 3, half = (warp - 4) >> 2;
    float acc[kGemmBN / 2];
#pragma unroll
    for (int j = 0; j < kGemmBN / 2; ++j) acc[j] = 0.0f;
    auto fold_chunk = [&](int ch) {
      const int buf = ch & 1;
      if (threadIdx.x == 128) EVOK_TRACE(10, (uint32_t)ch);
      bar_wait_relaxed(&tmem_full[buf], (ch >> 1) & 1);
      if (threadIdx.x == 128) EVOK_TRACE(11, (uint32_t)ch);
      tc_fence_after();
#pragma unroll
      for (int g = 0; g < 4; ++g) {
        uint32_t r[32];
        tmem_ld32(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(buf * kGemmBN + half * (kGemmBN / 2) + g * 32), r);
#pragma unroll
        for (int j = 0; j < 32; ++j) acc[g * 32 + j] += __uint_as_float(r[j]);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(s32(&tmem_empty[buf])) : "memory");
    };
    for (int ch = 0; ch < num_chunks; ++ch) fold_chunk(ch);
    if (threadIdx.x == 128) EVOK_TRACE(13, 1u);  // all chunks folded: the store phase starts
    // all MMAs have completed (the last tmem_full has fired), so the pipeline stages are free: use them as transpose scratch
    float* stile = reinterpret_cast<float*>(base) + (size_t)(warp - 4) * (32 * kEpiPitch);
    const float alpha = (p.C2 && p.alpha_dev) ? *p.alpha_dev : 1.0f;
    const bool affine = p.affine_k != nullptr && gridDim.z == 1;
    const float k0 = affine ? p.affine_k[0] : 1.0f, k1 = affine ? p.affine_k[1] : 0.0f, k2 = affine ? p.affine_k[2] : 0.0f;
    float* cbase = p.C + (int64_t)blockIdx.z * p.split_stride;
    const bool vec_ok = ((reinterpret_cast<uintptr_t>(cbase) & 15) == 0) && (p.ldc % 4 == 0);
    const int sub_row = lane >> 3, sub_col = (lane & 7) * 4;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
#pragma unroll
      for (int j = 0; j < 32; j += 4)
        *reinterpret_cast<float4*>(stile + lane * kEpiPitch + j) = make_float4(acc[g * 32 + j], acc[g * 32 + j + 1], acc[g * 32 + j + 2], acc[g * 32 + j + 3]);
      __syncwarp();
      const int col = n0 + half * (kGemmBN / 2) + g * 32 + sub_col;
#pragma unroll
      for (int it = 0; it < 8; ++it) {
        const int rr = it * 4 + sub_row;
        const int row = m0 + quad * 32 + rr;
        const float4 v = *reinterpret_cast<const float4*>(stile + rr * kEpiPitch + sub_col);
        if (row < p.M) {
          float* cp = cbase + (int64_t)row * p.ldc + col;
          float e[4] = {v.x, v.y, v.z, v.w};
          if (affine) {
            const float ur = p.affine_u ? __ldg(p.affine_u + row) : 0.0f;
            for (int t = 0; t < 4; ++t)
              if (col + t < p.N)
                e[t] = fmaf(k0, e[t], fmaf(k1, p.affine_E ? p.affine_E[(int64_t)row * p.lde + col + t] : 0.0f,
                                          k2 * ur * (p.affine_u ? __ldg(p.affine_u + col + t) : 0.0f)));
          }
          if (!affine && vec_ok && col + 4 <= p.N) {
            *reinterpret_cast<float4*>(cp) = v;
          } else {
            for (int t = 0; t < 4; ++t)
              if (col + t < p.N) cp[t] = e[t];
          }
          if (p.C2) {
            float* c2 = p.C2 + (int64_t)row * p.ldc2 + col;
            for (int t = 0; t < 4; ++t)
              if (col + t < p.N) c2[t] = fmaf(alpha, e[t], p.bias ? __ldg(p.bias + col + t) : 0.0f);
          }
        }
      }
      __syncwarp();
    }
  }
  if (threadIdx.x == 128) EVOK_TRACE(13, 2u);  // stores issued
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 2 * kGemmBN);
  }
}

// ---- persistent gather GEMM (batched policy forward on ONE shared minibatch) ------------------------------------------------
// Same arithmetic as gemm_tf32x3_kernel, for an A operand that is not TMA-addressable (rows only 4-byte aligned, non-uniform pitch: the
// stacked first-layer weights of a population of flat parameter vectors, GatherParams): the two converter warps fetch its tile with
// cp.async row copies and write BOTH the raw and the lo tile in the 128-byte-swizzled layout the tensor core expects, so the weights are
// read from HBM once.  Built for the shape this path has -- millions of A rows, a small B operand (the minibatch) that every tile re-reads:
//   * PERSISTENT: one CTA per SM walks the output tiles (tile = blockIdx.x + q * gridDim.x), so barrier set-up and the TMEM allocation
//     happen once, and the epilogue of tile q (bias, activation, 128 KB of stores) runs while the tensor core is already two
//     accumulator chunks into tile q + 1 (the two TMEM accumulators of the chunked accumulation double as the overlap buffer);
//   * the minibatch is split into hi / lo ONCE by a pre-pass (it is a few hundred KB) and both tiles arrive by TMA: the converter
//     warps only derive the lo tile of the gathered A operand (a third of the element-wise work of the generic kernel);
//   * the gathered A tiles live in a 4-deep ring of raw tiles (three 16 KB gathers in flight per SM while one is converted) with only
//     two lo buffers behind it (a lo tile is derived right before its MMAs); the minibatch tiles (2 stages of hi + lo, 128 KB) come
//     from L2;
//   * the epilogue warps store straight from registers, unit-fastest (GatherParams): the 32 lanes of a warp, consecutive rows of one
//     batch, write 128 consecutive bytes per store instruction.
// the minibatch operand, pre-split into hi / lo and stored four times, copy s shifted right by s floats (xs[b][k'] = x[b][k' - s], zero
// outside): TMA needs 16-byte aligned box coordinates (an odd K coordinate is an illegal instruction), so a tile whose rows sit sh
// floats past a 16-byte boundary reads copy sh at the aligned coordinate 32 i instead of the original at 32 i - sh
struct GatherMaps {
  CUtensorMap hi[4];
  CUtensorMap lo[4];
};

// K-blocks per TMEM accumulator chunk, as in the generic kernel.  (6 -- two chunks per 12-block tile, so that the tensor core could finish
// a whole tile while the epilogue stores the previous one -- was tried: 28.7 vs 29.0 ms, not worth the larger round-toward-zero error.
// The timeline shows why: during the store phase the converter warps themselves slow down 3-5x -- the epilogue's row-per-thread 16-byte
// stores are 32 cache-line operations per warp instruction, 8192 per tile, in the same LSU pipe as the converters' LDS / STS / LDGSTS.)
constexpr int kPersChunk = 4;
constexpr int kPersRawStages = 4, kPersLoStages = 2, kPersBStages = 2;
constexpr uint32_t kPersBStageBytes = 2 * kTileBBytes;
constexpr size_t kPersSmemBytes =
    (size_t)(kPersRawStages + kPersLoStages) * kTileABytes + (size_t)kPersBStages * kPersBStageBytes + 1024 /*align*/ + 256;

__global__ void __launch_bounds__(kGemmThreads, 1)
    gemm_gather_persistent_kernel(const __grid_constant__ GatherMaps maps, const GatherParams p) {
  extern __shared__ unsigned char gemm_smem_raw[];
  unsigned char* base = reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(gemm_smem_raw) + 1023) & ~(uintptr_t)1023);
  unsigned char* raw_base = base;                                             // gathered A tiles (= the hi operand)
  unsigned char* lo_base = base + (size_t)kPersRawStages * kTileABytes;       // their lo tiles
  unsigned char* b_base = lo_base + (size_t)kPersLoStages * kTileABytes;
  uint64_t* full_b = reinterpret_cast<uint64_t*>(b_base + (size_t)kPersBStages * kPersBStageBytes);
  uint64_t* empty_b = full_b + kPersBStages;
  uint64_t* empty_raw = empty_b + kPersBStages;
  uint64_t* empty_lo = empty_raw + kPersRawStages;
  uint64_t* conv_a = empty_lo + kPersLoStages;
  uint64_t* tmem_full = conv_a + kPersLoStages;  // [2]
  uint64_t* tmem_empty = tmem_full + 2;         // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + 2);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // VECTOR mode (rows of K % 4 == 0 floats at pitch K, a tile never straddles two batches): all rows of a tile share one misalignment
  // `sh` (0..3 floats past a 16-byte boundary), so the K axis of that tile is simply cut at 16-byte-aligned source addresses --
  // K-block i covers k = 32 i - sh .. 32 i - sh + 31 for BOTH operands (the minibatch tile comes from the copy shifted by sh floats,
  // GatherMaps; zeros for k < 0 and k >= K) -- and the gather moves 16 bytes per copy.  4-byte cp.async copies turned out to cost ~57 issue
  // cycles per warp instruction (ncu: 70 % of the converter warps' samples sat on the 64 LDGSTS of a K-block), which bounded the
  // whole kernel at 2.6 us per K-block against 0.9 us of tensor-core work.
  const bool vec_mode = (p.K % 4 == 0) && (p.ga_row_stride == p.K) && (p.ga_rows_per_batch % kGemmBM == 0);
  const int num_kb = (p.K + (vec_mode ? 3 : 0) + kGemmBK - 1) / kGemmBK;
  const int num_chunks = (num_kb + kPersChunk - 1) / kPersChunk;
  const int n_tiles = (p.N + kGemmBN - 1) / kGemmBN;
  const int64_t total_tiles = (int64_t)((p.M + kGemmBM - 1) / kGemmBM) * n_tiles;
  auto tile_rows = [&](int64_t t, int& m0, int& sh) -> const float* {  // first row of tile t (VECTOR mode) and its misalignment
    m0 = ((int)t / n_tiles) * kGemmBM;  // (fewer than 2^31 tiles: M < 2^31)
    const int rpb = (int)p.ga_rows_per_batch;
    const int bi = m0 / rpb;
    const float* tb = p.gather_a + (int64_t)bi * p.ga_batch_stride + (int64_t)(m0 - bi * rpb) * p.ga_row_stride;
    sh = vec_mode ? (int)((reinterpret_cast<uintptr_t>(tb) >> 2) & 3) : 0;
    return tb;
  };
  const int64_t my_tiles = total_tiles > blockIdx.x ? (total_tiles - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;

  if (threadIdx.x == 0) {
    for (int s = 0; s < kPersBStages; ++s) {
      bar_init(&full_b[s], 1);
      bar_init(&empty_b[s], 1);
    }
    for (int s = 0; s < kPersRawStages; ++s) bar_init(&empty_raw[s], 1);
    for (int s = 0; s < kPersLoStages; ++s) {
      bar_init(&empty_lo[s], 1);
      bar_init(&conv_a[s], 2);  // one arrival per converter warp
    }
    for (int t = 0; t < 2; ++t) {
      bar_init(&tmem_full[t], 1);
      bar_init(&tmem_empty[t], 8);  // one arrival per epilogue warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(tmem_slot, 2 * kGemmBN);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===== TMA producer of the minibatch tiles (hi, lo) =====
    if (lane == 0) {
      uint32_t g = 0;
      for (int64_t q = 0; q < my_tiles; ++q) {
        const int64_t t = blockIdx.x + q * gridDim.x;
        const int n0 = (int)(t % n_tiles) * kGemmBN;
        int m0_unused, sh;
        tile_rows(t, m0_unused, sh);
        for (int i = 0; i < num_kb; ++i, ++g) {
          const int s = g % kPersBStages;
          bar_wait(&empty_b[s], ((g / kPersBStages) & 1) ^ 1);  // tight poll: the minibatch tile of block g + 2 is needed ~1 block later
          EVOK_TRACE(9, g);
          unsigned char* st = b_base + (size_t)s * kPersBStageBytes;
          bar_expect_tx(&full_b[s], kPersBStageBytes);
          tma_load_2d(st, &maps.hi[sh], i * kGemmBK, n0, &full_b[s]);
          tma_load_2d(st + kTileBBytes, &maps.lo[sh], i * kGemmBK, n0, &full_b[s]);
        }
      }
    }
  } else if (warp == 1) {
    // ===== MMA issue =====
    if (lane == 0) {
      uint32_t g = 0, gch = 0;
      for (int64_t q = 0; q < my_tiles; ++q) {
        for (int i = 0; i < num_kb; ++i, ++g) {
          const int sr = g % kPersRawStages, sl = g % kPersLoStages, sb = g % kPersBStages;
          const int in_chunk = i % kPersChunk;
          const int buf = gch & 1;
          if (in_chunk == 0 && gch >= 2) {  // the epilogue must have folded the chunk that used this accumulator (two chunks ago)
            bar_wait(&tmem_empty[buf], ((gch >> 1) - 1) & 1);
            tc_fence_after();
          }
          bar_wait(&conv_a[sl], (g / kPersLoStages) & 1);
          EVOK_TRACE(6, g);
          bar_wait(&full_b[sb], (g / kPersBStages) & 1);
          EVOK_TRACE(7, g);
          tc_fence_after();
          const uint32_t acc = tmem_base + (uint32_t)(buf * kGemmBN);
          const uint32_t stb = s32(b_base + (size_t)sb * kPersBStageBytes);
          const uint64_t a_hi = make_sw128_desc(s32(raw_base + (size_t)sr * kTileABytes));
          const uint64_t a_lo = make_sw128_desc(s32(lo_base + (size_t)sl * kTileABytes));
          const uint64_t b_hi = make_sw128_desc(stb), b_lo = make_sw128_desc(stb + kTileBBytes);
#pragma unroll
          for (int k = 0; k < kGemmBK / kUmmaK; ++k) {
            const uint64_t adv = (uint64_t)((k * kUmmaK * 4) >> 4);
            umma_tf32(acc, a_hi + adv, b_lo + adv, kIdesc, (in_chunk | k) != 0);
            umma_tf32(acc, a_lo + adv, b_hi + adv, kIdesc, 1);
            umma_tf32(acc, a_hi + adv, b_hi + adv, kIdesc, 1);
          }
          umma_commit(&empty_raw[sr]);
          umma_commit(&empty_lo[sl]);
          umma_commit(&empty_b[sb]);
          EVOK_TRACE(8, g);
          if (in_chunk == kPersChunk - 1 || i == num_kb - 1) {
            umma_commit(&tmem_full[buf]);
            ++gch;
          }
        }
      }
    }
  } else if (warp < 4) {
    // ===== 2 converter warps: gather the A tile of K-block g (64 rows per warp), derive its lo tile =====
    // One warp executes a dependent instruction stream at ~0.2 IPC, so what bounds this role is its instruction COUNT per K-block:
    // everything that does not change between K-blocks is hoisted (lane offsets, per-tile base / misalignment), shared memory is
    // addressed through 32-bit shared-space addresses (LDS / STS / LDGSTS with immediate offsets), and the rare cases (first chunk of a
    // misaligned row, partial tiles) live in their own branches.
    const int ct = threadIdx.x - 64;
    const uint32_t total_g = (uint32_t)(my_tiles * num_kb);
    const int wrow0 = (warp - 2) * 64;
    const uint32_t raw_s = s32(raw_base), lo_s = s32(lo_base);
    // the issue cursor (tile, K-block) with the per-tile constants of its tile
    int64_t is_t = blockIdx.x;
    int is_i = 0, is_m0 = 0, is_sh = 0;
    const float* is_base = p.gather_a;
    if (my_tiles > 0) is_base = tile_rows(is_t, is_m0, is_sh);
    // VECTOR mode: lane = (row within a group of 4, 16-byte chunk c of the 128-byte row segment); rows wrow0 + 8 j + rsub ("even") and
    // wrow0 + 8 j + 4 + rsub ("odd") for j = 0..7; chunk c of row r sits at r * 128 + ((c ^ (r % 8)) << 4)
    const int c = lane & 7, rsub = lane >> 3;
    const uint32_t off_even = (uint32_t)(wrow0 + rsub) * 128u + ((uint32_t)(c ^ rsub) << 4);
    const uint32_t off_odd = (uint32_t)(wrow0 + 4 + rsub) * 128u + ((uint32_t)(c ^ (4 + rsub)) << 4);
    // 4-byte mode: lane = column of the K-block; element (r, lane) sits at r * 128 + sw[r % 8]
    uint32_t sw[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) sw[j] = ((((uint32_t)lane >> 2) ^ (uint32_t)j) << 4) + (((uint32_t)lane & 3u) << 2);
    const bool rows_regular = (p.ga_rows_per_batch % 64) == 0;  // a warp's 64 rows never straddle two batches
    auto issue_gather = [&](uint32_t g) {
      const int s = g % kPersRawStages;
      bar_wait(&empty_raw[s], ((g / kPersRawStages) & 1) ^ 1);
      if (threadIdx.x == 64) EVOK_TRACE(4, g);
      const uint32_t st_a = raw_s + (uint32_t)s * kTileABytes;
      const int i = is_i, m0 = is_m0;
      if (vec_mode) {
        const int k_first = i * kGemmBK + 4 * c - is_sh;  // first element of this lane's chunk (16-byte aligned in memory)
        if (k_first >= 0 && m0 + kGemmBM <= p.M) {
          const uint32_t sz = (uint32_t)min(max(p.K - k_first, 0), 4) * 4u;  // bytes read; the rest of the 16 is zero-filled
          const float* src = sz ? is_base + (int64_t)(wrow0 + rsub) * p.K + k_first : is_base - is_sh;  // (any aligned address if sz = 0)
          const int64_t pitch4 = sz ? 4 * (int64_t)p.K : 0;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(st_a + off_even + (uint32_t)j * 1024u), "l"(src + (2 * j) * pitch4),
                         "r"(sz)
                         : "memory");
            asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(st_a + off_odd + (uint32_t)j * 1024u),
                         "l"(src + (2 * j + 1) * pitch4), "r"(sz)
                         : "memory");
          }
        } else {
          // the chunk in front of a misaligned row (K-block 0: its first sh floats are NOT this row's -- they are zeroed rather than
          // left to the minibatch's zero fill, a NaN there would leak into the row), and the rows of a partial last tile
#pragma unroll 1
          for (int it = 0; it < 16; ++it) {
            const int r = wrow0 + it * 4 + rsub;
            const bool row_ok = m0 + r < p.M;
            const uint32_t dst = st_a + (uint32_t)r * 128u + ((uint32_t)(c ^ (r & 7)) << 4);
            const float* src = is_base + (int64_t)r * p.K + k_first;
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const bool ok = row_ok && (k_first + e >= 0) && (k_first + e < p.K);
              asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst + 4u * e), "l"(ok ? src + e : p.gather_a), "r"(ok ? 4 : 0)
                           : "memory");
            }
          }
        }
      } else {
        const int kcol = i * kGemmBK + lane;
        const bool k_ok = kcol < p.K;
        const int m_first = m0 + wrow0;
        const uint32_t dst0 = st_a + (uint32_t)wrow0 * 128u;
        const int rpb = (int)p.ga_rows_per_batch;
        int hrow = m_first % rpb;
        const float* rowp = p.gather_a + (int64_t)(m_first / rpb) * p.ga_batch_stride + (int64_t)hrow * p.ga_row_stride + kcol;
        if (rows_regular && m_first + 64 <= p.M) {
          const float* src = k_ok ? rowp : p.gather_a;
          const int64_t pitch = k_ok ? p.ga_row_stride : 0;
          const uint32_t sz = k_ok ? 4u : 0u;
#pragma unroll
          for (int it = 0; it < 64; ++it)
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst0 + (uint32_t)it * 128u + sw[it & 7]), "l"(src + it * pitch), "r"(sz)
                         : "memory");
        } else {
          const int64_t wrap = p.ga_batch_stride - p.ga_rows_per_batch * p.ga_row_stride;
#pragma unroll 8
          for (int it = 0; it < 64; ++it) {
            const bool ok = k_ok && (m_first + it < p.M);
            const float* src = ok ? rowp : p.gather_a;
            asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst0 + (uint32_t)it * 128u + sw[it & 7]), "l"(src), "r"(ok ? 4 : 0)
                         : "memory");
            rowp += p.ga_row_stride;
            if (++hrow == rpb) {
              hrow = 0;
              rowp += wrap;
            }
          }
        }
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
      if (++is_i == num_kb) {  // the cursor moves on to the next tile of this CTA
        is_i = 0;
        is_t += gridDim.x;
        if (is_t < total_tiles) is_base = tile_rows(is_t, is_m0, is_sh);
      }
    };
    if (total_g > 0) issue_gather(0);
    if (total_g > 1) issue_gather(1);
    if (total_g > 2) issue_gather(2);
    for (uint32_t g = 0; g < total_g; ++g) {
      const int sr = g % kPersRawStages, sl = g % kPersLoStages;
      if (threadIdx.x == 64) EVOK_TRACE(0, g);
      // block g has landed (blocks g + 1, g + 2 may still be in flight)
      if (g + 2 < total_g) asm volatile("cp.async.wait_group 2;" ::: "memory");
      else if (g + 1 < total_g) asm volatile("cp.async.wait_group 1;" ::: "memory");
      else asm volatile("cp.async.wait_group 0;" ::: "memory");
      if (threadIdx.x == 64) EVOK_TRACE(14, g);
      asm volatile("bar.sync 1, 64;" ::: "memory");  // ... and so have the other converter warp's rows
      if (threadIdx.x == 64) EVOK_TRACE(1, g);
      bar_wait(&empty_lo[sl], ((g / kPersLoStages) & 1) ^ 1);  // the MMAs of block g - 2 are done with this lo buffer
      if (threadIdx.x == 64) EVOK_TRACE(2, g);
      // lo = x - trunc_tf32(x), element-wise (every element keeps its swizzled position): 16 float4 per thread, all loads first
      const uint32_t ra = raw_s + (uint32_t)sr * kTileABytes + (uint32_t)ct * 16u, la = lo_s + (uint32_t)sl * kTileABytes + (uint32_t)ct * 16u;
      split_lo_tile<kTileABytes>(ra, la);
      asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
      __syncwarp();
      if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(s32(&conv_a[sl])) : "memory");
      if (threadIdx.x == 64) EVOK_TRACE(3, g);
      if (g + 3 < total_g) issue_gather(g + 3);
      if (threadIdx.x == 64) EVOK_TRACE(5, g);
    }
  } else {
    // ===== 8 epilogue warps: TMEM lane quadrant = warp % 4 (tile row = quadrant * 32 + lane), column half = (warp - 4) / 4 =====
    const int quad = warp & 3, half = (warp - 4) >> 2;
    uint32_t gch = 0;
    for (int64_t q = 0; q < my_tiles; ++q) {
      const int64_t t = blockIdx.x + q * gridDim.x;
      const int m0 = (int)(t / n_tiles) * kGemmBM, n0 = (int)(t % n_tiles) * kGemmBN;
      float acc[kGemmBN / 2];
#pragma unroll
      for (int j = 0; j < kGemmBN / 2; ++j) acc[j] = 0.0f;
      for (int ch = 0; ch < num_chunks; ++ch, ++gch) {
        const int buf = gch & 1;
        if (threadIdx.x == 128) EVOK_TRACE(10, gch);
        bar_wait_relaxed(&tmem_full[buf], (gch >> 1) & 1);
        if (threadIdx.x == 128) EVOK_TRACE(11, gch);
        tc_fence_after();
#pragma unroll
        for (int g8 = 0; g8 < 8; ++g8) {
          uint32_t r[16];
          tmem_ld16(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(buf * kGemmBN + half * (kGemmBN / 2) + g8 * 16), r);
#pragma unroll
          for (int j = 0; j < 16; ++j) acc[g8 * 16 + j] += __uint_as_float(r[j]);
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(s32(&tmem_empty[buf])) : "memory");
        if (threadIdx.x == 128) EVOK_TRACE(12, gch);
      }
      const int64_t m = (int64_t)m0 + quad * 32 + lane;
      if (m < p.M) {
        float b = 0.0f;
        if (p.row_bias) {
          const int64_t bi = m / p.ga_rows_per_batch;
          b = __ldg(p.row_bias + bi * p.rb_batch_stride + (m - bi * p.ga_rows_per_batch));
        }
        // bias + activation applied four values at a time on the way out; one unrolled copy of the store loop per activation (a
        // per-element switch would not fit the instruction cache)
        const int col0 = n0 + half * (kGemmBN / 2);
        // unit-fastest layout: the 32 lanes of a warp (consecutive rows of one batch) write 128 consecutive bytes per instruction
        const int64_t bi_c = m / p.ga_rows_per_batch;
        float* ccol = p.C + (bi_c * p.N + col0) * p.ga_rows_per_batch + (m - bi_c * p.ga_rows_per_batch);
        const int64_t cstride = p.ga_rows_per_batch;
        // (the full-width case stores unconditionally: with only per-element guards the compiler moves each activation under its
        // own branch and the four no longer overlap -- measured 2 % slower over the whole forward)
        auto store4 = [&](int j, float v0, float v1, float v2, float v3) {
          const int col = col0 + j;
          const float v[4] = {v0, v1, v2, v3};
          if (col + 4 <= p.N) {
#pragma unroll
            for (int u = 0; u < 4; ++u) ccol[(int64_t)(j + u) * cstride] = v[u];
          } else {
#pragma unroll
            for (int u = 0; u < 4; ++u)
              if (col + u < p.N) ccol[(int64_t)(j + u) * cstride] = v[u];
          }
        };
        if (p.row_act == EVOK_ACT_NONE) {
#pragma unroll
          for (int j = 0; j < kGemmBN / 2; j += 4) store4(j, acc[j] + b, acc[j + 1] + b, acc[j + 2] + b, acc[j + 3] + b);
        } else if (p.row_act == EVOK_ACT_RELU) {
#pragma unroll
          for (int j = 0; j < kGemmBN / 2; j += 4)
            store4(j, fmaxf(acc[j] + b, 0.0f), fmaxf(acc[j + 1] + b, 0.0f), fmaxf(acc[j + 2] + b, 0.0f), fmaxf(acc[j + 3] + b, 0.0f));
        } else if (p.row_act == EVOK_ACT_TANH) {
#pragma unroll
          for (int j = 0; j < kGemmBN / 2; j += 4)
            store4(j, tanh_abs1e7(acc[j] + b), tanh_abs1e7(acc[j + 1] + b), tanh_abs1e7(acc[j + 2] + b), tanh_abs1e7(acc[j + 3] + b));
        } else {
#pragma unroll
          for (int j = 0; j < kGemmBN / 2; j += 4)
            store4(j, activate_fast(acc[j] + b, EVOK_ACT_SIGMOID), activate_fast(acc[j + 1] + b, EVOK_ACT_SIGMOID),
                   activate_fast(acc[j + 2] + b, EVOK_ACT_SIGMOID), activate_fast(acc[j + 3] + b, EVOK_ACT_SIGMOID));
        }
      }
    }
  }
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 2 * kGemmBN);
  }
}

// ---- operand preparation -----------------------------------------------------------------------------------------
// hi = x with the 13 low mantissa bits cleared (exactly representable in TF32), lo = x - hi (exact in fp32)
__global__ void __launch_bounds__(256) split_tf32_kernel(const float* __restrict__ x, int64_t ldx, int64_t rows, int64_t cols, float* __restrict__ hi,
                                                         float* __restrict__ lo, int64_t ldo) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * cols) return;
  const int64_t r = i / cols, c = i % cols;
  const float v = x[r * ldx + c];
  const float h = __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
  hi[r * ldo + c] = h;
  lo[r * ldo + c] = v - h;
}

// the four shifted hi / lo copies of the minibatch (GatherMaps): hi[s][r][c] / lo[s][r][c] of x[r][c - s], zero for c - s outside [0, cols)
__global__ void __launch_bounds__(256) split_shifted_kernel(const float* __restrict__ x, int64_t ldx, int64_t rows, int64_t cols, float* __restrict__ hi,
                                                            float* __restrict__ lo, int64_t ldo) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= 4 * rows * ldo) return;
  const int64_t s = i / (rows * ldo), rem = i - s * rows * ldo;
  const int64_t r = rem / ldo, c = rem - r * ldo - s;
  const float v = (c >= 0 && c < cols) ? x[r * ldx + c] : 0.0f;
  const float h = __uint_as_float(__float_as_uint(v) & 0xFFFFE000u);
  hi[i] = h;
  lo[i] = v - h;
}

// out[c, r] = (w ? w[r] : 1) * in[r, c]   (32 x 32 tiles through shared memory)
__global__ void __launch_bounds__(256) transpose_scale_kernel(const float* __restrict__ in, int64_t ldi, int64_t rows, int64_t cols,
                                                              const float* __restrict__ w, float* __restrict__ out, int64_t ldo) {
  __shared__ float tile[32][33];
  const int64_t r0 = (int64_t)blockIdx.y * 32, c0 = (int64_t)blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int k = ty; k < 32; k += 8) {
    const int64_t r = r0 + k, c = c0 + tx;
    tile[k][tx] = (r < rows && c < cols) ? in[r * ldi + c] * (w ? w[r] : 1.0f) : 0.0f;
  }
  __syncthreads();
  for (int k = ty; k < 32; k += 8) {
    const int64_t c = c0 + k, r = r0 + tx;
    if (c < cols && r < rows) out[c * ldo + r] = tile[tx][k];
  }
}

__global__ void __launch_bounds__(256) reduce_splits_kernel(const float* __restrict__ partial, int splits, int64_t split_stride, int64_t M,
                                                            int64_t N, int64_t ldp, float* C, int64_t ldc, const float* __restrict__ affine_k,
                                                            const float* affine_E, int64_t lde, const float* __restrict__ affine_u) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M * N) return;
  const int64_t r = i / N, c = i % N;
  float acc = 0.0f;
  for (int s = 0; s < splits; ++s) acc += partial[(int64_t)s * split_stride + r * ldp + c];
  if (affine_k) {  // same update as the epilogue's (GemmParams::affine_*); E may alias C (element read before it is written)
    const float e = affine_E ? affine_E[r * lde + c] : 0.0f;
    const float uu = affine_u ? affine_u[r] * affine_u[c] : 0.0f;
    acc = fmaf(affine_k[0], acc, fmaf(affine_k[1], e, affine_k[2] * uu));
  }
  C[r * ldc + c] = acc;
}

// Operands of the weighted SYRK  S = Y^T diag(w) Y  as K-major matrices (K = the population axis), built in ONE pass over Y:
//   out_w[c, r] = w[r] * Y[r, c]      out_p[c, r] = Y[r, c]          (32 x 32 tiles through shared memory)
__global__ void __launch_bounds__(256) transpose_pair_kernel(const float* __restrict__ in, int64_t ldi, int64_t rows, int64_t cols,
                                                             const float* __restrict__ w, float* __restrict__ out_w, float* __restrict__ out_p,
                                                             int64_t ldo) {
  __shared__ float tile[32][33];
  __shared__ float wrow[32];
  const int64_t r0 = (int64_t)blockIdx.y * 32, c0 = (int64_t)blockIdx.x * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  if (ty == 0) wrow[tx] = (r0 + tx < rows) ? w[r0 + tx] : 0.0f;
  for (int k = ty; k < 32; k += 8) {
    const int64_t r = r0 + k, c = c0 + tx;
    tile[k][tx] = (r < rows && c < cols) ? in[r * ldi + c] : 0.0f;
  }
  __syncthreads();
  for (int k = ty; k < 32; k += 8) {
    const int64_t c = c0 + k, r = r0 + tx;
    if (c < cols && r < rows) {
      const float v = tile[tx][k];
      out_p[c * ldo + r] = v;
      out_w[c * ldo + r] = v * wrow[tx];
    }
  }
}

// ---- host side -------------------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
  }
  return fn;
}

// 2-D fp32 tensor [rows x K], K contiguous (pitch ld floats); box = 32 floats (128 B) x box_rows; 128-byte swizzle
static int make_map(CUtensorMap* map, const float* ptr, int64_t rows, int64_t K, int64_t ld, int box_rows) {
  EncodeTiledFn enc = get_encode_fn();
  if (!enc) return (int)cudaErrorNotSupported;
  const cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)ld * sizeof(float)};
  const cuuint32_t box[2] = {(cuuint32_t)kGemmBK, (cuuint32_t)box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                         CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : (int)cudaErrorInvalidValue;
}

static inline int64_t round_up(int64_t x, int64_t m) { return (x + m - 1) / m * m; }

struct GemmPlan {
  int64_t ldk;  // pitch of the split operands (floats), multiple of 4
  int splits, kblocks_per_split;
  size_t off_a_hi, off_a_lo, off_b_hi, off_b_lo, off_partial, total;
};

static GemmPlan plan_gemm(int64_t M, int64_t N, int64_t K, bool allow_split = true) {
  GemmPlan g;
  g.ldk = round_up(K, 4);
  const int64_t tiles = ((M + kGemmBM - 1) / kGemmBM) * ((N + kGemmBN - 1) / kGemmBN);
  const int total_kb = (int)((K + kGemmBK - 1) / kGemmBK);
  int splits = 1;
  while (allow_split && tiles * splits * 2 <= kNumSMs && splits * 2 <= total_kb && splits < 16) splits *= 2;
  g.kblocks_per_split = (total_kb + splits - 1) / splits;
  g.splits = (total_kb + g.kblocks_per_split - 1) / g.kblocks_per_split;
  auto al = [](size_t x) { return (x + 1023) & ~(size_t)1023; };
  size_t o = 0;
  g.off_a_hi = o; o += al((size_t)M * g.ldk * 4);
  g.off_a_lo = o; o += al((size_t)M * g.ldk * 4);
  g.off_b_hi = o; o += al((size_t)N * g.ldk * 4);
  g.off_b_lo = o; o += al((size_t)N * g.ldk * 4);
  g.off_partial = o; o += g.splits > 1 ? al((size_t)g.splits * M * N * 4) : 0;
  g.total = o;
  return g;
}

}  // namespace evok

using namespace evok;

extern "C" EVOK_API size_t evok_gemm_workspace_bytes(int64_t M, int64_t N, int64_t K) {
  if (M <= 0 || N <= 0 || K <= 0) return 1024;
  return plan_gemm(M, N, K).total + 1024;
}

struct GemmAffine {
  const float* k;
  const float* E;
  int64_t lde;
  const float* u;
};

static bool tma_ok(const float* p, int64_t ld) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0 && ld % 4 == 0; }

static int gemm_impl(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t M, int64_t N, int64_t K, float* C, int64_t ldc, float* C2,
                     int64_t ldc2, const float* alpha_dev, const float* bias, const GemmAffine* aff, void* ws, size_t ws_bytes, void* stream) {
  if (!A || !B || !C || !ws) return EVOK_E_NULLPTR;
  if (M <= 0 || N <= 0 || K <= 0 || lda < K || ldb < K || ldc < N || (C2 && ldc2 < N)) return EVOK_E_BADSIZE;
  if (M >= (1ll << 31) || N >= (1ll << 31) || K >= (1ll << 31)) return EVOK_E_BADSIZE;
  if (aff && (!aff->k || (aff->u && M != N) || (aff->E && aff->lde < N))) return EVOK_E_BADSIZE;
  const GemmPlan g = plan_gemm(M, N, K, C2 == nullptr);  // the fused second output needs the whole K range in one CTA
  char* w8 = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(ws) + 1023) & ~(uintptr_t)1023);
  if (ws_bytes < g.total + (size_t)(w8 - (char*)ws)) return EVOK_E_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  float* partial = (float*)(w8 + g.off_partial);
  // Operands that TMA can address directly (16-byte aligned base and pitch: every matrix this package allocates) are read from
  // HBM once, by the GEMM itself, which derives the lo halves in shared memory; otherwise a pre-pass writes aligned split copies.
  const bool convert = tma_ok(A, lda) && tma_ok(B, ldb);
  CUtensorMap ma_hi, ma_lo, mb_hi, mb_lo;
  int rc;
  if (convert) {
    if ((rc = make_map(&ma_hi, A, M, K, lda, kGemmBM))) return rc;
    if ((rc = make_map(&mb_hi, B, N, K, ldb, kGemmBN))) return rc;
    ma_lo = ma_hi;
    mb_lo = mb_hi;
  } else {
    float* a_hi = (float*)(w8 + g.off_a_hi);
    float* a_lo = (float*)(w8 + g.off_a_lo);
    float* b_hi = (float*)(w8 + g.off_b_hi);
    float* b_lo = (float*)(w8 + g.off_b_lo);
    split_tf32_kernel<<<(unsigned)((M * K + 255) / 256), 256, 0, st>>>(A, lda, M, K, a_hi, a_lo, g.ldk);
    split_tf32_kernel<<<(unsigned)((N * K + 255) / 256), 256, 0, st>>>(B, ldb, N, K, b_hi, b_lo, g.ldk);
    EVOK_CHECK_LAUNCH_N(2);
    if ((rc = make_map(&ma_hi, a_hi, M, K, g.ldk, kGemmBM))) return rc;
    if ((rc = make_map(&ma_lo, a_lo, M, K, g.ldk, kGemmBM))) return rc;
    if ((rc = make_map(&mb_hi, b_hi, N, K, g.ldk, kGemmBN))) return rc;
    if ((rc = make_map(&mb_lo, b_lo, N, K, g.ldk, kGemmBN))) return rc;
  }
  GemmParams p;
  p.M = (int)M; p.N = (int)N; p.K = (int)K;
  p.kblocks_per_split = g.kblocks_per_split;
  const bool split = g.splits > 1;
  p.C = split ? partial : C;
  p.ldc = split ? N : ldc;
  p.split_stride = split ? M * N : 0;
  p.C2 = split ? nullptr : C2;
  p.ldc2 = ldc2;
  p.alpha_dev = alpha_dev;
  p.bias = bias;
  p.affine_k = (aff && !split) ? aff->k : nullptr;
  p.affine_E = aff ? aff->E : nullptr;
  p.lde = aff ? aff->lde : 0;
  p.affine_u = aff ? aff->u : nullptr;
  p.trace = nullptr;
#ifdef EVOK_GEMM_TRACE
  {
    const char* e = getenv("EVOK_GATHER_TRACE_PTR");
    p.trace = e ? reinterpret_cast<long long*>(strtoull(e, nullptr, 16)) : nullptr;
  }
#endif
  static bool attr_set = false;
  if (!attr_set) {
    if (cudaFuncSetAttribute(gemm_tf32x3_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGemmSmemBytes) != cudaSuccess ||
        cudaFuncSetAttribute(gemm_tf32x3_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kGemmSmemBytes) != cudaSuccess)
      return (int)cudaGetLastError();
    attr_set = true;
  }
  dim3 grid((unsigned)((M + kGemmBM - 1) / kGemmBM), (unsigned)((N + kGemmBN - 1) / kGemmBN), (unsigned)g.splits);
  if (convert) gemm_tf32x3_kernel<true><<<grid, kGemmThreads, kGemmSmemBytes, st>>>(ma_hi, ma_lo, mb_hi, mb_lo, p);
  else gemm_tf32x3_kernel<false><<<grid, kGemmThreads, kGemmSmemBytes, st>>>(ma_hi, ma_lo, mb_hi, mb_lo, p);
  EVOK_CHECK_LAUNCH();
  if (split) {
    reduce_splits_kernel<<<(unsigned)((M * N + 255) / 256), 256, 0, st>>>(partial, g.splits, M * N, M, N, N, C, ldc, aff ? aff->k : nullptr,
                                                                          aff ? aff->E : nullptr, aff ? aff->lde : 0, aff ? aff->u : nullptr);
    EVOK_CHECK_LAUNCH();
  }
  return 0;
}

extern "C" EVOK_API int evok_gemm_nt(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t M, int64_t N, int64_t K, float* C,
                                     int64_t ldc, float* C2, int64_t ldc2, const float* alpha_dev, const float* bias, void* ws, size_t ws_bytes,
                                     void* stream) {
  return gemm_impl(A, lda, B, ldb, M, N, K, C, ldc, C2, ldc2, alpha_dev, bias, nullptr, ws, ws_bytes, stream);
}

extern "C" EVOK_API int evok_gemm_nt_affine(const float* A, int64_t lda, const float* B, int64_t ldb, int64_t M, int64_t N, int64_t K, float* C,
                                            int64_t ldc, const float* k_dev, const float* E, int64_t lde, const float* u, void* ws, size_t ws_bytes,
                                            void* stream) {
  if (!k_dev) return EVOK_E_NULLPTR;
  const GemmAffine aff{k_dev, E, lde, u};
  return gemm_impl(A, lda, B, ldb, M, N, K, C, ldc, nullptr, 0, nullptr, nullptr, &aff, ws, ws_bytes, stream);
}

// Stacked-rows GEMM of the batched policy forward (declared in evok_common.cuh) on the persistent kernel: X is split into four shifted
// hi / lo copies in `ws` first, so any alignment / pitch of X is fine.
size_t evok::gemm_gather_rows_workspace_bytes(int64_t n_cols, int64_t K) {
  if (n_cols <= 0 || K <= 0) return 512;
  return (size_t)8 * n_cols * round_up(K + 3, 4) * sizeof(float) + 512;  // 4 shifted copies of the hi and of the lo part
}

int evok::gemm_gather_rows_ws(const float* params, int64_t batch_stride, int64_t w_offset, int64_t rows_per_batch, int64_t n_batches,
                              const float* X, int64_t ldx, int64_t n_cols, int64_t K, int64_t bias_offset, int act, float* C, void* ws,
                              size_t ws_bytes, void* stream) {
  if (!params || !X || !C || !ws) return EVOK_E_NULLPTR;
  const int64_t M = rows_per_batch * n_batches;
  if (rows_per_batch <= 0 || n_batches <= 0 || n_cols <= 0 || K <= 0 || ldx < K || M >= (1ll << 31)) return EVOK_E_BADSIZE;
  if (act < EVOK_ACT_NONE || act > EVOK_ACT_SIGMOID) return EVOK_E_BADENUM;
  const int64_t ldk = round_up(K + 3, 4);
  char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
  if (ws_bytes < (size_t)(base - (char*)ws) + (size_t)8 * n_cols * ldk * sizeof(float)) return EVOK_E_WORKSPACE;
  float* x_hi = reinterpret_cast<float*>(base);
  float* x_lo = x_hi + 4 * n_cols * ldk;
  split_shifted_kernel<<<(unsigned)((4 * n_cols * ldk + 255) / 256), 256, 0, (cudaStream_t)stream>>>(X, ldx, n_cols, K, x_hi, x_lo, ldk);
  EVOK_CHECK_LAUNCH();
  GatherMaps maps;
  int rc;
  for (int s = 0; s < 4; ++s) {
    if ((rc = make_map(&maps.hi[s], x_hi + s * n_cols * ldk, n_cols, ldk, ldk, kGemmBN))) return rc;
    if ((rc = make_map(&maps.lo[s], x_lo + s * n_cols * ldk, n_cols, ldk, ldk, kGemmBN))) return rc;
  }
  GatherParams p{};
  p.M = (int)M; p.N = (int)n_cols; p.K = (int)K;
  p.C = C;
  p.gather_a = params + w_offset;
  p.ga_rows_per_batch = rows_per_batch;
  p.ga_batch_stride = batch_stride;
  p.ga_row_stride = K;
  p.row_bias = bias_offset >= 0 ? params + bias_offset : nullptr;
  p.rb_batch_stride = batch_stride;
  p.row_act = act;
#ifdef EVOK_GEMM_TRACE
  {
    const char* e = getenv("EVOK_GATHER_TRACE_PTR");  // device pointer (hex) of a 512 x 16 int64 buffer
    p.trace = e ? reinterpret_cast<long long*>(strtoull(e, nullptr, 16)) : nullptr;
  }
#endif
  static int sm_count = 0;
  if (!sm_count) {
    int dev = 0;
    cudaGetDevice(&dev);
    if (cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || sm_count <= 0) sm_count = 148;
    if (cudaFuncSetAttribute(gemm_gather_persistent_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPersSmemBytes) != cudaSuccess) {
      sm_count = 0;
      return (int)cudaGetLastError();
    }
  }
  const int64_t tiles = ((M + kGemmBM - 1) / kGemmBM) * ((n_cols + kGemmBN - 1) / kGemmBN);
  const unsigned grid = (unsigned)(tiles < sm_count ? tiles : sm_count);
  gemm_gather_persistent_kernel<<<grid, kGemmThreads, kPersSmemBytes, (cudaStream_t)stream>>>(maps, p);
  EVOK_CHECK_LAUNCH();
  return 0;
}

extern "C" EVOK_API int evok_transpose_pair(const float* in, int64_t ldi, int64_t rows, int64_t cols, const float* w, float* out_w, float* out_p,
                                            int64_t ldo, void* stream) {
  if (!in || !w || !out_w || !out_p) return EVOK_E_NULLPTR;
  if (rows <= 0 || cols <= 0 || ldi < cols || ldo < rows) return EVOK_E_BADSIZE;
  dim3 grid((unsigned)((cols + 31) / 32), (unsigned)((rows + 31) / 32));
  transpose_pair_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(in, ldi, rows, cols, w, out_w, out_p, ldo);
  EVOK_CHECK_LAUNCH();
  return 0;
}

extern "C" EVOK_API int evok_transpose_scale(const float* in, int64_t ldi, int64_t rows, int64_t cols, const float* w, float* out, int64_t ldo,
                                             void* stream) {
  if (!in || !out) return EVOK_E_NULLPTR;
  if (rows <= 0 || cols <= 0 || ldi < cols || ldo < rows) return EVOK_E_BADSIZE;
  dim3 grid((unsigned)((cols + 31) / 32), (unsigned)((rows + 31) / 32));
  transpose_scale_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(in, ldi, rows, cols, w, out, ldo);
  EVOK_CHECK_LAUNCH();
  return 0;
}
