// K8: batched flat-parameter MLP policy forward -- one observation per policy (the reference's `Policy.__call__`,
// neuroevolution/net/vecrl.py:1240-1279, which vmaps `functional_call` over the rows of an N x L parameter matrix).
// Every policy has its OWN weights, so this is a batched GEMV: 0.5 flop per parameter byte, i.e. purely HBM-read bound
// (26.4 GB of parameters at N = 65 536, L = 100 881).  Tensor cores cannot help: no operand is shared between rows.
//
// Layout of a parameter row (net/functional.py:118-129, torch.nn.Linear order): for each layer, W (out x in, row-major)
// then b (out).  L is odd in general (100 881), so rows are only 4-byte aligned: the kernel reads weights with coalesced
// 32-bit loads (a warp covers 128 contiguous bytes per instruction, 4 neuron rows in flight per warp).
// One CTA per policy (persistent grid-stride); activations ping-pong through shared memory.
#include "evok_common.cuh"

namespace evok {

constexpr int kMlpThreads = 256;
constexpr int kMlpWarps = kMlpThreads / 32;
constexpr int kMlpMaxLayers = 8;
constexpr int kMlpMaxWidth = 2048;
constexpr int kMlpNeuronsPerPass = 4;

struct MlpSpec {
  int n_layers;
  int dims[kMlpMaxLayers + 1];
  int acts[kMlpMaxLayers];
  int64_t w_off[kMlpMaxLayers];  // offset of W_l inside a parameter row; b_l follows at w_off + in*out
  int max_width;
};

// Observation pre-processing of the rollout loop (vecgymne.py:604-660, 822-836; net/runningnorm.py:412-533), fused into the
// observation load: x = clamp((obs - mean) / stdev, lo, hi) with mean / stdev derived on the fly from the running sums
// (mean = sum / count, var = max(sumsq / count - mean^2, min_variance)); policies whose environment is inactive are skipped
// altogether -- their 4*L parameter bytes are never read -- and get zero actions.
struct ObsPrep {
  const float* sum;        // n_in running sums, nullptr = no normalisation
  const float* sumsq;      // n_in running sums of squares
  const long long* count;  // number of observations behind the sums (device scalar)
  const unsigned char* active;  // N flags, nullptr = all active
  float min_variance, lo, hi;   // lo / hi = NaN: no clipping on that side
  unsigned int* ticket;         // zeroed work counter (nullptr: static round-robin).  With a mask the number of active policies per
                                // CTA is binomial under round-robin (1.9x imbalance at 10 % active); CTAs then draw chunks of rows
};

constexpr int kMlpTicketRows = 4;  // rows per ticket: 1/4 of the atomics, balance to within 4 rows

__device__ __forceinline__ float prep_obs(const ObsPrep& p, int k, float o) {
  if (!p.sum) return o;
  const float n = (float)(*p.count);
  const float mean = __fdiv_rn(p.sum[k], n);
  const float var = fmaxf(__fdiv_rn(p.sumsq[k], n) - mean * mean, p.min_variance);
  float v = __fdiv_rn(o - mean, __fsqrt_rn(var));
  if (p.lo == p.lo) v = fmaxf(v, p.lo);
  if (p.hi == p.hi) v = fminf(v, p.hi);
  return v;
}

__device__ __forceinline__ float activate(float v, int act) {
  switch (act) {
    case EVOK_ACT_TANH: return tanhf(v);
    case EVOK_ACT_RELU: return fmaxf(v, 0.0f);
    case EVOK_ACT_SIGMOID: return 1.0f / (1.0f + expf(-v));
    default: return v;
  }
}

// Activations live in shared memory SHIFTED by the 16-byte phase of the layer's weight rows: if every neuron row of a layer
// starts `ph` floats past a 16-byte boundary (true for all rows of a layer whenever n_in % 4 == 0), lane l loads the ALIGNED
// float4 chunks of the row and multiplies them with xs[4c .. 4c+3] where xs[u] = x[u - ph] and xs is zero outside the valid
// range -- the `ph` leading floats of the first chunk (they belong to the previous neuron) and the trailing floats of the last
// chunk meet zeros.  This turns 4-byte-aligned rows into 128-bit coalesced loads without any masking in the inner loop.
// The first and the last policy row use the scalar path so that no load ever touches bytes outside the parameter matrix.
constexpr int kMlpPad = 8;  // floats of zero padding in front of / behind an activation vector

__device__ __forceinline__ void store_shifted(float* buf, int ph, int j, float v) { buf[kMlpPad + ph + j] = v; }

__global__ void __launch_bounds__(kMlpThreads)
    mlp_forward_kernel(const float* __restrict__ params, int64_t ldp, const float* __restrict__ obs, int64_t ldo, float* __restrict__ out,
                       int64_t ldout, int64_t N, const __grid_constant__ MlpSpec spec, const __grid_constant__ ObsPrep prep) {
  extern __shared__ __align__(16) float act_buf[];  // 2 x (max_width + 2 * kMlpPad)
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int stride = (spec.max_width + 2 * kMlpPad + 3) & ~3;  // keeps both ping-pong buffers 16-byte aligned
  __shared__ unsigned int next_chunk;
  const bool dynamic = prep.ticket != nullptr;
  int64_t i = dynamic ? 0 : (int64_t)blockIdx.x - gridDim.x;
  int in_chunk = kMlpTicketRows;  // forces a ticket draw on the first iteration
  for (;;) {
    if (dynamic) {
      if (in_chunk == kMlpTicketRows) {
        __syncthreads();
        if (threadIdx.x == 0) next_chunk = atomicAdd(prep.ticket, 1u);
        __syncthreads();
        i = (int64_t)next_chunk * kMlpTicketRows;
        in_chunk = 0;
      } else {
        ++i;
      }
      ++in_chunk;
      if (i >= N) {
        if (in_chunk == 1) break;  // the chunk starts beyond the end: no work left anywhere
        continue;                  // tail of the last chunk
      }
    } else {
      i += gridDim.x;
      if (i >= N) break;
    }
    if (prep.active && !prep.active[i]) {  // CTA-uniform: the whole policy is skipped
      for (int k = threadIdx.x; k < spec.dims[spec.n_layers]; k += kMlpThreads) out[i * ldout + k] = 0.0f;
      continue;
    }
    const float* prow = params + i * ldp;
    const bool edge_row = (i == 0) || (i == N - 1);
    float* cur = act_buf;
    float* nxt = act_buf + stride;
    // phase of layer 0's weight rows (floats past a 16-byte boundary)
    int ph = (int)((reinterpret_cast<uintptr_t>(prow + spec.w_off[0]) >> 2) & 3);
    for (int k = threadIdx.x; k < stride; k += kMlpThreads) cur[k] = 0.0f;
    __syncthreads();
    for (int k = threadIdx.x; k < spec.dims[0]; k += kMlpThreads) store_shifted(cur, ph, k, prep_obs(prep, k, ld_stream1(obs + i * ldo + k)));
    __syncthreads();
    for (int l = 0; l < spec.n_layers; ++l) {
      const int n_in = spec.dims[l], n_out = spec.dims[l + 1];
      const float* W = prow + spec.w_off[l];
      const float* b = W + (int64_t)n_in * n_out;
      const bool last = l == spec.n_layers - 1;
      const int ph_next = last ? 0 : (int)((reinterpret_cast<uintptr_t>(prow + spec.w_off[l + 1]) >> 2) & 3);
      const bool vec = ((n_in & 3) == 0) && !edge_row;
      // zero the destination (including its pads) before the neurons of this layer are written into it
      if (!last)
        for (int k = threadIdx.x; k < stride; k += kMlpThreads) nxt[k] = 0.0f;
      __syncthreads();
      const float* xs = cur + kMlpPad;  // xs[u] = x[u - ph]
      const int nchunks = (n_in + ph + 3) >> 2;
      for (int j0 = warp * kMlpNeuronsPerPass; j0 < n_out; j0 += kMlpWarps * kMlpNeuronsPerPass) {
        float acc[kMlpNeuronsPerPass];
#pragma unroll
        for (int t = 0; t < kMlpNeuronsPerPass; ++t) acc[t] = 0.0f;
        const int n_here = min(kMlpNeuronsPerPass, n_out - j0);
        if (vec && n_here == kMlpNeuronsPerPass) {
          const float* w0 = W + (int64_t)j0 * n_in - ph;  // 16-byte aligned
          for (int c = lane; c < nchunks; c += 32) {
            const float4 x4 = *reinterpret_cast<const float4*>(xs + 4 * c);
#pragma unroll
            for (int t = 0; t < kMlpNeuronsPerPass; ++t) {
              const float4 w4 = ld_stream4(w0 + (int64_t)t * n_in + 4 * c);
              acc[t] = fmaf(w4.x, x4.x, fmaf(w4.y, x4.y, fmaf(w4.z, x4.z, fmaf(w4.w, x4.w, acc[t]))));
            }
          }
        } else {
          for (int t = 0; t < n_here; ++t) {
            const float* w0 = W + (int64_t)(j0 + t) * n_in;
            for (int k = lane; k < n_in; k += 32) acc[t] = fmaf(ld_stream1(w0 + k), xs[ph + k], acc[t]);
          }
        }
#pragma unroll
        for (int t = 0; t < kMlpNeuronsPerPass; ++t) acc[t] = warp_sum(acc[t]);
        if (lane < n_here) {
          float v = acc[0];
#pragma unroll
          for (int t = 1; t < kMlpNeuronsPerPass; ++t) v = lane == t ? acc[t] : v;
          v = activate(v + ld_stream1(b + j0 + lane), spec.acts[l]);
          if (last) out[i * ldout + j0 + lane] = v;
          else store_shifted(nxt, ph_next, j0 + lane, v);
        }
      }
      __syncthreads();
      float* tmp = cur;
      cur = nxt;
      nxt = tmp;
      ph = ph_next;
    }
  }
}

// ---- shared-minibatch forward (SupervisedNE with common_minibatch, supervisedne.py:337-347): layers 2..n of N networks on B samples.
// The first layer is the tensor-core GEMM over the stacked weight rows (gemm_gather_rows_ws), which leaves
//   hid[(i * B + b) * H1 + h] = act_0(W_0^i x_b + b_0^i)[h]      (unit fastest: one cache line per store instruction of the GEMM epilogue);
// this kernel takes one (network i, tile of 32 samples) per CTA, keeps the tile's activations in shared memory ([width][33]) and runs
// the remaining layers with fp32 FMAs: thread = (sample lane, output neuron), the weight row is a broadcast load shared by the 32
// samples of the warp.  out[(i * B + b) * O + o].
constexpr int kTailSamples = 32;
constexpr int kTailThreads = 256;
constexpr int kTailMaxWidth = 512;
constexpr int kTailOutBlock = 4;  // outputs per thread per pass (register blocking over the weight rows)

// tanh to ~1e-6 absolute: odd polynomial near 0, (1 - e) / (1 + e) with e = exp(-2|x|) elsewhere.  The accurate tanhf costs ~50
// instructions; 65 536 networks x 256 hidden units x 256 samples of them were a third of the forward.
// hid holds the first layer's PRE-activation (W_0 x + b_0); its activation is applied while the tile is loaded.
__global__ void __launch_bounds__(kTailThreads)
    mlp_tail_kernel(const float* __restrict__ params, int64_t ldp, const float* __restrict__ hid, int64_t ldh, int64_t n_first, int64_t B,
                    float* __restrict__ out, const __grid_constant__ MlpSpec spec) {
  extern __shared__ float tail_smem[];
  const int pitch = kTailSamples + 1;
  float* cur = tail_smem;
  float* nxt = cur + (size_t)spec.max_width * pitch;
  float* wsm = nxt + (size_t)spec.max_width * pitch;  // the current layer's weights + bias, staged once per CTA
  const int64_t net = blockIdx.y;
  const int64_t b0 = (int64_t)blockIdx.x * kTailSamples;
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int64_t b = b0 + lane;
  const bool b_ok = b < B;
  const float* prow = params + (net + n_first) * ldp;
  const int h1 = spec.dims[1];
  // hid[(net * B + sample) * h1 + unit]: lanes over the units (coalesced), one sample of the tile per warp pass
  for (int s = wid; s < kTailSamples; s += kTailThreads / 32) {
    const int64_t bs = b0 + s;
    for (int h = lane; h < h1; h += 32) cur[h * pitch + s] = bs < B ? activate_fast(hid[(net * B + bs) * h1 + h], spec.acts[0]) : 0.0f;
  }
  for (int l = 1; l < spec.n_layers; ++l) {
    const int din = spec.dims[l], dout = spec.dims[l + 1];
    const float* W = prow + spec.w_off[l];
    const int wcount = din * dout + dout;
    __syncthreads();  // cur complete; wsm free
    for (int e = threadIdx.x; e < wcount; e += kTailThreads) wsm[e] = __ldg(W + e);
    __syncthreads();
    const float* bias = wsm + (size_t)din * dout;
    // thread = (sample lane, block of kTailOutBlock consecutive outputs): per k one activation load + kTailOutBlock broadcast weight loads
    const int ob = min(kTailOutBlock, (dout + kTailThreads / 32 - 1) / (kTailThreads / 32));  // outputs per warp pass: spread dout over the 8 warps
    for (int o0 = wid * ob; o0 < dout; o0 += (kTailThreads / 32) * ob) {
      float acc[kTailOutBlock];
#pragma unroll
      for (int j = 0; j < kTailOutBlock; ++j) acc[j] = 0.0f;
      const int nj = min(ob, dout - o0);
#pragma unroll 4
      for (int k = 0; k < din; ++k) {
        const float a = cur[k * pitch + lane];
#pragma unroll
        for (int j = 0; j < kTailOutBlock; ++j)
          if (j < nj) acc[j] = fmaf(wsm[(size_t)(o0 + j) * din + k], a, acc[j]);
      }
#pragma unroll
      for (int j = 0; j < kTailOutBlock; ++j) {
        if (j < nj) {
          const float v = activate_fast(acc[j] + bias[o0 + j], spec.acts[l]);
          if (l == spec.n_layers - 1) {
            if (b_ok) out[((net * B) + b) * dout + o0 + j] = v;
          } else {
            nxt[(o0 + j) * pitch + lane] = v;
          }
        }
      }
    }
    float* t = cur;
    cur = nxt;
    nxt = t;
  }
}

// Two-layer nets with a narrow output (the usual policy / regression shape, e.g. 376-256-17): ONE CTA per network.  The second
// layer's weights are staged once in shared memory; a warp owns 64 samples (two per lane), streams the hidden pre-activations
// hid[h][b] straight from global memory (coalesced along b, each read exactly once), applies act_0 and accumulates all outputs
// in registers: per hidden unit one load, one activation and dout broadcast weight reads serving 2 x dout FMAs.
constexpr int kTail2MaxOut = 32;

// The hidden tile of 64 samples (h1 x 64 floats) is brought into shared memory with 16-byte cp.async copies, all of them issued up
// front in four commit groups (streaming the rows from inside the accumulation loop, or filling the tile with plain loads, was
// latency-bound: 35 ms of a 74 ms forward); each thread applies act_0 in place to the pieces it copied as its group lands, and the
// accumulation over a quarter of the hidden units starts while the other quarters are still in flight.  Thread = (sample pair,
// output group): per hidden unit two activation reads and one or two 16-byte broadcast weight reads serve 2 x OG FMAs.  96 KB of
// shared memory per CTA: two CTAs per SM cover each other's fill latency.
constexpr int kTail2Threads = 256;  // 8 warps = 4 output groups x 2 halves of the hidden units of each quarter
constexpr int kTail2Samples = 64;   // samples per pass
constexpr int kTail2Groups = 4;     // output groups (one warp each)
constexpr int kTail2Slots = 8;      // padded outputs per group: weights of hidden unit h, group g at wsm[(h * 4 + g) * 8 ..]

__device__ __forceinline__ void cp_async_16(void* smem_dst, const void* gmem_src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_4(void* smem_dst, const void* gmem_src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

template <int OG>  // outputs per thread (dout <= 4 * OG)
__global__ void __launch_bounds__(kTail2Threads)
    mlp_tail2_kernel(const float* __restrict__ params, int64_t ldp, const float* __restrict__ hid, int64_t ldh, int64_t n_first, int64_t B,
                     float* __restrict__ out, const __grid_constant__ MlpSpec spec) {
  extern __shared__ __align__(16) float tail_smem[];
  const int64_t net = blockIdx.x;
  const int h1 = spec.dims[1], dout = spec.dims[2];
  float* tile = tail_smem;                                                  // [64][h1 + 4]
  float* wsm = tile + (size_t)(h1 + 4) * kTail2Samples;                     // [h1][4][8]
  float* bsm = wsm + (size_t)h1 * kTail2Groups * kTail2Slots;               // [32]
  float* red = bsm + kTail2Groups * kTail2Slots;                            // [128][2 * OG] partial sums of the second half
  const float* W = params + (net + n_first) * ldp + spec.w_off[1];
  for (int e = threadIdx.x; e < h1 * kTail2Groups * kTail2Slots; e += kTail2Threads) wsm[e] = 0.0f;
  if (threadIdx.x < kTail2Groups * kTail2Slots) bsm[threadIdx.x] = 0.0f;
  __syncthreads();
  for (int e = threadIdx.x; e < h1 * dout; e += kTail2Threads) {
    const int o = e / h1, h = e - o * h1;
    wsm[(h * kTail2Groups + o / OG) * kTail2Slots + o % OG] = __ldg(W + e);
  }
  if (threadIdx.x < dout) bsm[(threadIdx.x / OG) * kTail2Slots + threadIdx.x % OG] = __ldg(W + h1 * dout + threadIdx.x);
  const int sp = threadIdx.x & 31, og = (threadIdx.x >> 5) & 3, hh = threadIdx.x >> 7;
  const int hq = ((h1 + 15) / 16) * 4;  // hidden units per commit group (a multiple of 4; h1 % 4 == 0)
  // The tile keeps the layout of hid -- [sample][unit], rows of h1 + 4 floats -- so it is filled with 16-byte copies; a thread reads FOUR
  // consecutive units of its two samples per 16-byte load: with a row pitch of 4 (mod 32) floats the 8 lanes of a quarter warp cover all
  // 32 banks exactly once.
  const int pitch = h1 + 4;
  const float* hnet = hid + net * B * h1;
  const int c4 = h1 / 4;  // 16-byte pieces per row
  for (int64_t b0 = 0; b0 < B; b0 += kTail2Samples) {
    __syncthreads();  // weights staged / the previous pass is done with the tile
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int qa = q * hq / 4, qb = min((q + 1) * hq, h1) / 4, qn = max(qb - qa, 0);  // this quarter's pieces [qa, qb) of every row
      for (int e = threadIdx.x; e < kTail2Samples * qn; e += kTail2Threads) {
        const int b = e / qn, v4 = qa + (e - b * qn);
        if (b0 + b < B) cp_async_16(tile + b * pitch + v4 * 4, hnet + (b0 + b) * h1 + v4 * 4);
      }
      cp_async_commit();
    }
    float acca[OG], accb[OG];
#pragma unroll
    for (int j = 0; j < OG; ++j) acca[j] = accb[j] = 0.0f;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      if (q == 0) cp_async_wait<3>();
      else if (q == 1) cp_async_wait<2>();
      else if (q == 2) cp_async_wait<1>();
      else cp_async_wait<0>();
      const int qa = q * hq / 4, qb = min((q + 1) * hq, h1) / 4, qn = max(qb - qa, 0);
      // act_0 in place, on the pieces this thread copied (its own cp.async writes are visible to it after the wait); nothing to do
      // when the producer (the GEMM epilogue) has already applied it
      if (spec.acts[0] != EVOK_ACT_NONE) {
        for (int e = threadIdx.x; e < kTail2Samples * qn; e += kTail2Threads) {
          const int b = e / qn, v4 = qa + (e - b * qn);
          if (b0 + b < B) {
            float4* p4 = reinterpret_cast<float4*>(tile + b * pitch + v4 * 4);
            float4 t = *p4;
            t.x = activate_fast(t.x, spec.acts[0]);
            t.y = activate_fast(t.y, spec.acts[0]);
            t.z = activate_fast(t.z, spec.acts[0]);
            t.w = activate_fast(t.w, spec.acts[0]);
            *p4 = t;
          }
        }
      }
      __syncthreads();
      const int qmid = qa + (qn + 1) / 2;
      const int v_lo = hh ? qmid : qa, v_hi = hh ? qb : qmid;  // this warp's half of the quarter (in 4-unit pieces)
#pragma unroll 2
      for (int v4 = v_lo; v4 < v_hi; ++v4) {
        const float4 xa4 = *reinterpret_cast<const float4*>(tile + sp * pitch + v4 * 4);
        const float4 xb4 = *reinterpret_cast<const float4*>(tile + (sp + 32) * pitch + v4 * 4);
        const float xa[4] = {xa4.x, xa4.y, xa4.z, xa4.w}, xb[4] = {xb4.x, xb4.y, xb4.z, xb4.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int h = v4 * 4 + u;
          const float4 w0 = *reinterpret_cast<const float4*>(wsm + (h * kTail2Groups + og) * kTail2Slots);
          float w[8] = {w0.x, w0.y, w0.z, w0.w, 0.0f, 0.0f, 0.0f, 0.0f};
          if (OG > 4) {
            const float4 w1 = *reinterpret_cast<const float4*>(wsm + (h * kTail2Groups + og) * kTail2Slots + 4);
            w[4] = w1.x, w[5] = w1.y, w[6] = w1.z, w[7] = w1.w;
          }
#pragma unroll
          for (int j = 0; j < OG; ++j) {
            acca[j] = fmaf(w[j], xa[u], acca[j]);
            accb[j] = fmaf(w[j], xb[u], accb[j]);
          }
        }
      }
    }
    // the second half hands its partial sums to the first through shared memory
    float* my_red = red + ((og * 32 + sp) * 2) * OG;
    if (hh) {
#pragma unroll
      for (int j = 0; j < OG; ++j) my_red[j] = acca[j], my_red[OG + j] = accb[j];
    }
    __syncthreads();
    if (!hh) {
      const int64_t ba = b0 + sp, bb = b0 + 32 + sp;
#pragma unroll
      for (int j = 0; j < OG; ++j) {
        const int o = og * OG + j;
        if (o < dout) {
          const float bias = bsm[og * kTail2Slots + j];
          if (ba < B) out[(net * B + ba) * dout + o] = activate_fast(acca[j] + my_red[j] + bias, spec.acts[1]);
          if (bb < B) out[(net * B + bb) * dout + o] = activate_fast(accb[j] + my_red[OG + j] + bias, spec.acts[1]);
        }
      }
    }
  }
  cp_async_wait<0>();
}

}  // namespace evok

using namespace evok;

extern "C" EVOK_API size_t evok_mlp_forward_shared_workspace_bytes(int64_t N, int64_t B, int n_layers, const int32_t* dims_host) {
  if (!dims_host || n_layers < 2 || N <= 0 || B <= 0) return 256;
  const int64_t ldh = (B + 3) / 4 * 4;
  int64_t chunk = ((int64_t)1 << 30) / (dims_host[1] * ldh * 4);  // about 1 GiB of first-layer activations at a time
  if (chunk < 1) chunk = 1;
  if (chunk > 65535) chunk = 65535;
  if (chunk > N) chunk = N;
  return (size_t)chunk * dims_host[1] * ldh * 4 + 256 + gemm_gather_rows_workspace_bytes(B, dims_host[0]);
}

// out[i, b, :] = net_i(X[b, :]) for N flat parameter rows and ONE shared input batch X (B x dims[0], 16-byte aligned rows).
extern "C" EVOK_API int evok_mlp_forward_shared(const float* params, int64_t ldp, int64_t N, const float* X, int64_t ldx, int64_t B, int n_layers,
                                                const int32_t* dims_host, const int32_t* acts_host, float* out, void* ws, size_t ws_bytes,
                                                void* stream) {
  if (!params || !X || !out || !dims_host || !acts_host || !ws) return EVOK_E_NULLPTR;
  if (n_layers < 2 || n_layers > kMlpMaxLayers || N < 0 || B <= 0) return EVOK_E_BADSIZE;
  MlpSpec spec;
  spec.n_layers = n_layers;
  int64_t off = 0;
  int maxw = 0;
  for (int l = 0; l <= n_layers; ++l) {
    const int d = dims_host[l];
    if (d < 1 || d > kMlpMaxWidth) return EVOK_E_BADSIZE;
    spec.dims[l] = d;
    if (l >= 1 && d > maxw) maxw = d;
  }
  if (maxw > kTailMaxWidth) return EVOK_E_BADSIZE;
  for (int l = 0; l < n_layers; ++l) {
    if (acts_host[l] < EVOK_ACT_NONE || acts_host[l] > EVOK_ACT_SIGMOID) return EVOK_E_BADENUM;
    spec.acts[l] = acts_host[l];
    spec.w_off[l] = off;
    off += (int64_t)spec.dims[l] * spec.dims[l + 1] + spec.dims[l + 1];
  }
  spec.max_width = maxw;
  if (ldp < off || ldx < spec.dims[0]) return EVOK_E_BADSIZE;
  if (N == 0) return 0;
  const int64_t h1 = spec.dims[1], ldh = (B + 3) / 4 * 4;
  int64_t chunk = ((int64_t)1 << 30) / (h1 * ldh * 4);
  if (chunk < 1) chunk = 1;
  if (chunk > 65535) chunk = 65535;  // gridDim.y of the tail kernel
  if (chunk > N) chunk = N;
  char* base = reinterpret_cast<char*>((reinterpret_cast<uintptr_t>(ws) + 255) & ~(uintptr_t)255);
  const size_t hid_bytes = ((size_t)chunk * h1 * ldh * 4 + 255) & ~(size_t)255;
  const size_t gws_bytes = gemm_gather_rows_workspace_bytes(B, spec.dims[0]);
  if (ws_bytes < (size_t)(base - (char*)ws) + hid_bytes + gws_bytes) return EVOK_E_WORKSPACE;
  float* hid = reinterpret_cast<float*>(base);
  void* gws = base + hid_bytes;
  // act_0 is applied by the GEMM epilogue (its warps have slack while the tensor core works on the next tile): the tail kernels
  // read activations
  MlpSpec tail_spec = spec;
  tail_spec.acts[0] = EVOK_ACT_NONE;
  size_t wmax = 0;  // largest staged layer (weights + bias) among the layers 1 .. n-1
  for (int l = 1; l < n_layers; ++l) {
    const size_t wl = (size_t)spec.dims[l] * spec.dims[l + 1] + spec.dims[l + 1];
    if (wl > wmax) wmax = wl;
  }
  const size_t smem = (2 * (size_t)maxw * (kTailSamples + 1) + wmax) * sizeof(float);
  if (smem > 200 * 1024) return EVOK_E_BADSIZE;  // a hidden layer too wide to stage: the caller falls back to the generic path
  static size_t attr_smem = 0;
  if (smem > attr_smem) {
    if (cudaFuncSetAttribute(mlp_tail_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem) != cudaSuccess) return (int)cudaGetLastError();
    attr_smem = smem;
  }
  for (int64_t i0 = 0; i0 < N; i0 += chunk) {
    const int64_t c = (N - i0) < chunk ? (N - i0) : chunk;
    // layer 0 of the c networks as ONE stacked-rows tensor-core product: (c * H1 x in) * (in x B)
    int rc = gemm_gather_rows_ws(params + i0 * ldp, ldp, spec.w_off[0], h1, c, X, ldx, B, spec.dims[0], spec.w_off[0] + (int64_t)spec.dims[0] * h1,
                                 spec.acts[0], hid, gws, gws_bytes, stream);
    if (rc) return rc;
    const size_t smem2 = ((size_t)(h1 + 4) * kTail2Samples + (size_t)h1 * kTail2Groups * kTail2Slots + kTail2Groups * kTail2Slots + 128 * 2 * 8) * sizeof(float);
    if (n_layers == 2 && spec.dims[2] <= kTail2MaxOut && smem2 <= 200 * 1024 && (reinterpret_cast<uintptr_t>(hid) & 15) == 0 && h1 % 4 == 0) {
      // 4 output groups x 32 sample pairs x 2 halves of the hidden units = 256 threads; outputs per thread = ceil(dout / 4)
      const int og = (spec.dims[2] + kTail2Groups - 1) / kTail2Groups;
#define EVOK_LAUNCH_TAIL2(OGV)                                                                                                      \
  do {                                                                                                                              \
    cudaFuncSetAttribute(mlp_tail2_kernel<OGV>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem2);                           \
    mlp_tail2_kernel<OGV><<<(unsigned)c, kTail2Threads, smem2, (cudaStream_t)stream>>>(params, ldp, hid, ldh, i0, B,                \
                                                                                       out + i0 * B * spec.dims[2], tail_spec);      \
  } while (0)
      if (og <= 1) EVOK_LAUNCH_TAIL2(1);
      else if (og <= 2) EVOK_LAUNCH_TAIL2(2);
      else if (og <= 4) EVOK_LAUNCH_TAIL2(4);
      else if (og <= 5) EVOK_LAUNCH_TAIL2(5);
      else EVOK_LAUNCH_TAIL2(8);
#undef EVOK_LAUNCH_TAIL2
    } else {
      dim3 grid((unsigned)((B + kTailSamples - 1) / kTailSamples), (unsigned)c);
      mlp_tail_kernel<<<grid, kTailThreads, smem, (cudaStream_t)stream>>>(params, ldp, hid, ldh, i0, B, out + i0 * B * spec.dims[n_layers], tail_spec);
    }
    EVOK_CHECK_LAUNCH();
  }
  return 0;
}

extern "C" EVOK_API int64_t evok_mlp_parameter_length(int n_layers, const int32_t* dims_host) {
  if (!dims_host || n_layers < 1 || n_layers > kMlpMaxLayers) return -1;
  int64_t total = 0;
  for (int l = 0; l < n_layers; ++l) total += (int64_t)dims_host[l] * dims_host[l + 1] + dims_host[l + 1];
  return total;
}

static int mlp_forward_impl(const float* params, int64_t ldp, const float* obs, int64_t ldo, float* out, int64_t ldout, int64_t N, int n_layers,
                            const int32_t* dims_host, const int32_t* acts_host, const ObsPrep& prep, void* stream) {
  if (!params || !obs || !out || !dims_host || !acts_host) return EVOK_E_NULLPTR;
  if (n_layers < 1 || n_layers > kMlpMaxLayers || N < 0) return EVOK_E_BADSIZE;
  MlpSpec spec;
  spec.n_layers = n_layers;
  int64_t off = 0;
  int maxw = 0;
  for (int l = 0; l <= n_layers; ++l) {
    const int d = dims_host[l];
    if (d < 1 || d > kMlpMaxWidth) return EVOK_E_BADSIZE;
    spec.dims[l] = d;
    if (d > maxw) maxw = d;
  }
  for (int l = 0; l < n_layers; ++l) {
    if (acts_host[l] < EVOK_ACT_NONE || acts_host[l] > EVOK_ACT_SIGMOID) return EVOK_E_BADENUM;
    spec.acts[l] = acts_host[l];
    spec.w_off[l] = off;
    off += (int64_t)spec.dims[l] * spec.dims[l + 1] + spec.dims[l + 1];
  }
  spec.max_width = maxw;
  if (ldp < off || ldo < spec.dims[0] || ldout < spec.dims[n_layers]) return EVOK_E_BADSIZE;
  if (N == 0) return 0;
  const size_t smem = 2 * (size_t)((maxw + 2 * 8 + 3) & ~3) * sizeof(float);
  int per_sm = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, mlp_forward_kernel, kMlpThreads, smem) != cudaSuccess || per_sm <= 0) per_sm = 4;
  int dev = 0, sms = kNumSMs;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  int64_t grid = (int64_t)per_sm * sms;
  if (grid > N) grid = N;
  mlp_forward_kernel<<<(unsigned)grid, kMlpThreads, smem, (cudaStream_t)stream>>>(params, ldp, obs, ldo, out, ldout, N, spec, prep);
  EVOK_CHECK_LAUNCH();
  return 0;
}

extern "C" EVOK_API int evok_mlp_forward(const float* params, int64_t ldp, const float* obs, int64_t ldo, float* out, int64_t ldout,
                                         int64_t N, int n_layers, const int32_t* dims_host, const int32_t* acts_host, void* stream) {
  ObsPrep prep{};
  return mlp_forward_impl(params, ldp, obs, ldo, out, ldout, N, n_layers, dims_host, acts_host, prep, stream);
}

extern "C" EVOK_API int evok_mlp_forward_prep(const float* params, int64_t ldp, const float* obs, int64_t ldo, float* out, int64_t ldout, int64_t N,
                                              int n_layers, const int32_t* dims_host, const int32_t* acts_host, const float* obs_sum,
                                              const float* obs_sumsq, const int64_t* obs_count_dev, float min_variance, float clip_lo, float clip_hi,
                                              const uint8_t* active, void* ws, size_t ws_bytes, void* stream) {
  if ((obs_sum != nullptr) != (obs_sumsq != nullptr) || (obs_sum != nullptr) != (obs_count_dev != nullptr)) return EVOK_E_NULLPTR;
  ObsPrep prep{};
  prep.sum = obs_sum;
  prep.sumsq = obs_sumsq;
  prep.count = reinterpret_cast<const long long*>(obs_count_dev);
  prep.active = active;
  prep.min_variance = min_variance;
  prep.lo = clip_lo;
  prep.hi = clip_hi;
  if (active && ws && ws_bytes >= sizeof(unsigned int) && N > 0) {  // masked: balance the surviving policies over the CTAs dynamically
    prep.ticket = static_cast<unsigned int*>(ws);
    cudaError_t e = cudaMemsetAsync(ws, 0, sizeof(unsigned int), (cudaStream_t)stream);
    if (e != cudaSuccess) return (int)e;
  }
  return mlp_forward_impl(params, ldp, obs, ldo, out, ldout, N, n_layers, dims_host, acts_host, prep, stream);
}
