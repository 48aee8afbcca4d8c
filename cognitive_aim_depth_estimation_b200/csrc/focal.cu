// Vector-sized stages of the focal / guidance path (fp32 throughout; block reductions via warp shuffles):
//   rowstats_merge   : merge the per-64-column softmax partials of GEMM pass A into (row max, weight / row sum)
//   focal_finalize   : column sums of pass B -> mean + centre bias -> L1 norm -> clamp -> renorm (+ re-focus scale)
//   guided_softmax   : softmax((0.7*mask + 0.3*a) / 0.05) and its argmax cell
//   weighted_pool    : sum_n w[b,n] * tokens[b,1+n,:]  (bandwidth-bound, split over N, deterministic partials)
//   guide_tail       : guided_softmax -> weighted_pool -> heads of one guided call in one launch
// Reference: src/model.py:197-200,234-282 (FocalStream), :426 (re-focus), :1404-1414 (_guided_focal_stream).
#include "common.cuh"
#include "focal.cuh"

#include <cuda_fp16.h>
#include "heads_row.cuh"
#include "host.h"

namespace ca {
namespace {

__device__ __forceinline__ float block_sum(float v, float* red) {
  v = warp_sum(v);
  const int w = warp_id(), l = lane_id(), nw = blockDim.x >> 5;
  __syncthreads();
  if (l == 0) red[w] = v;
  __syncthreads();
  float t = (l < nw) ? red[l] : 0.f;
  t = warp_sum(t);
  return t;  // every thread holds the total
}

// pm, ps: [batch, P, N] span-major (row max / sum-exp2 per 64-column span, as CA_EPI_ROWSTATS writes them)
//   -> rmax[batch * N], rinv[batch * N] = weight[row] / sum
// wtab (optional): [batch, P, N], wtab[b, s, r] = exp2(m[b, s, r] - rmax[r]) * rinv[r] — the factor that turns the
// span-relative exponentials E kept by GEMM pass A into (weighted) softmax probabilities.
// One thread per row; with the span-major layout every load and store of a warp is one contiguous 128-byte line.
constexpr int kMergeMaxSpans = 128;  // N <= 8192 columns
__global__ void __launch_bounds__(256) rowstats_merge_kernel(const float* __restrict__ pm, const float* __restrict__ ps,
                                      const float* __restrict__ weight, float* __restrict__ rmax,
                                      float* __restrict__ rinv, float* __restrict__ wtab, int rows, int N, int P) {
  griddep_sync();  // PDL: nothing before this line reads or writes global memory
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= rows) return;
  const int b = r / N;
  const size_t base = static_cast<size_t>(b) * P * N + (r - b * N);
  const float* m = pm + base;
  const float* s = ps + base;
  float mx = -INFINITY;
  for (int i = 0; i < P; i += 8) {
    float t[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) t[u] = (i + u < P) ? m[static_cast<size_t>(i + u) * N] : -INFINITY;
#pragma unroll
    for (int u = 0; u < 8; ++u) mx = fmaxf(mx, t[u]);
  }
  float sum = 0.f;
  for (int i = 0; i < P; i += 8) {
    float t[8], q[8];
#pragma unroll
    for (int u = 0; u < 8; ++u) {
      const bool in = i + u < P;
      t[u] = in ? m[static_cast<size_t>(i + u) * N] : -INFINITY;
      q[u] = in ? s[static_cast<size_t>(i + u) * N] : 0.f;
    }
#pragma unroll
    for (int u = 0; u < 8; ++u)
      if (i + u < P) sum += q[u] * exp2f(t[u] - mx);  // s = 0 where the span is fully masked (m = -inf)
  }
  const float ri = (weight ? weight[r] : 1.0f) / sum;
  if (rmax) rmax[r] = mx;
  if (rinv) rinv[r] = ri;
  if (wtab)
    for (int i = 0; i < P; ++i) wtab[base + static_cast<size_t>(i) * N] = exp2f(m[static_cast<size_t>(i) * N] - mx) * ri;
}

// Column sums of the (weighted) row softmax from the stored exponentials: pc[b, p, j] = sum over the 64 rows i of row
// span p of E[b, i, j] * wtab[b, i, j / 64].  One thread = 8 consecutive columns (one 16-byte fp16 load per row);
// grid = (column chunks, row spans, images).  Bandwidth-bound: reads E once (2 bytes per score).  The partials are
// span-major ([B, P, N]): a CTA's results are one contiguous row (the column-major form, 4-byte stores 4 P bytes apart,
// cost this kernel half its time in partial-sector writes: 0.38 -> see profiles/README.md of the HBM rate).
__global__ void __launch_bounds__(192) colsum_e_kernel(const __half* __restrict__ E, int lde, long long e_batch_stride,
                                                        const float* __restrict__ wtab, float* __restrict__ pc, int N,
                                                        int P) {
  griddep_sync();  // PDL: nothing before this line reads or writes global memory
  // The statistics GEMM wrote E image by image, row span by row span: walk it LAST-WRITTEN-FIRST, so that the CTAs that start
  // first read what the L2 still holds (E of a batch is about the size of the L2) instead of evicting it unread.
  const int b = gridDim.z - 1 - blockIdx.z;
  const int p = gridDim.y - 1 - blockIdx.y;
  const int j0 = (blockIdx.x * blockDim.x + threadIdx.x) * 8;
  if (j0 >= lde) return;
  const int span = j0 >> 6;
  const int i0 = min(p * 64, N);
  const int i1 = min(i0 + 64, N);
  const __half* e = E + static_cast<size_t>(b) * e_batch_stride + static_cast<size_t>(i0) * lde + j0;
  const float* w = wtab + (static_cast<size_t>(b) * P + span) * N + i0;  // span-major [B, P, N]: the rows of a span are contiguous
  float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  // 8 rows per batch, double-buffered: the loads of batch k + 1 are issued before batch k is consumed, so a warp always has
  // 8-16 x 512 B in flight.  (Written as one load-use loop the compiler kept two loads in flight per thread: 0.38 of the
  // HBM rate; with 16-row batches consumed before the next batch was issued the memory pipe drained four times per CTA.)
  constexpr int kBatch = 8;
  uint4 q[2][kBatch];
  float wi[2][kBatch];
  auto fetch = [&](int buf, int i) {
#pragma unroll
    for (int u = 0; u < kBatch; ++u) {
      const bool in = i + u < i1;
      q[buf][u] = in ? __ldg(reinterpret_cast<const uint4*>(e + static_cast<size_t>(i - i0 + u) * lde)) : make_uint4(0u, 0u, 0u, 0u);
      wi[buf][u] = in ? __ldg(w + (i - i0 + u)) : 0.f;
    }
  };
  auto consume = [&](int buf) {
#pragma unroll
    for (int u = 0; u < kBatch; ++u) {
      const __half2* h = reinterpret_cast<const __half2*>(&q[buf][u]);
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const float2 f = __half22float2(h[t]);
        acc[2 * t + 0] = fmaf(f.x, wi[buf][u], acc[2 * t + 0]);
        acc[2 * t + 1] = fmaf(f.y, wi[buf][u], acc[2 * t + 1]);
      }
    }
  };
  fetch(0, i0);
#pragma unroll 1
  for (int i = i0; i < i1; i += 2 * kBatch) {
    fetch(1, i + kBatch);
    consume(0);
    fetch(0, i + 2 * kBatch);
    consume(1);
  }
  float* out = pc + (static_cast<size_t>(b) * P + p) * N + j0;
#pragma unroll
  for (int t = 0; t < 8; ++t)
    if (j0 + t < N) out[t] = acc[t];
}

// One CTA per image.  pc: [B, P, N] column-sum partials (span-major, as ca_colsum_e writes them).  attn[b, j] = final_attention of the iteration.
// rowscale_out[b, j] = rowscale_in[b, j] * (1 + focus_strength * attn)  when rowscale_out != nullptr.
// mode 0: FocalStream attention  (mean over rows, centre bias, L1, clamp, renorm)   src/model.py:234-282
// mode 1: plain sum of partials (weighted column sums for the un-guided value path; no bias / normalisation)
// cur_weight[b] (optional): curiosity modulation between the L1 normalisation and the clamp (src/model.py:264-276).
constexpr int kFinalizeThreads = 1024;
constexpr int kFinalizeCols = 8;  // columns a thread keeps in registers: N <= 8192 (1036 x 1036 images: N = 5476)
__global__ void __launch_bounds__(kFinalizeThreads) focal_finalize_kernel(const float* __restrict__ pc, const float* __restrict__ cbias,
                                                              float* __restrict__ attn, const float* __restrict__ rs_in,
                                                              float* __restrict__ rs_out, int N, int P,
                                                              float focus_strength, int mode,
                                                              const float* __restrict__ cur_weight,
                                                              float adaptive_weight) {
  griddep_sync();  // PDL: nothing before this line reads or writes global memory
  __shared__ float red[32];
  const int b = blockIdx.x;
  const float* pcb = pc + static_cast<size_t>(b) * P * N;
  float* ab = attn + static_cast<size_t>(b) * N;
  const float invN = 1.0f / static_cast<float>(N);
  // A latency kernel (one CTA per image, 130 KB of partials): every thread owns up to 8 columns and keeps them in
  // registers through the three passes; the P partials of a column are fetched 8 at a time (independent loads) and
  // added in ascending order — the same sums as a plain loop, without one L2 round trip per addend.
  float v[kFinalizeCols];
  float local = 0.f;
#pragma unroll
  for (int c = 0; c < kFinalizeCols; ++c) {
    const int j = threadIdx.x + c * kFinalizeThreads;
    v[c] = 0.f;
    if (j < N) {
      float s = 0.f;
      for (int i = 0; i < P; i += 8) {
        float t[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) t[u] = (i + u < P) ? pcb[static_cast<size_t>(i + u) * N + j] : 0.f;
#pragma unroll
        for (int u = 0; u < 8; ++u)
          if (i + u < P) s += t[u];
      }
      v[c] = (mode == 0) ? (s * invN + cbias[j]) : s;
      local += v[c];
      if (mode != 0) ab[j] = v[c];
    }
  }
  if (mode != 0) return;
  const float tot1 = block_sum(local, red);
  const float d1 = tot1 + 1e-8f;
  const float cw = cur_weight ? cur_weight[b] : 0.f;
  local = 0.f;
#pragma unroll
  for (int c = 0; c < kFinalizeCols; ++c) {
    const int j = threadIdx.x + c * kFinalizeThreads;
    if (j < N) {
      float a = v[c] / d1;
      if (cur_weight) a = adaptive_weight * (a * (1.0f + cw)) + (1.0f - adaptive_weight) * a;  // src/model.py:270-274
      a = fmaxf(a, 1e-8f);
      v[c] = a;
      local += a;
    }
  }
  const float tot2 = block_sum(local, red);
  const float d2 = tot2 + 1e-8f;
#pragma unroll
  for (int c = 0; c < kFinalizeCols; ++c) {
    const int j = threadIdx.x + c * kFinalizeThreads;
    if (j < N) {
      const float a = v[c] / d2;
      ab[j] = a;
      if (rs_out) {
        const size_t o = static_cast<size_t>(b) * N + j;
        rs_out[o] = (rs_in ? rs_in[o] : 1.0f) * (1.0f + focus_strength * a);
      }
    }
  }
}

// heat[r, :] = softmax((alpha*mask + (1-alpha)*base[b, :]) / temperature), argmax[r] = first index of the maximum.
// One CTA per row r = k * B + b (instruction k of a sweep, image b; k = 0 for a single call): the mask row is
// mask + k * mask_k_stride + b * mask_batch_stride, the base row base + k * base_k_stride + b * N.
__global__ void __launch_bounds__(256) guided_softmax_kernel(const float* __restrict__ base, long long base_k_stride,
                                                              const float* __restrict__ mask, long long mask_k_stride,
                                                              long long mask_batch_stride, float* __restrict__ heat,
                                                              int* __restrict__ argmax, int B, int N, float alpha,
                                                              float temperature) {
  griddep_sync();  // PDL: nothing before this line reads or writes global memory
  __shared__ float red[32];
  __shared__ int redi[32];
  const int r = blockIdx.x;
  const int b = r % B, k = r / B;
  // mask_batch_stride 0: one instruction for the whole batch (src/model.py:1401)
  mask += static_cast<size_t>(k) * mask_k_stride + static_cast<size_t>(b) * mask_batch_stride;
  const float* bb = base + static_cast<size_t>(k) * base_k_stride + static_cast<size_t>(b) * N;
  float* hb = heat + static_cast<size_t>(r) * N;
  float mx = -INFINITY;
  int mi = 0x7fffffff;
  for (int j = threadIdx.x; j < N; j += blockDim.x) {
    const float t = (alpha * mask[j] + (1.0f - alpha) * bb[j]) / temperature;
    hb[j] = t;
    if (t > mx) {
      mx = t;
      mi = j;
    }
  }
  // block arg-max with first-index tie-break
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, mx, o);
    const int oi = __shfl_xor_sync(0xffffffffu, mi, o);
    if (om > mx || (om == mx && oi < mi)) {
      mx = om;
      mi = oi;
    }
  }
  const int w = warp_id(), l = lane_id(), nw = blockDim.x >> 5;
  if (l == 0) {
    red[w] = mx;
    redi[w] = mi;
  }
  __syncthreads();
  mx = (l < nw) ? red[l] : -INFINITY;
  mi = (l < nw) ? redi[l] : 0x7fffffff;
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, mx, o);
    const int oi = __shfl_xor_sync(0xffffffffu, mi, o);
    if (om > mx || (om == mx && oi < mi)) {
      mx = om;
      mi = oi;
    }
  }
  float local = 0.f;
  for (int j = threadIdx.x; j < N; j += blockDim.x) {
    const float e = expf(hb[j] - mx);
    hb[j] = e;
    local += e;
  }
  const float tot = block_sum(local, red);
  for (int j = threadIdx.x; j < N; j += blockDim.x) hb[j] = hb[j] / tot;
  if (threadIdx.x == 0 && argmax) argmax[r] = mi;
}

// partial[b, split, :] = sum_{n in split} w[b, n] * (w2 ? w2[b, n] : 1) * src[b*src_batch_stride + (row_offset+n)*D + :]
// D = 768: 192 threads x float4.  grid = (splits, B).
__global__ void __launch_bounds__(192) weighted_pool_kernel(const float* __restrict__ src, long long src_batch_stride,
                                                             int row_offset, const float* __restrict__ w,
                                                             const float* __restrict__ w2, float* __restrict__ partial,
                                                             int N, int D, int rows_per_split) {
  griddep_sync();  // PDL: nothing before this line reads or writes global memory
  const int b = blockIdx.y;
  const int split = blockIdx.x;
  const int n0 = split * rows_per_split;
  const int n1 = min(N, n0 + rows_per_split);
  const float4* s4 = reinterpret_cast<const float4*>(src + static_cast<size_t>(b) * src_batch_stride +
                                                     static_cast<size_t>(row_offset) * D);
  const float* wb = w + static_cast<size_t>(b) * N;
  const float* w2b = w2 ? w2 + static_cast<size_t>(b) * N : nullptr;
  const int dv = D / 4;
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  constexpr int kBatch = 8;  // loads of a batch issued together (memory-level parallelism), then the FMAs in row order
  for (int n = n0; n < n1; n += kBatch) {
    float4 t[kBatch];
    float g[kBatch];
#pragma unroll
    for (int u = 0; u < kBatch; ++u) {
      const bool in = n + u < n1;
      t[u] = in ? s4[static_cast<size_t>(n + u) * dv + threadIdx.x] : make_float4(0.f, 0.f, 0.f, 0.f);
      g[u] = in ? (w2b ? wb[n + u] * w2b[n + u] : wb[n + u]) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < kBatch; ++u) {
      acc.x = fmaf(g[u], t[u].x, acc.x);
      acc.y = fmaf(g[u], t[u].y, acc.y);
      acc.z = fmaf(g[u], t[u].z, acc.z);
      acc.w = fmaf(g[u], t[u].w, acc.w);
    }
  }
  reinterpret_cast<float4*>(partial + (static_cast<size_t>(b) * gridDim.x + split) * D)[threadIdx.x] = acc;
}

// weighted_pool_kernel for K weight vectors at once (an instruction sweep): w is [K, B, N] (row k * B + b), partial is
// [K * B, splits, D].  A CTA reads its rows of image b's tokens ONCE and keeps one float4 accumulator per vector.  Each
// accumulator goes through weighted_pool_kernel's exact sequence — same rows per split, same batches of 8 rows with the
// same zero padding in the tail, same fmaf chain — so partial row k * B + b is bit for bit what weighted_pool_kernel
// writes for weight vector k.  KMAX accumulators live in registers (16 x 4 at the largest instantiation, no spills).
template <int KMAX>
__global__ void __launch_bounds__(192) weighted_pool_sweep_kernel(const float* __restrict__ src, long long src_batch_stride,
                                                                   int row_offset, const float* __restrict__ w,
                                                                   float* __restrict__ partial, int K, int B, int N, int D,
                                                                   int rows_per_split) {
  griddep_sync();  // PDL: nothing before this line reads or writes global memory
  const int b = blockIdx.y;
  const int split = blockIdx.x;
  const int n0 = split * rows_per_split;
  const int n1 = min(N, n0 + rows_per_split);
  const float4* s4 = reinterpret_cast<const float4*>(src + static_cast<size_t>(b) * src_batch_stride +
                                                     static_cast<size_t>(row_offset) * D);
  const float* wb = w + static_cast<size_t>(b) * N;
  const size_t w_k_stride = static_cast<size_t>(B) * N;
  const int dv = D / 4;
  float4 acc[KMAX];
#pragma unroll
  for (int k = 0; k < KMAX; ++k) acc[k] = make_float4(0.f, 0.f, 0.f, 0.f);
  constexpr int kBatch = 8;
  for (int n = n0; n < n1; n += kBatch) {
    float4 t[kBatch];
#pragma unroll
    for (int u = 0; u < kBatch; ++u)
      t[u] = (n + u < n1) ? s4[static_cast<size_t>(n + u) * dv + threadIdx.x] : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int k = 0; k < KMAX; ++k) {
      if (k < K) {
        const float* wk = wb + k * w_k_stride;
        float g[kBatch];
#pragma unroll
        for (int u = 0; u < kBatch; ++u) g[u] = (n + u < n1) ? wk[n + u] : 0.f;
#pragma unroll
        for (int u = 0; u < kBatch; ++u) {
          acc[k].x = fmaf(g[u], t[u].x, acc[k].x);
          acc[k].y = fmaf(g[u], t[u].y, acc[k].y);
          acc[k].z = fmaf(g[u], t[u].z, acc[k].z);
          acc[k].w = fmaf(g[u], t[u].w, acc[k].w);
        }
      }
    }
  }
#pragma unroll
  for (int k = 0; k < KMAX; ++k)
    if (k < K)
      reinterpret_cast<float4*>(partial + ((static_cast<size_t>(k) * B + b) * gridDim.x + split) * D)[threadIdx.x] = acc[k];
}

// The guided tail of one call in one launch: guided_softmax -> weighted_pool -> heads, bit for bit.
// grid = (splits, B), kHeadsThreads threads.  Every CTA of image b recomputes the image's guided softmax (N <= 8192 logits
// in shared memory) with threads 0..255 in guided_softmax_kernel's striding and reductions — both depend on the thread
// count, so the other 768 threads only contribute the neutral elements a 256-thread block has in its idle lanes.  CTA
// `split` then pools its rows of the tokens with threads 0..191 exactly as weighted_pool_kernel does and writes its
// partial; the last CTA of the image (a per-image ticket, re-armed by that CTA, so nothing has to be cleared between
// launches) runs the heads body on the 32 partials.  Split 0 writes the heat map and the argmax.
constexpr int kTailSoftmaxThreads = 256;  // guided_softmax_kernel's block size
constexpr int kTailPoolThreads = 192;     // weighted_pool_kernel's block size (D = 768 as float4)
constexpr int kTailMaxN = kFinalizeThreads * kFinalizeCols;
__global__ void __launch_bounds__(kHeadsThreads) guide_tail_kernel(const HeadsWeights wt, const HeadsInputs in,
                                                                   const float* __restrict__ base,
                                                                   const float* __restrict__ mask,
                                                                   long long mask_batch_stride, float* __restrict__ heat,
                                                                   int* __restrict__ argmax, float* partial,
                                                                   unsigned int* __restrict__ ticket,
                                                                   float* __restrict__ depth, float* __restrict__ conf,
                                                                   int N, float alpha, float temperature) {
  griddep_sync();  // PDL: nothing before this line reads or writes global memory
  __shared__ float s_p[kTailMaxN];
  __shared__ float red[32];
  __shared__ int redi[32];
  __shared__ bool s_last;
  const int b = blockIdx.y;
  const int split = blockIdx.x;
  const int tid = threadIdx.x;
  const bool soft = tid < kTailSoftmaxThreads;

  // ---- guided softmax (guided_softmax_kernel, row b) ----
  const float* mb = mask + static_cast<size_t>(b) * mask_batch_stride;
  const float* bb = base + static_cast<size_t>(b) * N;
  float mx = -INFINITY;
  int mi = 0x7fffffff;
  if (soft)
    for (int j = tid; j < N; j += kTailSoftmaxThreads) {
      const float t = (alpha * mb[j] + (1.0f - alpha) * bb[j]) / temperature;
      s_p[j] = t;
      if (t > mx) {
        mx = t;
        mi = j;
      }
    }
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, mx, o);
    const int oi = __shfl_xor_sync(0xffffffffu, mi, o);
    if (om > mx || (om == mx && oi < mi)) {
      mx = om;
      mi = oi;
    }
  }
  const int w = warp_id(), l = lane_id();
  if (l == 0) {
    red[w] = mx;
    redi[w] = mi;
  }
  __syncthreads();
  // lanes of the idle warps hold (-inf, INT_MAX): what lanes >= 8 read in a 256-thread block
  mx = red[l];
  mi = redi[l];
  for (int o = 16; o > 0; o >>= 1) {
    const float om = __shfl_xor_sync(0xffffffffu, mx, o);
    const int oi = __shfl_xor_sync(0xffffffffu, mi, o);
    if (om > mx || (om == mx && oi < mi)) {
      mx = om;
      mi = oi;
    }
  }
  float local = 0.f;
  if (soft)
    for (int j = tid; j < N; j += kTailSoftmaxThreads) {
      const float e = expf(s_p[j] - mx);
      s_p[j] = e;
      local += e;
    }
  const float tot = block_sum(local, red);  // idle warps add 0: the zero lanes of a 256-thread block_sum
  float* hb = heat + static_cast<size_t>(b) * N;
  if (soft)
    for (int j = tid; j < N; j += kTailSoftmaxThreads) {
      const float h = s_p[j] / tot;
      s_p[j] = h;
      if (split == 0) hb[j] = h;
    }
  if (split == 0 && tid == 0 && argmax) argmax[b] = mi;
  __syncthreads();

  // ---- weighted pool of this split's rows (weighted_pool_kernel, w2 = NULL, row offset 1) ----
  if (tid < kTailPoolThreads) {
    const int rps = (N + gridDim.x - 1) / gridDim.x;
    const int n0 = split * rps;
    const int n1 = min(N, n0 + rps);
    const float4* s4 = reinterpret_cast<const float4*>(in.tokens + static_cast<size_t>(b) * in.tokens_per_img * 768 + 768);
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    constexpr int kBatch = 8;
    for (int n = n0; n < n1; n += kBatch) {
      float4 t[kBatch];
      float g[kBatch];
#pragma unroll
      for (int u = 0; u < kBatch; ++u) {
        const bool inr = n + u < n1;
        t[u] = inr ? s4[static_cast<size_t>(n + u) * 192 + tid] : make_float4(0.f, 0.f, 0.f, 0.f);
        g[u] = inr ? s_p[n + u] : 0.f;
      }
#pragma unroll
      for (int u = 0; u < kBatch; ++u) {
        acc.x = fmaf(g[u], t[u].x, acc.x);
        acc.y = fmaf(g[u], t[u].y, acc.y);
        acc.z = fmaf(g[u], t[u].z, acc.z);
        acc.w = fmaf(g[u], t[u].w, acc.w);
      }
    }
    reinterpret_cast<float4*>(partial + (static_cast<size_t>(b) * gridDim.x + split) * 768)[tid] = acc;
  }

  // ---- the last CTA of the image runs the heads ----
  __threadfence();
  __syncthreads();
  if (tid == 0) {
    const unsigned int t = atomicAdd(ticket + b, 1u);
    s_last = t == gridDim.x - 1;
    if (s_last) ticket[b] = 0u;  // every CTA of this image has taken its ticket: re-arm for the next launch
  }
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  heads_row(wt, in, depth, conf, nullptr, b, gridDim.y);
}

}  // namespace

int rowstats_merge_launch(const float* pm, const float* ps, const float* weight, float* rmax, float* rinv, float* wtab,
                          int rows, int rows_per_image, int P, cudaStream_t stream) {
  CA_REQUIRE(pm && ps, "rowstats_merge: null pointer");
  CA_REQUIRE((rmax && rinv) || wtab, "rowstats_merge: no output requested");
  CA_REQUIRE(P > 0 && P <= kMergeMaxSpans, "rowstats_merge: 1..128 spans per row");
  CA_REQUIRE(rows > 0 && rows_per_image > 0 && rows % rows_per_image == 0, "rowstats_merge: rows must be batch * rows_per_image");
  CA_TRY(launch_kernel(rowstats_merge_kernel, dim3((rows + 255) / 256), dim3(256), 0, stream, pm, ps, weight, rmax, rinv, wtab, rows,
                       rows_per_image, P));
  CA_CUDA(cudaGetLastError());
  return 0;
}

int colsum_e_launch(const void* E, int lde, long long e_batch_stride, const float* wtab, float* pc, int B, int N, int P,
                    cudaStream_t stream) {
  CA_REQUIRE(E && wtab && pc, "colsum_e: null pointer");
  CA_REQUIRE(lde % 64 == 0 && lde >= N, "colsum_e: lde must be a multiple of 64 and >= N");
  CA_REQUIRE(P * 64 >= N && lde <= P * 64, "colsum_e: P row/column spans of 64 must cover N");
  CA_REQUIRE((reinterpret_cast<uintptr_t>(E) & 15) == 0 && e_batch_stride % 8 == 0, "colsum_e: E must be 16-byte aligned");
  dim3 grid((lde / 8 + 191) / 192, P, B);  // every partial slot is written (row spans past N contribute zeros)
  CA_TRY(launch_kernel(colsum_e_kernel, dim3(grid), dim3(192), 0, stream, reinterpret_cast<const __half*>(E), lde, e_batch_stride, wtab, pc, N, P));
  CA_CUDA(cudaGetLastError());
  return 0;
}

int focal_finalize_launch(const float* pc, const float* cbias, float* attn, const float* rs_in, float* rs_out, int B,
                          int N, int P, float focus_strength, int mode, const float* cur_weight, float adaptive_weight,
                          cudaStream_t stream) {
  CA_REQUIRE(pc && attn, "focal_finalize: null pointer");
  CA_REQUIRE(mode != 0 || cbias, "focal_finalize: null centre bias");
  CA_REQUIRE(N <= kFinalizeThreads * kFinalizeCols, "focal_finalize: more than 8192 patch tokens per image");
  CA_TRY(launch_kernel(focal_finalize_kernel, dim3(B), dim3(kFinalizeThreads), 0, stream, pc, cbias, attn, rs_in, rs_out, N, P, focus_strength, mode,
                                                  cur_weight, adaptive_weight));
  CA_CUDA(cudaGetLastError());
  return 0;
}

int guided_softmax_launch(const float* base, const float* mask, long long mask_batch_stride, float* heat, int* argmax,
                          int B, int N, float alpha, float temperature, cudaStream_t stream) {
  CA_REQUIRE(base && mask && heat, "guided_softmax: null pointer");
  CA_REQUIRE(mask_batch_stride == 0 || mask_batch_stride >= N, "guided_softmax: mask batch stride must be 0 or >= N");
  CA_TRY(launch_kernel(guided_softmax_kernel, dim3(B), dim3(256), 0, stream, base, 0LL, mask, 0LL, mask_batch_stride, heat,
                       argmax, B, N, alpha, temperature));
  CA_CUDA(cudaGetLastError());
  return 0;
}

int guided_softmax_sweep_launch(const float* base, long long base_k_stride, const float* mask, long long mask_k_stride,
                                long long mask_batch_stride, float* heat, int* argmax, int K, int B, int N, float alpha,
                                float temperature, cudaStream_t stream) {
  CA_REQUIRE(base && mask && heat, "guided_softmax_sweep: null pointer");
  CA_REQUIRE(K >= 1 && K <= kSweepMaxK && B > 0 && N > 0, "guided_softmax_sweep: 1..16 instructions, B > 0, N > 0");
  CA_REQUIRE(base_k_stride == 0 || base_k_stride >= static_cast<long long>(B) * N,
             "guided_softmax_sweep: base stride per instruction must be 0 or >= B * N");
  CA_REQUIRE(mask_batch_stride == 0 || mask_batch_stride >= N, "guided_softmax_sweep: mask batch stride must be 0 or >= N");
  CA_REQUIRE(mask_k_stride == 0 || mask_k_stride >= N, "guided_softmax_sweep: mask stride per instruction must be 0 or >= N");
  CA_TRY(launch_kernel(guided_softmax_kernel, dim3(K * B), dim3(256), 0, stream, base, base_k_stride, mask, mask_k_stride,
                       mask_batch_stride, heat, argmax, B, N, alpha, temperature));
  CA_CUDA(cudaGetLastError());
  return 0;
}

int weighted_pool_launch(const float* src, long long src_batch_stride, int row_offset, const float* w, const float* w2,
                         float* partial, int B, int N, int D, int splits, cudaStream_t stream) {
  CA_REQUIRE(src && w && partial, "weighted_pool: null pointer");
  CA_REQUIRE(D == 768, "weighted_pool: only D = 768 is instantiated");
  CA_REQUIRE(splits > 0, "weighted_pool: splits must be positive");
  const int rps = (N + splits - 1) / splits;
  CA_TRY(launch_kernel(weighted_pool_kernel, dim3(dim3(splits, B)), dim3(192), 0, stream, src, src_batch_stride, row_offset, w, w2, partial, N, D, rps));
  CA_CUDA(cudaGetLastError());
  return 0;
}

int weighted_pool_sweep_launch(const float* src, long long src_batch_stride, int row_offset, const float* w, float* partial,
                               int K, int B, int N, int D, int splits, cudaStream_t stream) {
  CA_REQUIRE(src && w && partial, "weighted_pool_sweep: null pointer");
  CA_REQUIRE(D == 768, "weighted_pool_sweep: only D = 768 is instantiated");
  CA_REQUIRE(splits > 0 && B > 0 && N > 0, "weighted_pool_sweep: splits, B and N must be positive");
  CA_REQUIRE(K >= 1 && K <= kSweepMaxK, "weighted_pool_sweep: 1..16 weight vectors");
  const int rps = (N + splits - 1) / splits;  // the split of weighted_pool_launch: the partials must line up with it
  const dim3 grid(splits, B);
  // the smallest instantiation that holds K accumulators: registers (and so occupancy) follow K
  if (K <= 4)
    CA_TRY(launch_kernel(weighted_pool_sweep_kernel<4>, grid, dim3(192), 0, stream, src, src_batch_stride, row_offset, w,
                         partial, K, B, N, D, rps));
  else if (K <= 8)
    CA_TRY(launch_kernel(weighted_pool_sweep_kernel<8>, grid, dim3(192), 0, stream, src, src_batch_stride, row_offset, w,
                         partial, K, B, N, D, rps));
  else
    CA_TRY(launch_kernel(weighted_pool_sweep_kernel<kSweepMaxK>, grid, dim3(192), 0, stream, src, src_batch_stride,
                         row_offset, w, partial, K, B, N, D, rps));
  CA_CUDA(cudaGetLastError());
  return 0;
}

int guide_tail_launch(const HeadsWeights& w, const HeadsInputs& in, const float* base, const float* mask,
                      long long mask_batch_stride, float* heat, int* argmax, unsigned int* ticket, float* depth,
                      float* conf, int B, int N, float alpha, float temperature, cudaStream_t stream) {
  CA_REQUIRE(base && mask && heat && ticket && depth && conf && in.tokens, "guide_tail: null pointer");
  CA_REQUIRE(in.focal_feat == nullptr && in.sweep_images == 0, "guide_tail: guided single calls only (no focal_feat, no sweep)");
  CA_REQUIRE(in.pool_partial && in.tmp_w && in.tmp_b && in.pool_splits > 0, "guide_tail: pool partials and projection needed");
  CA_REQUIRE(in.exif == nullptr || in.camera_idx != nullptr, "guide_tail: EXIF given without camera_idx");
  CA_REQUIRE(B > 0 && N > 0 && N <= kTailMaxN, "guide_tail: B > 0 and 0 < N <= 8192");
  CA_REQUIRE(in.tokens_per_img == N + 1, "guide_tail: tokens_per_img must be N + 1 (CLS + patch tokens)");
  CA_REQUIRE(mask_batch_stride == 0 || mask_batch_stride >= N, "guide_tail: mask batch stride must be 0 or >= N");
  CA_TRY(launch_kernel(guide_tail_kernel, dim3(in.pool_splits, B), dim3(kHeadsThreads), 0, stream, w, in, base, mask,
                       mask_batch_stride, heat, argmax, const_cast<float*>(in.pool_partial), ticket, depth, conf, N, alpha,
                       temperature));
  CA_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace ca
