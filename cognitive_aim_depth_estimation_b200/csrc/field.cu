// Depth fields: the guided depth and confidence of one scene with the focus on every cell of the g x g patch grid
// (CognitiveAimModel.depth_field, ca_depth_field).  Cell c is the guided call whose mask is tables.focus_mask(c): 5.0 on
// the disk dy^2 + dx^2 <= r^2 around c, 2.0 on the ring out to 2r, 1.0 elsewhere, r = max(1, g / 6).
//
//   token_project     : P[b, n, :] = tokens[b, 1 + n, :] . Wtmp^T, the call's projection applied to every patch token once
//                       (it is linear, so pooling P with the guided weights is pooling the tokens and projecting after)
//   field_const       : per image, the fusion layer's pre-activation without its focal slot: ambient stream on CLS,
//                       EXIF prior and fusion bias (the focal slot zeroed), as heads_row computes them
//   depth_field_cells : per cell, the guided softmax over the cell's disk, the pooled 64-vector of P, the focal slice of
//                       the fusion layer (192 x 64) and the decision / confidence heads
// No atomics in any reduction: every sum has a fixed order, so results do not depend on scheduling.
#include "common.cuh"
#include "dense.cuh"
#include "field.cuh"
#include "host.h"

namespace ca {
namespace {

// ---- token projection: fp32 tiles of 128 tokens x 64 outputs, K = 768 in chunks of 32 staged in shared memory ----
constexpr int kProjRows = 128, kProjK = 32, kProjThreads = 256;

__global__ void __launch_bounds__(kProjThreads) token_project_kernel(const float* __restrict__ src,
                                                                    long long src_batch_stride, int row_offset,
                                                                    const float* __restrict__ W, float* __restrict__ P,
                                                                    int N, int M) {
  griddep_sync();  // PDL: nothing before this line reads or writes global memory
  __shared__ __align__(16) float As[kProjK][kProjRows + 4];  // [k][token]
  __shared__ __align__(16) float Ws[kProjK][64 + 4];         // [k][output]
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;  // outputs tx*4 .. +3, tokens ty*8 .. +7
  const int m0 = blockIdx.x * kProjRows;
  // loader roles: 1024 float4 of the token tile (4 per thread) and 512 of the weight tile (2 per thread), 8 per row
  const float4* arow[4];
  bool aok[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int f = tid + kProjThreads * j;
    const int m = m0 + (f >> 3);
    aok[j] = m < M;
    const int mm = aok[j] ? m : M - 1;
    const int b = mm / N, n = mm - b * N;
    arow[j] = reinterpret_cast<const float4*>(src + static_cast<size_t>(b) * src_batch_stride +
                                              static_cast<size_t>(row_offset + n) * 768) + (f & 7);
  }
  const float4* wrow[2];
#pragma unroll
  for (int j = 0; j < 2; ++j) {
    const int f = tid + kProjThreads * j;
    wrow[j] = reinterpret_cast<const float4*>(W + static_cast<size_t>(f >> 3) * 768) + (f & 7);
  }
  float acc[8][4];
#pragma unroll
  for (int r = 0; r < 8; ++r)
#pragma unroll
    for (int o = 0; o < 4; ++o) acc[r][o] = 0.f;

  float4 av[4], wv[2];
#pragma unroll
  for (int j = 0; j < 4; ++j) av[j] = aok[j] ? __ldg(arow[j]) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
  for (int j = 0; j < 2; ++j) wv[j] = __ldg(wrow[j]);
  for (int k0 = 0; k0 < 768; k0 += kProjK) {
    __syncthreads();  // the previous chunk has been consumed
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int f = tid + kProjThreads * j, row = f >> 3, k = (f & 7) * 4;
      As[k + 0][row] = av[j].x;
      As[k + 1][row] = av[j].y;
      As[k + 2][row] = av[j].z;
      As[k + 3][row] = av[j].w;
    }
#pragma unroll
    for (int j = 0; j < 2; ++j) {
      const int f = tid + kProjThreads * j, o = f >> 3, k = (f & 7) * 4;
      Ws[k + 0][o] = wv[j].x;
      Ws[k + 1][o] = wv[j].y;
      Ws[k + 2][o] = wv[j].z;
      Ws[k + 3][o] = wv[j].w;
    }
    __syncthreads();
    if (k0 + kProjK < 768) {  // the next chunk's loads are in flight during this chunk's FMAs
      const int q = (k0 + kProjK) / 4;
#pragma unroll
      for (int j = 0; j < 4; ++j) av[j] = aok[j] ? __ldg(arow[j] + q) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int j = 0; j < 2; ++j) wv[j] = __ldg(wrow[j] + q);
    }
#pragma unroll
    for (int k = 0; k < kProjK; ++k) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[k][ty * 8]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[k][ty * 8 + 4]);
      const float4 w = *reinterpret_cast<const float4*>(&Ws[k][tx * 4]);
      const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
#pragma unroll
      for (int r = 0; r < 8; ++r) {
        ffma2v(acc[r][0], acc[r][1], w.x, w.y, a[r], a[r], acc[r][0], acc[r][1]);
        ffma2v(acc[r][2], acc[r][3], w.z, w.w, a[r], a[r], acc[r][2], acc[r][3]);
      }
    }
  }
#pragma unroll
  for (int r = 0; r < 8; ++r) {
    const int m = m0 + ty * 8 + r;
    if (m < M)
      reinterpret_cast<float4*>(P + static_cast<size_t>(m) * 64)[tx] =
          make_float4(acc[r][0], acc[r][1], acc[r][2], acc[r][3]);
  }
}

// ---- per-image constant of the fusion layer: heads_row's ambient and EXIF stages, then fusion with a zero focal slot ----
__global__ void __launch_bounds__(kHeadsThreads) field_const_kernel(const HeadsWeights wt, const HeadsInputs in,
                                                                   float* __restrict__ cst) {
  griddep_sync();  // PDL: nothing before this line reads or writes global memory
  __shared__ __align__(16) float s_in[768];
  __shared__ __align__(16) float s_a[256];
  __shared__ __align__(16) float s_b[256];
  __shared__ __align__(16) float s_cat[192];
  __shared__ __align__(16) float s_f[192];
  const int b = blockIdx.x;
  const int tid = threadIdx.x;

  const float* cls = in.tokens + static_cast<size_t>(b) * in.tokens_per_img * 768;
  for (int i = tid; i < 768; i += kHeadsThreads) s_in[i] = cls[i];
  __syncthreads();
  dense(wt.amb_w0, wt.amb_b0, s_in, s_a, 768, 256, true);
  dense(wt.amb_w1, wt.amb_b1, s_a, s_b, 256, 128, true);
  dense(wt.amb_w2, wt.amb_b2, s_b, s_cat + 0, 128, 64, false);
  for (int i = tid; i < 64; i += kHeadsThreads) s_cat[64 + i] = 0.f;  // the focal slot is added per cell

  if (in.exif != nullptr) {
    const float* e = in.exif + static_cast<size_t>(b) * 3;
    if (tid == 0) {
      s_in[0] = e[0];
      s_in[1] = e[1];
      s_in[2] = logf(e[2] + 1.0f);
    }
    // the camera index is range-checked here, as heads_row does: clamped, and reported through the fault word
    long long cam = in.camera_idx[b];
    if (in.num_cameras > 0 && (cam < 0 || cam >= in.num_cameras)) {
      if (tid == 0 && in.fault) atomicOr(in.fault, 1);
      cam = cam < 0 ? 0 : in.num_cameras - 1;
    }
    for (int i = tid; i < 64; i += kHeadsThreads) s_b[i] = wt.cam_emb[cam * 64 + i];
    __syncthreads();
    dense(wt.exif_w0, wt.exif_b0, s_in, s_a, 3, 64, true);
    dense(wt.exif_w1, wt.exif_b1, s_a, s_b + 64, 64, 64, false);
    dense(wt.exif_f0, wt.exif_fb0, s_b, s_a, 128, 256, true);
    dense(wt.exif_f1, wt.exif_fb1, s_a, s_cat + 128, 256, 64, false);
  } else {
    for (int i = tid; i < 64; i += kHeadsThreads) s_cat[128 + i] = 0.f;
    __syncthreads();
  }
  dense(wt.fus_w, wt.fus_b, s_cat, s_f, 192, 192, false);  // ReLU after the focal slot is added
  for (int i = tid; i < 192; i += kHeadsThreads) cst[static_cast<size_t>(b) * 192 + i] = s_f[i];
}

// ---- cells: one warp per group of 4 cells, 8 warps and 64 cells per CTA, grid (cell tiles, B) ----
constexpr int kCellThreads = 256, kCellWarps = kCellThreads / 32, kCellGroup = 4, kCellsPerCta = 64;
constexpr int kFusPitch = 65;  // focal slice of fusion.0 as [192][65]: lane o reads row o, conflict-free at any column
constexpr float kFocusInner = 5.0f;  // the focus mask's value on the disk (tables.focus_mask)
constexpr size_t kCellSmemBytes = (192 * kFusPitch + 3 * 192 + kCellWarps * 64 * kCellGroup) * sizeof(float);

__global__ void __launch_bounds__(kCellThreads) depth_field_cells_kernel(const HeadsWeights wt,
                                                                        const float* __restrict__ tmp_b,
                                                                        const float* __restrict__ base,
                                                                        const float* __restrict__ P,
                                                                        const float* __restrict__ cst,
                                                                        float* __restrict__ depth,
                                                                        float* __restrict__ conf, int g, float alpha,
                                                                        float temperature) {
  griddep_sync();  // PDL: nothing before this line reads or writes global memory
  extern __shared__ __align__(16) float smem[];
  float* s_w = smem;                    // fusion.0 weight columns 64..127: s_w[o * kFusPitch + j] = W[o, 64 + j]
  float* s_cst = s_w + 192 * kFusPitch;  // this image's constant
  float* s_dec = s_cst + 192;
  float* s_cw = s_dec + 192;
  float* s_feat = s_cw + 192;  // per warp [64][kCellGroup]: the pooled focal features of its cells
  const int b = blockIdx.y, tid = threadIdx.x, w = warp_id(), l = lane_id();
  const int N = g * g;
  for (int i = tid; i < 192 * 64; i += kCellThreads) s_w[(i >> 6) * kFusPitch + (i & 63)] = __ldg(wt.fus_w + (i >> 6) * 192 + 64 + (i & 63));
  for (int i = tid; i < 192; i += kCellThreads) {
    s_cst[i] = cst[static_cast<size_t>(b) * 192 + i];
    s_dec[i] = __ldg(wt.dec_w + i);
    s_cw[i] = __ldg(wt.conf_w0 + i);
  }
  __syncthreads();

  const int r = max(1, g / 6), r2 = r * r, box = 2 * r + 1;
  const float* ab = base + static_cast<size_t>(b) * N;
  const float* Pb = P + static_cast<size_t>(b) * N * 64;
  const float2 tb = reinterpret_cast<const float2*>(tmp_b)[l];
  float* feat = s_feat + w * 64 * kCellGroup;
  const float beta = 1.0f - alpha;
  const float inner = alpha * kFocusInner;
  const int c_end = min(N, (blockIdx.x + 1) * kCellsPerCta);
  for (int c0 = blockIdx.x * kCellsPerCta + w * kCellGroup; c0 < c_end; c0 += kCellWarps * kCellGroup) {
#pragma unroll 1
    for (int q = 0; q < kCellGroup; ++q) {
      const int c = min(c0 + q, N - 1);  // a tail group repeats the last cell (not stored)
      const int cy = c / g, cx = c - cy * g;
      // The guided weights of cell c are softmax(L) with L[n] = (alpha * mask[n] + (1 - alpha) * a[n]) / temperature,
      // the expression of guided_softmax_kernel.  a is a probability vector (0 <= a <= 1) and alpha = 0.7,
      // temperature = 0.05, so L >= 70 on the r-disk (mask 5), L <= 34 on the 2r-ring (mask 2) and L <= 20 elsewhere
      // (mask 1): everything outside the disk weighs less than N * e^-36 relative to it, 2e-12 for N <= 8192, far below
      // fp32 rounding.  The softmax is therefore taken over the disk alone (its maximum is the global one).
      float mx = -INFINITY;
      for (int t = l; t < box * box; t += 32) {
        const int dy = t / box - r, dx = t % box - r, y = cy + dy, x = cx + dx;
        if (dy * dy + dx * dx <= r2 && y >= 0 && y < g && x >= 0 && x < g)
          mx = fmaxf(mx, (inner + beta * ab[y * g + x]) / temperature);
      }
      mx = warp_max(mx);
      float tot = 0.f;
      for (int t = l; t < box * box; t += 32) {
        const int dy = t / box - r, dx = t % box - r, y = cy + dy, x = cx + dx;
        if (dy * dy + dx * dx <= r2 && y >= 0 && y < g && x >= 0 && x < g)
          tot += expf((inner + beta * ab[y * g + x]) / temperature - mx);
      }
      tot = warp_sum(tot);  // every lane holds the same bits (xor butterfly)
      // pooled 64-vector: lane l owns channels 2l, 2l + 1; the disk row by row, each row a contiguous run of P
      float a0 = 0.f, a1 = 0.f;
      const int dy0 = max(-r, -cy), dy1 = min(r, g - 1 - cy);
      for (int dy = dy0; dy <= dy1; ++dy) {
        int half = r;
        while (dy * dy + half * half > r2) --half;
        const int y = cy + dy, x0 = max(cx - half, 0), x1 = min(cx + half, g - 1);
#pragma unroll 4
        for (int x = x0; x <= x1; ++x) {
          const int n = y * g + x;
          const float h = expf((inner + beta * ab[n]) / temperature - mx) / tot;
          const float2 p = reinterpret_cast<const float2*>(Pb + static_cast<size_t>(n) * 64)[l];
          a0 = fmaf(h, p.x, a0);
          a1 = fmaf(h, p.y, a1);
        }
      }
      feat[(2 * l) * kCellGroup + q] = a0 + tb.x;
      feat[(2 * l + 1) * kCellGroup + q] = a1 + tb.y;
    }
    __syncwarp();
    // fusion (focal slice) + heads for the group: lane l owns outputs l + 32 i, i < 6, for the 4 cells
    float acc[6][kCellGroup];
#pragma unroll
    for (int i = 0; i < 6; ++i)
#pragma unroll
      for (int q = 0; q < kCellGroup; ++q) acc[i][q] = s_cst[l + 32 * i];
#pragma unroll 4
    for (int j = 0; j < 64; ++j) {
      const float4 f = reinterpret_cast<const float4*>(feat)[j];
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        const float wv = s_w[(l + 32 * i) * kFusPitch + j];
        ffma2v(acc[i][0], acc[i][1], f.x, f.y, wv, wv, acc[i][0], acc[i][1]);
        ffma2v(acc[i][2], acc[i][3], f.z, f.w, wv, wv, acc[i][2], acc[i][3]);
      }
    }
    __syncwarp();  // feat is rewritten by the next group
    float zd[kCellGroup], zc[kCellGroup];
#pragma unroll
    for (int q = 0; q < kCellGroup; ++q) {
      zd[q] = 0.f;
      zc[q] = 0.f;
#pragma unroll
      for (int i = 0; i < 6; ++i) {
        const float f = fmaxf(acc[i][q], 0.f);
        zd[q] = fmaf(s_dec[l + 32 * i], f, zd[q]);
        zc[q] = fmaf(s_cw[l + 32 * i], f, zc[q]);
      }
      zd[q] = warp_sum(zd[q]);
      zc[q] = warp_sum(zc[q]);
    }
    if (l == 0) {
#pragma unroll
      for (int q = 0; q < kCellGroup; ++q) {
        if (c0 + q >= N) break;
        const size_t o = static_cast<size_t>(b) * N + c0 + q;
        const float z = zd[q] + wt.dec_b[0];
        depth[o] = z > 20.0f ? z : log1pf(expf(z));  // Softplus(beta=1, threshold=20)
        const float cc = fmaxf(zc[q] + wt.conf_b0[0], 0.f);
        const float zz = cc * wt.conf_w2[0] + wt.conf_b2[0];
        conf[o] = 1.0f / (1.0f + expf(-zz));
      }
    }
  }
}

}  // namespace

int token_project_launch(const float* src, long long src_batch_stride, int row_offset, const float* tmp_w, float* P,
                         int B, int N, cudaStream_t stream) {
  CA_REQUIRE(src && tmp_w && P, "token_project: null pointer");
  CA_REQUIRE(B > 0 && N > 0 && row_offset >= 0, "token_project: B > 0, N > 0 and row_offset >= 0");
  CA_REQUIRE(src_batch_stride >= static_cast<long long>(row_offset + N) * 768,
             "token_project: src batch stride must hold row_offset + N rows of 768");
  CA_REQUIRE(static_cast<long long>(B) * N <= 0x7fffffffLL, "token_project: B * N must fit in int");
  CA_REQUIRE((reinterpret_cast<uintptr_t>(src) & 15) == 0 && src_batch_stride % 4 == 0 &&
                 (reinterpret_cast<uintptr_t>(tmp_w) & 15) == 0 && (reinterpret_cast<uintptr_t>(P) & 15) == 0,
             "token_project: src, tmp_w and P must be 16-byte aligned (src batch stride a multiple of 4)");
  const int M = B * N;
  CA_TRY(launch_kernel(token_project_kernel, dim3((M + kProjRows - 1) / kProjRows), dim3(kProjThreads), 0, stream, src,
                       src_batch_stride, row_offset, tmp_w, P, N, M));
  CA_CUDA(cudaGetLastError());
  return 0;
}

int depth_field_cells_launch(const HeadsWeights& w, const HeadsInputs& in, const float* base, const float* P, float* cst,
                             float* depth, float* conf, int B, int g, float alpha, float temperature,
                             cudaStream_t stream) {
  CA_REQUIRE(base && P && cst && depth && conf && in.tokens && in.tmp_b, "depth_field_cells: null pointer");
  CA_REQUIRE(in.exif == nullptr || in.camera_idx != nullptr, "depth_field_cells: EXIF given without camera_idx");
  CA_REQUIRE(B > 0 && g > 0 && g <= 4096, "depth_field_cells: B > 0 and 0 < g <= 4096");
  // the disk-only softmax needs the disk's logits (>= 5 alpha / T) to exceed all others (<= (1 + alpha) / T) by ~36
  CA_REQUIRE(alpha > 0.25f && alpha <= 1.0f && temperature > 0.f && (4.0f * alpha - 1.0f) / temperature >= 35.9f,
             "depth_field_cells: alpha / temperature leave the focus disk less than e^36 above the rest of the grid");
  CA_REQUIRE(in.tokens_per_img >= 1, "depth_field_cells: tokens_per_img must be positive");
  CA_REQUIRE((reinterpret_cast<uintptr_t>(P) & 7) == 0 && (reinterpret_cast<uintptr_t>(in.tmp_b) & 7) == 0,
             "depth_field_cells: P and tmp_b must be 8-byte aligned");
  static PerDeviceOnce configured;
  CA_TRY(configured.run([&]() -> int {
    CA_CUDA(cudaFuncSetAttribute(depth_field_cells_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 static_cast<int>(kCellSmemBytes)));
    return 0;
  }));
  CA_TRY(launch_kernel(field_const_kernel, dim3(B), dim3(kHeadsThreads), 0, stream, w, in, cst));
  CA_CUDA(cudaGetLastError());
  const int N = g * g;
  CA_TRY(launch_kernel(depth_field_cells_kernel, dim3((N + kCellsPerCta - 1) / kCellsPerCta, B), dim3(kCellThreads),
                       kCellSmemBytes, stream, w, in.tmp_b, base, P, static_cast<const float*>(cst), depth, conf, g, alpha,
                       temperature));
  CA_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace ca
