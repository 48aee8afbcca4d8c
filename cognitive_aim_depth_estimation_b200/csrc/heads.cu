// Fused "everything after the token matrices" kernel: ambient MLP, (guided) focal projection, EXIF prior,
// fusion layer, depth and confidence heads.  One CTA per image, fp32, weights read straight from L2
// (~1.3 MB total, shared by every CTA), activations in shared memory; every dot product is one warp with
// coalesced weight-row reads and a shuffle reduction.
// Reference: src/model.py:46-53 (AmbientStream), :482-519 (EXIFPriorDatabase), :1418-1422 (temporary projection),
// :311,430 (FocalStream.projection / IterativeFocalStream.fusion, un-guided), :908-945,1223-1230 (fusion + heads).
#include "common.cuh"
#include "dense.cuh"
#include "heads.cuh"
#include "heads_row.cuh"
#include "host.h"

namespace ca {
namespace {

__global__ void __launch_bounds__(kHeadsThreads) heads_kernel(const HeadsWeights wt, const HeadsInputs in,
                                                              float* __restrict__ depth, float* __restrict__ conf,
                                                              float* __restrict__ fused_out) {
  griddep_sync();  // PDL: nothing before this line reads or writes global memory
  // r: output row.  In an instruction sweep r = k * B + b (k = call, sweep_images = B), otherwise r = b.
  heads_row(wt, in, depth, conf, fused_out, blockIdx.x, in.sweep_images > 0 ? in.sweep_images : gridDim.x);
}

// Un-guided focal features of ONE iteration (reference src/model.py:204,308-311 re-associated):
//   weighted = (sum_j c_j x~_j) Wv^T + bv   with  sum_j c_j = 1,   feat = projection(weighted)
// pooled x~ arrives as split partials of (tokens*rowscale) plus split partials of the PE table.
__global__ void __launch_bounds__(kHeadsThreads) focal_value_kernel(const FocalValueArgs a) {
  griddep_sync();  // PDL: nothing before this line reads or writes global memory
  __shared__ __align__(16) float s_x[768];
  __shared__ __align__(16) float s_v[768];
  __shared__ __align__(16) float s_h[256];
  const int b = blockIdx.x;
  const int tid = threadIdx.x;
  for (int i = tid; i < 768; i += kHeadsThreads) {
    float acc = 0.f;
    for (int s = 0; s < a.splits; ++s) {
      acc += a.tok_partial[(static_cast<size_t>(b) * a.splits + s) * 768 + i];
      acc += a.pe_partial[(static_cast<size_t>(b) * a.splits + s) * 768 + i];
    }
    s_x[i] = acc;
  }
  __syncthreads();
  dense(a.wv, a.bv, s_x, s_v, 768, 768, false);
  dense(a.proj_w0, a.proj_b0, s_v, s_h, 768, 256, true);
  dense(a.proj_w1, a.proj_b1, s_h, s_x, 256, 64, false);
  for (int i = tid; i < 64; i += kHeadsThreads) a.feat_out[(static_cast<size_t>(b) * a.n_iters + a.iter) * 64 + i] = s_x[i];
}

// fused[b, :] = fusion(cat(feat[b, 0..iters-1, :]))   (src/model.py:430)
__global__ void __launch_bounds__(kHeadsThreads) focal_fusion_kernel(const float* __restrict__ feats, int n_iters,
                                                                     const float* w0, const float* b0, const float* w1,
                                                                     const float* b1, float* __restrict__ out) {
  griddep_sync();  // PDL: nothing before this line reads or writes global memory
  __shared__ __align__(16) float s_in[256];
  __shared__ __align__(16) float s_h[128];
  __shared__ __align__(16) float s_o[64];
  const int b = blockIdx.x;
  const int n = n_iters * 64;
  for (int i = threadIdx.x; i < n; i += kHeadsThreads) s_in[i] = feats[static_cast<size_t>(b) * n + i];
  __syncthreads();
  dense(w0, b0, s_in, s_h, n, 128, true);
  dense(w1, b1, s_h, s_o, 128, 64, false);
  for (int i = threadIdx.x; i < 64; i += kHeadsThreads) out[static_cast<size_t>(b) * 64 + i] = s_o[i];
}

}  // namespace

int heads_launch(const HeadsWeights& w, const HeadsInputs& in, float* depth, float* conf, float* fused_out, int B,
                 cudaStream_t stream) {
  CA_REQUIRE(depth && conf && in.tokens, "heads: null pointer");
  CA_REQUIRE(in.focal_feat || (in.pool_partial && in.tmp_w && in.tmp_b && in.pool_splits > 0),
             "heads: neither focal features nor pooled partials + projection given");
  CA_REQUIRE(in.exif == nullptr || in.camera_idx != nullptr, "heads: EXIF given without camera_idx");
  CA_REQUIRE(in.sweep_images >= 0 && (in.sweep_images == 0 || (in.focal_feat == nullptr && B % in.sweep_images == 0)),
             "heads: an instruction sweep is guided only and needs B = K * sweep_images rows");
  CA_TRY(launch_kernel(heads_kernel, dim3(B), dim3(kHeadsThreads), 0, stream, w, in, depth, conf, fused_out));
  CA_CUDA(cudaGetLastError());
  return 0;
}

int focal_value_launch(const FocalValueArgs& a, int B, cudaStream_t stream) {
  CA_REQUIRE(a.tok_partial && a.pe_partial && a.wv && a.bv && a.feat_out, "focal_value: null pointer");
  CA_REQUIRE(a.n_iters >= 1 && a.n_iters <= 4, "focal_value: 1..4 iterations supported");
  CA_TRY(launch_kernel(focal_value_kernel, dim3(B), dim3(kHeadsThreads), 0, stream, a));
  CA_CUDA(cudaGetLastError());
  return 0;
}

int focal_fusion_launch(const float* feats, int n_iters, const float* w0, const float* b0, const float* w1,
                        const float* b1, float* out, int B, cudaStream_t stream) {
  CA_REQUIRE(feats && w0 && b0 && w1 && b1 && out, "focal_fusion: null pointer");
  CA_REQUIRE(n_iters >= 1 && n_iters <= 4, "focal_fusion: 1..4 iterations supported");
  CA_TRY(launch_kernel(focal_fusion_kernel, dim3(B), dim3(kHeadsThreads), 0, stream, feats, n_iters, w0, b0, w1, b1, out));
  CA_CUDA(cudaGetLastError());
  return 0;
}

}  // namespace ca
