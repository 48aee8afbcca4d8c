// The body of the fused heads kernel for ONE output row: ambient MLP on the CLS token, focal slot (un-guided features or
// the guided pool + per-call projection), EXIF prior, fusion, depth and confidence.  Shared by heads_kernel (csrc/heads.cu,
// one CTA per row) and guide_tail_kernel (csrc/focal.cu, the last CTA of an image), so both give the same bits.
// Needs a CTA of kHeadsThreads threads: every dense() output is reduced within one warp, so the result does not depend
// on the warp count, but the strided loops below assume the whole CTA takes part.
#pragma once

#include "common.cuh"
#include "dense.cuh"
#include "heads.cuh"

namespace ca {
namespace {

// r: output row; b = r % nb: image; k = r / nb: instruction of a sweep (0 otherwise), or in.call_of_row[r] (the rows of
// several guide calls).
__device__ __forceinline__ void heads_row(const HeadsWeights& wt, const HeadsInputs& in, float* __restrict__ depth,
                                          float* __restrict__ conf, float* __restrict__ fused_out, int r, int nb) {
  __shared__ __align__(16) float s_in[768];
  __shared__ __align__(16) float s_a[256];
  __shared__ __align__(16) float s_b[256];
  __shared__ __align__(16) float s_cat[192];
  __shared__ __align__(16) float s_f[192];
  const int b = r % nb;
  const int tid = threadIdx.x;

  // ---- ambient stream on the CLS token ----
  const float* cls = in.tokens + static_cast<size_t>(b) * in.tokens_per_img * 768;
  for (int i = tid; i < 768; i += kHeadsThreads) s_in[i] = cls[i];
  __syncthreads();
  dense(wt.amb_w0, wt.amb_b0, s_in, s_a, 768, 256, true);
  dense(wt.amb_w1, wt.amb_b1, s_a, s_b, 256, 128, true);
  dense(wt.amb_w2, wt.amb_b2, s_b, s_cat + 0, 128, 64, false);

  // ---- focal slot ----
  if (in.focal_feat != nullptr) {  // un-guided: features already computed by the focal value path
    for (int i = tid; i < 64; i += kHeadsThreads) s_cat[64 + i] = in.focal_feat[static_cast<size_t>(b) * 64 + i];
    __syncthreads();
  } else {  // guided: pooled = sum of the split partials (fixed order => deterministic), then the per-call projection
    for (int i = tid; i < 768; i += kHeadsThreads) {
      float acc = 0.f;
      // L2-coherent loads: in guide_tail_kernel other CTAs of the same launch wrote these partials
      for (int s = 0; s < in.pool_splits; ++s)
        acc += __ldcg(in.pool_partial + (static_cast<size_t>(r) * in.pool_splits + s) * 768 + i);
      s_in[i] = acc;
      if (in.pooled_out) in.pooled_out[static_cast<size_t>(r) * 768 + i] = acc;
    }
    __syncthreads();
    const size_t k = in.call_of_row ? static_cast<size_t>(in.call_of_row[r]) : static_cast<size_t>(r / nb);
    dense(in.tmp_w + k * 64 * 768, in.tmp_b + k * 64, s_in, s_cat + 64, 768, 64, false);
  }

  // ---- EXIF prior (zero slot when EXIF is absent: the reference zero-pads, src/model.py:1035-1039) ----
  if (in.exif != nullptr) {
    const float* e = in.exif + static_cast<size_t>(b) * 3;
    if (tid == 0) {
      s_in[0] = e[0];
      s_in[1] = e[1];
      s_in[2] = logf(e[2] + 1.0f);
    }
    // camera index checked HERE, not on the host: no device-to-host sync on the call path.  An index outside the
    // embedding table is clamped (no out-of-bounds read) and reported through the fault word, which the host reads
    // without synchronising (pinned memory) before its next call — nn.Embedding would have raised (src/model.py:491).
    long long cam = in.camera_idx[b];
    if (in.num_cameras > 0 && (cam < 0 || cam >= in.num_cameras)) {
      if (tid == 0 && in.fault) atomicOr(in.fault, 1);
      cam = cam < 0 ? 0 : in.num_cameras - 1;
    }
    for (int i = tid; i < 64; i += kHeadsThreads) s_b[i] = wt.cam_emb[cam * 64 + i];  // cat([camera, exif]) slot 0..63
    __syncthreads();
    dense(wt.exif_w0, wt.exif_b0, s_in, s_a, 3, 64, true);
    dense(wt.exif_w1, wt.exif_b1, s_a, s_b + 64, 64, 64, false);
    dense(wt.exif_f0, wt.exif_fb0, s_b, s_a, 128, 256, true);
    dense(wt.exif_f1, wt.exif_fb1, s_a, s_cat + 128, 256, 64, false);
  } else {
    for (int i = tid; i < 64; i += kHeadsThreads) s_cat[128 + i] = 0.f;
    __syncthreads();
  }

  // ---- fusion + heads ----
  dense(wt.fus_w, wt.fus_b, s_cat, s_f, 192, 192, true);
  if (fused_out)
    for (int i = tid; i < 192; i += kHeadsThreads) fused_out[static_cast<size_t>(r) * 192 + i] = s_f[i];
  if (warp_id() < 2) {
    const float* w = warp_id() == 0 ? wt.dec_w : wt.conf_w0;
    float acc = 0.f;
    for (int i = lane_id(); i < 192; i += 32) acc = fmaf(w[i], s_f[i], acc);
    acc = warp_sum(acc);
    if (lane_id() == 0) {
      if (warp_id() == 0) {
        const float z = acc + wt.dec_b[0];
        depth[r] = z > 20.0f ? z : log1pf(expf(z));  // Softplus(beta=1, threshold=20)
      } else {
        const float c = fmaxf(acc + wt.conf_b0[0], 0.f);
        const float z = c * wt.conf_w2[0] + wt.conf_b2[0];
        conf[r] = 1.0f / (1.0f + expf(-z));
      }
    }
  }
}

}  // namespace
}  // namespace ca
