// Launchers of the depth-field kernels (csrc/field.cu): the guided depth and confidence with the focus on every cell of
// the g x g patch grid, from a scene's tokens and last focal attention.
#pragma once

#include <cuda_runtime.h>

#include "heads.cuh"

namespace ca {

// Largest patch grid of a field: the model's largest image side (1260 = 90 x 14).
constexpr int kFieldMaxGrid = 90;

// P[b, n, :] = src[b * src_batch_stride + (row_offset + n) * 768 + :] . tmp_w^T  ->  [B, N, 64] fp32.
int token_project_launch(const float* src, long long src_batch_stride, int row_offset, const float* tmp_w, float* P,
                         int B, int N, cudaStream_t stream);
// depth[b, c], conf[b, c] of a guided call with the focus mask of cell c (tables.focus_mask), for every cell c of the
// g x g grid.  in.tokens (CLS rows), in.tmp_b, in.exif / camera_idx / num_cameras / fault are read as ca_heads reads
// them; in.tmp_w and in.pool_partial are not (the projection is already in P).  cst: [B, 192] scratch.
int depth_field_cells_launch(const HeadsWeights& w, const HeadsInputs& in, const float* base, const float* P, float* cst,
                             float* depth, float* conf, int B, int g, float alpha, float temperature, cudaStream_t stream);

}  // namespace ca
