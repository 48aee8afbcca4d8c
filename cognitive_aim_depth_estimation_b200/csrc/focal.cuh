// Launchers of the vector-sized focal / guidance kernels (csrc/focal.cu).
#pragma once

#include <cuda_runtime.h>

#include "heads.cuh"

namespace ca {

int rowstats_merge_launch(const float* pm, const float* ps, const float* weight, float* rmax, float* rinv, float* wtab,
                          int rows, int rows_per_image, int P, cudaStream_t stream);
int colsum_e_launch(const void* E, int lde, long long e_batch_stride, const float* wtab, float* pc, int B, int N, int P,
                    cudaStream_t stream);
int focal_finalize_launch(const float* pc, const float* cbias, float* attn, const float* rs_in, float* rs_out, int B,
                          int N, int P, float focus_strength, int mode, const float* cur_weight, float adaptive_weight,
                          cudaStream_t stream);
// Instruction sweeps (include/cogaim_b200.h, CA_SWEEP_MAX_K): K guidance rows per image in one launch (K = 1: one call).
constexpr int kSweepMaxK = 16;
int guided_softmax_launch(const float* base, long long base_k_stride, const float* mask, long long mask_k_stride,
                          long long mask_batch_stride, float* heat, int* argmax, int K, int B, int N, float alpha,
                          float temperature, cudaStream_t stream);
// w: [K, B, N], partial: [K * B, splits, D]; w2 ([B, N], optional) with K = 1 only
int weighted_pool_launch(const float* src, long long src_batch_stride, int row_offset, const float* w, const float* w2,
                         float* partial, int K, int B, int N, int D, int splits, cudaStream_t stream);
// rows of several scenes (ca_guide_many): the pool of row r reads rows[r].tokens; gather_rows copies the per-row inputs
int weighted_pool_rows_launch(const ca_guide_many_row* rows, const float* w, float* partial, int R, int N, int D,
                              int splits, cudaStream_t stream);
int gather_rows_launch(const ca_guide_many_row* rows, int R, int N, int num_cameras, float* cls, float* base,
                       float* exif, long long* camera_idx, int* call_of_row, cudaStream_t stream);
// guided_softmax -> weighted_pool (in.pool_splits splits) -> heads in one launch, bit for bit; ticket: [B] zero-initialised
// counters, left at zero by every launch.
int guide_tail_launch(const HeadsWeights& w, const HeadsInputs& in, const float* base, const float* mask,
                      long long mask_batch_stride, float* heat, int* argmax, unsigned int* ticket, float* depth,
                      float* conf, int B, int N, float alpha, float temperature, cudaStream_t stream);

}  // namespace ca
