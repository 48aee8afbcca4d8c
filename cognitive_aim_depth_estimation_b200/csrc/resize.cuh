// Launchers of the exact-Pillow bilinear resize (csrc/resize.cu).
#pragma once

#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/cogaim_b200.h"

namespace ca {

constexpr int kMaxResizeSide = CA_RESIZE_MAX_SIDE;

size_t resize_tmp_bytes(int B, int H0, int W0, int out_h, int out_w);
int resize_u8_launch(const uint8_t* src, int B, int H0, int W0, int out_h, int out_w, uint8_t* tmp, uint8_t* out,
                     cudaStream_t stream);
// B images of individual sizes (HOST arrays of device pointers and (H0, W0) pairs) -> out [B, out_h, out_w, 3];
// *launches (optional) receives the number of kernels enqueued.
size_t resize_list_tmp_bytes(const int* h_hw, int B, int out_h, int out_w);
int resize_list_launch(const uint8_t* const* h_images, const int* h_hw, int B, int out_h, int out_w, uint8_t* tmp,
                       size_t tmp_bytes, uint8_t* out, cudaStream_t stream, int* launches);

}  // namespace ca
