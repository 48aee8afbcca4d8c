// C-ABI of libcogaim_b200.so (declared in include/cogaim_b200.h).  No torch types, no exceptions.
#include "../../include/cogaim_b200.h"

#include "attention.cuh"
#include "curiosity.cuh"
#include "focal.cuh"
#include "gemm.cuh"
#include "heads.cuh"
#include "jpeg.cuh"
#include "visual.cuh"
#include "resize.cuh"
#include "rowops.cuh"
#include "host.h"

namespace ca {
const char* last_error_cstr();
}

extern "C" {

const char* ca_last_error(void) { return ca::last_error_cstr(); }

int ca_version(void) { return 1; }

int ca_device_check(int device) {
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess || count <= 0) {
    ca::set_error("no CUDA device visible: the Cognitive-Aim B200 path has no CPU fallback");
    (void)cudaGetLastError();
    return CA_STATUS_UNSUPPORTED;
  }
  if (device < 0 || device >= count) return ca::invalid("device index out of range");
  int major = 0;
  CA_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
  if (major != 10) {
    ca::set_error("device is not compute capability 10.x (sm_100a kernels only)");
    return CA_STATUS_UNSUPPORTED;
  }
  return CA_STATUS_OK;
}

int ca_gemm_bf16(const uint16_t* A, const uint16_t* W, int M, int N, int K, int lda, int ldw, int batch,
                 long long a_batch_stride, long long w_batch_stride, int epilogue, void* out, int ldo,
                 long long out_batch_stride, const float* bias, const float* ls, const float* pos,
                 int patches_per_img, float scale_log2, float* part_a, float* part_b, const float* col_max,
                 const float* col_rinv, void* stream) {
  ca::GemmArgs a;
  a.A = reinterpret_cast<const __nv_bfloat16*>(A);
  a.W = reinterpret_cast<const __nv_bfloat16*>(W);
  a.M = M;
  a.N = N;
  a.K = K;
  a.lda = lda;
  a.ldw = ldw;
  a.batch = batch;
  a.a_batch_stride = a_batch_stride;
  a.w_batch_stride = w_batch_stride;
  a.epilogue = epilogue;
  a.out = out;
  a.ldo = ldo;
  a.out_batch_stride = out_batch_stride;
  a.bias = bias;
  a.ls = ls;
  a.pos = pos;
  a.patches_per_img = patches_per_img;
  a.scale_log2 = scale_log2;
  a.part_a = part_a;
  a.part_b = part_b;
  a.col_max = col_max;
  a.col_rinv = col_rinv;
  return ca::gemm_launch(a, static_cast<cudaStream_t>(stream));
}

int ca_gemm_bf16_ln(const uint16_t* A, const uint16_t* W, int M, int N, int K, int lda, int ldw, int epilogue, void* out,
                    int ldo, const float* bias, const float* ls, float* ln_stats, int ln_slots,
                    float ln_eps, uint16_t* shadow, int ld_shadow, void* stream) {
  if (epilogue != ca::EPI_LN_BIAS_BF16 && epilogue != ca::EPI_LN_GELU_BF16 && epilogue != ca::EPI_RESID_LN_F32)
    return ca::invalid("ca_gemm_bf16_ln: epilogue must be one of CA_EPI_LN_BIAS_BF16, CA_EPI_LN_GELU_BF16, CA_EPI_RESID_LN_F32");
  ca::GemmArgs a;
  a.A = reinterpret_cast<const __nv_bfloat16*>(A);
  a.W = reinterpret_cast<const __nv_bfloat16*>(W);
  a.M = M;
  a.N = N;
  a.K = K;
  a.lda = lda;
  a.ldw = ldw;
  a.batch = 1;
  a.a_batch_stride = 0;
  a.w_batch_stride = 0;
  a.epilogue = epilogue;
  a.out = out;
  a.ldo = ldo;
  a.out_batch_stride = 0;
  a.bias = bias;
  a.ls = ls;
  a.pos = nullptr;
  a.patches_per_img = 0;
  a.scale_log2 = 0.f;
  a.part_a = a.part_b = nullptr;
  a.col_max = a.col_rinv = nullptr;
  a.ln_stats = ln_stats;
  a.ln_slots = ln_slots;
  a.ln_eps = ln_eps;
  a.shadow = reinterpret_cast<__nv_bfloat16*>(shadow);
  a.ld_shadow = ld_shadow;
  return ca::gemm_launch(a, static_cast<cudaStream_t>(stream));
}

int ca_ln_shadow(const float* x, uint16_t* shadow, int ld_shadow, float* stats, int rows, int D, void* stream) {
  return ca::ln_shadow_launch(x, reinterpret_cast<__nv_bfloat16*>(shadow), ld_shadow, stats, rows, D,
                              static_cast<cudaStream_t>(stream));
}

int ca_attention_bf16(const uint16_t* qkv, uint16_t* out, int B, int T, int H, void* stream) {
  return ca::attention_launch(reinterpret_cast<const __nv_bfloat16*>(qkv), reinterpret_cast<__nv_bfloat16*>(out), B, T,
                              H, static_cast<cudaStream_t>(stream));
}

int ca_attention_bf16_ld(const uint16_t* qkv, uint16_t* out, int ldo, int B, int T, int H, void* stream) {
  return ca::attention_launch(reinterpret_cast<const __nv_bfloat16*>(qkv), reinterpret_cast<__nv_bfloat16*>(out), B, T,
                              H, static_cast<cudaStream_t>(stream), ldo);
}

int ca_patchify_f32(const float* images, uint16_t* patches, int B, int S, void* stream) {
  return ca::patchify_f32_launch(images, reinterpret_cast<__nv_bfloat16*>(patches), B, S,
                                 static_cast<cudaStream_t>(stream));
}

int ca_preprocess_u8(const uint8_t* images, uint16_t* patches, int B, int S, const float* h_mean3,
                     const float* h_std3, void* stream) {
  return ca::preprocess_u8_launch(images, reinterpret_cast<__nv_bfloat16*>(patches), B, S, h_mean3, h_std3,
                                  static_cast<cudaStream_t>(stream));
}

int ca_cls_rows(float* x, const float* cls, const float* pos, int B, int T, int D, void* stream) {
  return ca::cls_rows_launch(x, cls, pos, B, T, D, static_cast<cudaStream_t>(stream));
}

int ca_layernorm(const float* x, const float* gamma, const float* beta, void* out, int out_is_bf16, int rows, int D,
                 float eps, void* stream) {
  return ca::layernorm_launch(x, gamma, beta, out, out_is_bf16, rows, D, eps, static_cast<cudaStream_t>(stream));
}

int ca_layernorm_ld(const float* x, const float* gamma, const float* beta, void* out, int out_is_bf16, int ld_out,
                    int rows, int D, float eps, void* stream) {
  return ca::layernorm_launch(x, gamma, beta, out, out_is_bf16, rows, D, eps, static_cast<cudaStream_t>(stream), ld_out);
}

int ca_focal_input(const float* tokens, const float* pe, const float* rowscale, uint16_t* xin, int B, int N, int D,
                   void* stream) {
  return ca::focal_input_launch(tokens, pe, rowscale, reinterpret_cast<__nv_bfloat16*>(xin), B, N, D,
                                static_cast<cudaStream_t>(stream));
}

int ca_fetch_pinned_f32(float* dst, const float* h_src_pinned, size_t n, void* stream) {
  return ca::fetch_pinned_launch(dst, h_src_pinned, n, static_cast<cudaStream_t>(stream));
}

int ca_rowstats_merge(const float* pm, const float* ps, const float* weight, float* rmax, float* rinv, float* wtab,
                      int rows, int rows_per_image, int P, void* stream) {
  return ca::rowstats_merge_launch(pm, ps, weight, rmax, rinv, wtab, rows, rows_per_image, P,
                                   static_cast<cudaStream_t>(stream));
}

int ca_colsum_e(const uint16_t* E, int lde, long long e_batch_stride, const float* wtab, float* pc, int B, int N, int P,
                void* stream) {
  return ca::colsum_e_launch(E, lde, e_batch_stride, wtab, pc, B, N, P, static_cast<cudaStream_t>(stream));
}

int ca_focal_finalize(const float* pc, const float* cbias, float* attn, const float* rs_in, float* rs_out, int B, int N,
                      int P, float focus_strength, int mode, const float* cur_weight, float adaptive_weight,
                      void* stream) {
  return ca::focal_finalize_launch(pc, cbias, attn, rs_in, rs_out, B, N, P, focus_strength, mode, cur_weight,
                                   adaptive_weight, static_cast<cudaStream_t>(stream));
}

int ca_guided_softmax(const float* base, const float* mask, long long mask_batch_stride, float* heat, int32_t* argmax,
                      int B, int N, float alpha, float temperature, void* stream) {
  return ca::guided_softmax_launch(base, mask, mask_batch_stride, heat, argmax, B, N, alpha, temperature,
                                   static_cast<cudaStream_t>(stream));
}

int ca_weighted_pool(const float* src, long long src_batch_stride, int row_offset, const float* w, const float* w2,
                     float* partial, int B, int N, int D, int splits, void* stream) {
  return ca::weighted_pool_launch(src, src_batch_stride, row_offset, w, w2, partial, B, N, D, splits,
                                  static_cast<cudaStream_t>(stream));
}

int ca_guided_softmax_sweep(const float* base, long long base_k_stride, const float* mask, long long mask_k_stride,
                            long long mask_batch_stride, float* heat, int32_t* argmax, int K, int B, int N, float alpha,
                            float temperature, void* stream) {
  return ca::guided_softmax_sweep_launch(base, base_k_stride, mask, mask_k_stride, mask_batch_stride, heat, argmax, K, B, N,
                                         alpha, temperature, static_cast<cudaStream_t>(stream));
}

int ca_weighted_pool_sweep(const float* src, long long src_batch_stride, int row_offset, const float* w, float* partial,
                           int K, int B, int N, int D, int splits, void* stream) {
  return ca::weighted_pool_sweep_launch(src, src_batch_stride, row_offset, w, partial, K, B, N, D, splits,
                                        static_cast<cudaStream_t>(stream));
}

int ca_heads(const ca_heads_weights* w, const ca_heads_inputs* in, float* depth, float* conf, float* fused_out, int B,
             void* stream) {
  if (!w || !in) return ca::invalid("heads: null argument struct");
  return ca::heads_launch(*w, *in, depth, conf, fused_out, B, static_cast<cudaStream_t>(stream));
}

int ca_guide_tail(const ca_heads_weights* w, const ca_heads_inputs* in, const float* base, const float* mask,
                  long long mask_batch_stride, float* heat, int32_t* argmax, uint32_t* ticket, float* depth, float* conf,
                  int B, int N, float alpha, float temperature, void* stream) {
  if (!w || !in) return ca::invalid("guide_tail: null argument struct");
  return ca::guide_tail_launch(*w, *in, base, mask, mask_batch_stride, heat, argmax, ticket, depth, conf, B, N, alpha,
                               temperature, static_cast<cudaStream_t>(stream));
}

int ca_focal_value(const ca_focal_value_args* a, int B, void* stream) {
  if (!a) return ca::invalid("focal_value: null argument struct");
  return ca::focal_value_launch(*a, B, static_cast<cudaStream_t>(stream));
}

int ca_focal_fusion(const float* feats, int n_iters, const float* w0, const float* b0, const float* w1, const float* b1,
                    float* out, int B, void* stream) {
  return ca::focal_fusion_launch(feats, n_iters, w0, b0, w1, b1, out, B, static_cast<cudaStream_t>(stream));
}

int ca_curiosity(const ca_curiosity_weights* w, const float* tokens, int tokens_per_img, const float* eps,
                 const float* noise, float* reward_raw, float* reward, float* history, int history_len,
                 long long* history_pointer, int B, void* stream) {
  if (!w) return ca::invalid("curiosity: null weight struct");
  return ca::curiosity_launch(*w, tokens, tokens_per_img, eps, noise, reward_raw, reward, history, history_len,
                              history_pointer, B, static_cast<cudaStream_t>(stream));
}

int ca_curiosity_modulation(const ca_curiosity_mod_weights* w, const float* reward, float lo, float hi, float* cur_weight,
                            int B, int n_iters, int mod_hidden, void* stream) {
  if (!w) return ca::invalid("curiosity_modulation: null weight struct");
  return ca::curiosity_modulation_launch(*w, reward, lo, hi, cur_weight, B, n_iters, mod_hidden,
                                         static_cast<cudaStream_t>(stream));
}

int ca_resize_u8(const uint8_t* src, int B, int H0, int W0, int out_h, int out_w, uint8_t* tmp, uint8_t* out,
                 void* stream) {
  return ca::resize_u8_launch(src, B, H0, W0, out_h, out_w, tmp, out, static_cast<cudaStream_t>(stream));
}

size_t ca_resize_u8_list_tmp_bytes(const int* h_hw, int B, int out_h, int out_w) {
  return ca::resize_list_tmp_bytes(h_hw, B, out_h, out_w);
}

int ca_resize_u8_list(const uint8_t* const* h_images, const int* h_hw, int B, int out_h, int out_w, uint8_t* tmp,
                      size_t tmp_bytes, uint8_t* out, void* stream) {
  return ca::resize_list_launch(h_images, h_hw, B, out_h, out_w, tmp, tmp_bytes, out, static_cast<cudaStream_t>(stream),
                                nullptr);
}

int ca_jpeg_info(const uint8_t* h_data, size_t len, int* width, int* height) {
  return ca::jpeg_info(h_data, len, width, height, nullptr);
}

int ca_jpeg_decode(const uint8_t* h_data, size_t len, uint8_t* out_rgb, int width, int height, void* stream) {
  return ca::jpeg_decode(h_data, len, out_rgb, width, height, static_cast<cudaStream_t>(stream));
}

int ca_jpeg_decode_batch(const uint8_t* const* h_data, const size_t* lens, int n, uint8_t* const* outs, const int* widths,
                         const int* heights, void* stream) {
  return ca::jpeg_decode_batch(h_data, lens, n, outs, widths, heights, static_cast<cudaStream_t>(stream));
}

int ca_focus_map(const float* heat, int B, int g, int out_h, int out_w, float* norm, float* out, void* stream) {
  return ca::focus_map_launch(heat, B, g, out_h, out_w, norm, out, static_cast<cudaStream_t>(stream));
}

}  // extern "C"
