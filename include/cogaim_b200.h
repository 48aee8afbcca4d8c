/* cogaim_b200.h — C-ABI of the B200-native Cognitive-Aim forward path.
 *
 * The reference (yenjane-dot/cognitive-aim-depth-estimation) has no FFI: its boundary is the Python
 * nn.Module surface of `CognitiveAimModel` (reference src/model.py:1064 `forward`, :1157
 * `forward_with_guidance`, :1534 `create_model`).  The Python host module in
 * `cognitive_aim_depth_estimation_b200/model.py` mirrors that surface and calls the entry points below through
 * ctypes.  Every entry point cites the reference call site whose arithmetic it replaces.
 *
 * Conventions
 *   - plain pointers and sizes only; all data pointers are DEVICE pointers unless named `h_*`;
 *   - every function returns 0 on success, non-zero (ca_status) on failure and never throws;
 *     `ca_last_error()` returns a thread-local description of the last failure;
 *   - the caller supplies the CUDA stream (as a `void*` holding a `cudaStream_t`), all outputs and
 *     all workspaces; nothing is allocated behind the caller's back on the hot path;
 *   - bf16 buffers are raw 16-bit storage (`uint16_t`), row-major.
 *   - there is NO CPU fallback: without an sm_100 device every compute entry point fails.
 */
#ifndef COGAIM_B200_H_
#define COGAIM_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum ca_status {
  CA_STATUS_OK = 0,
  CA_STATUS_INVALID = 1,    /* bad shape / alignment / null pointer */
  CA_STATUS_CUDA = 2,       /* CUDA runtime or driver failure */
  CA_STATUS_UNSUPPORTED = 3 /* no sm_100 device */
} ca_status;

/* GEMM epilogues (see ca_gemm_bf16). */
typedef enum ca_epilogue {
  CA_EPI_BIAS_BF16 = 0, /* out_bf16 = acc + bias                      HF modeling_dinov2.py:199-201 (q/k/v Linear); src/model.py:192-193 */
  CA_EPI_GELU_BF16 = 1, /* out_bf16 = gelu_erf(acc + bias)            HF modeling_dinov2.py:324-326 (fc1 + GELU) */
  CA_EPI_RESID_F32 = 2, /* x_f32 += ls * (acc + bias), in place       HF modeling_dinov2.py:246,278,376-385 (dense + LayerScale + residual) */
  CA_EPI_PATCH_F32 = 3, /* x_f32[b*T+1+p] = acc + bias + pos[1+p]     HF modeling_dinov2.py:148,112 (patch conv + pos-embed) */
  CA_EPI_ROWSTATS = 4,  /* softmax row statistics of acc*scale        src/model.py:197-200 (pass A); with `out` != NULL also keeps
                           exp2(acc*scale - span max) as fp16 [batch, M, ldo] for ca_colsum_e */
  CA_EPI_COLSUM = 5,    /* column sums of softmax(acc*scale)          src/model.py:234 (pass B, transposed) */
  CA_EPI_F32 = 6,       /* out_f32 = acc (test hook) */
  /* LayerNorm (HF modeling_dinov2.py:354,359: norm1 / norm2) folded into the GEMMs either side of it — see ca_gemm_bf16_ln */
  CA_EPI_LN_BIAS_BF16 = 7, /* out_bf16 = rstd * acc + bias, W row-centred                (norm1 -> q/k/v Linear) */
  CA_EPI_LN_GELU_BF16 = 8, /* out_bf16 = gelu_erf(the same)                              (norm2 -> fc1 -> GELU) */
  CA_EPI_RESID_LN_F32 = 9  /* x_f32 += ls * (acc + bias); shadow_bf16 = bf16(x); row statistics of the new x */
} ca_epilogue;

/* Library / device introspection -------------------------------------------------------------- */
const char* ca_last_error(void);
int ca_version(void);                       /* ABI version, currently 1 */
int ca_device_check(int device);            /* CA_STATUS_OK iff `device` is compute capability 10.x */

/* Dense contraction on tcgen05 tensor cores --------------------------------------------------- */
/* C[b] = epilogue(A[b] (M x K, lda) * W[b] (N x K, ldw)^T), bf16 operands, fp32 TMEM accumulators.
 * w_batch_stride == 0 shares W across the batch.  Unused epilogue operands may be NULL.
 * For CA_EPI_ROWSTATS/COLSUM the per-row partial buffers have P = 4*ceil(N/256) entries per row (one per 64-column
 * span of the 256-wide tiles; spans past N hold max = -inf, sum = 0) and are SPAN-MAJOR: [batch, P, M]. */
int ca_gemm_bf16(const uint16_t* A, const uint16_t* W, int M, int N, int K, int lda, int ldw, int batch,
                 long long a_batch_stride, long long w_batch_stride, int epilogue, void* out, int ldo,
                 long long out_batch_stride, const float* bias, const float* ls, const float* pos,
                 int patches_per_img, float scale_log2, float* part_a, float* part_b, const float* col_max,
                 const float* col_rinv, void* stream);

/* The same contraction with the LayerNorm of HF modeling_dinov2.py:354 / :359 folded in (no LayerNorm pass over HBM):
 *   LN(x) W^T + b  =  rstd * (x W'^T) + b',   b' = b + W beta,   W' = W diag(gamma) with every row centred,
 *   W'[n,:] -= mean_k W'[n,k]   (then x W'^T = (x - mean(x)) W'^T: the row mean never has to be subtracted).
 * CA_EPI_RESID_LN_F32 (dense + LayerScale + residual, :246,278,376-385) updates x in place and leaves, for the LayerNorm
 * that follows, `shadow` = the new rows as bf16 [M, N] (pitch ld_shadow) and ln_stats[M, ln_slots, 2] = (sum, sum of
 * squared deviations from the span mean) of each 128-column span of the new row; N == 128 * ln_slots.
 * CA_EPI_LN_BIAS_BF16 / CA_EPI_LN_GELU_BF16 take A = that shadow (K == 128 * ln_slots), W = W' (bf16), bias = b' and
 * ln_stats, and apply the row's 1/sqrt(var + ln_eps) in the epilogue.  ca_ln_shadow produces shadow + ln_stats from fp32 rows (the entry of the chain, after the embeddings). */
int ca_gemm_bf16_ln(const uint16_t* A, const uint16_t* W, int M, int N, int K, int lda, int ldw, int epilogue, void* out,
                    int ldo, const float* bias, const float* ls, float* ln_stats, int ln_slots,
                    float ln_eps, uint16_t* shadow, int ld_shadow, void* stream);
int ca_ln_shadow(const float* x, uint16_t* shadow, int ld_shadow, float* stats, int rows, int D, void* stream);

/* Backbone attention --------------------------------------------------------------------------- */
/* out[B*T, H*64] = softmax(Q K^T / 8) V per (image, head); qkv is the fused [B*T, 3*H*64] activation
 * (Q | K | V column blocks).  Replaces F.scaled_dot_product_attention at HF modeling_dinov2.py:215-229. */
int ca_attention_bf16(const uint16_t* qkv, uint16_t* out, int B, int T, int H, void* stream);
/* the same with an output row pitch of `ldo` elements (>= H*64): the output feeds a GEMM whose K dimension is extended by
 * the LoRA columns stored behind each row (see ca_gemm_bf16 with K > 768 in model.py, `lora_mode: fused`). */
int ca_attention_bf16_ld(const uint16_t* qkv, uint16_t* out, int ldo, int B, int T, int H, void* stream);

/* Bandwidth-bound row kernels ------------------------------------------------------------------- */
/* fp32 CHW images [B,3,S,S] (the tensor `forward` receives) -> bf16 patch rows [B*(S/14)^2, 592]
 * (column k = c*196 + ky*14 + kx, columns 588..591 zero).  HF modeling_dinov2.py:139-148 (im2col of the conv). */
int ca_patchify_f32(const float* images, uint16_t* patches, int B, int S, void* stream);
/* uint8 HWC images [B,S,S,3] -> /255 -> (x-mean)/std -> bf16 patch rows.  demo.py:162-166 (ToTensor + Normalize;
 * the source is already S x S so Resize is the identity).  h_mean3 / h_std3 are HOST pointers to 3 floats. */
int ca_preprocess_u8(const uint8_t* images, uint16_t* patches, int B, int S, const float* h_mean3,
                     const float* h_std3, void* stream);
/* x[b, 0, :] = cls + pos[0]  (HF modeling_dinov2.py:108-112). x is the fp32 residual stream [B, T, D]. */
int ca_cls_rows(float* x, const float* cls, const float* pos, int B, int T, int D, void* stream);
/* LayerNorm(D=768) of fp32 rows -> bf16 (out_is_bf16=1) or fp32.  HF modeling_dinov2.py:354,359,449. */
int ca_layernorm(const float* x, const float* gamma, const float* beta, void* out, int out_is_bf16, int rows, int D,
                 float eps, void* stream);
/* the same with an output row pitch of `ld_out` elements (>= D). */
int ca_layernorm_ld(const float* x, const float* gamma, const float* beta, void* out, int out_is_bf16, int ld_out,
                    int rows, int D, float eps, void* stream);
/* xin[b,n,:] = bf16(tokens[b,1+n,:] * rowscale[b,n] + pe[n,:]); rowscale may be NULL (=1).
 * reference src/model.py:184 (PE add) and :426 (re-focus, folded into a per-row scale). */
int ca_focal_input(const float* tokens, const float* pe, const float* rowscale, uint16_t* xin, int B, int N, int D,
                   void* stream);

/* dst[0..n) (device) = h_src_pinned[0..n) (PAGE-LOCKED host memory), read by the SMs over PCIe instead of by the copy
 * engine: the per-call inputs of src/model.py:609, :744, :1421 (Gaussian draws, fresh projection; a few hundred KB) must
 * not queue on the H2D copy engine behind the application's bulk image upload.  Fails for pageable memory. */
int ca_fetch_pinned_f32(float* dst, const float* h_src_pinned, size_t n, void* stream);

/* Focal / guidance vector stages (fp32) ---------------------------------------------------------- */
/* Merge the per-64-column partials of CA_EPI_ROWSTATS (pm, ps: span-major [batch, P, rows_per_image]; rows = batch *
 * rows_per_image): rmax[r] = max, rinv[r] = (weight ? weight[r] : 1) / sumexp, wtab[b, s, i] = exp2(pm[b, s, i] - rmax) * rinv
 * (span-major like pm); any of the three outputs may be null (not all).
 * reference src/model.py:200 (row softmax statistics). */
int ca_rowstats_merge(const float* pm, const float* ps, const float* weight, float* rmax, float* rinv, float* wtab,
                      int rows, int rows_per_image, int P, void* stream);
/* Column sums of the (weighted) row softmax from the span-relative exponentials E (fp16 [B, N, lde], written by
 * ca_gemm_bf16 with CA_EPI_ROWSTATS when `out` is given): pc[b, p, j] = sum_{i in row span p} E[b,i,j] * wtab[b,j/64,i]
 * (span-major [B, P, N]: every CTA writes one contiguous row).
 * Replaces the second Q K^T pass (CA_EPI_COLSUM) by one bandwidth-bound read of E.  src/model.py:234 (col mean), :308. */
int ca_colsum_e(const uint16_t* E, int lde, long long e_batch_stride, const float* wtab, float* pc, int B, int N, int P,
                void* stream);
/* pc: the span-major [B, P, N] partials of ca_colsum_e.
 * mode 0: FocalStream attention: mean over rows + centre bias, L1 normalise, clamp 1e-8,
 *         renormalise; optionally rs_out = rs_in * (1 + focus_strength * attn)   (src/model.py:234-282, :426).
 * mode 1: attn = plain sum of the partials (weighted column sums of the un-guided value path). */
/*         cur_weight (optional, [B]) with adaptive_weight: the curiosity modulation of src/model.py:264-276,
 *         p <- aw * p * (1 + cur_weight[b]) + (1 - aw) * p between the L1 normalisation and the clamp. */
int ca_focal_finalize(const float* pc, const float* cbias, float* attn, const float* rs_in, float* rs_out, int B, int N,
                      int P, float focus_strength, int mode, const float* cur_weight, float adaptive_weight,
                      void* stream);
/* heat = softmax((alpha*mask + (1-alpha)*base)/temperature) per image; argmax = first index of the maximum.
 * src/model.py:1404-1409.  mask_batch_stride = 0: one mask [N] for the whole batch (the reference broadcasts one
 * instruction per call, :1401); = N (or more): one mask per image, i.e. per-sample instructions in one batch
 * (what demo.py:406-432 `predict_batch` does with a Python loop over single-image calls). */
int ca_guided_softmax(const float* base, const float* mask, long long mask_batch_stride, float* heat, int32_t* argmax,
                      int B, int N, float alpha, float temperature, void* stream);
/* partial[b, s, :] = sum_{n in split s} w[b,n] * (w2 ? w2[b,n] : 1) * src[b*src_batch_stride + (row_offset+n)*D + :]
 * (src/model.py:1412-1414 guided pooling; :308 weighted features).  D must be 768. */
int ca_weighted_pool(const float* src, long long src_batch_stride, int row_offset, const float* w, const float* w2,
                     float* partial, int B, int N, int D, int splits, void* stream);

/* Instruction sweeps: K guidance instructions over the same batch (K successive forward_with_guidance calls that share
 * the backbone and the focal pass).  Rows r = k * B + b, k-major.  K is at most CA_SWEEP_MAX_K: the sweep pool keeps one
 * float4 accumulator per instruction in registers. */
#define CA_SWEEP_MAX_K 16
/* ca_guided_softmax for K * B rows: row r = k * B + b reads mask + k * mask_k_stride + b * mask_batch_stride and base +
 * k * base_k_stride + b * N (base_k_stride 0: one focal pass shared by every instruction; B * N: one per instruction,
 * curiosity-guided attention), writes heat [K * B, N] and argmax [K * B].  Each row is computed exactly as
 * ca_guided_softmax computes it. */
int ca_guided_softmax_sweep(const float* base, long long base_k_stride, const float* mask, long long mask_k_stride,
                            long long mask_batch_stride, float* heat, int32_t* argmax, int K, int B, int N, float alpha,
                            float temperature, void* stream);
/* partial[k * B + b, s, :] = sum_{n in split s} w[k, b, n] * src[b*src_batch_stride + (row_offset+n)*D + :] for K weight
 * vectors w [K, B, N]: the tokens are read once for all K.  Bit for bit what K ca_weighted_pool launches (w2 = NULL) with
 * the same `splits` write.  D must be 768. */
int ca_weighted_pool_sweep(const float* src, long long src_batch_stride, int row_offset, const float* w, float* partial,
                           int K, int B, int N, int D, int splits, void* stream);

/* Rows of several scenes: m guide calls answered together (ca_guide_many, CognitiveAimModel.guide_many).  Row r of the
 * batch is one image of one call's scene, r in call order; the row table holds, per row, DEVICE pointers into the scene
 * that owns the image.  Nothing of a scene is copied but the few values below. */
#define CA_GUIDE_MANY_MAX_CALLS 64 /* guide calls per ca_guide_many */
#define CA_GUIDE_MANY_MAX_ROWS 256 /* rows (the images of all calls) per ca_guide_many */
typedef struct ca_guide_many_row {
  const float* tokens;          /* the image's tokens [1 + N, 768] fp32 (row 0: CLS), 16-byte aligned */
  const float* base;            /* its focal attention [N] */
  const float* exif;            /* its EXIF [3] */
  const long long* camera_idx;  /* its camera index */
  int* fault;                   /* the fault word a bad camera index of this image is reported in (bit 0), or NULL */
  long long call;               /* j: the guide call the row belongs to */
} ca_guide_many_row;
/* One launch: cls[r, :] = rows[r].tokens[0, :] ([R, 768]), base[r, :] = rows[r].base ([R, N]), exif[r, :] ([R, 3]),
 * camera_idx[r] ([R] int64) and call_of_row[r] = rows[r].call ([R] int32).  A camera index outside [0, num_cameras)
 * sets bit 0 of rows[r].fault (the heads clamp it).  `rows` is a DEVICE array of R entries. */
int ca_gather_rows(const ca_guide_many_row* rows, int R, int N, int num_cameras, float* cls, float* base, float* exif,
                   long long* camera_idx, int32_t* call_of_row, void* stream);
/* ca_weighted_pool with the tokens of row r read through the row table: partial[r, s, :] = sum_{n in split s} w[r, n] *
 * rows[r].tokens[(1 + n) * 768 + :].  Partial r is bit for bit what ca_weighted_pool writes for that image alone with
 * the same `splits`.  `rows`: DEVICE [R]; w: [R, N]; D must be 768. */
int ca_weighted_pool_rows(const ca_guide_many_row* rows, const float* w, float* partial, int R, int N, int D, int splits,
                          void* stream);

/* Heads ------------------------------------------------------------------------------------------ */
/* All members are DEVICE pointers to fp32 row-major [out, in] weights / [out] biases of the reference modules. */
typedef struct ca_heads_weights {
  const float *amb_w0, *amb_b0, *amb_w1, *amb_b1, *amb_w2, *amb_b2; /* ambient_stream.mlp.{0,3,5}   src/model.py:37-44 */
  const float* cam_emb;                                             /* exif_prior.camera_embedding [num_cameras, 64] */
  const float *exif_w0, *exif_b0, *exif_w1, *exif_b1;               /* exif_prior.exif_encoder.{0,2} */
  const float *exif_f0, *exif_fb0, *exif_f1, *exif_fb1;             /* exif_prior.fusion.{0,3} */
  const float *fus_w, *fus_b;                                       /* fusion.0 [192,192] */
  const float *dec_w, *dec_b;                                       /* decision_head.0 [1,192] */
  const float *conf_w0, *conf_b0, *conf_w2, *conf_b2;               /* confidence_head.{0,2} */
} ca_heads_weights;

typedef struct ca_heads_inputs {
  const float* tokens;        /* [B, tokens_per_img, 768] fp32 backbone output; row 0 of each image is CLS */
  int tokens_per_img;
  const float* focal_feat;    /* [B, 64] un-guided focal features, or NULL for the guided path */
  const float* pool_partial;  /* guided: [B, pool_splits, 768] partial weighted sums of the patch tokens */
  int pool_splits;
  const float* tmp_w;         /* guided: per-call projection [64, 768]  (src/model.py:1421) */
  const float* tmp_b;         /* [64] */
  float* pooled_out;          /* optional [B, 768] (debug / tests) */
  const float* exif;          /* [B, 3] raw focal_length, aperture, iso — or NULL (zero EXIF slot) */
  const long long* camera_idx;/* [B] */
  int num_cameras;            /* rows of cam_emb; an index outside [0, num_cameras) is clamped and reported in *fault */
  int* fault;                 /* optional device-visible word (e.g. pinned host memory): bit 0 set on a bad camera_idx */
  int sweep_images;           /* 0: one CTA per image.  > 0 (instruction sweep, guided only): the B passed to ca_heads is
                                 K * sweep_images; CTA r reads image b = r % sweep_images (CLS token, EXIF, camera index),
                                 projection k = r / sweep_images of tmp_w [K, 64, 768] / tmp_b [K, 64], pool_partial row r,
                                 and writes depth[r], conf[r] */
  const int32_t* call_of_row; /* guided only, with sweep_images 0: [B] device; row r uses projection call_of_row[r] of
                                 tmp_w [m, 64, 768] / tmp_b [m, 64] (rows of several guide calls, ca_guide_many).  NULL:
                                 the projection follows sweep_images as above */
} ca_heads_inputs;

/* depth[B], conf[B] (and optionally fused_out[B,192]) from the backbone tokens + focal slot + EXIF.
 * `w` and `in` are HOST pointers to the structs above.  src/model.py:1195-1230. */
int ca_heads(const ca_heads_weights* w, const ca_heads_inputs* in, float* depth, float* conf, float* fused_out, int B,
             void* stream);
/* The guided tail of one call in ONE launch: ca_guided_softmax(base, mask) -> ca_weighted_pool(tokens, heat,
 * in->pool_splits splits) -> ca_heads(in), with results bit-identical to that chain.  Grid (in->pool_splits, B); every CTA
 * recomputes its image's softmax, pools its split into in->pool_partial (a [B, pool_splits, 768] scratch this call
 * overwrites) and the image's last CTA runs the heads.  in->focal_feat must be NULL and in->sweep_images 0;
 * in->tokens_per_img must be N + 1.  ticket: [B] device counters, zero before the first launch; every launch leaves them
 * at zero (no clearing between launches).  argmax may be NULL.  N <= 8192. */
/* Largest batch for which a single guided call (K = 1: forward_with_guidance, guide and sweeps of one instruction;
 * ca_forward_guided, ca_guide and their sweeps) uses ca_guide_tail; larger batches and sweeps of K > 1 run the
 * three-kernel chain.  A single image is launch-bound, and one launch replaces three.  A batch is bandwidth-bound: a
 * ca_guide_tail CTA of 1024 threads fills an SM's register file, and only 6 of its warps stream tokens, while several
 * 192-thread pool CTAs of the chain share an SM.  tools/bench_scene.py times both at B = 1 and B = 32. */
#define CA_GUIDE_TAIL_MAX_B 1
int ca_guide_tail(const ca_heads_weights* w, const ca_heads_inputs* in, const float* base, const float* mask,
                  long long mask_batch_stride, float* heat, int32_t* argmax, uint32_t* ticket, float* depth, float* conf,
                  int B, int N, float alpha, float temperature, void* stream);

/* Depth fields (CognitiveAimModel.depth_field): the guided call with the focus on every cell of the g x g grid.
 * P[b, n, :] = src[b * src_batch_stride + (row_offset + n) * 768 + :] . tmp_w^T for n < N: [B, N, 64] fp32, the per-call
 * projection tmp_w [64, 768] applied to every patch token once.  src, tmp_w and P 16-byte aligned. */
int ca_token_project(const float* src, long long src_batch_stride, int row_offset, const float* tmp_w, float* P, int B,
                     int N, void* stream);
/* depth[b, c], conf[b, c] for every cell c = y * g + x of the g x g grid: the guided call (ca_guided_softmax ->
 * ca_weighted_pool -> ca_heads) whose mask is 5 on the disk dy^2 + dx^2 <= r^2 around (y, x), 2 out to 2r and 1 elsewhere,
 * r = max(1, g / 6).  base [B, g * g] is the focal attention, a probability vector per image (0 <= base <= 1): then the
 * disk's logits exceed all others by (4 alpha - 1) / temperature = 36 at the reference's 0.7 / 0.05, and the softmax is
 * taken over the disk alone (the rest weighs < N e^-36).  Other alpha / temperature are refused when that gap is below 36.
 * P [B, g * g, 64] from ca_token_project; tmp_b [64] the projection bias (in->tmp_b).  `in` supplies tokens (the CLS rows,
 * tokens_per_img), tmp_b, exif, camera_idx, num_cameras and fault as for ca_heads; its other members are not read.
 * cst: [B, 192] scratch (the fusion layer's per-image part).  Two launches; no atomics in any reduction. */
int ca_depth_field_cells(const ca_heads_weights* w, const ca_heads_inputs* in, const float* base, const float* P,
                         float* cst, float* depth, float* conf, int B, int g, float alpha, float temperature,
                         void* stream);

typedef struct ca_focal_value_args {
  const float* tok_partial;  /* [B, splits, 768] partial sums of c_j * rowscale_j * tokens_j */
  const float* pe_partial;   /* [B, splits, 768] partial sums of c_j * PE_j */
  int splits;
  const float *wv, *bv;              /* value_proj [768,768], [768] */
  const float *proj_w0, *proj_b0;    /* projection.0 [256,768] */
  const float *proj_w1, *proj_b1;    /* projection.3 [64,256] */
  float* feat_out;                   /* [B, n_iters, 64] */
  int iter, n_iters;
} ca_focal_value_args;

/* Un-guided focal features of one iteration: ((sum_j c_j x~_j) Wv^T + bv) -> projection (src/model.py:204,308-311). */
int ca_focal_value(const ca_focal_value_args* a, int B, void* stream);
/* fused[B,64] = IterativeFocalStream.fusion(cat(feats))  (src/model.py:430); feats is [B, n_iters, 64]. */
int ca_focal_fusion(const float* feats, int n_iters, const float* w0, const float* b0, const float* w1, const float* b1,
                    float* out, int B, void* stream);

/* Curiosity module -------------------------------------------------------------------------------- */
/* DEVICE pointers to the fp32 weights of reference `CuriosityModule` (src/model.py:524-583). */
typedef struct ca_curiosity_weights {
  const float *em_w0, *em_b0, *em_w1, *em_b1;     /* encoder_mean.{0,3}      [384,768] [192,384] */
  const float *el_w0, *el_b0, *el_w1, *el_b1;     /* encoder_logvar.{0,3}    [384,768] [192,384] */
  const float *dec_w0, *dec_b0, *dec_w1, *dec_b1; /* decoder.{0,3}           [384,192] [192,384] */
  const float *unc_w0, *unc_b0, *unc_w1, *unc_b1; /* uncertainty_head.{0,2}  [192,768] [1,192] */
  const float *loc_w0, *loc_b0, *loc_w1, *loc_b1; /* local_curiosity.{0,2}   [128,768] [1,128]; NULL = not hierarchical */
  const float* cur_w;                             /* curiosity_weights [3] (geometric, local, variational) */
} ca_curiosity_weights;

/* CuriosityModule.forward(cls, exif_data=None) (src/model.py:586-688 with :690-700, :731-758): reward_raw[B] (before the
 * final clamp; what the ring buffer records), reward[B] = clamp(reward_raw, 0, 100) (what callers get), and the
 * sequential ring-buffer update history[ptr] = reward_raw[b]; ptr = (ptr + 1) % history_len for b = 0..B-1
 * (src/model.py:760-773) on `history` / `history_pointer` (device int64) when `history` is not NULL.
 * tokens: fp32 [B, tokens_per_img, 768], row 0 of each image is the CLS token.  eps [B,192] and noise [B,768] are the
 * two standard-normal draws of :609 and :744, made by the caller (the reference takes them from the global generator).
 * `w` is a HOST pointer. */
int ca_curiosity(const ca_curiosity_weights* w, const float* tokens, int tokens_per_img, const float* eps,
                 const float* noise, float* reward_raw, float* reward, float* history, int history_len,
                 long long* history_pointer, int B, void* stream);

/* DEVICE pointers to the curiosity-guided attention weights (only built when `curiosity_guided_attention.enabled`). */
typedef struct ca_curiosity_mod_weights {
  const float *amp_w0, *amp_b0, *amp_w1, *amp_b1; /* focal_stream.curiosity_amplifier.{0,2}  [32,1] [n_iters,32]  src/model.py:333-339 */
  const float* mod_w0[8];                         /* focal_streams.{i}.curiosity_modulator.0 [32,1]   src/model.py:73-79 */
  const float* mod_b0[8];
  const float* mod_w1[8];                         /* focal_streams.{i}.curiosity_modulator.2 [8,32] */
  const float* mod_b1[8];
} ca_curiosity_mod_weights;

/* cur_weight[i, b] = mean_h sigmoid(modulator_i(score_b * softmax(amplifier(score_b))[i]))  for i < n_iters <= 8, where
 * score_b = clamp(reward[b], lo, hi)  (src/model.py:406-417, 266-269; the un-guided attention calls clamp the score to
 * [0.5, 1], :1107, :1141; pass lo > hi for no clamp).  mod_hidden = focal_hidden_dim / 8 (<= 64), 8 modulator outputs.
 * `w` is a HOST pointer. */
int ca_curiosity_modulation(const ca_curiosity_mod_weights* w, const float* reward, float lo, float hi, float* cur_weight,
                            int B, int n_iters, int mod_hidden, void* stream);

/* ---- demo.py:162-163 `Resize((S, S))` on a PIL image = Pillow's antialiased bilinear resample, bit-exact ----------
 * src: uint8 [B, H0, W0, 3] (device), out: uint8 [B, out_h, out_w, 3].  tmp: uint8 [B, H0, out_w, 3] scratch, needed
 * only when both axes change.  The fixed-point coefficient tables are built on the host as Pillow's Resample.c builds
 * them and cached per (device, source size, target size) — the first call for a new size allocates and synchronises. */
int ca_resize_u8(const uint8_t* src, int B, int H0, int W0, int out_h, int out_w, uint8_t* tmp, uint8_t* out,
                 void* stream);
/* Largest source (and target) side the resize accepts: the horizontal pass stages 4 source rows of up to this many
 * pixels in shared memory.  Larger images are rejected with CA_STATUS_INVALID. */
#define CA_RESIZE_MAX_SIDE 16384
/* Images per launch of each resize pass: the per-image descriptors travel as one kernel parameter.  Larger batches are
 * resized in chunks of this many images. */
#define CA_RESIZE_LIST_CHUNK 128
/* B images of individual sizes -> uint8 [B, out_h, out_w, 3]; bit-exact PIL.Image.resize(..., BILINEAR) per image.
 * h_images: HOST array of B device pointers (uint8 HWC, contiguous); h_hw: HOST [B, 2] (H0, W0).  Per image a pass runs
 * only on an axis whose size changes (Pillow's semantics); an image of the target size is copied.  Each pass is one
 * launch for the whole batch (per CA_RESIZE_LIST_CHUNK images), whatever its mix of sizes.  tmp: at least
 * ca_resize_u8_list_tmp_bytes(h_hw, B, out_h, out_w) bytes (0 when no image changes both axes; tmp may then be NULL). */
size_t ca_resize_u8_list_tmp_bytes(const int* h_hw, int B, int out_h, int out_w);
int ca_resize_u8_list(const uint8_t* const* h_images, const int* h_hw, int B, int out_h, int out_w, uint8_t* tmp,
                      size_t tmp_bytes, uint8_t* out, void* stream);

/* ---- demo.py:312 `Image.open(path).convert('RGB')`: JPEG ingest through nvJPEG (CUDA toolkit; loaded lazily) ---------
 * h_data / len: one JPEG file's bytes in HOST memory.  ca_jpeg_info fills the decoded size; ca_jpeg_decode writes
 * height*width*3 bytes of interleaved RGB to the DEVICE buffer out_rgb on `stream` (grayscale streams are expanded to
 * RGB like PIL's convert).  Without nvJPEG both return CA_STATUS_UNSUPPORTED: there is no CPU decode fallback.
 * nvJPEG and libjpeg-turbo (inside Pillow) are different decoders: with the interpolating chroma up-sampler requested
 * here the results agree to <= 5 LSB (mean ~0.6), not bit for bit (tests/test_jpeg_gpu.py states the tolerance). */
int ca_jpeg_info(const uint8_t* h_data, size_t len, int* width, int* height);
int ca_jpeg_decode(const uint8_t* h_data, size_t len, uint8_t* out_rgb, int width, int height, void* stream);
/* n JPEG files in ONE call (nvjpegDecodeBatched: the Huffman stage of the whole batch on a host thread pool, one set of
 * GPU kernels): h_data[i] / lens[i] host bytes, outs[i] device RGB HWC buffers of widths[i] x heights[i] (from
 * ca_jpeg_info).  Replaces the per-file loop of reference demo.py:406-432 (`predict_batch`). */
int ca_jpeg_decode_batch(const uint8_t* const* h_data, const size_t* lens, int n, uint8_t* const* outs, const int* widths,
                         const int* heights, void* stream);

/* ---- visualisation post-processing (the consumer right after the hot path; replaces demo.py:530-563) ------------
 * norm[b, :]  = min-max( where(a > percentile70(a), a, 0.3 a) ),  a = heat[b, :]^3            (numpy float32 semantics)
 * out[b,y,x]  = scipy.ndimage.zoom(norm[b].reshape(g, g), (out_h / g, out_w / g), order=1)    (skipped when out is null)
 * heat, norm: [B, g*g] fp32; out: [B, out_h, out_w] fp32.  g*g <= 16384. */
int ca_focus_map(const float* heat, int B, int g, int out_h, int out_w, float* norm, float* out, void* stream);

/* ================================================================================================
 * Handle-level entry points: the whole forward behind ONE call (SURVEY.md §8b).
 *
 * The per-kernel entry points above are what the tests drive; a host that is not Python (or that wants no per-kernel
 * orchestration) creates a handle from a table of packed device weights and calls ca_forward_guided / ca_forward.  The
 * handle owns what the reference keeps in Python objects between calls: the per-resolution tables (position-embedding
 * interpolation, focal position encoding, centre bias, instruction masks — reference src/model.py:140-231, 1270-1376,
 * HF modeling_dinov2.py:57-95), the activation workspace per (batch, resolution), a ring of pinned staging buffers for the
 * per-call host inputs, a side stream for the CuriosityModule branch and one CUDA graph per (path, batch, resolution).
 * One handle per device; calls on one handle must be serialised by the caller (the reference is single-threaded too,
 * demo.py:79,338).  Replaces the flow of reference demo.py:298-405 (`predict`) / src/model.py:1157-1240, 1064-1155.
 * ================================================================================================ */
typedef struct ca_handle ca_handle;

/* DEVICE pointers to one encoder layer's operands: bf16 GEMM weights [out, in] (torch Linear layout), fp32 the rest. */
typedef struct ca_layer_weights {
  const float *n1w, *n1b;       /* norm1                                                    HF modeling_dinov2.py:354 */
  const uint16_t* wqkv;         /* [2304, 768] = query | key | value weights stacked         HF:203-214 */
  const float* bqkv;            /* [2304] */
  const uint16_t* wo;           /* attention.output.dense [768, 768]                         HF:246 */
  const float *bo, *ls1;        /* bias, layer_scale1.lambda1                                HF:278 */
  const float *n2w, *n2b;       /* norm2 */
  const uint16_t* w1;           /* mlp.fc1 [3072, 768] */
  const float* b1;
  const uint16_t* w2;           /* mlp.fc2 [768, 3072] */
  const float *b2, *ls2;
} ca_layer_weights;

typedef struct ca_focal_weights {
  const uint16_t* wqk;          /* [1536, 768] = query_proj | key_proj of one FocalStream      src/model.py:192-193 */
  const float* bqk;             /* [1536] */
  const float *wv, *bv;         /* value_proj [768,768], [768] fp32 (un-guided features only)  :194 */
  const float *pw0, *pb0, *pw1, *pb1; /* projection.{0,3} [256,768] [64,256]                   :311 */
} ca_focal_weights;

typedef struct ca_model_weights {
  const uint16_t* patch_w;      /* [768, 592] bf16: conv weight flattened (c, ky, kx), columns 588..591 zero */
  const float* patch_b;         /* [768] */
  const float* cls_token;       /* [768] */
  const float* pos_embed;       /* HOST pointer, fp32 [1 + 37*37, 768]: the native-grid position embedding (row 0 = CLS);
                                   interpolated per resolution by the handle */
  ca_layer_weights layer[12];
  const float *lnw, *lnb;       /* backbone.layernorm */
  int n_focal;                  /* focal iterations (1..4) */
  float focus_strength;         /* src/model.py:426 re-focus strength (1.5 under every shipped YAML) */
  ca_focal_weights focal[4];
  const float *ffw0, *ffb0, *ffw1, *ffb1;   /* focal_stream.fusion.{0,2}  [128,192] [64,128]   :430 */
  ca_heads_weights heads;
  ca_curiosity_weights curiosity;
  float* exploration_history;   /* curiosity_module.exploration_history (device, mutated)      :760-773 */
  int history_len;
  long long* history_pointer;   /* device int64 */
  int num_cameras;              /* rows of heads.cam_emb; 0 = the model has no EXIF prior */
  int layernorm_folded;         /* 1 = the caller folded norm1 into (wqkv, bqkv) and norm2 into (w1, b1) of every layer
                                   (W' = bf16(rows of W diag(gamma), centred), b' = b + W beta; see ca_gemm_bf16_ln): the
                                   encoder runs without LayerNorm passes and n1w / n1b / n2w / n2b are not read */
} ca_model_weights;

/* Per-call inputs.  Device pointers unless marked HOST.  The two Gaussian draws of the CuriosityModule and the per-call
 * random projection come from the caller because the reference takes them from ITS global generator (src/model.py:609,
 * 744, 1421): parity under a shared seed is the caller's RNG, not this library's. */
typedef struct ca_forward_call {
  const void* images;           /* fp32 [B,3,S,S] normalised, or (images_u8) uint8 [B,S,S,3] at model resolution */
  int images_u8;
  int B, S;
  const float* exif;            /* [B,3] raw focal_length, aperture, iso; NULL = no EXIF (zero slot; un-guided only) */
  const long long* camera_idx;  /* [B] */
  const char* instruction;      /* guided: one of the 9 instructions / aliases (HOST string); NULL when `mask` is given */
  const float* mask;            /* guided: explicit guidance [N] (mask_batch_stride 0) or per image [B,N] (stride N) */
  long long mask_batch_stride;
  const float* tmp_w;           /* HOST [64,768]: per-call projection weight (guided only)       src/model.py:1421 */
  const float* tmp_b;           /* HOST [64] */
  const float* eps;             /* HOST [runs,B,192]: CuriosityModule draw of :609, one per run (guided: 1 run) */
  const float* noise;           /* HOST [runs,B,768]: draw of :744 */
  int curiosity_runs;           /* un-guided: 1..3 runs as the reference makes them (:992, :1104, :1138); guided: 1 */
  float* depth;                 /* out [B] */
  float* conf;                  /* out [B] */
  float* attention;             /* out [B,N]: guided heat map / last-iteration focal attention */
  int* argmax;                  /* out [B] (guided) or NULL */
  float* fused;                 /* out [B,192] fusion features (un-guided) or NULL */
  int* fault;                   /* optional device-visible word: bit 0 = camera_idx out of range */
  int use_graph;                /* 1: capture the launch sequence once per (path, B, S) and replay it */
  /* Photographs of individual sizes (demo.py:406-432 `predict_batch` over a folder): when set, `images` must be NULL
   * and the handle resizes each image to S x S (exactly as ca_resize_u8_list does) into a buffer it owns, then
   * normalises and patchifies the batch.  The resize runs in front of the (possibly replayed) graph, so batches of
   * other sizes at the same (B, S) replay the same graph.  Zero-initialised callers keep the `images` behaviour. */
  const uint8_t* const* image_list; /* HOST [B]: device pointers to uint8 [H_i, W_i, 3] (contiguous) */
  const int* image_hw;              /* HOST [B, 2]: (H_i, W_i), each side at most CA_RESIZE_MAX_SIDE */
} ca_forward_call;

/* `w` (HOST struct of device pointers) is copied; the weights themselves must outlive the handle. */
int ca_create(ca_handle** out, const ca_model_weights* w, int device);
int ca_destroy(ca_handle* h);
/* forward_with_guidance(images, exif, instruction | guidance tensor) -> depth, confidence, heat map, arg-max cell. */
int ca_forward_guided(ca_handle* h, const ca_forward_call* call, void* stream);
/* Instruction sweep: K = 1..CA_SWEEP_MAX_K guided calls over one batch.  HOST pointers where marked, device otherwise. */
typedef struct ca_sweep_call {
  int K;
  const char* const* instructions; /* HOST [K] instruction strings / aliases, or NULL when `masks` is given */
  const float* masks;              /* [K, N] explicit guidance, one row per call, shared by the batch; or NULL */
  const float* tmp_w;              /* HOST [K, 64, 768]: the per-call projections, in call order  src/model.py:1421 */
  const float* tmp_b;              /* HOST [K, 64] */
  const float* eps;                /* HOST [K, B, 192]: the CuriosityModule draw of :609 of each call */
  const float* noise;              /* HOST [K, B, 768]: the draw of :744 of each call */
  float* depth;                    /* out [K, B] */
  float* conf;                     /* out [K, B] */
  float* attention;                /* out [K, B, N] heat maps */
  int* argmax;                     /* out [K, B] or NULL */
} ca_sweep_call;
/* K forward_with_guidance calls on the same images and EXIF, in one: the backbone and the focal iterations run once, the
 * CuriosityModule K times (the ring buffer receives K runs of B entries in call order), the guidance, pooling and heads
 * once for all K * B rows.  Bit-identical to K ca_forward_guided calls given the same per-call draws.  `call` supplies
 * images, images_u8, B, S, exif, camera_idx, fault and use_graph; its per-call fields (instruction, mask, tmp_w, tmp_b,
 * eps, noise, depth, conf, attention, argmax, fused) must be NULL. */
int ca_forward_guided_sweep(ca_handle* h, const ca_forward_call* call, const ca_sweep_call* sweep, void* stream);
/* forward(images, exif or none) -> depth, confidence, last-iteration focal attention, fusion features. */
int ca_forward(ca_handle* h, const ca_forward_call* call, void* stream);
/* DINOv2 tokens only: tokens_out fp32 [B, 1+N, 768] (BASELINE.json configs[2]). */
int ca_backbone(ca_handle* h, const void* images, int images_u8, int B, int S, float* tokens_out, void* stream);
/* The same from B photographs of individual sizes (HOST arrays as in ca_forward_call.image_list / image_hw), resized to
 * S x S by the handle. */
int ca_backbone_list(ca_handle* h, const uint8_t* const* image_list, const int* image_hw, int B, int S, float* tokens_out,
                     void* stream);
/* kernels launched by the last ca_forward* / ca_backbone call of this handle (the launch-count claim of bench.py). */
int ca_last_launch_count(const ca_handle* h);

/* Scenes: encode a batch once, guide it any number of times.  A scene owns the backbone tokens [B, 1+N, 768], the last
 * focal iteration's attention [B, N], the EXIF and camera indices of the batch, and the graphs captured on them; it
 * belongs to the handle that encoded it.  A scene of a destroyed handle (or of another handle) is refused with
 * CA_STATUS_INVALID and never dereferenced through its handle; so is a scene already destroyed. */
typedef struct ca_scene ca_scene;
/* The instruction-independent part of ca_forward_guided: `call` supplies images (or image_list / image_hw), images_u8,
 * B, S, exif, camera_idx (both required), fault (used by the scene's guide calls) and use_graph; its per-call fields
 * (instruction, mask, tmp_w, tmp_b, eps, noise, depth, conf, attention, argmax, fused) must be NULL. */
int ca_encode(ca_handle* h, const ca_forward_call* call, ca_scene** out, void* stream);
/* One guided call on a scene: HOST pointers where marked, device otherwise. */
typedef struct ca_guide_call {
  const char* instruction;      /* HOST instruction string / alias, or NULL when `mask` is given */
  const float* mask;            /* explicit guidance [N] (mask_batch_stride 0) or per image [B, N] (stride N) */
  long long mask_batch_stride;
  const float* tmp_w;           /* HOST [64, 768]: per-call projection weight   src/model.py:1421 */
  const float* tmp_b;           /* HOST [64] */
  const float* eps;             /* HOST [B, 192]: CuriosityModule draw of :609 */
  const float* noise;           /* HOST [B, 768]: draw of :744 */
  float* depth;                 /* out [B] */
  float* conf;                  /* out [B] */
  float* attention;             /* out [B, N] heat map */
  int* argmax;                  /* out [B] or NULL */
} ca_guide_call;
/* ca_forward_guided on the encoded images, bit for bit given the same draws, without the backbone and the focal pass:
 * the CuriosityModule run and the fused tail (ca_guide_tail).  With use_graph the launches are captured on the scene's
 * buffers at its second guide call and replayed after. */
int ca_guide(ca_handle* h, ca_scene* scene, const ca_guide_call* call, void* stream);
/* ca_forward_guided_sweep on the encoded images, bit for bit given the same draws (ca_sweep_call as there). */
int ca_guide_sweep(ca_handle* h, ca_scene* scene, const ca_sweep_call* sweep, void* stream);
/* A depth field of a scene: HOST pointers where marked, device otherwise. */
typedef struct ca_depth_field_call {
  const float* tmp_w;           /* HOST [64, 768]: per-call projection weight   src/model.py:1421 */
  const float* tmp_b;           /* HOST [64] */
  const float* eps;             /* HOST [B, 192]: CuriosityModule draw of :609 */
  const float* noise;           /* HOST [B, 768]: draw of :744 */
  float* depth;                 /* out [B, N]: cell c = y * g + x */
  float* conf;                  /* out [B, N] */
} ca_depth_field_call;
/* The guided depth and confidence with the focus mask of every cell of the grid (ca_depth_field_cells), from one call's
 * draws: one projection for every cell and one CuriosityModule run (B ring entries).  The scene graph policy and the
 * refusals are those of ca_guide. */
int ca_depth_field(ca_handle* h, ca_scene* scene, const ca_depth_field_call* call, void* stream);
/* One guide call on each of m scenes in one: HOST pointers where marked, device otherwise.  Rows r = 0..R-1 are the
 * images of the calls in call order, R = sum of the scenes' B. */
typedef struct ca_guide_many_call {
  int m;                           /* 1..CA_GUIDE_MANY_MAX_CALLS; R at most CA_GUIDE_MANY_MAX_ROWS */
  ca_scene* const* scenes;         /* HOST [m]: scenes of this handle, all of one side S; a scene may repeat */
  const char* const* instructions; /* HOST [m] instruction strings / aliases, or NULL when `masks` is given */
  const float* masks;              /* [R, N] explicit guidance, one row per image; or NULL */
  const float* tmp_w;              /* HOST [m, 64, 768]: the per-call projections, in call order  src/model.py:1421 */
  const float* tmp_b;              /* HOST [m, 64] */
  const float* eps;                /* HOST [R, 192]: the CuriosityModule draw of :609 of each call, rows in call order */
  const float* noise;              /* HOST [R, 768]: the draw of :744 */
  float* depth;                    /* out [R] */
  float* conf;                     /* out [R] */
  float* attention;                /* out [R, N] heat maps */
  int* argmax;                     /* out [R] or NULL */
  int use_graph;                   /* 1: capture the launches at the second call of this (S, R, m) and replay them after,
                                      for any scenes */
} ca_guide_many_call;
/* m ca_guide calls, one per scene, bit for bit given the same draws, in ONE pass over the R rows: the row inputs
 * gathered through a row table (ca_gather_rows), one CuriosityModule run over the R CLS rows (the ring receives them in
 * call order), the guided softmax, ca_weighted_pool_rows and the heads with call_of_row.  Each scene's graphs are left
 * alone.  Every scene is checked as ca_guide checks it before anything is enqueued; a bad camera index of scene j is
 * reported in scene j's fault word. */
int ca_guide_many(ca_handle* h, const ca_guide_many_call* call, void* stream);
/* Release a scene's memory and graphs (waits for the device).  NULL is a no-op. */
int ca_scene_destroy(ca_scene* scene);

#ifdef __cplusplus
}
#endif
#endif /* COGAIM_B200_H_ */
