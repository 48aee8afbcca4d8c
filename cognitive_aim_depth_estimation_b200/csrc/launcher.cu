// Handle-level C-ABI (include/cogaim_b200.h, "Handle-level entry points"): the whole forward of the Cognitive-Aim model
// behind one call, for hosts that do not want to orchestrate ~110 kernel launches themselves.
//
// This file is host code only.  It owns what the reference keeps alive in Python objects between calls:
//   * per-resolution tables — DINOv2 position-embedding interpolation (HF modeling_dinov2.py:57-95: identity at the native
//     37 x 37 grid, bicubic align_corners=False otherwise), the focal 2-D sinusoidal position encoding
//     (src/model.py:140-166), the Gaussian centre bias (:208-231) and the instruction masks (:1270-1376);
//   * one activation workspace per (batch, resolution), carved out of a single device allocation;
//   * a ring of pinned staging buffers for the per-call HOST inputs (per-call projection, curiosity draws), pulled to the
//     device by SM-side reads so they never queue on the H2D copy engine behind the application's image upload;
//   * the launch sequence itself (the same kernels, in the same order, as cognitive_aim_depth_estimation_b200/model.py),
//     the CuriosityModule on a forked side stream, and one CUDA graph per (path, batch, resolution).
// The first call of a (path, batch, resolution) runs eagerly (one-time allocations and kernel attributes are illegal
// during capture), the second is captured and launched as a graph, later calls replay it.
#include "../../include/cogaim_b200.h"

#include <math.h>
#include <string.h>

#include <atomic>

#include <map>
#include <mutex>
#include <set>
#include <string>
#include <tuple>
#include <vector>

#include "attention.cuh"
#include "curiosity.cuh"
#include "focal.cuh"
#include "gemm.cuh"
#include "heads.cuh"
#include "host.h"
#include "resize.cuh"
#include "rowops.cuh"

namespace {

constexpr int kD = 768, kHeads = 12, kLayers = 12, kMlp = 3072, kPoolSplits = 32, kMaxRuns = 3, kNativeGrid = 37;
constexpr float kLog2e = 1.4426950408889634f;

struct Tables {
  float* pos = nullptr;    // [1 + N, 768]
  float* pe = nullptr;     // [N, 768]
  float* cbias = nullptr;  // [N]
  std::map<std::string, float*> masks;
};

struct Workspace {
  int B = 0, S = 0;
  unsigned long long gen = 0;  // unique per allocation: a scene's graphs captured on another workspace are not replayed
  void* arena = nullptr;
  __nv_bfloat16 *patches, *h, *qkv, *att, *mlp, *xin, *qk;
  float *x, *tokens, *pm, *ps, *pc, *wtab, *attn, *cvec, *rowscale, *heat, *pool, *pool_pe, *pooled, *feats, *focal_feat,
      *fused, *depth, *conf, *mask_in, *tmpw, *tmpb, *exif_in, *cur_eps, *cur_noise, *cur_raw, *cur_reward, *ln_stats;
  void* E;
  int* argmax;
  int* tail_ticket;  // [B] per-image tickets of the fused guide tail, zero when idle
  long long* cam_in;
  int P = 0, lde = 0;
  std::map<int, std::pair<cudaGraphExec_t, int>> graphs;  // path key -> (executable graph, launches)
  std::map<int, int> seen;                                // path key -> calls so far
  // instruction sweeps: the per-call buffers of K calls (rows k * B + b), one arena per K; the backbone and focal
  // buffers above are shared with the single-call paths
  struct Sweep {
    void* arena = nullptr;
    float *mask_in, *heat, *pool, *depth, *conf, *tmpw, *tmpb, *cur_eps, *cur_noise, *cur_raw, *cur_reward;
    int* argmax;
  };
  std::map<int, Sweep> sweeps;  // K -> buffers
};

void free_workspace(Workspace& w) {
  for (auto& g : w.graphs) cudaGraphExecDestroy(g.second.first);
  for (auto& s : w.sweeps) cudaFree(s.second.arena);
  cudaFree(w.arena);
}

struct PinnedSlot {
  float* buf = nullptr;
  size_t cap = 0;
  cudaEvent_t done = nullptr;
};

}  // namespace

struct ca_handle {
  ca_model_weights w;
  std::vector<float> pos_native;  // host copy of the native-grid position embedding
  int device = 0;
  std::map<int, Tables> tables;
  std::map<std::pair<int, int>, Workspace> ws;
  PinnedSlot ring[4];
  int ring_next = 0;
  cudaStream_t side = nullptr;
  cudaEvent_t fork = nullptr, join = nullptr;
  int launches = 0;       // running count of the sequence being issued
  int last_launches = 0;  // of the last completed call
  // photographs of individual sizes (ca_forward_call.image_list): the resized uint8 [B, S, S, 3] batch followed by the
  // resize temporary, grow-only
  uint8_t* resize_buf = nullptr;
  size_t resize_cap = 0;
  unsigned long long id = 0;  // unique per handle: scenes record it (a later handle may reuse the address)
};

// A scene (ca_encode): buffers it owns in one device allocation, the handle it belongs to (by id, never dereferenced
// once that handle is gone), and the graphs of its guide calls, captured on its own buffers and one workspace.
struct ca_scene {
  unsigned long long handle_id = 0;
  int device = 0, B = 0, S = 0;
  void* arena = nullptr;
  float *tokens = nullptr, *base = nullptr, *exif = nullptr;
  long long* cam = nullptr;
  int* fault = nullptr;
  bool use_graph = false;
  unsigned long long ws_gen = 0;                           // workspace the graphs below were captured on
  std::map<int, std::pair<cudaGraphExec_t, int>> graphs;  // path key -> (executable graph, launches)
  std::map<int, int> seen;                                // path key -> calls so far
};

namespace {

using ca::invalid;
using ca::set_error;

// ------------------------------------------------------------------------------------------------------------------
// host-side tables
// ------------------------------------------------------------------------------------------------------------------
// torch.nn.functional.interpolate(mode="bicubic", align_corners=False) as ATen's upsample_bicubic2d computes it in fp32:
// source coordinate scale * (dst + 0.5) - 0.5 with scale = in / out, cubic-convolution coefficients with A = -0.75, border
// samples clamped, rows interpolated along x first, then along y.
inline float cubic1(float x, float A) { return ((A + 2.f) * x - (A + 3.f)) * x * x + 1.f; }
inline float cubic2(float x, float A) { return ((A * x - 5.f * A) * x + 8.f * A) * x - 4.f * A; }
inline void cubic_coeffs(float t, float c[4]) {
  const float A = -0.75f;
  c[0] = cubic2(t + 1.f, A);
  c[1] = cubic1(t, A);
  c[2] = cubic1(1.f - t, A);
  c[3] = cubic2(2.f - t, A);
}

std::vector<float> interpolate_pos(const std::vector<float>& native, int g) {
  const int g0 = kNativeGrid;
  std::vector<float> out(static_cast<size_t>(1 + g * g) * kD);
  memcpy(out.data(), native.data(), kD * sizeof(float));  // CLS row
  if (g == g0) {
    memcpy(out.data(), native.data(), out.size() * sizeof(float));
    return out;
  }
  const float scale = static_cast<float>(g0) / static_cast<float>(g);
  std::vector<int> ix(g);
  std::vector<float> cx(static_cast<size_t>(g) * 4);
  for (int o = 0; o < g; ++o) {
    const float real = scale * (o + 0.5f) - 0.5f;
    const float fl = floorf(real);
    ix[o] = static_cast<int>(fl);
    cubic_coeffs(real - fl, &cx[static_cast<size_t>(o) * 4]);
  }
  auto clampi = [&](int v) { return v < 0 ? 0 : (v > g0 - 1 ? g0 - 1 : v); };
  const float* src = native.data() + kD;  // [g0, g0, D]
  for (int oy = 0; oy < g; ++oy) {
    const float* cy = &cx[static_cast<size_t>(oy) * 4];
    for (int ox = 0; ox < g; ++ox) {
      const float* cxx = &cx[static_cast<size_t>(ox) * 4];
      float* dst = out.data() + (static_cast<size_t>(1) + static_cast<size_t>(oy) * g + ox) * kD;
      for (int d = 0; d < kD; ++d) {
        float rows[4];
        for (int i = 0; i < 4; ++i) {
          const float* r = src + (static_cast<size_t>(clampi(ix[oy] - 1 + i)) * g0) * kD + d;
          rows[i] = r[static_cast<size_t>(clampi(ix[ox] - 1)) * kD] * cxx[0] + r[static_cast<size_t>(clampi(ix[ox])) * kD] * cxx[1] +
                    r[static_cast<size_t>(clampi(ix[ox] + 1)) * kD] * cxx[2] + r[static_cast<size_t>(clampi(ix[ox] + 2)) * kD] * cxx[3];
        }
        dst[d] = rows[0] * cy[0] + rows[1] * cy[1] + rows[2] * cy[2] + rows[3] * cy[3];
      }
    }
  }
  return out;
}

// src/model.py:140-166: first half of the channels encodes the patch row, second half the column; even index sin, odd cos
std::vector<float> focal_pe(int g) {
  const int n = g * g, half = kD / 2;
  std::vector<float> pe(static_cast<size_t>(n) * kD, 0.f);
  std::vector<float> div(half / 2);
  const float k = static_cast<float>(-(log(10000.0) / half));
  for (int i = 0; i < half / 2; ++i) div[i] = expf(static_cast<float>(2 * i) * k);
  for (int idx = 0; idx < n; ++idx) {
    const float row = static_cast<float>(idx / g), col = static_cast<float>(idx % g);
    float* p = pe.data() + static_cast<size_t>(idx) * kD;
    for (int i = 0; i < half / 2; ++i) {
      p[2 * i] = sinf(row * div[i]);
      p[2 * i + 1] = cosf(row * div[i]);
      p[half + 2 * i] = sinf(col * div[i]);
      p[half + 2 * i + 1] = cosf(col * div[i]);
    }
  }
  return pe;
}

// src/model.py:208-231: 0.3 * exp(-d^2 / (2 sigma^2)), sigma = g / 6, centre (g // 2, g // 2)
std::vector<float> center_bias(int g) {
  std::vector<float> b(static_cast<size_t>(g) * g);
  const int c = g / 2;
  const float denom = static_cast<float>(2.0 * (g / 6.0) * (g / 6.0));
  for (int y = 0; y < g; ++y)
    for (int x = 0; x < g; ++x) {
      const float fx = static_cast<float>(x - c), fy = static_cast<float>(y - c);
      const float dist = sqrtf(fx * fx + fy * fy);
      b[static_cast<size_t>(y) * g + x] = expf(-(dist * dist) / denom) * 0.3f;
    }
  return b;
}

// src/model.py:1270-1376: `.lower()`, aliases without the hyphen, unknown strings -> all ones
bool instruction_mask(const char* instruction, int g, std::vector<float>* out) {
  std::string s(instruction);
  for (auto& ch : s) ch = static_cast<char>(tolower(ch));
  if (s == "topleft") s = "top-left";
  if (s == "topright") s = "top-right";
  if (s == "bottomleft") s = "bottom-left";
  if (s == "bottomright") s = "bottom-right";
  out->assign(static_cast<size_t>(g) * g, 1.0f);
  const int q = g / 4, h = g / 2, t = g * 3 / 4;
  int fy, fx, r;
  float hi, lo;
  if (s == "center") { fy = h; fx = h; r = g / 4 > 1 ? g / 4 : 1; hi = 3.0f; lo = 1.5f; }
  else {
    r = g / 6 > 1 ? g / 6 : 1; hi = 5.0f; lo = 2.0f;
    if (s == "left") { fy = h; fx = q; }
    else if (s == "right") { fy = h; fx = t; }
    else if (s == "top") { fy = q; fx = h; }
    else if (s == "bottom") { fy = t; fx = h; }
    else if (s == "top-left") { fy = q; fx = q; }
    else if (s == "top-right") { fy = q; fx = t; }
    else if (s == "bottom-left") { fy = t; fx = q; }
    else if (s == "bottom-right") { fy = t; fx = t; }
    else return true;  // unknown instruction: uniform guidance (reference behaviour)
  }
  for (int y = 0; y < g; ++y)
    for (int x = 0; x < g; ++x) {
      const double dist = sqrt(static_cast<double>((y - fy) * (y - fy) + (x - fx) * (x - fx)));
      float& m = (*out)[static_cast<size_t>(y) * g + x];
      if (dist <= 2 * r) m = lo;
      if (dist <= r) m = hi;
    }
  return true;
}

int upload(const std::vector<float>& v, float** dst) {
  CA_CUDA(cudaMalloc(dst, v.size() * sizeof(float)));
  CA_CUDA(cudaMemcpy(*dst, v.data(), v.size() * sizeof(float), cudaMemcpyHostToDevice));
  return 0;
}

int get_tables(ca_handle* h, int g, Tables** out) {
  auto it = h->tables.find(g);
  if (it == h->tables.end()) {
    CA_REQUIRE(g >= 4, "patch grids smaller than 4 x 4 are not supported (the reference's degenerate-variance fallbacks, "
                       "src/model.py:242-257, are not built)");
    Tables t;
    CA_TRY(upload(interpolate_pos(h->pos_native, g), &t.pos));
    CA_TRY(upload(focal_pe(g), &t.pe));
    CA_TRY(upload(center_bias(g), &t.cbias));
    it = h->tables.emplace(g, t).first;
  }
  *out = &it->second;
  return 0;
}

int get_mask(Tables* t, const char* instruction, int g, float** out) {
  std::string key(instruction);
  auto it = t->masks.find(key);
  if (it == t->masks.end()) {
    std::vector<float> m;
    instruction_mask(instruction, g, &m);
    float* d = nullptr;
    CA_TRY(upload(m, &d));
    it = t->masks.emplace(key, d).first;
  }
  *out = it->second;
  return 0;
}

// ------------------------------------------------------------------------------------------------------------------
// workspace
// ------------------------------------------------------------------------------------------------------------------
int get_workspace(ca_handle* h, int B, int S, Workspace** out) {
  const auto key = std::make_pair(B, S);
  auto it = h->ws.find(key);
  if (it != h->ws.end()) {
    *out = &it->second;
    return 0;
  }
  if (h->ws.size() >= 4) {  // keep the cache bounded: drop the oldest entry
    auto old = h->ws.begin();
    free_workspace(old->second);
    h->ws.erase(old);
  }
  Workspace w;
  w.B = B;
  w.S = S;
  const int g = S / 14;
  const size_t N = static_cast<size_t>(g) * g, T = N + 1, M = B * T, BN = B * N;
  w.P = ca::gemm_stats_partials(static_cast<int>(N));
  w.lde = 64 * static_cast<int>((N + 63) / 64);
  const int iters = h->w.n_focal;
  size_t off = 0;
  auto take = [&](size_t bytes) {
    const size_t o = off;
    off += (bytes + 255) & ~static_cast<size_t>(255);
    return o;
  };
  struct Slot { void** p; size_t o; };
  std::vector<Slot> slots;
  auto want = [&](auto** p, size_t bytes) { slots.push_back({reinterpret_cast<void**>(p), take(bytes)}); };
  want(&w.patches, BN * ca::kPatchRowStride * 2);
  want(&w.x, M * kD * 4);
  want(&w.h, M * kD * 2);
  want(&w.ln_stats, M * (kD / 128) * 2 * 4);
  want(&w.qkv, M * 3 * kD * 2);
  want(&w.att, M * kD * 2);
  want(&w.mlp, M * kMlp * 2);
  want(&w.tokens, M * kD * 4);
  want(&w.xin, BN * kD * 2);
  want(&w.qk, BN * 2 * kD * 2);
  want(&w.pm, BN * w.P * 4);
  want(&w.ps, BN * w.P * 4);
  want(&w.pc, BN * w.P * 4);
  want(&w.wtab, BN * w.P * 4);
  want(&w.E, BN * w.lde * 2);
  want(&w.attn, iters * BN * 4);
  want(&w.cvec, BN * 4);
  want(&w.rowscale, 2 * BN * 4);
  want(&w.heat, BN * 4);
  want(&w.argmax, B * 4);
  want(&w.pool, static_cast<size_t>(B) * kPoolSplits * kD * 4);
  want(&w.pool_pe, static_cast<size_t>(B) * kPoolSplits * kD * 4);
  want(&w.pooled, static_cast<size_t>(B) * kD * 4);
  want(&w.feats, static_cast<size_t>(B) * iters * 64 * 4);
  want(&w.focal_feat, static_cast<size_t>(B) * 64 * 4);
  want(&w.fused, static_cast<size_t>(B) * 192 * 4);
  want(&w.depth, B * 4);
  want(&w.conf, B * 4);
  want(&w.mask_in, BN * 4);
  want(&w.tmpw, 64 * kD * 4);
  want(&w.tmpb, 64 * 4);
  want(&w.exif_in, B * 3 * 4);
  want(&w.cam_in, B * 8);
  want(&w.tail_ticket, B * 4);
  want(&w.cur_eps, static_cast<size_t>(kMaxRuns) * B * 192 * 4);
  want(&w.cur_noise, static_cast<size_t>(kMaxRuns) * B * kD * 4);
  want(&w.cur_raw, static_cast<size_t>(kMaxRuns) * B * 4);
  want(&w.cur_reward, static_cast<size_t>(kMaxRuns) * B * 4);
  CA_CUDA(cudaMalloc(&w.arena, off));
  for (auto& s : slots) *s.p = static_cast<char*>(w.arena) + s.o;
  CA_CUDA(cudaMemset(w.exif_in, 0, B * 3 * 4));
  CA_CUDA(cudaMemset(w.cam_in, 0, B * 8));
  CA_CUDA(cudaMemset(w.tail_ticket, 0, B * 4));
  static std::atomic<unsigned long long> next_gen{1};
  w.gen = next_gen.fetch_add(1);
  *out = &h->ws.emplace(key, w).first->second;
  return 0;
}

int get_sweep(Workspace& w, int K, Workspace::Sweep** out) {
  auto it = w.sweeps.find(K);
  if (it == w.sweeps.end()) {
    const int g = w.S / 14;
    const size_t N = static_cast<size_t>(g) * g, KB = static_cast<size_t>(K) * w.B;
    size_t off = 0;
    std::vector<std::pair<void**, size_t>> slots;
    Workspace::Sweep s;
    auto want = [&](auto** p, size_t bytes) {
      slots.push_back({reinterpret_cast<void**>(p), off});
      off += (bytes + 255) & ~static_cast<size_t>(255);
    };
    want(&s.mask_in, K * N * 4);
    want(&s.heat, KB * N * 4);
    want(&s.argmax, KB * 4);
    want(&s.pool, KB * kPoolSplits * kD * 4);
    want(&s.depth, KB * 4);
    want(&s.conf, KB * 4);
    want(&s.tmpw, static_cast<size_t>(K) * 64 * kD * 4);
    want(&s.tmpb, static_cast<size_t>(K) * 64 * 4);
    want(&s.cur_eps, KB * 192 * 4);
    want(&s.cur_noise, KB * kD * 4);
    want(&s.cur_raw, KB * 4);
    want(&s.cur_reward, KB * 4);
    CA_CUDA(cudaMalloc(&s.arena, off));
    for (auto& sl : slots) *sl.first = static_cast<char*>(s.arena) + sl.second;
    it = w.sweeps.emplace(K, s).first;
  }
  *out = &it->second;
  return 0;
}

// ------------------------------------------------------------------------------------------------------------------
// launch sequences (same kernels and order as model.py)
// ------------------------------------------------------------------------------------------------------------------
#define LAUNCH(expr)       \
  do {                     \
    CA_TRY(expr);          \
    ++h->launches;         \
  } while (0)

int gemm(ca_handle* h, const void* A, const void* W, int M, int N, int K, int epi, void* out, int ldo, const float* bias,
         const float* ls, const float* pos, int patches_per_img, cudaStream_t st, int lda = 0, int ldw = 0) {
  ca::GemmArgs a{};
  a.A = static_cast<const __nv_bfloat16*>(A);
  a.W = static_cast<const __nv_bfloat16*>(W);
  a.M = M;
  a.N = N;
  a.K = K;
  a.lda = lda ? lda : K;
  a.ldw = ldw ? ldw : K;
  a.batch = 1;
  a.epilogue = epi;
  a.out = out;
  a.ldo = ldo;
  a.bias = bias;
  a.ls = ls;
  a.pos = pos;
  a.patches_per_img = patches_per_img;
  LAUNCH(ca::gemm_launch(a, st));
  return 0;
}

int gemm_ln(ca_handle* h, const void* A, const void* W, int M, int N, int K, int epi, void* out, int ldo, const float* bias,
            const float* ls, float* stats, __nv_bfloat16* shadow, cudaStream_t st) {
  ca::GemmArgs a{};
  a.A = static_cast<const __nv_bfloat16*>(A);
  a.W = static_cast<const __nv_bfloat16*>(W);
  a.M = M;
  a.N = N;
  a.K = K;
  a.lda = K;
  a.ldw = K;
  a.batch = 1;
  a.epilogue = epi;
  a.out = out;
  a.ldo = ldo;
  a.bias = bias;
  a.ls = ls;
  a.ln_stats = stats;
  a.ln_slots = kD / 128;
  a.ln_eps = 1e-6f;
  a.shadow = shadow;
  a.ld_shadow = kD;
  LAUNCH(ca::gemm_launch(a, st));
  return 0;
}

int backbone_layers(ca_handle* h, Workspace& w, const Tables& tb, cudaStream_t st) {
  const int B = w.B, g = w.S / 14, N = g * g, T = N + 1, M = B * T;
  const ca_model_weights& mw = h->w;
  LAUNCH(ca::cls_rows_launch(w.x, mw.cls_token, tb.pos, B, T, kD, st));
  CA_TRY(gemm(h, w.patches, mw.patch_w, B * N, kD, ca::kPatchRowStride, ca::EPI_PATCH_F32, w.x, kD, mw.patch_b, nullptr, tb.pos, N, st,
              ca::kPatchRowStride, ca::kPatchRowStride));
  // LayerNorm-folded operands (ca_model_weights.layernorm_folded): norm1 / norm2 live in the epilogues of the GEMMs either
  // side of them; `w.h` then carries the raw residual rows as bf16 and `w.ln_stats` their statistics.
  const bool fold = mw.layernorm_folded != 0;
  if (fold) LAUNCH(ca::ln_shadow_launch(w.x, w.h, kD, w.ln_stats, M, kD, st));
  for (int l = 0; l < kLayers; ++l) {
    const ca_layer_weights& L = mw.layer[l];
    if (fold) {
      CA_TRY(gemm_ln(h, w.h, L.wqkv, M, 3 * kD, kD, ca::EPI_LN_BIAS_BF16, w.qkv, 3 * kD, L.bqkv, nullptr, w.ln_stats, nullptr, st));
    } else {
      LAUNCH(ca::layernorm_launch(w.x, L.n1w, L.n1b, w.h, 1, M, kD, 1e-6f, st));
      CA_TRY(gemm(h, w.h, L.wqkv, M, 3 * kD, kD, ca::EPI_BIAS_BF16, w.qkv, 3 * kD, L.bqkv, nullptr, nullptr, 0, st));
    }
    LAUNCH(ca::attention_launch(w.qkv, w.att, B, T, kHeads, st));
    if (fold) {
      CA_TRY(gemm_ln(h, w.att, L.wo, M, kD, kD, ca::EPI_RESID_LN_F32, w.x, kD, L.bo, L.ls1, w.ln_stats, w.h, st));
      CA_TRY(gemm_ln(h, w.h, L.w1, M, kMlp, kD, ca::EPI_LN_GELU_BF16, w.mlp, kMlp, L.b1, nullptr, w.ln_stats, nullptr, st));
    } else {
      CA_TRY(gemm(h, w.att, L.wo, M, kD, kD, ca::EPI_RESID_F32, w.x, kD, L.bo, L.ls1, nullptr, 0, st));
      LAUNCH(ca::layernorm_launch(w.x, L.n2w, L.n2b, w.h, 1, M, kD, 1e-6f, st));
      CA_TRY(gemm(h, w.h, L.w1, M, kMlp, kD, ca::EPI_GELU_BF16, w.mlp, kMlp, L.b1, nullptr, nullptr, 0, st));
    }
    if (fold && l + 1 < kLayers)
      CA_TRY(gemm_ln(h, w.mlp, L.w2, M, kD, kMlp, ca::EPI_RESID_LN_F32, w.x, kD, L.b2, L.ls2, w.ln_stats, w.h, st));
    else  // the final LayerNorm reads the fp32 rows itself
      CA_TRY(gemm(h, w.mlp, L.w2, M, kD, kMlp, ca::EPI_RESID_F32, w.x, kD, L.b2, L.ls2, nullptr, 0, st));
  }
  LAUNCH(ca::layernorm_launch(w.x, mw.lnw, mw.lnb, w.tokens, 0, M, kD, 1e-6f, st));
  return 0;
}

// IterativeFocalStream (src/model.py:391-455); returns the last iteration's attention in *attn_out
int focal_iterations(ca_handle* h, Workspace& w, const Tables& tb, bool want_features, cudaStream_t st, float** attn_out) {
  const int B = w.B, g = w.S / 14, N = g * g, T = N + 1;
  const ca_model_weights& mw = h->w;
  const float scale_log2 = kLog2e / sqrtf(static_cast<float>(kD / 8));  // single head, sqrt(768 // 8)  (src/model.py:69)
  const size_t BN = static_cast<size_t>(B) * N;
  const float* rs = nullptr;
  for (int i = 0; i < mw.n_focal; ++i) {
    const ca_focal_weights& F = mw.focal[i];
    LAUNCH(ca::focal_input_launch(w.tokens, tb.pe, rs, w.xin, B, N, kD, st));
    CA_TRY(gemm(h, w.xin, F.wqk, B * N, 2 * kD, kD, ca::EPI_BIAS_BF16, w.qk, 2 * kD, F.bqk, nullptr, nullptr, 0, st));
    ca::GemmArgs a{};
    a.A = w.qk;
    a.W = w.qk + kD;
    a.M = N;
    a.N = N;
    a.K = kD;
    a.lda = 2 * kD;
    a.ldw = 2 * kD;
    a.batch = B;
    a.a_batch_stride = static_cast<long long>(N) * 2 * kD;
    a.w_batch_stride = static_cast<long long>(N) * 2 * kD;
    a.epilogue = ca::EPI_ROWSTATS;
    a.out = w.E;
    a.ldo = w.lde;
    a.out_batch_stride = static_cast<long long>(N) * w.lde;
    a.scale_log2 = scale_log2;
    a.part_a = w.pm;
    a.part_b = w.ps;
    LAUNCH(ca::gemm_launch(a, st));
    LAUNCH(ca::rowstats_merge_launch(w.pm, w.ps, nullptr, nullptr, nullptr, w.wtab, B * N, N, w.P, st));
    LAUNCH(ca::colsum_e_launch(w.E, w.lde, static_cast<long long>(N) * w.lde, w.wtab, w.pc, B, N, w.P, st));
    const bool last = i == mw.n_focal - 1;
    float* rs_out = last ? nullptr : w.rowscale + (i % 2) * BN;
    float* attn = w.attn + static_cast<size_t>(i) * BN;
    LAUNCH(ca::focal_finalize_launch(w.pc, tb.cbias, attn, rs, rs_out, B, N, w.P, mw.focus_strength, 0, nullptr, 0.5f, st));
    if (want_features) {
      // value path re-associated: sum_i a_i (A V)_i = ((a^T A) x~) Wv^T + bv   (src/model.py:204,308)
      LAUNCH(ca::rowstats_merge_launch(w.pm, w.ps, attn, nullptr, nullptr, w.wtab, B * N, N, w.P, st));
      LAUNCH(ca::colsum_e_launch(w.E, w.lde, static_cast<long long>(N) * w.lde, w.wtab, w.pc, B, N, w.P, st));
      LAUNCH(ca::focal_finalize_launch(w.pc, nullptr, w.cvec, nullptr, nullptr, B, N, w.P, 0.0f, 1, nullptr, 0.5f, st));
      LAUNCH(ca::weighted_pool_launch(w.tokens, static_cast<long long>(T) * kD, 1, w.cvec, rs, w.pool, B, N, kD, kPoolSplits, st));
      LAUNCH(ca::weighted_pool_launch(tb.pe, 0, 0, w.cvec, nullptr, w.pool_pe, B, N, kD, kPoolSplits, st));
      ca_focal_value_args v{};
      v.tok_partial = w.pool;
      v.pe_partial = w.pool_pe;
      v.splits = kPoolSplits;
      v.wv = F.wv;
      v.bv = F.bv;
      v.proj_w0 = F.pw0;
      v.proj_b0 = F.pb0;
      v.proj_w1 = F.pw1;
      v.proj_b1 = F.pb1;
      v.feat_out = w.feats;
      v.iter = i;
      v.n_iters = mw.n_focal;
      LAUNCH(ca::focal_value_launch(v, B, st));
    }
    rs = rs_out;
  }
  if (want_features)
    LAUNCH(ca::focal_fusion_launch(w.feats, mw.n_focal, mw.ffw0, mw.ffb0, mw.ffw1, mw.ffb1, w.focal_feat, B, st));
  *attn_out = w.attn + static_cast<size_t>(mw.n_focal - 1) * BN;
  return 0;
}

// CuriosityModule runs of one call on the side stream (forked here, joined by curiosity_join): output-dead under the
// shipped configurations and latency-bound, so it runs under the focal stream's GEMMs.  The fork / join are stream
// dependencies: during capture they become a parallel branch of the graph.
// eps / noise / raw / reward: [runs, B, ...] buffers of the runs (the workspace's, or an instruction sweep's).
int curiosity_fork(ca_handle* h, Workspace& w, int runs, const float* eps, const float* noise, float* raw, float* reward,
                   cudaStream_t st, const float* tokens = nullptr) {
  const int B = w.B, g = w.S / 14, T = g * g + 1;
  CA_CUDA(cudaEventRecord(h->fork, st));
  CA_CUDA(cudaStreamWaitEvent(h->side, h->fork, 0));
  for (int j = 0; j < runs; ++j) {
    CA_TRY(ca::curiosity_launch(h->w.curiosity, tokens ? tokens : w.tokens, T, eps + static_cast<size_t>(j) * B * 192,
                                noise + static_cast<size_t>(j) * B * kD, raw + static_cast<size_t>(j) * B,
                                reward + static_cast<size_t>(j) * B, h->w.exploration_history, h->w.history_len,
                                h->w.history_pointer, B, h->side));
    h->launches += h->w.exploration_history ? 2 : 1;
  }
  return 0;
}

int curiosity_join(ca_handle* h, cudaStream_t st) {
  CA_CUDA(cudaEventRecord(h->join, h->side));
  CA_CUDA(cudaStreamWaitEvent(st, h->join, 0));
  return 0;
}

int heads(ca_handle* h, Workspace& w, bool guided, bool has_exif, int* fault, cudaStream_t st) {
  const int g = w.S / 14, T = g * g + 1;
  ca_heads_inputs in{};
  in.tokens = w.tokens;
  in.tokens_per_img = T;
  if (guided) {
    in.pool_partial = w.pool;
    in.pool_splits = kPoolSplits;
    in.tmp_w = w.tmpw;
    in.tmp_b = w.tmpb;
    in.pooled_out = w.pooled;
  } else {
    in.focal_feat = w.focal_feat;
  }
  in.exif = has_exif ? w.exif_in : nullptr;
  in.camera_idx = has_exif ? w.cam_in : nullptr;
  in.num_cameras = h->w.num_cameras;
  in.fault = fault;
  LAUNCH(ca::heads_launch(h->w.heads, in, w.depth, w.conf, guided ? nullptr : w.fused, w.B, st));
  return 0;
}

// per-call HOST inputs -> pinned staging slot -> fixed device buffers (SM-side reads of the pinned memory)
// next slot of the pinned ring, holding at least `need` floats
int pinned_slot(ca_handle* h, size_t need, PinnedSlot** out) {
  PinnedSlot& s = h->ring[h->ring_next];
  h->ring_next = (h->ring_next + 1) % 4;
  if (s.done) CA_CUDA(cudaEventSynchronize(s.done));  // the reads of four calls ago (normally long finished)
  if (s.cap < need) {
    if (s.buf) CA_CUDA(cudaFreeHost(s.buf));
    CA_CUDA(cudaHostAlloc(&s.buf, need * sizeof(float), cudaHostAllocDefault));
    s.cap = need;
  }
  if (!s.done) CA_CUDA(cudaEventCreateWithFlags(&s.done, cudaEventDisableTiming));
  *out = &s;
  return 0;
}

int stage_host_inputs(ca_handle* h, Workspace& w, const ca_forward_call& c, bool guided, int runs, cudaStream_t st) {
  const size_t B = w.B;
  const size_t n_w = guided ? 64 * kD + 64 : 0;
  const size_t need = n_w + static_cast<size_t>(runs) * B * (192 + kD);
  PinnedSlot* sp = nullptr;
  CA_TRY(pinned_slot(h, need, &sp));
  PinnedSlot& s = *sp;
  float* p = s.buf;
  if (guided) {
    memcpy(p, c.tmp_w, 64 * kD * sizeof(float));
    memcpy(p + 64 * kD, c.tmp_b, 64 * sizeof(float));
    CA_TRY(ca::fetch_pinned_launch(w.tmpw, p, 64 * kD, st));
    CA_TRY(ca::fetch_pinned_launch(w.tmpb, p + 64 * kD, 64, st));
    h->launches += 2;
    p += n_w;
  }
  memcpy(p, c.eps, static_cast<size_t>(runs) * B * 192 * sizeof(float));
  memcpy(p + static_cast<size_t>(runs) * B * 192, c.noise, static_cast<size_t>(runs) * B * kD * sizeof(float));
  CA_TRY(ca::fetch_pinned_launch(w.cur_eps, p, static_cast<size_t>(runs) * B * 192, st));
  CA_TRY(ca::fetch_pinned_launch(w.cur_noise, p + static_cast<size_t>(runs) * B * 192, static_cast<size_t>(runs) * B * kD, st));
  h->launches += 2;
  CA_CUDA(cudaEventRecord(s.done, st));
  return 0;
}

// the K calls' projections and curiosity draws (HOST) -> one pinned slot sized for K -> the sweep's device buffers
int stage_sweep_inputs(ca_handle* h, Workspace& w, Workspace::Sweep& s, const ca_sweep_call& c, cudaStream_t st) {
  const size_t K = c.K, B = w.B;
  const size_t n_tw = K * 64 * kD, n_tb = K * 64, n_eps = K * B * 192, n_noise = K * B * kD;
  PinnedSlot* slot = nullptr;
  CA_TRY(pinned_slot(h, n_tw + n_tb + n_eps + n_noise, &slot));
  float* p = slot->buf;
  memcpy(p, c.tmp_w, n_tw * sizeof(float));
  memcpy(p + n_tw, c.tmp_b, n_tb * sizeof(float));
  memcpy(p + n_tw + n_tb, c.eps, n_eps * sizeof(float));
  memcpy(p + n_tw + n_tb + n_eps, c.noise, n_noise * sizeof(float));
  CA_TRY(ca::fetch_pinned_launch(s.tmpw, p, n_tw, st));
  CA_TRY(ca::fetch_pinned_launch(s.tmpb, p + n_tw, n_tb, st));
  CA_TRY(ca::fetch_pinned_launch(s.cur_eps, p + n_tw + n_tb, n_eps, st));
  CA_TRY(ca::fetch_pinned_launch(s.cur_noise, p + n_tw + n_tb + n_eps, n_noise, st));
  h->launches += 4;
  CA_CUDA(cudaEventRecord(slot->done, st));
  return 0;
}

// The images of one call: a uniform tensor (`images`, fp32 or uint8 at model resolution) or B photographs of
// individual sizes (`list` / `hw`, HOST arrays).
struct ImagesIn {
  const void* images;
  int u8;
  const uint8_t* const* list;
  const int* hw;
};

ImagesIn images_of(const ca_forward_call& c) { return {c.images, c.images_u8, c.image_list, c.image_hw}; }

int check_images(const ImagesIn& in) {
  CA_REQUIRE((in.images != nullptr) != (in.list != nullptr), "forward: give images OR image_list");
  CA_REQUIRE(!in.list || in.hw, "forward: image_list needs image_hw");
  return 0;
}

// Eager, in front of the (possibly replayed) graph: nothing here depends on a captured address except w.patches.
int patch_rows(ca_handle* h, Workspace& w, const ImagesIn& in, cudaStream_t st) {
  static const float mean[3] = {0.485f, 0.456f, 0.406f}, stdv[3] = {0.229f, 0.224f, 0.225f};
  const void* images = in.images;
  if (in.list) {
    const size_t out_bytes = (static_cast<size_t>(w.B) * w.S * w.S * 3 + 255) & ~static_cast<size_t>(255);
    const size_t tmp_bytes = ca::resize_list_tmp_bytes(in.hw, w.B, w.S, w.S);
    if (h->resize_cap < out_bytes + tmp_bytes) {
      // cudaFree waits for the device: the previous batch's reads of the old buffer have finished
      if (h->resize_buf) CA_CUDA(cudaFree(h->resize_buf));
      h->resize_buf = nullptr;
      h->resize_cap = 0;
      CA_CUDA(cudaMalloc(&h->resize_buf, out_bytes + tmp_bytes));
      h->resize_cap = out_bytes + tmp_bytes;
    }
    int n = 0;
    CA_TRY(ca::resize_list_launch(in.list, in.hw, w.B, w.S, w.S, h->resize_buf + out_bytes, tmp_bytes, h->resize_buf, st,
                                  &n));
    h->launches += n;
    images = h->resize_buf;
  }
  if (in.u8 || in.list)
    LAUNCH(ca::preprocess_u8_launch(static_cast<const uint8_t*>(images), w.patches, w.B, w.S, mean, stdv, st));
  else
    LAUNCH(ca::patchify_f32_launch(static_cast<const float*>(images), w.patches, w.B, w.S, st));
  return 0;
}

// Run `seq` eagerly the first time a path key is seen on this workspace, capture + instantiate it the second time, replay
// the graph afterwards.
template <class F>
int run_captured(ca_handle* h, std::map<int, std::pair<cudaGraphExec_t, int>>& graphs, std::map<int, int>& seen, int key,
                 bool use_graph, cudaStream_t st, F&& seq) {
  const int calls = seen[key]++;
  auto g = graphs.find(key);
  // (the legacy default stream cannot be captured: such callers get eager launches)
  if (!use_graph || calls == 0 || st == nullptr) return seq();
  if (g == graphs.end()) {
    const int before = h->launches;
    CA_CUDA(cudaStreamBeginCapture(st, cudaStreamCaptureModeRelaxed));
    const int status = seq();
    cudaGraph_t graph = nullptr;
    const cudaError_t e = cudaStreamEndCapture(st, &graph);
    if (status != 0) {
      if (graph) cudaGraphDestroy(graph);
      return status;
    }
    CA_CUDA(e);
    cudaGraphExec_t exec = nullptr;
    const cudaError_t ei = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    CA_CUDA(ei);
    g = graphs.emplace(key, std::make_pair(exec, h->launches - before)).first;
    h->launches = before;
  }
  CA_CUDA(cudaGraphLaunch(g->second.first, st));
  h->launches += g->second.second;
  return 0;
}

template <class F>
int run_sequence(ca_handle* h, Workspace& w, int key, bool use_graph, cudaStream_t st, F&& seq) {
  return run_captured(h, w.graphs, w.seen, key, use_graph, st, static_cast<F&&>(seq));
}

// Live handles and scenes: a scene is only used while its handle lives, and a destroyed scene is never touched again.
std::mutex g_live_mu;
std::map<const ca_handle*, unsigned long long> g_live_handles;
std::set<const ca_scene*> g_live_scenes;
std::atomic<unsigned long long> g_next_handle_id{1};

int check_scene(const ca_handle* h, const ca_scene* sc) {
  std::lock_guard<std::mutex> lock(g_live_mu);
  CA_REQUIRE(h && sc, "null handle / scene");
  auto it = g_live_handles.find(h);
  CA_REQUIRE(it != g_live_handles.end(), "the handle has been destroyed");
  CA_REQUIRE(g_live_scenes.count(sc) != 0, "the scene has been destroyed");
  CA_REQUIRE(sc->handle_id == it->second, "the scene belongs to another (possibly destroyed) handle");
  return 0;
}

void drop_scene_graphs(ca_scene* sc) {
  for (auto& g : sc->graphs) cudaGraphExecDestroy(g.second.first);
  sc->graphs.clear();
  sc->seen.clear();
}

// The workspace a guide call of `sc` runs on; the scene's graphs are dropped when it is not the one they were captured on.
int scene_workspace(ca_handle* h, ca_scene* sc, Workspace** out, Tables** tb) {
  CA_TRY(get_workspace(h, sc->B, sc->S, out));
  CA_TRY(get_tables(h, sc->S / 14, tb));
  if (sc->ws_gen != (*out)->gen) {
    drop_scene_graphs(sc);
    sc->ws_gen = (*out)->gen;
  }
  return 0;
}

int check_call(const ca_handle* h, const ca_forward_call* c) {
  CA_REQUIRE(h && c, "null handle / call");
  CA_REQUIRE(c->B > 0, "forward: empty batch");
  CA_TRY(check_images(images_of(*c)));
  CA_REQUIRE(c->S >= 56 && c->S % 14 == 0 && c->S <= 1260, "forward: image side must be a multiple of 14 in [56, 1260]");
  CA_REQUIRE(c->depth && c->conf, "forward: null output");
  CA_REQUIRE(c->eps && c->noise, "forward: null CuriosityModule draws (HOST pointers, src/model.py:609,744)");
  return 0;
}

struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    cudaGetDevice(&prev);
    if (prev != dev) cudaSetDevice(dev);
    else prev = -1;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

}  // namespace

extern "C" {

int ca_create(ca_handle** out, const ca_model_weights* w, int device) {
  CA_REQUIRE(out && w, "ca_create: null argument");
  CA_TRY(ca_device_check(device));
  CA_REQUIRE(w->n_focal >= 1 && w->n_focal <= 4, "ca_create: 1..4 focal iterations are built");
  CA_REQUIRE(w->pos_embed && w->patch_w && w->cls_token && w->lnw, "ca_create: null weight");
  for (int l = 0; l < kLayers; ++l) {
    const ca_layer_weights& L = w->layer[l];
    CA_REQUIRE(w->layernorm_folded || (L.n1w && L.n1b && L.n2w && L.n2b), "ca_create: null LayerNorm weight");
  }
  DeviceGuard guard(device);
  ca_handle* h = new ca_handle();
  h->w = *w;
  h->device = device;
  h->pos_native.assign(w->pos_embed, w->pos_embed + static_cast<size_t>(1 + kNativeGrid * kNativeGrid) * kD);
  h->w.pos_embed = nullptr;
  if (cudaStreamCreateWithFlags(&h->side, cudaStreamNonBlocking) != cudaSuccess ||
      cudaEventCreateWithFlags(&h->fork, cudaEventDisableTiming) != cudaSuccess ||
      cudaEventCreateWithFlags(&h->join, cudaEventDisableTiming) != cudaSuccess) {
    delete h;
    return ca::cuda_fail(cudaGetLastError(), "ca_create: stream / event creation", __FILE__, __LINE__);
  }
  {
    std::lock_guard<std::mutex> lock(g_live_mu);
    h->id = g_next_handle_id.fetch_add(1);
    g_live_handles[h] = h->id;
  }
  *out = h;
  return 0;
}

int ca_destroy(ca_handle* h) {
  if (!h) return 0;
  {
    std::lock_guard<std::mutex> lock(g_live_mu);
    g_live_handles.erase(h);  // its scenes are refused from now on
  }
  DeviceGuard guard(h->device);
  cudaDeviceSynchronize();
  for (auto& kv : h->ws) free_workspace(kv.second);
  for (auto& kv : h->tables) {
    cudaFree(kv.second.pos);
    cudaFree(kv.second.pe);
    cudaFree(kv.second.cbias);
    for (auto& m : kv.second.masks) cudaFree(m.second);
  }
  for (auto& s : h->ring) {
    if (s.buf) cudaFreeHost(s.buf);
    if (s.done) cudaEventDestroy(s.done);
  }
  if (h->resize_buf) cudaFree(h->resize_buf);
  cudaStreamDestroy(h->side);
  cudaEventDestroy(h->fork);
  cudaEventDestroy(h->join);
  delete h;
  return 0;
}

int ca_last_launch_count(const ca_handle* h) { return h ? h->last_launches : 0; }

namespace {

int backbone(ca_handle* h, const ImagesIn& in, int B, int S, float* tokens_out, void* stream) {
  CA_REQUIRE(h && B > 0 && S >= 56 && S % 14 == 0, "ca_backbone: bad argument");
  CA_TRY(check_images(in));
  DeviceGuard guard(h->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Workspace* w = nullptr;
  Tables* tb = nullptr;
  CA_TRY(get_workspace(h, B, S, &w));
  CA_TRY(get_tables(h, S / 14, &tb));
  h->launches = 0;
  CA_TRY(patch_rows(h, *w, in, st));
  CA_TRY(run_sequence(h, *w, 0, true, st, [&]() { return backbone_layers(h, *w, *tb, st); }));
  if (tokens_out) {
    const size_t g = S / 14;
    CA_CUDA(cudaMemcpyAsync(tokens_out, w->tokens, static_cast<size_t>(B) * (g * g + 1) * kD * 4, cudaMemcpyDeviceToDevice, st));
  }
  h->last_launches = h->launches;
  return 0;
}

}  // namespace

int ca_backbone(ca_handle* h, const void* images, int images_u8, int B, int S, float* tokens_out, void* stream) {
  return backbone(h, ImagesIn{images, images_u8, nullptr, nullptr}, B, S, tokens_out, stream);
}

int ca_backbone_list(ca_handle* h, const uint8_t* const* image_list, const int* image_hw, int B, int S, float* tokens_out,
                     void* stream) {
  CA_REQUIRE(image_list, "ca_backbone_list: null image list");
  return backbone(h, ImagesIn{nullptr, 0, image_list, image_hw}, B, S, tokens_out, stream);
}

int ca_forward_guided(ca_handle* h, const ca_forward_call* c, void* stream) {
  CA_TRY(check_call(h, c));
  CA_REQUIRE(c->exif && c->camera_idx, "forward_guided: EXIF inputs are required (without them the reference falls back "
                                       "to forward(): call ca_forward)");
  CA_REQUIRE(c->tmp_w && c->tmp_b, "forward_guided: null per-call projection (HOST pointers, src/model.py:1421)");
  CA_REQUIRE((c->instruction != nullptr) != (c->mask != nullptr), "forward_guided: give an instruction OR a mask");
  CA_REQUIRE(c->attention, "forward_guided: null heat-map output");
  DeviceGuard guard(h->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int B = c->B, S = c->S, g = S / 14, N = g * g, T = N + 1;
  Workspace* wp = nullptr;
  Tables* tb = nullptr;
  CA_TRY(get_workspace(h, B, S, &wp));
  CA_TRY(get_tables(h, g, &tb));
  Workspace& w = *wp;
  h->launches = 0;
  const float* mask = c->mask;
  long long mstride = c->mask_batch_stride;
  if (c->instruction) {
    float* m = nullptr;
    CA_TRY(get_mask(tb, c->instruction, g, &m));
    mask = m;
    mstride = 0;
  }
  CA_REQUIRE(mstride == 0 || mstride == N, "forward_guided: mask batch stride must be 0 or N");
  CA_TRY(stage_host_inputs(h, w, *c, true, 1, st));
  CA_CUDA(cudaMemcpyAsync(w.mask_in, mask, static_cast<size_t>(mstride ? B : 1) * N * 4, cudaMemcpyDeviceToDevice, st));
  CA_CUDA(cudaMemcpyAsync(w.exif_in, c->exif, static_cast<size_t>(B) * 3 * 4, cudaMemcpyDeviceToDevice, st));
  CA_CUDA(cudaMemcpyAsync(w.cam_in, c->camera_idx, static_cast<size_t>(B) * 8, cudaMemcpyDeviceToDevice, st));
  CA_TRY(patch_rows(h, w, images_of(*c), st));
  int* fault = c->fault;
  const int key = 100 + (mstride ? 1 : 0);
  CA_TRY(run_sequence(h, w, key, c->use_graph != 0, st, [&]() -> int {
    CA_TRY(backbone_layers(h, w, *tb, st));
    CA_TRY(curiosity_fork(h, w, 1, w.cur_eps, w.cur_noise, w.cur_raw, w.cur_reward, st));
    float* base = nullptr;
    CA_TRY(focal_iterations(h, w, *tb, false, st, &base));
    LAUNCH(ca::guided_softmax_launch(base, w.mask_in, mstride ? N : 0, w.heat, w.argmax, B, N, 0.7f, 0.05f, st));
    LAUNCH(ca::weighted_pool_launch(w.tokens, static_cast<long long>(T) * kD, 1, w.heat, nullptr, w.pool, B, N, kD, kPoolSplits, st));
    CA_TRY(heads(h, w, true, true, fault, st));
    CA_TRY(curiosity_join(h, st));
    return 0;
  }));
  CA_CUDA(cudaMemcpyAsync(c->depth, w.depth, B * 4, cudaMemcpyDeviceToDevice, st));
  CA_CUDA(cudaMemcpyAsync(c->conf, w.conf, B * 4, cudaMemcpyDeviceToDevice, st));
  CA_CUDA(cudaMemcpyAsync(c->attention, w.heat, static_cast<size_t>(B) * N * 4, cudaMemcpyDeviceToDevice, st));
  if (c->argmax) CA_CUDA(cudaMemcpyAsync(c->argmax, w.argmax, B * 4, cudaMemcpyDeviceToDevice, st));
  h->last_launches = h->launches;
  return 0;
}

int ca_forward_guided_sweep(ca_handle* h, const ca_forward_call* c, const ca_sweep_call* sw, void* stream) {
  CA_REQUIRE(h && c && sw, "forward_guided_sweep: null handle / call / sweep");
  CA_REQUIRE(c->B > 0, "forward_guided_sweep: empty batch");
  CA_TRY(check_images(images_of(*c)));
  CA_REQUIRE(c->S >= 56 && c->S % 14 == 0 && c->S <= 1260,
             "forward_guided_sweep: image side must be a multiple of 14 in [56, 1260]");
  CA_REQUIRE(c->exif && c->camera_idx, "forward_guided_sweep: EXIF inputs are required (without them the reference falls "
                                       "back to forward(): call ca_forward)");
  CA_REQUIRE(!c->instruction && !c->mask && !c->tmp_w && !c->tmp_b && !c->eps && !c->noise && !c->depth && !c->conf &&
                 !c->attention && !c->argmax && !c->fused,
             "forward_guided_sweep: the per-call fields of ca_forward_call must be NULL (they go in ca_sweep_call)");
  const int K = sw->K;
  CA_REQUIRE(K >= 1 && K <= CA_SWEEP_MAX_K, "forward_guided_sweep: K must be in 1..CA_SWEEP_MAX_K (16)");
  CA_REQUIRE((sw->instructions != nullptr) != (sw->masks != nullptr), "forward_guided_sweep: give instructions OR masks");
  if (sw->instructions)
    for (int k = 0; k < K; ++k) CA_REQUIRE(sw->instructions[k], "forward_guided_sweep: null instruction string");
  CA_REQUIRE(sw->tmp_w && sw->tmp_b && sw->eps && sw->noise,
             "forward_guided_sweep: null per-call projections or CuriosityModule draws (HOST pointers)");
  CA_REQUIRE(sw->depth && sw->conf && sw->attention, "forward_guided_sweep: null output");
  DeviceGuard guard(h->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int B = c->B, S = c->S, g = S / 14, N = g * g, T = N + 1;
  Workspace* wp = nullptr;
  Tables* tb = nullptr;
  Workspace::Sweep* sp = nullptr;
  CA_TRY(get_workspace(h, B, S, &wp));
  CA_TRY(get_tables(h, g, &tb));
  Workspace& w = *wp;
  CA_TRY(get_sweep(w, K, &sp));
  Workspace::Sweep& s = *sp;
  h->launches = 0;
  // mask set [K, N], one row per call, shared by the batch (mask stride per image 0)
  if (sw->instructions) {
    for (int k = 0; k < K; ++k) {
      float* m = nullptr;
      CA_TRY(get_mask(tb, sw->instructions[k], g, &m));
      CA_CUDA(cudaMemcpyAsync(s.mask_in + static_cast<size_t>(k) * N, m, static_cast<size_t>(N) * 4, cudaMemcpyDeviceToDevice, st));
    }
  } else {
    CA_CUDA(cudaMemcpyAsync(s.mask_in, sw->masks, static_cast<size_t>(K) * N * 4, cudaMemcpyDeviceToDevice, st));
  }
  CA_TRY(stage_sweep_inputs(h, w, s, *sw, st));
  CA_CUDA(cudaMemcpyAsync(w.exif_in, c->exif, static_cast<size_t>(B) * 3 * 4, cudaMemcpyDeviceToDevice, st));
  CA_CUDA(cudaMemcpyAsync(w.cam_in, c->camera_idx, static_cast<size_t>(B) * 8, cudaMemcpyDeviceToDevice, st));
  CA_TRY(patch_rows(h, w, images_of(*c), st));
  int* fault = c->fault;
  CA_TRY(run_sequence(h, w, 300 + K, c->use_graph != 0, st, [&]() -> int {
    CA_TRY(backbone_layers(h, w, *tb, st));
    CA_TRY(curiosity_fork(h, w, K, s.cur_eps, s.cur_noise, s.cur_raw, s.cur_reward, st));
    float* base = nullptr;
    CA_TRY(focal_iterations(h, w, *tb, false, st, &base));  // shared by the K calls: it does not read the instruction
    LAUNCH(ca::guided_softmax_sweep_launch(base, 0, s.mask_in, N, 0, s.heat, s.argmax, K, B, N, 0.7f, 0.05f, st));
    LAUNCH(ca::weighted_pool_sweep_launch(w.tokens, static_cast<long long>(T) * kD, 1, s.heat, s.pool, K, B, N, kD,
                                          kPoolSplits, st));
    ca_heads_inputs in{};
    in.tokens = w.tokens;
    in.tokens_per_img = T;
    in.pool_partial = s.pool;
    in.pool_splits = kPoolSplits;
    in.tmp_w = s.tmpw;
    in.tmp_b = s.tmpb;
    in.exif = w.exif_in;
    in.camera_idx = w.cam_in;
    in.num_cameras = h->w.num_cameras;
    in.fault = fault;
    in.sweep_images = B;
    LAUNCH(ca::heads_launch(h->w.heads, in, s.depth, s.conf, nullptr, K * B, st));
    CA_TRY(curiosity_join(h, st));
    return 0;
  }));
  const size_t KB = static_cast<size_t>(K) * B;
  CA_CUDA(cudaMemcpyAsync(sw->depth, s.depth, KB * 4, cudaMemcpyDeviceToDevice, st));
  CA_CUDA(cudaMemcpyAsync(sw->conf, s.conf, KB * 4, cudaMemcpyDeviceToDevice, st));
  CA_CUDA(cudaMemcpyAsync(sw->attention, s.heat, KB * N * 4, cudaMemcpyDeviceToDevice, st));
  if (sw->argmax) CA_CUDA(cudaMemcpyAsync(sw->argmax, s.argmax, KB * 4, cudaMemcpyDeviceToDevice, st));
  h->last_launches = h->launches;
  return 0;
}

int ca_forward(ca_handle* h, const ca_forward_call* c, void* stream) {
  CA_TRY(check_call(h, c));
  CA_REQUIRE(c->curiosity_runs >= 1 && c->curiosity_runs <= kMaxRuns, "forward: 1..3 CuriosityModule runs");
  CA_REQUIRE((c->exif == nullptr) == (c->camera_idx == nullptr), "forward: exif and camera_idx go together");
  DeviceGuard guard(h->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int B = c->B, S = c->S, g = S / 14, N = g * g;
  Workspace* wp = nullptr;
  Tables* tb = nullptr;
  CA_TRY(get_workspace(h, B, S, &wp));
  CA_TRY(get_tables(h, g, &tb));
  Workspace& w = *wp;
  h->launches = 0;
  const bool has_exif = c->exif != nullptr && h->w.num_cameras > 0;
  const int runs = c->curiosity_runs;
  CA_TRY(stage_host_inputs(h, w, *c, false, runs, st));
  if (has_exif) {
    CA_CUDA(cudaMemcpyAsync(w.exif_in, c->exif, static_cast<size_t>(B) * 3 * 4, cudaMemcpyDeviceToDevice, st));
    CA_CUDA(cudaMemcpyAsync(w.cam_in, c->camera_idx, static_cast<size_t>(B) * 8, cudaMemcpyDeviceToDevice, st));
  }
  CA_TRY(patch_rows(h, w, images_of(*c), st));
  int* fault = c->fault;
  float* att = nullptr;
  const int key = 200 + (has_exif ? 1 : 0) + 2 * runs;
  CA_TRY(run_sequence(h, w, key, c->use_graph != 0, st, [&]() -> int {
    CA_TRY(backbone_layers(h, w, *tb, st));
    CA_TRY(curiosity_fork(h, w, runs, w.cur_eps, w.cur_noise, w.cur_raw, w.cur_reward, st));
    CA_TRY(focal_iterations(h, w, *tb, true, st, &att));
    CA_TRY(heads(h, w, false, has_exif, fault, st));
    CA_TRY(curiosity_join(h, st));
    return 0;
  }));
  att = w.attn + static_cast<size_t>(h->w.n_focal - 1) * B * N;
  CA_CUDA(cudaMemcpyAsync(c->depth, w.depth, B * 4, cudaMemcpyDeviceToDevice, st));
  CA_CUDA(cudaMemcpyAsync(c->conf, w.conf, B * 4, cudaMemcpyDeviceToDevice, st));
  if (c->attention) CA_CUDA(cudaMemcpyAsync(c->attention, att, static_cast<size_t>(B) * N * 4, cudaMemcpyDeviceToDevice, st));
  if (c->fused) CA_CUDA(cudaMemcpyAsync(c->fused, w.fused, static_cast<size_t>(B) * 192 * 4, cudaMemcpyDeviceToDevice, st));
  h->last_launches = h->launches;
  return 0;
}


int ca_encode(ca_handle* h, const ca_forward_call* c, ca_scene** out, void* stream) {
  CA_REQUIRE(h && c && out, "encode: null handle / call / out");
  {
    std::lock_guard<std::mutex> lock(g_live_mu);
    CA_REQUIRE(g_live_handles.count(h) != 0, "encode: the handle has been destroyed");
  }
  CA_REQUIRE(c->B > 0, "encode: empty batch");
  CA_TRY(check_images(images_of(*c)));
  CA_REQUIRE(c->S >= 56 && c->S % 14 == 0 && c->S <= 1260, "encode: image side must be a multiple of 14 in [56, 1260]");
  CA_REQUIRE(c->exif && c->camera_idx, "encode: EXIF inputs are required (without them the reference falls back to "
                                       "forward(): call ca_forward)");
  CA_REQUIRE(!c->instruction && !c->mask && !c->tmp_w && !c->tmp_b && !c->eps && !c->noise && !c->depth && !c->conf &&
                 !c->attention && !c->argmax && !c->fused,
             "encode: the per-call fields of ca_forward_call must be NULL (they go in ca_guide_call / ca_sweep_call)");
  DeviceGuard guard(h->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int B = c->B, S = c->S, g = S / 14, N = g * g, T = N + 1;
  Workspace* wp = nullptr;
  Tables* tb = nullptr;
  CA_TRY(get_workspace(h, B, S, &wp));
  CA_TRY(get_tables(h, g, &tb));
  Workspace& w = *wp;
  h->launches = 0;
  CA_TRY(patch_rows(h, w, images_of(*c), st));
  float* base = nullptr;
  CA_TRY(run_sequence(h, w, 400, c->use_graph != 0, st, [&]() -> int {
    CA_TRY(backbone_layers(h, w, *tb, st));
    return focal_iterations(h, w, *tb, false, st, &base);
  }));
  base = w.attn + static_cast<size_t>(h->w.n_focal - 1) * B * N;
  const size_t tok = static_cast<size_t>(B) * T * kD * 4, bn = static_cast<size_t>(B) * N * 4;
  const size_t o_base = (tok + 255) & ~size_t(255), o_exif = o_base + ((bn + 255) & ~size_t(255));
  const size_t o_cam = o_exif + 256 * ((static_cast<size_t>(B) * 12 + 255) / 256);
  ca_scene* sc = new ca_scene();
  if (cudaMalloc(&sc->arena, o_cam + static_cast<size_t>(B) * 8) != cudaSuccess) {
    delete sc;
    return ca::cuda_fail(cudaGetLastError(), "encode: scene allocation", __FILE__, __LINE__);
  }
  char* a = static_cast<char*>(sc->arena);
  sc->tokens = reinterpret_cast<float*>(a);
  sc->base = reinterpret_cast<float*>(a + o_base);
  sc->exif = reinterpret_cast<float*>(a + o_exif);
  sc->cam = reinterpret_cast<long long*>(a + o_cam);
  sc->handle_id = h->id;
  sc->device = h->device;
  sc->B = B;
  sc->S = S;
  sc->fault = c->fault;
  sc->use_graph = c->use_graph != 0;
  const int status = [&]() -> int {
    CA_CUDA(cudaMemcpyAsync(sc->tokens, w.tokens, tok, cudaMemcpyDeviceToDevice, st));
    CA_CUDA(cudaMemcpyAsync(sc->base, base, bn, cudaMemcpyDeviceToDevice, st));
    CA_CUDA(cudaMemcpyAsync(sc->exif, c->exif, static_cast<size_t>(B) * 12, cudaMemcpyDeviceToDevice, st));
    CA_CUDA(cudaMemcpyAsync(sc->cam, c->camera_idx, static_cast<size_t>(B) * 8, cudaMemcpyDeviceToDevice, st));
    return 0;
  }();
  if (status != 0) {
    cudaFree(sc->arena);
    delete sc;
    return status;
  }
  {
    std::lock_guard<std::mutex> lock(g_live_mu);
    g_live_scenes.insert(sc);
  }
  h->last_launches = h->launches;
  *out = sc;
  return 0;
}

int ca_guide(ca_handle* h, ca_scene* sc, const ca_guide_call* c, void* stream) {
  CA_TRY(check_scene(h, sc));
  CA_REQUIRE(c, "guide: null call");
  CA_REQUIRE((c->instruction != nullptr) != (c->mask != nullptr), "guide: give an instruction OR a mask");
  CA_REQUIRE(c->tmp_w && c->tmp_b && c->eps && c->noise,
             "guide: null per-call projection or CuriosityModule draws (HOST pointers, src/model.py:609,744,1421)");
  CA_REQUIRE(c->depth && c->conf && c->attention, "guide: null output");
  DeviceGuard guard(h->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int B = sc->B, g = sc->S / 14, N = g * g, T = N + 1;
  Workspace* wp = nullptr;
  Tables* tb = nullptr;
  CA_TRY(scene_workspace(h, sc, &wp, &tb));
  Workspace& w = *wp;
  h->launches = 0;
  const float* mask = c->mask;
  long long mstride = c->mask_batch_stride;
  if (c->instruction) {
    float* m = nullptr;
    CA_TRY(get_mask(tb, c->instruction, g, &m));
    mask = m;
    mstride = 0;
  }
  CA_REQUIRE(mstride == 0 || mstride == N, "guide: mask batch stride must be 0 or N");
  ca_forward_call staged{};
  staged.tmp_w = c->tmp_w;
  staged.tmp_b = c->tmp_b;
  staged.eps = c->eps;
  staged.noise = c->noise;
  CA_TRY(stage_host_inputs(h, w, staged, true, 1, st));
  CA_CUDA(cudaMemcpyAsync(w.mask_in, mask, static_cast<size_t>(mstride ? B : 1) * N * 4, cudaMemcpyDeviceToDevice, st));
  CA_TRY(run_captured(h, sc->graphs, sc->seen, 1 + (mstride ? 1 : 0), sc->use_graph, st, [&]() -> int {
    CA_TRY(curiosity_fork(h, w, 1, w.cur_eps, w.cur_noise, w.cur_raw, w.cur_reward, st, sc->tokens));
    ca_heads_inputs in{};
    in.tokens = sc->tokens;
    in.tokens_per_img = T;
    in.pool_partial = w.pool;
    in.pool_splits = kPoolSplits;
    in.tmp_w = w.tmpw;
    in.tmp_b = w.tmpb;
    in.exif = sc->exif;
    in.camera_idx = sc->cam;
    in.num_cameras = h->w.num_cameras;
    in.fault = sc->fault;
    if (B <= CA_GUIDE_TAIL_MAX_B) {
      LAUNCH(ca::guide_tail_launch(h->w.heads, in, sc->base, w.mask_in, mstride ? N : 0, w.heat, w.argmax, reinterpret_cast<unsigned int*>(w.tail_ticket),
                                   w.depth, w.conf, B, N, 0.7f, 0.05f, st));
    } else {
      LAUNCH(ca::guided_softmax_launch(sc->base, w.mask_in, mstride ? N : 0, w.heat, w.argmax, B, N, 0.7f, 0.05f, st));
      LAUNCH(ca::weighted_pool_launch(sc->tokens, static_cast<long long>(T) * kD, 1, w.heat, nullptr, w.pool, B, N, kD,
                                      kPoolSplits, st));
      LAUNCH(ca::heads_launch(h->w.heads, in, w.depth, w.conf, nullptr, B, st));
    }
    return curiosity_join(h, st);
  }));
  CA_CUDA(cudaMemcpyAsync(c->depth, w.depth, B * 4, cudaMemcpyDeviceToDevice, st));
  CA_CUDA(cudaMemcpyAsync(c->conf, w.conf, B * 4, cudaMemcpyDeviceToDevice, st));
  CA_CUDA(cudaMemcpyAsync(c->attention, w.heat, static_cast<size_t>(B) * N * 4, cudaMemcpyDeviceToDevice, st));
  if (c->argmax) CA_CUDA(cudaMemcpyAsync(c->argmax, w.argmax, B * 4, cudaMemcpyDeviceToDevice, st));
  h->last_launches = h->launches;
  return 0;
}

int ca_guide_sweep(ca_handle* h, ca_scene* sc, const ca_sweep_call* sw, void* stream) {
  CA_TRY(check_scene(h, sc));
  CA_REQUIRE(sw, "guide_sweep: null sweep");
  const int K = sw->K;
  CA_REQUIRE(K >= 1 && K <= CA_SWEEP_MAX_K, "guide_sweep: K must be in 1..CA_SWEEP_MAX_K (16)");
  CA_REQUIRE((sw->instructions != nullptr) != (sw->masks != nullptr), "guide_sweep: give instructions OR masks");
  if (sw->instructions)
    for (int k = 0; k < K; ++k) CA_REQUIRE(sw->instructions[k], "guide_sweep: null instruction string");
  CA_REQUIRE(sw->tmp_w && sw->tmp_b && sw->eps && sw->noise,
             "guide_sweep: null per-call projections or CuriosityModule draws (HOST pointers)");
  CA_REQUIRE(sw->depth && sw->conf && sw->attention, "guide_sweep: null output");
  DeviceGuard guard(h->device);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int B = sc->B, g = sc->S / 14, N = g * g, T = N + 1;
  Workspace* wp = nullptr;
  Tables* tb = nullptr;
  CA_TRY(scene_workspace(h, sc, &wp, &tb));
  Workspace& w = *wp;
  Workspace::Sweep* sp = nullptr;
  CA_TRY(get_sweep(w, K, &sp));
  Workspace::Sweep& s = *sp;
  h->launches = 0;
  if (sw->instructions) {
    for (int k = 0; k < K; ++k) {
      float* m = nullptr;
      CA_TRY(get_mask(tb, sw->instructions[k], g, &m));
      CA_CUDA(cudaMemcpyAsync(s.mask_in + static_cast<size_t>(k) * N, m, static_cast<size_t>(N) * 4, cudaMemcpyDeviceToDevice, st));
    }
  } else {
    CA_CUDA(cudaMemcpyAsync(s.mask_in, sw->masks, static_cast<size_t>(K) * N * 4, cudaMemcpyDeviceToDevice, st));
  }
  CA_TRY(stage_sweep_inputs(h, w, s, *sw, st));
  CA_TRY(run_captured(h, sc->graphs, sc->seen, 100 + K, sc->use_graph, st, [&]() -> int {
    CA_TRY(curiosity_fork(h, w, K, s.cur_eps, s.cur_noise, s.cur_raw, s.cur_reward, st, sc->tokens));
    LAUNCH(ca::guided_softmax_sweep_launch(sc->base, 0, s.mask_in, N, 0, s.heat, s.argmax, K, B, N, 0.7f, 0.05f, st));
    LAUNCH(ca::weighted_pool_sweep_launch(sc->tokens, static_cast<long long>(T) * kD, 1, s.heat, s.pool, K, B, N, kD,
                                          kPoolSplits, st));
    ca_heads_inputs in{};
    in.tokens = sc->tokens;
    in.tokens_per_img = T;
    in.pool_partial = s.pool;
    in.pool_splits = kPoolSplits;
    in.tmp_w = s.tmpw;
    in.tmp_b = s.tmpb;
    in.exif = sc->exif;
    in.camera_idx = sc->cam;
    in.num_cameras = h->w.num_cameras;
    in.fault = sc->fault;
    in.sweep_images = B;
    LAUNCH(ca::heads_launch(h->w.heads, in, s.depth, s.conf, nullptr, K * B, st));
    return curiosity_join(h, st);
  }));
  const size_t KB = static_cast<size_t>(K) * B;
  CA_CUDA(cudaMemcpyAsync(sw->depth, s.depth, KB * 4, cudaMemcpyDeviceToDevice, st));
  CA_CUDA(cudaMemcpyAsync(sw->conf, s.conf, KB * 4, cudaMemcpyDeviceToDevice, st));
  CA_CUDA(cudaMemcpyAsync(sw->attention, s.heat, KB * N * 4, cudaMemcpyDeviceToDevice, st));
  if (sw->argmax) CA_CUDA(cudaMemcpyAsync(sw->argmax, s.argmax, KB * 4, cudaMemcpyDeviceToDevice, st));
  h->last_launches = h->launches;
  return 0;
}

int ca_scene_destroy(ca_scene* sc) {
  if (!sc) return 0;
  {
    std::lock_guard<std::mutex> lock(g_live_mu);
    CA_REQUIRE(g_live_scenes.count(sc) != 0, "scene_destroy: not a live scene (already destroyed?)");
    g_live_scenes.erase(sc);
  }
  DeviceGuard guard(sc->device);
  drop_scene_graphs(sc);
  cudaFree(sc->arena);  // waits for the work that still reads it
  delete sc;
  return 0;
}

}  // extern "C"
