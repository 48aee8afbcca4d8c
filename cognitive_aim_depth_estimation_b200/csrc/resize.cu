// Exact-Pillow antialiased bilinear resize on the GPU: the `Resize((S, S))` of demo.py:162-163 (torchvision on a PIL
// image = PIL.Image.resize(..., BILINEAR) = Pillow's ImagingResample with the triangle filter), batched.
//
// Pillow's algorithm is integer after the coefficient tables: per output column a window [xmin, xmin + n) of source
// columns with 22-bit fixed-point weights (double-precision triangle filter, normalised, rounded half away from zero),
// accumulate from 1 << 21, shift right by 22, clamp to 8 bits; horizontal pass first into a uint8 intermediate (only
// the source rows the vertical pass will read), then the vertical pass.  A pass runs only on an axis whose size changes;
// with neither, the image is copied.  The tables are built on the host in double exactly as Resample.c builds them and
// cached per (source size, target size); the two passes are bit-exact against PIL
// (tests/test_rowops_gpu.py::test_resize_matches_pillow, tests/test_ragged_gpu.py).
//
// A batch may be ragged: every image carries its own source size, tables and offsets in a descriptor, and each pass is
// ONE launch over the whole batch (up to CA_RESIZE_LIST_CHUNK images), its flat block index mapped to (image, rows)
// through the descriptors' block offsets.  The descriptors travel by value as a __grid_constant__ kernel parameter, so
// nothing is copied host-to-device on the stream.  A uniform batch is the case where every descriptor is alike.
#include "common.cuh"
#include "host.h"
#include "resize.cuh"

#include <math.h>

#include <algorithm>
#include <map>
#include <memory>
#include <mutex>
#include <vector>

namespace ca {
namespace {

constexpr int kPrecisionBits = 32 - 8 - 2;
constexpr int kRowsPerCta = 4;     // source rows the horizontal pass stages per CTA: each tap's coefficient serves 4 rows
constexpr int kHThreads = 128;
constexpr int kVThreads = 256;
// shared memory of the horizontal pass: kRowsPerCta rows of up to kMaxResizeSide pixels, 16-byte aligned, plus the
// misalignment of each row's start
constexpr size_t kMaxSmemPitch = static_cast<size_t>(kMaxResizeSide) * 3 + 16;
static_assert(kRowsPerCta * kMaxSmemPitch <= 227 * 1024, "horizontal pass staging exceeds shared memory");

struct AxisTable {
  int ksize = 0;
  int first = 0;  // first source index any output reads
  int last = 0;   // one past the last source index any output reads
  int* d_xmin = nullptr;
  int* d_cnt = nullptr;
  int* d_kk = nullptr;
};

// Resample.c precompute_coeffs + normalize_coeffs_8bpc, triangle filter (support 1.0), box = the whole axis.
int build_axis_table(int in_size, int out_size, AxisTable* t) {
  const double scale = static_cast<double>(in_size) / out_size;
  const double filterscale = scale < 1.0 ? 1.0 : scale;
  const double support = 1.0 * filterscale;
  const int ksize = static_cast<int>(ceil(support)) * 2 + 1;
  std::vector<int> xmin(out_size), cnt(out_size), kk(static_cast<size_t>(out_size) * ksize, 0);
  std::vector<double> w(ksize);
  const double ss = 1.0 / filterscale;
  for (int xx = 0; xx < out_size; ++xx) {
    const double center = (xx + 0.5) * scale;
    int lo = static_cast<int>(center - support + 0.5);
    if (lo < 0) lo = 0;
    int hi = static_cast<int>(center + support + 0.5);
    if (hi > in_size) hi = in_size;
    const int n = hi - lo;
    double ww = 0.0;
    for (int x = 0; x < n; ++x) {
      double a = (x + lo - center + 0.5) * ss;
      if (a < 0.0) a = -a;
      w[x] = a < 1.0 ? 1.0 - a : 0.0;
      ww += w[x];
    }
    for (int x = 0; x < n; ++x) {
      if (ww != 0.0) w[x] /= ww;
      kk[static_cast<size_t>(xx) * ksize + x] = w[x] < 0 ? static_cast<int>(-0.5 + w[x] * (1 << kPrecisionBits))
                                                          : static_cast<int>(0.5 + w[x] * (1 << kPrecisionBits));
    }
    xmin[xx] = lo;
    cnt[xx] = n;
  }
  t->ksize = ksize;
  t->first = xmin[0];
  t->last = xmin[out_size - 1] + cnt[out_size - 1];
  CA_CUDA(cudaMalloc(&t->d_xmin, out_size * sizeof(int)));
  CA_CUDA(cudaMalloc(&t->d_cnt, out_size * sizeof(int)));
  CA_CUDA(cudaMalloc(&t->d_kk, kk.size() * sizeof(int)));
  CA_CUDA(cudaMemcpy(t->d_xmin, xmin.data(), out_size * sizeof(int), cudaMemcpyHostToDevice));
  CA_CUDA(cudaMemcpy(t->d_cnt, cnt.data(), out_size * sizeof(int), cudaMemcpyHostToDevice));
  CA_CUDA(cudaMemcpy(t->d_kk, kk.data(), kk.size() * sizeof(int), cudaMemcpyHostToDevice));
  return 0;
}

int axis_table(int in_size, int out_size, const AxisTable** out) {
  static std::mutex mu;
  static std::map<std::tuple<int, int, int>, AxisTable> cache;  // (device, in, out)
  int dev = 0;
  CA_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(mu);
  auto key = std::make_tuple(dev, in_size, out_size);
  auto it = cache.find(key);
  if (it == cache.end()) {
    AxisTable t;
    CA_TRY(build_axis_table(in_size, out_size, &t));
    it = cache.emplace(key, t).first;
  }
  *out = &it->second;
  return 0;
}

// One image of a batch.  The horizontal pass covers source rows [row0, row0 + hrows) in ceil(hrows / kRowsPerCta)
// blocks from hblock0; the vertical pass covers the out_h output rows in out_h blocks from vblock0 (none when the
// height does not change).
struct ResizeImage {
  const uint8_t* src;   // uint8 [H0, W0, 3]
  uint8_t* hdst;        // horizontal pass output [hrows, out_w, 3]: the temporary, or the output when only W changes
  const uint8_t* vsrc;  // vertical pass input, row vrow0 first: the temporary, or the source when only H changes
  uint8_t* out;         // uint8 [out_h, out_w, 3]
  const int *hx, *hc, *hk;  // horizontal table: window start, length, coefficients [out_w, hks]
  const int *vy, *vc, *vk;  // vertical table [out_h, vks]
  int hks, vks;
  int W0, row0, hrows, vrow0;
  int hblock0, vblock0;
};

struct ResizeBatch {
  int n, out_w, smem_pitch;
  int hblocks, vblocks;
  ResizeImage im[CA_RESIZE_LIST_CHUNK];
};
static_assert(sizeof(ResizeBatch) <= 32764, "resize descriptors exceed the kernel parameter space");

// the image whose block range holds `b`: the last descriptor with block0 <= b (images without blocks in this pass share
// their block0 with the next image, which comes later and therefore wins)
template <bool kH>
__device__ __forceinline__ int image_of_block(const ResizeBatch& p, int b) {
  int lo = 0, hi = p.n;  // upper bound of b in the block offsets
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    const int b0 = kH ? p.im[mid].hblock0 : p.im[mid].vblock0;
    if (b0 <= b) lo = mid + 1;
    else hi = mid;
  }
  return lo - 1;
}

__device__ __forceinline__ uint8_t clip8(int v) {
  v >>= kPrecisionBits;
  return static_cast<uint8_t>(v < 0 ? 0 : (v > 255 ? 255 : v));
}

// dst[r, xx, :] = sum_j src[row0 + r, xmin[xx] + j, :] * kk[xx, j]     (3 interleaved channels)
// One CTA stages kRowsPerCta source rows in shared memory with 16-byte loads; each thread then produces output columns
// of all staged rows, so every coefficient it loads serves kRowsPerCta rows.
__global__ void __launch_bounds__(kHThreads) resize_h_kernel(const __grid_constant__ ResizeBatch p) {
  griddep_sync();  // PDL: nothing before this line reads or writes global memory
  extern __shared__ uint4 smem_v[];
  uint8_t* smem = reinterpret_cast<uint8_t*>(smem_v);
  const int b = blockIdx.x;
  const ResizeImage& im = p.im[image_of_block<true>(p, b)];
  const int r0 = (b - im.hblock0) * kRowsPerCta;
  const int nr = min(kRowsPerCta, im.hrows - r0);
  const int row_bytes = im.W0 * 3;
  const uint8_t* srow[kRowsPerCta];
#pragma unroll
  for (int r = 0; r < kRowsPerCta; ++r) {
    const uint8_t* g = im.src + (static_cast<size_t>(im.row0 + r0 + min(r, nr - 1))) * row_bytes;
    const int mis = static_cast<int>(reinterpret_cast<uintptr_t>(g) & 15);
    uint8_t* s = smem + r * p.smem_pitch + mis;  // s[k] = g[k]; s and g share their alignment modulo 16
    srow[r] = s;
    if (r >= nr) continue;
    const int head = min((16 - mis) & 15, row_bytes);
    const int nv = (row_bytes - head) >> 4;
    const uint4* gv = reinterpret_cast<const uint4*>(g + head);
    uint4* sv = reinterpret_cast<uint4*>(s + head);
    for (int k = threadIdx.x; k < nv; k += kHThreads) sv[k] = __ldcs(gv + k);  // the source is read once: stream it
    const int tail = head + nv * 16;
    if (static_cast<int>(threadIdx.x) < head) s[threadIdx.x] = g[threadIdx.x];
    if (tail + static_cast<int>(threadIdx.x) < row_bytes) s[tail + threadIdx.x] = g[tail + threadIdx.x];
  }
  __syncthreads();
  const int out_w = p.out_w;
  for (int xx = threadIdx.x; xx < out_w; xx += kHThreads) {
    const int x0 = 3 * __ldg(im.hx + xx);
    const int n = __ldg(im.hc + xx);
    const int* k = im.hk + static_cast<size_t>(xx) * im.hks;
    int a[kRowsPerCta][3];
#pragma unroll
    for (int r = 0; r < kRowsPerCta; ++r) a[r][0] = a[r][1] = a[r][2] = 1 << (kPrecisionBits - 1);
    for (int j = 0; j < n; ++j) {
      const int c = __ldg(k + j);
#pragma unroll
      for (int r = 0; r < kRowsPerCta; ++r) {
        const uint8_t* s = srow[r] + x0 + 3 * j;
        a[r][0] += s[0] * c;
        a[r][1] += s[1] * c;
        a[r][2] += s[2] * c;
      }
    }
#pragma unroll
    for (int r = 0; r < kRowsPerCta; ++r) {
      if (r >= nr) break;
      uint8_t* d = im.hdst + (static_cast<size_t>(r0 + r) * out_w + xx) * 3;
      d[0] = clip8(a[r][0]);
      d[1] = clip8(a[r][1]);
      d[2] = clip8(a[r][2]);
    }
  }
}

// out[yy, e] = sum_j vsrc[ymin[yy] - vrow0 + j, e] * kk[yy, j]   over e in [0, 3 * out_w) (channels interleaved)
// One CTA per output row: its window and coefficients are shared by the whole CTA.
__global__ void __launch_bounds__(kVThreads) resize_v_kernel(const __grid_constant__ ResizeBatch p) {
  griddep_sync();  // PDL: nothing before this line reads or writes global memory
  const int b = blockIdx.x;
  const ResizeImage& im = p.im[image_of_block<false>(p, b)];
  const int yy = b - im.vblock0;
  const int row_elems = p.out_w * 3;
  const uint8_t* s = im.vsrc + static_cast<size_t>(__ldg(im.vy + yy) - im.vrow0) * row_elems;
  const int* k = im.vk + static_cast<size_t>(yy) * im.vks;
  const int n = __ldg(im.vc + yy);
  uint8_t* d = im.out + static_cast<size_t>(yy) * row_elems;
  for (int e = threadIdx.x; e < row_elems; e += kVThreads) {
    int a = 1 << (kPrecisionBits - 1);
    for (int j = 0; j < n; ++j) a += s[static_cast<size_t>(j) * row_elems + e] * __ldg(k + j);
    d[e] = clip8(a);
  }
}

size_t two_pass_tmp_bytes(int H0, int out_w) { return static_cast<size_t>(H0) * out_w * 3; }

}  // namespace

size_t resize_tmp_bytes(int B, int H0, int W0, int out_h, int out_w) {
  if (H0 == out_h || W0 == out_w) return 0;
  return static_cast<size_t>(B) * two_pass_tmp_bytes(H0, out_w);  // upper bound (the horizontal pass may skip unread rows)
}

size_t resize_list_tmp_bytes(const int* h_hw, int B, int out_h, int out_w) {
  if (!h_hw || B <= 0) return 0;
  size_t total = 0;
  for (int i = 0; i < B; ++i)
    if (h_hw[2 * i] != out_h && h_hw[2 * i + 1] != out_w) total += two_pass_tmp_bytes(h_hw[2 * i], out_w);
  return total;
}

int resize_list_launch(const uint8_t* const* h_images, const int* h_hw, int B, int out_h, int out_w, uint8_t* tmp,
                       size_t tmp_bytes, uint8_t* out, cudaStream_t stream, int* launches) {
  CA_REQUIRE(h_images && h_hw && out, "resize: null pointer");
  CA_REQUIRE(B > 0 && out_h > 0 && out_w > 0, "resize: non-positive dimension");
  CA_REQUIRE(out_h <= kMaxResizeSide && out_w <= kMaxResizeSide, "resize: target side above CA_RESIZE_MAX_SIDE (16384)");
  for (int i = 0; i < B; ++i) {
    CA_REQUIRE(h_images[i], "resize: null image pointer");
    CA_REQUIRE(h_hw[2 * i] > 0 && h_hw[2 * i + 1] > 0, "resize: non-positive source dimension");
    CA_REQUIRE(h_hw[2 * i] <= kMaxResizeSide && h_hw[2 * i + 1] <= kMaxResizeSide,
               "resize: source side above CA_RESIZE_MAX_SIDE (16384)");
  }
  CA_REQUIRE(tmp_bytes >= resize_list_tmp_bytes(h_hw, B, out_h, out_w), "resize: temporary buffer too small");
  CA_REQUIRE(tmp || resize_list_tmp_bytes(h_hw, B, out_h, out_w) == 0, "resize: a two-pass resize needs the temporary buffer");
  static PerDeviceOnce configured;
  CA_TRY(configured.run([&]() -> int {
    CA_CUDA(cudaFuncSetAttribute(resize_h_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 static_cast<int>(kRowsPerCta * kMaxSmemPitch)));
    return 0;
  }));
  const size_t out_bytes = static_cast<size_t>(out_h) * out_w * 3;
  auto batch = std::make_unique<ResizeBatch>();
  size_t tmp_off = 0;
  int n_launches = 0;
  for (int c0 = 0; c0 < B; c0 += CA_RESIZE_LIST_CHUNK) {
    ResizeBatch& p = *batch;
    p = ResizeBatch{};
    p.out_w = out_w;
    int max_row_bytes = 0;
    for (int i = c0; i < B && i < c0 + CA_RESIZE_LIST_CHUNK; ++i) {
      const int H0 = h_hw[2 * i], W0 = h_hw[2 * i + 1];
      uint8_t* dst = out + static_cast<size_t>(i) * out_bytes;
      const bool need_h = W0 != out_w, need_v = H0 != out_h;
      if (!need_h && !need_v) {  // Pillow returns a copy
        CA_CUDA(cudaMemcpyAsync(dst, h_images[i], out_bytes, cudaMemcpyDeviceToDevice, stream));
        continue;
      }
      const AxisTable *th = nullptr, *tv = nullptr;
      if (need_h) CA_TRY(axis_table(W0, out_w, &th));
      if (need_v) CA_TRY(axis_table(H0, out_h, &tv));
      ResizeImage& d = p.im[p.n++];
      d.src = h_images[i];
      d.out = dst;
      d.W0 = W0;
      d.hblock0 = p.hblocks;
      d.vblock0 = p.vblocks;
      if (need_h) {
        d.hx = th->d_xmin;
        d.hc = th->d_cnt;
        d.hk = th->d_kk;
        d.hks = th->ksize;
        d.row0 = need_v ? tv->first : 0;
        d.hrows = need_v ? tv->last - tv->first : H0;
        if (need_v) {
          d.hdst = tmp + tmp_off;
          tmp_off += two_pass_tmp_bytes(H0, out_w);
        } else {
          d.hdst = dst;
        }
        p.hblocks += (d.hrows + kRowsPerCta - 1) / kRowsPerCta;
        max_row_bytes = std::max(max_row_bytes, W0 * 3);
      }
      if (need_v) {
        d.vy = tv->d_xmin;
        d.vc = tv->d_cnt;
        d.vk = tv->d_kk;
        d.vks = tv->ksize;
        d.vsrc = need_h ? d.hdst : d.src;
        d.vrow0 = need_h ? d.row0 : 0;
        p.vblocks += out_h;
      }
    }
    p.smem_pitch = ((max_row_bytes + 15) & ~15) + 16;
    if (p.hblocks > 0) {
      CA_TRY(launch_kernel(resize_h_kernel, dim3(p.hblocks), dim3(kHThreads),
                           static_cast<size_t>(kRowsPerCta) * p.smem_pitch, stream, p));
      CA_CUDA(cudaGetLastError());
      ++n_launches;
    }
    if (p.vblocks > 0) {
      CA_TRY(launch_kernel(resize_v_kernel, dim3(p.vblocks), dim3(kVThreads), 0, stream, p));
      CA_CUDA(cudaGetLastError());
      ++n_launches;
    }
  }
  if (launches) *launches = n_launches;
  return 0;
}

int resize_u8_launch(const uint8_t* src, int B, int H0, int W0, int out_h, int out_w, uint8_t* tmp, uint8_t* out,
                     cudaStream_t stream) {
  CA_REQUIRE(src && out, "resize: null pointer");
  CA_REQUIRE(B > 0 && H0 > 0 && W0 > 0 && out_h > 0 && out_w > 0, "resize: non-positive dimension");
  const size_t img_bytes = static_cast<size_t>(H0) * W0 * 3;
  std::vector<const uint8_t*> images(B);
  std::vector<int> hw(2 * static_cast<size_t>(B));
  for (int b = 0; b < B; ++b) {
    images[b] = src + b * img_bytes;
    hw[2 * b] = H0;
    hw[2 * b + 1] = W0;
  }
  return resize_list_launch(images.data(), hw.data(), B, out_h, out_w, tmp, resize_tmp_bytes(B, H0, W0, out_h, out_w),
                            out, stream, nullptr);
}

}  // namespace ca
