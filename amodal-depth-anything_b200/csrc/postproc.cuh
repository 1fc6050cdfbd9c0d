// Device-side pre/post-processing of the reference's single-image inference (infer.py:16-28, 72-103; SURVEY.md section 8
// row f2). In the reference these steps bounce through the host (cv2.resize, depth_raw.cpu() -> normalise -> .cuda(),
// pred.cpu() -> numpy blend -> cv2.blur); here they are small bandwidth kernels on the forward's stream. All fp32 except
// the uint8 resize. Every kernel runs over a batch: image b is blockIdx.y. Images of different sizes are read from one
// packed uint8 buffer through a device table of ada_img_desc rows; the single-image entry points launch the same kernels
// with one image and no table.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

#include "../../include/amodal_b200.h"

namespace ada {

// Geometry of image blockIdx.y: its row of the descriptor table, or, without a table (the single-image entry points),
// the one image at src of H0 x W0.
__device__ __forceinline__ ada_img_desc image_desc(const ada_img_desc* __restrict__ table, int H0, int W0) {
  if (table) return table[blockIdx.y];
  return ada_img_desc{0, H0, W0};
}

// ATen nearest (F.interpolate default / torchvision Resize(NEAREST), infer.py:85-87,97-100): src = min(floor(dst * in/out), in-1)
__device__ __forceinline__ int nearest_src(int dst, float scale, int in) {
  return min(static_cast<int>(floorf(static_cast<float>(dst) * scale)), in - 1);
}

// cv2.resize(img, (W, H)) with INTER_LINEAR on uint8 HWC, 3 channels (infer.py:17), bit-exact. Source coordinate and
// 11-bit coefficients of output index d along an axis of `src` -> `dst` samples, as OpenCV computes them: the coordinate
// in double rounded to float, the fraction in float, each coefficient rounded half to even on its own. Explicit _rn
// intrinsics keep the compiler from contracting these into FMAs, which would round differently.
__device__ __forceinline__ void linear_coeff(int d, int dst, int src, int& s, int& a0, int& a1) {
  const double scale = __ddiv_rn(1.0, __ddiv_rn(static_cast<double>(dst), static_cast<double>(src)));
  float f = __double2float_rn(__dadd_rn(__dmul_rn(__dadd_rn(static_cast<double>(d), 0.5), scale), -0.5));
  const float fs = floorf(f);
  s = static_cast<int>(fs);
  f = __fsub_rn(f, fs);
  a0 = __float2int_rn(__fmul_rn(__fsub_rn(1.0f, f), 2048.0f));
  a1 = __float2int_rn(__fmul_rn(f, 2048.0f));
}
// One thread per output pixel of image blockIdx.y; out is [B, H, W, 3]. Along x the border resets the fraction; along y
// it does not, only the two source rows are clamped (OpenCV's vertical pass clamps row pointers, not coefficients).
// OpenCV takes its INTER_AREA fast path, (a + b + c + d + 2) >> 2, when the image is exactly 2H x 2W; this arithmetic
// gives the same bits there (all four coefficients are 1024, so each vertical term is exactly a + b).
__global__ void __launch_bounds__(256)
resize_linear_kernel(const uint8_t* __restrict__ src, const ada_img_desc* __restrict__ table, uint8_t* __restrict__ out,
                     int H, int W) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= H * W) return;
  const int y = i / W, x = i - y * W;
  const ada_img_desc g = table[blockIdx.y];
  const int H0 = static_cast<int>(g.H0), W0 = static_cast<int>(g.W0);
  const uint8_t* img = src + g.offset;
  uint8_t* o = out + (static_cast<long long>(blockIdx.y) * H * W + i) * 3;
  int sx, a0, a1, sy, b0, b1;
  linear_coeff(x, W, W0, sx, a0, a1);
  linear_coeff(y, H, H0, sy, b0, b1);
  if (sx < 0 || sx >= W0 - 1) {
    sx = sx < 0 ? 0 : W0 - 1;
    a0 = 2048;
    a1 = 0;
  }
  const int sx1 = min(sx + 1, W0 - 1);
  const uint8_t* r0 = img + static_cast<long long>(min(max(sy, 0), H0 - 1)) * W0 * 3;
  const uint8_t* r1 = img + static_cast<long long>(min(max(sy + 1, 0), H0 - 1)) * W0 * 3;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const int S0 = r0[sx * 3 + c] * a0 + r0[sx1 * 3 + c] * a1;
    const int S1 = r1[sx * 3 + c] * a0 + r1[sx1 * 3 + c] * a1;
    o[c] = static_cast<uint8_t>((((b0 * (S0 >> 4)) >> 16) + ((b1 * (S1 >> 4)) >> 16) + 2) >> 2);
  }
}

// DepthAnythingV2.image2tensor (depth_anything_v2_raw/dpt.py:186-222), bit-exact: cvtColor(BGR -> RGB) / 255.0, then
// cv2.resize(..., INTER_CUBIC) of that float64 image, then (x - mean) / std in float64, then astype(float32). OpenCV's
// float64 cubic path computes the source coordinate as linear_coeff does, the four coefficients in float (A = -0.75, each
// operation rounded on its own, the last one 1 - c0 - c1 - c2) and every sum in double, left to right, with the float
// coefficients widened. Out-of-range source columns and rows are clamped (replicated), never reflected.
__device__ __forceinline__ void cubic_coeff(int d, int dst, int src, int& s, float c[4]) {
  const double scale = __ddiv_rn(1.0, __ddiv_rn(static_cast<double>(dst), static_cast<double>(src)));
  float f = __double2float_rn(__dadd_rn(__dmul_rn(__dadd_rn(static_cast<double>(d), 0.5), scale), -0.5));
  const float fs = floorf(f);
  s = static_cast<int>(fs);
  f = __fsub_rn(f, fs);
  constexpr float A = -0.75f;
  const float f1 = __fadd_rn(f, 1.0f), g = __fsub_rn(1.0f, f);
  c[0] = __fsub_rn(__fmul_rn(__fadd_rn(__fmul_rn(__fsub_rn(__fmul_rn(A, f1), 5.0f * A), f1), 8.0f * A), f1), 4.0f * A);
  c[1] = __fadd_rn(__fmul_rn(__fmul_rn(__fsub_rn(__fmul_rn(A + 2.0f, f), A + 3.0f), f), f), 1.0f);
  c[2] = __fadd_rn(__fmul_rn(__fmul_rn(__fsub_rn(__fmul_rn(A + 2.0f, g), A + 3.0f), g), g), 1.0f);
  c[3] = __fsub_rn(__fsub_rn(__fsub_rn(1.0f, c[0]), c[1]), c[2]);
}
// One thread per output pixel of image blockIdx.y (source geometry from its ada_img_desc row); out is [B, 3, H, W], the
// ImageNet-normalised input DepthAnythingV2.forward expects. u / 255.0 comes from a per-block table of the 256 doubles.
__global__ void __launch_bounds__(256)
resize_cubic_normalize_kernel(const uint8_t* __restrict__ src, const ada_img_desc* __restrict__ table,
                              float* __restrict__ out, int H, int W) {
  __shared__ double unit[256];
  unit[threadIdx.x] = __ddiv_rn(static_cast<double>(threadIdx.x), 255.0);
  __syncthreads();
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= H * W) return;
  const int y = i / W, x = i - y * W;
  const ada_img_desc g = table[blockIdx.y];
  const int H0 = static_cast<int>(g.H0), W0 = static_cast<int>(g.W0);
  const uint8_t* img = src + g.offset;
  int sx, sy;
  float cx[4], cy[4];
  cubic_coeff(x, W, W0, sx, cx);
  cubic_coeff(y, H, H0, sy, cy);
  int col[4];
#pragma unroll
  for (int k = 0; k < 4; ++k) col[k] = min(max(sx - 1 + k, 0), W0 - 1) * 3;
  double v[3];
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const uint8_t* r = img + static_cast<long long>(min(max(sy - 1 + k, 0), H0 - 1)) * W0 * 3;
    const double wy = static_cast<double>(cy[k]);
#pragma unroll
    for (int c = 0; c < 3; ++c) {   // output channel c reads source channel 2 - c (BGR -> RGB)
      double h = __dmul_rn(unit[r[col[0] + 2 - c]], static_cast<double>(cx[0]));
#pragma unroll
      for (int j = 1; j < 4; ++j) h = __dadd_rn(h, __dmul_rn(unit[r[col[j] + 2 - c]], static_cast<double>(cx[j])));
      v[c] = k == 0 ? __dmul_rn(h, wy) : __dadd_rn(v[c], __dmul_rn(h, wy));
    }
  }
  const double mean[3] = {0.485, 0.456, 0.406}, sd[3] = {0.229, 0.224, 0.225};
  float* o = out + static_cast<long long>(blockIdx.y) * 3 * H * W + i;
#pragma unroll
  for (int c = 0; c < 3; ++c)
    o[static_cast<long long>(c) * H * W] = __double2float_rn(__ddiv_rn(__dsub_rn(v[c], mean[c]), sd[c]));
}

// uint8 HWC image (cv2 order, infer.py:76) -> fp32 CHW in [0,1] at (H, W) by nearest sampling: rgb/255 then Resize(NEAREST)
// (infer.py:84-86). normalize != 0 additionally applies (x - mean) / std with the ImageNet constants per channel index
// (infer.py:18, the un-guided model's input). One thread per output pixel, 3 channels; out is [B, 3, H, W].
__global__ void __launch_bounds__(256)
image_nearest_kernel(const uint8_t* __restrict__ src, const ada_img_desc* __restrict__ table, int H0_, int W0_,
                     float* __restrict__ out, int H, int W, int normalize) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= H * W) return;
  const ada_img_desc g = image_desc(table, H0_, W0_);
  const int H0 = static_cast<int>(g.H0), W0 = static_cast<int>(g.W0);
  const int y = i / W, x = i - y * W;
  const int sy = nearest_src(y, static_cast<float>(H0) / static_cast<float>(H), H0);
  const int sx = nearest_src(x, static_cast<float>(W0) / static_cast<float>(W), W0);
  const uint8_t* p = src + g.offset + (static_cast<long long>(sy) * W0 + sx) * 3;
  float* o = out + static_cast<long long>(blockIdx.y) * 3 * H * W;
  const float mean[3] = {0.485f, 0.456f, 0.406f}, sd[3] = {0.229f, 0.224f, 0.225f};
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    float v = static_cast<float>(p[c]) / 255.0f;
    if (normalize) v = __fdiv_rn(__fsub_rn(v, mean[c]), sd[c]);  // same two roundings as the tensor expression
    o[static_cast<long long>(c) * H * W + i] = v;
  }
}

// uint8 mask (any non-zero = inside, infer.py:80-81) -> nearest resize -> mask01 (0/1, infer.py:87,100-101) and the
// network guide mask01 * 2 - 1 (infer.py:91), each [B, H, W]. Either output may be null.
__global__ void __launch_bounds__(256)
mask_nearest_kernel(const uint8_t* __restrict__ src, const ada_img_desc* __restrict__ table, int H0_, int W0_,
                    float* __restrict__ mask01, float* __restrict__ guide, int H, int W) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= H * W) return;
  const ada_img_desc g = image_desc(table, H0_, W0_);
  const int H0 = static_cast<int>(g.H0), W0 = static_cast<int>(g.W0);
  const int y = i / W, x = i - y * W;
  const int sy = nearest_src(y, static_cast<float>(H0) / static_cast<float>(H), H0);
  const int sx = nearest_src(x, static_cast<float>(W0) / static_cast<float>(W), W0);
  const float m = src[g.offset + static_cast<long long>(sy) * W0 + sx] > 0 ? 1.0f : 0.0f;
  const long long j = static_cast<long long>(blockIdx.y) * H * W + i;
  if (mask01) mask01[j] = m;
  if (guide) guide[j] = m * 2.0f - 1.0f;
}

// min / max of each of B fp32 maps of n values (infer.py:22): mm[2b] / mm[2b+1] for map b = blockIdx.y.
// Order-preserving float <-> uint mapping so atomicMin/Max work for any sign.
__device__ __forceinline__ uint32_t f2ord(float f) {
  const uint32_t u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(uint32_t o) {
  return __uint_as_float((o & 0x80000000u) ? (o & 0x7fffffffu) : ~o);
}
__global__ void minmax_init_kernel(uint32_t* mm, int B) {
  for (int b = threadIdx.x; b < B; b += blockDim.x) {
    mm[2 * b] = 0xffffffffu;  // min
    mm[2 * b + 1] = 0u;       // max
  }
}
__global__ void __launch_bounds__(256)
minmax_kernel(const float* __restrict__ d, long long n, uint32_t* mm) {
  d += static_cast<long long>(blockIdx.y) * n;
  mm += 2 * blockIdx.y;
  uint32_t lo = 0xffffffffu, hi = 0u;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const uint32_t o = f2ord(d[i]);
    lo = min(lo, o);
    hi = max(hi, o);
  }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) {
    lo = min(lo, __shfl_xor_sync(0xffffffffu, lo, s));
    hi = max(hi, __shfl_xor_sync(0xffffffffu, hi, s));
  }
  if ((threadIdx.x & 31) == 0) {
    atomicMin(mm, lo);
    atomicMax(mm + 1, hi);
  }
}
// base01 = (d - min) / (max - min) (infer.py:22); observation = base01 * 2 - 1 (infer.py:92), per map. Either output may
// be null. A constant map gives 0/0 = NaN, as the reference does.
__global__ void __launch_bounds__(256)
normalize_kernel(const float* __restrict__ d, long long n, const uint32_t* __restrict__ mm, float* __restrict__ base01,
                 float* __restrict__ obs) {
  const long long off = static_cast<long long>(blockIdx.y) * n;
  const float lo = ord2f(mm[2 * blockIdx.y]), hi = ord2f(mm[2 * blockIdx.y + 1]);
  const float range = hi - lo;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const float v = (d[off + i] - lo) / range;
    if (base01) base01[off + i] = v;
    if (obs) obs[off + i] = v * 2.0f - 1.0f;
  }
}

// median_filter_blend (infer.py:30-44, filter_width 3): blended = mask ? amodal : raw; the seam = pixels whose 3x3
// zero-padded mask sum is in (0, 9) is replaced by the 3x3 box mean of `blended` (cv2.blur: BORDER_REFLECT_101, row sums
// then column sum, times 1/9 in fp32). All maps [B, H, W]; map b = blockIdx.y.
__device__ __forceinline__ int reflect101(int i, int n) {
  if (i < 0) return -i;
  if (i >= n) return 2 * n - 2 - i;
  return i;
}
__global__ void __launch_bounds__(256)
blend_seam_kernel(const float* __restrict__ raw, const float* __restrict__ amodal, const float* __restrict__ mask01,
                  float* __restrict__ out, int H, int W) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= H * W) return;
  const long long off = static_cast<long long>(blockIdx.y) * H * W;
  raw += off;
  amodal += off;
  mask01 += off;
  const int y = i / W, x = i - y * W;
  auto blended = [&](int yy, int xx) {
    const int j = yy * W + xx;
    return mask01[j] > 0.f ? amodal[j] : raw[j];
  };
  float dil = 0.f;
#pragma unroll
  for (int dy = -1; dy <= 1; ++dy)
#pragma unroll
    for (int dx = -1; dx <= 1; ++dx) {
      const int yy = y + dy, xx = x + dx;
      if (yy >= 0 && yy < H && xx >= 0 && xx < W) dil += mask01[yy * W + xx];
    }
  float v = blended(y, x);
  if (dil > 0.f && dil < 9.f) {
    float rows[3];
#pragma unroll
    for (int dy = -1; dy <= 1; ++dy) {
      const int yy = reflect101(y + dy, H);
      rows[dy + 1] = (blended(yy, reflect101(x - 1, W)) + blended(yy, x)) + blended(yy, reflect101(x + 1, W));
    }
    v = ((rows[0] + rows[1]) + rows[2]) * (1.0f / 9.0f);
  }
  out[off + i] = v;
}

// F.interpolate(depth[:, None], (h, w), mode="bilinear", align_corners=True) of DepthAnythingV2.infer_image
// (depth_anything_v2_raw/dpt.py:186-222), with ATen's index math: scale (in - 1) / (out - 1) in fp32 (0 when out == 1),
// src = scale * dst, i1 = i0 + (i0 < in - 1), lambda = src - i0. Every product and sum is rounded on its own. Map b =
// blockIdx.y of depth [B, H, W] goes to its own (h, w) = (H0, W0) of its ada_img_desc row, at that row's byte offset
// from out. The output sizes live on the device, so the threads of an image stride over its pixels.
__device__ __forceinline__ void restore_coord(int d, int out, int in, int& i0, int& i1, float& l0, float& l1) {
  const float scale = out > 1 ? __fdiv_rn(static_cast<float>(in - 1), static_cast<float>(out - 1)) : 0.0f;
  const float s = __fmul_rn(scale, static_cast<float>(d));
  i0 = static_cast<int>(s);
  i1 = i0 + (i0 < in - 1 ? 1 : 0);
  l1 = __fsub_rn(s, static_cast<float>(i0));
  l0 = __fsub_rn(1.0f, l1);
}
__global__ void __launch_bounds__(256)
upsample_restore_kernel(const float* __restrict__ depth, int H, int W, const ada_img_desc* __restrict__ table,
                        float* __restrict__ out) {
  const ada_img_desc g = table[blockIdx.y];
  const int h = static_cast<int>(g.H0), w = static_cast<int>(g.W0);
  const float* d = depth + static_cast<long long>(blockIdx.y) * H * W;
  float* o = reinterpret_cast<float*>(reinterpret_cast<char*>(out) + g.offset);
  const long long n = static_cast<long long>(h) * w;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int y = static_cast<int>(i / w), x = static_cast<int>(i - static_cast<long long>(y) * w);
    int y0, y1, x0, x1;
    float h0, h1, w0, w1;
    restore_coord(y, h, H, y0, y1, h0, h1);
    restore_coord(x, w, W, x0, x1, w0, w1);
    const float* r0 = d + static_cast<long long>(y0) * W;
    const float* r1 = d + static_cast<long long>(y1) * W;
    const float top = __fadd_rn(__fmul_rn(w0, r0[x0]), __fmul_rn(w1, r0[x1]));
    const float bot = __fadd_rn(__fmul_rn(w0, r1[x0]), __fmul_rn(w1, r1[x1]));
    o[i] = __fadd_rn(__fmul_rn(h0, top), __fmul_rn(h1, bot));
  }
}

}  // namespace ada
