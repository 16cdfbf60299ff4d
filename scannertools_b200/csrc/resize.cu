// Resize op (SURVEY §8f rank 1): cv::resize(..., INTER_LINEAR) on 8-bit frames, bit-exact with
// OpenCV's fixed-point path (scannertools_cpp/imgproc/resize_kernel.cpp:69-71 on CPU,
// cvc::resize :75-79 on GPU).  It is the step in front of OpticalFlow in the shipped
// flow-histogram pipeline (scannertools/old/histograms.py:64-68, 426x240).
//
// One thread per output pixel (all channels).  11-bit coefficients cvRound(f * 2048), horizontal
// taps in int, vertical (((b0 * (S0 >> 4)) >> 16) + ((b1 * (S1 >> 4)) >> 16) + 2) >> 2.  The x
// index/fraction are clamped when the coefficient is formed, y keeps the unclamped fraction and
// clips the two row indices -- exactly OpenCV's asymmetry (it changes results on up-scaled
// border rows).  Exact 2x down-scaling takes OpenCV's INTER_AREA fast path (a+b+c+d+2)>>2.
//
// The other interpolation names the reference maps (resize_kernel.cpp:9-20) that are implemented:
// INTER_NEAREST and INTER_AREA (integer-factor block averages, the general weighted-cell tables with
// OpenCV's float accumulation order, and the linear "area" coefficients when an axis is up-scaled),
// all bit-exact with cv2 4.13.
//
// INTER_CUBIC / INTER_LANCZOS4 (resize_kernel.cpp:13,15): OpenCV's generic separable fixed-point path
// (resizeGeneric_ with HResizeCubic / HResizeLanczos4 in int and 11-bit short coefficients).  The tap
// tables (first source index + 4 / 8 shorts per destination column and row) are built on the HOST with
// the same float / double expressions OpenCV uses (interpolateCubic, A = -0.75; interpolateLanczos4 with
// libm's sin / cos) and uploaded stream-ordered; resize_taps_u8_kernel applies them.  The vertical pass
// reproduces OpenCV's two code paths: VResizeCubicVec_32s8u combines the four int rows in float
// (beta * 2^-22, mul / add without contraction, round half even) for the first floor(W * cn / 8) * 8
// elements of a row and the exact integer (sum + 2^21) >> 22 for the scalar tail; Lanczos4 has no vector
// path for 8-bit frames.  Bit-exact with cv2's own implementation (cv2.ipp.setUseIPP(False)); builds of
// OpenCV that dispatch 8-bit cubic to IPP differ from OpenCV's own code by one grey level on ~5 % of pixels.
//
// Float32 frames with 1 to 4 channels (OpticalFlow's H x W x 2 fields) take the same five paths, chosen by the same
// host routine (plan_resize), with the same coordinates, area tables and tap tables, and OpenCV's float arithmetic
// (resize_*_f32_kernel below).
#include <cmath>
#include <string>
#include <vector>

#include "stb_rt.h"

namespace stb {

enum { kInterpLinear = 0, kInterpNearest = 1, kInterpArea = 2, kInterpCubic = 3, kInterpLanczos4 = 4 };

__device__ __forceinline__ int cv_round_f(float v) { return __float2int_rn(v); }

__device__ __forceinline__ int clamp_index(int i, int n) { return min(max(i, 0), n - 1); }

// Source taps of one linear output pixel, shared by the 8-bit and the float kernels: columns sx, sx1 with fraction
// fx, rows y0, y1 with fraction fy.
struct LinearTaps {
  int sx, sx1, y0, y1;
  float fx, fy;
};

__device__ __forceinline__ LinearTaps linear_taps(int dx, int dy, int sw, int sh, int dw, int dh, double scale_x,
                                                  double scale_y, int area_mode) {
  float fx, fy;
  int sx, sy;
  if (!area_mode) {
    fx = (float)((dx + 0.5) * scale_x - 0.5);
    sx = __float2int_rd(fx);
    fx -= (float)sx;
    fy = (float)((dy + 0.5) * scale_y - 0.5);
    sy = __float2int_rd(fy);
    fy -= (float)sy;
  } else {
    // INTER_AREA with an up-scaled axis: linear arithmetic, "area" coefficients
    // (inv_scale is the double dsize/ssize, scale = 1/inv_scale, as cv::resize forms them)
    const double inv_x = (double)dw / sw, inv_y = (double)dh / sh;
    sx = __double2int_rd(dx * scale_x);
    fx = (float)((dx + 1) - (sx + 1) * inv_x);
    fx = fx <= 0.f ? 0.f : fx - floorf(fx);
    sy = __double2int_rd(dy * scale_y);
    fy = (float)((dy + 1) - (sy + 1) * inv_y);
    fy = fy <= 0.f ? 0.f : fy - floorf(fy);
  }
  if (sx < 0) { fx = 0.f; sx = 0; }
  if (sx >= sw - 1) { fx = 0.f; sx = sw - 1; }
  LinearTaps t;
  t.sx = sx;
  t.sx1 = sx + 1 < sw ? sx + 1 : sx;
  t.y0 = clamp_index(sy, sh);
  t.y1 = clamp_index(sy + 1, sh);
  t.fx = fx;
  t.fy = fy;
  return t;
}

template <int CN>
__global__ void __launch_bounds__(256)
resize_linear_u8_kernel(PtrBatch<const uint8_t> srcs, PtrBatch<uint8_t> dsts, int sw, int sh, int dw, int dh,
                        double scale_x, double scale_y, int area2x, int area_mode) {
  const int dx = blockIdx.x * 32 + (threadIdx.x & 31);
  const int dy = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (dx >= dw || dy >= dh) return;
  const uint8_t* src = srcs.p[blockIdx.z];
  uint8_t* dst = dsts.p[blockIdx.z] + ((size_t)dy * dw + dx) * CN;
  if (area2x) {
    const uint8_t* p = src + ((size_t)(2 * dy) * sw + 2 * dx) * CN;
    const size_t rs = (size_t)sw * CN;
#pragma unroll
    for (int c = 0; c < CN; ++c) dst[c] = (uint8_t)((p[c] + p[CN + c] + p[rs + c] + p[rs + CN + c] + 2) >> 2);
    return;
  }
  const LinearTaps t = linear_taps(dx, dy, sw, sh, dw, dh, scale_x, scale_y, area_mode);
  const int sx = t.sx, sx1 = t.sx1;
  const int a0 = cv_round_f(__fmul_rn(1.f - t.fx, 2048.f)), a1 = cv_round_f(__fmul_rn(t.fx, 2048.f));
  const int b0 = cv_round_f(__fmul_rn(1.f - t.fy, 2048.f)), b1 = cv_round_f(__fmul_rn(t.fy, 2048.f));
  const uint8_t* r0 = src + (size_t)t.y0 * sw * CN;
  const uint8_t* r1 = src + (size_t)t.y1 * sw * CN;
#pragma unroll
  for (int c = 0; c < CN; ++c) {
    const int h0 = r0[sx * CN + c] * a0 + r0[sx1 * CN + c] * a1;
    const int h1 = r1[sx * CN + c] * a0 + r1[sx1 * CN + c] * a1;
    const int v = (((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2;
    dst[c] = (uint8_t)min(max(v, 0), 255);
  }
}

// INTER_NEAREST: sx = min(floor(dx * scale_x), sw - 1) (cv::resizeNN)
__device__ __forceinline__ int nearest_index(int d, double scale, int sn) { return min(__double2int_rd(d * scale), sn - 1); }

template <int CN>
__global__ void __launch_bounds__(256)
resize_nearest_u8_kernel(PtrBatch<const uint8_t> srcs, PtrBatch<uint8_t> dsts, int sw, int sh, int dw, int dh,
                         double scale_x, double scale_y) {
  const int dx = blockIdx.x * 32 + (threadIdx.x & 31);
  const int dy = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (dx >= dw || dy >= dh) return;
  const int sx = nearest_index(dx, scale_x, sw), sy = nearest_index(dy, scale_y, sh);
  const uint8_t* p = srcs.p[blockIdx.z] + ((size_t)sy * sw + sx) * CN;
  uint8_t* dst = dsts.p[blockIdx.z] + ((size_t)dy * dw + dx) * CN;
#pragma unroll
  for (int c = 0; c < CN; ++c) dst[c] = p[c];
}

// INTER_AREA, integer factors (cv::ResizeAreaFast): block sum, (s + 2) >> 2 for 2x2, otherwise
// saturate(round(sum * (1.f / area)))
template <int CN>
__global__ void __launch_bounds__(256)
resize_area_int_u8_kernel(PtrBatch<const uint8_t> srcs, PtrBatch<uint8_t> dsts, int sw, int dw, int dh, int isx, int isy) {
  const int dx = blockIdx.x * 32 + (threadIdx.x & 31);
  const int dy = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (dx >= dw || dy >= dh) return;
  const uint8_t* p = srcs.p[blockIdx.z] + ((size_t)(dy * isy) * sw + (size_t)dx * isx) * CN;
  uint8_t* dst = dsts.p[blockIdx.z] + ((size_t)dy * dw + dx) * CN;
  int sum[CN];
#pragma unroll
  for (int c = 0; c < CN; ++c) sum[c] = 0;
  for (int j = 0; j < isy; ++j) {
    const uint8_t* r = p + (size_t)j * sw * CN;
    for (int i = 0; i < isx; ++i) {
#pragma unroll
      for (int c = 0; c < CN; ++c) sum[c] += r[i * CN + c];
    }
  }
  const float scale = __fdiv_rn(1.f, (float)(isx * isy));
#pragma unroll
  for (int c = 0; c < CN; ++c) {
    const int v = (isx == 2 && isy == 2) ? (sum[c] + 2) >> 2 : __float2int_rn(__fmul_rn((float)sum[c], scale));
    dst[c] = (uint8_t)min(max(v, 0), 255);
  }
}

// One destination index of cv::computeResizeAreaTab: the source cells [first, first + n) it covers
// and their float weights, in table order (optional partial first cell, full cells, optional
// partial last cell).
struct AreaSpan {
  int first, n;
  float a_first, a_mid, a_last;
  bool has_first, has_last;
  __device__ __forceinline__ float alpha(int k) const {
    if (k == 0 && has_first) return a_first;
    if (k == n - 1 && has_last) return a_last;
    return a_mid;
  }
};

__device__ __forceinline__ AreaSpan area_span(int d, double scale, int ssize) {
  const double f1 = d * scale, f2 = f1 + scale;
  const double cell = fmin(scale, ssize - f1);
  int s1 = __double2int_ru(f1), s2 = __double2int_rd(f2);
  s2 = min(s2, ssize - 1);
  s1 = min(s1, s2);
  AreaSpan sp;
  sp.has_first = (s1 - f1) > 1e-3;
  sp.has_last = (f2 - s2) > 1e-3;
  sp.a_first = (float)((s1 - f1) / cell);
  sp.a_mid = (float)(1.0 / cell);
  sp.a_last = (float)(fmin(fmin(f2 - s2, 1.0), cell) / cell);
  sp.first = sp.has_first ? s1 - 1 : s1;
  sp.n = (s2 - s1) + (sp.has_first ? 1 : 0) + (sp.has_last ? 1 : 0);
  return sp;
}

// INTER_AREA, general down-scaling (cv::ResizeArea_Invoker): float accumulation in table order,
// no FMA contraction: buf = sum_x S * alpha (from 0), sum = beta_0 * buf_0, sum += beta_j * buf_j.
template <int CN>
__global__ void __launch_bounds__(256)
resize_area_u8_kernel(PtrBatch<const uint8_t> srcs, PtrBatch<uint8_t> dsts, int sw, int sh, int dw, int dh,
                      double scale_x, double scale_y) {
  const int dx = blockIdx.x * 32 + (threadIdx.x & 31);
  const int dy = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (dx >= dw || dy >= dh) return;
  const AreaSpan xs = area_span(dx, scale_x, sw), ys = area_span(dy, scale_y, sh);
  const uint8_t* src = srcs.p[blockIdx.z];
  uint8_t* dst = dsts.p[blockIdx.z] + ((size_t)dy * dw + dx) * CN;
  float sum[CN];
#pragma unroll
  for (int c = 0; c < CN; ++c) sum[c] = 0.f;
  for (int j = 0; j < ys.n; ++j) {
    const uint8_t* r = src + ((size_t)(ys.first + j) * sw + xs.first) * CN;
    float buf[CN];
#pragma unroll
    for (int c = 0; c < CN; ++c) buf[c] = 0.f;
    for (int i = 0; i < xs.n; ++i) {
      const float a = xs.alpha(i);
#pragma unroll
      for (int c = 0; c < CN; ++c) buf[c] = __fadd_rn(buf[c], __fmul_rn((float)r[i * CN + c], a));
    }
    const float beta = ys.alpha(j);
#pragma unroll
    for (int c = 0; c < CN; ++c) sum[c] = j == 0 ? __fmul_rn(beta, buf[c]) : __fadd_rn(sum[c], __fmul_rn(beta, buf[c]));
  }
#pragma unroll
  for (int c = 0; c < CN; ++c) dst[c] = (uint8_t)min(max(__float2int_rn(sum[c]), 0), 255);
}

// INTER_CUBIC (K = 4) / INTER_LANCZOS4 (K = 8): host-built tap tables.  xofs / yofs = index of the first
// tap (may be outside the image: taps are clamped to the border, cv::resizeGeneric_'s xmin / xmax handling);
// xa / ya = K short coefficients per destination column / row.  One thread per output pixel.
template <int CN, int K>
__global__ void __launch_bounds__(256)
resize_taps_u8_kernel(PtrBatch<const uint8_t> srcs, PtrBatch<uint8_t> dsts, int sw, int sh, int dw, int dh,
                      const int* __restrict__ xofs, const short* __restrict__ xa, const int* __restrict__ yofs,
                      const short* __restrict__ ya, int vec_elems) {
  const int dx = blockIdx.x * 32 + (threadIdx.x & 31);
  const int dy = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (dx >= dw || dy >= dh) return;
  const uint8_t* src = srcs.p[blockIdx.z];
  uint8_t* dst = dsts.p[blockIdx.z] + ((size_t)dy * dw + dx) * CN;
  const int sx0 = xofs[dx], sy0 = yofs[dy];
  int a[K], b[K], cx[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    a[k] = xa[dx * K + k];
    b[k] = ya[dy * K + k];
    cx[k] = clamp_index(sx0 + k, sw) * CN;
  }
  int hsum[K][CN];
#pragma unroll
  for (int j = 0; j < K; ++j) {
    const uint8_t* r = src + (size_t)clamp_index(sy0 + j, sh) * sw * CN;
#pragma unroll
    for (int c = 0; c < CN; ++c) {
      int h = 0;
#pragma unroll
      for (int k = 0; k < K; ++k) h += r[cx[k] + c] * a[k];
      hsum[j][c] = h;
    }
  }
#pragma unroll
  for (int c = 0; c < CN; ++c) {
    int v;
    if (K == 4 && dx * CN + c < vec_elems) {
      // VResizeCubicVec_32s8u: float, S3 * b3 first, then + S2 * b2, + S1 * b1, + S0 * b0 (mul and add rounded separately)
      const float sc = 1.f / (2048.f * 2048.f);
      float acc = __fmul_rn((float)hsum[3][c], __fmul_rn((float)b[3], sc));
      acc = __fadd_rn(__fmul_rn((float)hsum[2][c], __fmul_rn((float)b[2], sc)), acc);
      acc = __fadd_rn(__fmul_rn((float)hsum[1][c], __fmul_rn((float)b[1], sc)), acc);
      acc = __fadd_rn(__fmul_rn((float)hsum[0][c], __fmul_rn((float)b[0], sc)), acc);
      v = __float2int_rn(acc);
    } else {
      int t = 0;
#pragma unroll
      for (int j = 0; j < K; ++j) t += hsum[j][c] * b[j];
      v = (t + (1 << 21)) >> 22;   // FixedPtCast<int, uchar, INTER_RESIZE_COEF_BITS * 2>
    }
    dst[c] = (uint8_t)min(max(v, 0), 255);
  }
}

// ---- float32 frames (a flow field is H x W x 2) ----------------------------------------------------------------
// The same taps as the 8-bit kernels with OpenCV's float arithmetic: every product and sum is rounded on its own
// (__fmul_rn / __fadd_rn, no FMA contraction) in the order cv::resize's float path uses, and nothing is rounded to
// an integer.  Frames are 4-byte aligned float arrays read and written one element at a time.

template <int CN>
__global__ void __launch_bounds__(256)
resize_nearest_f32_kernel(PtrBatch<const float> srcs, PtrBatch<float> dsts, int sw, int sh, int dw, int dh,
                          double scale_x, double scale_y) {
  const int dx = blockIdx.x * 32 + (threadIdx.x & 31);
  const int dy = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (dx >= dw || dy >= dh) return;
  const int sx = nearest_index(dx, scale_x, sw), sy = nearest_index(dy, scale_y, sh);
  const float* p = srcs.p[blockIdx.z] + ((size_t)sy * sw + sx) * CN;
  float* dst = dsts.p[blockIdx.z] + ((size_t)dy * dw + dx) * CN;
#pragma unroll
  for (int c = 0; c < CN; ++c) dst[c] = p[c];
}

// INTER_LINEAR, and INTER_AREA with an up-scaled axis: h = S[sx] * a0 + S[sx1] * a1 per row (a0 = 1 - fx, a1 = fx),
// out = h0 * b0 + h1 * b1 (HResizeLinear / VResizeLinear in float).  Columns clamped at the right border (sx1 == sx,
// OpenCV's dx >= xmax) take h = S[sx] * 1 without the neighbour term, so an inf there stays inf, as in OpenCV.
template <int CN>
__global__ void __launch_bounds__(256)
resize_linear_f32_kernel(PtrBatch<const float> srcs, PtrBatch<float> dsts, int sw, int sh, int dw, int dh,
                         double scale_x, double scale_y, int area_mode) {
  const int dx = blockIdx.x * 32 + (threadIdx.x & 31);
  const int dy = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (dx >= dw || dy >= dh) return;
  const LinearTaps t = linear_taps(dx, dy, sw, sh, dw, dh, scale_x, scale_y, area_mode);
  const float a0 = 1.f - t.fx, a1 = t.fx, b0 = 1.f - t.fy, b1 = t.fy;
  const float* src = srcs.p[blockIdx.z];
  const float* r0 = src + (size_t)t.y0 * sw * CN;
  const float* r1 = src + (size_t)t.y1 * sw * CN;
  const size_t x0 = (size_t)t.sx * CN, x1 = (size_t)t.sx1 * CN;
  float* dst = dsts.p[blockIdx.z] + ((size_t)dy * dw + dx) * CN;
#pragma unroll
  for (int c = 0; c < CN; ++c) {
    const float h0 = x1 == x0 ? __fmul_rn(r0[x0 + c], a0) : __fadd_rn(__fmul_rn(r0[x0 + c], a0), __fmul_rn(r0[x1 + c], a1));
    const float h1 = x1 == x0 ? __fmul_rn(r1[x0 + c], a0) : __fadd_rn(__fmul_rn(r1[x0 + c], a0), __fmul_rn(r1[x1 + c], a1));
    dst[c] = __fadd_rn(__fmul_rn(h0, b0), __fmul_rn(h1, b1));
  }
}

// INTER_AREA with integer factors, and INTER_LINEAR at exactly 2x down (cv::resizeAreaFast_ on float).  With
// a = (y0, x0), b = (y0, x1), c = (y1, x0), d = (y1, x1) a 2x2 block is ((a + b) + (c + d)) * 0.25 where OpenCV's
// 4-float vector body runs (every element at 4 channels, the first floor(dw / 4) * 4 pixels of a row at 1 channel)
// and (0 + (((a + b) + c) + d)) * 0.25 in its scalar code (its sum starts at +0, so a block of -0 gives +0 there).  Other factors: the block in row-major order, summed four
// elements at a time, (((s0 + s1) + s2) + s3) added to the running sum, the rest one by one, times 1 / area.
template <int CN>
__global__ void __launch_bounds__(256)
resize_area_int_f32_kernel(PtrBatch<const float> srcs, PtrBatch<float> dsts, int sw, int dw, int dh, int isx, int isy) {
  const int dx = blockIdx.x * 32 + (threadIdx.x & 31);
  const int dy = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (dx >= dw || dy >= dh) return;
  const size_t rs = (size_t)sw * CN;
  const float* p = srcs.p[blockIdx.z] + (size_t)dy * isy * rs + (size_t)dx * isx * CN;
  float* dst = dsts.p[blockIdx.z] + ((size_t)dy * dw + dx) * CN;
  if (isx == 2 && isy == 2) {
    const bool vec = CN == 4 || (CN == 1 && dx < (dw & ~3));
#pragma unroll
    for (int c = 0; c < CN; ++c) {
      const float a = p[c], b = p[CN + c], cc = p[rs + c], d = p[rs + CN + c];
      const float s = vec ? __fadd_rn(__fadd_rn(a, b), __fadd_rn(cc, d))
                          : __fadd_rn(0.f, __fadd_rn(__fadd_rn(__fadd_rn(a, b), cc), d));
      dst[c] = __fmul_rn(s, 0.25f);
    }
    return;
  }
  const int area = isx * isy;
  const float scale = __fdiv_rn(1.f, (float)area);
#pragma unroll
  for (int c = 0; c < CN; ++c) {
    float sum = 0.f;
    int i = 0, j = 0;   // block element k = j * isx + i
    auto next = [&]() {
      const float v = p[(size_t)j * rs + (size_t)i * CN + c];
      if (++i == isx) { i = 0; ++j; }
      return v;
    };
    int k = 0;
    for (; k + 4 <= area; k += 4) {
      float g = next();
      g = __fadd_rn(g, next());
      g = __fadd_rn(g, next());
      g = __fadd_rn(g, next());
      sum = __fadd_rn(sum, g);
    }
    for (; k < area; ++k) sum = __fadd_rn(sum, next());
    dst[c] = __fmul_rn(sum, scale);
  }
}

// INTER_AREA, general down-scaling: the table order of resize_area_u8_kernel without the final rounding.
template <int CN>
__global__ void __launch_bounds__(256)
resize_area_f32_kernel(PtrBatch<const float> srcs, PtrBatch<float> dsts, int sw, int sh, int dw, int dh,
                       double scale_x, double scale_y) {
  const int dx = blockIdx.x * 32 + (threadIdx.x & 31);
  const int dy = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (dx >= dw || dy >= dh) return;
  const AreaSpan xs = area_span(dx, scale_x, sw), ys = area_span(dy, scale_y, sh);
  const float* src = srcs.p[blockIdx.z];
  float* dst = dsts.p[blockIdx.z] + ((size_t)dy * dw + dx) * CN;
  float sum[CN];
#pragma unroll
  for (int c = 0; c < CN; ++c) sum[c] = 0.f;
  for (int j = 0; j < ys.n; ++j) {
    const float* r = src + ((size_t)(ys.first + j) * sw + xs.first) * CN;
    float buf[CN];
#pragma unroll
    for (int c = 0; c < CN; ++c) buf[c] = 0.f;
    for (int i = 0; i < xs.n; ++i) {
      const float a = xs.alpha(i);
#pragma unroll
      for (int c = 0; c < CN; ++c) buf[c] = __fadd_rn(buf[c], __fmul_rn(r[(size_t)i * CN + c], a));
    }
    const float beta = ys.alpha(j);
#pragma unroll
    for (int c = 0; c < CN; ++c) sum[c] = j == 0 ? __fmul_rn(beta, buf[c]) : __fadd_rn(sum[c], __fmul_rn(beta, buf[c]));
  }
#pragma unroll
  for (int c = 0; c < CN; ++c) dst[c] = sum[c];
}

// INTER_CUBIC (K = 4) / INTER_LANCZOS4 (K = 8) with the float coefficients of the host tap tables: per source row
// h = S[x0] * a0 + S[x1] * a1 + ... left to right, then out = h0 * b0 + h1 * b1 + ... top to bottom.
template <int CN, int K>
__global__ void __launch_bounds__(256)
resize_taps_f32_kernel(PtrBatch<const float> srcs, PtrBatch<float> dsts, int sw, int sh, int dw, int dh,
                       const int* __restrict__ xofs, const float* __restrict__ xa, const int* __restrict__ yofs,
                       const float* __restrict__ ya) {
  const int dx = blockIdx.x * 32 + (threadIdx.x & 31);
  const int dy = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (dx >= dw || dy >= dh) return;
  const float* src = srcs.p[blockIdx.z];
  float* dst = dsts.p[blockIdx.z] + ((size_t)dy * dw + dx) * CN;
  const int sx0 = xofs[dx], sy0 = yofs[dy];
  float a[K];
  size_t cx[K];
#pragma unroll
  for (int k = 0; k < K; ++k) {
    a[k] = xa[(size_t)dx * K + k];
    cx[k] = (size_t)clamp_index(sx0 + k, sw) * CN;
  }
  float acc[CN];
#pragma unroll
  for (int j = 0; j < K; ++j) {
    const float* r = src + (size_t)clamp_index(sy0 + j, sh) * sw * CN;
    const float b = ya[(size_t)dy * K + j];
#pragma unroll
    for (int c = 0; c < CN; ++c) {
      float h = __fmul_rn(r[cx[0] + c], a[0]);
#pragma unroll
      for (int k = 1; k < K; ++k) h = __fadd_rn(h, __fmul_rn(r[cx[k] + c], a[k]));
      acc[c] = j == 0 ? __fmul_rn(h, b) : __fadd_rn(acc[c], __fmul_rn(h, b));
    }
  }
#pragma unroll
  for (int c = 0; c < CN; ++c) dst[c] = acc[c];
}

// ---- host side of the tap tables: OpenCV's expressions in OpenCV's precision -------------------------
#if defined(__GNUC__) && !defined(__clang__)
#define STB_NO_CONTRACT __attribute__((optimize("fp-contract=off")))
#else
#define STB_NO_CONTRACT
#endif

static STB_NO_CONTRACT void cubic_coeffs(float x, float* c) {          // cv::interpolateCubic
  const float A = -0.75f;
  c[0] = ((A * (x + 1) - 5 * A) * (x + 1) + 8 * A) * (x + 1) - 4 * A;
  c[1] = ((A + 2) * x - (A + 3)) * x * x + 1;
  c[2] = ((A + 2) * (1 - x) - (A + 3)) * (1 - x) * (1 - x) + 1;
  c[3] = 1.f - c[0] - c[1] - c[2];
}

static STB_NO_CONTRACT void lanczos4_coeffs(float x, float* c) {       // cv::interpolateLanczos4
  static const double s45 = 0.70710678118654752440;
  static const double cs[][2] = {{1, 0}, {-s45, -s45}, {0, 1}, {s45, -s45}, {-1, 0}, {s45, s45}, {0, -1}, {-s45, s45}};
  if (x < 1.1920928955078125e-07f) {                                   // FLT_EPSILON
    for (int i = 0; i < 8; ++i) c[i] = 0.f;
    c[3] = 1.f;
    return;
  }
  float sum = 0.f;
  const double y0 = -(x + 3) * 3.1415926535897932384626433832795 * 0.25, s0 = std::sin(y0), c0 = std::cos(y0);
  for (int i = 0; i < 8; ++i) {
    const double y = -(x + 3 - i) * 3.1415926535897932384626433832795 * 0.25;
    c[i] = (float)((cs[i][0] * s0 + cs[i][1] * c0) / (y * y));
    sum += c[i];
  }
  sum = 1.f / sum;
  for (int i = 0; i < 8; ++i) c[i] *= sum;
}

// cv::resize's tap tables for INTER_CUBIC / INTER_LANCZOS4: per destination index the first source index (it may lie
// outside the image) and K float coefficients.
static STB_NO_CONTRACT void build_taps(int dn, int sn, int K, bool cubic, std::vector<int>& ofs, std::vector<float>& al) {
  const double scale = 1. / ((double)dn / sn);
  ofs.resize(dn);
  al.resize((size_t)dn * K);
  for (int d = 0; d < dn; ++d) {
    float f = (float)((d + 0.5) * scale - 0.5);
    const int s0 = (int)std::floor(f);
    f -= s0;
    float c[8];
    if (cubic) cubic_coeffs(f, c); else lanczos4_coeffs(f, c);
    ofs[d] = s0 - (K / 2 - 1);
    for (int k = 0; k < K; ++k) al[(size_t)d * K + k] = c[k];
  }
}

// the 8-bit coefficient of a float one: saturate_cast<short>(cbuf[k] * INTER_RESIZE_COEF_SCALE)
static STB_NO_CONTRACT short tap_coef_u8(float c) {
  const float v = c * 2048.f;
  const long r = std::lrint(v);                                        // round half to even (default rounding mode)
  return (short)(r < -32768 ? -32768 : (r > 32767 ? 32767 : r));
}

static float tap_coef_f32(float c) { return c; }

// Tap tables on the device, in one allocation [xofs | yofs | xa | ya]; mem is released with cudaFreeAsync.
template <class Coef>
struct TapTables {
  int* mem = nullptr;
  const int *xofs = nullptr, *yofs = nullptr;
  const Coef *xa = nullptr, *ya = nullptr;
};

// Builds the tables on the host and uploads them in stream order.
template <class Coef>
static int upload_taps(const char* who, int sw, int sh, int dw, int dh, int K, bool cubic, Coef (*coef)(float),
                       cudaStream_t s, TapTables<Coef>* t) {
  std::vector<int> xo, yo;
  std::vector<float> xa, ya;
  build_taps(dw, sw, K, cubic, xo, xa);
  build_taps(dh, sh, K, cubic, yo, ya);
  const size_t n_int = (size_t)dw + dh, n_coef = xa.size() + ya.size();
  std::vector<int> host(n_int + (n_coef * sizeof(Coef) + sizeof(int) - 1) / sizeof(int));
  std::copy(xo.begin(), xo.end(), host.begin());
  std::copy(yo.begin(), yo.end(), host.begin() + dw);
  Coef* hc = reinterpret_cast<Coef*>(host.data() + n_int);
  for (size_t i = 0; i < xa.size(); ++i) hc[i] = coef(xa[i]);
  for (size_t i = 0; i < ya.size(); ++i) hc[xa.size() + i] = coef(ya[i]);
  STB_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&t->mem), host.size() * sizeof(int), s));
  // pageable source: the runtime stages it before returning, so `host` may go out of scope
  cudaError_t e = cudaMemcpyAsync(t->mem, host.data(), host.size() * sizeof(int), cudaMemcpyHostToDevice, s);
  if (e != cudaSuccess) {
    cudaFreeAsync(t->mem, s);
    t->mem = nullptr;
    return cuda_fail(e, (std::string(who) + ": tap table upload").c_str());
  }
  t->xofs = t->mem;
  t->yofs = t->mem + dw;
  t->xa = reinterpret_cast<const Coef*>(t->mem + n_int);
  t->ya = t->xa + (size_t)dw * K;
  return STB_OK;
}

// Which of OpenCV's code paths cv::resize takes for an interpolation code and a pair of sizes.  Both element types
// select the same way.
enum ResizePath {
  kPathNearest,    // INTER_NEAREST, and every mode at dsize == ssize (cv::resize copies the frame; nearest at scale 1
                   // is that copy, element for element)
  kPathAreaFast,   // integer factors: INTER_AREA scaled down by whole numbers, INTER_LINEAR by exactly 2
  kPathArea,       // INTER_AREA scaled down on both axes, other factors
  kPathLinear,     // INTER_LINEAR, and INTER_AREA with an up-scaled axis (area_coeffs)
  kPathTaps,       // INTER_CUBIC / INTER_LANCZOS4
};

struct ResizePlan {
  ResizePath path;
  double scale_x, scale_y;   // 1 / (dsize / ssize), as cv::resize forms them
  int isx, isy;              // kPathAreaFast: the integer factors
  int area_coeffs;           // kPathLinear: INTER_AREA's coefficients
};

static ResizePlan plan_resize(int interp, int sw, int sh, int dw, int dh) {
  ResizePlan p;
  p.scale_x = 1. / ((double)dw / sw);
  p.scale_y = 1. / ((double)dh / sh);
  // cv::resize: iscale = saturate_cast<int>(scale) (round half even); "fast area" when both are integers
  p.isx = (int)std::nearbyint(p.scale_x);
  p.isy = (int)std::nearbyint(p.scale_y);
  const bool int_scale = std::fabs(p.scale_x - p.isx) < 2.220446049250313e-16 && std::fabs(p.scale_y - p.isy) < 2.220446049250313e-16;
  const bool down = p.scale_x >= 1 && p.scale_y >= 1;
  p.area_coeffs = interp == kInterpArea ? 1 : 0;
  if (sw == dw && sh == dh) p.path = kPathNearest;
  else if (interp == kInterpCubic || interp == kInterpLanczos4) p.path = kPathTaps;
  else if (interp == kInterpNearest) p.path = kPathNearest;
  else if (interp == kInterpLinear && sw == 2 * dw && sh == 2 * dh) p.path = kPathAreaFast;
  else if (interp == kInterpArea && down && int_scale) p.path = kPathAreaFast;
  else if (interp == kInterpArea && down) p.path = kPathArea;
  else p.path = kPathLinear;
  return p;
}

// The scalar checks of a resize entry point, in the order both report them.
static int check_resize_args(const char* who, int n, int src_w, int src_h, int dst_w, int dst_h, int channels,
                             bool channels_ok, const char* channel_list, int interp) {
  if (n < 0 || src_w <= 0 || src_h <= 0 || dst_w <= 0 || dst_h <= 0) {
    set_error("%s: invalid argument (n=%d, %dx%d -> %dx%d)", who, n, src_w, src_h, dst_w, dst_h);
    return STB_ERR_INVALID;
  }
  if (!channels_ok) {
    set_error("%s: %d channels not supported (%s)", who, channels, channel_list);
    return STB_ERR_UNSUPPORTED;
  }
  if (interp < kInterpLinear || interp > kInterpLanczos4) {
    set_error("%s: interpolation %d is not implemented (INTER_LINEAR, INTER_NEAREST, INTER_AREA, INTER_CUBIC, INTER_LANCZOS4)", who, interp);
    return STB_ERR_UNSUPPORTED;
  }
  return STB_OK;
}

// float frames are read and written as floats: every entry must be 4-byte aligned
static int check_float_aligned(const float* const* tab, int n, const char* who, const char* what) {
  for (int i = 0; i < n; ++i)
    if (reinterpret_cast<uintptr_t>(tab[i]) % alignof(float)) {
      set_error("%s: %s %d is not 4-byte aligned", who, what, i);
      return STB_ERR_INVALID;
    }
  return STB_OK;
}

template <class F>
static F by_channels(int channels, F c1, F c2, F c3, F c4) {
  return channels == 1 ? c1 : channels == 2 ? c2 : channels == 3 ? c3 : c4;
}

}  // namespace stb

using namespace stb;

extern "C" {

int stb_resize_target(int frame_w, int frame_h, int width, int height, int min_flag, int preserve_aspect, int* out_w,
                      int* out_h) {
  // resize_kernel.cpp:43-61, verbatim semantics (integer division included)
  if (frame_w <= 0 || frame_h <= 0 || !out_w || !out_h) { set_error("stb_resize_target: invalid argument"); return STB_ERR_INVALID; }
  int tw = width, th = height;
  if (preserve_aspect) {
    if (tw == 0) tw = frame_w * th / frame_h;
    else th = frame_h * tw / frame_w;
  }
  if (min_flag) {
    if (frame_w <= tw && frame_h <= th) { tw = frame_w; th = frame_h; }
  }
  *out_w = tw; *out_h = th;
  return STB_OK;
}

int stb_resize_interp_code(const char* name) {
  if (!name || !*name) return kInterpLinear;
  const char* names[] = {"INTER_LINEAR", "INTER_NEAREST", "INTER_AREA", "INTER_CUBIC", "INTER_LANCZOS4"};
  for (int i = 0; i < 5; ++i) {
    const char* a = names[i];
    const char* b = name;
    while (*a && *a == *b) { ++a; ++b; }
    if (*a == 0 && *b == 0) return i;
  }
  return -1;
}

int stb_resize_bilinear_u8(const uint8_t* const* d_src, int n, int src_w, int src_h, int channels, uint8_t* const* d_dst,
                           int dst_w, int dst_h, stb_stream_t stream) {
  return stb_resize_u8(d_src, n, src_w, src_h, channels, d_dst, dst_w, dst_h, kInterpLinear, stream);
}

#define STB_RESIZE_DISPATCH(KERNEL, ...)                                                     \
  do {                                                                                       \
    if (channels == 3) stb_launch(KERNEL<3>, grid, dim3(256), 0, s, a, b, __VA_ARGS__);      \
    else if (channels == 1) stb_launch(KERNEL<1>, grid, dim3(256), 0, s, a, b, __VA_ARGS__); \
    else stb_launch(KERNEL<4>, grid, dim3(256), 0, s, a, b, __VA_ARGS__);                    \
  } while (0)

int stb_resize_u8(const uint8_t* const* d_src, int n, int src_w, int src_h, int channels, uint8_t* const* d_dst,
                  int dst_w, int dst_h, int interp, stb_stream_t stream) {
  if (n == 0) return STB_OK;
  if (int rc = check_resize_args("stb_resize_u8", n, src_w, src_h, dst_w, dst_h, channels,
                                 channels == 1 || channels == 3 || channels == 4, "1, 3, 4", interp))
    return rc;
  if (int rc = check_ptr_table(d_src, n, "stb_resize_u8", "source frame")) return rc;
  if (int rc = check_ptr_table(d_dst, n, "stb_resize_u8", "destination frame")) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  const ResizePlan p = plan_resize(interp, src_w, src_h, dst_w, dst_h);
  // INTER_CUBIC / INTER_LANCZOS4: tap tables built here, uploaded and released in stream order
  const int K = interp == kInterpCubic ? 4 : 8;
  TapTables<short> t;
  if (p.path == kPathTaps)
    if (int rc = upload_taps("stb_resize_u8", src_w, src_h, dst_w, dst_h, K, interp == kInterpCubic, tap_coef_u8, s, &t)) return rc;
  const int vec_elems = interp == kInterpCubic ? (dst_w * channels / 8) * 8 : 0;
  const double scale_x = p.scale_x, scale_y = p.scale_y;
  for (int base = 0; base < n; base += kMaxPtrBatch) {
    const int m = n - base < kMaxPtrBatch ? n - base : kMaxPtrBatch;
    const PtrBatch<const uint8_t> a = ptr_chunk(d_src, base, m);
    const PtrBatch<uint8_t> b = ptr_chunk(d_dst, base, m);
    const dim3 grid(ceil_div(dst_w, 32), ceil_div(dst_h, 8), m);
    if (p.path == kPathTaps) {
      if (K == 4) {
        if (channels == 3) stb_launch(resize_taps_u8_kernel<3, 4>, grid, dim3(256), 0, s, a, b, src_w, src_h, dst_w, dst_h, t.xofs, t.xa, t.yofs, t.ya, vec_elems);
        else if (channels == 1) stb_launch(resize_taps_u8_kernel<1, 4>, grid, dim3(256), 0, s, a, b, src_w, src_h, dst_w, dst_h, t.xofs, t.xa, t.yofs, t.ya, vec_elems);
        else stb_launch(resize_taps_u8_kernel<4, 4>, grid, dim3(256), 0, s, a, b, src_w, src_h, dst_w, dst_h, t.xofs, t.xa, t.yofs, t.ya, vec_elems);
      } else {
        if (channels == 3) stb_launch(resize_taps_u8_kernel<3, 8>, grid, dim3(256), 0, s, a, b, src_w, src_h, dst_w, dst_h, t.xofs, t.xa, t.yofs, t.ya, vec_elems);
        else if (channels == 1) stb_launch(resize_taps_u8_kernel<1, 8>, grid, dim3(256), 0, s, a, b, src_w, src_h, dst_w, dst_h, t.xofs, t.xa, t.yofs, t.ya, vec_elems);
        else stb_launch(resize_taps_u8_kernel<4, 8>, grid, dim3(256), 0, s, a, b, src_w, src_h, dst_w, dst_h, t.xofs, t.xa, t.yofs, t.ya, vec_elems);
      }
    }
    else if (p.path == kPathNearest) STB_RESIZE_DISPATCH(resize_nearest_u8_kernel, src_w, src_h, dst_w, dst_h, scale_x, scale_y);
    // exact 2x INTER_LINEAR: (a + b + c + d + 2) >> 2 inside the linear kernel
    else if (p.path == kPathAreaFast && interp == kInterpLinear) STB_RESIZE_DISPATCH(resize_linear_u8_kernel, src_w, src_h, dst_w, dst_h, scale_x, scale_y, 1, 0);
    else if (p.path == kPathAreaFast) STB_RESIZE_DISPATCH(resize_area_int_u8_kernel, src_w, dst_w, dst_h, p.isx, p.isy);
    else if (p.path == kPathArea) STB_RESIZE_DISPATCH(resize_area_u8_kernel, src_w, src_h, dst_w, dst_h, scale_x, scale_y);
    else STB_RESIZE_DISPATCH(resize_linear_u8_kernel, src_w, src_h, dst_w, dst_h, scale_x, scale_y, 0, p.area_coeffs);
    if (cudaPeekAtLastError() != cudaSuccess && t.mem) cudaFreeAsync(t.mem, s);
    STB_CHECK_LAUNCH("resize kernel");
  }
  if (t.mem) STB_CUDA(cudaFreeAsync(t.mem, s));
  return STB_OK;
}

int stb_resize_f32(const float* const* d_src, int n, int src_w, int src_h, int channels, float* const* d_dst, int dst_w,
                   int dst_h, int interp, stb_stream_t stream) {
  const char* who = "stb_resize_f32";
  if (n == 0) return STB_OK;
  if (int rc = check_resize_args(who, n, src_w, src_h, dst_w, dst_h, channels, channels >= 1 && channels <= 4, "1..4", interp))
    return rc;
  if (int rc = check_ptr_table(d_src, n, who, "source frame")) return rc;
  if (int rc = check_ptr_table(d_dst, n, who, "destination frame")) return rc;
  if (int rc = check_float_aligned(d_src, n, who, "source frame")) return rc;
  if (int rc = check_float_aligned(d_dst, n, who, "destination frame")) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  const ResizePlan p = plan_resize(interp, src_w, src_h, dst_w, dst_h);
  TapTables<float> t;
  if (p.path == kPathTaps)
    if (int rc = upload_taps(who, src_w, src_h, dst_w, dst_h, interp == kInterpCubic ? 4 : 8, interp == kInterpCubic, tap_coef_f32, s, &t))
      return rc;
  const int c = channels;
  for (int base = 0; base < n; base += kMaxPtrBatch) {
    const int m = n - base < kMaxPtrBatch ? n - base : kMaxPtrBatch;
    const PtrBatch<const float> a = ptr_chunk(d_src, base, m);
    const PtrBatch<float> b = ptr_chunk(d_dst, base, m);
    const dim3 grid(ceil_div(dst_w, 32), ceil_div(dst_h, 8), m), block(256);
    switch (p.path) {
      case kPathNearest:
        stb_launch(by_channels(c, resize_nearest_f32_kernel<1>, resize_nearest_f32_kernel<2>, resize_nearest_f32_kernel<3>,
                               resize_nearest_f32_kernel<4>),
                   grid, block, 0, s, a, b, src_w, src_h, dst_w, dst_h, p.scale_x, p.scale_y);
        break;
      case kPathAreaFast:
        stb_launch(by_channels(c, resize_area_int_f32_kernel<1>, resize_area_int_f32_kernel<2>, resize_area_int_f32_kernel<3>,
                               resize_area_int_f32_kernel<4>),
                   grid, block, 0, s, a, b, src_w, dst_w, dst_h, p.isx, p.isy);
        break;
      case kPathArea:
        stb_launch(by_channels(c, resize_area_f32_kernel<1>, resize_area_f32_kernel<2>, resize_area_f32_kernel<3>,
                               resize_area_f32_kernel<4>),
                   grid, block, 0, s, a, b, src_w, src_h, dst_w, dst_h, p.scale_x, p.scale_y);
        break;
      case kPathLinear:
        stb_launch(by_channels(c, resize_linear_f32_kernel<1>, resize_linear_f32_kernel<2>, resize_linear_f32_kernel<3>,
                               resize_linear_f32_kernel<4>),
                   grid, block, 0, s, a, b, src_w, src_h, dst_w, dst_h, p.scale_x, p.scale_y, p.area_coeffs);
        break;
      case kPathTaps:
        stb_launch(interp == kInterpCubic
                       ? by_channels(c, resize_taps_f32_kernel<1, 4>, resize_taps_f32_kernel<2, 4>, resize_taps_f32_kernel<3, 4>,
                                     resize_taps_f32_kernel<4, 4>)
                       : by_channels(c, resize_taps_f32_kernel<1, 8>, resize_taps_f32_kernel<2, 8>, resize_taps_f32_kernel<3, 8>,
                                     resize_taps_f32_kernel<4, 8>),
                   grid, block, 0, s, a, b, src_w, src_h, dst_w, dst_h, t.xofs, t.xa, t.yofs, t.ya);
        break;
    }
    if (cudaPeekAtLastError() != cudaSuccess && t.mem) cudaFreeAsync(t.mem, s);
    STB_CHECK_LAUNCH("resize kernel");
  }
  if (t.mem) STB_CUDA(cudaFreeAsync(t.mem, s));
  return STB_OK;
}

}  // extern "C"
