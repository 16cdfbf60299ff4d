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
#include <cmath>
#include <vector>

#include "stb_rt.h"

namespace stb {

enum { kInterpLinear = 0, kInterpNearest = 1, kInterpArea = 2, kInterpCubic = 3, kInterpLanczos4 = 4 };

__device__ __forceinline__ int cv_round_f(float v) { return __float2int_rn(v); }

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
  const int sx1 = sx + 1 < sw ? sx + 1 : sx;
  const int a0 = cv_round_f(__fmul_rn(1.f - fx, 2048.f)), a1 = cv_round_f(__fmul_rn(fx, 2048.f));
  const int b0 = cv_round_f(__fmul_rn(1.f - fy, 2048.f)), b1 = cv_round_f(__fmul_rn(fy, 2048.f));
  const int y0 = min(max(sy, 0), sh - 1), y1 = min(max(sy + 1, 0), sh - 1);
  const uint8_t* r0 = src + (size_t)y0 * sw * CN;
  const uint8_t* r1 = src + (size_t)y1 * sw * CN;
#pragma unroll
  for (int c = 0; c < CN; ++c) {
    const int h0 = r0[sx * CN + c] * a0 + r0[sx1 * CN + c] * a1;
    const int h1 = r1[sx * CN + c] * a0 + r1[sx1 * CN + c] * a1;
    const int v = (((b0 * (h0 >> 4)) >> 16) + ((b1 * (h1 >> 4)) >> 16) + 2) >> 2;
    dst[c] = (uint8_t)min(max(v, 0), 255);
  }
}

// INTER_NEAREST: sx = min(floor(dx * scale_x), sw - 1) (cv::resizeNN)
template <int CN>
__global__ void __launch_bounds__(256)
resize_nearest_u8_kernel(PtrBatch<const uint8_t> srcs, PtrBatch<uint8_t> dsts, int sw, int sh, int dw, int dh,
                         double scale_x, double scale_y) {
  const int dx = blockIdx.x * 32 + (threadIdx.x & 31);
  const int dy = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (dx >= dw || dy >= dh) return;
  const int sx = min(__double2int_rd(dx * scale_x), sw - 1), sy = min(__double2int_rd(dy * scale_y), sh - 1);
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
    cx[k] = min(max(sx0 + k, 0), sw - 1) * CN;
  }
  int hsum[K][CN];
#pragma unroll
  for (int j = 0; j < K; ++j) {
    const uint8_t* r = src + (size_t)min(max(sy0 + j, 0), sh - 1) * sw * CN;
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

static STB_NO_CONTRACT void build_taps(int dn, int sn, int K, bool cubic, std::vector<int>& ofs, std::vector<short>& al) {
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
    for (int k = 0; k < K; ++k) {
      const float v = c[k] * 2048.f;                                   // saturate_cast<short>(cbuf[k] * INTER_RESIZE_COEF_SCALE)
      const long r = std::lrint(v);                                    // round half to even (default rounding mode)
      al[(size_t)d * K + k] = (short)(r < -32768 ? -32768 : (r > 32767 ? 32767 : r));
    }
  }
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
  if (n < 0 || src_w <= 0 || src_h <= 0 || dst_w <= 0 || dst_h <= 0) {
    set_error("stb_resize_u8: invalid argument (n=%d, %dx%d -> %dx%d)", n, src_w, src_h, dst_w, dst_h);
    return STB_ERR_INVALID;
  }
  if (channels != 1 && channels != 3 && channels != 4) {
    set_error("stb_resize_u8: %d channels not supported (1, 3, 4)", channels);
    return STB_ERR_UNSUPPORTED;
  }
  if (interp < kInterpLinear || interp > kInterpLanczos4) {
    set_error("stb_resize_u8: interpolation %d is not implemented (INTER_LINEAR, INTER_NEAREST, INTER_AREA, INTER_CUBIC, INTER_LANCZOS4)", interp);
    return STB_ERR_UNSUPPORTED;
  }
  if (int rc = check_ptr_table(d_src, n, "stb_resize_u8", "source frame")) return rc;
  if (int rc = check_ptr_table(d_dst, n, "stb_resize_u8", "destination frame")) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  // INTER_CUBIC / INTER_LANCZOS4: tap tables built here, uploaded and released in stream order
  const bool taps = interp == kInterpCubic || interp == kInterpLanczos4;
  const int K = interp == kInterpCubic ? 4 : 8;
  int* d_tab = nullptr;
  const int *d_xofs = nullptr, *d_yofs = nullptr;
  const short *d_xa = nullptr, *d_ya = nullptr;
  if (taps) {
    std::vector<int> xo, yo;
    std::vector<short> xa, ya;
    build_taps(dst_w, src_w, K, interp == kInterpCubic, xo, xa);
    build_taps(dst_h, src_h, K, interp == kInterpCubic, yo, ya);
    // one allocation: [xofs | yofs | xa | ya]
    const size_t n_int = (size_t)dst_w + dst_h, n_short = ((size_t)dst_w + dst_h) * K;
    std::vector<int> host(n_int + (n_short + 1) / 2);
    std::copy(xo.begin(), xo.end(), host.begin());
    std::copy(yo.begin(), yo.end(), host.begin() + dst_w);
    short* hs = reinterpret_cast<short*>(host.data() + n_int);
    std::copy(xa.begin(), xa.end(), hs);
    std::copy(ya.begin(), ya.end(), hs + (size_t)dst_w * K);
    STB_CUDA(cudaMallocAsync(reinterpret_cast<void**>(&d_tab), host.size() * sizeof(int), s));
    // pageable source: the runtime stages it before returning, so `host` may go out of scope
    cudaError_t e = cudaMemcpyAsync(d_tab, host.data(), host.size() * sizeof(int), cudaMemcpyHostToDevice, s);
    if (e != cudaSuccess) { cudaFreeAsync(d_tab, s); return cuda_fail(e, "stb_resize_u8: tap table upload"); }
    d_xofs = d_tab;
    d_yofs = d_tab + dst_w;
    d_xa = reinterpret_cast<const short*>(d_tab + n_int);
    d_ya = d_xa + (size_t)dst_w * K;
  }
  const int vec_elems = interp == kInterpCubic ? (dst_w * channels / 8) * 8 : 0;
  const double scale_x = 1. / ((double)dst_w / src_w), scale_y = 1. / ((double)dst_h / src_h);
  // cv::resize: iscale = saturate_cast<int>(scale) (round half even); "fast area" when both are integers
  const int isx = (int)std::nearbyint(scale_x), isy = (int)std::nearbyint(scale_y);
  const bool int_scale = std::fabs(scale_x - isx) < 2.220446049250313e-16 && std::fabs(scale_y - isy) < 2.220446049250313e-16;
  const bool down = scale_x >= 1 && scale_y >= 1;
  const int area2x = (interp == kInterpLinear && src_w == 2 * dst_w && src_h == 2 * dst_h) ? 1 : 0;
  for (int base = 0; base < n; base += kMaxPtrBatch) {
    const int m = n - base < kMaxPtrBatch ? n - base : kMaxPtrBatch;
    const PtrBatch<const uint8_t> a = ptr_chunk(d_src, base, m);
    const PtrBatch<uint8_t> b = ptr_chunk(d_dst, base, m);
    const dim3 grid(ceil_div(dst_w, 32), ceil_div(dst_h, 8), m);
    if (taps) {
      if (K == 4) {
        if (channels == 3) stb_launch(resize_taps_u8_kernel<3, 4>, grid, dim3(256), 0, s, a, b, src_w, src_h, dst_w, dst_h, d_xofs, d_xa, d_yofs, d_ya, vec_elems);
        else if (channels == 1) stb_launch(resize_taps_u8_kernel<1, 4>, grid, dim3(256), 0, s, a, b, src_w, src_h, dst_w, dst_h, d_xofs, d_xa, d_yofs, d_ya, vec_elems);
        else stb_launch(resize_taps_u8_kernel<4, 4>, grid, dim3(256), 0, s, a, b, src_w, src_h, dst_w, dst_h, d_xofs, d_xa, d_yofs, d_ya, vec_elems);
      } else {
        if (channels == 3) stb_launch(resize_taps_u8_kernel<3, 8>, grid, dim3(256), 0, s, a, b, src_w, src_h, dst_w, dst_h, d_xofs, d_xa, d_yofs, d_ya, vec_elems);
        else if (channels == 1) stb_launch(resize_taps_u8_kernel<1, 8>, grid, dim3(256), 0, s, a, b, src_w, src_h, dst_w, dst_h, d_xofs, d_xa, d_yofs, d_ya, vec_elems);
        else stb_launch(resize_taps_u8_kernel<4, 8>, grid, dim3(256), 0, s, a, b, src_w, src_h, dst_w, dst_h, d_xofs, d_xa, d_yofs, d_ya, vec_elems);
      }
    }
    else if (interp == kInterpNearest) STB_RESIZE_DISPATCH(resize_nearest_u8_kernel, src_w, src_h, dst_w, dst_h, scale_x, scale_y);
    else if (interp == kInterpArea && down && int_scale) STB_RESIZE_DISPATCH(resize_area_int_u8_kernel, src_w, dst_w, dst_h, isx, isy);
    else if (interp == kInterpArea && down) STB_RESIZE_DISPATCH(resize_area_u8_kernel, src_w, src_h, dst_w, dst_h, scale_x, scale_y);
    else STB_RESIZE_DISPATCH(resize_linear_u8_kernel, src_w, src_h, dst_w, dst_h, scale_x, scale_y, area2x, interp == kInterpArea ? 1 : 0);
    if (cudaPeekAtLastError() != cudaSuccess && d_tab) cudaFreeAsync(d_tab, s);
    STB_CHECK_LAUNCH("resize kernel");
  }
  if (d_tab) STB_CUDA(cudaFreeAsync(d_tab, s));
  return STB_OK;
}

}  // extern "C"
