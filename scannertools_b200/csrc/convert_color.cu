// ConvertColor op (SURVEY §8f rank 3) for the conversions the shipped pipelines use:
// cv::cvtColor(frame, out, COLOR_RGB2HSV) (scannertools/old/cpp_ops/imgproc.cpp:41, behind
// compute_hsv_histograms, old/histograms.py:32-36) and the gray / channel-swap codes of
// scannertools_cpp/imgproc/convert_color_kernel.cpp:24-25,19-20,61.  8-bit, bit-exact with OpenCV:
//   HSV: OpenCV's integer path -- sdiv_table[v] = cvRound(255*4096/v), hdiv_table[d] =
//        cvRound(180*4096/(6 d)), s = (d*sdiv[v] + 2048) >> 12, h from the max channel, +180 if
//        negative (H in [0,180)).
//   GRAY: (c0*k0 + c1*k1 + c2*k2 + 16384) >> 15 with the 15-bit coefficients {3735,19235,9798}
//        in B,G,R order.
#include "stb_rt.h"
#include "hsv.cuh"

namespace stb {

enum { kCodeRGB2HSV = 0, kCodeBGR2HSV = 1, kCodeRGB2GRAY = 2, kCodeBGR2GRAY = 3, kCodeSwapRB = 4 };

__device__ __forceinline__ void hsv_px(int r, int g, int b, const int* sdiv, const int* hdiv, unsigned char* o) {
  int h, s, v;
  hsv_vals(r, g, b, sdiv, hdiv, h, s, v);
  o[0] = (unsigned char)min(max(h, 0), 255);
  o[1] = (unsigned char)s;
  o[2] = (unsigned char)v;
}

__global__ void __launch_bounds__(256)
convert_color_kernel(PtrBatch<const uint8_t> srcs, PtrBatch<uint8_t> dsts, unsigned long long npx, int code) {
  __shared__ int sdiv[256], hdiv[256];
  if (code <= kCodeBGR2HSV) {
    hsv_tables_init(sdiv, hdiv, threadIdx.x);
    __syncthreads();
  }
  const uint8_t* src = srcs.p[blockIdx.y];
  uint8_t* dst = dsts.p[blockIdx.y];
  const unsigned long long gt = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned long long T = (unsigned long long)gridDim.x * blockDim.x;
  for (unsigned long long i = gt; i < npx; i += T) {
    const int c0 = src[3 * i], c1 = src[3 * i + 1], c2 = src[3 * i + 2];
    if (code == kCodeRGB2HSV) hsv_px(c0, c1, c2, sdiv, hdiv, dst + 3 * i);
    else if (code == kCodeBGR2HSV) hsv_px(c2, c1, c0, sdiv, hdiv, dst + 3 * i);
    else if (code == kCodeBGR2GRAY) dst[i] = (uint8_t)((c0 * 3735 + c1 * 19235 + c2 * 9798 + (1 << 14)) >> 15);
    else if (code == kCodeRGB2GRAY) dst[i] = (uint8_t)((c2 * 3735 + c1 * 19235 + c0 * 9798 + (1 << 14)) >> 15);
    else { dst[3 * i] = (uint8_t)c2; dst[3 * i + 1] = (uint8_t)c1; dst[3 * i + 2] = (uint8_t)c0; }
  }
}

}  // namespace stb

using namespace stb;

extern "C" {

int stb_color_code(const char* name) {
  if (!name) return -1;
  const char* names[] = {"COLOR_RGB2HSV", "COLOR_BGR2HSV", "COLOR_RGB2GRAY", "COLOR_BGR2GRAY", "COLOR_BGR2RGB", "COLOR_RGB2BGR"};
  const int codes[] = {kCodeRGB2HSV, kCodeBGR2HSV, kCodeRGB2GRAY, kCodeBGR2GRAY, kCodeSwapRB, kCodeSwapRB};
  for (int i = 0; i < 6; ++i) {
    const char* a = names[i];
    const char* b = name;
    while (*a && *a == *b) { ++a; ++b; }
    if (*a == 0 && *b == 0) return codes[i];
  }
  return -1;
}

int stb_color_out_channels(int code) {
  if (code == kCodeRGB2GRAY || code == kCodeBGR2GRAY) return 1;
  if (code >= 0 && code <= kCodeSwapRB) return 3;
  return 0;
}

int stb_convert_color_u8(const uint8_t* const* d_src, int n, int width, int height, int code, uint8_t* const* d_dst,
                         stb_stream_t stream) {
  if (n == 0) return STB_OK;
  if (n < 0 || width <= 0 || height <= 0) {
    set_error("stb_convert_color_u8: invalid argument (n=%d, %dx%d)", n, width, height);
    return STB_ERR_INVALID;
  }
  if (code < 0 || code > kCodeSwapRB) {
    set_error("stb_convert_color_u8: conversion code %d is not implemented (RGB/BGR2HSV, RGB/BGR2GRAY, RGB<->BGR)", code);
    return STB_ERR_UNSUPPORTED;
  }
  if (int rc = check_ptr_table(d_src, n, "stb_convert_color_u8", "source frame")) return rc;
  if (int rc = check_ptr_table(d_dst, n, "stb_convert_color_u8", "destination frame")) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  const unsigned long long npx = (unsigned long long)width * height;
  long long blocks = (long long)((npx + 255) / 256);
  for (int base = 0; base < n; base += kMaxPtrBatch) {
    const int m = n - base < kMaxPtrBatch ? n - base : kMaxPtrBatch;
    long long cap = (long long)num_sms() * 8 / m;
    if (cap < 1) cap = 1;
    const long long bx = blocks < cap ? blocks : cap;
    stb_launch(convert_color_kernel, dim3((unsigned)bx, (unsigned)m), dim3(256), 0, s, ptr_chunk(d_src, base, m),
               ptr_chunk(d_dst, base, m), npx, code);
    STB_CHECK_LAUNCH("convert_color_kernel");
  }
  return STB_OK;
}

}  // extern "C"
