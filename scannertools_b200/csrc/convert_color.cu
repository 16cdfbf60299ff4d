// ConvertColor op (SURVEY §8f rank 3): cv::cvtColor on packed 8-bit frames, bit-exact with OpenCV's integer paths.
// The shipped pipelines use COLOR_RGB2HSV (scannertools/old/cpp_ops/imgproc.cpp:41, behind
// compute_hsv_histograms, old/histograms.py:32-36) and the gray / channel-swap codes of
// scannertools_cpp/imgproc/convert_color_kernel.cpp:24-25,19-20,61; the reference accepts any COLOR_* name, and
// these are the ones with an exact integer definition in OpenCV and an H x W x C frame on both sides:
//   HSV, HSV_FULL: OpenCV's integer path (hsv.cuh), hue range 180 or 256.
//   GRAY: (c0*k0 + c1*k1 + c2*k2 + 16384) >> 15 with the 15-bit coefficients {3735,19235,9798} in B,G,R order.
//   YCrCb, YUV (4:4:4): 14-bit fixed point.  Y = (R*4899 + G*9617 + B*1868 + 2^13) >> 14 -- not the gray value,
//        whose coefficients are 15-bit -- then Cr/V = (R - Y)*{11682, 14369} and Cb/U = (B - Y)*{9241, 8061}, each
//        + (128 << 14) and descaled the same way.  The inverse adds to Y the descaled (Cr - 128)*{22987, 18678}
//        (R), (Cb - 128)*{-5636, -6472} + (Cr - 128)*{-11698, -9519} (G) and (Cb - 128)*{29049, 33292} (B).
//   alpha / channel order: byte moves; an added alpha is 255, a kept one is copied.
// Each conversion is one instantiation of convert_color_kernel, with its channel counts and constants fixed at
// compile time; kConversions maps the public code to it.
#include "stb_rt.h"
#include "hsv.cuh"

namespace stb {

__device__ __forceinline__ int sat_u8(int x) { return min(max(x, 0), 255); }
__device__ __forceinline__ int descale14(int x) { return (x + (1 << 13)) >> 14; }

// A conversion maps the IN bytes of one pixel to its OUT bytes; HUE != 0 means it reads the HSV tables of that
// hue range.  BGR: the colour input (or output, for the inverse colour spaces) is in B,G,R order.
template <int IN, int OUT, int HUE = 0>
struct Conv {
  static constexpr int kIn = IN, kOut = OUT, kHue = HUE;
};

// channel reorder, alpha added (255), dropped or copied
template <int IN, int OUT, bool SWAP>
struct Reorder : Conv<IN, OUT> {
  __device__ static void px(const int (&c)[IN], int (&o)[OUT], const int*, const int*) {
    o[0] = c[SWAP ? 2 : 0];
    o[1] = c[1];
    o[2] = c[SWAP ? 0 : 2];
    if constexpr (OUT == 4) o[3] = IN == 4 ? c[3] : 255;
  }
};

template <int OUT>
struct FromGray : Conv<1, OUT> {
  __device__ static void px(const int (&c)[1], int (&o)[OUT], const int*, const int*) {
    o[0] = o[1] = o[2] = c[0];
    if constexpr (OUT == 4) o[3] = 255;
  }
};

template <int IN, bool BGR>
struct ToGray : Conv<IN, 1> {
  __device__ static void px(const int (&c)[IN], int (&o)[1], const int*, const int*) {
    const int r = c[BGR ? 2 : 0], g = c[1], b = c[BGR ? 0 : 2];
    o[0] = (b * 3735 + g * 19235 + r * 9798 + (1 << 14)) >> 15;
  }
};

template <int HUE, bool BGR>
struct ToHsv : Conv<3, 3, HUE> {
  __device__ static void px(const int (&c)[3], int (&o)[3], const int* sdiv, const int* hdiv) {
    int h, s, v;
    hsv_vals<HUE>(c[BGR ? 2 : 0], c[1], c[BGR ? 0 : 2], sdiv, hdiv, h, s, v);
    o[0] = sat_u8(h);
    o[1] = s;
    o[2] = v;
  }
};

// YCrCb (CRCB) stores Y, Cr, Cb; YUV stores Y, U, V
template <bool CRCB, bool BGR>
struct ToLumaChroma : Conv<3, 3> {
  __device__ static void px(const int (&c)[3], int (&o)[3], const int*, const int*) {
    const int r = c[BGR ? 2 : 0], g = c[1], b = c[BGR ? 0 : 2];
    const int y = descale14(r * 4899 + g * 9617 + b * 1868);
    const int v = sat_u8(descale14((r - y) * (CRCB ? 11682 : 14369) + (128 << 14)));
    const int u = sat_u8(descale14((b - y) * (CRCB ? 9241 : 8061) + (128 << 14)));
    o[0] = y;
    o[1] = CRCB ? v : u;
    o[2] = CRCB ? u : v;
  }
};

template <bool CRCB, bool BGR>
struct FromLumaChroma : Conv<3, 3> {
  __device__ static void px(const int (&c)[3], int (&o)[3], const int*, const int*) {
    const int y = c[0], v = (CRCB ? c[1] : c[2]) - 128, u = (CRCB ? c[2] : c[1]) - 128;
    const int r = sat_u8(y + descale14(v * (CRCB ? 22987 : 18678)));
    const int g = sat_u8(y + descale14(u * (CRCB ? -5636 : -6472) + v * (CRCB ? -11698 : -9519)));
    const int b = sat_u8(y + descale14(u * (CRCB ? 29049 : 33292)));
    o[BGR ? 2 : 0] = r;
    o[1] = g;
    o[BGR ? 0 : 2] = b;
  }
};

template <class Op>
__global__ void __launch_bounds__(256)
convert_color_kernel(PtrBatch<const uint8_t> srcs, PtrBatch<uint8_t> dsts, unsigned long long npx) {
  constexpr int IN = Op::kIn, OUT = Op::kOut;
  __shared__ int sdiv[Op::kHue ? 256 : 1], hdiv[Op::kHue ? 256 : 1];
  if constexpr (Op::kHue != 0) {
    hsv_tables_init<Op::kHue>(sdiv, hdiv, threadIdx.x);
    __syncthreads();
  }
  const uint8_t* src = srcs.p[blockIdx.y];
  uint8_t* dst = dsts.p[blockIdx.y];
  const unsigned long long gt = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned long long T = (unsigned long long)gridDim.x * blockDim.x;
  for (unsigned long long i = gt; i < npx; i += T) {
    int c[IN], o[OUT];
#pragma unroll
    for (int k = 0; k < IN; ++k) c[k] = src[IN * i + k];
    Op::px(c, o, sdiv, hdiv);
#pragma unroll
    for (int k = 0; k < OUT; ++k) dst[OUT * i + k] = (uint8_t)o[k];
  }
}

using ColorKernel = void (*)(PtrBatch<const uint8_t>, PtrBatch<uint8_t>, unsigned long long);

struct ColorConversion {
  const char* name;
  const char* alias;  // OpenCV's other name for the same conversion, or NULL
  ColorKernel kernel;
  int in, out;
};

template <class Op>
ColorConversion conversion(const char* name, const char* alias = nullptr) {
  return ColorConversion{name, alias, convert_color_kernel<Op>, Op::kIn, Op::kOut};
}

// index = the public code (stb_color_code); append only, codes stay below 99
static const ColorConversion kConversions[] = {
    conversion<ToHsv<180, false>>("COLOR_RGB2HSV"),
    conversion<ToHsv<180, true>>("COLOR_BGR2HSV"),
    conversion<ToGray<3, false>>("COLOR_RGB2GRAY"),
    conversion<ToGray<3, true>>("COLOR_BGR2GRAY"),
    conversion<Reorder<3, 3, true>>("COLOR_BGR2RGB", "COLOR_RGB2BGR"),
    conversion<Reorder<3, 4, false>>("COLOR_BGR2BGRA", "COLOR_RGB2RGBA"),
    conversion<Reorder<3, 4, true>>("COLOR_BGR2RGBA", "COLOR_RGB2BGRA"),
    conversion<Reorder<4, 3, false>>("COLOR_BGRA2BGR", "COLOR_RGBA2RGB"),
    conversion<Reorder<4, 3, true>>("COLOR_RGBA2BGR", "COLOR_BGRA2RGB"),
    conversion<Reorder<4, 4, true>>("COLOR_BGRA2RGBA", "COLOR_RGBA2BGRA"),
    conversion<FromGray<3>>("COLOR_GRAY2BGR", "COLOR_GRAY2RGB"),
    conversion<FromGray<4>>("COLOR_GRAY2BGRA", "COLOR_GRAY2RGBA"),
    conversion<ToGray<4, true>>("COLOR_BGRA2GRAY"),
    conversion<ToGray<4, false>>("COLOR_RGBA2GRAY"),
    conversion<ToLumaChroma<true, true>>("COLOR_BGR2YCrCb"),
    conversion<ToLumaChroma<true, false>>("COLOR_RGB2YCrCb"),
    conversion<FromLumaChroma<true, true>>("COLOR_YCrCb2BGR"),
    conversion<FromLumaChroma<true, false>>("COLOR_YCrCb2RGB"),
    conversion<ToLumaChroma<false, true>>("COLOR_BGR2YUV"),
    conversion<ToLumaChroma<false, false>>("COLOR_RGB2YUV"),
    conversion<FromLumaChroma<false, true>>("COLOR_YUV2BGR"),
    conversion<FromLumaChroma<false, false>>("COLOR_YUV2RGB"),
    conversion<ToHsv<256, true>>("COLOR_BGR2HSV_FULL"),
    conversion<ToHsv<256, false>>("COLOR_RGB2HSV_FULL"),
};
constexpr int kNumConversions = (int)(sizeof(kConversions) / sizeof(kConversions[0]));

static bool same_name(const char* a, const char* b) {
  while (*a && *a == *b) { ++a; ++b; }
  return *a == 0 && *b == 0;
}

}  // namespace stb

using namespace stb;

extern "C" {

int stb_color_code(const char* name) {
  if (!name) return -1;
  for (int i = 0; i < kNumConversions; ++i)
    if (same_name(kConversions[i].name, name) || (kConversions[i].alias && same_name(kConversions[i].alias, name)))
      return i;
  return -1;
}

int stb_color_in_channels(int code) { return code >= 0 && code < kNumConversions ? kConversions[code].in : 0; }

int stb_color_out_channels(int code) { return code >= 0 && code < kNumConversions ? kConversions[code].out : 0; }

int stb_convert_color_u8(const uint8_t* const* d_src, int n, int width, int height, int code, uint8_t* const* d_dst,
                         stb_stream_t stream) {
  if (n == 0) return STB_OK;
  if (n < 0 || width <= 0 || height <= 0) {
    set_error("stb_convert_color_u8: invalid argument (n=%d, %dx%d)", n, width, height);
    return STB_ERR_INVALID;
  }
  if (code < 0 || code >= kNumConversions) {
    set_error("stb_convert_color_u8: conversion code %d is not implemented (see stb_color_code)", code);
    return STB_ERR_UNSUPPORTED;
  }
  if (int rc = check_ptr_table(d_src, n, "stb_convert_color_u8", "source frame")) return rc;
  if (int rc = check_ptr_table(d_dst, n, "stb_convert_color_u8", "destination frame")) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  const ColorKernel kernel = kConversions[code].kernel;
  const unsigned long long npx = (unsigned long long)width * height;
  long long blocks = (long long)((npx + 255) / 256);
  for (int base = 0; base < n; base += kMaxPtrBatch) {
    const int m = n - base < kMaxPtrBatch ? n - base : kMaxPtrBatch;
    long long cap = (long long)num_sms() * 8 / m;
    if (cap < 1) cap = 1;
    const long long bx = blocks < cap ? blocks : cap;
    stb_launch(kernel, dim3((unsigned)bx, (unsigned)m), dim3(256), 0, s, ptr_chunk(d_src, base, m),
               ptr_chunk(d_dst, base, m), npx);
    STB_CHECK_LAUNCH("convert_color_kernel");
  }
  return STB_OK;
}

}  // extern "C"
