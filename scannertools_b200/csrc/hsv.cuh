// OpenCV's 8-bit integer RGB->HSV (cv::cvtColor COLOR_RGB2HSV / COLOR_BGR2HSV with HUE = 180, H in [0,180);
// COLOR_*2HSV_FULL with HUE = 256, H in [0,256)):
//   sdiv[v] = cvRound(255*4096 / v), hdiv[d] = cvRound(HUE*4096 / (6 d))  (both 0 at index 0)
//   s = (d*sdiv[v] + 2048) >> 12, h = (hnum*hdiv[d] + 2048) >> 12, h += HUE if negative.
// Used by the ConvertColor kernel; the fused HSV histogram restates the same arithmetic.
#pragma once
#include "stb_rt.h"

namespace stb {

// fills sdiv[256] and hdiv[256] (threads 0..255 of the block; the caller synchronises)
template <int HUE>
__device__ __forceinline__ void hsv_tables_init(int* sdiv, int* hdiv, unsigned tid) {
  if (tid < 256u) {
    const int i = (int)tid;
    // cvRound of an exact double quotient: round half to even (no exact ties occur for i < 256)
    sdiv[i] = i ? __double2int_rn((double)(255 << 12) / (double)i) : 0;
    hdiv[i] = i ? __double2int_rn((double)(HUE << 12) / (6.0 * (double)i)) : 0;
  }
}

template <int HUE>
__device__ __forceinline__ void hsv_vals(int r, int g, int b, const int* sdiv, const int* hdiv, int& h, int& s, int& v) {
  v = max(max(b, g), r);
  const int vmin = min(min(b, g), r);
  const int diff = v - vmin;
  const int vr = (v == r) ? -1 : 0, vg = (v == g) ? -1 : 0;
  s = (diff * sdiv[v] + (1 << 11)) >> 12;
  h = (vr & (g - b)) + (~vr & ((vg & (b - r + 2 * diff)) + ((~vg) & (r - g + 4 * diff))));
  h = (h * hdiv[diff] + (1 << 11)) >> 12;
  h += h < 0 ? HUE : 0;
}

}  // namespace stb
