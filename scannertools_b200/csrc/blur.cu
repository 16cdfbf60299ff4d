// Blur op: the box blur of the reference's BlurKernel (scannertools_cpp/imgproc/blur_kernel_cpu.cpp) on packed
// 8-bit frames with 1, 3 or 4 channels.  With k = kernel_size, L = ceil(k/2) - 1 and R = k/2, an interior pixel
// (L <= x < W - R, L <= y < H - R) gets, per channel, the unsigned sum of the k x k window [y-L, y+R] x [x-L, x+R]
// divided by k*k with truncation; every other pixel is a copy of the input (the reference leaves those bytes
// unwritten).  The reference's sigma is parsed by the kernel class and never read: this is not a Gaussian.
//
// One CTA owns kBlurTileBytes output bytes of a row (channel-agnostic: horizontal neighbours are C bytes apart)
// and a strip of rows.  Per row it
//   1. updates the running vertical sums of the span it needs, [x0 - L*C, x0 + tile + R*C), in registers: two
//      u16 sums per 32-bit register (a column sum is at most 255 * k <= 65025), incoming row y+R added and row
//      y-L-1, read k rows earlier and still cached, subtracted; the sums go to shared memory as a u16 row;
//   2. sums k taps of that row per output byte (u16 pairs added as 32-bit words while a pair cannot overflow,
//      then widened), divides by k*k with a host-computed multiply-shift and stores 4 bytes per thread;
//      non-interior bytes are copied from the input in the same pass.
// Global loads and stores are aligned 32-bit words, so frames may start at any address: a word that straddles
// the frame's first or last byte is only ever read (it lies in the same 4-byte granule as a frame byte), and
// words the CTA does not own completely are stored byte by byte.
#include "stb_rt.h"

namespace stb {

constexpr int kBlurThreads = 256;
constexpr int kBlurTileBytes = 4 * kBlurThreads;  // output bytes of a row per CTA: one word per thread
constexpr int kBlurMaxK = 255;
// vertical-sum groups (4 bytes each) of a span: the tile, a halo of up to (255 - 1) * 4 bytes and one group for a
// span that does not start on a group boundary
constexpr int kBlurMaxGroups = (kBlurTileBytes + (kBlurMaxK - 1) * 4 + 3) / 4 + 1;
constexpr int kBlurGroupsPerThread = (kBlurMaxGroups + kBlurThreads - 1) / kBlurThreads;

// floor(n / (k*k)) = (n * m) >> s for every n <= 255 * k*k (blur_div_constants)
struct BlurDiv {
  unsigned long long m;
  int s;
};

__device__ __forceinline__ uint32_t blur_div(uint32_t n, BlurDiv d) { return (uint32_t)((n * d.m) >> d.s); }

// the 4 bytes at row byte x (any alignment) as one word, byte i of the word = byte x + i; `aligned`: every row
// start is 4-byte aligned.  `last` is the frame's last aligned word: a funnel load never reads a word past it.
__device__ __forceinline__ uint32_t load_word(const uint8_t* p, bool aligned, const uint8_t* last) {
  if (aligned) return *reinterpret_cast<const uint32_t*>(p);
  const uint8_t* a = reinterpret_cast<const uint8_t*>(reinterpret_cast<uintptr_t>(p) & ~(uintptr_t)3);
  const uint8_t* b = a + 4 <= last ? a + 4 : a;
  const uint32_t w0 = *reinterpret_cast<const uint32_t*>(a), w1 = *reinterpret_cast<const uint32_t*>(b);
  const int sh = (int)(reinterpret_cast<uintptr_t>(p) & 3) * 8;
  return (uint32_t)((((unsigned long long)w1 << 32) | w0) >> sh);
}

// the four u16 vertical sums at u16 index q of the shared row, as pairs (q, q+1) and (q+2, q+3)
__device__ __forceinline__ void load_pairs(const uint32_t* vs, int q, uint32_t& p0, uint32_t& p1) {
  const uint32_t* w = vs + (q >> 1);
  if (q & 1) {
    const uint32_t w0 = w[0], w1 = w[1], w2 = w[2];
    p0 = (w0 >> 16) | (w1 << 16);
    p1 = (w1 >> 16) | (w2 << 16);
  } else {
    p0 = w[0];
    p1 = w[1];
  }
}

// grid: x = tile of row bytes, y = strip of rows, z = frame of this launch
template <int C>
__global__ void __launch_bounds__(kBlurThreads)
blur_kernel(PtrBatch<const uint8_t> srcs, PtrBatch<uint8_t> dsts, int width, int height, int k, int strip_rows,
            int pair_taps, BlurDiv div) {
  __shared__ __align__(16) uint32_t vs_buf[2][kBlurMaxGroups * 2 + 2];
  const uint8_t* src = srcs.p[blockIdx.z];
  uint8_t* dst = dsts.p[blockIdx.z];
  const int row_bytes = width * C;
  const size_t frame_bytes = (size_t)row_bytes * height;
  const uint8_t* last_word =
      reinterpret_cast<const uint8_t*>(reinterpret_cast<uintptr_t>(src + frame_bytes - 1) & ~(uintptr_t)3);
  const bool aligned = ((reinterpret_cast<uintptr_t>(src) | (uintptr_t)row_bytes) & 3) == 0;
  const int L = (k + 1) / 2 - 1, R = k / 2;
  const int x0 = blockIdx.x * kBlurTileBytes;
  const int x_end = min(x0 + kBlurTileBytes, row_bytes);
  // interior bytes of a row, [in_lo, in_hi); empty when the frame is narrower than the window
  const int in_lo = L * C, in_hi = max(width - R, L) * C;
  const int y0 = blockIdx.y * strip_rows, y1 = min(y0 + strip_rows, height);
  const int yi_lo = max(y0, L), yi_hi = min(y1, height - R);  // interior rows of the strip
  // vertical-sum groups: 4 row bytes each, 4g .. 4g+3, over the span the tile's interior outputs read
  const int g_begin = max(x0 - L * C, 0) >> 2;
  const int g_end = (min(x_end + R * C, row_bytes) + 3) >> 2;
  const int t = threadIdx.x;

  uint32_t lo[kBlurGroupsPerThread], hi[kBlurGroupsPerThread];  // bytes 0,2 and 1,3 of each group, u16 each
#pragma unroll
  for (int i = 0; i < kBlurGroupsPerThread; ++i) lo[i] = hi[i] = 0;
  // the k-1 rows above the first interior row, y_first - L .. y_first + R - 1
  if (yi_lo < yi_hi) {
    for (int r = yi_lo - L; r < yi_lo + R; ++r) {
      const uint8_t* row = src + (size_t)r * row_bytes;
#pragma unroll
      for (int i = 0; i < kBlurGroupsPerThread; ++i) {
        const int g = g_begin + t + i * kBlurThreads;
        if (g < g_end) {
          const uint32_t w = load_word(row + 4 * g, aligned, last_word);
          lo[i] += w & 0x00ff00ffu;
          hi[i] += (w >> 8) & 0x00ff00ffu;
        }
      }
    }
  }

  for (int y = y0; y < y1; ++y) {
    const bool interior_row = y >= yi_lo && y < yi_hi;
    uint32_t* vs = vs_buf[y & 1];
    if (interior_row) {
      const uint8_t* in_row = src + (size_t)(y + R) * row_bytes;
      const uint8_t* out_row = src + (size_t)(y - L) * row_bytes;  // leaves the window after this row
#pragma unroll
      for (int i = 0; i < kBlurGroupsPerThread; ++i) {
        const int g = g_begin + t + i * kBlurThreads;
        if (g < g_end) {
          const uint32_t w = load_word(in_row + 4 * g, aligned, last_word);
          lo[i] += w & 0x00ff00ffu;
          hi[i] += (w >> 8) & 0x00ff00ffu;
          // u16 order in shared memory: byte 0 | byte 1 << 16, byte 2 | byte 3 << 16
          reinterpret_cast<uint2*>(vs)[g - g_begin] =
              make_uint2((lo[i] & 0xffffu) | (hi[i] << 16), (lo[i] >> 16) | (hi[i] & 0xffff0000u));
          const uint32_t o = load_word(out_row + 4 * g, aligned, last_word);
          lo[i] -= o & 0x00ff00ffu;
          hi[i] -= (o >> 8) & 0x00ff00ffu;
        }
      }
      __syncthreads();
    }
    const uint8_t* srow = src + (size_t)y * row_bytes;
    uint8_t* drow = dst + (size_t)y * row_bytes;
    // the destination words that hold bytes [x0, x_end) of this row
    const uintptr_t wa = reinterpret_cast<uintptr_t>(drow + x0) & ~(uintptr_t)3;
    const int nwords = (int)((reinterpret_cast<uintptr_t>(drow + x_end) - wa + 3) >> 2);
    const int q_base = -4 * g_begin;  // u16 index in the shared row of row byte 0
    for (int wi = t; wi < nwords; wi += kBlurThreads) {
      const int x = (int)(wa + 4 * (uintptr_t)wi - reinterpret_cast<uintptr_t>(drow));  // row byte of the word's byte 0
      if (interior_row && x >= x0 && x + 4 <= x_end && x >= in_lo && x + 4 <= in_hi) {
        uint32_t a0 = 0, a1 = 0, a2 = 0, a3 = 0;
        int q = q_base + x - L * C;
        for (int j = 0; j < k; j += pair_taps) {
          const int jn = min(j + pair_taps, k);
          uint32_t s0 = 0, s1 = 0;
          for (int jj = j; jj < jn; ++jj, q += C) {
            uint32_t p0, p1;
            load_pairs(vs, q, p0, p1);
            s0 += p0;
            s1 += p1;
          }
          a0 += s0 & 0xffffu;
          a1 += s0 >> 16;
          a2 += s1 & 0xffffu;
          a3 += s1 >> 16;
        }
        *reinterpret_cast<uint32_t*>(drow + x) =
            blur_div(a0, div) | blur_div(a1, div) << 8 | blur_div(a2, div) << 16 | blur_div(a3, div) << 24;
      } else {
        // border bytes, bytes next to the interior's edge and the words shared with another CTA, one by one
        const uint16_t* vs16 = reinterpret_cast<const uint16_t*>(vs);
        for (int b = 0; b < 4; ++b) {
          const int xb = x + b;
          if (xb < x0 || xb >= x_end) continue;
          if (interior_row && xb >= in_lo && xb < in_hi) {
            uint32_t a = 0;
            for (int j = 0, q = q_base + xb - L * C; j < k; ++j, q += C) a += vs16[q];
            drow[xb] = (uint8_t)blur_div(a, div);
          } else {
            drow[xb] = srow[xb];
          }
        }
      }
    }
  }
}

using BlurKernel = void (*)(PtrBatch<const uint8_t>, PtrBatch<uint8_t>, int, int, int, int, int, BlurDiv);

// floor(n / d) = (n * m) >> s for 0 <= n <= 255 d, d = k*k <= 65025: with l = ceil(log2 d), s = 8 + 2l and
// m = ceil(2^s / d) = (2^s + e) / d, 0 <= e < d, n*m / 2^s = n/d + n*e / (d 2^s) and n*e < 2^(8+l) * 2^l = 2^s, so
// the error stays below 1/d and never carries past the next multiple of d.  n*m < 2^50 is a 64-bit product.
static BlurDiv blur_div_constants(int k) {
  const unsigned long long d = (unsigned long long)k * k;
  int l = 0;
  while ((1ull << l) < d) ++l;
  const int s = 8 + 2 * l;
  return BlurDiv{((1ull << s) + d - 1) / d, s};
}

static bool bytes_overlap(const uint8_t* a, const uint8_t* b, size_t n) {
  const uintptr_t x = reinterpret_cast<uintptr_t>(a), y = reinterpret_cast<uintptr_t>(b);
  return x < y + n && y < x + n;
}

}  // namespace stb

using namespace stb;

extern "C" {

int stb_blur_u8(const uint8_t* const* d_src, int n, int width, int height, int channels, int kernel_size,
                uint8_t* const* d_dst, stb_stream_t stream) {
  if (n == 0) return STB_OK;
  if (n < 0 || width <= 0 || height <= 0 || !(channels == 1 || channels == 3 || channels == 4) || kernel_size < 1) {
    set_error("stb_blur_u8: invalid argument (n=%d, %dx%d, channels=%d, kernel_size=%d)", n, width, height, channels,
              kernel_size);
    return STB_ERR_INVALID;
  }
  if (kernel_size > kBlurMaxK) {
    set_error("stb_blur_u8: kernel_size %d is not supported (1..%d)", kernel_size, kBlurMaxK);
    return STB_ERR_UNSUPPORTED;
  }
  if ((long long)width * channels > 0x7fffffffLL - kBlurTileBytes) {
    set_error("stb_blur_u8: rows of %d x %d bytes are not supported", width, channels);
    return STB_ERR_UNSUPPORTED;
  }
  if (int rc = check_ptr_table(d_src, n, "stb_blur_u8", "source frame")) return rc;
  if (int rc = check_ptr_table(d_dst, n, "stb_blur_u8", "destination frame")) return rc;
  const size_t frame_bytes = (size_t)width * channels * height;
  for (int i = 0; i < n; ++i)
    if (bytes_overlap(d_src[i], d_dst[i], frame_bytes)) {
      set_error("stb_blur_u8: destination frame %d overlaps its source frame", i);
      return STB_ERR_INVALID;
    }
  const BlurKernel kernel = channels == 1 ? blur_kernel<1> : channels == 3 ? blur_kernel<3> : blur_kernel<4>;
  const int k = kernel_size;
  // taps whose u16 pair sums cannot overflow: k-row column sums are <= 255 k
  const int pair_taps = max(65535 / (255 * k), 1);
  // strips long enough that the k-1 rows read before a strip's first output row stay a small share
  const int strip_rows = min(max(64, 4 * (k - 1)), height);
  const int tiles = (width * channels + kBlurTileBytes - 1) / kBlurTileBytes;
  const int strips = (height + strip_rows - 1) / strip_rows;
  const BlurDiv div = blur_div_constants(k);
  cudaStream_t s = (cudaStream_t)stream;
  for (int base = 0; base < n; base += kMaxPtrBatch) {
    const int m = n - base < kMaxPtrBatch ? n - base : kMaxPtrBatch;
    stb_launch(kernel, dim3((unsigned)tiles, (unsigned)strips, (unsigned)m), dim3(kBlurThreads), 0, s,
               ptr_chunk(d_src, base, m), ptr_chunk(d_dst, base, m), width, height, k, strip_rows, pair_taps, div);
    STB_CHECK_LAUNCH("blur_kernel");
  }
  return STB_OK;
}

}  // extern "C"
