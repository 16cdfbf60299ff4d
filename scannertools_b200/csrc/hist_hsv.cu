// Fused ConvertToHSV -> Histogram (SURVEY §8f rank 3): the HSV variant of the shot-detection
// histogram, scannertools/old/histograms.py:32-36 (ConvertToHSVCPP, old/cpp_ops/imgproc.cpp:14-48,
// then the Histogram op on the HSV frame, histogram_kernel_cpu.cpp:16-46).  The HSV frame is never
// written: each RGB byte is read once, converted in registers with OpenCV's integer tables
// (hsv.cuh) and counted.  Result == stb_hist_rgb16(stb_convert_color_u8(frame, RGB2HSV)).
//
// Counting uses per-LANE private counters (bank == lane), one table of 44 planes per block (H < 180 only
// reaches bins 0..11); updates of different warps are different instructions and serialise in the atomic
// unit anyway.  The two division tables of OpenCV's integer HSV (sdiv[v], hdiv[diff]) are replicated per
// lane as well -- [256][32] words each, 64 KB -- so a look-up is one conflict-free wavefront whatever the 32
// indices are: with one shared copy the random indices of a warp collided on banks, 3.1 wavefronts per
// look-up, which was two thirds of this kernel's shared-memory traffic (round 2 ncu: 12.9 M of 19.7 M).
#include "stb_rt.h"
#include "hsv.cuh"

namespace stb {

constexpr int kHsvThreads = 384;
constexpr int kHsvPlanes = 12 + 16 + 16;                       // H bins 0..11, S, V
constexpr int kHsvPlaneS = 12, kHsvPlaneV = 28;
constexpr int kHsvTableWords = kHsvPlanes * 32;                // 1 408 words = 5.5 KB of counters
constexpr int kHsvDivWords = 256 * 32;                         // one division table, replicated per lane: 32 KB
constexpr int kHsvSmemBytes = (kHsvTableWords + 2 * kHsvDivWords) * 4;   // 71 168 B: three blocks per SM
constexpr int kHsvGroupPx = 16;                                // pixels per thread per step (48 bytes)

__device__ __forceinline__ int hsv_byte(unsigned w, int k) {
#ifdef STB_CPU_EMU
  return (int)((w >> (8 * k)) & 255u);
#else
  return (int)__byte_perm(w, 0u, 0x4440u + (unsigned)k);
#endif
}

// Counter / table addressing.  On the device both are 32-bit shared-window addresses, so one
// counter update is SHF (bin) + LEA (base + bin*128) + RED; the emulator uses plain pointers.
#ifdef STB_CPU_EMU
struct HsvSmem {
  unsigned* my;          // this lane's column of this warp's planes
  const int* sdiv;
  const int* hdiv;
  template <int SHIFT>
  __device__ __forceinline__ void inc(int plane, int x) const { atomicAdd(my + (plane + (x >> SHIFT)) * 32, 1u); }
  __device__ __forceinline__ int s_div(int v) const { return sdiv[v * 32]; }
  __device__ __forceinline__ int h_div(int d) const { return hdiv[d * 32]; }
};
__device__ __forceinline__ HsvSmem hsv_smem(unsigned* sh, unsigned lane, const int* sdiv, const int* hdiv) {
  return HsvSmem{sh + lane, sdiv + lane, hdiv + lane};
}
#else
struct HsvSmem {
  unsigned my, sdiv, hdiv;   // shared-window byte addresses
  // x >> SHIFT selects the bin (x >= 0).  The shift is opaque to the compiler so that it stays
  // SHF + LEA instead of being rewritten into shift-left / mask / add.
  template <int SHIFT>
  __device__ __forceinline__ void inc(int plane, int x) const {
    unsigned bin;
    asm("shr.u32 %0, %1, %2;" : "=r"(bin) : "r"((unsigned)x), "n"(SHIFT));
    asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(my + (unsigned)plane * 128u + (bin << 7)) : "memory");
  }
  __device__ __forceinline__ int s_div(int v) const {
    int r;
    asm volatile("ld.shared.s32 %0, [%1];" : "=r"(r) : "r"(sdiv + ((unsigned)v << 7)));
    return r;
  }
  __device__ __forceinline__ int h_div(int d) const {
    int r;
    asm volatile("ld.shared.s32 %0, [%1];" : "=r"(r) : "r"(hdiv + ((unsigned)d << 7)));
    return r;
  }
};
__device__ __forceinline__ HsvSmem hsv_smem(unsigned* sh, unsigned lane, const int* sdiv, const int* hdiv) {
  const unsigned base = (unsigned)__cvta_generic_to_shared(sh);
  return HsvSmem{base + lane * 4u, (unsigned)__cvta_generic_to_shared(sdiv) + lane * 4u,
                 (unsigned)__cvta_generic_to_shared(hdiv) + lane * 4u};
}
#endif

template <bool SWAP>
__device__ __forceinline__ void hsv_count_px(const HsvSmem& m, int c0, int c1, int c2) {
  const int r = SWAP ? c2 : c0, g = c1, b = SWAP ? c0 : c2;   // SWAP: BGR input
  // hsv_vals (hsv.cuh) with the two table reads going through m
  const int v = max(max(b, g), r), vmin = min(min(b, g), r);
  const int diff = v - vmin;
  const int vr = (v == r) ? -1 : 0, vg = (v == g) ? -1 : 0;
  const int s4096 = diff * m.s_div(v) + (1 << 11);             // s = s4096 >> 12, its bin = s4096 >> 16
  int h = (vr & (g - b)) + (~vr & ((vg & (b - r + 2 * diff)) + ((~vg) & (r - g + 4 * diff))));
  h = (h * m.h_div(diff) + (1 << 11)) >> 12;
  h += h < 0 ? 180 : 0;
  m.inc<4>(0, h);
  m.inc<16>(kHsvPlaneS, s4096);
  m.inc<4>(kHsvPlaneV, v);
}

// 16 pixels held in twelve 32-bit words
template <bool SWAP>
__device__ __forceinline__ void hsv_count_group(const HsvSmem& m, const unsigned (&w)[12]) {
#pragma unroll
  for (int j = 0; j < kHsvGroupPx; ++j) {
    const int b = 3 * j;
    hsv_count_px<SWAP>(m, hsv_byte(w[b >> 2], b & 3), hsv_byte(w[(b + 1) >> 2], (b + 1) & 3),
                       hsv_byte(w[(b + 2) >> 2], (b + 2) & 3));
  }
}

__device__ __forceinline__ void hsv_load_group(const uint8_t* p, bool aligned, unsigned (&w)[12]) {
  if (aligned) {
    const uint4* v = reinterpret_cast<const uint4*>(p);
    const uint4 a = __ldg(v), b = __ldg(v + 1), c = __ldg(v + 2);
    w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w;
    w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
    w[8] = c.x; w[9] = c.y; w[10] = c.z; w[11] = c.w;
  } else {
    // frame base not 16-byte aligned (odd frame sizes inside a packed batch): byte loads
#pragma unroll
    for (int k = 0; k < 12; ++k)
      w[k] = (unsigned)p[4 * k] | ((unsigned)p[4 * k + 1] << 8) | ((unsigned)p[4 * k + 2] << 16) | ((unsigned)p[4 * k + 3] << 24);
  }
}

template <class Addr, bool SWAP>
__global__ void __launch_bounds__(kHsvThreads, 3)
hist_hsv16_kernel(Addr addr, unsigned long long npx, int32_t* __restrict__ out, unsigned base_blocks, unsigned rem) {
  // 1-D grid over (frame, part), as in hist_rgb16_kernel
  unsigned frame, part, nparts;
  flat_grid_decode(blockIdx.x, base_blocks, rem, frame, part, nparts);
  STB_DYN_SMEM(unsigned, sh);
  int* sdiv = reinterpret_cast<int*>(sh + kHsvTableWords);   // [256][32]
  int* hdiv = sdiv + kHsvDivWords;                           // [256][32]
  const unsigned tid = threadIdx.x, lane = tid & 31u;
  {
    uint4* z = reinterpret_cast<uint4*>(sh);
    for (unsigned i = tid; i < kHsvTableWords / 4; i += kHsvThreads) z[i] = make_uint4(0u, 0u, 0u, 0u);
  }
  if (tid < 256u) {
    // thread i computes entry i of both tables (hsv.cuh) and writes it into all 32 lane slots
    const int i = (int)tid;
    const int sv = i ? __double2int_rn((double)(255 << 12) / (double)i) : 0;
    const int hv = i ? __double2int_rn((double)(180 << 12) / (6.0 * (double)i)) : 0;
    const int4 s4 = make_int4(sv, sv, sv, sv), h4 = make_int4(hv, hv, hv, hv);
#pragma unroll
    for (int l = 0; l < 8; ++l) {
      reinterpret_cast<int4*>(sdiv + i * 32)[l] = s4;
      reinterpret_cast<int4*>(hdiv + i * 32)[l] = h4;
    }
  }
  __syncthreads();

  const uint8_t* f = addr(frame);
  const bool aligned = (reinterpret_cast<uintptr_t>(f) & 15u) == 0;
  const HsvSmem m = hsv_smem(sh, lane, sdiv, hdiv);
  const unsigned long long ngroups = npx / kHsvGroupPx;
  const unsigned long long gt = (unsigned long long)part * kHsvThreads + tid;
  const unsigned long long T = (unsigned long long)nparts * kHsvThreads;

  // one group in flight while the previous one is converted and counted
  unsigned long long i = gt;
  if (i < ngroups) {
    unsigned cur[12];
    hsv_load_group(f + i * (3 * kHsvGroupPx), aligned, cur);
    for (i += T; i < ngroups; i += T) {
      unsigned nxt[12];
      hsv_load_group(f + i * (3 * kHsvGroupPx), aligned, nxt);
      hsv_count_group<SWAP>(m, cur);
#pragma unroll
      for (int k = 0; k < 12; ++k) cur[k] = nxt[k];
    }
    hsv_count_group<SWAP>(m, cur);
  }
  // ragged end: fewer than 16 pixels
  if (part == 0) {
    const unsigned long long p = ngroups * kHsvGroupPx + tid;
    if (p < npx) hsv_count_px<SWAP>(m, f[3 * p], f[3 * p + 1], f[3 * p + 2]);
  }
  __syncthreads();

  // block reduce: 8 threads per output bin (bin = ch*16 + b), each sums 4 lanes
  const unsigned bin = tid >> 3, rpart = tid & 7u;
  const unsigned ch = bin >> 4, b = bin & 15u;
  const bool live = !(ch == 0 && b >= 12u);                       // H bins 12..15 stay zero
  const unsigned plane = ch == 0 ? b : (ch == 1 ? kHsvPlaneS + b : kHsvPlaneV + b);
  unsigned s = 0;
  if (live) {
    const uint4 q = *reinterpret_cast<const uint4*>(sh + plane * 32 + rpart * 4);
    s = q.x + q.y + q.z + q.w;
  }
  s += __shfl_xor_sync(0xffffffffu, s, 1);
  s += __shfl_xor_sync(0xffffffffu, s, 2);
  s += __shfl_xor_sync(0xffffffffu, s, 4);
  if (rpart == 0 && s != 0) atomicAdd(out + (size_t)frame * STB_HIST_INTS + bin, (int)s);
}

template <class Addr, bool SWAP>
static int launch_hist_hsv_t(Addr addr, int n, unsigned long long npx, int32_t* d_out, cudaStream_t s) {
  if (int rc = set_max_dyn_smem_once<hist_hsv16_kernel<Addr, SWAP>>(kHsvSmemBytes)) return rc;
  // one resident wave (3 blocks/SM) split over the frames as evenly as possible, never more
  // blocks per frame than there are two-group iterations of work
  const unsigned long long ngroups = npx / kHsvGroupPx;
  const long long max_useful = (long long)((ngroups + (unsigned long long)kHsvThreads * 2 - 1) / ((unsigned long long)kHsvThreads * 2));
  long long total;
  unsigned base_blocks, rem;
  one_wave_split(n, 3, max_useful, &total, &base_blocks, &rem);
  stb_launch(hist_hsv16_kernel<Addr, SWAP>, dim3((unsigned)total), dim3(kHsvThreads), kHsvSmemBytes, s, addr, npx, d_out,
             base_blocks, rem);
  STB_CHECK_LAUNCH("hist_hsv16_kernel");
  return STB_OK;
}

template <class Addr>
static int launch_hist_hsv(Addr addr, int n, unsigned long long npx, bool swap, int32_t* d_out, cudaStream_t s) {
  return swap ? launch_hist_hsv_t<Addr, true>(addr, n, npx, d_out, s) : launch_hist_hsv_t<Addr, false>(addr, n, npx, d_out, s);
}

static int hsv_code_swap(int code, const char* who, bool* swap) {
  const int rgb = stb_color_code("COLOR_RGB2HSV"), bgr = stb_color_code("COLOR_BGR2HSV");
  if (code != rgb && code != bgr) {
    set_error("%s: conversion code %d is not an HSV conversion (COLOR_RGB2HSV / COLOR_BGR2HSV)", who, code);
    return STB_ERR_UNSUPPORTED;
  }
  *swap = code == bgr;
  return STB_OK;
}

}  // namespace stb

using namespace stb;

extern "C" {

int stb_hist_hsv16(const uint8_t* const* d_frames, int n, int width, int height, int code, int32_t* d_out,
                   stb_stream_t stream) {
  if (n == 0) return STB_OK;
  if (!d_out || n < 0 || width <= 0 || height <= 0) {
    set_error("stb_hist_hsv16: invalid argument (n=%d, %dx%d)", n, width, height);
    return STB_ERR_INVALID;
  }
  bool swap = false;
  if (int rc = hsv_code_swap(code, "stb_hist_hsv16", &swap)) return rc;
  if (int rc = check_ptr_table(d_frames, n, "stb_hist_hsv16", "frame")) return rc;
  const unsigned long long npx = (unsigned long long)width * (unsigned long long)height;
  size_t stride = 0;
  if (uniform_stride(d_frames, n, 3 * npx, &stride))
    return stb_hist_hsv16_strided(d_frames[0], stride, n, width, height, code, d_out, stream);
  cudaStream_t s = (cudaStream_t)stream;
  STB_CUDA(cudaMemsetAsync(d_out, 0, (size_t)n * STB_HIST_INTS * sizeof(int32_t), s));
  for (int base = 0; base < n; base += kMaxPtrBatch) {
    const int m = n - base < kMaxPtrBatch ? n - base : kMaxPtrBatch;
    PtrAddr<const uint8_t> a{ptr_chunk(d_frames, base, m)};
    if (int rc = launch_hist_hsv(a, m, npx, swap, d_out + (size_t)base * STB_HIST_INTS, s)) return rc;
  }
  return STB_OK;
}

int stb_hist_hsv16_strided(const uint8_t* d_base, size_t stride_bytes, int n, int width, int height, int code,
                           int32_t* d_out, stb_stream_t stream) {
  if (n == 0) return STB_OK;
  const unsigned long long npx = (unsigned long long)(width > 0 ? width : 0) * (unsigned long long)(height > 0 ? height : 0);
  if (!d_base || !d_out || n < 0 || width <= 0 || height <= 0 || stride_bytes < 3 * npx) {
    set_error("stb_hist_hsv16_strided: invalid argument (n=%d, %dx%d, stride=%zu)", n, width, height, stride_bytes);
    return STB_ERR_INVALID;
  }
  bool swap = false;
  if (int rc = hsv_code_swap(code, "stb_hist_hsv16_strided", &swap)) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  STB_CUDA(cudaMemsetAsync(d_out, 0, (size_t)n * STB_HIST_INTS * sizeof(int32_t), s));
  for (int base = 0; base < n; base += kMaxStridedFrames) {
    const int m = n - base < kMaxStridedFrames ? n - base : kMaxStridedFrames;
    StrideAddr<const uint8_t> a{d_base + (size_t)base * stride_bytes, (unsigned long long)stride_bytes};
    if (int rc = launch_hist_hsv(a, m, npx, swap, d_out + (size_t)base * STB_HIST_INTS, s)) return rc;
  }
  return STB_OK;
}

}  // extern "C"
