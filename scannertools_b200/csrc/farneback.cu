// Dense Farneback optical flow for sm_100a -- the OpticalFlow op's arithmetic.
//
// Replaces cv::cvtColor(BGR2GRAY) + cv::FarnebackOpticalFlow(3, .5, false, 15, 3, 5, 1.2, 0)
// ::calc as called by scannertools_cpp/imgproc/optical_flow_kernel_cpu.cpp:36-41 (and the
// cv::cuda variant, optical_flow_kernel_gpu.cpp:66-89).  Algorithm = SURVEY.md Appendix A.
// This is a from-scratch design, not a port of OpenCV's cudaoptflow:
//
//   * planar (SoA) 5-channel polynomial-expansion arrays R and matrix arrays M, so every
//     global access of a warp is a contiguous run of floats (the CPU code's 5-float
//     interleaved pixels are hostile to coalescing);
//   * each pyramid level is produced straight from the full-resolution gray plane by one
//     kernel (separable Gaussian evaluated only at the columns/rows the bilinear
//     down-sampler needs), no intermediate full-resolution blurred image exists;
//   * one fused kernel per displacement-update iteration: 15x15 box sums of the 5 M planes
//     (pairwise-doubling window sums, no subtract recurrence) -> 2x2 solve -> new
//     flow -> bilinear gather of R1 -> next M, so M is read once and written once per
//     iteration and the flow of inner iterations never touches HBM;
//   * frames are processed level-major, a whole batch of pairs per launch (grid.z), so every
//     launch is many waves deep and the small pyramid levels are not launch-bound;
//   * polynomial expansions are computed once per frame and shared by the two pairs that
//     contain it (the reference recomputes both pyramids for every pair).
#include "stb_rt.h"
#include "flow_bins.cuh"

#include <cmath>
#include <cstdlib>
#include <cstring>
#include <new>
#include <vector>

namespace stb {

constexpr int kMaxScales = 4;     // numLevels = 3 -> up to 4 scales (Appendix A.1)
constexpr int kMaxGaussTaps = 19; // sigma 3.5 -> ksize 19
constexpr int kPolyN = 5;

constexpr int kMaxPolyN = 7;   // polyN = 5 (the reference) has the tiled kernel; 3..7 run a generic one
struct PolyConsts {
  float g[kMaxPolyN + 1], xg[kMaxPolyN + 1], xxg[kMaxPolyN + 1];
  float ig11, ig03, ig33, ig55;
  // the taps duplicated into (t, t) pairs: 64-bit constant-bank operands of the packed f32x2 vertical pass
  float2 g2[kMaxPolyN + 1], xg2[kMaxPolyN + 1], xxg2[kMaxPolyN + 1];
};

// packed f32x2 arithmetic (sm_100a FADD2 / FMUL2 / FFMA2): two independent IEEE single-precision operations per
// instruction, same rounding as the scalar forms
__device__ __forceinline__ float2 f2add(float2 a, float2 b) {
#ifdef STB_CPU_EMU
  return make_float2(a.x + b.x, a.y + b.y);
#else
  unsigned long long ra, rb, rc;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(rc) : "l"(ra), "l"(rb));
  float2 r;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(rc));
  return r;
#endif
}
__device__ __forceinline__ float2 f2sub(float2 a, float2 b) {
#ifdef STB_CPU_EMU
  return make_float2(a.x - b.x, a.y - b.y);
#else
  unsigned long long ra, rb, rc;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(rc) : "l"(ra), "l"(rb));
  float2 r;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(rc));
  return r;
#endif
}
__device__ __forceinline__ float2 f2mul(float2 a, float2 b) {
#ifdef STB_CPU_EMU
  return make_float2(a.x * b.x, a.y * b.y);
#else
  unsigned long long ra, rb, rc;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(rc) : "l"(ra), "l"(rb));
  float2 r;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(rc));
  return r;
#endif
}
__device__ __forceinline__ float2 f2fma(float2 a, float2 b, float2 c) {   // a * b + c
#ifdef STB_CPU_EMU
  return make_float2(fmaf(a.x, b.x, c.x), fmaf(a.y, b.y, c.y));
#else
  unsigned long long ra, rb, rc, rd;
  asm("mov.b64 %0, {%1, %2};" : "=l"(ra) : "f"(a.x), "f"(a.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rb) : "f"(b.x), "f"(b.y));
  asm("mov.b64 %0, {%1, %2};" : "=l"(rc) : "f"(c.x), "f"(c.y));
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(rd) : "l"(ra), "l"(rb), "l"(rc));
  float2 r;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(r.x), "=f"(r.y) : "l"(rd));
  return r;
#endif
}

struct PyrParams {
  int W, H;          // full resolution
  int w, h;          // this level
  int r;             // Gaussian radius (ksize = 2r+1)
  int max_rows;      // rows of the shared-memory strip
  double scale_x, scale_y;  // W / w, H / h  (cv::resize's 1/inv_scale)
  float taps[kMaxGaussTaps];
};

// ---------------------------------------------------------------------------------------------
// gray: COLOR_BGR2GRAY fixed point applied to the RGB bytes as they lie in memory
// (optical_flow_kernel_cpu.cpp:38-39; SURVEY Appendix B).  16 pixels (48 B in, 16 B out) per
// thread iteration with 16-byte accesses when the frame base is 16-byte aligned.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned gray_of(unsigned c0, unsigned c1, unsigned c2) {
  return (c0 * 3735u + c1 * 19235u + c2 * 9798u + (1u << 14)) >> 15;
}

__global__ void __launch_bounds__(256)
gray_kernel(PtrBatch<const uint8_t> frames, uint8_t* __restrict__ gray, unsigned long long npx) {
  const uint8_t* f = frames.p[blockIdx.y];
  uint8_t* g = gray + (unsigned long long)blockIdx.y * npx;
  const unsigned long long gt = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned long long T = (unsigned long long)gridDim.x * blockDim.x;
  unsigned long long done = 0;
  if (((reinterpret_cast<uintptr_t>(f) | reinterpret_cast<uintptr_t>(g)) & 15u) == 0) {
    const unsigned long long ngroups = npx >> 4;
    const uint4* v = reinterpret_cast<const uint4*>(f);
    uint4* o = reinterpret_cast<uint4*>(g);
    for (unsigned long long i = gt; i < ngroups; i += T) {
      const uint4 a = __ldg(v + 3 * i), b = __ldg(v + 3 * i + 1), c = __ldg(v + 3 * i + 2);
      const unsigned wd[12] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, c.x, c.y, c.z, c.w};
      unsigned res[4];
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        unsigned packed = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const int px = q * 4 + k;  // pixel within the group; bytes 3px, 3px+1, 3px+2
          const int b0 = 3 * px, b1 = 3 * px + 1, b2 = 3 * px + 2;
          const unsigned c0 = (wd[b0 >> 2] >> ((b0 & 3) * 8)) & 0xffu;
          const unsigned c1 = (wd[b1 >> 2] >> ((b1 & 3) * 8)) & 0xffu;
          const unsigned c2 = (wd[b2 >> 2] >> ((b2 & 3) * 8)) & 0xffu;
          packed |= gray_of(c0, c1, c2) << (8 * k);
        }
        res[q] = packed;
      }
      o[i] = make_uint4(res[0], res[1], res[2], res[3]);
    }
    done = ngroups << 4;
  }
  for (unsigned long long i = done + gt; i < npx; i += T)
    g[i] = (uint8_t)gray_of(f[3 * i], f[3 * i + 1], f[3 * i + 2]);
}

// ---------------------------------------------------------------------------------------------
// pyramid level: I_k = resize_bilinear(GaussianBlur(float(gray), ksize_k, sigma_k), (w_k, h_k))
// (Appendix A.2).  Tile = 32 x 8 outputs.  Phase 1 evaluates, for every source row the tile
// needs, the horizontally blurred + horizontally interpolated value at the tile's 32 output
// columns (REFLECT_101 in x) into shared memory; phase 2 blurs vertically and interpolates in
// y (REFLECT_101 in y is applied when a row is stored in phase 1).
// ---------------------------------------------------------------------------------------------
constexpr int kPyrTW = 32, kPyrTH = 8, kPyrThreads = 256;

__device__ __forceinline__ int reflect101(int i, int n) {
  // OpenCV BORDER_REFLECT_101; |overshoot| < n for every kernel used here
  if (n == 1) return 0;
  if (i < 0) i = -i;
  if (i >= n) i = 2 * (n - 1) - i;
  if (i < 0) i = -i;
  return i < n ? i : n - 1;
}

__device__ __forceinline__ void resize_src(int d, double scale, int n_src, int& s, float& f) {
  // cv::resize INTER_LINEAR source coordinate for destination index d
  f = (float)((d + 0.5) * scale - 0.5);
  s = __float2int_rd(f);
  f -= (float)s;
  if (s < 0) { s = 0; f = 0.f; }
  if (s >= n_src - 1) { s = n_src - 1; f = 0.f; }
}

__global__ void __launch_bounds__(kPyrThreads)
pyr_kernel(const uint8_t* __restrict__ gray, float* __restrict__ I, PyrParams p, int frame0) {
  STB_DYN_SMEM(float, hx);  // [max_rows][32]
  __shared__ float taps[kMaxGaussTaps];
  const int tid = threadIdx.x;
  if (tid < kMaxGaussTaps) taps[tid] = p.taps[tid];
  __syncthreads();
  const int frame = frame0 + blockIdx.z;
  const uint8_t* G = gray + (size_t)frame * p.W * p.H;
  float* out = I + (size_t)frame * p.w * p.h;
  const int ox0 = blockIdx.x * kPyrTW, oy0 = blockIdx.y * kPyrTH;
  const int oy_last = min(oy0 + kPyrTH - 1, p.h - 1);
  int sy_first, sy_last; float fdummy;
  resize_src(oy0, p.scale_y, p.H, sy_first, fdummy);
  resize_src(oy_last, p.scale_y, p.H, sy_last, fdummy);
  const int row_lo = sy_first - p.r;
  const int nrows = min(sy_last + 1 + p.r - row_lo + 1, p.max_rows);

  // phase 1
  {
    const int ox = tid & 31;
    const int x = ox0 + ox;
    int sx = 0; float fx = 0.f;
    if (x < p.w) resize_src(x, p.scale_x, p.W, sx, fx);
    for (int rr = tid >> 5; rr < nrows; rr += kPyrThreads / 32) {
      float v = 0.f;
      if (x < p.w) {
        const uint8_t* row = G + (size_t)reflect101(row_lo + rr, p.H) * p.W;
        float a = 0.f, b = 0.f;
        for (int t = 0; t <= 2 * p.r; ++t) a = fmaf(taps[t], (float)row[reflect101(sx + t - p.r, p.W)], a);
        if (fx != 0.f)
          for (int t = 0; t <= 2 * p.r; ++t) b = fmaf(taps[t], (float)row[reflect101(sx + 1 + t - p.r, p.W)], b);
        v = a * (1.f - fx) + b * fx;
      }
      hx[rr * kPyrTW + ox] = v;
    }
  }
  __syncthreads();
  // phase 2
  {
    const int ox = tid & 31, oy = oy0 + (tid >> 5);
    const int x = ox0 + ox;
    if (x < p.w && oy < p.h) {
      int sy; float fy;
      resize_src(oy, p.scale_y, p.H, sy, fy);
      const int base = sy - p.r - row_lo;  // >= 0 by construction
      float a = 0.f, b = 0.f;
      for (int t = 0; t <= 2 * p.r; ++t) a = fmaf(taps[t], hx[(base + t) * kPyrTW + ox], a);
      if (fy != 0.f)
        for (int t = 0; t <= 2 * p.r; ++t) b = fmaf(taps[t], hx[(base + 1 + t) * kPyrTW + ox], b);
      out[(size_t)oy * p.w + x] = a * (1.f - fy) + b * fy;
    }
  }
}

// ---------------------------------------------------------------------------------------------
// pyramid levels 1..3 when the level size is exactly (W / 2^K, H / 2^K) -- the common case
// (1080p, 720p, 640x480 ...).  cv::resize's bilinear taps are then exactly (0.5, 0.5) at source
// offset S*o + S/2 - 1, so Gaussian + down-sampling collapse into ONE separable FIR of
// 2r+2 merged taps c[t] = (g[t] + g[t-1]) / 2 evaluated at stride S = 2^K.
// Tile = 32 x 16 outputs (32 x 8 for K = 3).  The u8 source region is staged in shared memory with aligned 4-byte
// loads (interior tiles) or per-byte REFLECT_101 (tiles touching the left/right image edge);
// phase 1 = horizontal FIR at the 32 output columns for every staged row, phase 2 = vertical FIR.
// ---------------------------------------------------------------------------------------------
struct MergedTaps { float c[kMaxGaussTaps + 1]; };

template <int K>
__global__ void __launch_bounds__(256)
pyr_pow2_kernel(const uint8_t* __restrict__ gray, float* __restrict__ I, int W, int H, MergedTaps mt, int frame0) {
  constexpr int S = 1 << K;
  constexpr int RAD = (K == 1) ? 1 : (K == 2 ? 4 : 9);
  constexpr int NT = 2 * RAD + 2;
  constexpr int TH = (K == 3) ? 8 : 16;                      // output rows per tile (K = 3 would need 56 KB of shared memory at 16)
  constexpr int NROWS = NT + S * (TH - 1);
  constexpr int LEAD = 8 - (RAD + 1 - S / 2);                 // byte offset of the first tap inside the aligned region
  constexpr int PITCH = ((LEAD + NT + S * 31) + 3) & ~3;      // bytes per staged row
  __shared__ __align__(16) uint8_t g8[NROWS * PITCH];
  __shared__ float hx[NROWS][32];
  __shared__ float taps[NT];

  const int tid = threadIdx.x;
  const int w = W >> K, h = H >> K;
  const int frame = frame0 + blockIdx.z;
  const uint8_t* G = gray + (size_t)frame * W * H;
  float* out = I + (size_t)frame * w * h;
  const int ox0 = blockIdx.x * 32, oy0 = blockIdx.y * TH;
  const int a_lo = S * ox0 - 8;                                // aligned first staged column
  const int r_lo = S * oy0 + S / 2 - 1 - RAD;                  // first staged row
  if (tid < NT) taps[tid] = mt.c[tid];

  // Staging.  W is a multiple of S (>= 2) here; when it is also a multiple of 4 every aligned
  // 4-byte word of a row lies entirely inside or entirely outside [0, W): inside words are one
  // aligned load, the few outside words (tiles touching the left / right edge) are rebuilt byte
  // by byte through REFLECT_101.
  constexpr int WPR = PITCH / 4;
  if ((W & 3) == 0) {
    for (int idx = tid; idx < NROWS * WPR; idx += 256) {
      const int rr = idx / WPR, wc = idx - rr * WPR;
      const int y = reflect101(r_lo + rr, H);
      const int c0 = a_lo + 4 * wc;
      const uint8_t* row = G + (size_t)y * W;
      unsigned v;
      if (c0 >= 0 && c0 + 3 < W) {
        v = __ldg(reinterpret_cast<const unsigned*>(row + c0));
      } else {
        v = (unsigned)__ldg(row + reflect101(c0, W)) | ((unsigned)__ldg(row + reflect101(c0 + 1, W)) << 8) |
            ((unsigned)__ldg(row + reflect101(c0 + 2, W)) << 16) | ((unsigned)__ldg(row + reflect101(c0 + 3, W)) << 24);
      }
      reinterpret_cast<unsigned*>(g8)[idx] = v;
    }
  } else {
    for (int idx = tid; idx < NROWS * PITCH; idx += 256) {
      const int rr = idx / PITCH, bc = idx - rr * PITCH;
      const int y = reflect101(r_lo + rr, H);
      g8[idx] = __ldg(G + (size_t)y * W + reflect101(a_lo + bc, W));
    }
  }
  __syncthreads();
  {
    const int ox = tid & 31;
    const uint8_t* base = g8 + LEAD + S * ox;
    for (int rr = tid >> 5; rr < NROWS; rr += 8) {
      const uint8_t* row = base + rr * PITCH;
      float a = 0.f;
#pragma unroll
      for (int t = 0; t < NT; ++t) a = fmaf(taps[t], (float)row[t], a);
      hx[rr][ox] = a;
    }
  }
  __syncthreads();
  {
    const int ox = tid & 31;
    const int x = ox0 + ox;
#pragma unroll
    for (int oyl = tid >> 5; oyl < TH; oyl += 8) {
      const int y = oy0 + oyl;
      if (x < w && y < h) {
        float a = 0.f;
#pragma unroll
        for (int t = 0; t < NT; ++t) a = fmaf(taps[t], hx[S * oyl + t][ox], a);
        out[(size_t)y * w + x] = a;
      }
    }
  }
}

// ---------------------------------------------------------------------------------------------
// Levels 1..3 in TWO launches when every level is an exact power-of-two size and W % 32 == 0 (1080p,
// 720p, 640x480, 4K): the same merged-tap separable FIRs as pyr_pow2_kernel, evaluated in the same
// fmaf order (bit-identical I_k), but
//   * pyr_h_kernel reads the gray plane ONCE for all three levels: a thread owns 32 source pixels
//     of one row (+ 8 either side), converts its 48 bytes to float once, and emits the horizontal
//     FIR of that row at the 16 / 8 / 4 output columns of levels 1 / 2 / 3 (taps are kernel
//     parameters, i.e. constant-bank FFMA operands) into a narrow intermediate Hx_K [H][w_K];
//   * pyr_v_kernel runs the three vertical FIRs (4 outputs per thread, 16-byte loads) over it.
// pyr_pow2_kernel re-did the horizontal FIR per 8/16-row tile, per level, with one LDS.U8 + I2F per
// tap: 144 us per 17 1080p frames; these two: 72 us.
// ---------------------------------------------------------------------------------------------
struct PyrTaps3 { float c1[4], c2[10], c3[20]; };

__device__ __forceinline__ void unpack4(unsigned wd, float* f) {
  f[0] = (float)(wd & 0xffu); f[1] = (float)((wd >> 8) & 0xffu); f[2] = (float)((wd >> 16) & 0xffu); f[3] = (float)(wd >> 24);
}

__global__ void __launch_bounds__(128)
pyr_h_kernel(const uint8_t* __restrict__ gray, float* __restrict__ Hx, int W, int H, PyrTaps3 tp, int nlev, int frame0) {
  const int nseg = W >> 5;
  const int item = blockIdx.x * 128 + threadIdx.x;
  if (item >= nseg * H) return;
  const int y = item / nseg, seg = item - y * nseg;
  const int frame = frame0 + blockIdx.y;
  const uint8_t* row = gray + ((size_t)frame * H + y) * W;
  const int x0 = seg * 32;
  float v[48];                      // v[j] = gray[x0 - 8 + j] with REFLECT_101 at the row ends
  {
    // The 8 bytes left of the first segment / right of the last one lie outside the row: they are not loaded
    // but mirrored from the segment's own bytes (REFLECT_101: x = -i -> i, x = W - 1 + i -> W - 1 - i), with
    // predicated register moves -- no divergent per-byte path (a warp of 32 consecutive (row, segment) items
    // crosses a row end every W / 32 items, so half the warps used to execute both paths).
    const bool first = seg == 0, last = seg == nseg - 1;
    uint2 a = make_uint2(0u, 0u), d = make_uint2(0u, 0u);
    if (!first) a = __ldg(reinterpret_cast<const uint2*>(row + x0 - 8));
    const uint4 b = __ldg(reinterpret_cast<const uint4*>(row + x0));
    const uint4 c = __ldg(reinterpret_cast<const uint4*>(row + x0 + 16));
    if (!last) d = __ldg(reinterpret_cast<const uint2*>(row + x0 + 32));
    unpack4(a.x, v); unpack4(a.y, v + 4);
    unpack4(b.x, v + 8); unpack4(b.y, v + 12); unpack4(b.z, v + 16); unpack4(b.w, v + 20);
    unpack4(c.x, v + 24); unpack4(c.y, v + 28); unpack4(c.z, v + 32); unpack4(c.w, v + 36);
    unpack4(d.x, v + 40); unpack4(d.y, v + 44);
    if (first) {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = v[16 - j];
    }
    if (last) {
#pragma unroll
      for (int k = 40; k < 48; ++k) v[k] = v[78 - k];
    }
  }
  // frame-major intermediate: [frame][level-1 rows | level-2 rows | level-3 rows]
  const int w1 = W >> 1, w2 = W >> 2, w3 = W >> 3;
  float* base = Hx + (size_t)frame * H * (w1 + w2 + w3);
  {   // level 1: S = 2, 4 taps, first tap of output o at source 2o - 1
    float* o = base + (size_t)y * w1 + seg * 16;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      float r[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float a = 0.f;
#pragma unroll
        for (int t = 0; t < 4; ++t) a = fmaf(tp.c1[t], v[8 + 2 * (4 * q + i) - 1 + t], a);
        r[i] = a;
      }
      *reinterpret_cast<float4*>(o + 4 * q) = make_float4(r[0], r[1], r[2], r[3]);
    }
  }
  if (nlev >= 2) {   // level 2: S = 4, 10 taps, first tap at 4o - 3
    float* o = base + (size_t)H * w1 + (size_t)y * w2 + seg * 8;
#pragma unroll
    for (int q = 0; q < 2; ++q) {
      float r[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float a = 0.f;
#pragma unroll
        for (int t = 0; t < 10; ++t) a = fmaf(tp.c2[t], v[8 + 4 * (4 * q + i) - 3 + t], a);
        r[i] = a;
      }
      *reinterpret_cast<float4*>(o + 4 * q) = make_float4(r[0], r[1], r[2], r[3]);
    }
  }
  if (nlev >= 3) {   // level 3: S = 8, 20 taps, first tap at 8o - 6
    float* o = base + (size_t)H * (w1 + w2) + (size_t)y * w3 + seg * 4;
    float r[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float a = 0.f;
#pragma unroll
      for (int t = 0; t < 20; ++t) a = fmaf(tp.c3[t], v[8 + 8 * i - 6 + t], a);
      r[i] = a;
    }
    *reinterpret_cast<float4*>(o) = make_float4(r[0], r[1], r[2], r[3]);
  }
}

// vertical FIRs: one thread = 4 adjacent outputs of one level; blockIdx.x walks the quads of
// level 1, then level 2, then level 3.  I_k of frame f lives at I + f * stride_f + off_k.
template <int K>
__device__ __forceinline__ void pyr_v_quad(const float* __restrict__ hx, float* __restrict__ out, int wK, int H, int q,
                                           const float* taps) {
  constexpr int S = 1 << K;
  constexpr int RAD = (K == 1) ? 1 : (K == 2 ? 4 : 9);
  constexpr int NT = 2 * RAD + 2;
  const int qpr = wK >> 2;                      // quads per row
  const int oy = q / qpr, ox = (q - oy * qpr) * 4;
  const int r_lo = S * oy + S / 2 - 1 - RAD;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  if (r_lo >= 0 && r_lo + NT - 1 < H) {          // interior rows (warp-uniform: a warp's quads share oy): no reflection
    const float* p = hx + (size_t)r_lo * wK + ox;
#pragma unroll
    for (int t = 0; t < NT; ++t) {
      const float4 h = __ldg(reinterpret_cast<const float4*>(p + (size_t)t * wK));
      a0 = fmaf(taps[t], h.x, a0); a1 = fmaf(taps[t], h.y, a1); a2 = fmaf(taps[t], h.z, a2); a3 = fmaf(taps[t], h.w, a3);
    }
  } else {
#pragma unroll
    for (int t = 0; t < NT; ++t) {
      const float4 h = __ldg(reinterpret_cast<const float4*>(hx + (size_t)reflect101(r_lo + t, H) * wK + ox));
      a0 = fmaf(taps[t], h.x, a0); a1 = fmaf(taps[t], h.y, a1); a2 = fmaf(taps[t], h.z, a2); a3 = fmaf(taps[t], h.w, a3);
    }
  }
  *reinterpret_cast<float4*>(out + (size_t)oy * wK + ox) = make_float4(a0, a1, a2, a3);
}

__global__ void __launch_bounds__(128)
pyr_v_kernel(const float* __restrict__ Hx, float* __restrict__ I, int W, int H, PyrTaps3 tp, int nlev, size_t frame_stride,
             int frame0) {
  const int w1 = W >> 1, w2 = W >> 2, w3 = W >> 3;
  const int n1 = (w1 >> 2) * (H >> 1), n2 = nlev >= 2 ? (w2 >> 2) * (H >> 2) : 0, n3 = nlev >= 3 ? (w3 >> 2) * (H >> 3) : 0;
  const int frame = frame0 + blockIdx.y;
  const float* hx = Hx + (size_t)frame * H * (w1 + w2 + w3);
  float* out = I + (size_t)frame * frame_stride;
  int q = blockIdx.x * 128 + threadIdx.x;
  if (q < n1) { pyr_v_quad<1>(hx, out, w1, H, q, tp.c1); return; }
  q -= n1;
  if (q < n2) { pyr_v_quad<2>(hx + (size_t)H * w1, out + (size_t)w1 * (H >> 1), w2, H, q, tp.c2); return; }
  q -= n2;
  if (q < n3) pyr_v_quad<3>(hx + (size_t)H * (w1 + w2), out + (size_t)w1 * (H >> 1) + (size_t)w2 * (H >> 2), w3, H, q, tp.c3);
}

// ---------------------------------------------------------------------------------------------
// level 0 of the pyramid: 3x3 separable Gaussian (taps t0,t1,t2; REFLECT_101), no resize.
// Each thread produces a 4 (x) by 4 (y) patch: 6 source rows x (one aligned 4-byte load + the
// two neighbouring bytes), horizontal blur per row, vertical combine, float4 stores.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
pyr0_kernel(const uint8_t* __restrict__ gray, float* __restrict__ I, int W, int H, float t0, float t1, float t2,
            int frame0, int vec_ok) {
  const int frame = frame0 + blockIdx.z;
  const uint8_t* G = gray + (size_t)frame * W * H;
  float* out = I + (size_t)frame * W * H;
  const int x0 = (blockIdx.x * 32 + (threadIdx.x & 31)) * 4;
  const int y0 = (blockIdx.y * 8 + (threadIdx.x >> 5)) * 4;
  if (x0 >= W || y0 >= H) return;
  const bool fast = vec_ok && (x0 + 4 <= W);
  float hrow[6][4];
#pragma unroll
  for (int r = 0; r < 6; ++r) {
    const int y = reflect101(y0 - 1 + r, H);
    const uint8_t* row = G + (size_t)y * W;
    float g[6];
    if (fast) {
      const unsigned wd = __ldg(reinterpret_cast<const unsigned*>(row + x0));
      g[1] = (float)(wd & 0xffu); g[2] = (float)((wd >> 8) & 0xffu);
      g[3] = (float)((wd >> 16) & 0xffu); g[4] = (float)(wd >> 24);
      g[0] = (float)__ldg(row + (x0 > 0 ? x0 - 1 : 1 % W));
      g[5] = (float)__ldg(row + (x0 + 4 < W ? x0 + 4 : reflect101(x0 + 4, W)));
    } else {
#pragma unroll
      for (int i = 0; i < 6; ++i) g[i] = (float)__ldg(row + reflect101(x0 - 1 + i, W));
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) hrow[r][i] = fmaf(t2, g[i + 2], fmaf(t1, g[i + 1], t0 * g[i]));
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int y = y0 + j;
    if (y >= H) break;
    float o[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) o[i] = fmaf(t2, hrow[j + 2][i], fmaf(t1, hrow[j + 1][i], t0 * hrow[j][i]));
    float* dst = out + (size_t)y * W + x0;
    if (fast) {
      *reinterpret_cast<float4*>(dst) = make_float4(o[0], o[1], o[2], o[3]);
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (x0 + i < W) dst[i] = o[i];
    }
  }
}

// Level 0 again, for W % 8 == 0: a thread owns an 8-pixel column strip and walks kPyr0Rows rows down it.  Per row:
// one 8-byte load (issued one row ahead of its use), the two horizontal halo bytes from the neighbouring lanes
// by shuffle (lanes 0 / 31 and the image edges load them), bytes converted to float once, the horizontal 3-tap
// into a rolling three-row window in registers, the vertical 3-tap, two 16-byte stores -- the same fmaf order
// as pyr0_kernel (bit-identical).  About a third of pyr0_kernel's instructions per pixel (that kernel spends
// them on per-byte halo loads and per-row border arithmetic for a 4 x 4 patch) and, unlike a one-shot
// patch-per-thread kernel (53 us against pyr0_kernel's 55 us: both latency-bound, issue 47 %, DRAM 26 %), the
// loads of the next row are always in flight.
constexpr int kPyr0Rows = 16;

__device__ __forceinline__ void pyr0_hrow(const uint8_t* __restrict__ row, uint2 wd, int x0, int W, int lane, bool act,
                                          float t0, float t1, float t2, float* hr) {
  unsigned left = __shfl_up_sync(0xffffffffu, wd.y >> 24, 1);
  unsigned right = __shfl_down_sync(0xffffffffu, wd.x & 0xffu, 1);
  if (act) {
    if (lane == 0 || x0 == 0) left = __ldg(row + (x0 > 0 ? x0 - 1 : 1 % W));
    if (lane == 31 || x0 + 8 >= W) right = __ldg(row + (x0 + 8 < W ? x0 + 8 : reflect101(x0 + 8, W)));
  }
  float g[10];
  g[0] = (float)left;
  g[1] = (float)(wd.x & 0xffu); g[2] = (float)((wd.x >> 8) & 0xffu); g[3] = (float)((wd.x >> 16) & 0xffu); g[4] = (float)(wd.x >> 24);
  g[5] = (float)(wd.y & 0xffu); g[6] = (float)((wd.y >> 8) & 0xffu); g[7] = (float)((wd.y >> 16) & 0xffu); g[8] = (float)(wd.y >> 24);
  g[9] = (float)right;
#pragma unroll
  for (int i = 0; i < 8; ++i) hr[i] = fmaf(t2, g[i + 2], fmaf(t1, g[i + 1], t0 * g[i]));
}

__global__ void __launch_bounds__(256)
pyr0x8_kernel(const uint8_t* __restrict__ gray, float* __restrict__ I, int W, int H, float t0, float t1, float t2, int frame0) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int frame = frame0 + blockIdx.z;
  const uint8_t* G = gray + (size_t)frame * W * H;
  float* out = I + (size_t)frame * W * H;
  const int x0 = (blockIdx.x * 32 + lane) * 8;
  const int yb = (blockIdx.y * 8 + warp) * kPyr0Rows;
  if (yb >= H) return;                           // whole warp
  const bool act = x0 < W;
  const int yend = min(yb + kPyr0Rows, H);        // warp-uniform
  auto row_ptr = [&](int yy) { return G + (size_t)reflect101(yy, H) * W; };
  auto load = [&](const uint8_t* row) { return act ? __ldg(reinterpret_cast<const uint2*>(row + x0)) : make_uint2(0u, 0u); };
  float hp[8], hc[8], hn[8];
  {
    const uint8_t* ra = row_ptr(yb - 1);
    const uint8_t* rb = row_ptr(yb);
    const uint2 wa = load(ra), wb = load(rb);
    pyr0_hrow(ra, wa, x0, W, lane, act, t0, t1, t2, hp);
    pyr0_hrow(rb, wb, x0, W, lane, act, t0, t1, t2, hc);
  }
  const uint8_t* rn = row_ptr(yb + 1);
  uint2 wn = load(rn);
  for (int y = yb; y < yend; ++y) {
    const uint8_t* rnn = row_ptr(y + 2);
    const uint2 wnn = load(rnn);                   // in flight while this row is finished
    pyr0_hrow(rn, wn, x0, W, lane, act, t0, t1, t2, hn);
    if (act) {
      float o[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] = fmaf(t2, hn[i], fmaf(t1, hc[i], t0 * hp[i]));
      float4* dst = reinterpret_cast<float4*>(out + (size_t)y * W + x0);
      dst[0] = make_float4(o[0], o[1], o[2], o[3]);
      dst[1] = make_float4(o[4], o[5], o[6], o[7]);
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) { hp[i] = hc[i]; hc[i] = hn[i]; }
    rn = rnn; wn = wnn;
  }
}

// ---------------------------------------------------------------------------------------------
// Tensor-map type and the TMA L2 prefetch, shared by updmat_init_kernel and iter15_tma_kernel.
// A prefetch has no shared-memory destination and nothing to wait for: it only pulls one box of
// the tensor towards L2.
// ---------------------------------------------------------------------------------------------
constexpr int kPfBoxW = 48, kPfBoxH = 32;   // iteration kernel: exactly its 48 x 32 tile (the flow-displaced part of R1 is
                                            // covered by the neighbouring tiles' own prefetches; a padded 64 x 40 box measured 1 % slower)
constexpr int kPfInitBoxH = 8;              // updmat_init_kernel: exactly one of its 64 x 8 tiles
#ifdef STB_CPU_EMU
struct TmaMap3D {            // emulator stand-in for a CUtensorMap over [planes][h][w] floats
  const float* base;
  int w, h, planes;
};
#define STB_GRID_CONSTANT
__device__ __forceinline__ void tma_prefetch_l2(const TmaMap3D*, int, int, int) {}
#else
}  // namespace stb
#include <cuda.h>
namespace stb {
typedef CUtensorMap TmaMap3D;
#define STB_GRID_CONSTANT __grid_constant__
__device__ __forceinline__ void tma_prefetch_l2(const TmaMap3D* map, int x0, int y0, int z) {
  asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];" ::"l"(reinterpret_cast<unsigned long long>(map)),
               "r"(x0), "r"(y0), "r"(z)
               : "memory");
}
#endif

// ---------------------------------------------------------------------------------------------
// polynomial expansion (Appendix A.3): separable 11-tap, replicate borders.  I (h x w) ->
// R (5 planes of h x w).  Tile 64 x 32, 256 threads.
// ---------------------------------------------------------------------------------------------
constexpr int kPeTW = 64, kPeTH = 32, kPeThreads = 256;
constexpr int kPeCols = kPeTW + 2 * kPolyN;   // 74 columns of vertical results per tile
constexpr int kPeStride = 80;                 // row stride (floats) of the shared arrays; col j <-> x = ox0 - 8 + j
constexpr int kPeRows = 8 + 2 * kPolyN;       // 18 input rows per vertical item (8 output rows)

// Vertical pass: item = (column, group of 8 rows); the 18 input rows come straight from global
// memory (coalesced along x, replicate clamp), results r0,r1,r2 go to shared memory row-major.
// Horizontal pass: item = (row, 4 adjacent columns): 16-byte shared loads of a 20-float window
// per component, 11-tap sums in registers, float4 stores of the 5 output planes.
__global__ void __launch_bounds__(kPeThreads, 4)
polyexp_kernel(const float* __restrict__ I, size_t i_stride, float* __restrict__ R, int w, int h, PolyConsts c, int frame0) {
  // (A prefetch-ahead of the I tile, as in updmat_init_kernel, measured neutral here: the reads are
  // 1/6 of this kernel's traffic.)
  __shared__ __align__(16) float V[3][kPeTH][kPeStride];
  const int tid = threadIdx.x;
  const int frame = frame0 + blockIdx.z;
  const int n = w * h;
  const float* src = I + (size_t)frame * i_stride;
  float* dst = R + (size_t)frame * 5 * n;
  const int ox0 = blockIdx.x * kPeTW, oy0 = blockIdx.y * kPeTH;

  if ((w & 1) == 0) {
    // Column PAIRS (x, x + 1), x even: one 8-byte load per row and packed f32x2 arithmetic -- half the instructions
    // of the scalar pass below, the same operations per element.  38 pairs cover columns ox0 - 6 .. ox0 + 69 (the
    // tile's 64 + 5 either side, plus one spare column each end that the horizontal pass never reads).
    constexpr int kPairs = (kPeCols + 2) / 2;   // 38
    for (int item = tid; item < kPairs * (kPeTH / 8); item += kPeThreads) {
      const int g = item / kPairs, q = item - g * kPairs;
      const int xa = ox0 + 2 * q - (kPolyN + 1);            // even
      const int y_first = oy0 + g * 8 - kPolyN;
      float2 v[kPeRows];
      const bool rows_in = y_first >= 0 && y_first + kPeRows - 1 <= h - 1;
      if (xa >= 0 && xa + 1 < w) {
        if (rows_in) {
          const float* p = src + y_first * w + xa;
#pragma unroll
          for (int j = 0; j < kPeRows; ++j) v[j] = __ldg(reinterpret_cast<const float2*>(p + j * w));
        } else {
#pragma unroll
          for (int j = 0; j < kPeRows; ++j) v[j] = __ldg(reinterpret_cast<const float2*>(src + min(max(y_first + j, 0), h - 1) * w + xa));
        }
      } else {
        const int x0c = min(max(xa, 0), w - 1), x1c = min(max(xa + 1, 0), w - 1);    // replicate columns
#pragma unroll
        for (int j = 0; j < kPeRows; ++j) {
          const float* row = src + min(max(y_first + j, 0), h - 1) * w;
          v[j] = make_float2(__ldg(row + x0c), __ldg(row + x1c));
        }
      }
      const int col = 2 * q + 2;          // x = ox0 - 8 + col
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        float2 r0 = f2mul(v[i + kPolyN], c.g2[0]);
        float2 r1 = make_float2(0.f, 0.f), r2 = make_float2(0.f, 0.f);
#pragma unroll
        for (int k = 1; k <= kPolyN; ++k) {
          const float2 a = v[i + kPolyN - k], b = v[i + kPolyN + k];
          const float2 pp = f2add(a, b);
          r0 = f2fma(c.g2[k], pp, r0);
          r1 = f2fma(c.xg2[k], f2sub(b, a), r1);
          r2 = f2fma(c.xxg2[k], pp, r2);
        }
        *reinterpret_cast<float2*>(&V[0][g * 8 + i][col]) = r0;
        *reinterpret_cast<float2*>(&V[1][g * 8 + i][col]) = r1;
        *reinterpret_cast<float2*>(&V[2][g * 8 + i][col]) = r2;
      }
    }
  } else
  for (int item = tid; item < kPeCols * (kPeTH / 8); item += kPeThreads) {
    const int g = item / kPeCols, cx = item - g * kPeCols;
    const int x = min(max(ox0 + cx - kPolyN, 0), w - 1);
    const int y_first = oy0 + g * 8 - kPolyN;
    float v[kPeRows];
    if (y_first >= 0 && y_first + kPeRows - 1 <= h - 1) {
      const float* p = src + y_first * w + x;
#pragma unroll
      for (int j = 0; j < kPeRows; ++j) v[j] = __ldg(p + j * w);
    } else {
#pragma unroll
      for (int j = 0; j < kPeRows; ++j) v[j] = __ldg(src + min(max(y_first + j, 0), h - 1) * w + x);
    }
    const int col = cx + 3;   // x = ox0 - 5 + cx  <->  j = cx + 3
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const float s0 = v[i + kPolyN];
      float r0 = s0 * c.g[0], r1 = 0.f, r2 = 0.f;
#pragma unroll
      for (int k = 1; k <= kPolyN; ++k) {
        const float a = v[i + kPolyN - k], b = v[i + kPolyN + k];
        const float pp = a + b;
        r0 = fmaf(c.g[k], pp, r0);
        r1 = fmaf(c.xg[k], b - a, r1);
        r2 = fmaf(c.xxg[k], pp, r2);
      }
      V[0][g * 8 + i][col] = r0;
      V[1][g * 8 + i][col] = r1;
      V[2][g * 8 + i][col] = r2;
    }
  }
  __syncthreads();

  const bool vec_ok = (w & 3) == 0;
  for (int item = tid; item < (kPeTW / 4) * kPeTH; item += kPeThreads) {
    const int ty = item / (kPeTW / 4), q = item - ty * (kPeTW / 4);
    const int x = ox0 + q * 4, y = oy0 + ty;
    if (x >= w || y >= h) continue;
    // window: shared columns [4q, 4q+20)  <->  x-8 .. x+11; pixel i, tap offset d -> index 8 + i + d
    float b1[4], b2[4], b3[4], b4[4], b5[4], b6[4];
    {
      float t[20];
      const float4* wp = reinterpret_cast<const float4*>(&V[0][ty][q * 4]);
#pragma unroll
      for (int j = 0; j < 5; ++j) { const float4 f = wp[j]; t[4 * j] = f.x; t[4 * j + 1] = f.y; t[4 * j + 2] = f.z; t[4 * j + 3] = f.w; }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float a1 = t[8 + i] * c.g[0], a2 = 0.f, a4 = 0.f;
#pragma unroll
        for (int k = 1; k <= kPolyN; ++k) {
          const float pl = t[8 + i + k], mi = t[8 + i - k];
          const float tg = pl + mi;
          a1 = fmaf(tg, c.g[k], a1);
          a4 = fmaf(tg, c.xxg[k], a4);
          a2 = fmaf(pl - mi, c.xg[k], a2);
        }
        b1[i] = a1; b2[i] = a2; b4[i] = a4;
      }
    }
    {
      float t[20];
      const float4* wp = reinterpret_cast<const float4*>(&V[1][ty][q * 4]);
#pragma unroll
      for (int j = 0; j < 5; ++j) { const float4 f = wp[j]; t[4 * j] = f.x; t[4 * j + 1] = f.y; t[4 * j + 2] = f.z; t[4 * j + 3] = f.w; }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float a3 = t[8 + i] * c.g[0], a6 = 0.f;
#pragma unroll
        for (int k = 1; k <= kPolyN; ++k) {
          const float pl = t[8 + i + k], mi = t[8 + i - k];
          a3 = fmaf(pl + mi, c.g[k], a3);
          a6 = fmaf(pl - mi, c.xg[k], a6);
        }
        b3[i] = a3; b6[i] = a6;
      }
    }
    {
      float t[20];
      const float4* wp = reinterpret_cast<const float4*>(&V[2][ty][q * 4]);
#pragma unroll
      for (int j = 0; j < 5; ++j) { const float4 f = wp[j]; t[4 * j] = f.x; t[4 * j + 1] = f.y; t[4 * j + 2] = f.z; t[4 * j + 3] = f.w; }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float a5 = t[8 + i] * c.g[0];
#pragma unroll
        for (int k = 1; k <= kPolyN; ++k) a5 = fmaf(t[8 + i + k] + t[8 + i - k], c.g[k], a5);
        b5[i] = a5;
      }
    }
    float o0[4], o1[4], o2[4], o3[4], o4[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      o0[i] = b3[i] * c.ig11;                          // d/dy
      o1[i] = b2[i] * c.ig11;                          // d/dx
      o2[i] = fmaf(b1[i], c.ig03, b5[i] * c.ig33);     // yy
      o3[i] = fmaf(b1[i], c.ig03, b4[i] * c.ig33);     // xx
      o4[i] = b6[i] * c.ig55;                          // xy
    }
    float* d0 = dst + y * w + x;
    if (vec_ok && x + 3 < w) {
      *reinterpret_cast<float4*>(d0) = make_float4(o0[0], o0[1], o0[2], o0[3]);
      *reinterpret_cast<float4*>(d0 + n) = make_float4(o1[0], o1[1], o1[2], o1[3]);
      *reinterpret_cast<float4*>(d0 + 2 * n) = make_float4(o2[0], o2[1], o2[2], o2[3]);
      *reinterpret_cast<float4*>(d0 + 3 * n) = make_float4(o3[0], o3[1], o3[2], o3[3]);
      *reinterpret_cast<float4*>(d0 + 4 * n) = make_float4(o4[0], o4[1], o4[2], o4[3]);
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i)
        if (x + i < w) { d0[i] = o0[i]; d0[n + i] = o1[i]; d0[2 * n + i] = o2[i]; d0[3 * n + i] = o3[i]; d0[4 * n + i] = o4[i]; }
    }
  }
}

// Generic polynomial expansion for polyN != 5 (not used by the reference, which hard-codes 5):
// one thread per pixel, the (2n+1)^2 neighbourhood read straight from global memory (L1/L2
// resident), same arithmetic as polyexp_kernel.  Correctness path, not tuned.
__device__ __forceinline__ void polyexp_column(const float* __restrict__ src, int w, int h, int xc, int y, int n,
                                               const PolyConsts& c, float& r0, float& r1, float& r2) {
  const float s0 = __ldg(src + y * w + xc);
  r0 = s0 * c.g[0]; r1 = 0.f; r2 = 0.f;
  for (int k = 1; k <= n; ++k) {
    const float a = __ldg(src + max(y - k, 0) * w + xc), b = __ldg(src + min(y + k, h - 1) * w + xc);
    const float pp = a + b;
    r0 = fmaf(c.g[k], pp, r0);
    r1 = fmaf(c.xg[k], b - a, r1);
    r2 = fmaf(c.xxg[k], pp, r2);
  }
}

__global__ void __launch_bounds__(256)
polyexp_generic_kernel(const float* __restrict__ I, size_t i_stride, float* __restrict__ R, int w, int h, PolyConsts c, int n, int frame0) {
  const int x = blockIdx.x * 32 + (threadIdx.x & 31), y = blockIdx.y * 8 + (threadIdx.x >> 5);
  if (x >= w || y >= h) return;
  const int frame = frame0 + blockIdx.z;
  const int npx = w * h;
  const float* src = I + (size_t)frame * i_stride;
  float* dst = R + (size_t)frame * 5 * npx + y * w + x;
  float c0, c1, c2;
  polyexp_column(src, w, h, x, y, n, c, c0, c1, c2);
  float b1 = c0 * c.g[0], b2 = 0.f, b3 = c1 * c.g[0], b4 = 0.f, b5 = c2 * c.g[0], b6 = 0.f;
  for (int k = 1; k <= n; ++k) {
    float p0, p1, p2, m0, m1, m2;
    polyexp_column(src, w, h, min(x + k, w - 1), y, n, c, p0, p1, p2);
    polyexp_column(src, w, h, max(x - k, 0), y, n, c, m0, m1, m2);
    b1 = fmaf(p0 + m0, c.g[k], b1);
    b4 = fmaf(p0 + m0, c.xxg[k], b4);
    b2 = fmaf(p0 - m0, c.xg[k], b2);
    b3 = fmaf(p1 + m1, c.g[k], b3);
    b6 = fmaf(p1 - m1, c.xg[k], b6);
    b5 = fmaf(p2 + m2, c.g[k], b5);
  }
  dst[0] = b3 * c.ig11;                          // d/dy
  dst[npx] = b2 * c.ig11;                        // d/dx
  dst[2 * npx] = fmaf(b1, c.ig03, b5 * c.ig33);  // yy
  dst[3 * npx] = fmaf(b1, c.ig03, b4 * c.ig33);  // xx
  dst[4 * npx] = b6 * c.ig55;                    // xy
}

// ---------------------------------------------------------------------------------------------
// UpdateMatrices for one pixel (Appendix A.5).  R0, R1: planar 5 x n.
// ---------------------------------------------------------------------------------------------
// p + elems floats as ONE instruction (IMAD.WIDE).  Written as pointer + int, nvcc forms the plane / row
// addresses of the R0 loads and M' stores of the update kernels from 64-bit IADD3 / IADD3.X / LEA / LEA.HI.X
// chains: 36 address instructions for 10 loads (ncu source view, round 2).
#ifdef STB_CPU_EMU
template <class T> __device__ __forceinline__ T* padd(T* p, int elems) { return p + elems; }
#else
template <class T> __device__ __forceinline__ T* padd(T* p, int elems) {
  static_assert(sizeof(T) == 4, "4-byte elements");
  T* r;
  asm("mad.wide.s32 %0, %1, 4, %2;" : "=l"(r) : "r"(elems), "l"(p));
  return r;
}
#endif

__device__ __forceinline__ float border_w(int d) { return d < 2 ? 0.14f : 0.4472f; }

// second half of UpdateMatrices: from R0's planes q0..q4 at (x, y) and the (interpolated) R1
// values r2..r6 (`inside` false = the out-of-range branch) to the five M entries
__device__ __forceinline__ void um_finish(float q0, float q1, float q2, float q3, float q4, bool inside,
                                          float r2, float r3, float r4, float r5, float r6,
                                          int w, int h, int x, int y, float dx, float dy, float m[5]) {
  if (inside) {
    r4 = (q2 + r4) * 0.5f;
    r5 = (q3 + r5) * 0.5f;
    r6 = (q4 + r6) * 0.25f;
  } else {
    r2 = r3 = 0.f;
    r4 = q2;
    r5 = q3;
    r6 = q4 * 0.5f;
  }
  r2 = (q0 - r2) * 0.5f;
  r3 = (q1 - r3) * 0.5f;
  r2 += r4 * dy + r6 * dx;
  r3 += r6 * dy + r5 * dx;
  if ((unsigned)(x - 5) >= (unsigned)(w - 10) || (unsigned)(y - 5) >= (unsigned)(h - 10)) {
    const float scale = (x < 5 ? border_w(x) : 1.f) * (x >= w - 5 ? border_w(w - x - 1) : 1.f) *
                        (y < 5 ? border_w(y) : 1.f) * (y >= h - 5 ? border_w(h - y - 1) : 1.f);
    r2 *= scale; r3 *= scale; r4 *= scale; r5 *= scale; r6 *= scale;
  }
  m[0] = r4 * r4 + r6 * r6;
  m[1] = (r4 + r5) * r6;
  m[2] = r5 * r5 + r6 * r6;
  m[3] = r4 * r2 + r6 * r3;
  m[4] = r6 * r2 + r5 * r3;
}

__device__ __forceinline__ void update_matrices_q(float q0, float q1, float q2, float q3, float q4,
                                                  const float* __restrict__ R1, int n, int w, int h, int x, int y,
                                                  float dx, float dy, float m[5]) {
  // q0..q4 = R0's five planes at (x, y).  n = w*h <= 2^28 (checked at create), so 5*n fits an
  // int: 32-bit offsets throughout
  float fx = (float)x + dx, fy = (float)y + dy;
  const int x1 = __float2int_rd(fx), y1 = __float2int_rd(fy);
  fx -= (float)x1; fy -= (float)y1;
  float r[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
  const bool inside = (unsigned)x1 < (unsigned)(w - 1) && (unsigned)y1 < (unsigned)(h - 1);
  if (inside) {
    const float a00 = (1.f - fx) * (1.f - fy), a01 = fx * (1.f - fy), a10 = (1.f - fx) * fy, a11 = fx * fy;
    const float* p = padd(R1, y1 * w + x1);
#pragma unroll
    for (int pl = 0; pl < 5; ++pl) {
      const float* pw = padd(p, w);
      r[pl] = a00 * __ldg(p) + a01 * __ldg(p + 1) + a10 * __ldg(pw) + a11 * __ldg(pw + 1);
      p = padd(p, n);
    }
  }
  um_finish(q0, q1, q2, q3, q4, inside, r[0], r[1], r[2], r[3], r[4], w, h, x, y, dx, dy, m);
}

// Two horizontally adjacent pixels (x, y) and (x+1, y).  Their bilinear footprints in R1 almost
// always overlap (the flow is a 15x15-window solution, so floor(x + dx) of neighbours differs by
// exactly 1 except at integer crossings): then 3 columns x 2 rows per plane serve both pixels
// instead of 4 + 4 loads.  Same values, same arithmetic: bit-identical to two single calls.
__device__ __forceinline__ void update_matrices_pair(const float2 q[5], const float* __restrict__ R1, int n, int w, int h,
                                                     int x, int y, float2 fa, float2 fb, float ma[5], float mb[5]) {
  float fxa = (float)x + fa.x, fya = (float)y + fa.y;
  float fxb = (float)(x + 1) + fb.x, fyb = (float)y + fb.y;
  const int x1a = __float2int_rd(fxa), y1a = __float2int_rd(fya);
  const int x1b = __float2int_rd(fxb), y1b = __float2int_rd(fyb);
  const bool ina = (unsigned)x1a < (unsigned)(w - 1) && (unsigned)y1a < (unsigned)(h - 1);
  const bool inb = (unsigned)x1b < (unsigned)(w - 1) && (unsigned)y1b < (unsigned)(h - 1);
  if (ina && inb && x1b == x1a + 1 && y1b == y1a) {
    fxa -= (float)x1a; fya -= (float)y1a; fxb -= (float)x1b; fyb -= (float)y1b;
    const float a00 = (1.f - fxa) * (1.f - fya), a01 = fxa * (1.f - fya), a10 = (1.f - fxa) * fya, a11 = fxa * fya;
    const float b00 = (1.f - fxb) * (1.f - fyb), b01 = fxb * (1.f - fyb), b10 = (1.f - fxb) * fyb, b11 = fxb * fyb;
    const float* p = padd(R1, y1a * w + x1a);
    float ra[5], rb[5];
#pragma unroll
    for (int pl = 0; pl < 5; ++pl) {
      const float* pw = padd(p, w);
      const float t0 = __ldg(p), t1 = __ldg(p + 1), t2 = __ldg(p + 2);
      const float u0 = __ldg(pw), u1 = __ldg(pw + 1), u2 = __ldg(pw + 2);
      ra[pl] = a00 * t0 + a01 * t1 + a10 * u0 + a11 * u1;
      rb[pl] = b00 * t1 + b01 * t2 + b10 * u1 + b11 * u2;
      p = padd(p, n);
    }
    um_finish(q[0].x, q[1].x, q[2].x, q[3].x, q[4].x, true, ra[0], ra[1], ra[2], ra[3], ra[4], w, h, x, y, fa.x, fa.y, ma);
    um_finish(q[0].y, q[1].y, q[2].y, q[3].y, q[4].y, true, rb[0], rb[1], rb[2], rb[3], rb[4], w, h, x + 1, y, fb.x, fb.y, mb);
  } else {
    update_matrices_q(q[0].x, q[1].x, q[2].x, q[3].x, q[4].x, R1, n, w, h, x, y, fa.x, fa.y, ma);
    update_matrices_q(q[0].y, q[1].y, q[2].y, q[3].y, q[4].y, R1, n, w, h, x + 1, y, fb.x, fb.y, mb);
  }
}

__device__ __forceinline__ void update_matrices_px(const float* __restrict__ R0, const float* __restrict__ R1,
                                                   int n, int w, int h, int x, int y, float dx, float dy,
                                                   float m[5]) {
  const int o = y * w + x;
  update_matrices_q(__ldg(R0 + o), __ldg(R0 + n + o), __ldg(R0 + 2 * n + o), __ldg(R0 + 3 * n + o),
                    __ldg(R0 + 4 * n + o), R1, n, w, h, x, y, dx, dy, m);
}

// Flow-compensated R1 window of iter15_win_kernel: the box [x0, x0 + kWinW) x [y0, y0 + kWinH) of the
// five R1 planes in shared memory, plane stride kWinPlaneFloats.  fits == false: no window, the
// footprints are gathered from global memory (kNoR1Win, a compile-time constant for the other kernels).
constexpr int kWinW = 56, kWinH = 38;
constexpr int kWinPlaneFloats = 2144;                         // 56 * 38 = 2128, rounded up to a multiple of 32 floats (128 B)
struct R1Win {
  const float* s;
  int x0, y0;
  bool fits;
};
constexpr R1Win kNoR1Win = {nullptr, 0, 0, false};

// Two VERTICALLY adjacent pixels (x, y) and (x, y+1) handled by one thread, consecutive lanes on
// consecutive x.  Their bilinear footprints in R1 almost always share a row (floor(y + dy) of
// vertical neighbours differs by exactly 1 except at integer crossings), so 3 rows x 2 columns
// per plane serve both pixels (30 loads instead of 40), and -- unlike a horizontal pair, whose
// lanes stride by two pixels -- every load of a warp covers one contiguous run of floats: about
// 1.3 L1 wavefronts per load instead of 3.  Same values and arithmetic as two single calls.
// With a window that fits, the shared footprint is read from it instead (same values).
__device__ __forceinline__ void update_matrices_vpair(const float* __restrict__ R0, const float* __restrict__ R1, R1Win win,
                                                      int n, int w, int h, int x, int y, float2 fa, float2 fb, float ma[5],
                                                      float mb[5]) {
  float qa[5], qb[5];
  {
    const float* q = padd(R0, y * w + x);
#pragma unroll
    for (int c = 0; c < 5; ++c) { qa[c] = __ldg(q); qb[c] = __ldg(padd(q, w)); q = padd(q, n); }
  }
  float fxa = (float)x + fa.x, fya = (float)y + fa.y;
  float fxb = (float)x + fb.x, fyb = (float)(y + 1) + fb.y;
  const int x1a = __float2int_rd(fxa), y1a = __float2int_rd(fya);
  const int x1b = __float2int_rd(fxb), y1b = __float2int_rd(fyb);
  const bool ina = (unsigned)x1a < (unsigned)(w - 1) && (unsigned)y1a < (unsigned)(h - 1);
  const bool inb = (unsigned)x1b < (unsigned)(w - 1) && (unsigned)y1b < (unsigned)(h - 1);
  if (ina && inb && x1b == x1a && y1b == y1a + 1) {
    fxa -= (float)x1a; fya -= (float)y1a; fxb -= (float)x1b; fyb -= (float)y1b;
    const float a00 = (1.f - fxa) * (1.f - fya), a01 = fxa * (1.f - fya), a10 = (1.f - fxa) * fya, a11 = fxa * fya;
    const float b00 = (1.f - fxb) * (1.f - fyb), b01 = fxb * (1.f - fyb), b10 = (1.f - fxb) * fyb, b11 = fxb * fyb;
    float ra[5], rb[5];
    if (win.fits) {
      const float* p = win.s + (y1a - win.y0) * kWinW + (x1a - win.x0);
#pragma unroll
      for (int pl = 0; pl < 5; ++pl) {
        const float t00 = p[pl * kWinPlaneFloats], t01 = p[pl * kWinPlaneFloats + 1];
        const float t10 = p[pl * kWinPlaneFloats + kWinW], t11 = p[pl * kWinPlaneFloats + kWinW + 1];
        const float t20 = p[pl * kWinPlaneFloats + 2 * kWinW], t21 = p[pl * kWinPlaneFloats + 2 * kWinW + 1];
        ra[pl] = a00 * t00 + a01 * t01 + a10 * t10 + a11 * t11;
        rb[pl] = b00 * t10 + b01 * t11 + b10 * t20 + b11 * t21;
      }
    } else {
      const float* p = padd(R1, y1a * w + x1a);
#pragma unroll
      for (int pl = 0; pl < 5; ++pl) {
        const float* p1 = padd(p, w);
        const float* p2 = padd(p1, w);
        const float t00 = __ldg(p), t01 = __ldg(p + 1);
        const float t10 = __ldg(p1), t11 = __ldg(p1 + 1);
        const float t20 = __ldg(p2), t21 = __ldg(p2 + 1);
        ra[pl] = a00 * t00 + a01 * t01 + a10 * t10 + a11 * t11;
        rb[pl] = b00 * t10 + b01 * t11 + b10 * t20 + b11 * t21;
        p = padd(p, n);
      }
    }
    um_finish(qa[0], qa[1], qa[2], qa[3], qa[4], true, ra[0], ra[1], ra[2], ra[3], ra[4], w, h, x, y, fa.x, fa.y, ma);
    um_finish(qb[0], qb[1], qb[2], qb[3], qb[4], true, rb[0], rb[1], rb[2], rb[3], rb[4], w, h, x, y + 1, fb.x, fb.y, mb);
  } else {
    update_matrices_q(qa[0], qa[1], qa[2], qa[3], qa[4], R1, n, w, h, x, y, fa.x, fa.y, ma);
    update_matrices_q(qb[0], qb[1], qb[2], qb[3], qb[4], R1, n, w, h, x, y + 1, fb.x, fb.y, mb);
  }
}

// ---------------------------------------------------------------------------------------------
// Block order of the kernels that read R (updmat_init_kernel and the iteration kernels): the grid
// is walked PAIR-FASTEST.  The polynomial expansion R of frame f+1 is read twice per level and pass:
// displaced, as R1 of pair f, and in place, as R0 of pair f+1.  With the pair index as the slowest
// grid dimension (round 1) those two reads were a whole pair (2.3 resident waves, ~200 MB of
// traffic) apart and both came from HBM; with the pairs of one tile adjacent in the grid they run
// at the same time on neighbouring SMs and the second read is an L2 hit: a quarter of the
// iteration's 80 B/px never reaches HBM.  Two orders are launched:
//   * the iteration kernels: a 1-D grid, pair, then kTileBand tile rows, then tile column, then
//     band, so a tile's vertical neighbours (whose M halos it shares) are co-resident too;
//   * updmat_init_kernel: a 3-D grid (pair, tile x, tile y) in the hardware's own rasterisation
//     order.
// Measured on B200 (1080p, 16-pair batches, one box, back to back): round-1 order through a 1-D grid
// 5117 fps; iteration kernels band 2 / 4 / 8 / all rows: 5284 / 5308 / 5317 / 5001; updmat_init_kernel
// band 8 / 16 / 32 / all rows: 5309 / 5308 / 5314 / 5193 and, as the 3-D grid: +1.5 % on top (5466 vs
// 5383) -- the iteration kernels lose 0.4 % that way.
// ---------------------------------------------------------------------------------------------
constexpr int kTileBand = 4;   // tile rows of 32 px walked before the column advances

struct TileOrder {
  int tiles_x, tiles_y, np;
};

// tile of block `id` of the iteration kernels' 1-D grid.  Unsigned divisions: shorter than signed
// ones, which keeps the 64-register kernels free of spills.
__device__ __forceinline__ void tile_of_band_order(const TileOrder& o, int id, int& tx, int& ty, int& pz) {
  const unsigned per_band = (unsigned)(o.tiles_x * kTileBand * o.np);
  const unsigned b = (unsigned)id / per_band, r = (unsigned)id - b * per_band;
  const unsigned bh = min((unsigned)kTileBand, (unsigned)o.tiles_y - b * kTileBand);   // the last band may be shorter
  const unsigned col = bh * (unsigned)o.np;
  tx = (int)(r / col);
  const unsigned r2 = r - (unsigned)tx * col;
  const unsigned tyb = r2 / (unsigned)o.np;
  ty = (int)(b * kTileBand + tyb);
  pz = (int)(r2 - tyb * (unsigned)o.np);
}

// initial M of a level from the up-sampled coarser flow (Appendix A.4-5).
__device__ __forceinline__ void upsample_axis(int d, double scale, int n_src, int& s, float& f) {
  if (scale == 0.5) {   // exact halving: (d + 0.5) * 0.5 - 0.5 is exact in float, skip the double path
    f = (float)d * 0.5f - 0.25f;
    s = __float2int_rd(f);
    f -= (float)s;
    if (s < 0) { s = 0; f = 0.f; }
    if (s >= n_src - 1) { s = n_src - 1; f = 0.f; }
  } else {
    resize_src(d, scale, n_src, s, f);
  }
}

__device__ __forceinline__ float2 upsample_flow(const float2* __restrict__ fc, int wc, int hc, int sy, float fy,
                                                int x, double scale_x, float flow_mul) {
  int sx; float fx;
  upsample_axis(x, scale_x, wc, sx, fx);
  const int sx1 = min(sx + 1, wc - 1), sy1 = min(sy + 1, hc - 1);
  const float2 f00 = __ldg(fc + (sy * wc + sx)), f01 = __ldg(fc + (sy * wc + sx1));
  const float2 f10 = __ldg(fc + (sy1 * wc + sx)), f11 = __ldg(fc + (sy1 * wc + sx1));
  const float ax0 = 1.f - fx, ay0 = 1.f - fy;
  const float h0x = f00.x * ax0 + f01.x * fx, h1x = f10.x * ax0 + f11.x * fx;
  const float h0y = f00.y * ax0 + f01.y * fx, h1y = f10.y * ax0 + f11.y * fx;
  return make_float2((h0x * ay0 + h1x * fy) * flow_mul, (h0y * ay0 + h1y * fy) * flow_mul);
}

// Two horizontally adjacent pixels per thread (8-byte accesses of R0 / M when w is even).  This
// kernel is DRAM-bound (69 % of peak): the vertical-pair mapping that helps the L1-bound iteration
// kernel measured 12 % slower here (495 vs 440 us per 16-pair level-0 launch).
// 5 blocks/SM (48 registers): with the prefetch-ahead in place the extra resident warps are
// worth +1 % of the step (before it, 5 blocks/SM measured slower: 500 vs 440 us in isolation).
// Grid (pair, tile x, tile y) of 64 x 8 tiles, see "Block order" above.
__global__ void __launch_bounds__(256, 5)
updmat_init_kernel(const float* __restrict__ R, const float* __restrict__ flow_coarse, float* __restrict__ M,
                   int w, int h, int wc, int hc, double scale_x, double scale_y, float flow_mul, int pair0,
                   const STB_GRID_CONSTANT TmaMap3D map_R, int prefetch_blocks) {
  const int bpz = (int)blockIdx.x, btx = (int)blockIdx.y, bty = (int)blockIdx.z;
  const int pair = pair0 + bpz;
  if (prefetch_blocks > 0 && threadIdx.x < 10) {
    // The block `prefetch_blocks` further on in the grid is picked up about two resident waves from
    // now.  Pull its R planes towards L2 so its loads hit L2 instead of waiting on DRAM.  Every plane
    // of every frame tile is prefetched by exactly one block: a block prefetches R0 (the planes of its
    // own frame, lanes 0-4); the block of the launch's last pair also prefetches R1 (lanes 5-9) -- for
    // the other pairs that frame is the R0 of the pair next to them.
    const int np = (int)gridDim.x, per = np * (int)gridDim.y;
    const int ahead = (int)(blockIdx.x + gridDim.x * (blockIdx.y + gridDim.y * blockIdx.z)) + prefetch_blocks;
    if (ahead < (int)(gridDim.x * gridDim.y * gridDim.z)) {
      const int aty = ahead / per, r = ahead - aty * per;
      const int atx = r / np, apz = r - atx * np;
      if ((int)threadIdx.x < 5 || apz == np - 1)
        tma_prefetch_l2(&map_R, atx * 64, aty * 8, (pair0 + apz) * 5 + (int)threadIdx.x);
    }
  }
  const int x = (btx * 32 + (threadIdx.x & 31)) * 2;
  const int y = bty * 8 + (threadIdx.x >> 5);
  if (x >= w || y >= h) return;
  const int n = w * h;
  const bool two = x + 1 < w;
  float2 da = make_float2(0.f, 0.f), db = make_float2(0.f, 0.f);
  if (flow_coarse != nullptr) {
    const float2* fc = reinterpret_cast<const float2*>(flow_coarse) + (size_t)pair * wc * hc;
    int sy; float fy;
    upsample_axis(y, scale_y, hc, sy, fy);
    const int cx = x >> 1;
    if (scale_x == 0.5 && two && cx >= 1 && cx + 1 < wc) {
      // Exact halving, interior: pixel x = 2 cx reads coarse columns (cx - 1, cx) with weights (0.25, 0.75) and
      // pixel x + 1 columns (cx, cx + 1) with (0.75, 0.25) -- upsample_axis's results -- so the pair shares the
      // middle column: 6 loads instead of 8, same arithmetic per pixel as upsample_flow.
      const int sy1 = min(sy + 1, hc - 1);
      const float2* r0 = fc + (sy * wc + cx - 1);
      const float2* r1 = fc + (sy1 * wc + cx - 1);
      const float2 t0 = __ldg(r0), t1 = __ldg(r0 + 1), t2 = __ldg(r0 + 2);
      const float2 u0 = __ldg(r1), u1 = __ldg(r1 + 1), u2 = __ldg(r1 + 2);
      const float ay0 = 1.f - fy;
      {
        const float fx = 0.75f, ax0 = 0.25f;
        const float h0x = t0.x * ax0 + t1.x * fx, h1x = u0.x * ax0 + u1.x * fx;
        const float h0y = t0.y * ax0 + t1.y * fx, h1y = u0.y * ax0 + u1.y * fx;
        da = make_float2((h0x * ay0 + h1x * fy) * flow_mul, (h0y * ay0 + h1y * fy) * flow_mul);
      }
      {
        const float fx = 0.25f, ax0 = 0.75f;
        const float h0x = t1.x * ax0 + t2.x * fx, h1x = u1.x * ax0 + u2.x * fx;
        const float h0y = t1.y * ax0 + t2.y * fx, h1y = u1.y * ax0 + u2.y * fx;
        db = make_float2((h0x * ay0 + h1x * fy) * flow_mul, (h0y * ay0 + h1y * fy) * flow_mul);
      }
    } else {
      da = upsample_flow(fc, wc, hc, sy, fy, x, scale_x, flow_mul);
      if (two) db = upsample_flow(fc, wc, hc, sy, fy, x + 1, scale_x, flow_mul);
    }
  }
  const float* R0 = R + (size_t)pair * 5 * n;
  const float* R1 = R0 + (size_t)5 * n;
  const int o = y * w + x;
  float ma[5], mb[5];
  float* Mo = M + (size_t)pair * 5 * n + o;
  if (two && (w & 1) == 0) {
    float2 q[5];
    {
      const float* qp = padd(R0, o);
#pragma unroll
      for (int c = 0; c < 5; ++c) { q[c] = __ldg(reinterpret_cast<const float2*>(qp)); qp = padd(qp, n); }
    }
    update_matrices_pair(q, R1, n, w, h, x, y, da, db, ma, mb);
#pragma unroll
    for (int c = 0; c < 5; ++c) { *reinterpret_cast<float2*>(Mo) = make_float2(ma[c], mb[c]); Mo = padd(Mo, n); }
  } else {
    update_matrices_px(R0, R1, n, w, h, x, y, da.x, da.y, ma);
#pragma unroll
    for (int c = 0; c < 5; ++c) Mo[c * n] = ma[c];
    if (two) {
      update_matrices_px(R0, R1, n, w, h, x + 1, y, db.x, db.y, mb);
#pragma unroll
      for (int c = 0; c < 5; ++c) Mo[c * n + 1] = mb[c];
    }
  }
}

// ---------------------------------------------------------------------------------------------
// one displacement-update iteration (Appendix A.6), fused:
//   box sums (2m+1)^2 of the 5 planes of M (replicate border) -> 2x2 solve -> flow
//   -> (UPDATE)  UpdateMatrices with the new flow -> M_out
//   -> (!UPDATE) flow written out (float2 per pixel, interleaved dx,dy -- the op's layout)
// Tile 64 x 32, 256 threads (generic window size; the production winSize = 15 path is
// iter15_kernel below).  Per plane: raw tile (+halo) -> shared; vertical window sums
// -> transposed shared array; horizontal window sums by
// (lane = row, warp = 8-column group) into registers.  After the solve, flow goes through
// shared memory so the global-memory phase runs with lanes along x (coalesced).
// ---------------------------------------------------------------------------------------------
constexpr int kItTW = 64, kItTH = 32, kItThreads = 256;
constexpr int kItMaxHalo = 15;  // win_size <= 31

// GAUSS (flags & OPTFLOW_FARNEBACK_GAUSSIAN, OpenCV's FarnebackUpdateFlow_GaussianBlur): the box
// sums become a separable Gaussian window, taps k[0..m] normalised to sum 1 per axis, accumulated
// centre first, then symmetric pairs (OpenCV's order); no division by the window area.
struct WinTaps {
  float k[kItMaxHalo + 1];
};

template <bool UPDATE, bool GAUSS>
__global__ void __launch_bounds__(kItThreads, 2)
iter_kernel(const float* __restrict__ Min, float* __restrict__ Mout, const float* __restrict__ R,
            PtrBatch<float> flow_out, int w, int h, int m, int pair0, WinTaps taps) {
  STB_DYN_SMEM(float, sm);
  const int rawW = kItTW + 2 * m, rawH = kItTH + 2 * m;
  const int rawS = rawW + 2;              // row stride of raw
  float* raw = sm;                        // [rawH][rawS]
  float* Vt = sm + rawH * rawS;           // [rawW][33]   (transposed vertical sums)
  float2* fl = reinterpret_cast<float2*>(sm);  // [32][64] aliases raw/Vt after the box phase

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int pair = pair0 + blockIdx.z;
  const size_t n = (size_t)w * h;
  const float* Mp = Min + (size_t)pair * 5 * n;
  const int ox0 = blockIdx.x * kItTW, oy0 = blockIdx.y * kItTH;
  const int win = 2 * m + 1;

  float sums[5][8];
#pragma unroll
  for (int c = 0; c < 5; ++c) {
    const float* plane = Mp + (size_t)c * n;
    for (int idx = tid; idx < rawH * rawW; idx += kItThreads) {
      const int yy = idx / rawW, xx = idx - yy * rawW;
      const int y = min(max(oy0 + yy - m, 0), h - 1);
      const int x = min(max(ox0 + xx - m, 0), w - 1);
      raw[yy * rawS + xx] = __ldg(plane + (size_t)y * w + x);
    }
    __syncthreads();
    // vertical: item = (column cx, row group g of 8 output rows)
    for (int item = tid; item < rawW * 4; item += kItThreads) {
      const int g = item / rawW, cx = item - g * rawW;
      const float* col = raw + (g * 8) * rawS + cx;
      for (int i = 0; i < 8; ++i) {      // direct sums: no add/subtract recurrence (see box15)
        float s;
        if (GAUSS) {
          s = col[(i + m) * rawS] * taps.k[0];
          for (int d = 1; d <= m; ++d) s += (col[(i + m + d) * rawS] + col[(i + m - d) * rawS]) * taps.k[d];
        } else {
          s = 0.f;
          for (int j = 0; j < win; ++j) s += col[(i + j) * rawS];
        }
        Vt[cx * 33 + g * 8 + i] = s;
      }
    }
    __syncthreads();
    // horizontal: lane = output row, warp = group of 8 output columns
    {
      const float* rowp = Vt + (warp * 8) * 33 + lane;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        float s;
        if (GAUSS) {
          s = rowp[(i + m) * 33] * taps.k[0];
          for (int d = 1; d <= m; ++d) s += taps.k[d] * (rowp[(i + m - d) * 33] + rowp[(i + m + d) * 33]);
        } else {
          s = 0.f;
          for (int j = 0; j < win; ++j) s += rowp[(i + j) * 33];
        }
        sums[c][i] = s;
      }
    }
    // the next plane's raw load may start now (raw was last read before the previous barrier);
    // its vertical pass only starts after the barrier that follows that load, i.e. after every
    // thread finished reading Vt above.
  }
  __syncthreads();  // all reads of raw/Vt done before fl (aliased) is written

  const float inv_area = GAUSS ? 1.f : 1.f / (float)(win * win);
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const float g11 = sums[0][i] * inv_area, g12 = sums[1][i] * inv_area, g22 = sums[2][i] * inv_area;
    const float h1 = sums[3][i] * inv_area, h2 = sums[4][i] * inv_area;
    // differences of products with the rounding error of one product recovered by FMA
    const float w12 = g12 * g12;
    const float det = fmaf(g11, g22, -w12) + fmaf(-g12, g12, w12);
    const float idet = 1.f / (det + 1e-3f);
    const float t1 = g12 * h1;
    const float nx = fmaf(g11, h2, -t1) + fmaf(-g12, h1, t1);
    const float t2 = g12 * h2;
    const float ny = fmaf(g22, h1, -t2) + fmaf(-g12, h2, t2);
    fl[lane * (kItTW + 1) + warp * 8 + i] = make_float2(nx * idet, ny * idet);
  }
  __syncthreads();

  // global phase: lanes along x
  const int tx = tid & 63;
  const int x = ox0 + tx;
  if (x < w) {
#pragma unroll 2
    for (int i = 0; i < 8; ++i) {
      const int ty = (tid >> 6) + 4 * i;
      const int y = oy0 + ty;
      if (y >= h) break;
      const float2 f = fl[ty * (kItTW + 1) + tx];
      if (UPDATE) {
        float mm[5];
        update_matrices_px(R + (size_t)pair * 5 * n, R + (size_t)(pair + 1) * 5 * n, (int)n, w, h, x, y, f.x, f.y, mm);
        float* Mo = Mout + (size_t)pair * 5 * n + (size_t)y * w + x;
#pragma unroll
        for (int c = 0; c < 5; ++c) Mo[c * n] = mm[c];
      } else {
        reinterpret_cast<float2*>(flow_out.p[blockIdx.z])[(size_t)y * w + x] = f;
      }
    }
  }
}

static inline size_t iter_smem_bytes(int m) {
  const int rawW = kItTW + 2 * m, rawH = kItTH + 2 * m;
  size_t box = ((size_t)rawH * (rawW + 2) + (size_t)rawW * 33) * sizeof(float);
  size_t fl = (size_t)(kItTW + 1) * kItTH * sizeof(float2);
  return box > fl ? box : fl;
}


// ---------------------------------------------------------------------------------------------
// The same iteration specialised for the reference's winSize = 15 (m = 7): the production path.
// Differences from the generic kernel above:
//   * no raw tile in shared memory: each thread item (column, 8-row group) pulls its 22 rows
//     straight from global memory (coalesced along x; the 2.75x re-reads between row groups
//     hit L1), forms the vertical 15-sums in registers and writes them transposed;
//   * the loads of plane c+1 are issued before the barrier and the horizontal pass of plane c,
//     so global latency overlaps shared-memory work (software pipeline, double-buffered Vt);
//   * tile 48 x 32 makes every phase fill the 256 threads: vertical 62 cols x 4 groups = 248
//     items, horizontal 32 rows x 8 groups of 6 columns = 256 items, update 6 pixels/thread;
//   * one barrier per plane.
// ---------------------------------------------------------------------------------------------
// 15-wide window sums WITHOUT a sliding (add-new / subtract-old) recurrence: after a window has
// passed over large values the subtraction leaves their rounding residue in sums that should be
// ~0 (flat regions next to strong edges), which the 2x2 solve then amplifies -- the reason
// OpenCV keeps these sums in double.  Instead (van Herk / Gil-Werman for sums): the NOUT+14
// inputs split into block A = t[0..14] and block B = t[15..]; window i = suffix_A[i] +
// prefix_B[i+14].  Only additions, 14 + (NOUT-2) + (NOUT-1) of them, and float accuracy
// relative to the window's own magnitude.
template <int NOUT>
__device__ __forceinline__ void box15(const float* t /* NOUT+14 */, float* out /* NOUT */) {
  static_assert(NOUT >= 2 && NOUT <= 15, "two blocks of 15 must cover every window");
  float suf[15];
  suf[14] = t[14];
#pragma unroll
  for (int j = 13; j >= 0; --j) suf[j] = suf[j + 1] + t[j];
  out[0] = suf[0];
  float pre = t[15];
  out[1] = suf[1] + pre;
#pragma unroll
  for (int i = 2; i < NOUT; ++i) {
    pre += t[14 + i];
    out[i] = suf[i] + pre;
  }
}

constexpr int kFiTW = 48, kFiTH = 32, kFiThreads = 256, kFiM = 7;
constexpr int kFiHistStride = 2 * 65;   // fused FlowHistogram: per-warp table of 64 + 1 trash + 64 + 1 trash counters
constexpr int kFiRawW = kFiTW + 2 * kFiM;     // 62
constexpr int kFiRows = 8 + 2 * kFiM;         // 22 input rows per vertical item
constexpr int kFiGC = 6;                      // output columns per horizontal item
constexpr int kFiVtWords = kFiRawW * 33;      // one transposed vertical-sum buffer
constexpr int kFiFlStride = kFiTW + 1;        // float2 row stride of the staged flow (bank spread)

// Global-memory phase shared by both winSize-15 kernels.
//   UPDATE: each thread takes two vertically adjacent pixels, consecutive lanes on consecutive x
//           (update_matrices_vpair): unit-stride R1 gathers with a shared middle row.  Measured on
//           B200 against the alternatives: one pixel per thread 618 us, two horizontally adjacent
//           pixels with 8-byte R0 / M' accesses 555 us per 16-pair level-0 launch.
//           R1 footprints come from `win` when it fits (iter15_win_kernel).
//   !UPDATE: two horizontally adjacent pixels per thread so the flow goes out as 16-byte stores.
template <bool UPDATE, bool HIST>
__device__ __forceinline__ void iter15_global_phase(const float2* fl, unsigned* fh, float* __restrict__ Mout,
                                                    const float* __restrict__ R, R1Win win, const PtrBatch<float>& flow_out,
                                                    int32_t* __restrict__ flow_hist, int w, int h, int pair, int pz, int ox0, int oy0) {
  const int tid = threadIdx.x, warp = tid >> 5;
  const size_t n = (size_t)w * h;
  const int ni = (int)n;
  if (UPDATE) {
    const float* R0 = R + (size_t)pair * 5 * n;
    const float* R1 = R0 + 5 * n;
    float* Mp = Mout + (size_t)pair * 5 * n;
#pragma unroll 1
    for (int i = 0; i < (kFiTW * kFiTH) / (2 * kFiThreads); ++i) {
      const int p2 = tid + i * kFiThreads;          // vertical pixel-pair index inside the tile
      const int tp = p2 / kFiTW, tx = p2 - tp * kFiTW;
      const int x = ox0 + tx, y = oy0 + 2 * tp;
      if (x >= w || y >= h) continue;
      const float2 fa = fl[(2 * tp) * kFiFlStride + tx];
      const float2 fb = fl[(2 * tp + 1) * kFiFlStride + tx];
      float* Mo = Mp + (y * w + x);
      float ma[5], mb[5];
      if (y + 1 < h) {
        update_matrices_vpair(R0, R1, win, ni, w, h, x, y, fa, fb, ma, mb);
#pragma unroll
        for (int c = 0; c < 5; ++c) { *Mo = ma[c]; *padd(Mo, w) = mb[c]; Mo = padd(Mo, ni); }
      } else {
        update_matrices_px(R0, R1, ni, w, h, x, y, fa.x, fa.y, ma);
#pragma unroll
        for (int c = 0; c < 5; ++c) Mo[c * ni] = ma[c];
      }
    }
    return;
  }
  const bool pair_ok = (w & 1) == 0;
#pragma unroll 1
  for (int i = 0; i < (kFiTW * kFiTH) / (2 * kFiThreads); ++i) {
    const int p2 = tid + i * kFiThreads;            // horizontal pixel-pair index inside the tile
    const int ty = p2 / (kFiTW / 2), tx = (p2 - ty * (kFiTW / 2)) * 2;
    const int x = ox0 + tx, y = oy0 + ty;
    if (x >= w || y >= h) continue;
    const float2 fa = fl[ty * kFiFlStride + tx];
    const float2 fb = fl[ty * kFiFlStride + tx + 1];
    const bool two = (x + 1 < w);
    const int o = y * w + x;
    if (flow_out.p[pz] != nullptr) {
      float2* fo = reinterpret_cast<float2*>(flow_out.p[pz]) + o;
      if (two && pair_ok && ((reinterpret_cast<uintptr_t>(fo) & 15u) == 0)) {
        *reinterpret_cast<float4*>(fo) = make_float4(fa.x, fa.y, fb.x, fb.y);
      } else {
        fo[0] = fa;
        if (two) fo[1] = fb;
      }
    }
    if (HIST) {
      // fused FlowHistogram (flow_histogram_kernel_cpu.cpp:33-49) of the flow just produced
      // per-warp rows: 64 magnitude bins, trash, 64 angle bins, trash -- dropped values are clamped onto the
      // trash entries so the updates need no predicate (see flow_hist_kernel)
      unsigned* my = fh + warp * kFiHistStride;
      int bm, ba;
      flow_bins_fast(fa.x, fa.y, bm, ba);
      atomicAdd(my + min((unsigned)bm, 64u), 1u);
      atomicAdd(my + 65 + min((unsigned)ba, 64u), 1u);
      if (two) {
        flow_bins_fast(fb.x, fb.y, bm, ba);
        atomicAdd(my + min((unsigned)bm, 64u), 1u);
        atomicAdd(my + 65 + min((unsigned)ba, 64u), 1u);
      }
    }
  }
  if (HIST) {
    __syncthreads();
    if (tid < STB_FLOWHIST_INTS) {
      unsigned sum = 0;
#pragma unroll
      for (int wq = 0; wq < kFiThreads / 32; ++wq) sum += fh[wq * kFiHistStride + tid + (tid >> 6)];
      if (sum) atomicAdd(flow_hist + (size_t)pair * STB_FLOWHIST_INTS + tid, (int)sum);
    }
  }
}

// 2x2 solve of the winSize-15 kernels on the UN-normalised window sums: the 1/225 factors of
// OpenCV's g = sum * scale cancel between numerator and determinant, only its +1e-3 scales by
// 225^2.  Differences of products carry the rounding error of one product through an FMA;
// the reciprocal is MUFU.RCP (1 ulp), 1.2e-7 relative on the flow.  Saves the five scalings and
// the ~10-instruction IEEE division per pixel (level-0 update launch 535 -> 525 us).
__device__ __forceinline__ float2 solve_flow15(float g11, float g12, float g22, float h1, float h2) {
  const float w12 = g12 * g12;
  const float det = fmaf(g11, g22, -w12) + fmaf(-g12, g12, w12);
  const float den = det + 1e-3f * 225.f * 225.f;
  float idet;
#ifdef STB_CPU_EMU
  idet = 1.f / den;
#else
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(idet) : "f"(den));
#endif
  const float t1 = g12 * h1;
  const float nx = fmaf(g11, h2, -t1) + fmaf(-g12, h1, t1);
  const float t2 = g12 * h2;
  const float ny = fmaf(g22, h1, -t2) + fmaf(-g12, h2, t2);
  return make_float2(nx * idet, ny * idet);
}

// Horizontal pass of one plane over its transposed vertical sums vt: lane = output row, warp = group
// of kFiGC output columns.
__device__ __forceinline__ void box15_rows(const float* vt, float out[kFiGC]) {
  const float* rowp = vt + ((threadIdx.x >> 5) * kFiGC) * 33 + (threadIdx.x & 31);
  float t[kFiGC + 14];
#pragma unroll
  for (int j = 0; j < kFiGC + 14; ++j) t[j] = rowp[j * 33];
  box15<kFiGC>(t, out);
}

// Flow of this thread's output i (row lane, column warp * kFiGC + i) from the window sums, staged in
// fl for the global phase.
__device__ __forceinline__ float2 stage_flow15(float2* fl, const float (&sums)[5][kFiGC], int i) {
  const float2 f = solve_flow15(sums[0][i], sums[1][i], sums[2][i], sums[3][i], sums[4][i]);
  fl[(threadIdx.x & 31) * kFiFlStride + (threadIdx.x >> 5) * kFiGC + i] = f;
  return f;
}

template <bool UPDATE, bool HIST>
__global__ void __launch_bounds__(kFiThreads, 4)
iter15_kernel(const float* __restrict__ Min, float* __restrict__ Mout, const float* __restrict__ R,
              PtrBatch<float> flow_out, int32_t* __restrict__ flow_hist, int w, int h, int pair0, TileOrder ord) {
  __shared__ float Vt[2][kFiVtWords];
  __shared__ float2 fl[kFiTH * kFiFlStride];
  __shared__ unsigned fh[HIST ? (kFiThreads / 32) * kFiHistStride : 1];   // warp-private 128-bin tables
  if (HIST) {
    for (int i = threadIdx.x; i < (kFiThreads / 32) * kFiHistStride; i += kFiThreads) fh[i] = 0u;
  }

  const int tid = threadIdx.x;
  int btx, bty, bpz;
  tile_of_band_order(ord, (int)blockIdx.x, btx, bty, bpz);
  const int pair = pair0 + bpz;
  const size_t n = (size_t)w * h;
  const float* Mp = Min + (size_t)pair * 5 * n;
  const int ox0 = btx * kFiTW, oy0 = bty * kFiTH;

  // vertical item of this thread
  // 64 thread slots per row group (62 active): a warp never straddles two groups, which would
  // make its shared accesses of the two groups collide in the same banks
  const int vg = tid >> 6, vcx = tid & 63;
  const bool vact = vcx < kFiRawW;
  const int gx = min(max(ox0 + vcx - kFiM, 0), w - 1);
  const int y_first = oy0 + vg * 8 - kFiM;
  // row offsets are the same for every plane
  const bool interior_rows = (y_first >= 0) && (y_first + kFiRows - 1 <= h - 1);
  const float* col0 = Mp + (size_t)min(max(y_first, 0), h - 1) * w + gx;

  float v[kFiRows];
  auto load_plane = [&](int c) {
    const float* pl = col0 + (size_t)c * n;
    if (interior_rows) {
#pragma unroll
      for (int j = 0; j < kFiRows; ++j) v[j] = __ldg(pl + (size_t)j * w);
    } else {
      const float* base = Mp + (size_t)c * n + gx;
#pragma unroll
      for (int j = 0; j < kFiRows; ++j) v[j] = __ldg(base + (size_t)min(max(y_first + j, 0), h - 1) * w);
    }
  };

  float sums[5][kFiGC];
  if (vact) load_plane(0);
#pragma unroll
  for (int c = 0; c < 5; ++c) {
    float* vt = Vt[c & 1];
    if (vact) {
      float vs[8];
      box15<8>(v, vs);
      float* o = vt + vcx * 33 + vg * 8;
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] = vs[i];
      if (c < 4) load_plane(c + 1);   // in flight across the barrier and the horizontal pass
    }
    __syncthreads();
    box15_rows(vt, sums[c]);
    // Vt[c&1] is next written for plane c+2, after the barrier of plane c+1: safe.
  }

#pragma unroll
  for (int i = 0; i < kFiGC; ++i) stage_flow15(fl, sums, i);
  __syncthreads();

  iter15_global_phase<UPDATE, HIST>(fl, fh, Mout, R, kNoR1Win, flow_out, flow_hist, w, h, pair, bpz, ox0, oy0);
}

// ---------------------------------------------------------------------------------------------
// TMA-staged variant of the winSize-15 iteration (the production path when rows are 16-byte
// aligned, i.e. w % 4 == 0).  The 46 x 64 raw tile of each M plane (tile + 7-pixel halo, box
// padded to 64 columns = 256 B) is fetched by ONE cp.async.bulk.tensor issued by one thread into
// a two-stage shared-memory ring (plane c+2 is in flight while plane c is consumed; completion
// through an mbarrier).  The box starts at x = tile_x - 8 so that its innermost coordinate is a
// multiple of 4 floats (TMA faults on an unaligned inner coordinate).  This removes the 110 per-thread global loads of the LDG variant above
// and all their 64-bit address arithmetic from the vertical pass (shared loads with immediate
// offsets instead) and keeps HBM latency off the critical path.  Out-of-image elements are
// zero-filled by TMA; tiles touching the image border therefore take a clamped-index read path
// (replicate border, as OpenCV's box filter).
// ---------------------------------------------------------------------------------------------
constexpr int kTmRawW = 64;                               // box width (>= kFiRawW = 62, 256-byte rows)
constexpr int kTmRawH = kFiTH + 2 * kFiM;                 // 46
constexpr int kTmStageFloats = kTmRawW * kTmRawH;         // 2944 floats = 11776 B per stage
constexpr unsigned kTmStageBytes = kTmStageFloats * sizeof(float);

#ifdef STB_CPU_EMU
__device__ __forceinline__ void tma_mbar_init(unsigned long long*, int) {}
// the emulated copy is synchronous in thread 0: a block barrier stands in for the mbarrier wait
__device__ __forceinline__ void tma_mbar_wait(unsigned long long*, unsigned) { __syncthreads(); }
template <int BW = kTmRawW, int BH = kTmRawH, bool TX = true>
__device__ __forceinline__ void tma_load_tile(float* dst, const TmaMap3D* m, int x0, int y0, int z, unsigned long long*) {
  if (x0 & 3) { fprintf(stderr, "cuda_emu: TMA inner coordinate %d is not 16-byte aligned\n", x0); abort(); }
  for (int r = 0; r < BH; ++r)
    for (int c = 0; c < BW; ++c) {
      const int x = x0 + c, y = y0 + r;
      dst[r * BW + c] = (x >= 0 && x < m->w && y >= 0 && y < m->h) ? m->base[((size_t)z * m->h + y) * m->w + x] : 0.f;
    }
}
__device__ __forceinline__ void tma_mbar_arrive(unsigned long long*) {}
#else
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void tma_mbar_init(unsigned long long* bar, int count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void tma_mbar_wait(unsigned long long* bar, unsigned parity) {
  const unsigned addr = smem_u32(bar);
  // try_wait suspends for a hardware-defined time slice; bound the retries so that a faulty
  // descriptor traps (reported as a launch failure) instead of hanging the GPU
  for (unsigned spin = 0; spin < (1u << 24); ++spin) {
    unsigned done;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(done)
        : "r"(addr), "r"(parity)
        : "memory");
    if (done) return;
  }
  __trap();
}
__device__ __forceinline__ void tma_mbar_arrive(unsigned long long* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// TX = false: the caller has already armed the barrier with the byte count of several copies
template <int BW = kTmRawW, int BH = kTmRawH, bool TX = true>
__device__ __forceinline__ void tma_load_tile(float* dst, const TmaMap3D* map, int x0, int y0, int z, unsigned long long* bar) {
  if (TX) asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"((unsigned)(BW * BH * sizeof(float))) : "memory");
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::"r"(smem_u32(dst)),
      "l"(reinterpret_cast<unsigned long long>(map)), "r"(x0), "r"(y0), "r"(z), "r"(smem_u32(bar))
      : "memory");
}
#endif

// Box phase of iter15_tma_kernel and iter15_win_kernel: initialises bars[0 .. NBARS) (the ones past the
// two of the ring are the caller's), streams the tile's five M planes through the ring raw / bars[0..1],
// and leaves the horizontal 15-sums of this thread's outputs in sums.  The shared buffers are passed in
// because one kernel holds them as static arrays and the other in its dynamic overlay.  Ends with a
// barrier after the last read of raw and Vt, so the caller may overlay them.
template <int NBARS>
__device__ __forceinline__ void iter15_tma_box(float (*raw)[kTmStageFloats], float (*Vt)[kFiVtWords], unsigned long long* bars,
                                               const TmaMap3D* map_in, const TmaMap3D* map_R, bool prefetch_R, bool last_pair,
                                               int w, int h, int pair, int ox0, int oy0, float (&sums)[5][kFiGC]) {
  static_assert(kFiRawW + 1 <= kTmRawW && (kFiTW % 4) == 0, "box covers the halo'd tile from an aligned origin");
  const int tid = threadIdx.x;
  // box origin (may be negative).  The innermost TMA coordinate must be 16-byte aligned (measured:
  // an unaligned x traps), so the box starts one column early: raw column cx lives at box column cx+1.
  const int bx0 = ox0 - kFiM - 1, by0 = oy0 - kFiM;

  if (tid == 0) {
#pragma unroll
    for (int b = 0; b < NBARS; ++b) tma_mbar_init(&bars[b], 1);
#ifndef STB_CPU_EMU
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
#endif
  }
  __syncthreads();
  if (tid == 0) {
    tma_load_tile(raw[0], map_in, bx0, by0, pair * 5 + 0, &bars[0]);
    tma_load_tile(raw[1], map_in, bx0, by0, pair * 5 + 1, &bars[1]);
  }
  // (pair-fastest order: R1 of this pair is the R0 of the pair next to it, whose block runs at the same time and
  // prefetches it; only the launch's last pair has to pull its own R1)
  if (prefetch_R && tid >= 32 && tid < (last_pair ? 42 : 37)) {
    // the update phase at the end of this block reads this tile of R0 (frame `pair`) and, displaced
    // by the flow, of R1 (frame pair + 1): pull both towards L2 while the box phase runs, so those
    // loads find L2 hits instead of paying DRAM latency on the critical path (543 -> 522 us per
    // 16-pair level-0 launch)
    const int q = tid - 32;                      // 0..4: R0 planes, 5..9: R1 planes
    tma_prefetch_l2(map_R, ox0, oy0, pair * 5 + q);
  }
  // (Prefetching the M boxes of a tile one or two waves ahead, the way updmat_init_kernel does for
  // R, was measured and rejected: 599-628 us vs 533-542 us per 16-pair level-0 launch, with
  // halo'd 64 x 46 boxes as well as exact 48 x 32 tiles -- the prefetched lines do not survive in
  // L2 until they are used, so the traffic is paid twice.)

  // vertical item of this thread
  const int vg = tid >> 6, vcx = tid & 63;                     // 64 slots per row group, 62 active (see iter15_kernel)
  const bool vact = vcx < kFiRawW;
  // tiles whose box pokes outside the image read through clamped indices (replicate border)
  const bool border = (bx0 + 1 < 0) || (by0 < 0) || (bx0 + 1 + kFiRawW > w) || (by0 + kTmRawH > h);
  const int ccol = min(max(bx0 + 1 + vcx, 0), w - 1) - bx0;  // clamped column inside the box

#pragma unroll
  for (int c = 0; c < 5; ++c) {
    const int st = c & 1;
    tma_mbar_wait(&bars[st], (unsigned)((c >> 1) & 1));
    float* vt = Vt[st];
    if (vact) {
      float v[kFiRows];
      if (!border) {
        const float* col = &raw[st][(vg * 8) * kTmRawW + vcx + 1];
#pragma unroll
        for (int j = 0; j < kFiRows; ++j) v[j] = col[j * kTmRawW];
      } else {
#pragma unroll
        for (int j = 0; j < kFiRows; ++j) {
          const int rr = min(max(by0 + vg * 8 + j, 0), h - 1) - by0;
          v[j] = raw[st][rr * kTmRawW + ccol];
        }
      }
      float vs[8];
      box15<8>(v, vs);
      float* o = vt + vcx * 33 + vg * 8;
#pragma unroll
      for (int i = 0; i < 8; ++i) o[i] = vs[i];
    }
    __syncthreads();                                           // raw[st] consumed, Vt[st] complete
    if (tid == 0 && c + 2 < 5) tma_load_tile(raw[st], map_in, bx0, by0, pair * 5 + c + 2, &bars[st]);
    box15_rows(vt, sums[c]);
  }
  __syncthreads();   // every read of raw (plane 4 lives in stage 0) and Vt is done before the caller overlays them
}

template <bool UPDATE, bool HIST>
__global__ void __launch_bounds__(kFiThreads, 4)
iter15_tma_kernel(const STB_GRID_CONSTANT TmaMap3D map_in, float* __restrict__ Mout, const float* __restrict__ R,
                  PtrBatch<float> flow_out, int32_t* __restrict__ flow_hist, int w, int h, int pair0,
                  const STB_GRID_CONSTANT TmaMap3D map_R, int prefetch_R, TileOrder ord) {
  __shared__ __align__(128) float raw[2][kTmStageFloats];     // also reused for the staged flow after the box phase
  __shared__ float Vt[2][kFiVtWords];
  __shared__ __align__(8) unsigned long long bars[2];
  __shared__ unsigned fh[HIST ? (kFiThreads / 32) * kFiHistStride : 1];
  float2* fl = reinterpret_cast<float2*>(&raw[0][0]);       // 32 x 49 float2 = 12544 B <= one stage + part of the next
  static_assert(kFiTH * kFiFlStride * sizeof(float2) <= 2 * kTmStageBytes, "staged flow must fit in the raw ring");

  int btx, bty, bpz;
  tile_of_band_order(ord, (int)blockIdx.x, btx, bty, bpz);
  const int pair = pair0 + bpz;
  const int ox0 = btx * kFiTW, oy0 = bty * kFiTH;

  if (HIST) {
    for (int i = threadIdx.x; i < (kFiThreads / 32) * kFiHistStride; i += kFiThreads) fh[i] = 0u;
  }
  float sums[5][kFiGC];
  iter15_tma_box<2>(raw, Vt, bars, &map_in, &map_R, UPDATE && prefetch_R, bpz == ord.np - 1, w, h, pair, ox0, oy0, sums);

#pragma unroll
  for (int i = 0; i < kFiGC; ++i) stage_flow15(fl, sums, i);
  __syncthreads();

  iter15_global_phase<UPDATE, HIST>(fl, fh, Mout, R, kNoR1Win, flow_out, flow_hist, w, h, pair, bpz, ox0, oy0);
}


// ---------------------------------------------------------------------------------------------
// The update iteration with a FLOW-COMPENSATED R1 WINDOW in shared memory.
// In iter15_tma_kernel the update phase gathers R1 at (x + dx, y + dy) with 30 global loads per
// pixel pair; every warp then sits on the first consumer of those loads (21 % of the kernel's stall
// samples; no pipe above 67 %) -- the register file is full (64 x 1024 threads per SM), so more
// loads in flight per thread are not to be had.  Here the gathers read shared memory instead:
// after the 2x2 solve the block reduces the bounding box of floor(x + dx), floor(y + dy) over its
// in-image pixels; if the box fits 56 x 38 (the 48 x 32 tile + 8 / 6 of slack, its origin rounded
// down to 4 floats for TMA), one thread fetches that box of the five R1 planes with five
// cp.async.bulk.tensor copies whose ORIGIN IS THE DATA-DEPENDENT box corner, while everybody
// issues their (flow-independent) R0 loads; the bilinear footprints are then LDS with immediate
// offsets off one base address.  Smooth flow -- any global motion, however large -- fits; tiles
// that straddle a motion boundary do not and take the global-memory gathers, as do pixel pairs
// whose footprints do not share a row.  Box phase and update loop are iter15_tma_kernel's
// (iter15_tma_box, iter15_global_phase), the latter given the window.
// Shared memory: raw ring + Vt (39.9 KB, dead after the box phase) are overlaid by the staged flow
// (12.25 KB) and the window (5 x 8.4 KB): 55.5 KB per block, still 4 blocks per SM.
// ---------------------------------------------------------------------------------------------
constexpr size_t kWinFlBytes = 12544;                         // 32 x 49 float2
constexpr size_t kWinSmemWin = kWinFlBytes;                   // window starts right after the staged flow
constexpr size_t kWinSmemBars = kWinSmemWin + 5 * kWinPlaneFloats * sizeof(float);   // 55424
constexpr size_t kWinSmemBytes = kWinSmemBars + 64;
static_assert(kWinW * kWinH <= kWinPlaneFloats && (kWinFlBytes % 128) == 0 && ((kWinPlaneFloats * 4) % 128) == 0, "TMA destinations are 128-byte aligned");
static_assert(2 * kTmStageBytes + 2 * kFiVtWords * sizeof(float) <= kWinSmemBars, "box-phase buffers fit under the barriers");

__global__ void __launch_bounds__(kFiThreads, 4)
iter15_win_kernel(const STB_GRID_CONSTANT TmaMap3D map_in, float* __restrict__ Mout, const float* __restrict__ R,
                  int w, int h, int pair0, const STB_GRID_CONSTANT TmaMap3D map_R, int prefetch_R,
                  const STB_GRID_CONSTANT TmaMap3D map_Rw, TileOrder ord) {
#ifdef STB_CPU_EMU
  unsigned char* smem = cuda_emu::dyn_smem();
#else
  extern __shared__ __align__(128) unsigned char smem[];
#endif
  float (*raw)[kTmStageFloats] = reinterpret_cast<float (*)[kTmStageFloats]>(smem);                       // box phase
  float (*Vt)[kFiVtWords] = reinterpret_cast<float (*)[kFiVtWords]>(smem + 2 * kTmStageBytes);            // box phase
  float2* fl = reinterpret_cast<float2*>(smem);                                                            // update phase
  float* win = reinterpret_cast<float*>(smem + kWinSmemWin);                                               // update phase
  unsigned long long* bars = reinterpret_cast<unsigned long long*>(smem + kWinSmemBars);                   // [0,1] M ring, [2] window
  int* wprm = reinterpret_cast<int*>(smem + kWinSmemBars + 24);                                            // wx0, wy0, fits
  __shared__ int s_wbox[8][4];                                                                             // per-warp footprint boxes

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  int btx, bty, bpz;
  tile_of_band_order(ord, (int)blockIdx.x, btx, bty, bpz);
  const int pair = pair0 + bpz;
  const int ox0 = btx * kFiTW, oy0 = bty * kFiTH;

  float sums[5][kFiGC];
  iter15_tma_box<3>(raw, Vt, bars, &map_in, &map_R, prefetch_R != 0, bpz == ord.np - 1, w, h, pair, ox0, oy0, sums);

  // ---- solve + bounding box of the bilinear footprints of this thread's pixels (row oy0 + lane, columns ox0 + 6 warp ..)
  int minx = 0x7fffffff, miny = 0x7fffffff, maxx = -1, maxy = -1;
  {
    const int y = oy0 + lane;
#pragma unroll
    for (int i = 0; i < kFiGC; ++i) {
      const float2 f = stage_flow15(fl, sums, i);
      const int x = ox0 + warp * kFiGC + i;
      if (x < w && y < h) {
        const int x1 = __float2int_rd((float)x + f.x), y1 = __float2int_rd((float)y + f.y);
        if ((unsigned)x1 < (unsigned)(w - 1) && (unsigned)y1 < (unsigned)(h - 1)) {
          minx = min(minx, x1); maxx = max(maxx, x1 + 1);
          miny = min(miny, y1); maxy = max(maxy, y1 + 1);
        }
      }
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
      minx = min(minx, __shfl_xor_sync(0xffffffffu, minx, d)); maxx = max(maxx, __shfl_xor_sync(0xffffffffu, maxx, d));
      miny = min(miny, __shfl_xor_sync(0xffffffffu, miny, d)); maxy = max(maxy, __shfl_xor_sync(0xffffffffu, maxy, d));
    }
  }
  if (lane == 0) { s_wbox[warp][0] = minx; s_wbox[warp][1] = maxx; s_wbox[warp][2] = miny; s_wbox[warp][3] = maxy; }
  __syncthreads();   // staged flow + warp boxes visible
  if (tid == 0) {
    int bx_lo = 0x7fffffff, bx_hi = -1, by_lo = 0x7fffffff, by_hi = -1;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      bx_lo = min(bx_lo, s_wbox[q][0]); bx_hi = max(bx_hi, s_wbox[q][1]);
      by_lo = min(by_lo, s_wbox[q][2]); by_hi = max(by_hi, s_wbox[q][3]);
    }
    const int wx0 = bx_lo & ~3, wy0 = by_lo;
    const int fits = (bx_hi >= 0) && (bx_hi - wx0 < kWinW) && (by_hi - wy0 < kWinH);
    wprm[0] = wx0; wprm[1] = wy0; wprm[2] = fits;
    if (fits) {
#ifndef STB_CPU_EMU
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(&bars[2])),
                   "r"((unsigned)(5 * kWinW * kWinH * sizeof(float))) : "memory");
#endif
#pragma unroll
      for (int c = 0; c < 5; ++c)
        tma_load_tile<kWinW, kWinH, false>(win + c * kWinPlaneFloats, &map_Rw, wx0, wy0, (pair + 1) * 5 + c, &bars[2]);
    } else {
      tma_mbar_arrive(&bars[2]);      // nothing to wait for: release the parameters
    }
  }

  // ---- update phase: vertical pixel pairs through the window when it fits
  tma_mbar_wait(&bars[2], 0u);
  const R1Win rw = {win, wprm[0], wprm[1], wprm[2] != 0};
  iter15_global_phase<true, false>(fl, nullptr, Mout, R, rw, PtrBatch<float>{}, nullptr, w, h, pair, bpz, ox0, oy0);
}

}  // namespace stb

// =============================================================================================
// host side: handle, workspace, level-major chunked schedule
// =============================================================================================
using namespace stb;

namespace stb { struct FbGraph; static void graph_free(FbGraph* g); }
struct stb_farneback {
  int W, H, max_pairs, device;
  stb_farneback_params prm;
  int nscales;
  int w[8], h[8];
  PolyConsts pc;
  WinTaps taps;     // Gaussian window taps (flags & OPTFLOW_FARNEBACK_GAUSSIAN), zero otherwise
  PyrParams pyr[kMaxScales];
  MergedTaps merged[kMaxScales];
  int pow2[kMaxScales];
  int fast_pyr;          // levels 1.. from one horizontal + one vertical launch (pyr_h_kernel / pyr_v_kernel)
  PyrTaps3 taps3;
  // device workspace
  uint8_t* gray;    // [F][H*W]
  float* I;         // [F][N_0] slots: I_k of frame f at I + I_off[k] + f * I_stride[k]
  size_t I_off[kMaxScales], I_stride[kMaxScales];
  float* R;         // [F][5][N_0]   level 0 (and, before its expansion is written, the pyramid's intermediate)
  float* Rk[kMaxScales];   // [F][5][N_k] per level: Rk[0] = R; separate buffers so that the expansions of all levels can be
                           // produced ahead of (and concurrently with) the displacement iterations of the coarser levels
  cudaStream_t s_prep;     // second lane: gray -> pyramid -> polynomial expansions of every level (low priority)
  cudaEvent_t ev_fork, ev_R[kMaxScales];
  // CUDA-graph replay of a whole batch (see graph_run): one instantiated graph per (pairs, outputs) shape
  int use_graph;
  cudaStream_t s_cap;
  std::vector<stb::FbGraph*> graphs;
  float* M[2];      // [P][5][N_k]   (N_0 sized)
  float* flow[2];   // [P][N_k*2]    level >= 1 only (N_1 sized)
  float* flow0;     // [P][N_0*2]    lazily allocated: level-0 flow when the caller wants only histograms
  size_t bytes;
  // debug taps
  int dbg_level, dbg_pair;
  float *dbg_I0, *dbg_I1, *dbg_R0, *dbg_R1, *dbg_M0, *dbg_flow;
  // TMA descriptors of the two M ping-pong buffers at every level ([5*P planes][h_k][w_k] floats)
  TmaMap3D tmap[2][kMaxScales];
  int use_tma[kMaxScales];
  // R at every level ([5*F planes][h_k][w_k]) for the L2 prefetch of the update phase's tiles
  TmaMap3D tmapR[kMaxScales];
  int prefetch_R[kMaxScales];
  TmaMap3D tmapRw[kMaxScales];   // same tensor, 56 x 38 boxes: iter15_win_kernel's flow-compensated R1 window
  int use_win[kMaxScales];
  TmaMap3D tmapRi[kMaxScales];   // same tensor, 64 x 8 boxes: updmat_init_kernel's prefetch-ahead
  int prefetch_Ri[kMaxScales];
  // measurement hook: event pairs around the level-0 update-iteration kernels
  int profile;
  std::vector<cudaEvent_t> ev_free;
  std::vector<cudaEvent_t> ev_used;   // (begin, end) pairs
  long long prof_launches;
  long long prof_pair_iters;   // sum over timed launches of the pairs each one processed
};

namespace stb {

static int cv_round_d(double v) { return (int)std::nearbyint(v); }

static void gaussian_taps(int ksize, double sigma, float* taps) {
  // cv::getGaussianKernel(ksize, sigma, CV_32F)
  if (ksize == 3 && sigma <= 0) { taps[0] = 0.25f; taps[1] = 0.5f; taps[2] = 0.25f; return; }
  if (sigma <= 0) sigma = 0.3 * ((ksize - 1) * 0.5 - 1) + 0.8;
  double t[kMaxGaussTaps], sum = 0;
  for (int i = 0; i < ksize; ++i) {
    const double x = i - (ksize - 1) * 0.5;
    t[i] = std::exp(-0.5 / (sigma * sigma) * x * x);
    sum += t[i];
  }
  for (int i = 0; i < ksize; ++i) taps[i] = (float)(t[i] / sum);
}

static bool invert_spd6(double A[6][6], double inv[6][6]) {
  // Cholesky A = L L^T, then solve for the identity columns
  double L[6][6] = {};
  for (int i = 0; i < 6; ++i)
    for (int j = 0; j <= i; ++j) {
      double s = A[i][j];
      for (int k = 0; k < j; ++k) s -= L[i][k] * L[j][k];
      if (i == j) { if (s <= 0) return false; L[i][i] = std::sqrt(s); }
      else L[i][j] = s / L[j][j];
    }
  for (int c = 0; c < 6; ++c) {
    double y[6], x[6];
    for (int i = 0; i < 6; ++i) {
      double s = (i == c) ? 1.0 : 0.0;
      for (int k = 0; k < i; ++k) s -= L[i][k] * y[k];
      y[i] = s / L[i][i];
    }
    for (int i = 5; i >= 0; --i) {
      double s = y[i];
      for (int k = i + 1; k < 6; ++k) s -= L[k][i] * x[k];
      x[i] = s / L[i][i];
    }
    for (int i = 0; i < 6; ++i) inv[i][c] = x[i];
  }
  return true;
}

static bool poly_consts(int n, double sigma, PolyConsts* pc) {
  // FarnebackPrepareGaussian (Appendix A.3)
  float gf[2 * kMaxPolyN + 1];
  if (sigma < 1.1920929e-07) sigma = n * 0.3;
  double s = 0;
  for (int x = -n; x <= n; ++x) { gf[x + n] = (float)std::exp(-x * x / (2 * sigma * sigma)); s += gf[x + n]; }
  s = 1. / s;
  for (int x = -n; x <= n; ++x) gf[x + n] = (float)(gf[x + n] * s);
  for (int x = 0; x <= n; ++x) {
    pc->g[x] = gf[x + n];
    pc->xg[x] = (float)(x * gf[x + n]);
    pc->xxg[x] = (float)(x * x * gf[x + n]);
    pc->g2[x] = make_float2(pc->g[x], pc->g[x]);
    pc->xg2[x] = make_float2(pc->xg[x], pc->xg[x]);
    pc->xxg2[x] = make_float2(pc->xxg[x], pc->xxg[x]);
  }
  double G[6][6] = {}, inv[6][6];
  for (int y = -n; y <= n; ++y)
    for (int x = -n; x <= n; ++x) {
      const float gg = gf[y + n] * gf[x + n];  // float products, accumulated in double, as OpenCV does
      G[0][0] += gg;
      G[1][1] += gg * x * x;
      G[3][3] += gg * x * x * x * x;
      G[5][5] += gg * x * x * y * y;
    }
  G[2][2] = G[0][3] = G[0][4] = G[3][0] = G[4][0] = G[1][1];
  G[4][4] = G[3][3];
  G[3][4] = G[4][3] = G[5][5];
  if (!invert_spd6(G, inv)) return false;
  pc->ig11 = (float)inv[1][1]; pc->ig03 = (float)inv[0][3]; pc->ig33 = (float)inv[3][3]; pc->ig55 = (float)inv[5][5];
  return true;
}

constexpr int kFlagGaussian = 256;   // cv::OPTFLOW_FARNEBACK_GAUSSIAN

static int validate_params(const stb_farneback_params& p) {
  if (p.num_levels < 0 || p.num_levels > kMaxScales - 1 || !(p.pyr_scale >= 0.5 && p.pyr_scale < 1.0) || (p.fast_pyramids != 0 && p.fast_pyramids != 1) ||
      p.win_size < 3 || (p.win_size & 1) == 0 || p.win_size > 2 * kItMaxHalo + 1 || p.num_iters < 1 ||
      p.poly_n < 3 || p.poly_n > kMaxPolyN || (p.flags & ~kFlagGaussian) != 0) {
    set_error("stb_farneback: unsupported parameters (levels=%d pyr_scale=%g fast=%d win=%d iters=%d poly_n=%d flags=%d)",
              p.num_levels, p.pyr_scale, p.fast_pyramids, p.win_size, p.num_iters, p.poly_n, p.flags);
    return STB_ERR_UNSUPPORTED;
  }
  return STB_OK;
}

static int plan_levels(int W, int H, const stb_farneback_params& p, int* ws, int* hs) {
  // Appendix A.1
  int k; double scale = 1;
  for (k = 0; k < p.num_levels; ++k) {
    scale *= p.pyr_scale;
    if (W * scale < 32 || H * scale < 32) break;
  }
  const int levels = k;
  for (k = 0; k <= levels; ++k) {
    double sc = 1;
    for (int i = 0; i < k; ++i) sc *= p.pyr_scale;
    ws[k] = cv_round_d(W * sc);
    hs[k] = cv_round_d(H * sc);
  }
  return levels + 1;
}

#ifdef STB_CPU_EMU
static bool make_tmap(TmaMap3D* m, float* base, int w, int h, int planes, int = 0, int = 0) {
  m->base = base; m->w = w; m->h = h; m->planes = planes;
  return true;
}
#else
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                    const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                    CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static PFN_encodeTiled get_encode_tiled() {
  static PFN_encodeTiled fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* sym = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(sym);
    else
      (void)cudaGetLastError();
  }
  return fn;
}
// [planes][h][w] f32, box = box_w x box_h x 1 (default: the 64 x 46 raw tile of the box filter), zero fill outside the tensor
static bool make_tmap(TmaMap3D* m, float* base, int w, int h, int planes, int box_w = kTmRawW, int box_h = kTmRawH) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc || (w & 3) != 0 || (reinterpret_cast<uintptr_t>(base) & 15u) != 0) return false;
  const cuuint64_t dims[3] = {(cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)planes};
  const cuuint64_t strides[2] = {(cuuint64_t)w * sizeof(float), (cuuint64_t)w * h * sizeof(float)};
  const cuuint32_t box[3] = {(cuuint32_t)box_w, (cuuint32_t)box_h, 1u};
  const cuuint32_t estr[3] = {1u, 1u, 1u};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
#endif

struct WsLayout { size_t gray, I, R, Rc, M, flow, total; };

static WsLayout ws_layout(int W, int H, int P, int nscales, const int* ws, const int* hs) {
  auto al = [](size_t b) { return (b + 255) & ~(size_t)255; };
  const size_t F = (size_t)P + 1, N0 = (size_t)W * H;
  const size_t N1 = nscales > 1 ? (size_t)ws[1] * hs[1] : 0;
  WsLayout l;
  l.gray = al(F * N0);
  l.I = al(F * N0 * sizeof(float));
  l.R = al(F * 5 * N0 * sizeof(float));
  l.Rc = 0;                                        // R_1 .. R_3, each 256-byte aligned (8 / 16-byte vector accesses)
  for (int k = 1; k < nscales; ++k) l.Rc += al(F * 5 * (size_t)ws[k] * hs[k] * sizeof(float));
  l.M = al((size_t)P * 5 * N0 * sizeof(float));
  l.flow = al((size_t)P * N1 * 2 * sizeof(float));
  l.total = l.gray + l.I + l.R + l.Rc + 2 * l.M + 2 * l.flow;
  return l;
}

}  // namespace stb

extern "C" {

void stb_farneback_default_params(stb_farneback_params* p) {
  if (!p) return;
  p->num_levels = 3; p->pyr_scale = 0.5; p->fast_pyramids = 0; p->win_size = 15;
  p->num_iters = 3; p->poly_n = 5; p->poly_sigma = 1.2; p->flags = 0;
}

size_t stb_farneback_workspace_bytes(int width, int height, int max_pairs, const stb_farneback_params* params) {
  stb_farneback_params p;
  if (params) p = *params; else stb_farneback_default_params(&p);
  if (width <= 0 || height <= 0 || max_pairs <= 0 || validate_params(p) != STB_OK) return 0;
  int ws[8], hs[8];
  const int ns = plan_levels(width, height, p, ws, hs);
  return ws_layout(width, height, max_pairs, ns, ws, hs).total;
}

int stb_farneback_create(int width, int height, int max_pairs, const stb_farneback_params* params, stb_farneback** out) {
  if (!out) { set_error("stb_farneback_create: out is NULL"); return STB_ERR_INVALID; }
  *out = nullptr;
  stb_farneback_params p;
  if (params) p = *params; else stb_farneback_default_params(&p);
  if (width <= 0 || height <= 0 || max_pairs <= 0 || (long long)width * height > (1ll << 28)) {
    set_error("stb_farneback_create: invalid geometry %dx%d, max_pairs=%d", width, height, max_pairs);
    return STB_ERR_INVALID;
  }
  int rc = validate_params(p);
  if (rc) return rc;
  stb_farneback* h = new (std::nothrow) stb_farneback();
  if (!h) { set_error("stb_farneback_create: out of host memory"); return STB_ERR_ALLOC; }
  h->W = width; h->H = height; h->max_pairs = max_pairs; h->prm = p; h->dbg_level = -1;
  h->device = current_device();
  h->nscales = plan_levels(width, height, p, h->w, h->h);
  {
    // FarnebackUpdateFlow_GaussianBlur's window: sigma = 0.3 * (winSize / 2), float taps exp(-i^2 /
    // (2 sigma^2)) normalised by their double-precision sum over the full (2m + 1)-tap window
    for (int i = 0; i <= kItMaxHalo; ++i) h->taps.k[i] = 0.f;
    const int m = p.win_size / 2;
    const double sigma = m * 0.3;
    double sum = 1;
    h->taps.k[0] = 1.f;
    for (int i = 1; i <= m; ++i) {
      const float t = (float)std::exp(-i * i / (2 * sigma * sigma));
      h->taps.k[i] = t;
      sum += t * 2;
    }
    sum = 1. / sum;
    for (int i = 0; i <= m; ++i) h->taps.k[i] = (float)(h->taps.k[i] * sum);
  }
  if (!poly_consts(p.poly_n, p.poly_sigma, &h->pc)) {
    delete h;
    set_error("stb_farneback_create: singular polynomial basis (poly_sigma=%g)", p.poly_sigma);
    return STB_ERR_INVALID;
  }
  for (int k = 0; k < h->nscales; ++k) {
    PyrParams& q = h->pyr[k];
    double scale = 1;
    for (int i = 0; i < k; ++i) scale *= p.pyr_scale;
    const double sigma = (1. / scale - 1) * 0.5;
    int ksize = cv_round_d(sigma * 5) | 1;
    if (ksize < 3) ksize = 3;
    q.W = width; q.H = height; q.w = h->w[k]; q.h = h->h[k]; q.r = ksize / 2;
    q.scale_x = 1. / ((double)q.w / width);
    q.scale_y = 1. / ((double)q.h / height);
    gaussian_taps(ksize, sigma, q.taps);
    q.max_rows = (int)std::ceil((kPyrTH - 1) * q.scale_y) + 3 + 2 * q.r;
    // exact power-of-two level (and the radii the specialised kernel is compiled for)
    const int expect_r = (k == 1) ? 1 : (k == 2 ? 4 : 9);
    h->pow2[k] = (k >= 1 && k <= 3 && (width % (1 << k)) == 0 && (height % (1 << k)) == 0 &&
                  q.w == (width >> k) && q.h == (height >> k) && q.r == expect_r) ? 1 : 0;
    for (int t = 0; t <= ksize; ++t)
      h->merged[k].c[t] = 0.5f * ((t < ksize ? q.taps[t] : 0.f) + (t > 0 ? q.taps[t - 1] : 0.f));
  }
  {
    // two-launch pyramid for levels >= 1: every level an exact power-of-two size, 32-pixel segments
    bool ok = h->nscales >= 2 && (width % 32) == 0;
    for (int k = 1; k < h->nscales; ++k) ok = ok && h->pow2[k];
    h->fast_pyr = ok ? 1 : 0;
    for (int t = 0; t < 4; ++t) h->taps3.c1[t] = h->nscales > 1 ? h->merged[1].c[t] : 0.f;
    for (int t = 0; t < 10; ++t) h->taps3.c2[t] = h->nscales > 2 ? h->merged[2].c[t] : 0.f;
    for (int t = 0; t < 20; ++t) h->taps3.c3[t] = h->nscales > 3 ? h->merged[3].c[t] : 0.f;
    // pyr_v_kernel packs I_1, I_2, .. one after the other into the frame's N_0 slot; the per-level
    // kernels give every level its own dense [F][N_k] layout
    size_t packed = 0;
    for (int k = 0; k < h->nscales; ++k) {
      const bool in_slot = h->fast_pyr && k >= 1;
      h->I_off[k] = in_slot ? packed : 0;
      h->I_stride[k] = in_slot ? (size_t)width * height : (size_t)h->w[k] * h->h[k];
      if (in_slot) packed += (size_t)h->w[k] * h->h[k];
    }
  }
  const WsLayout l = ws_layout(width, height, max_pairs, h->nscales, h->w, h->h);
  uint8_t* base = nullptr;
  cudaError_t e = cudaMalloc((void**)&base, l.total);
  if (e != cudaSuccess) {
    delete h;
    (void)cudaGetLastError();
    set_error("stb_farneback_create: cudaMalloc(%zu bytes) failed: %s", l.total, cudaGetErrorString(e));
    return (int)e == 100 || (int)e == 35 ? STB_ERR_NO_DEVICE : STB_ERR_ALLOC;
  }
  h->bytes = l.total;
  size_t off = 0;
  h->gray = base; off += l.gray;
  h->I = (float*)(base + off); off += l.I;
  h->R = (float*)(base + off); off += l.R;
  h->Rk[0] = h->R;
  {
    size_t roff = off;
    for (int k = 1; k < h->nscales; ++k) {
      h->Rk[k] = (float*)(base + roff);
      roff += ((size_t)(max_pairs + 1) * 5 * h->w[k] * h->h[k] * sizeof(float) + 255) & ~(size_t)255;
    }
    off += l.Rc;
  }
  h->M[0] = (float*)(base + off); off += l.M;
  h->M[1] = (float*)(base + off); off += l.M;
  h->flow[0] = (float*)(base + off); off += l.flow;
  h->flow[1] = (float*)(base + off); off += l.flow;
  {
    // STB_NO_WIN selects iter15_tma_kernel, the global-gather reference the window kernel is tested against
    const bool no_win = getenv("STB_NO_WIN") != nullptr;
    for (int k = 0; k < h->nscales; ++k) {
      // one box (64 x 46) must make sense for the level; tiny levels keep the LDG kernel
      if (h->w[k] < kTmRawW || h->h[k] < 8) continue;
      if (make_tmap(&h->tmap[0][k], h->M[0], h->w[k], h->h[k], 5 * max_pairs) &&
          make_tmap(&h->tmap[1][k], h->M[1], h->w[k], h->h[k], 5 * max_pairs))
        h->use_tma[k] = 1;
      if (h->use_tma[k] && h->h[k] >= kPfBoxH &&
          make_tmap(&h->tmapR[k], h->Rk[k], h->w[k], h->h[k], 5 * (max_pairs + 1), kPfBoxW, kPfBoxH))
        h->prefetch_R[k] = 1;
      if (h->use_tma[k] && h->prefetch_R[k] && !no_win && h->w[k] >= kWinW && h->h[k] >= kWinH &&
          make_tmap(&h->tmapRw[k], h->Rk[k], h->w[k], h->h[k], 5 * (max_pairs + 1), kWinW, kWinH))
        h->use_win[k] = 1;
      if (make_tmap(&h->tmapRi[k], h->Rk[k], h->w[k], h->h[k], 5 * (max_pairs + 1), 64, kPfInitBoxH))
        h->prefetch_Ri[k] = 1;
    }
  }
#ifndef STB_CPU_EMU
  e = cudaFuncSetAttribute(iter_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)iter_smem_bytes(kItMaxHalo));
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(iter_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)iter_smem_bytes(kItMaxHalo));
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(iter_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)iter_smem_bytes(kItMaxHalo));
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(iter_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)iter_smem_bytes(kItMaxHalo));
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(pyr_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
  if (e == cudaSuccess)
    e = cudaFuncSetAttribute(iter15_win_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kWinSmemBytes);
  if (e != cudaSuccess) {
    cudaFree(base);
    delete h;
    return cuda_fail(e, "cudaFuncSetAttribute");
  }
#endif
  {
    // second lane for the pyramid / polynomial-expansion chain (see run_levels); lowest priority, so the
    // displacement-iteration chain is scheduled first whenever both have blocks ready
    h->use_graph = getenv("STB_NO_GRAPH") ? 0 : 1;   // direct launches, the reference the graph replay is tested against
    int lo = 0, hi = 0;
    cudaError_t e2 = cudaDeviceGetStreamPriorityRange(&lo, &hi);
    if (e2 == cudaSuccess) e2 = cudaStreamCreateWithPriority(&h->s_prep, cudaStreamNonBlocking, lo);
    if (e2 == cudaSuccess) e2 = cudaStreamCreateWithFlags(&h->s_cap, cudaStreamNonBlocking);
    if (e2 == cudaSuccess) e2 = cudaEventCreateWithFlags(&h->ev_fork, cudaEventDisableTiming);
    for (int k = 0; k < kMaxScales && e2 == cudaSuccess; ++k) e2 = cudaEventCreateWithFlags(&h->ev_R[k], cudaEventDisableTiming);
    if (e2 != cudaSuccess) {
      int rc2 = cuda_fail(e2, "stb_farneback_create: second lane");
      stb_farneback_destroy(h);
      return rc2;
    }
  }
  *out = h;
  return STB_OK;
}

int stb_farneback_destroy(stb_farneback* h) {
  if (!h) return STB_OK;
  if (h->s_prep) { cudaStreamSynchronize(h->s_prep); cudaStreamDestroy(h->s_prep); }
  if (h->s_cap) cudaStreamDestroy(h->s_cap);
  for (FbGraph* g : h->graphs) graph_free(g);
  h->graphs.clear();
  if (h->ev_fork) cudaEventDestroy(h->ev_fork);
  for (int k = 0; k < kMaxScales; ++k)
    if (h->ev_R[k]) cudaEventDestroy(h->ev_R[k]);
  if (h->gray) cudaFree(h->gray);
  if (h->flow0) cudaFree(h->flow0);
  for (cudaEvent_t e : h->ev_free) cudaEventDestroy(e);
  for (cudaEvent_t e : h->ev_used) cudaEventDestroy(e);
  delete h;
  return STB_OK;
}

int stb_farneback_levels(const stb_farneback* h, int* widths, int* heights) {
  if (!h) return 0;
  for (int k = 0; k < h->nscales; ++k) {
    if (widths) widths[k] = h->w[k];
    if (heights) heights[k] = h->h[k];
  }
  return h->nscales;
}

int stb_farneback_profile(stb_farneback* h, int enable) {
  if (!h) { set_error("stb_farneback_profile: NULL handle"); return STB_ERR_INVALID; }
  h->profile = enable ? 1 : 0;
  return STB_OK;
}

int stb_farneback_profile_read(stb_farneback* h, double* ms_total, long long* launches, long long* pair_iterations) {
  if (!h) { set_error("stb_farneback_profile_read: NULL handle"); return STB_ERR_INVALID; }
  double total = 0;
  for (size_t i = 0; i + 1 < h->ev_used.size(); i += 2) {
    float ms = 0;
    STB_CUDA(cudaEventSynchronize(h->ev_used[i + 1]));
    STB_CUDA(cudaEventElapsedTime(&ms, h->ev_used[i], h->ev_used[i + 1]));
    total += ms;
  }
  for (cudaEvent_t e : h->ev_used) h->ev_free.push_back(e);
  h->ev_used.clear();
  if (ms_total) *ms_total = total;
  if (launches) *launches = h->prof_launches;
  if (pair_iterations) *pair_iterations = h->prof_pair_iters;
  h->prof_launches = 0;
  h->prof_pair_iters = 0;
  return STB_OK;
}

int stb_farneback_debug_set(stb_farneback* h, int level, int pair, float* d_I0, float* d_I1, float* d_R0, float* d_R1,
                            float* d_M0, float* d_flow_level) {
  if (!h) { set_error("stb_farneback_debug_set: NULL handle"); return STB_ERR_INVALID; }
  h->dbg_level = level; h->dbg_pair = pair;
  h->dbg_I0 = d_I0; h->dbg_I1 = d_I1; h->dbg_R0 = d_R0; h->dbg_R1 = d_R1; h->dbg_M0 = d_M0; h->dbg_flow = d_flow_level;
  return STB_OK;
}

}  // extern "C"

namespace stb {

static int prof_mark(stb_farneback* h, cudaStream_t s) {
  cudaEvent_t e;
  if (!h->ev_free.empty()) { e = h->ev_free.back(); h->ev_free.pop_back(); }
  else STB_CUDA(cudaEventCreate(&e));
  h->ev_used.push_back(e);
  STB_CUDA(cudaEventRecord(e, s));
  return STB_OK;
}

static inline bool fused_hist_available(const stb_farneback* h) {
  return h->prm.win_size / 2 == kFiM && (h->prm.flags & kFlagGaussian) == 0;
}

// I_k and R_k of frames [fa, fb) at level k on stream `sp` (the "prep" work of a level)
static int prep_level(stb_farneback* h, int k, int fa, int fb, cudaStream_t sp) {
  const int w = h->w[k], hh = h->h[k];
  const PyrParams& pp = h->pyr[k];
  const float* Ik = h->I + h->I_off[k];
  const size_t i_stride = h->I_stride[k];
  if (h->fast_pyr && k >= 1) {
    // I_k already produced by pyr_h_kernel / pyr_v_kernel
  } else if (k == 0) {
    // rows of the gray plane and of I are 4/16-byte aligned iff W % 4 == 0 (bases are 256-byte aligned)
    if ((w % 8) == 0)
      stb_launch(pyr0x8_kernel, dim3(ceil_div(w, 256), ceil_div(hh, 8 * kPyr0Rows), fb - fa), dim3(256), 0, sp,
                 (const uint8_t*)h->gray, h->I, w, hh, pp.taps[0], pp.taps[1], pp.taps[2], fa);
    else
      stb_launch(pyr0_kernel, dim3(ceil_div(w, 128), ceil_div(hh, 32), fb - fa), dim3(256), 0, sp,
                 (const uint8_t*)h->gray, h->I, w, hh, pp.taps[0], pp.taps[1], pp.taps[2], fa, (w % 4 == 0) ? 1 : 0);
    STB_CHECK_LAUNCH("pyr0_kernel");
  } else if (h->pow2[k]) {
    const dim3 g(ceil_div(w, 32), ceil_div(hh, k == 3 ? 8 : 16), fb - fa);
    if (k == 1) stb_launch(pyr_pow2_kernel<1>, g, dim3(256), 0, sp, (const uint8_t*)h->gray, h->I, h->W, h->H, h->merged[k], fa);
    else if (k == 2) stb_launch(pyr_pow2_kernel<2>, g, dim3(256), 0, sp, (const uint8_t*)h->gray, h->I, h->W, h->H, h->merged[k], fa);
    else stb_launch(pyr_pow2_kernel<3>, g, dim3(256), 0, sp, (const uint8_t*)h->gray, h->I, h->W, h->H, h->merged[k], fa);
    STB_CHECK_LAUNCH("pyr_pow2_kernel");
  } else {
    const size_t pyr_smem = (size_t)pp.max_rows * kPyrTW * sizeof(float);
    stb_launch(pyr_kernel, dim3(ceil_div(w, kPyrTW), ceil_div(hh, kPyrTH), fb - fa), dim3(kPyrThreads), pyr_smem, sp,
               (const uint8_t*)h->gray, h->I, pp, fa);
    STB_CHECK_LAUNCH("pyr_kernel");
  }
  if (h->prm.poly_n == kPolyN)
    stb_launch(polyexp_kernel, dim3(ceil_div(w, kPeTW), ceil_div(hh, kPeTH), fb - fa), dim3(kPeThreads), 0, sp,
               Ik, i_stride, h->Rk[k], w, hh, h->pc, fa);
  else
    stb_launch(polyexp_generic_kernel, dim3(ceil_div(w, 32), ceil_div(hh, 8), fb - fa), dim3(256), 0, sp,
               Ik, i_stride, h->Rk[k], w, hh, h->pc, h->prm.poly_n, fa);
  STB_CHECK_LAUNCH("polyexp_kernel");
  return STB_OK;
}

// d_hist != NULL: fused FlowHistogram (n*128 int32, pre-zeroed) in the level-0 last iteration, for parameter
// sets with fused_hist_available(h) only; then d_flow entries may be NULL.
//
// Schedule.  A level needs (a) I_k and the polynomial expansion R_k of every frame -- which depend on the
// gray planes only -- and (b) the chain updmat_init -> iterations, which depends on R_k and on the coarser
// level's flow.  (a) for ALL levels runs on the handle's own low-priority stream (forked from the caller's
// stream after the gray conversion, every R_k in its own buffer) while the caller's stream walks the chain
// (b) from the coarsest level in pointer-table chunks of pairs, waiting per level on an event: the small,
// latency-bound launches of the coarse levels (less than one resident wave at level 3) share the GPU with
// the bandwidth-heavy expansion of the fine levels instead of running alone.  The caller's stream waits on
// the level-0 event, recorded last, so the lanes join before the call returns control of the stream.
// The debug taps of I_k / R_k are copied on the prep lane right after level k's prep: with the two-launch
// pyramid I_k (k >= 1) lives in the frame's level-0 slot, which the level-0 pyramid overwrites next.
static int run_levels(stb_farneback* h, int n, float* const* d_flow, cudaStream_t s, int32_t* d_hist = nullptr) {
  const int F = n + 1;
  const int slice = kMaxPtrBatch + 1;    // frames per prep launch: a batch of up to 64 pairs is one slice
  const int m = h->prm.win_size / 2;
  const size_t it_smem = iter_smem_bytes(m);
  int fl_cur = 0;  // h->flow[fl_cur] receives this level's flow (levels >= 1)
  const bool dbg_in_batch = h->dbg_pair >= 0 && h->dbg_pair < n;
  cudaStream_t sp = h->s_prep;
  STB_CUDA(cudaEventRecord(h->ev_fork, s));            // gray planes ready; the previous call on `s` is done with R / I
  STB_CUDA(cudaStreamWaitEvent(sp, h->ev_fork, 0));
  if (h->fast_pyr) {
    // Levels >= 1 from two launches per slice.  The intermediate lives in the level-0 R buffer, which is not
    // written before the level-0 polynomial expansion; I_1.. are packed into the I slots, which the level-0
    // pyramid only overwrites after every level >= 1 has been expanded.
    const int nlev = h->nscales - 1;
    const int items = (h->W >> 5) * h->H;
    int quads = 0;
    for (int k = 1; k <= nlev; ++k) quads += (h->w[k] >> 2) * h->h[k];
    for (int f0 = 0; f0 < F; f0 += slice) {
      const int nf = (f0 + slice < F ? f0 + slice : F) - f0;
      stb_launch(pyr_h_kernel, dim3(ceil_div(items, 128), nf), dim3(128), 0, sp, (const uint8_t*)h->gray, h->R, h->W, h->H, h->taps3,
                 nlev, f0);
      STB_CHECK_LAUNCH("pyr_h_kernel");
      stb_launch(pyr_v_kernel, dim3(ceil_div(quads, 128), nf), dim3(128), 0, sp, (const float*)h->R, h->I, h->W, h->H, h->taps3, nlev,
                 h->I_stride[1], f0);
      STB_CHECK_LAUNCH("pyr_v_kernel");
    }
  }
  for (int k = h->nscales - 1; k >= 0; --k) {
    for (int f0 = 0; f0 < F; f0 += slice) {
      int prc = prep_level(h, k, f0, f0 + slice < F ? f0 + slice : F, sp);
      if (prc) return prc;
    }
    if (h->dbg_level == k && dbg_in_batch) {
      const size_t nk = (size_t)h->w[k] * h->h[k];
      const float* I0 = h->I + h->I_off[k] + (size_t)h->dbg_pair * h->I_stride[k];
      const float* R0 = h->Rk[k] + (size_t)h->dbg_pair * 5 * nk;
      if (h->dbg_I0) STB_CUDA(cudaMemcpyAsync(h->dbg_I0, I0, nk * 4, cudaMemcpyDeviceToDevice, sp));
      if (h->dbg_I1) STB_CUDA(cudaMemcpyAsync(h->dbg_I1, I0 + h->I_stride[k], nk * 4, cudaMemcpyDeviceToDevice, sp));
      if (h->dbg_R0) STB_CUDA(cudaMemcpyAsync(h->dbg_R0, R0, nk * 20, cudaMemcpyDeviceToDevice, sp));
      if (h->dbg_R1) STB_CUDA(cudaMemcpyAsync(h->dbg_R1, R0 + 5 * nk, nk * 20, cudaMemcpyDeviceToDevice, sp));
    }
    STB_CUDA(cudaEventRecord(h->ev_R[k], sp));
  }
  for (int k = h->nscales - 1; k >= 0; --k) {
    const int w = h->w[k], hh = h->h[k];
    const size_t nk = (size_t)w * hh;
    const float* Rk = h->Rk[k];
    const float* coarse = (k == h->nscales - 1) ? nullptr : h->flow[fl_cur ^ 1];
    const int wc = coarse ? h->w[k + 1] : 0, hc = coarse ? h->h[k + 1] : 0;
    const double up_sx = coarse ? 1. / ((double)w / wc) : 0, up_sy = coarse ? 1. / ((double)hh / hc) : 0;
    const bool dbg = (h->dbg_level == k);
    STB_CUDA(cudaStreamWaitEvent(s, h->ev_R[k], 0));
    // Pairs per launch: the whole batch (up to the pointer-table size).  Measured on B200 (1080p,
    // 16-pair batches): 1 pair per level-0 launch 3585 fps, 2 -> 3944, 4 -> 4276, 8 -> 4499.  The
    // kernels are issue/latency bound, so wave quantisation and launch tails (1360 blocks over
    // 592 resident slots = 2.3 waves for one 1080p pair) cost more than keeping one pair's
    // working set (~92 B/px) resident in the 126 MB L2 buys.
    for (int p0 = 0; p0 < n; p0 += kMaxPtrBatch) {
      const int p1 = (p0 + kMaxPtrBatch < n) ? p0 + kMaxPtrBatch : n;
      const int np = p1 - p0;
      {
        // prefetch distance in blocks of the grid's linear order: two resident waves of 4 blocks per SM
        // (the occupancy it was tuned at; about 1.6 waves at the kernel's 5)
        const int ahead = h->prefetch_Ri[k] ? 2 * 4 * num_sms() : 0;
        stb_launch(updmat_init_kernel, dim3(np, ceil_div(w, 64), ceil_div(hh, 8)), dim3(256), 0, s, Rk, coarse, h->M[0], w, hh,
                   wc, hc, up_sx, up_sy, (float)(1. / h->prm.pyr_scale), p0, h->tmapRi[k], ahead);
      }
      STB_CHECK_LAUNCH("updmat_init_kernel");
      if (dbg && h->dbg_M0 && h->dbg_pair >= p0 && h->dbg_pair < p1)
        STB_CUDA(cudaMemcpyAsync(h->dbg_M0, h->M[0] + (size_t)h->dbg_pair * 5 * nk, nk * 20, cudaMemcpyDeviceToDevice, s));
      PtrBatch<float> fo;
      for (int i = 0; i < kMaxPtrBatch; ++i) fo.p[i] = nullptr;
      for (int i = 0; i < np; ++i)
        fo.p[i] = (k == 0) ? d_flow[p0 + i] : h->flow[fl_cur] + (size_t)(p0 + i) * nk * 2;
      int mc = 0;
      const bool gauss = (h->prm.flags & kFlagGaussian) != 0;
      const bool fast15 = (m == kFiM) && !gauss;   // the winSize-15 kernels are box-window only
      const TileOrder ot = {ceil_div(w, kFiTW), ceil_div(hh, kFiTH), np};
      const dim3 grid = fast15 ? dim3((unsigned)(ot.tiles_x * ot.tiles_y * np)) : dim3(ceil_div(w, kItTW), ceil_div(hh, kItTH), np);
      const bool prof = h->profile && k == 0 && h->prm.num_iters > 1;
      for (int it = 0; it < h->prm.num_iters; ++it) {
        if (it < h->prm.num_iters - 1) {
          if (prof && it == 0) { int prc = prof_mark(h, s); if (prc) return prc; }
          if (fast15 && h->use_tma[k] && h->use_win[k])
            stb_launch(iter15_win_kernel, grid, dim3(kFiThreads), kWinSmemBytes, s, h->tmap[mc][k], h->M[mc ^ 1],
                       Rk, w, hh, p0, h->tmapR[k], h->prefetch_R[k], h->tmapRw[k], ot);
          else if (fast15 && h->use_tma[k])
            stb_launch(iter15_tma_kernel<true, false>, grid, dim3(kFiThreads), 0, s, h->tmap[mc][k], h->M[mc ^ 1],
                       Rk, fo, (int32_t*)nullptr, w, hh, p0, h->tmapR[k], h->prefetch_R[k], ot);
          else if (fast15)
            stb_launch(iter15_kernel<true, false>, grid, dim3(kFiThreads), 0, s, (const float*)h->M[mc], h->M[mc ^ 1],
                       Rk, fo, (int32_t*)nullptr, w, hh, p0, ot);
          else if (gauss)
            stb_launch(iter_kernel<true, true>, grid, dim3(kItThreads), it_smem, s, (const float*)h->M[mc], h->M[mc ^ 1],
                       Rk, fo, w, hh, m, p0, h->taps);
          else
            stb_launch(iter_kernel<true, false>, grid, dim3(kItThreads), it_smem, s, (const float*)h->M[mc], h->M[mc ^ 1],
                       Rk, fo, w, hh, m, p0, h->taps);
          mc ^= 1;
          if (prof && it == h->prm.num_iters - 2) {
            int prc = prof_mark(h, s);
            if (prc) return prc;
            h->prof_launches += h->prm.num_iters - 1;
            h->prof_pair_iters += (long long)(h->prm.num_iters - 1) * np;
          }
        } else {
          if (fast15 && h->use_tma[k] && k == 0 && d_hist != nullptr)
            stb_launch(iter15_tma_kernel<false, true>, grid, dim3(kFiThreads), 0, s, h->tmap[mc][k], (float*)nullptr,
                       Rk, fo, d_hist, w, hh, p0, h->tmapR[k], 0, ot);
          else if (fast15 && h->use_tma[k])
            stb_launch(iter15_tma_kernel<false, false>, grid, dim3(kFiThreads), 0, s, h->tmap[mc][k], (float*)nullptr,
                       Rk, fo, (int32_t*)nullptr, w, hh, p0, h->tmapR[k], 0, ot);
          else if (fast15 && k == 0 && d_hist != nullptr)
            stb_launch(iter15_kernel<false, true>, grid, dim3(kFiThreads), 0, s, (const float*)h->M[mc], (float*)nullptr,
                       Rk, fo, d_hist, w, hh, p0, ot);
          else if (fast15)
            stb_launch(iter15_kernel<false, false>, grid, dim3(kFiThreads), 0, s, (const float*)h->M[mc], (float*)nullptr,
                       Rk, fo, (int32_t*)nullptr, w, hh, p0, ot);
          else if (gauss)
            stb_launch(iter_kernel<false, true>, grid, dim3(kItThreads), it_smem, s, (const float*)h->M[mc], (float*)nullptr,
                       Rk, fo, w, hh, m, p0, h->taps);
          else
            stb_launch(iter_kernel<false, false>, grid, dim3(kItThreads), it_smem, s, (const float*)h->M[mc], (float*)nullptr,
                       Rk, fo, w, hh, m, p0, h->taps);
        }
        STB_CHECK_LAUNCH("iter_kernel");
      }
      if (dbg && h->dbg_flow && h->dbg_pair >= p0 && h->dbg_pair < p1)
        STB_CUDA(cudaMemcpyAsync(h->dbg_flow, fo.p[h->dbg_pair - p0], nk * 8, cudaMemcpyDeviceToDevice, s));
    }
    fl_cur ^= 1;
  }
  return STB_OK;
}

// Checks the caller's tables before anything is enqueued: frames[0..n] and (when given, or always with
// `need_flow`) d_flow[0..n-1] must not hold NULL.  An empty batch is accepted without looking at them.
static int check_run_args(stb_farneback* h, const uint8_t* const* frames, int n, float* const* d_flow, bool need_flow, const char* who) {
  if (!h || !frames || n < 0) { set_error("%s: invalid argument", who); return STB_ERR_INVALID; }
  if (n > h->max_pairs) { set_error("%s: n=%d exceeds max_pairs=%d", who, n, h->max_pairs); return STB_ERR_INVALID; }
  if (n == 0) return STB_OK;
  if (int rc = check_ptr_table(frames, n + 1, who, "frame")) return rc;
  return d_flow || need_flow ? check_ptr_table(d_flow, n, who, "flow") : STB_OK;
}

static int ensure_flow0(stb_farneback* h) {
  if (h->flow0) return STB_OK;
  cudaError_t e = cudaMalloc((void**)&h->flow0, (size_t)h->max_pairs * h->W * h->H * 2 * sizeof(float));
  if (e != cudaSuccess) {
    (void)cudaGetLastError();
    set_error("stb_farneback: cudaMalloc of the internal flow buffer failed: %s", cudaGetErrorString(e));
    return STB_ERR_ALLOC;
  }
  return STB_OK;
}

static int to_gray(stb_farneback* h, const uint8_t* const* d_rgb, int F, cudaStream_t s) {
  const unsigned long long npx = (unsigned long long)h->W * h->H;
  long long blocks = (long long)((npx / 16 + 255) / 256);
  const long long cap = (long long)num_sms() * 8;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  for (int base = 0; base < F; base += kMaxPtrBatch) {
    const int mcount = F - base < kMaxPtrBatch ? F - base : kMaxPtrBatch;
    stb_launch(gray_kernel, dim3((unsigned)blocks, (unsigned)mcount), dim3(256), 0, s, ptr_chunk(d_rgb, base, mcount),
               h->gray + (size_t)base * npx, npx);
    STB_CHECK_LAUNCH("gray_kernel");
  }
  return STB_OK;
}

// enqueue of one batch on `s` (shared by the direct path and the capture)
static int enqueue_batch(stb_farneback* h, const uint8_t* const* d_rgb, int n, float* const* fl, int32_t* d_hist, cudaStream_t s) {
  int rc = to_gray(h, d_rgb, n + 1, s);
  if (rc) return rc;
  if (d_hist) {
    cudaError_t e = cudaMemsetAsync(d_hist, 0, (size_t)n * STB_FLOWHIST_INTS * sizeof(int32_t), s);
    if (e != cudaSuccess) return cuda_fail(e, "cudaMemsetAsync(flow_hist)");
  }
  return run_levels(h, n, fl, s, d_hist);
}


// ---------------------------------------------------------------------------------------------
// CUDA-graph replay.  A batch is ~25 launches on two lanes; at small resolutions (640x480, 720p
// streams) the launches are a few microseconds each and the per-launch CPU + front-end cost shows.
// The first call of a given shape (number of pairs, which outputs) is stream-captured -- the very
// same enqueue code, fork / join of the second lane included -- and instantiated; later calls of
// that shape patch the kernel nodes that carry caller pointers (gray_kernel: the frame table; the
// level-0 last-iteration kernel: the flow table and the histogram pointer; the histogram memset)
// and replay the graph with one cudaGraphLaunch.  Everything else in the graph only touches
// handle-owned workspace.  Not used with the debug taps, the event profiler, chunked batches
// (> 64 pairs) or parameter sets that need the unfused histogram kernel.
// ---------------------------------------------------------------------------------------------
#ifndef STB_CPU_EMU
struct GrayArgs { PtrBatch<const uint8_t> frames; uint8_t* gray; unsigned long long npx; };
struct LastArgs {
  TmaMap3D map_in; float* Mout; const float* R; PtrBatch<float> flow_out; int32_t* flow_hist;
  int w, h, pair0; TmaMap3D map_R; int prefetch_R; TileOrder ord;
};
struct FbGraph {
  int n, kind;                       // kind: 0 = flow frames, 1 = flow frames + histogram, 2 = histogram only
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  std::vector<cudaGraphNode_t> gray_nodes;
  std::vector<cudaKernelNodeParams> gray_np;
  std::vector<GrayArgs> gray_args;
  cudaGraphNode_t last_node = nullptr;
  cudaKernelNodeParams last_np;
  LastArgs last_args;
  cudaGraphNode_t memset_node = nullptr;
  cudaMemsetParams memset_p;
  long long kernel_nodes = 0;
};

static void graph_free(FbGraph* g) {
  if (!g) return;
  if (g->exec) cudaGraphExecDestroy(g->exec);
  if (g->graph) cudaGraphDestroy(g->graph);
  delete g;
}

static bool graph_eligible(const stb_farneback* h, int n) {
  if (!h->use_graph || h->profile || h->dbg_level >= 0 || !h->s_cap) return false;
  if (!fused_hist_available(h) || !h->use_tma[0]) return false;
  return n + 1 <= kMaxPtrBatch;      // one gray launch (and so one chunk per level)
}

static int graph_build(stb_farneback* h, const uint8_t* const* d_rgb, int n, float* const* fl, int32_t* d_hist, int kind, FbGraph** out) {
  *out = nullptr;
  FbGraph* g = new (std::nothrow) FbGraph();
  if (!g) { set_error("out of host memory"); return STB_ERR_ALLOC; }
  g->n = n; g->kind = kind;
  const long long l0 = g_launches.load(std::memory_order_relaxed);
  cudaError_t e = cudaStreamBeginCapture(h->s_cap, cudaStreamCaptureModeThreadLocal);
  if (e != cudaSuccess) { graph_free(g); return cuda_fail(e, "cudaStreamBeginCapture"); }
  int rc = enqueue_batch(h, d_rgb, n, fl, d_hist, h->s_cap);
  e = cudaStreamEndCapture(h->s_cap, &g->graph);
  g_launches.store(l0, std::memory_order_relaxed);           // nothing ran: the capture only recorded
  if (rc || e != cudaSuccess || !g->graph) {
    graph_free(g);
    (void)cudaGetLastError();
    return rc ? rc : cuda_fail(e, "cudaStreamEndCapture");
  }
  size_t nn = 0;
  e = cudaGraphGetNodes(g->graph, nullptr, &nn);
  std::vector<cudaGraphNode_t> nodes(nn);
  if (e == cudaSuccess && nn) e = cudaGraphGetNodes(g->graph, nodes.data(), &nn);
  const void* f_last = kind == 0 ? (const void*)iter15_tma_kernel<false, false> : (const void*)iter15_tma_kernel<false, true>;
  for (size_t i = 0; i < nn && e == cudaSuccess; ++i) {
    cudaGraphNodeType ty;
    e = cudaGraphNodeGetType(nodes[i], &ty);
    if (e != cudaSuccess) break;
    if (ty == cudaGraphNodeTypeKernel) {
      ++g->kernel_nodes;
      cudaKernelNodeParams kp;
      e = cudaGraphKernelNodeGetParams(nodes[i], &kp);
      if (e != cudaSuccess) break;
      if (kp.func == (void*)gray_kernel) {
        // (the graph's parameter copies carry no alignment guarantee: memcpy, never a typed load)
        GrayArgs a;
        std::memcpy(&a.frames, kp.kernelParams[0], sizeof(a.frames));
        std::memcpy(&a.gray, kp.kernelParams[1], sizeof(a.gray));
        std::memcpy(&a.npx, kp.kernelParams[2], sizeof(a.npx));
        g->gray_nodes.push_back(nodes[i]); g->gray_np.push_back(kp); g->gray_args.push_back(a);
      } else if (kp.func == f_last) {
        int pw = 0, ph = 0;
        std::memcpy(&pw, kp.kernelParams[5], sizeof(int));
        std::memcpy(&ph, kp.kernelParams[6], sizeof(int));
        if (pw != h->w[0] || ph != h->h[0]) continue;            // the last iteration of a coarser level
        LastArgs& a = g->last_args;
        std::memcpy(&a.map_in, kp.kernelParams[0], sizeof(a.map_in));
        std::memcpy(&a.Mout, kp.kernelParams[1], sizeof(a.Mout));
        std::memcpy(&a.R, kp.kernelParams[2], sizeof(a.R));
        std::memcpy(&a.flow_out, kp.kernelParams[3], sizeof(a.flow_out));
        std::memcpy(&a.flow_hist, kp.kernelParams[4], sizeof(a.flow_hist));
        a.w = pw; a.h = ph;
        std::memcpy(&a.pair0, kp.kernelParams[7], sizeof(a.pair0));
        std::memcpy(&a.map_R, kp.kernelParams[8], sizeof(a.map_R));
        std::memcpy(&a.prefetch_R, kp.kernelParams[9], sizeof(a.prefetch_R));
        std::memcpy(&a.ord, kp.kernelParams[10], sizeof(a.ord));
        g->last_node = nodes[i]; g->last_np = kp;
      }
    } else if (ty == cudaGraphNodeTypeMemset) {
      g->memset_node = nodes[i];
      e = cudaGraphMemsetNodeGetParams(nodes[i], &g->memset_p);
    }
  }
  // exactly the nodes we know how to re-point, or no graph at all
  const bool ok = e == cudaSuccess && g->gray_nodes.size() == 1 && g->last_node && ((d_hist != nullptr) == (g->memset_node != nullptr));
  if (ok) e = cudaGraphInstantiate(&g->exec, g->graph, 0);
  if (!ok || e != cudaSuccess) {
    graph_free(g);
    (void)cudaGetLastError();
    return STB_OK;      // *out stays NULL: the caller falls back to direct launches
  }
  *out = g;
  return STB_OK;
}

// returns STB_OK with *used = true when the batch was enqueued through a graph
static int graph_run(stb_farneback* h, const uint8_t* const* d_rgb, int n, float* const* fl, int32_t* d_hist, int kind, cudaStream_t s,
                     bool* used) {
  *used = false;
  if (!graph_eligible(h, n)) return STB_OK;
  FbGraph* g = nullptr;
  for (FbGraph* c : h->graphs)
    if (c->n == n && c->kind == kind) { g = c; break; }
  if (!g) {
    int rc = graph_build(h, d_rgb, n, fl, d_hist, kind, &g);
    if (rc) return rc;
    if (!g) { h->use_graph = 0; return STB_OK; }       // capture not possible here: stay on direct launches
    if (h->graphs.size() >= 16) { graph_free(h->graphs.front()); h->graphs.erase(h->graphs.begin()); }
    h->graphs.push_back(g);
  }
  {
    GrayArgs& a = g->gray_args[0];
    for (int i = 0; i < kMaxPtrBatch; ++i) a.frames.p[i] = i <= n ? d_rgb[i] : nullptr;
    void* args[3] = {&a.frames, &a.gray, &a.npx};
    cudaKernelNodeParams kp = g->gray_np[0];
    kp.kernelParams = args; kp.extra = nullptr;
    STB_CUDA(cudaGraphExecKernelNodeSetParams(g->exec, g->gray_nodes[0], &kp));
  }
  {
    LastArgs& a = g->last_args;
    for (int i = 0; i < kMaxPtrBatch; ++i) a.flow_out.p[i] = i < n ? fl[i] : nullptr;
    a.flow_hist = d_hist;
    void* args[11] = {&a.map_in, &a.Mout, &a.R, &a.flow_out, &a.flow_hist, &a.w, &a.h, &a.pair0, &a.map_R, &a.prefetch_R, &a.ord};
    cudaKernelNodeParams kp = g->last_np;
    kp.kernelParams = args; kp.extra = nullptr;
    STB_CUDA(cudaGraphExecKernelNodeSetParams(g->exec, g->last_node, &kp));
  }
  if (g->memset_node) {
    cudaMemsetParams mp = g->memset_p;
    mp.dst = d_hist;
    STB_CUDA(cudaGraphExecMemsetNodeSetParams(g->exec, g->memset_node, &mp));
  }
  STB_CUDA(cudaGraphLaunch(g->exec, s));
  g_launches.fetch_add(g->kernel_nodes, std::memory_order_relaxed);
  *used = true;
  return STB_OK;
}
#else
struct FbGraph {};
static void graph_free(FbGraph*) {}
static int graph_run(stb_farneback*, const uint8_t* const*, int, float* const*, int32_t*, int, cudaStream_t, bool* used) { *used = false; return STB_OK; }
#endif

}  // namespace stb

extern "C" {

int stb_farneback_run(stb_farneback* h, const uint8_t* const* d_rgb, int n, float* const* d_flow, stb_stream_t stream) {
  int rc = check_run_args(h, d_rgb, n, d_flow, true, "stb_farneback_run");
  if (rc || n == 0) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  bool via_graph = false;
  rc = graph_run(h, d_rgb, n, d_flow, nullptr, 0, s, &via_graph);
  if (rc || via_graph) return rc;
  return enqueue_batch(h, d_rgb, n, d_flow, nullptr, s);
}

int stb_farneback_run_gray(stb_farneback* h, const uint8_t* const* d_gray, int n, float* const* d_flow, stb_stream_t stream) {
  int rc = check_run_args(h, d_gray, n, d_flow, true, "stb_farneback_run_gray");
  if (rc || n == 0) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  const size_t npx = (size_t)h->W * h->H;
  for (int i = 0; i <= n; ++i)
    STB_CUDA(cudaMemcpyAsync(h->gray + (size_t)i * npx, d_gray[i], npx, cudaMemcpyDeviceToDevice, s));
  return run_levels(h, n, d_flow, s);
}

int stb_farneback_run_hist(stb_farneback* h, const uint8_t* const* d_rgb, int n, float* const* d_flow,
                           int32_t* d_flow_hist, stb_stream_t stream) {
  int rc = check_run_args(h, d_rgb, n, d_flow, false, "stb_farneback_run_hist");
  if (rc || n == 0) return rc;
  if (!d_flow_hist) { set_error("stb_farneback_run_hist: d_flow_hist is NULL"); return STB_ERR_INVALID; }
  cudaStream_t s = (cudaStream_t)stream;
  const bool fused = fused_hist_available(h);   // the winSize-15 box kernel bins the flow it produces
  float* tmp[kMaxPtrBatch * 4];
  float** fl = (n <= kMaxPtrBatch * 4) ? tmp : nullptr;
  float** heap = nullptr;
  if (!fl) { heap = new (std::nothrow) float*[n]; if (!heap) { set_error("out of host memory"); return STB_ERR_ALLOC; } fl = heap; }
  if (d_flow) {
    for (int i = 0; i < n; ++i) fl[i] = d_flow[i];
  } else if (fused) {
    for (int i = 0; i < n; ++i) fl[i] = nullptr;       // histogram only: the flow frames never touch HBM
  } else {
    rc = ensure_flow0(h);
    if (rc) { delete[] heap; return rc; }
    for (int i = 0; i < n; ++i) fl[i] = h->flow0 + (size_t)i * h->W * h->H * 2;
  }
  if (fused) {
    bool via_graph = false;
    rc = graph_run(h, d_rgb, n, fl, d_flow_hist, d_flow ? 1 : 2, s, &via_graph);
    if (rc || via_graph) { delete[] heap; return rc; }
  }
  rc = enqueue_batch(h, d_rgb, n, fl, fused ? d_flow_hist : nullptr, s);
  if (!rc && !fused) rc = flow_hist_device(fl, n, (unsigned long long)h->W * h->H, d_flow_hist, s, true);
  delete[] heap;
  return rc;
}

}  // extern "C"
