// Histogram, shot-score, FlowHistogram and FrameDifference kernels (sm_100a) + their C ABI.
//
// All four are HBM-bound byte/word streaming kernels: each input byte is read exactly once
// with 16-byte coalesced loads; counting happens in shared memory that is privatised per
// lane (bank == lane), so shared-memory reductions never conflict regardless of image content
// (constant frames are the worst case for a shared table); the RGB histogram counts byte PAIRS
// into a joint table (half the reductions); one global merge per block.
//
// Reference call sites replaced: see include/stb.h.
#include <cstdlib>

#include "stb_rt.h"
#include "flow_bins.cuh"

namespace stb {

// -------------------------------------------------------------------------------------------
// RGB histogram, 16 bins/channel.  The packed RGB24 frame is a flat byte stream: byte at
// offset a belongs to channel a % 3 and falls in bin (byte >> 4).
// Block = 384 threads (a multiple of 3 and of 32), so with a grid-stride of gridDim.x*384
// sixteen-byte vectors every thread sees a constant channel phase: byte b of each of its
// vectors is channel (phase + b) % 3 -- the table bases are fixed registers.
//
// JOINT counting: a shared-memory reduction costs ~2 cycles of the SM's atomic unit per warp
// instruction whatever it adds and however many lanes are active (tools/probe/atoms_probe.cu), so one
// RED per input byte caps the kernel at ~17 B/clk/SM = 0.75 of HBM -- where round 1 / early round 2
// sat.  Two vectors of one thread have the same channel phase, so byte k of vector A and byte k of
// vector B are the same channel: the pair is counted with ONE reduction into a 256-entry joint table
// indexed by (bin_A | bin_B << 4), and the block's epilogue folds the joint table into the two
// marginals.  Half the reductions for any content, and fewer instructions per byte (the joint indices
// of four byte pairs come from one shift + one LOP3 on the two words).
// Tables are private per LANE (bank == lane, never a conflict); one table per block -- updates of
// different warps are different instructions and serialise in the atomic unit anyway.
//   joint  [3 channels][256][32 lanes] u32 = 96 KB, single [3][16][32] u32 = 6 KB (odd vector, ragged ends)
// -------------------------------------------------------------------------------------------
constexpr int kHistThreads = 384;
constexpr int kHistBlocksPerSM = 2;
#ifndef STB_HIST_VECS
#define STB_HIST_VECS 4
#endif
constexpr int kHistVecs = STB_HIST_VECS;                                // 16-byte vectors in flight per thread (even)
constexpr int kHistJointBytes = 3 * 256 * 32 * 4;                       // 98304
constexpr int kHistSingleBytes = STB_HIST_INTS * 32 * 4;                // 6144
constexpr int kHistSmemBytes = kHistJointBytes + kHistSingleBytes;      // 104448: two blocks per SM

#ifdef STB_CPU_EMU
typedef unsigned char* hist_addr_t;   // emulator: a plain pointer into the table
__device__ __forceinline__ hist_addr_t hist_origin(unsigned char* dyn) { return dyn; }
__device__ __forceinline__ void hist_inc(hist_addr_t a) { atomicAdd(reinterpret_cast<unsigned*>(a), 1u); }
__device__ __forceinline__ unsigned hist_byte(unsigned w, int k) { return (w >> (8 * k)) & 255u; }
#else
typedef unsigned hist_addr_t;         // 32-bit address in the shared window
__device__ __forceinline__ hist_addr_t hist_origin(unsigned char* dyn) { return (unsigned)__cvta_generic_to_shared(dyn); }
__device__ __forceinline__ void hist_inc(hist_addr_t a) {
  asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(a) : "memory");   // fire-and-forget shared-memory reduction
}
__device__ __forceinline__ unsigned hist_byte(unsigned w, int k) { return __byte_perm(w, 0u, 0x4440u + (unsigned)k); }
#endif

// four byte pairs (byte k of wa with byte k of wb); their channels use bases (b0, b1, b2, b0): the caller
// rotates them per word.  m holds the four joint indices, one per byte: bin_A in the low nibble, bin_B in the high.
__device__ __forceinline__ void hist_count_pair_word(unsigned wa, unsigned wb, hist_addr_t b0, hist_addr_t b1, hist_addr_t b2) {
#ifdef STB_CPU_EMU
  const unsigned m = ((wa >> 4) & 0x0f0f0f0fu) | (wb & 0xf0f0f0f0u);
#else
  unsigned m;   // bitwise select in one LOP3: mask ? (wa >> 4) : wb
  asm("lop3.b32 %0, %1, %2, %3, 0xCA;" : "=r"(m) : "r"(0x0f0f0f0fu), "r"(wa >> 4), "r"(wb));
#endif
  hist_inc(b0 + (hist_byte(m, 0) << 7));
  hist_inc(b1 + (hist_byte(m, 1) << 7));
  hist_inc(b2 + (hist_byte(m, 2) << 7));
  hist_inc(b0 + (hist_byte(m, 3) << 7));
}

__device__ __forceinline__ void hist_count_pair_vec(const uint4& a, const uint4& b, hist_addr_t c0, hist_addr_t c1, hist_addr_t c2) {
  // word j starts at byte 4j: channel of its first byte is (phase + 4j) % 3 = (phase + j) % 3
  hist_count_pair_word(a.x, b.x, c0, c1, c2);
  hist_count_pair_word(a.y, b.y, c1, c2, c0);
  hist_count_pair_word(a.z, b.z, c2, c0, c1);
  hist_count_pair_word(a.w, b.w, c0, c1, c2);
}

__device__ __forceinline__ void hist_count_word(unsigned wd, hist_addr_t b0, hist_addr_t b1, hist_addr_t b2) {
  // single bytes: bin << 7 == ((byte >> 4) & 15) << 7, taken straight out of the word with one shift + mask
  hist_inc(b0 + ((wd << 3) & 0x780u));
  hist_inc(b1 + ((wd >> 5) & 0x780u));
  hist_inc(b2 + ((wd >> 13) & 0x780u));
  hist_inc(b0 + ((wd >> 21) & 0x780u));
}

__device__ __forceinline__ void hist_count_vec(const uint4& q, hist_addr_t c0, hist_addr_t c1, hist_addr_t c2) {
  hist_count_word(q.x, c0, c1, c2);
  hist_count_word(q.y, c1, c2, c0);
  hist_count_word(q.z, c2, c0, c1);
  hist_count_word(q.w, c0, c1, c2);
}

template <class Addr>
__global__ void __launch_bounds__(kHistThreads, kHistBlocksPerSM)
hist_rgb16_kernel(Addr addr, unsigned long long nbytes, int32_t* __restrict__ out, unsigned base_blocks, unsigned rem) {
  // 1-D grid over (frame, part): the first `rem` frames get base_blocks + 1 blocks, the others
  // base_blocks, so a batch fills the resident wave exactly whatever the frame count
  unsigned frame, part, nparts;
  flat_grid_decode(blockIdx.x, base_blocks, rem, frame, part, nparts);
  STB_DYN_SMEM(unsigned char, dyn);
  const hist_addr_t origin = hist_origin(dyn);
  const unsigned tid = threadIdx.x, lane = tid & 31u;
  {
    uint4* z = reinterpret_cast<uint4*>(dyn);
    for (unsigned i = tid; i < kHistSmemBytes / 16; i += kHistThreads) z[i] = make_uint4(0u, 0u, 0u, 0u);
  }
  __syncthreads();

  const uint8_t* f = addr(frame);
  unsigned long long head = (16u - (unsigned)(reinterpret_cast<uintptr_t>(f) & 15u)) & 15u;
  if (head > nbytes) head = nbytes;
  const uint4* v = reinterpret_cast<const uint4*>(f + head);
  const unsigned long long nvec = (nbytes - head) >> 4;

  const unsigned gt = part * kHistThreads + tid;
  const unsigned long long T = (unsigned long long)nparts * kHistThreads;
  const unsigned ph = (unsigned)((head + gt) % 3u);
  const hist_addr_t jbase = origin + lane * 4u, sbase = origin + kHistJointBytes + lane * 4u;
  const hist_addr_t j0 = jbase + ((ph + 0u) % 3u) * 32768u, j1 = jbase + ((ph + 1u) % 3u) * 32768u,
                    j2 = jbase + ((ph + 2u) % 3u) * 32768u;
  const hist_addr_t s0 = sbase + ((ph + 0u) % 3u) * 2048u, s1 = sbase + ((ph + 1u) % 3u) * 2048u,
                    s2 = sbase + ((ph + 2u) % 3u) * 2048u;

  // software pipeline: the next kHistVecs vectors are in flight while the current ones (kHistVecs / 2 pairs) are counted
  unsigned long long i = gt;
  if (i + (kHistVecs - 1) * T < nvec) {
    uint4 q[kHistVecs];
#pragma unroll
    for (int k = 0; k < kHistVecs; ++k) q[k] = __ldg(v + i + k * T);
    i += kHistVecs * T;
#pragma unroll 2
    for (; i + (kHistVecs - 1) * T < nvec; i += kHistVecs * T) {
      uint4 nx[kHistVecs];
#pragma unroll
      for (int k = 0; k < kHistVecs; ++k) nx[k] = __ldg(v + i + k * T);
#pragma unroll
      for (int k = 0; k < kHistVecs; k += 2) hist_count_pair_vec(q[k], q[k + 1], j0, j1, j2);
#pragma unroll
      for (int k = 0; k < kHistVecs; ++k) q[k] = nx[k];
    }
#pragma unroll
    for (int k = 0; k < kHistVecs; k += 2) hist_count_pair_vec(q[k], q[k + 1], j0, j1, j2);
  }
  for (; i + T < nvec; i += 2 * T) {
    const uint4 qa = __ldg(v + i), qb = __ldg(v + i + T);
    hist_count_pair_vec(qa, qb, j0, j1, j2);
  }
  if (i < nvec) {
    const uint4 q = __ldg(v + i);
    hist_count_vec(q, s0, s1, s2);
  }
  // ragged ends (unaligned base pointer / byte count not a multiple of 16): at most 30 bytes
  if (part == 0) {
    const unsigned long long tail0 = head + (nvec << 4);
    const unsigned long long ntail = nbytes - tail0;
    if (tid < head + ntail) {
      const unsigned long long a = tid < head ? tid : tail0 + (tid - head);
      hist_inc(sbase + (unsigned)(a % 3u) * 2048u + (((unsigned)(f[a] >> 4)) << 7));
    }
  }
  __syncthreads();

  // block reduce: 8 threads per output bin (ch, b), each over 4 lanes: the single table's row plus the
  // joint table's rows (b | j << 4) -- first byte of a pair in bin b -- and (j | b << 4) -- second byte
  const unsigned bin = tid >> 3, rpart = tid & 7u;
  const unsigned ch = bin >> 4, b = bin & 15u;
  const unsigned* jt = reinterpret_cast<const unsigned*>(dyn) + ch * (256 * 32) + rpart * 4;
  const unsigned* st = reinterpret_cast<const unsigned*>(dyn + kHistJointBytes) + bin * 32 + rpart * 4;
  unsigned s;
  {
    const uint4 q = *reinterpret_cast<const uint4*>(st);
    s = q.x + q.y + q.z + q.w;
  }
#pragma unroll 4
  for (unsigned j = 0; j < 16; ++j) {
    const uint4 qa = *reinterpret_cast<const uint4*>(jt + (b | (j << 4)) * 32);
    const uint4 qb = *reinterpret_cast<const uint4*>(jt + (j | (b << 4)) * 32);
    s += qa.x + qa.y + qa.z + qa.w + qb.x + qb.y + qb.z + qb.w;
  }
  s += __shfl_xor_sync(0xffffffffu, s, 1);
  s += __shfl_xor_sync(0xffffffffu, s, 2);
  s += __shfl_xor_sync(0xffffffffu, s, 4);
  if (rpart == 0 && s != 0) atomicAdd(out + (size_t)frame * STB_HIST_INTS + bin, (int)s);
}

// -------------------------------------------------------------------------------------------
// shot scores: S[i] = sum_j max_b |h[i-1][j][b] - h[i][j][b]|
// one warp per frame: lane l handles bins l and l+32 (48 bins), segmented max over 16 lanes.
// -------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
shot_scores_kernel(const int32_t* __restrict__ hist, int n, const int32_t* __restrict__ prev_hist,
                   int32_t* __restrict__ S) {
  const int lane = threadIdx.x & 31;
  const int i = (int)(blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5));
  if (i >= n) return;  // whole warp exits together
  const int32_t* cur = hist + (size_t)i * STB_HIST_INTS;
  const int32_t* prv = i > 0 ? cur - STB_HIST_INTS : prev_hist;
  int d0 = 0, d1 = 0;
  if (prv != nullptr) {
    d0 = abs(cur[lane] - prv[lane]);                       // channels 0 (lanes 0-15) and 1 (16-31)
    if (lane < 16) d1 = abs(cur[32 + lane] - prv[32 + lane]);  // channel 2
  }
#pragma unroll
  for (int m = 1; m < 16; m <<= 1) {
    d0 = max(d0, __shfl_xor_sync(0xffffffffu, d0, m));
    d1 = max(d1, __shfl_xor_sync(0xffffffffu, d1, m));
  }
  const int other = __shfl_sync(0xffffffffu, d0, 16);
  if (lane == 0) S[i] = d0 + other + d1;
}

// -------------------------------------------------------------------------------------------
// FlowHistogram: 64-bin magnitude [0,64) + 64-bin angle [0,360) of an HxWx2 f32 flow field.
// Arithmetic reproduces OpenCV's cartToPolar (polynomial fastAtan, angleInDegrees) and
// calcHist's double-precision bin index bit-for-bit (SURVEY Appendix B).
// Per-lane private u32 counters, ONE table per block: [128 bins][32 lanes] (bank == lane, so a warp's
// update never conflicts whatever the content; updates of different warps are different instructions
// and serialise in the atomic unit anyway).  One update = LEA (base + bin * 128) + predicated RED.
// History: one packed-16-bit table per warp (64 KB, 3 blocks / SM, 0.32 of HBM) -> one per 4 warps
// (0.35) -> this form, with the ~11-instruction packed-counter update gone.
// -------------------------------------------------------------------------------------------
constexpr int kFlowHistThreads = 256;
// rows: 64 magnitude bins, one trash row, 64 angle bins, one trash row.  A dropped value (bin outside 0..63)
// is clamped onto the trash row, so the update needs no predicate: ptxas turns a predicated shared RED into
// a BSSY / BRA / BSYNC region (+4 instructions per update).
constexpr int kFlowHistRows = 2 * 65;
constexpr int kFlowHistSmemWords = kFlowHistRows * 32;        // 16.25 KB
constexpr int kFlowHistBlocksPerSM = 6;

#ifdef STB_CPU_EMU
typedef unsigned* flow_tab_t;
__device__ __forceinline__ flow_tab_t flow_tab(unsigned* sh, unsigned lane) { return sh + lane; }
__device__ __forceinline__ void flow_inc(flow_tab_t my, int bin, int plane) {
  atomicAdd(my + (plane * 65 + min((unsigned)bin, 64u)) * 32, 1u);
}
#else
typedef unsigned flow_tab_t;                                  // 32-bit address in the shared window
__device__ __forceinline__ flow_tab_t flow_tab(unsigned* sh, unsigned lane) {
  return (unsigned)__cvta_generic_to_shared(sh) + lane * 4u;
}
__device__ __forceinline__ void flow_inc(flow_tab_t my, int bin, int plane) {
  asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(my + (unsigned)plane * (65u * 128u) + (min((unsigned)bin, 64u) << 7)) : "memory");
}
#endif

__device__ __forceinline__ void flow_count(flow_tab_t my, float x, float y) {
  int bm, ba;
  flow_bins_fast(x, y, bm, ba);
  flow_inc(my, bm, 0);
  flow_inc(my, ba, 1);
}

template <class Addr>
__global__ void __launch_bounds__(kFlowHistThreads, kFlowHistBlocksPerSM)
flow_hist_kernel(Addr addr, unsigned long long npx, int32_t* __restrict__ out, unsigned base_blocks, unsigned rem) {
  // 1-D grid over (frame, part), as in hist_rgb16_kernel
  unsigned frame, part, nparts;
  flat_grid_decode(blockIdx.x, base_blocks, rem, frame, part, nparts);
  STB_DYN_SMEM(unsigned, sh);
  const unsigned tid = threadIdx.x, lane = tid & 31u;
  {
    uint4* z = reinterpret_cast<uint4*>(sh);
    for (unsigned i = tid; i < kFlowHistSmemWords / 4; i += kFlowHistThreads) z[i] = make_uint4(0u, 0u, 0u, 0u);
  }
  __syncthreads();
  const float* f = addr(frame);
  const flow_tab_t my = flow_tab(sh, lane);
  const unsigned long long gt = (unsigned long long)part * kFlowHistThreads + tid;
  const unsigned long long T = (unsigned long long)nparts * kFlowHistThreads;
  if ((reinterpret_cast<uintptr_t>(f) & 15u) == 0) {
    const float4* v = reinterpret_cast<const float4*>(f);
    const unsigned long long nvec = npx >> 1;
    unsigned long long i = gt;
    for (; i + T < nvec; i += 2 * T) {
      const float4 q0 = __ldg(v + i);
      const float4 q1 = __ldg(v + i + T);
      flow_count(my, q0.x, q0.y);
      flow_count(my, q0.z, q0.w);
      flow_count(my, q1.x, q1.y);
      flow_count(my, q1.z, q1.w);
    }
    for (; i < nvec; i += T) {
      const float4 q = __ldg(v + i);
      flow_count(my, q.x, q.y);
      flow_count(my, q.z, q.w);
    }
    if ((npx & 1ull) && gt == 0) flow_count(my, f[2 * (npx - 1)], f[2 * (npx - 1) + 1]);
  } else {
    for (unsigned long long i = gt; i < npx; i += T) flow_count(my, __ldg(f + 2 * i), __ldg(f + 2 * i + 1));
  }
  __syncthreads();
  // reduce: 2 threads per bin, each sums 16 lanes
  const unsigned bin = tid >> 1, rpart = tid & 1u;
  const unsigned* row = sh + (bin + (bin >> 6)) * 32 + rpart * 16;   // skip the magnitude trash row
  unsigned s = 0;
#pragma unroll
  for (int l = 0; l < 16; l += 4) {
    const uint4 q = *reinterpret_cast<const uint4*>(row + l);
    s += q.x + q.y + q.z + q.w;
  }
  s += __shfl_xor_sync(0xffffffffu, s, 1);
  if (rpart == 0 && s != 0) atomicAdd(out + (size_t)frame * STB_FLOWHIST_INTS + bin, (int)s);
}

// -------------------------------------------------------------------------------------------
// FrameDifference: out = (u8)(cur - prev)
// -------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
frame_diff_kernel(const uint8_t* __restrict__ prev, const uint8_t* __restrict__ cur, uint8_t* __restrict__ out,
                  unsigned long long n, int vec_ok) {
  const unsigned long long gt = (unsigned long long)blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned long long T = (unsigned long long)gridDim.x * blockDim.x;
  unsigned long long done = 0;
  if (vec_ok) {
    const unsigned long long nvec = n >> 4;
    const uint4* p = reinterpret_cast<const uint4*>(prev);
    const uint4* c = reinterpret_cast<const uint4*>(cur);
    uint4* o = reinterpret_cast<uint4*>(out);
    for (unsigned long long i = gt; i < nvec; i += T) {
      const uint4 a = __ldg(c + i), b = __ldg(p + i);
      o[i] = make_uint4(__vsub4(a.x, b.x), __vsub4(a.y, b.y), __vsub4(a.z, b.z), __vsub4(a.w, b.w));
    }
    done = nvec << 4;
  }
  for (unsigned long long i = done + gt; i < n; i += T) out[i] = (uint8_t)(cur[i] - prev[i]);
}

// -------------------------------------------------------------------------------------------
// host side
// -------------------------------------------------------------------------------------------
template <class Addr>
static int launch_hist(Addr addr, int n, unsigned long long nbytes, int32_t* d_out, cudaStream_t s) {
  if (int rc = set_max_dyn_smem_once<hist_rgb16_kernel<Addr>>(kHistSmemBytes)) return rc;
  // One resident wave (kHistBlocksPerSM blocks/SM) split over the frames as evenly as possible
  // (some frames get one block more); spilling a handful of blocks into a second wave costs ~25 %,
  // leaving slots empty costs proportionally (n = 32 on 444 slots: 416 blocks 66.8 %, 444 blocks ~71 %).
  // Never more blocks per frame than there are 4-vector iterations of work; with more frames than
  // slots, one block per frame.
  const unsigned long long nvec = nbytes >> 4;
  const long long max_useful = (long long)((nvec + (unsigned long long)kHistThreads * 4 - 1) / ((unsigned long long)kHistThreads * 4));
  long long total;
  unsigned base_blocks, rem;
  one_wave_split(n, kHistBlocksPerSM, max_useful, &total, &base_blocks, &rem);
  stb_launch(hist_rgb16_kernel<Addr>, dim3((unsigned)total), dim3(kHistThreads), kHistSmemBytes, s, addr, nbytes, d_out,
             base_blocks, rem);
  STB_CHECK_LAUNCH("hist_rgb16_kernel");
  return STB_OK;
}

template <class Addr>
static int launch_flow_hist(Addr addr, int n, unsigned long long npx, int32_t* d_out, cudaStream_t s) {
  if (int rc = set_max_dyn_smem_once<flow_hist_kernel<Addr>>((int)(kFlowHistSmemWords * sizeof(unsigned)))) return rc;
  const long long max_useful = (long long)((npx / 2 + (unsigned long long)kFlowHistThreads * 2 - 1) / ((unsigned long long)kFlowHistThreads * 2));
  long long total;
  unsigned base_blocks, rem;
  one_wave_split(n, kFlowHistBlocksPerSM, max_useful, &total, &base_blocks, &rem);
  stb_launch(flow_hist_kernel<Addr>, dim3((unsigned)total), dim3(kFlowHistThreads), kFlowHistSmemWords * sizeof(unsigned), s,
             addr, npx, d_out, base_blocks, rem);
  STB_CHECK_LAUNCH("flow_hist_kernel");
  return STB_OK;
}

int flow_hist_device(const float* const* d_flow, int n, unsigned long long npx, int32_t* d_out, cudaStream_t s,
                     bool zero_out) {
  if (zero_out) STB_CUDA(cudaMemsetAsync(d_out, 0, (size_t)n * STB_FLOWHIST_INTS * sizeof(int32_t), s));
  for (int base = 0; base < n; base += kMaxPtrBatch) {
    const int m = n - base < kMaxPtrBatch ? n - base : kMaxPtrBatch;
    int rc = launch_flow_hist(PtrAddr<const float>{ptr_chunk(d_flow, base, m)}, m, npx, d_out + (size_t)base * STB_FLOWHIST_INTS, s);
    if (rc) return rc;
  }
  return STB_OK;
}

}  // namespace stb

using namespace stb;

extern "C" {

int stb_hist_rgb16(const uint8_t* const* d_frames, int n, int width, int height, int32_t* d_out, stb_stream_t stream) {
  if (n == 0) return STB_OK;
  if (!d_out || n < 0 || width <= 0 || height <= 0) {
    set_error("stb_hist_rgb16: invalid argument (n=%d, %dx%d)", n, width, height);
    return STB_ERR_INVALID;
  }
  if (int rc = check_ptr_table(d_frames, n, "stb_hist_rgb16", "frame")) return rc;
  const unsigned long long nbytes = 3ull * (unsigned long long)width * (unsigned long long)height;
  size_t stride = 0;
  if (uniform_stride(d_frames, n, nbytes, &stride))
    return stb_hist_rgb16_strided(d_frames[0], stride, n, width, height, d_out, stream);
  cudaStream_t s = (cudaStream_t)stream;
  STB_CUDA(cudaMemsetAsync(d_out, 0, (size_t)n * STB_HIST_INTS * sizeof(int32_t), s));
  for (int base = 0; base < n; base += kMaxPtrBatch) {
    const int m = n - base < kMaxPtrBatch ? n - base : kMaxPtrBatch;
    int rc = launch_hist(PtrAddr<const uint8_t>{ptr_chunk(d_frames, base, m)}, m, nbytes, d_out + (size_t)base * STB_HIST_INTS, s);
    if (rc) return rc;
  }
  return STB_OK;
}

int stb_hist_rgb16_strided(const uint8_t* d_base, size_t stride_bytes, int n, int width, int height, int32_t* d_out,
                           stb_stream_t stream) {
  if (n == 0) return STB_OK;
  const unsigned long long nbytes = 3ull * (unsigned long long)(width > 0 ? width : 0) * (unsigned long long)(height > 0 ? height : 0);
  if (!d_base || !d_out || n < 0 || width <= 0 || height <= 0 || stride_bytes < nbytes) {
    set_error("stb_hist_rgb16_strided: invalid argument (n=%d, %dx%d, stride=%zu)", n, width, height, stride_bytes);
    return STB_ERR_INVALID;
  }
  cudaStream_t s = (cudaStream_t)stream;
  STB_CUDA(cudaMemsetAsync(d_out, 0, (size_t)n * STB_HIST_INTS * sizeof(int32_t), s));
  for (int base = 0; base < n; base += kMaxStridedFrames) {
    const int m = n - base < kMaxStridedFrames ? n - base : kMaxStridedFrames;
    StrideAddr<const uint8_t> a{d_base + (size_t)base * stride_bytes, (unsigned long long)stride_bytes};
    int rc = launch_hist(a, m, nbytes, d_out + (size_t)base * STB_HIST_INTS, s);
    if (rc) return rc;
  }
  return STB_OK;
}

int stb_shot_scores(const int32_t* d_hist, int n, const int32_t* d_prev_hist, int32_t* d_S, stb_stream_t stream) {
  if (n == 0) return STB_OK;
  if (!d_hist || !d_S || n < 0) {
    set_error("stb_shot_scores: invalid argument (n=%d)", n);
    return STB_ERR_INVALID;
  }
  const int warps_per_block = 8;
  stb_launch(shot_scores_kernel, dim3((unsigned)ceil_div(n, warps_per_block)), dim3(warps_per_block * 32), 0,
             (cudaStream_t)stream, d_hist, n, d_prev_hist, d_S);
  STB_CHECK_LAUNCH("shot_scores_kernel");
  return STB_OK;
}

int stb_flow_hist(const float* const* d_flow, int n, int width, int height, int32_t* d_out, stb_stream_t stream) {
  if (n == 0) return STB_OK;
  if (!d_out || n < 0 || width <= 0 || height <= 0) {
    set_error("stb_flow_hist: invalid argument (n=%d, %dx%d)", n, width, height);
    return STB_ERR_INVALID;
  }
  if (int rc = check_ptr_table(d_flow, n, "stb_flow_hist", "flow")) return rc;
  return flow_hist_device(d_flow, n, (unsigned long long)width * (unsigned long long)height, d_out, (cudaStream_t)stream, true);
}

int stb_flow_hist_strided(const float* d_base, size_t stride_bytes, int n, int width, int height, int32_t* d_out,
                          stb_stream_t stream) {
  if (n == 0) return STB_OK;
  const unsigned long long npx = (unsigned long long)(width > 0 ? width : 0) * (unsigned long long)(height > 0 ? height : 0);
  if (!d_base || !d_out || n < 0 || width <= 0 || height <= 0 || stride_bytes < npx * 8 || (stride_bytes & 3)) {
    set_error("stb_flow_hist_strided: invalid argument (n=%d, %dx%d, stride=%zu)", n, width, height, stride_bytes);
    return STB_ERR_INVALID;
  }
  cudaStream_t s = (cudaStream_t)stream;
  STB_CUDA(cudaMemsetAsync(d_out, 0, (size_t)n * STB_FLOWHIST_INTS * sizeof(int32_t), s));
  for (int base = 0; base < n; base += kMaxStridedFrames) {
    const int m = n - base < kMaxStridedFrames ? n - base : kMaxStridedFrames;
    StrideAddr<const float> a{reinterpret_cast<const float*>(reinterpret_cast<const uint8_t*>(d_base) + (size_t)base * stride_bytes),
                              (unsigned long long)stride_bytes};
    int rc = launch_flow_hist(a, m, npx, d_out + (size_t)base * STB_FLOWHIST_INTS, s);
    if (rc) return rc;
  }
  return STB_OK;
}

int stb_frame_diff(const uint8_t* d_prev, const uint8_t* d_cur, uint8_t* d_out, size_t bytes, stb_stream_t stream) {
  if (bytes == 0) return STB_OK;
  if (!d_prev || !d_cur || !d_out) {
    set_error("stb_frame_diff: NULL pointer");
    return STB_ERR_INVALID;
  }
  const int vec_ok = (((reinterpret_cast<uintptr_t>(d_prev) | reinterpret_cast<uintptr_t>(d_cur) |
                        reinterpret_cast<uintptr_t>(d_out)) & 15u) == 0) ? 1 : 0;
  unsigned long long work = vec_ok ? (bytes >> 4) + 15 : bytes;
  long long blocks = (long long)((work + 255) / 256);
  const long long cap = (long long)num_sms() * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  stb_launch(frame_diff_kernel, dim3((unsigned)blocks), dim3(256), 0, (cudaStream_t)stream, d_prev, d_cur, d_out,
             (unsigned long long)bytes, vec_ok);
  STB_CHECK_LAUNCH("frame_diff_kernel");
  return STB_OK;
}

}  // extern "C"
