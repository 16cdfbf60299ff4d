// Common runtime glue for the scannertools_b200 CUDA sources.
// Product builds: nvcc, sm_100a.  (STB_CPU_EMU is defined only by tests/cuda_emu, which
// compiles the same kernel source against a CPU emulation of the CUDA execution model.)
#pragma once
#ifdef STB_CPU_EMU_BUILD
#include "cuda_emu.h"
#else
#include <cuda_runtime.h>
#endif
#include <cstdarg>
#include <cstddef>
#include <cstdint>
#include <cstdio>
#include <utility>

#include "stb.h"

#ifndef STB_CPU_EMU
#include <atomic>
namespace stb { extern std::atomic<long long> g_launches; }
template <class... KArgs, class... Args>
static inline void stb_launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args) {
  kernel<<<grid, block, smem, s>>>(args...);
  stb::g_launches.fetch_add(1, std::memory_order_relaxed);
}
#define STB_DYN_SMEM(T, name)                                      \
  extern __shared__ __align__(16) unsigned char stb_dyn_smem_[];   \
  T* name = reinterpret_cast<T*>(stb_dyn_smem_)
#else
#define STB_DYN_SMEM(T, name) T* name = reinterpret_cast<T*>(cuda_emu::dyn_smem())
#endif

namespace stb {

constexpr int kMaxPtrBatch = 64;
// device pointers passed by value in kernel parameter space (no table upload, no sync)
template <class T>
struct PtrBatch {
  T* p[kMaxPtrBatch];
};

// How a batched kernel finds frame i: entry i of a pointer table, or base + i * stride bytes.
template <class T>
struct PtrAddr {
  PtrBatch<T> t;
  __device__ __forceinline__ T* operator()(unsigned i) const { return t.p[i]; }
};
template <class T>
struct StrideAddr {
  T* base;
  unsigned long long stride;  // bytes
  __device__ __forceinline__ T* operator()(unsigned i) const {
    return reinterpret_cast<T*>(reinterpret_cast<const uint8_t*>(base) + (unsigned long long)i * stride);
  }
};

// frames per launch of the strided entry points
constexpr int kMaxStridedFrames = 32768;

void set_error(const char* fmt, ...);
int cuda_fail(cudaError_t e, const char* what);

#define STB_CUDA(expr)                                        \
  do {                                                        \
    cudaError_t stb_e_ = (expr);                              \
    if (stb_e_ != cudaSuccess) return stb::cuda_fail(stb_e_, #expr); \
  } while (0)

#define STB_CHECK_LAUNCH(what)                                \
  do {                                                        \
    cudaError_t stb_e_ = cudaGetLastError();                  \
    if (stb_e_ != cudaSuccess) return stb::cuda_fail(stb_e_, what); \
  } while (0)

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// The per-frame streaming kernels (histograms) run on a flattened 1-D grid of exactly one
// resident wave: `total` blocks are split over n frames as evenly as possible -- the first
// rem = total % n frames get base_blocks + 1 blocks, the others base_blocks = total / n -- so a
// batch fills every block slot whatever the frame count.  This maps a block index to
// (frame, part of that frame, number of parts of that frame).
__host__ __device__ inline void flat_grid_decode(unsigned b, unsigned base_blocks, unsigned rem, unsigned& frame,
                                                 unsigned& part, unsigned& nparts) {
  const unsigned big = rem * (base_blocks + 1u);
  if (b < big) {
    frame = b / (base_blocks + 1u);
    part = b - frame * (base_blocks + 1u);
    nparts = base_blocks + 1u;
  } else {
    const unsigned bb = b - big;
    frame = rem + bb / base_blocks;
    part = bb - (bb / base_blocks) * base_blocks;
    nparts = base_blocks;
  }
}

int num_sms();
int current_device();

// Sizes the grid that flat_grid_decode walks: one resident wave of blocks_per_sm blocks per SM over the n frames of
// a launch, never more than max_useful blocks per frame (when max_useful >= 1) and never less than one.
inline void one_wave_split(int n, int blocks_per_sm, long long max_useful, long long* total, unsigned* base_blocks,
                           unsigned* rem) {
  long long t = (long long)num_sms() * blocks_per_sm;
  if (max_useful >= 1 && t > max_useful * n) t = max_useful * n;
  if (t < n) t = n;
  *total = t;
  *base_blocks = (unsigned)(t / n);
  *rem = (unsigned)(t % n);
}

// cudaFuncSetAttribute(MaxDynamicSharedMemorySize) on the first launch of Kernel on each device: the attribute
// belongs to the (function, device) pair.
template <auto Kernel>
int set_max_dyn_smem_once(int bytes) {
  static bool done[64] = {};
  const int dev = current_device();
  if (!done[dev]) {
    STB_CUDA(cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    done[dev] = true;
  }
  return STB_OK;
}

// Checks a caller's table of n device pointers before anything is enqueued: a NULL table or entry is
// STB_ERR_INVALID, reported as "<who>: <what> <i> is NULL".
template <class T>
int check_ptr_table(T* const* tab, int n, const char* who, const char* what) {
  if (!tab) {
    set_error("%s: %s table is NULL", who, what);
    return STB_ERR_INVALID;
  }
  for (int i = 0; i < n; ++i)
    if (!tab[i]) {
      set_error("%s: %s %d is NULL", who, what, i);
      return STB_ERR_INVALID;
    }
  return STB_OK;
}

// entries [base, base + m) of a caller's table as one kernel-parameter table, the rest NULL
template <class T>
PtrBatch<T> ptr_chunk(T* const* tab, int base, int m) {
  PtrBatch<T> b;
  for (int i = 0; i < kMaxPtrBatch; ++i) b.p[i] = i < m ? tab[base + i] : nullptr;
  return b;
}

// A batch of more than one pointer table whose frames lie in one buffer at a constant stride of at least
// min_stride bytes (a decoder batch, a block buffer) can be read by a strided launch with no table at all.
inline bool uniform_stride(const uint8_t* const* tab, int n, unsigned long long min_stride, size_t* stride) {
  if (n <= kMaxPtrBatch) return false;
  const ptrdiff_t d = tab[1] - tab[0];
  if (d <= 0 || (unsigned long long)d < min_stride) return false;
  for (int i = 2; i < n; ++i)
    if (tab[i] - tab[i - 1] != d) return false;
  *stride = (size_t)d;
  return true;
}

int flow_hist_device(const float* const* d_flow, int n, unsigned long long npx, int32_t* d_out, cudaStream_t s,
                     bool zero_out);

}  // namespace stb
