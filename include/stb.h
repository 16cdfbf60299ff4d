/* scannertools_b200 -- C ABI of the B200-native per-frame analysis hot path.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  The reference library
 * (libscannertools_imgproc.so / libimgproc_op.so) exports no C symbols: its Scanner kernel
 * classes call OpenCV directly.  The replacement kernel classes (scannertools_b200/csrc/scanner_ops/)
 * keep the reference's REGISTER_OP / REGISTER_KERNEL names and call the functions below
 * instead of cv:: / cv::cuda::.  Every entry point cites the reference call it replaces
 * (paths relative to /root/reference/scannertools/).
 *
 * Conventions
 *   - plain pointers and sizes only; no C++/torch types.
 *   - `d_` pointers are device memory on the CURRENT CUDA device; pointer tables
 *     (`const T* const*`) are HOST arrays of device pointers.
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream).
 *   - work is enqueued asynchronously on `stream`; nothing synchronises unless stated.
 *   - outputs are caller-allocated (Scanner allocators: new_block_buffer / new_frames).
 *   - return 0 on success, negative stb_status or positive cudaError_t otherwise;
 *     stb_last_error() returns a thread-local message.  No exceptions cross the boundary,
 *     no CPU fallback exists: without a usable CUDA device every compute call fails.
 *   - frames are packed row-major HWC with no row pitch (blur_kernel_cpu.cpp:70).
 */
#ifndef SCANNERTOOLS_B200_STB_H_
#define SCANNERTOOLS_B200_STB_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define STB_API
#else
#define STB_API __attribute__((visibility("default")))
#endif

typedef void* stb_stream_t;

enum stb_status {
  STB_OK = 0,
  STB_ERR_INVALID = -1,     /* bad argument (null pointer, non-positive size, n > capacity) */
  STB_ERR_NO_DEVICE = -2,   /* no CUDA device / driver */
  STB_ERR_ALLOC = -3,       /* workspace allocation failed */
  STB_ERR_UNSUPPORTED = -4  /* parameter combination not implemented (see stb_farneback_params) */
};

#define STB_HIST_BINS 16       /* histogram_kernel_cpu.cpp:8  */
#define STB_HIST_INTS 48       /* int32[3][16] = 192 B per frame (histogram_kernel_cpu.cpp:20) */
#define STB_FLOWHIST_BINS 64   /* old/cpp_ops/flow_histogram_kernel_cpu.cpp:9 */
#define STB_FLOWHIST_INTS 128  /* int32[2][64] = 512 B per frame (flow_histogram_kernel_cpu.cpp:21) */

STB_API int stb_version(void);
STB_API const char* stb_last_error(void);
/* number of usable CUDA devices (0 if none); never fails */
STB_API int stb_device_count(void);

/* ---- Histogram ---------------------------------------------------------------------------
 * Replaces, per frame, cvc::split + 3 x cvc::histEven(plane, 16, 0, 256)
 * (scannertools_cpp/imgproc/histogram_kernel_gpu.cpp:49-57) == 3 x cv::calcHist + convertTo
 * (histogram_kernel_cpu.cpp:33-41).  d_out[i*48 + j*16 + b] = #{pixels of frame i whose
 * channel-j byte >> 4 == b}.  Bit-exact. */
STB_API int stb_hist_rgb16(const uint8_t* const* d_frames, int n, int width, int height,
                           int32_t* d_out /* n*48 */, stb_stream_t stream);
/* same, frames at d_base + i*stride_bytes (e.g. one Scanner block buffer / decoder batch) */
STB_API int stb_hist_rgb16_strided(const uint8_t* d_base, size_t stride_bytes, int n, int width,
                                   int height, int32_t* d_out, stb_stream_t stream);

/* ---- frame-difference scoring behind ShotBoundaries ----------------------------------------
 * Replaces the Chebyshev part of shot_boundaries (scannertools/shot_detection.py:14-18):
 * d_S[i] = sum_{j<3} max_b |h[i-1][j][b] - h[i][j][b]|  (= 3*diffs[i], an exact integer).
 * d_S[0] uses d_prev_hist (the histogram of the frame before this range, for frame-range
 * shards) or is 0 when d_prev_hist is NULL (stream start, diffs[0] = 0, shot_detection.py:18).
 * The +-500-frame windowed outlier test (shot_detection.py:22-26) stays on the host in
 * float64 (scannertools_b200/shot_detection.py) so it is bit-identical to numpy. */
STB_API int stb_shot_scores(const int32_t* d_hist /* n*48 */, int n, const int32_t* d_prev_hist /* 48 or NULL */,
                            int32_t* d_S /* n */, stb_stream_t stream);

/* ---- FlowHistogram -------------------------------------------------------------------------
 * Replaces split + cv::cartToPolar(x, y, mag, deg, true) + 2 x cv::calcHist(64 bins)
 * (scannertools/old/cpp_ops/flow_histogram_kernel_cpu.cpp:27-54).  d_out[i*128 + 0..63] =
 * magnitude histogram over [0,64), [64..127] = angle (degrees) histogram over [0,360);
 * values outside the range are dropped, as calcHist does.  Uses OpenCV's polynomial fastAtan
 * and double-precision bin index, so counts match the reference exactly on identical flow. */
STB_API int stb_flow_hist(const float* const* d_flow, int n, int width, int height,
                          int32_t* d_out /* n*128 */, stb_stream_t stream);
STB_API int stb_flow_hist_strided(const float* d_base, size_t stride_bytes, int n, int width, int height,
                                  int32_t* d_out, stb_stream_t stream);

/* ---- FrameDifference -----------------------------------------------------------------------
 * Intended semantics of the (dead, uncompilable) frame_difference_kernel_cpu.cpp:51-61:
 * out[k] = (uint8)(cur[k] - prev[k]) for every byte. */
STB_API int stb_frame_diff(const uint8_t* d_prev, const uint8_t* d_cur, uint8_t* d_out, size_t bytes,
                           stb_stream_t stream);

/* ---- OpticalFlow (dense Farneback) ---------------------------------------------------------
 * Replaces cv::cvtColor(BGR2GRAY) x2 + cv::FarnebackOpticalFlow::create(3, 0.5, false, 15, 3,
 * 5, 1.2, 0)->calc(gray0, gray1, flow) (scannertools_cpp/imgproc/optical_flow_kernel_cpu.cpp:
 * 15-16,36-41) and the cv::cuda equivalent (optical_flow_kernel_gpu.cpp:24,66-89).
 * Direction follows the CPU kernel: flow i maps frame i -> frame i+1 (SURVEY Appendix C). */
typedef struct stb_farneback_params {
  int num_levels;     /* 3   */
  double pyr_scale;   /* 0.5  (0.5 <= pyr_scale < 1)               */
  int fast_pyramids;  /* 0    (0 or 1; no effect, exactly as in OpenCV's CPU implementation, which is the parity target) */
  int win_size;       /* 15   (odd, <= 31)                         */
  int num_iters;      /* 3                                         */
  int poly_n;         /* 5    (3..7; 5 has the tuned kernel)       */
  double poly_sigma;  /* 1.2                                       */
  int flags;          /* 0 = box window (the reference); 256 = cv::OPTFLOW_FARNEBACK_GAUSSIAN
                         (Gaussian window, generic kernel); OPTFLOW_USE_INITIAL_FLOW is not supported */
} stb_farneback_params;

typedef struct stb_farneback stb_farneback;

/* the reference's hard-coded parameters (optical_flow_kernel_cpu.cpp:16) */
STB_API void stb_farneback_default_params(stb_farneback_params* p);
/* device bytes a handle for (width,height,max_pairs) allocates; 0 on invalid arguments */
STB_API size_t stb_farneback_workspace_bytes(int width, int height, int max_pairs,
                                             const stb_farneback_params* params /* NULL = defaults */);
/* Creates a handle on the current device (the reference constructs its cv::cuda objects in the
 * kernel constructor, optical_flow_kernel_gpu.cpp:14-26).  Scratch is handle-owned; one handle
 * may be used by one thread at a time. */
STB_API int stb_farneback_create(int width, int height, int max_pairs, const stb_farneback_params* params,
                                 stb_farneback** out);
STB_API int stb_farneback_destroy(stb_farneback* h);
/* n frame pairs from n+1 RGB24 frames (the batch layout of optical_flow_kernel_gpu.cpp:52-57):
 * d_flow[i] (H*W*2 f32, interleaved dx,dy) = flow(frame i -> frame i+1).  n <= max_pairs. */
STB_API int stb_farneback_run(stb_farneback* h, const uint8_t* const* d_rgb /* n+1 */, int n,
                              float* const* d_flow /* n */, stb_stream_t stream);
/* same on already-gray frames (H*W u8): the cv::FarnebackOpticalFlow::calc contract itself */
STB_API int stb_farneback_run_gray(stb_farneback* h, const uint8_t* const* d_gray /* n+1 */, int n,
                                   float* const* d_flow /* n */, stb_stream_t stream);
/* Fused OpticalFlow -> FlowHistogram (SURVEY §8f rank 2): additionally writes n*128 int32
 * flow histograms; d_flow may be NULL to skip materialising the flow frames. */
STB_API int stb_farneback_run_hist(stb_farneback* h, const uint8_t* const* d_rgb, int n,
                                   float* const* d_flow /* n or NULL */, int32_t* d_flow_hist /* n*128 */,
                                   stb_stream_t stream);
/* pyramid geometry actually used: returns the number of scales (<= 4), fills w[k], h[k] */
STB_API int stb_farneback_levels(const stb_farneback* h, int* widths /* 8 */, int* heights /* 8 */);
/* debugging / stage-by-stage parity: copies level-k intermediates of the LAST run for pair
 * `pair` into caller DEVICE buffers (any may be NULL): I0,I1: h*w f32; R0,R1,M: 5 planes of
 * h*w f32 (planar, unlike OpenCV's interleaved layout).  Synchronises the stream. */
STB_API int stb_farneback_debug_set(stb_farneback* h, int level, int pair, float* d_I0, float* d_I1,
                                    float* d_R0, float* d_R1, float* d_M0, float* d_flow_level);

/* ---- Resize (SURVEY 8f rank 1, the op in front of OpticalFlow in old/histograms.py:64-68) ---
 * Replaces cv::resize / cvc::resize(img, out, Size(w, h), 0, 0, INTER_LINEAR) on 8-bit frames
 * (scannertools_cpp/imgproc/resize_kernel.cpp:69-79); bit-exact with OpenCV's fixed-point
 * bilinear (including its INTER_AREA fast path for exact 2x down-scaling).  channels: 1, 3, 4.
 * stb_resize_target reproduces the op's target-size rules (width/height/min/preserve_aspect,
 * resize_kernel.cpp:43-61). */
STB_API int stb_resize_target(int frame_w, int frame_h, int width, int height, int min_flag, int preserve_aspect,
                              int* out_w, int* out_h);
STB_API int stb_resize_bilinear_u8(const uint8_t* const* d_src, int n, int src_w, int src_h, int channels,
                                   uint8_t* const* d_dst, int dst_w, int dst_h, stb_stream_t stream);
/* The same with ResizeArgs.interpolation (resize_kernel.cpp:9-20,31-35): stb_resize_interp_code maps
 * "INTER_LINEAR" (also "" / NULL, the reference's default), "INTER_NEAREST", "INTER_AREA", "INTER_CUBIC",
 * "INTER_LANCZOS4" to codes 0..4 and anything else to -1 (stb_resize_u8 then returns
 * STB_ERR_UNSUPPORTED).  Bit-exact with cv::resize on 8-bit frames for all five (INTER_CUBIC: with
 * OpenCV's own code path; OpenCV builds that hand 8-bit cubic to IPP differ from it by one grey level on
 * ~5 % of pixels).  INTER_CUBIC / INTER_LANCZOS4 build their tap tables on the host and upload them in
 * stream order (cudaMallocAsync / cudaFreeAsync): the call stays asynchronous but is not graph-capturable. */
STB_API int stb_resize_interp_code(const char* name);
STB_API int stb_resize_u8(const uint8_t* const* d_src, int n, int src_w, int src_h, int channels,
                          uint8_t* const* d_dst, int dst_w, int dst_h, int interp, stb_stream_t stream);
/* The same on float32 frames with 1 to 4 channels (an OpticalFlow field is H x W x 2), with the interpolation codes
 * of stb_resize_interp_code and OpenCV's float arithmetic (cv2.ipp.setUseIPP(False)).  Bit-exact with cv::resize
 * for INTER_NEAREST, INTER_LINEAR (exact 2x down included) and INTER_AREA up-scaling and integer factors, signed zeros
 * and infinities included, and for every mode at dst == src size (a copy, as in OpenCV); within
 * 8 * 2^-23 * max|src| of OpenCV's double-precision result for general INTER_AREA down-scaling, INTER_CUBIC and
 * INTER_LANCZOS4.  Every frame pointer must be 4-byte aligned.  STB_ERR_UNSUPPORTED: channels outside 1..4, unknown
 * interp; STB_ERR_INVALID: bad sizes, NULL or misaligned table entries (nothing is enqueued then); n == 0 does
 * nothing.  INTER_CUBIC / INTER_LANCZOS4 upload their tap tables in stream order, as stb_resize_u8 does: asynchronous,
 * not graph-capturable. */
STB_API int stb_resize_f32(const float* const* d_src, int n, int src_w, int src_h, int channels,
                           float* const* d_dst, int dst_w, int dst_h, int interp, stb_stream_t stream);

/* ---- ConvertColor (SURVEY 8f rank 3) -------------------------------------------------------------
 * Replaces cv::cvtColor(frame, out, code) on packed 8-bit frames (scannertools_cpp/imgproc/
 * convert_color_kernel.cpp:270-276; COLOR_RGB2HSV also for old/cpp_ops/imgproc.cpp:41, feeding the HSV
 * histogram of old/histograms.py:32-36); bit-exact with OpenCV's integer paths on every input.
 * stb_color_code maps the reference's conversion names to codes, both spellings where OpenCV has an
 * alias (-1 = not implemented; every code is below 99):
 *   0 RGB2HSV, 1 BGR2HSV, 2 RGB2GRAY, 3 BGR2GRAY, 4 BGR2RGB = RGB2BGR            (3 -> 3 or 1)
 *   5 BGR2BGRA = RGB2RGBA, 6 BGR2RGBA = RGB2BGRA                                  (3 -> 4, alpha 255)
 *   7 BGRA2BGR = RGBA2RGB, 8 RGBA2BGR = BGRA2RGB                                  (4 -> 3)
 *   9 BGRA2RGBA = RGBA2BGRA                                                       (4 -> 4, alpha kept)
 *  10 GRAY2BGR = GRAY2RGB, 11 GRAY2BGRA = GRAY2RGBA                               (1 -> 3 / 4, alpha 255)
 *  12 BGRA2GRAY, 13 RGBA2GRAY                                                     (4 -> 1)
 *  14 BGR2YCrCb, 15 RGB2YCrCb, 16 YCrCb2BGR, 17 YCrCb2RGB                         (3 -> 3)
 *  18 BGR2YUV, 19 RGB2YUV, 20 YUV2BGR, 21 YUV2RGB  (packed 4:4:4)                 (3 -> 3)
 *  22 BGR2HSV_FULL, 23 RGB2HSV_FULL  (H over [0,256))                             (3 -> 3)
 * (names without their COLOR_ prefix).  stb_color_in_channels / stb_color_out_channels give a code's
 * channel counts (0 for an unknown code); stb_convert_color_u8 reads in-channel frames and writes
 * out-channel frames, n of them, width x height pixels each. */
STB_API int stb_color_code(const char* name);
STB_API int stb_color_in_channels(int code);
STB_API int stb_color_out_channels(int code);
STB_API int stb_convert_color_u8(const uint8_t* const* d_src, int n, int width, int height, int code,
                                 uint8_t* const* d_dst, stb_stream_t stream);

/* ---- Blur ----------------------------------------------------------------------------------------
 * Replaces the box blur of the reference's BlurKernel (scannertools_cpp/imgproc/blur_kernel_cpu.cpp), which runs
 * on the CPU only; its BlurArgs.sigma is never read, so this is a box filter, not a Gaussian.  With
 * k = kernel_size, L = ceil(k/2) - 1 and R = k/2 (an even k puts the extra row and column on the bottom and right),
 * a pixel with L <= x < width - R and L <= y < height - R gets, for each channel c independently,
 *   out[y][x][c] = (sum over dy, dx in [-L, R] of in[y+dy][x+dx][c]) / (k*k)
 * as an unsigned integer sum divided with truncation.  Every other pixel is a copy of the input pixel (the
 * reference leaves those bytes unwritten), so k = 1 is the identity and a frame smaller than the window is copied
 * unchanged.  channels: 1, 3 or 4.  n frames of width x height, d_src[i] -> d_dst[i], any alignment.
 * STB_ERR_INVALID: n < 0, width or height <= 0, other channel counts, kernel_size < 1, or d_dst[i] overlapping
 * d_src[i] (a blur in place would read half-written rows); aliasing between different frames is the caller's
 * responsibility.  STB_ERR_UNSUPPORTED: kernel_size > 255.  n == 0 does nothing. */
STB_API int stb_blur_u8(const uint8_t* const* d_src, int n, int width, int height, int channels, int kernel_size,
                        uint8_t* const* d_dst, stb_stream_t stream);

/* ---- fused ConvertToHSV -> Histogram (SURVEY 8f rank 3) -------------------------------------------
 * The HSV variant of the shot-detection histogram: scannertools/old/histograms.py:32-36 chains
 * ConvertToHSVCPP (old/cpp_ops/imgproc.cpp:14-48, cv::cvtColor COLOR_RGB2HSV) into the Histogram
 * op (histogram_kernel_cpu.cpp:16-46).  One pass over the RGB bytes, the HSV frame is never
 * materialised; d_out[n][3][16] = histogram of (H, S, V), identical to
 * stb_hist_rgb16(stb_convert_color_u8(frame, code)).  H < 180, so H bins 12..15 are zero.
 * code = stb_color_code("COLOR_RGB2HSV") or ("COLOR_BGR2HSV"); anything else is STB_ERR_UNSUPPORTED. */
STB_API int stb_hist_hsv16(const uint8_t* const* d_frames, int n, int width, int height, int code,
                           int32_t* d_out, stb_stream_t stream);
STB_API int stb_hist_hsv16_strided(const uint8_t* d_base, size_t stride_bytes, int n, int width, int height,
                                   int code, int32_t* d_out, stb_stream_t stream);

/* ---- measurement hooks (bench.py) -----------------------------------------------------------
 * stb_launch_count: kernels this library has launched in this process (all entry points).
 * stb_farneback_profile: when enabled, every level-0 pair brackets its fused update-iteration
 * kernels (the dominant kernel, DESIGN.md) with CUDA events on the launching stream;
 * _profile_read synchronises those events and returns their summed duration, the number of
 * kernel launches they cover and the number of (pair x iteration) units those launches
 * processed (one launch handles a whole batch of pairs). */
STB_API long long stb_launch_count(void);
STB_API int stb_farneback_profile(stb_farneback* h, int enable);
STB_API int stb_farneback_profile_read(stb_farneback* h, double* ms_total, long long* launches,
                                       long long* pair_iterations);

/* ---- host-buffer entry points (end-to-end path) ---------------------------------------------
 * The reference's kernels receive device frames from the Scanner engine; when this library is
 * driven directly with HOST frames (bench e2e, python wrappers on numpy arrays) these calls own
 * the pinned staging ring, the async H2D/D2H copies and their overlap with compute on two
 * streams.  They synchronise before returning; outputs are host memory. */
typedef struct stb_pipe stb_pipe;
STB_API int stb_pipe_create(int width, int height, int max_batch, int want_flow, stb_pipe** out);
STB_API int stb_pipe_destroy(stb_pipe* p);
/* n frames -> n*48 int32 histograms (+ n int32 scores S, S[0] = 0, when h_S != NULL) */
STB_API int stb_pipe_hist(stb_pipe* p, const uint8_t* h_frames, int n, int32_t* h_hist, int32_t* h_S);
/* n+1 frames -> n flow frames (h_flow may be NULL) and/or n*128 flow histograms (may be NULL) */
STB_API int stb_pipe_flow(stb_pipe* p, const uint8_t* h_frames, int n, float* h_flow, int32_t* h_flow_hist);
/* Asynchronous form: enqueues the whole call and returns a ticket (0 or 1; -1 when n == 0); the host
 * buffers must stay valid and untouched until stb_pipe_wait(ticket).  At most two calls may be in
 * flight; the second call's uploads overlap the first call's kernels, so a stream of calls keeps
 * the GPU busy without the per-call start-up bubble. */
STB_API int stb_pipe_flow_async(stb_pipe* p, const uint8_t* h_frames, int n, float* h_flow, int32_t* h_flow_hist,
                                int* ticket);
STB_API int stb_pipe_wait(stb_pipe* p, int ticket);
/* Page-locked host staging memory for the calls above (they are only asynchronous on pinned buffers).
 * write_combined != 0 allocates write-combined memory (cudaHostAllocWriteCombined): fast for the device
 * to read over PCIe, slow for the host to read back -- for upload-only frame buffers. */
STB_API int stb_host_alloc(size_t bytes, int write_combined, void** out);
STB_API int stb_host_free(void* p);

#ifdef __cplusplus
}
#endif
#endif /* SCANNERTOOLS_B200_STB_H_ */
