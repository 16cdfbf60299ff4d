"""Python host-side mirror of the reference ops on this path, driving the C ABI (include/stb.h).

Reference ops mirrored (paths relative to /root/reference/scannertools/):
  Histogram       scannertools_cpp/imgproc/histogram_kernel_{cpu,gpu}.cpp   -> histogram()
  OpticalFlow     scannertools_cpp/imgproc/optical_flow_kernel_{cpu,gpu}.cpp -> OpticalFlow
  FlowHistogram   scannertools/old/cpp_ops/flow_histogram_kernel_cpu.cpp     -> flow_histogram()
  FrameDifference scannertools_cpp/imgproc/frame_difference_kernel_cpu.cpp   -> frame_difference()
  ShotBoundaries  scannertools/shot_detection.py                              -> shot_detection.py

Like Scanner's GPU kernels, these take frames that are already device resident (torch CUDA
tensors are used purely as device-memory handles) and return device tensors.  Host (numpy /
pinned torch) frames go through `Pipe`, which owns the async copy/compute overlap.
torch is plumbing only: every byte of arithmetic happens in the CUDA kernels behind the C ABI.
There is no CPU fallback: on a machine without the built library or a GPU these calls raise.
"""
import ctypes as C

import numpy as np

from . import _lib

HIST_BINS = 16       # histogram_kernel_cpu.cpp:8
FLOW_HIST_BINS = 64  # flow_histogram_kernel_cpu.cpp:9
# names of resize_kernel.cpp:9-20's table without a kernel here
RESIZE_TABLE_UNIMPLEMENTED = ('INTER_MAX', 'WARP_FILL_OUTLIERS', 'WARP_INVERSE_MAP')   # flag values, not interpolation modes


def _torch():
    import torch
    return torch


def _stream_ptr(stream=None):
    torch = _torch()
    s = stream if stream is not None else torch.cuda.current_stream()
    return C.c_void_p(s.cuda_stream)


def _require_cuda(t, dtype, what):
    torch = _torch()
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise TypeError('%s must be a CUDA tensor (device-resident frames, as Scanner GPU kernels receive); '
                        'use scannertools_b200.ops.Pipe for host buffers' % what)
    if t.dtype != dtype:
        raise TypeError('%s must have dtype %s, got %s' % (what, dtype, t.dtype))
    if not t.is_contiguous():
        raise ValueError('%s must be contiguous (packed HWC, no row pitch)' % what)


def _frames_list(frames, dtype, what, last):
    """Accepts one [n,H,W,last] tensor or a sequence of [H,W,last] tensors (separate buffers,
    as a Scanner batch of Frame* is).  Returns (list_of_tensors, H, W)."""
    torch = _torch()
    if isinstance(frames, torch.Tensor):
        if frames.dim() == 3:
            frames = frames.unsqueeze(0)
        _require_cuda(frames, dtype, what)
        lst = [frames[i] for i in range(frames.shape[0])]
    else:
        lst = list(frames)
        for f in lst:
            _require_cuda(f, dtype, what)
    if lst:
        H, W, c = lst[0].shape
        if c != last:
            raise ValueError('%s: expected %d channels, got %d' % (what, last, c))
        for f in lst:
            if tuple(f.shape) != (H, W, last):
                raise ValueError('%s: all frames of a batch must share one FrameInfo' % what)
        return lst, H, W
    return lst, 0, 0


def histogram(frames, stream=None, hsv=None):
    """Histogram op: n RGB24 frames -> int32 [n, 3, 16] (192 B per frame, channel-major, the
    layout `types.histograms` parses).  Bit-exact with the reference (bin = byte >> 4).

    hsv='COLOR_RGB2HSV' (or 'COLOR_BGR2HSV') gives the HSV variant of the shot-detection
    histogram (scannertools/old/histograms.py:32-36: ConvertToHSVCPP -> Histogram) in one fused
    pass, identical to histogram(convert_color(frames, hsv))."""
    torch = _torch()
    lib = _lib.load()
    code = None
    if hsv is not None:
        code = lib.stb_color_code(hsv.encode())
        if code < 0 or hsv not in ('COLOR_RGB2HSV', 'COLOR_BGR2HSV'):
            raise ValueError('histogram: hsv must be COLOR_RGB2HSV or COLOR_BGR2HSV, got %r' % (hsv,))
    if isinstance(frames, torch.Tensor) and frames.dim() == 4 and frames.shape[0] > 0:
        # one contiguous batch (a decoder batch / block buffer): strided entry point, one launch
        _require_cuda(frames, torch.uint8, 'frames')
        n, H, W, c = frames.shape
        if c != 3:
            raise ValueError('frames: expected 3 channels, got %d' % c)
        out = torch.empty((n, 3, HIST_BINS), dtype=torch.int32, device=frames.device)
        with torch.cuda.device(frames.device):
            if code is None:
                rc = lib.stb_hist_rgb16_strided(C.c_void_p(frames.data_ptr()), H * W * 3, n, W, H,
                                                C.c_void_p(out.data_ptr()), _stream_ptr(stream))
            else:
                rc = lib.stb_hist_hsv16_strided(C.c_void_p(frames.data_ptr()), H * W * 3, n, W, H, code,
                                                C.c_void_p(out.data_ptr()), _stream_ptr(stream))
            _lib.check(rc, lib)
        return out
    lst, H, W = _frames_list(frames, torch.uint8, 'frames', 3)
    n = len(lst)
    dev = lst[0].device if n else torch.device('cuda')
    out = torch.empty((n, 3, HIST_BINS), dtype=torch.int32, device=dev)
    if n == 0:
        return out
    with torch.cuda.device(dev):
        tab = _lib.ptr_table([f.data_ptr() for f in lst])
        if code is None:
            rc = lib.stb_hist_rgb16(tab, n, W, H, C.c_void_p(out.data_ptr()), _stream_ptr(stream))
        else:
            rc = lib.stb_hist_hsv16(tab, n, W, H, code, C.c_void_p(out.data_ptr()), _stream_ptr(stream))
        _lib.check(rc, lib)
    return out


def shot_scores(hist, prev_hist=None, stream=None):
    """S[i] = 3 * diffs[i] of shot_detection.py:14-18 as exact int32.  `prev_hist` is the
    histogram of the frame preceding this range (frame-range shards); without it S[0] = 0."""
    torch = _torch()
    lib = _lib.load()
    _require_cuda(hist, torch.int32, 'hist')
    n = hist.shape[0]
    if hist.numel() != n * 3 * HIST_BINS:
        raise ValueError('hist must be [n, 3, 16]')
    S = torch.empty((n,), dtype=torch.int32, device=hist.device)
    if n == 0:
        return S
    pp = None
    if prev_hist is not None:
        _require_cuda(prev_hist, torch.int32, 'prev_hist')
        pp = C.c_void_p(prev_hist.data_ptr())
    with torch.cuda.device(hist.device):
        _lib.check(lib.stb_shot_scores(C.c_void_p(hist.data_ptr()), n, pp, C.c_void_p(S.data_ptr()), _stream_ptr(stream)), lib)
    return S


def flow_histogram(flows, stream=None):
    """FlowHistogram op: n flow frames (HxWx2 f32) -> int32 [n, 2, 64] (512 B per frame:
    magnitude bins then angle bins, the layout `flow_hist_reader` parses)."""
    torch = _torch()
    lib = _lib.load()
    if isinstance(flows, torch.Tensor) and flows.dim() == 4 and flows.shape[0] > 0:
        _require_cuda(flows, torch.float32, 'flows')
        n, H, W, c = flows.shape
        if c != 2:
            raise ValueError('flows: expected 2 channels, got %d' % c)
        out = torch.empty((n, 2, FLOW_HIST_BINS), dtype=torch.int32, device=flows.device)
        with torch.cuda.device(flows.device):
            _lib.check(lib.stb_flow_hist_strided(C.c_void_p(flows.data_ptr()), H * W * 8, n, W, H,
                                                 C.c_void_p(out.data_ptr()), _stream_ptr(stream)), lib)
        return out
    lst, H, W = _frames_list(flows, torch.float32, 'flows', 2)
    n = len(lst)
    dev = lst[0].device if n else torch.device('cuda')
    out = torch.empty((n, 2, FLOW_HIST_BINS), dtype=torch.int32, device=dev)
    if n == 0:
        return out
    with torch.cuda.device(dev):
        tab = _lib.ptr_table([f.data_ptr() for f in lst])
        _lib.check(lib.stb_flow_hist(tab, n, W, H, C.c_void_p(out.data_ptr()), _stream_ptr(stream)), lib)
    return out


def frame_difference(prev, cur, stream=None):
    """FrameDifference op (intended semantics, stencil {-1, 0}): (cur - prev) mod 256 per byte."""
    torch = _torch()
    lib = _lib.load()
    _require_cuda(prev, torch.uint8, 'prev')
    _require_cuda(cur, torch.uint8, 'cur')
    if prev.shape != cur.shape:
        raise ValueError('prev and cur must have the same FrameInfo')
    out = torch.empty_like(cur)
    with torch.cuda.device(cur.device):
        _lib.check(lib.stb_frame_diff(C.c_void_p(prev.data_ptr()), C.c_void_p(cur.data_ptr()), C.c_void_p(out.data_ptr()),
                                      cur.numel(), _stream_ptr(stream)), lib)
    return out


def resize_target(frame_w, frame_h, width=0, height=0, min=False, preserve_aspect=False):
    """Target size of the Resize op for ResizeArgs(width, height, min, preserve_aspect)
    (scannertools_cpp/imgproc/resize_kernel.cpp:43-61)."""
    lib = _lib.load()
    w, h = C.c_int(), C.c_int()
    _lib.check(lib.stb_resize_target(frame_w, frame_h, int(width), int(height), 1 if min else 0,
                                     1 if preserve_aspect else 0, C.byref(w), C.byref(h)), lib)
    return w.value, h.value


def resize(frames, width=0, height=0, min=False, preserve_aspect=False, interpolation='INTER_LINEAR', stream=None):
    """Resize op (scannertools_cpp/imgproc/resize_kernel.cpp:22-105): n frames -> [n, height, width, C] of the
    input's dtype.  `frames` is one [n,H,W,C] / [H,W,C] tensor or a sequence of [H,W,C] tensors.

    uint8, C in {1, 3, 4}: bit-exact with cv::resize for INTER_LINEAR (the default), INTER_NEAREST, INTER_AREA,
    INTER_LANCZOS4 and INTER_CUBIC (OpenCV's own code path; builds that dispatch 8-bit cubic to IPP differ from it by
    one grey level on ~5 % of pixels).

    float32, C in 1..4 (an OpticalFlow field is [H,W,2]), against cv::resize's float code (cv2.ipp.setUseIPP(False)):
      INTER_NEAREST, INTER_LINEAR (exact 2x down included), INTER_AREA up-scaling and integer factors: bit-exact,
      signed zeros and infinities included; every mode at the frame's own size: a copy, as in OpenCV;
      INTER_AREA general down-scaling, INTER_CUBIC, INTER_LANCZOS4: every element within 8 * 2^-23 * max|frame| of
      OpenCV's double-precision result (general INTER_AREA matches cv2 bit for bit on every size tested).
    OpenCV builds that send float INTER_LINEAR to IPP differ from OpenCV's own code by up to ~2^-18.6 * max|frame|.

    Other dtypes raise TypeError.  The remaining names of the reference's table (:9-20: INTER_MAX, WARP_*, flag
    values rather than modes) raise NotImplementedError."""
    torch = _torch()
    lib = _lib.load()
    interp = lib.stb_resize_interp_code((interpolation or '').encode())
    if interp < 0:
        # resize_kernel.cpp:31-35: names outside the reference's INTERP_TYPES table silently mean INTER_LINEAR
        # (mirrored, like ResizeKernelGPU does); names INSIDE the table that are not implemented here raise
        if interpolation in RESIZE_TABLE_UNIMPLEMENTED:
            raise NotImplementedError('Resize: INTER_LINEAR, INTER_NEAREST, INTER_AREA, INTER_CUBIC and INTER_LANCZOS4 are implemented (got %r)' % (interpolation,))
        interp = lib.stb_resize_interp_code(b'INTER_LINEAR')
    if isinstance(frames, torch.Tensor) and frames.dim() == 3:
        frames = frames.unsqueeze(0)
    lst = [frames[i] for i in range(frames.shape[0])] if isinstance(frames, torch.Tensor) else list(frames)
    if not lst:
        raise ValueError('Resize needs at least one frame')
    dtype = lst[0].dtype if isinstance(lst[0], torch.Tensor) else None
    if dtype not in (torch.uint8, torch.float32):
        raise TypeError('Resize: frames must be uint8 or float32 CUDA tensors, got %s' % (dtype,))
    for f in lst:
        _require_cuda(f, dtype, 'frames')
    H, W, c = lst[0].shape
    if dtype == torch.float32:
        if not 1 <= c <= 4:
            raise ValueError('Resize: float32 frames must have 1 to 4 channels, got %d' % c)
        if any(tuple(f.shape) != (H, W, c) for f in lst):
            raise ValueError('Resize: every frame of a batch must have the same shape')
    tw, th = resize_target(W, H, width, height, min, preserve_aspect)
    if tw <= 0 or th <= 0:
        raise ValueError('Resize: target size %dx%d' % (tw, th))
    out = torch.empty((len(lst), th, tw, c), dtype=dtype, device=lst[0].device)
    fn = lib.stb_resize_u8 if dtype == torch.uint8 else lib.stb_resize_f32
    with torch.cuda.device(lst[0].device):
        st = _lib.ptr_table([f.data_ptr() for f in lst])
        dt = _lib.ptr_table([out[i].data_ptr() for i in range(len(lst))])
        _lib.check(fn(st, len(lst), W, H, c, dt, tw, th, interp, _stream_ptr(stream)), lib)
    return out


def convert_color(frames, conversion='COLOR_RGB2HSV', stream=None):
    """ConvertColor op (scannertools_cpp/imgproc/convert_color_kernel.cpp:239-281) / ConvertToHSVCPP
    (old/cpp_ops/imgproc.cpp:14-48) on uint8 frames; bit-exact with cv::cvtColor.  `frames` is one
    [n,H,W,C] / [H,W,C] tensor or a sequence of [H,W,C] tensors, C the conversion's input channel count
    (1-channel inputs are [n,H,W,1] / [H,W,1]); returns uint8 [n,H,W,out channels].  Implemented
    (both spellings where OpenCV has an alias):
      COLOR_RGB2HSV, COLOR_BGR2HSV, COLOR_RGB2HSV_FULL, COLOR_BGR2HSV_FULL (3 -> 3);
      COLOR_RGB2GRAY, COLOR_BGR2GRAY (3 -> 1); COLOR_RGBA2GRAY, COLOR_BGRA2GRAY (4 -> 1);
      COLOR_BGR2RGB / RGB2BGR (3 -> 3); COLOR_BGR2BGRA / RGB2RGBA, COLOR_BGR2RGBA / RGB2BGRA (3 -> 4, alpha 255);
      COLOR_BGRA2BGR / RGBA2RGB, COLOR_RGBA2BGR / BGRA2RGB (4 -> 3); COLOR_BGRA2RGBA / RGBA2BGRA (4 -> 4);
      COLOR_GRAY2BGR / GRAY2RGB (1 -> 3), COLOR_GRAY2BGRA / GRAY2RGBA (1 -> 4, alpha 255);
      COLOR_BGR2YCrCb, COLOR_RGB2YCrCb, COLOR_YCrCb2BGR, COLOR_YCrCb2RGB,
      COLOR_BGR2YUV, COLOR_RGB2YUV, COLOR_YUV2BGR, COLOR_YUV2RGB (packed 4:4:4, 3 -> 3).
    Any other name raises NotImplementedError; frames with the wrong channel count raise ValueError."""
    torch = _torch()
    lib = _lib.load()
    code = lib.stb_color_code(conversion.encode())
    if code < 0:
        raise NotImplementedError('ConvertColor: %s is not implemented' % conversion)
    if isinstance(frames, torch.Tensor) and frames.dim() == 3:
        frames = frames.unsqueeze(0)
    lst, H, W = _frames_list(frames, torch.uint8, 'frames', lib.stb_color_in_channels(code))
    if not lst:
        raise ValueError('ConvertColor needs at least one frame')
    oc = lib.stb_color_out_channels(code)
    out = torch.empty((len(lst), H, W, oc), dtype=torch.uint8, device=lst[0].device)
    with torch.cuda.device(lst[0].device):
        st = _lib.ptr_table([f.data_ptr() for f in lst])
        dt = _lib.ptr_table([out[i].data_ptr() for i in range(len(lst))])
        _lib.check(lib.stb_convert_color_u8(st, len(lst), W, H, code, dt, _stream_ptr(stream)), lib)
    return out


def blur(frames, kernel_size, stream=None):
    """Blur op (scannertools_cpp/imgproc/blur_kernel_cpu.cpp) on uint8 frames with 1, 3 or 4 channels: the
    reference's k x k box mean (its BlurArgs.sigma is never read), per channel, the window [-L, R] with
    L = ceil(k/2) - 1 and R = k/2, sum / k^2 truncated.  Pixels whose window leaves the frame are copies of the
    input (the reference leaves them unwritten).  `frames` is one [n,H,W,C] / [H,W,C] tensor or a sequence of
    [H,W,C] tensors; returns uint8 [n,H,W,C].  kernel_size < 1 raises ValueError, kernel_size > 255 StbError."""
    torch = _torch()
    lib = _lib.load()
    k = int(kernel_size)
    if k < 1:
        raise ValueError('Blur: kernel_size must be >= 1, got %d' % k)
    if isinstance(frames, torch.Tensor):
        if frames.dim() == 3:
            frames = frames.unsqueeze(0)
        if frames.dim() != 4:
            raise ValueError('Blur: frames must be [n,H,W,C] or [H,W,C], got shape %s' % (tuple(frames.shape),))
    else:
        frames = list(frames)
    if len(frames) == 0:
        raise ValueError('Blur needs at least one frame')
    first = frames[0]
    if isinstance(first, torch.Tensor) and (first.dim() != 3 or first.shape[-1] not in (1, 3, 4)):
        raise ValueError('Blur: frames must be [H,W,C] with C in 1, 3, 4, got %s' % (tuple(first.shape),))
    c = int(first.shape[-1]) if isinstance(first, torch.Tensor) else 0
    lst, H, W = _frames_list(frames, torch.uint8, 'frames', c)
    out = torch.empty((len(lst), H, W, c), dtype=torch.uint8, device=lst[0].device)
    with torch.cuda.device(lst[0].device):
        st = _lib.ptr_table([f.data_ptr() for f in lst])
        dt = _lib.ptr_table([out[i].data_ptr() for i in range(len(lst))])
        _lib.check(lib.stb_blur_u8(st, len(lst), W, H, c, k, dt, _stream_ptr(stream)), lib)
    return out


class OpticalFlow:
    """OpticalFlow op (dense Farneback, the reference's hard-coded parameters).

    Mirrors OpticalFlowKernelGPU (optical_flow_kernel_gpu.cpp:12-107): constructed once per
    device/FrameInfo, `execute` takes the B+1 unique frames of a stenciled batch and returns B
    flow frames (H x W x 2 f32); flow i maps frame i -> frame i+1 (the CPU kernel's direction,
    optical_flow_kernel_cpu.cpp:41)."""

    OPTFLOW_FARNEBACK_GAUSSIAN = 256

    def __init__(self, width, height, max_batch=16, device=None, num_levels=3, win_size=15, num_iters=3, flags=0,
                 pyr_scale=0.5, poly_n=5, poly_sigma=1.2):
        """The keyword defaults are the reference's hard-coded FarnebackOpticalFlow arguments
        (optical_flow_kernel_cpu.cpp:16).  Other pyramid depths (<= 3), 0.5 <= pyr_scale < 1, odd windows <= 31, polyN 3..7, iteration
        counts and flags=OPTFLOW_FARNEBACK_GAUSSIAN run on the generic kernels; anything else
        raises StbError (STB_ERR_UNSUPPORTED)."""
        torch = _torch()
        self._lib = _lib.load()
        self.width, self.height, self.max_batch = int(width), int(height), int(max_batch)
        self.device = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
        self._h = C.c_void_p()
        prm = _lib.FarnebackParams(int(num_levels), float(pyr_scale), 0, int(win_size), int(num_iters), int(poly_n),
                                   float(poly_sigma), int(flags))
        with torch.cuda.device(self.device):
            _lib.check(self._lib.stb_farneback_create(self.width, self.height, self.max_batch, C.byref(prm), C.byref(self._h)), self._lib)

    def close(self):
        if getattr(self, '_h', None) is not None and self._h:
            self._lib.stb_farneback_destroy(self._h)
            self._h = None

    __del__ = close

    def reset(self):
        """Scanner calls reset() at stream discontinuities; the kernel keeps no cross-call state."""

    def levels(self):
        ws = (C.c_int * 8)()
        hs = (C.c_int * 8)()
        n = self._lib.stb_farneback_levels(self._h, ws, hs)
        return [(ws[k], hs[k]) for k in range(n)]

    def workspace_bytes(self):
        return int(self._lib.stb_farneback_workspace_bytes(self.width, self.height, self.max_batch, None))

    def _check(self, lst, H, W):
        if (H, W) != (self.height, self.width):
            raise ValueError('frame size %dx%d does not match the kernel FrameInfo %dx%d' % (W, H, self.width, self.height))
        if len(lst) - 1 > self.max_batch:
            raise ValueError('batch of %d pairs exceeds max_batch=%d' % (len(lst) - 1, self.max_batch))
        for f in lst:
            if f.device != self.device:     # the handle's workspace lives on self.device (check_frame(device_, ...))
                raise ValueError('frame on %s, but this OpticalFlow kernel was created on %s' % (f.device, self.device))

    def execute(self, frames, out=None, stream=None, gray=False):
        torch = _torch()
        lst, H, W = _frames_list(frames, torch.uint8, 'frames', 1 if gray else 3)
        n = len(lst) - 1
        if n < 0:
            raise ValueError('OpticalFlow needs at least the two frames of its {0, 1} stencil')
        self._check(lst, H, W)
        if out is None:
            out = torch.empty((max(n, 0), H, W, 2), dtype=torch.float32, device=self.device)
        else:
            _require_cuda(out, torch.float32, 'out')
            if tuple(out.shape) != (max(n, 0), H, W, 2) or out.device != self.device:
                raise ValueError('out must be float32 [%d, %d, %d, 2] on %s, got %s on %s'
                                 % (max(n, 0), H, W, self.device, tuple(out.shape), out.device))
        if n == 0:
            return out
        with torch.cuda.device(self.device):
            ft = _lib.ptr_table([f.data_ptr() for f in lst])
            ot = _lib.ptr_table([out[i].data_ptr() for i in range(n)])
            fn = self._lib.stb_farneback_run_gray if gray else self._lib.stb_farneback_run
            _lib.check(fn(self._h, ft, n, ot, _stream_ptr(stream)), self._lib)
        return out

    def execute_with_histogram(self, frames, want_flow=True, stream=None):
        """OpticalFlow -> FlowHistogram without a round trip (SURVEY §8f rank 2).
        Returns (flow or None, int32 [n, 2, 64])."""
        torch = _torch()
        lst, H, W = _frames_list(frames, torch.uint8, 'frames', 3)
        n = len(lst) - 1
        self._check(lst, H, W)
        hist = torch.empty((max(n, 0), 2, FLOW_HIST_BINS), dtype=torch.int32, device=self.device)
        flow = torch.empty((max(n, 0), H, W, 2), dtype=torch.float32, device=self.device) if want_flow else None
        if n <= 0:
            return flow, hist
        with torch.cuda.device(self.device):
            ft = _lib.ptr_table([f.data_ptr() for f in lst])
            ot = _lib.ptr_table([flow[i].data_ptr() for i in range(n)]) if want_flow else None
            _lib.check(self._lib.stb_farneback_run_hist(self._h, ft, n, ot, C.c_void_p(hist.data_ptr()), _stream_ptr(stream)), self._lib)
        return flow, hist

    def debug_level(self, frames, level, pair=0):
        """Stage-by-stage parity helper: runs the batch and returns level-`level` intermediates
        of `pair` (I0, I1: [h,w]; R0, R1, M0: [5,h,w] planar; flow: [h,w,2])."""
        torch = _torch()
        w, h = self.levels()[level]
        mk = lambda *s: torch.zeros(s, dtype=torch.float32, device=self.device)
        d = dict(I0=mk(h, w), I1=mk(h, w), R0=mk(5, h, w), R1=mk(5, h, w), M0=mk(5, h, w), flow=mk(h, w, 2))
        p = lambda t: C.c_void_p(t.data_ptr())
        self._lib.stb_farneback_debug_set(self._h, level, pair, p(d['I0']), p(d['I1']), p(d['R0']), p(d['R1']), p(d['M0']), p(d['flow']))
        try:
            out = self.execute(frames)
            torch.cuda.synchronize(self.device)
        finally:
            self._lib.stb_farneback_debug_set(self._h, -1, 0, None, None, None, None, None, None)
        return out, d


class Pipe:
    """Host-buffer front end (stb_pipe_* in include/stb.h): numpy / pinned-host frames in,
    numpy results out; H2D copies of batch c+1 overlap the kernels of batch c."""

    def __init__(self, width, height, max_batch=16, want_flow=False, device=None):
        torch = _torch()
        self._lib = _lib.load()
        self.width, self.height, self.max_batch = int(width), int(height), int(max_batch)
        self.device = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
        self._p = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self._lib.stb_pipe_create(self.width, self.height, self.max_batch, 1 if want_flow else 0, C.byref(self._p)), self._lib)

    def close(self):
        if getattr(self, '_p', None) is not None and self._p:
            self._lib.stb_pipe_destroy(self._p)
            self._p = None

    __del__ = close

    @staticmethod
    def _host_ptr(a):
        torch = _torch()
        if isinstance(a, torch.Tensor):
            if a.is_cuda or not a.is_contiguous():
                raise TypeError('Pipe takes contiguous HOST buffers')
            return a.data_ptr(), a.shape
        a = np.ascontiguousarray(a)
        return a.ctypes.data, a.shape

    def histogram(self, frames, scores=True):
        """frames: host uint8 [n,H,W,3] -> (int32 [n,3,16], int32 [n] scores or None)."""
        torch = _torch()
        ptr, shape = self._host_ptr(frames)
        n = shape[0]
        hist = np.empty((n, 3, HIST_BINS), np.int32)
        S = np.empty((n,), np.int32) if scores else None
        with torch.cuda.device(self.device):
            _lib.check(self._lib.stb_pipe_hist(self._p, C.c_void_p(ptr), n, C.c_void_p(hist.ctypes.data),
                                               C.c_void_p(S.ctypes.data) if scores else None), self._lib)
        return hist, S

    def flow_async(self, frames, hist_out, flow_out=None):
        """Asynchronous OpticalFlow -> FlowHistogram: enqueues the call and returns a ticket for
        `wait`.  `frames` (host, ideally pinned) and `hist_out` (int32 [n,2,64] numpy or pinned
        tensor) must stay untouched until then.  Two calls may be in flight: submit call i+1, then
        wait for call i, and the uploads of one call hide behind the kernels of the other.
        flow_out (float32 [n,H,W,2] host buffer, ideally pinned) additionally returns the flow frames."""
        torch = _torch()
        ptr, shape = self._host_ptr(frames)
        n = shape[0] - 1
        optr, oshape = self._host_ptr(hist_out)
        if int(np.prod(oshape)) != n * 2 * FLOW_HIST_BINS:
            raise ValueError('hist_out must hold n x 2 x 64 int32')
        flp = None
        if flow_out is not None:
            fptr, fshape = self._host_ptr(flow_out)
            if tuple(fshape) != (n, self.height, self.width, 2) or getattr(flow_out, 'dtype', None) not in (np.float32, torch.float32):
                raise ValueError('flow_out must be float32 [n, H, W, 2]')
            flp = C.c_void_p(fptr)
        t = C.c_int(-1)
        with torch.cuda.device(self.device):
            _lib.check(self._lib.stb_pipe_flow_async(self._p, C.c_void_p(ptr), n, flp, C.c_void_p(optr), C.byref(t)), self._lib)
        return t.value

    def wait(self, ticket):
        if ticket >= 0:
            _lib.check(self._lib.stb_pipe_wait(self._p, ticket), self._lib)

    def flow(self, frames, want_flow=True, want_hist=False, flow_out=None):
        """frames: host uint8 [n+1,H,W,3] -> (float32 [n,H,W,2] or None, int32 [n,2,64] or None)."""
        torch = _torch()
        ptr, shape = self._host_ptr(frames)
        n = shape[0] - 1
        fl = None
        flp = None
        if want_flow:
            fl = flow_out if flow_out is not None else np.empty((n, self.height, self.width, 2), np.float32)
            flp = C.c_void_p(self._host_ptr(fl)[0])
        fh = np.empty((n, 2, FLOW_HIST_BINS), np.int32) if want_hist else None
        with torch.cuda.device(self.device):
            _lib.check(self._lib.stb_pipe_flow(self._p, C.c_void_p(ptr), n, flp,
                                               C.c_void_p(fh.ctypes.data) if want_hist else None), self._lib)
        return fl, fh
