"""Float32 Resize on the GPU: OpticalFlow's 1080p flow fields resized to the shipped pipeline's 426x240 and to 960x540
(exact 2x) in all five modes, and one 4K four-channel frame, bit for bit against the restatement of
tests/resize_f32_restate.py, and against live cv2 by tier (bit for bit, or within 8 * 2^-23 * max|src| of cv2's
float64 run); batches as one tensor and as separate buffers; ops.resize's dtype and channel errors; the Scanner kernel
class on F32 frames; and launches per call."""
import ctypes as C

import numpy as np
import pytest

import resize_f32_restate as rr
from scannertools_b200 import _lib, synth

gpu = pytest.mark.gpu
MODES = list(rr.INTERP)

try:
    import cv2
except Exception:  # cv2 missing on the box: the restatement alone, which test_resize_f32_oracle.py pins to it
    cv2 = None


@pytest.fixture(scope='module')
def torch():
    import torch
    assert torch.cuda.is_available(), 'gpu tests need a CUDA device'
    return torch


@pytest.fixture(scope='module')
def ops(torch):
    from scannertools_b200 import ops
    return ops


@pytest.fixture(scope='module')
def flows(torch, ops):
    """Two real 1920x1080 flow fields from ops.OpticalFlow on a textured synth clip."""
    clip = synth.textured_clip(11, 3, 1080, 1920)
    of = ops.OpticalFlow(1920, 1080, max_batch=2)
    try:
        return of.execute(torch.from_numpy(clip).cuda()).cpu().numpy()
    finally:
        of.close()


def same_bits(a, b):
    return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))


def check(got, x, dw, dh, interp):
    ref = rr.resize(x, dw, dh, interp)
    assert same_bits(got, ref), (interp, x.shape, dw, dh, int((got != ref).sum()))
    if cv2 is None:
        return
    old = cv2.ipp.useIPP()
    cv2.ipp.setUseIPP(False)
    try:
        code = getattr(cv2, interp)
        live = cv2.resize(x, (dw, dh), interpolation=code).reshape(dh, dw, x.shape[2])
        sh, sw = x.shape[:2]
        if rr.path(interp, sw, sh, dw, dh) in ('nearest', 'linear', 'area_fast'):
            assert same_bits(got, live), (interp, x.shape, dw, dh, int((got != live).sum()))
        else:
            r64 = cv2.resize(x.astype(np.float64), (dw, dh), interpolation=code).reshape(dh, dw, x.shape[2])
            err = np.abs(got.astype(np.float64) - r64).max()
            assert err <= rr.bound(x), (interp, x.shape, dw, dh, err / rr.bound(x) * 8)
    finally:
        cv2.ipp.setUseIPP(old)


@gpu
@pytest.mark.parametrize('interp', MODES)
def test_flow_fields_at_1080p(torch, ops, flows, interp):
    d = torch.from_numpy(flows).cuda()
    for dw, dh in [(426, 240), (960, 540)]:
        out = ops.resize(d, dw, dh, interpolation=interp).cpu().numpy()
        assert out.shape == (2, dh, dw, 2) and out.dtype == np.float32
        for i in range(2):
            check(out[i], flows[i], dw, dh, interp)
        # the same batch as separate buffers
        sep = ops.resize([torch.from_numpy(f.copy()).cuda() for f in flows], dw, dh, interpolation=interp).cpu().numpy()
        assert same_bits(sep, out)


@gpu
@pytest.mark.parametrize('interp', MODES)
def test_one_4k_four_channel_frame(torch, ops, interp):
    x = (np.random.default_rng(4).standard_normal((2160, 3840, 4)) * 50).astype(np.float32)
    out = ops.resize(torch.from_numpy(x).cuda(), 1920, 1080, interpolation=interp).cpu().numpy()
    check(out[0], x, 1920, 1080, interp)


@gpu
def test_resize_dtype_and_channel_errors(torch, ops):
    for dt in (torch.float64, torch.int16, torch.float16):
        with pytest.raises(TypeError, match='uint8 or float32'):
            ops.resize(torch.zeros((1, 8, 8, 2), dtype=dt, device='cuda'), 4, 4)
    with pytest.raises(ValueError, match='1 to 4 channels'):
        ops.resize(torch.zeros((1, 8, 8, 5), dtype=torch.float32, device='cuda'), 4, 4)
    with pytest.raises(TypeError):
        ops.resize(torch.zeros((1, 8, 8, 2), dtype=torch.float32), 4, 4)          # host tensor
    with pytest.raises(TypeError):
        ops.resize([torch.zeros((8, 8, 2), dtype=torch.float32, device='cuda'),
                    torch.zeros((8, 8, 2), dtype=torch.uint8, device='cuda')], 4, 4)
    with pytest.raises(_lib.StbError):
        ops.resize(torch.zeros((1, 8, 8, 2), dtype=torch.uint8, device='cuda'), 4, 4)   # no 2-channel 8-bit kernel
    # a [H,W,C] tensor is one frame
    assert ops.resize(torch.zeros((8, 8, 2), dtype=torch.float32, device='cuda'), 4, 4).shape == (1, 4, 4, 2)


@gpu
def test_resize_kernel_class_on_f32_frames(ops):
    from scannertools_b200 import build
    from test_scanner_ops import _resize_args
    shim = C.CDLL(build.build_scanner_ops())
    n, h, w = 3, 270, 480
    fr = synth.textured_flow_field(3, h, w)[None].repeat(n, 0).astype(np.float32)
    fr[1] *= -0.5
    fr[2] += 1.25
    fr = np.ascontiguousarray(fr)
    out = np.zeros(n * h * w * 2, np.float32)
    ow, oh = C.c_int(), C.c_int()
    for name in MODES:
        args = _resize_args(width=213, preserve_aspect=True, interpolation=name.encode())
        rc = shim.stb_shim_resize_f32(C.c_void_p(fr.ctypes.data), n, w, h, 2, args, len(args), C.c_void_p(out.ctypes.data),
                                      out.size, C.byref(ow), C.byref(oh), 0)
        assert rc == 0 and (ow.value, oh.value) == (213, h * 213 // w), (name, rc)
        got = out[:n * oh.value * ow.value * 2].reshape(n, oh.value, ow.value, 2)
        for i in range(n):
            assert same_bits(got[i], rr.resize(fr[i], ow.value, oh.value, name)), (name, i)
    bad = _resize_args(width=10, height=10, interpolation=b'INTER_MAX')
    assert shim.stb_shim_resize_f32(C.c_void_p(fr.ctypes.data), 1, w, h, 2, bad, len(bad), C.c_void_p(out.ctypes.data),
                                    out.size, C.byref(ow), C.byref(oh), 0) == -4


@gpu
def test_resize_f32_launch_counts(torch, ops):
    """One launch per 64-entry pointer table (the cubic tap tables are uploaded, not launched); none for a rejected
    table."""
    lib = _lib.load()
    n, h, w = 130, 6, 8
    src = torch.randn((n, h, w, 2), device='cuda')
    dst = torch.empty((n, 3, 4, 2), device='cuda')
    st = _lib.ptr_table([src[i].data_ptr() for i in range(n)])
    dt = _lib.ptr_table([dst[i].data_ptr() for i in range(n)])
    for interp in range(5):
        l0 = lib.stb_launch_count()
        assert lib.stb_resize_f32(st, n, w, h, 2, dt, 4, 3, interp, None) == 0
        torch.cuda.synchronize()
        assert lib.stb_launch_count() - l0 == 3, interp
        for i in (0, 64, 129):
            assert same_bits(dst[i].cpu().numpy(), rr.resize(src[i].cpu().numpy(), 4, 3, MODES[interp])), (interp, i)
    bad = _lib.ptr_table([src[i].data_ptr() if i != 65 else 0 for i in range(n)])
    mis = _lib.ptr_table([dst[i].data_ptr() + (2 if i == 100 else 0) for i in range(n)])
    l0 = lib.stb_launch_count()
    assert lib.stb_resize_f32(bad, n, w, h, 2, dt, 4, 3, 3, None) == -1
    assert lib.stb_resize_f32(st, n, w, h, 2, mis, 4, 3, 0, None) == -1
    assert lib.stb_launch_count() == l0


def same_values(a, b):
    """Bit for bit, with NaN matched by NaN-ness (the GPU's NaN payload is its own)."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint32), b[~nb].view(np.uint32))


@gpu
@pytest.mark.parametrize('interp', MODES)
def test_signed_zeros_infinities_and_same_size_copies(torch, ops, flows, interp):
    """A flow field with -0 blocks resized by exactly 2x (OpenCV's scalar order at 2 channels gives +0 there), and
    a field with +-inf / NaN / -0 resized to its own size, which is a copy in every mode."""
    x = flows[0].copy()
    x[:200:2, :300:2] = -0.0
    x[:200:2, 1:300:2] = -0.0
    x[1:200:2, :300] = -0.0
    out = ops.resize(torch.from_numpy(x).cuda(), 960, 540, interpolation=interp).cpu().numpy()[0]
    assert same_bits(out, rr.resize(x, 960, 540, interp)), interp
    if rr.path(interp, 1920, 1080, 960, 540) == 'area_fast':
        assert not np.signbit(out[:100, :150]).any()
    y = flows[1].copy()
    y[::97, ::89] = np.inf
    y[5::101, ::83] = -np.inf
    y[7::61, 3::67] = np.nan
    y[::7, ::5] = -0.0
    same = ops.resize(torch.from_numpy(y).cuda(), 1920, 1080, interpolation=interp).cpu().numpy()[0]
    assert same_values(same, y), interp
