"""Blur on the GPU: stb_blur_u8 through ops.blur bit for bit against the restatement of tests/blur_restate.py (and
OpenCV's unnormalised box filter on the interior) on 1080p batches given as one tensor and as separate buffers, on
1- and 4-channel frames and on one 4K frame; ops.blur's argument errors; and the Scanner kernel class."""
import ctypes as C
import struct

import numpy as np
import pytest

import blur_restate as br
from scannertools_b200 import synth

gpu = pytest.mark.gpu

try:
    import cv2
except Exception:  # cv2 missing on the box: the restatement alone, which test_blur_oracle.py pins to it
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


def dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def check(got, x, k):
    ref = br.blur(x, k)
    assert np.array_equal(got, ref), (k, x.shape, int((got != ref).any(-1).sum()))
    if cv2 is not None:
        ys, xs = br.interior(x.shape[0], x.shape[1], k)
        assert np.array_equal(got[ys, xs], br.cv2_interior(x, k)), (k, x.shape)


@gpu
@pytest.mark.parametrize('k', [1, 2, 3, 4, 5, 7, 15, 31, 64, 255])
def test_blur_1080p_batch_as_tensor_and_as_list(torch, ops, k):
    fr = synth.noise_clip(40 + k, 3, 1080, 1920)
    one = ops.blur(dev(torch, fr), k)
    lst = ops.blur([dev(torch, f) for f in fr], k)
    assert tuple(one.shape) == tuple(lst.shape) == (3, 1080, 1920, 3)
    one, lst = one.cpu().numpy(), lst.cpu().numpy()
    assert np.array_equal(one, lst), k
    for i in range(3):
        check(one[i], fr[i], k)


@gpu
@pytest.mark.parametrize('c', [1, 4])
@pytest.mark.parametrize('k', [3, 15])
def test_blur_1080p_one_and_four_channels(torch, ops, k, c):
    rng = np.random.default_rng(k * c)
    fr = rng.integers(0, 256, (2, 1080, 1920, c), dtype=np.uint8)
    out = ops.blur(dev(torch, fr), k).cpu().numpy()
    assert out.shape == fr.shape
    for i in range(2):
        check(out[i], fr[i], k)


@gpu
def test_blur_one_4k_frame(torch, ops):
    fr = synth.noise_clip(9, 1, 2160, 3840)[0]
    out = ops.blur(dev(torch, fr), 3)
    assert tuple(out.shape) == (1, 2160, 3840, 3)
    check(out.cpu().numpy()[0], fr, 3)


@gpu
def test_blur_errors(torch, ops):
    from scannertools_b200._lib import StbError
    fr = dev(torch, synth.noise_clip(2, 2, 36, 52))
    assert tuple(ops.blur(fr[0], 3).shape) == (1, 36, 52, 3)
    for frames in [fr[..., :2].contiguous(), fr[..., :1].expand(2, 36, 52, 5).contiguous(), fr[0, :, :, 0],
                   [fr[0], fr[1, :20]], [fr[0], fr[1, ..., :1].contiguous()], []]:
        with pytest.raises(ValueError):
            ops.blur(frames, 3)
    with pytest.raises(ValueError):
        ops.blur(fr[:, :, ::2], 3)                       # not contiguous
    with pytest.raises(TypeError):
        ops.blur(fr.cpu(), 3)
    with pytest.raises(TypeError):
        ops.blur(fr.float(), 3)
    for k in (0, -1):
        with pytest.raises(ValueError):
            ops.blur(fr, k)
    with pytest.raises(StbError) as e:
        ops.blur(fr, 256)
    assert e.value.code == -4


@pytest.fixture(scope='module')
def shim():
    from scannertools_b200 import build
    lib = C.CDLL(build.build_scanner_ops())
    lib.stb_shim_registered.argtypes = [C.c_char_p, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    return lib


def blur_args(kernel_size=None, sigma=None, double=False):
    """Serialized BlurArgs { int32 kernel_size = 1; float sigma = 2; }; sigma as fixed64 when `double`."""
    out = b''
    if kernel_size is not None:
        v = kernel_size & ((1 << 64) - 1)
        out += b'\x08'
        while True:
            b = v & 0x7f
            v >>= 7
            out += bytes([b | (0x80 if v else 0)])
            if not v:
                break
    if sigma is not None:
        out += b'\x11' + struct.pack('<d', sigma) if double else b'\x15' + struct.pack('<f', sigma)
    return out


def test_blur_registered_under_the_reference_name(shim):
    b, l, h = C.c_int(-1), C.c_int(99), C.c_int(99)
    assert shim.stb_shim_registered(b'Blur', C.byref(b), C.byref(l), C.byref(h)) == 1
    assert (b.value, l.value, h.value) == (1, 0, 0)


@gpu
@pytest.mark.parametrize('c', [1, 3, 4])
def test_blur_kernel_class(shim, c):
    n, h, w = 3, 45, 64
    fr = np.random.default_rng(c).integers(0, 256, (n, h, w, c), dtype=np.uint8)
    for args, k in [(blur_args(3, 0.5), 3), (blur_args(4, 2.0, double=True), 4), (blur_args(5), 5)]:
        out = np.zeros_like(fr)
        rc = shim.stb_shim_blur(C.c_void_p(fr.ctypes.data), n, w, h, c, args, len(args), C.c_void_p(out.ctypes.data),
                                out.size, 0)
        assert rc == 0, (rc, args)
        for i in range(n):
            assert np.array_equal(out[i], br.blur(fr[i], k)), (k, c, i)
    # empty args, kernel_size 0 (absent), 0 (explicit), negative and 256 fail validate()
    for args in [b'', blur_args(None, 0.5), blur_args(0, 0.5), blur_args(-3), blur_args(256, 0.5), b'\x08']:
        out = np.zeros_like(fr)
        assert shim.stb_shim_blur(C.c_void_p(fr.ctypes.data), n, w, h, c, args, len(args),
                                  C.c_void_p(out.ctypes.data), out.size, 0) == -4, args
