"""ConvertColor on the GPU for every conversion beyond HSV / gray / RGB<->BGR: bit for bit against cv2.cvtColor (or, where
cv2 is missing, the numpy restatements that tests/test_color_oracle.py pins to it) on all 2^24 inputs, on 1080p
batches, through ops.convert_color and through the Scanner kernel class."""
import ctypes as C

import numpy as np
import pytest

import color_restate as cr
from scannertools_b200 import synth

pytestmark = pytest.mark.gpu

try:
    import cv2
except Exception:  # cv2 missing on the box: fall back to the pinned restatement
    cv2 = None

NEW = sorted(cr.CONVERSIONS)


def reference(x, name):
    cin, cout = cr.CONVERSIONS[name]
    if cv2 is not None:
        out = cv2.cvtColor(np.ascontiguousarray(x[..., 0] if cin == 1 else x), getattr(cv2, name))
    else:
        out = cr.convert(x, name)
    return out.reshape(x.shape[:-1] + (cout,))


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


def with_channels(rgb, name):
    """Frames (..., 3) turned into inputs of the conversion: as they are, with a varied alpha, or their first byte."""
    cin = cr.CONVERSIONS[name][0]
    if cin == 3:
        return np.ascontiguousarray(rgb)
    if cin == 1:
        return np.ascontiguousarray(rgb[..., :1])
    a = (rgb[..., 0].astype(np.uint32) * 3 + rgb[..., 1] + 5 * rgb[..., 2]) & 255
    return np.ascontiguousarray(np.concatenate([rgb, a[..., None].astype(np.uint8)], -1))


@pytest.mark.parametrize('name', NEW)
def test_convert_color_every_input(torch, ops, name):
    """All 2^24 colours as one 4096 x 4096 frame (4-channel inputs with alpha varied over all 256 values, 1-channel
    inputs a ramp holding every value)."""
    x = cr.cube_input(name)
    out = ops.convert_color(dev(torch, x), name)
    assert tuple(out.shape) == (1, 4096, 4096, cr.CONVERSIONS[name][1])
    ref = reference(x, name)
    got = out.cpu().numpy()[0]
    assert np.array_equal(got, ref), (name, int((got != ref).any(-1).sum()))


@pytest.mark.parametrize('name', NEW)
def test_convert_color_1080p_batch_as_tensor_and_as_list(torch, ops, name):
    fr = with_channels(synth.noise_clip(19, 3, 1080, 1920), name)
    one = ops.convert_color(dev(torch, fr), name)
    lst = ops.convert_color([dev(torch, f) for f in fr], name)
    cout = cr.CONVERSIONS[name][1]
    assert tuple(one.shape) == tuple(lst.shape) == (3, 1080, 1920, cout)
    one, lst = one.cpu().numpy(), lst.cpu().numpy()
    assert np.array_equal(one, lst), name
    for i in range(3):
        assert np.array_equal(one[i], reference(fr[i], name)), (name, i)


def test_convert_color_shapes_and_channel_errors(torch, ops):
    rgb = dev(torch, synth.noise_clip(2, 2, 36, 52))
    rgba = dev(torch, with_channels(synth.noise_clip(3, 2, 36, 52), 'COLOR_RGBA2RGB'))
    gray = rgb[..., :1].contiguous()
    assert tuple(ops.convert_color(rgb, 'COLOR_RGB2RGBA').shape) == (2, 36, 52, 4)
    assert tuple(ops.convert_color(rgb[0], 'COLOR_RGB2YCrCb').shape) == (1, 36, 52, 3)
    assert tuple(ops.convert_color(rgba, 'COLOR_BGRA2GRAY').shape) == (2, 36, 52, 1)
    assert tuple(ops.convert_color(gray, 'COLOR_GRAY2BGRA').shape) == (2, 36, 52, 4)
    single = ops.convert_color(gray[1], 'COLOR_GRAY2RGB')
    assert tuple(single.shape) == (1, 36, 52, 3)
    assert torch.equal(single[0], gray[1].expand(36, 52, 3))
    for frames, name in [(rgb, 'COLOR_RGBA2BGR'), (rgba, 'COLOR_RGB2YUV'), (rgb, 'COLOR_GRAY2BGR'),
                         (gray, 'COLOR_BGR2HSV_FULL'), (rgba, 'COLOR_YCrCb2RGB'),
                         (rgb[..., 0].contiguous(), 'COLOR_GRAY2BGR'), ([rgba[0], rgb[1]], 'COLOR_RGBA2RGB')]:
        with pytest.raises(ValueError):
            ops.convert_color(frames, name)
    with pytest.raises(TypeError):
        ops.convert_color(rgba.float(), 'COLOR_RGBA2GRAY')
    with pytest.raises(ValueError):
        ops.convert_color(rgba[:, :, ::2], 'COLOR_RGBA2GRAY')          # not contiguous
    with pytest.raises(ValueError):
        ops.convert_color([], 'COLOR_GRAY2RGB')
    for name in ('COLOR_BGR2HLS', 'COLOR_HSV2BGR', 'COLOR_BGR2Lab', 'COLOR_YUV2RGB_NV12', 'COLOR_BGR2XYZ'):
        with pytest.raises(NotImplementedError):
            ops.convert_color(rgb, name)


@pytest.fixture(scope='module')
def shim():
    from scannertools_b200 import build
    return C.CDLL(build.build_scanner_ops())


@pytest.mark.parametrize('name', ['COLOR_BGR2RGBA', 'COLOR_RGBA2BGR', 'COLOR_BGRA2RGBA', 'COLOR_GRAY2RGBA',
                                  'COLOR_RGBA2GRAY', 'COLOR_RGB2YCrCb', 'COLOR_YUV2BGR', 'COLOR_RGB2HSV_FULL'])
def test_convert_color_kernel_class(shim, name):
    """ConvertColorKernelGPU takes frames of the conversion's input channel count and allocates output frames of
    its output channel count."""
    cin, cout = cr.CONVERSIONS[name]
    fr = with_channels(synth.noise_clip(8, 3, 45, 64), name)
    assert fr.shape == (3, 45, 64, cin)
    out = np.zeros((3, 45, 64, cout), np.uint8)
    oc = C.c_int()
    args = b'\x0a' + bytes([len(name)]) + name.encode()
    rc = shim.stb_shim_convert_color(C.c_void_p(fr.ctypes.data), 3, 64, 45, args, len(args),
                                     C.c_void_p(out.ctypes.data), C.byref(oc), 0)
    assert rc == 0 and oc.value == cout, (rc, oc.value)
    for i in range(3):
        assert np.array_equal(out[i], reference(fr[i], name)), (name, i)
