"""ConvertColor's conversion kernels without a GPU (tests/cuda_emu): every code beyond HSV / gray / RGB<->BGR against
the numpy restatements of tests/color_restate.py (pinned to cv2 on all 2^24 colours by test_color_oracle.py), on
ragged sizes, unaligned bases, batches past one 64-entry pointer table, and the C ABI's name and channel tables."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

import color_restate as cr
from conftest import ROOT
from scannertools_b200 import _lib

sys.path.insert(0, os.path.join(ROOT, 'tests', 'cuda_emu'))

NEW = sorted(cr.CONVERSIONS)
# (name, in, out) of the conversions implemented before the table grew; their codes 0..4 are fixed
OLD = [('COLOR_RGB2HSV', 3, 3), ('COLOR_BGR2HSV', 3, 3), ('COLOR_RGB2GRAY', 3, 1), ('COLOR_BGR2GRAY', 3, 1),
       ('COLOR_BGR2RGB', 3, 3), ('COLOR_RGB2BGR', 3, 3)]
OUT_OF_SCOPE = ['COLOR_BGR2XYZ', 'COLOR_XYZ2BGR', 'COLOR_RGB2XYZ', 'COLOR_BGR2HLS', 'COLOR_RGB2HLS_FULL',
                'COLOR_HSV2BGR', 'COLOR_HSV2RGB_FULL', 'COLOR_HLS2RGB', 'COLOR_BGR2Lab', 'COLOR_Lab2BGR', 'COLOR_RGB2Luv',
                'COLOR_YUV2RGB_NV12', 'COLOR_YUV2BGR_I420', 'COLOR_RGB2YUV_I420', 'COLOR_YUV2RGB_YUY2',
                'COLOR_BayerBG2BGR', 'COLOR_BGR2BGR565', 'COLOR_BGR5552BGR', 'COLOR_RGBA2mRGBA', 'COLOR_mRGBA2RGBA',
                'COLOR_rgb2hsv', 'COLOR_RGB2YCRCB', 'RGB2YCrCb', 'COLOR_RGB2HSV_FULL ', '']


@pytest.fixture(scope='module')
def emu():
    import build_emu
    return _lib.bind(C.CDLL(build_emu.build()))


def channels(name):
    return cr.CONVERSIONS[name]


def as_input(rgb, name, rng=None):
    """An input of the conversion's channel count holding the colours `rgb` (..., 3): the colour itself, the colour
    with a varied alpha, or its first byte as a gray value."""
    cin = channels(name)[0]
    if cin == 3:
        return np.ascontiguousarray(rgb)
    if cin == 1:
        return np.ascontiguousarray(rgb[..., :1])
    a = (rgb[..., 0].astype(np.uint32) + 7 * rgb[..., 1] + 13 * rgb[..., 2]) & 255
    return np.ascontiguousarray(np.concatenate([rgb, a[..., None].astype(np.uint8)], -1))


def reference(x, name):
    return cr.convert(x, name).reshape(x.shape[:-1] + (channels(name)[1],))


def run(emu, frames, name, w, h, out=None):
    """frames: list of host arrays (or raw addresses); returns the n output frames as one array."""
    code = emu.stb_color_code(name.encode())
    cout = channels(name)[1]
    if out is None:
        out = np.full((len(frames), h, w, cout), 0xA5, np.uint8)
    src = [f if isinstance(f, int) else f.ctypes.data for f in frames]
    rc = emu.stb_convert_color_u8(_lib.ptr_table(src), len(frames), w, h, code, _lib.ptr_table([o.ctypes.data for o in out]), None)
    assert rc == 0, (name, rc, emu.stb_last_error())
    return out


@pytest.mark.parametrize('name', NEW)
def test_emu_color_ragged_sizes_and_unaligned_bases(emu, name):
    rng = np.random.default_rng(31)
    for (h, w) in [(1, 1), (37, 53)]:
        x = as_input(rng.integers(0, 256, (h, w, 3), dtype=np.uint8), name)
        ref = reference(x, name)
        assert np.array_equal(run(emu, [x], name, w, h)[0], ref), (name, h, w)
        for off in (1, 3):
            buf = np.zeros(x.size + 8, np.uint8)
            buf[off:off + x.size] = x.reshape(-1)
            assert np.array_equal(run(emu, [buf.ctypes.data + off], name, w, h)[0], ref), (name, h, w, off)
            # the destination at an odd base as well
            cout = channels(name)[1]
            obuf = np.full(h * w * cout + 8, 0xA5, np.uint8)
            code = emu.stb_color_code(name.encode())
            assert emu.stb_convert_color_u8(_lib.ptr_table([x.ctypes.data]), 1, w, h, code,
                                            _lib.ptr_table([obuf.ctypes.data + off]), None) == 0
            assert np.array_equal(obuf[off:off + ref.size], ref.reshape(-1)), (name, h, w, off)
            assert (obuf[:off] == 0xA5).all() and (obuf[off + ref.size:] == 0xA5).all()


@pytest.mark.parametrize('name', ['COLOR_RGB2RGBA', 'COLOR_BGRA2RGB', 'COLOR_GRAY2BGRA', 'COLOR_RGBA2GRAY',
                                  'COLOR_YCrCb2BGR', 'COLOR_RGB2HSV_FULL'])
def test_emu_color_batch_past_one_pointer_table(emu, name):
    """67 frames: two launches (64 + 3 frames); every frame equals its single-frame call."""
    n, h, w = 67, 5, 9
    rng = np.random.default_rng(5)
    xs = [as_input(rng.integers(0, 256, (h, w, 3), dtype=np.uint8), name) for _ in range(n)]
    out = run(emu, xs, name, w, h)
    for i, x in enumerate(xs):
        assert np.array_equal(out[i], run(emu, [x], name, w, h)[0]), (name, i)
        assert np.array_equal(out[i], reference(x, name)), (name, i)


def cube_sample():
    """Every 61st colour of the RGB cube (275,037 colours) plus every colour whose channels are all extremal or next
    to an extreme / the chroma midpoint, as one frame."""
    v = np.arange(0, 1 << 24, 61, dtype=np.uint32)
    sample = np.stack([(v >> 16) & 255, (v >> 8) & 255, v & 255], -1).astype(np.uint8)
    ext = np.array([0, 1, 2, 126, 127, 128, 129, 253, 254, 255], np.uint8)
    corners = np.stack(np.meshgrid(ext, ext, ext, indexing='ij'), -1).reshape(-1, 3)
    px = np.concatenate([sample, corners])
    w = 1000
    pad = (-len(px)) % w
    px = np.concatenate([px, px[:pad]])
    return px.reshape(-1, w, 3)


@pytest.mark.parametrize('name', NEW)
def test_emu_color_cube_sample_and_extremes(emu, name):
    rgb = cube_sample()
    if channels(name)[0] == 1:
        rgb = np.repeat(np.arange(256, dtype=np.uint8), 3).reshape(1, 256, 3)
    x = as_input(rgb, name)
    if channels(name)[0] == 4:
        # alpha 0 and 255 on the extremal colours as well
        x = np.concatenate([x, x.copy()], 0)
        x[x.shape[0] // 2:, :, 3] = np.where(np.arange(x.shape[1]) % 2, 0, 255)
    h, w = x.shape[:2]
    assert np.array_equal(run(emu, [x], name, w, h)[0], reference(x, name)), name


@pytest.mark.parametrize('name,side', [('COLOR_RGB2RGBA', 'src'), ('COLOR_RGB2RGBA', 'dst'), ('COLOR_RGBA2BGR', 'src'),
                                       ('COLOR_GRAY2RGB', 'dst'), ('COLOR_RGB2YCrCb', 'src'), ('COLOR_YUV2RGB', 'dst'),
                                       ('COLOR_BGRA2GRAY', 'dst'), ('COLOR_BGR2HSV_FULL', 'src')])
def test_emu_color_null_entry_at_65_leaves_every_output_untouched(emu, name, side):
    n, h, w, bad = 67, 4, 8, 65
    cin, cout = channels(name)
    src = np.random.default_rng(3).integers(0, 256, (n, h, w, cin), dtype=np.uint8)
    out = np.full((n, h, w, cout), 0xA5, np.uint8)
    st = _lib.ptr_table([0 if side == 'src' and i == bad else src[i].ctypes.data for i in range(n)])
    dt = _lib.ptr_table([0 if side == 'dst' and i == bad else out[i].ctypes.data for i in range(n)])
    rc = emu.stb_convert_color_u8(st, n, w, h, emu.stb_color_code(name.encode()), dt, None)
    assert rc == -1 and b'NULL' in emu.stb_last_error(), (rc, emu.stb_last_error())
    assert b'%s frame 65' % (b'source' if side == 'src' else b'destination') in emu.stb_last_error()
    assert (out == 0xA5).all()


def test_emu_color_codes_and_channel_counts(emu):
    codes = {}
    for name, cin, cout in OLD + [(k, *v) for k, v in cr.CONVERSIONS.items()]:
        code = emu.stb_color_code(name.encode())
        assert 0 <= code < 99, name
        assert (emu.stb_color_in_channels(code), emu.stb_color_out_channels(code)) == (cin, cout), name
        codes.setdefault(code, set()).add(name)
    # the codes of the first five conversions are part of the ABI
    assert [emu.stb_color_code(n.encode()) for n, _, _ in OLD] == [0, 1, 2, 3, 4, 4]
    # aliases share a code exactly where OpenCV gives the two names one value
    cv_value = {}
    try:
        import cv2
        cv_value = {n: getattr(cv2, n) for c in codes.values() for n in c}
    except ImportError:
        pass
    for names in codes.values():
        assert len(names) <= 2, names
        if cv_value:
            assert len({cv_value[n] for n in names}) == 1, names
    if cv_value:
        assert len({cv_value[n] for c in codes.values() for n in c}) == len(codes)
    for bad in (-1, len(codes), 98, 99, 1 << 20):
        assert emu.stb_color_in_channels(bad) == 0 and emu.stb_color_out_channels(bad) == 0, bad
    x = np.zeros(12, np.uint8)
    assert emu.stb_convert_color_u8(_lib.ptr_table([x.ctypes.data]), 1, 2, 2, len(codes), _lib.ptr_table([x.ctypes.data]), None) == -4


@pytest.mark.parametrize('name', OUT_OF_SCOPE)
def test_emu_color_out_of_scope_names_stay_unimplemented(emu, name):
    assert emu.stb_color_code(name.encode()) == -1
