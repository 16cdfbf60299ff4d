"""TEST INFRASTRUCTURE ONLY: numpy integer restatements of the 8-bit cv::cvtColor conversions that
ConvertColor implements beyond HSV / gray / RGB<->BGR (those are in oracle/restate.c).  OpenCV-free, so
the GPU tests can use them where cv2 is missing; tests/test_color_oracle.py pins every one of them
against cv2.cvtColor on all 2^24 colours.

OpenCV's fixed point (modules/imgproc/src/color_yuv.simd.hpp, color_hsv.simd.hpp), all 8-bit:
  YCrCb / YUV forward: Y = (R*4899 + G*9617 + B*1868 + 2^13) >> 14,
                       Cr = ((R - Y)*11682 + (128 << 14) + 2^13) >> 14, Cb = ((B - Y)*9241 + ...) >> 14;
                       YUV uses V = (R - Y)*14369, U = (B - Y)*8061 and stores Y, U, V (YCrCb stores Y, Cr, Cb).
  inverse:             R = Y + ((Cr - 128)*22987 + 2^13) >> 14, G = Y + ((Cb - 128)*-5636 + (Cr - 128)*-11698 + 2^13) >> 14,
                       B = Y + ((Cb - 128)*29049 + 2^13) >> 14; YUV: V*18678, U*-6472 + V*-9519, U*33292.
  HSV_FULL:            the HSV-180 integer path with hdiv[d] = cvRound(256*4096 / (6 d)) and +256 on a negative hue.
"""
import numpy as np

# name -> (in channels, out channels); aliases OpenCV defines with the same value share a row's function
CONVERSIONS = {
    'COLOR_BGR2BGRA': (3, 4), 'COLOR_RGB2RGBA': (3, 4), 'COLOR_BGR2RGBA': (3, 4), 'COLOR_RGB2BGRA': (3, 4),
    'COLOR_BGRA2BGR': (4, 3), 'COLOR_RGBA2RGB': (4, 3), 'COLOR_RGBA2BGR': (4, 3), 'COLOR_BGRA2RGB': (4, 3),
    'COLOR_BGRA2RGBA': (4, 4), 'COLOR_RGBA2BGRA': (4, 4),
    'COLOR_GRAY2BGR': (1, 3), 'COLOR_GRAY2RGB': (1, 3), 'COLOR_GRAY2BGRA': (1, 4), 'COLOR_GRAY2RGBA': (1, 4),
    'COLOR_BGRA2GRAY': (4, 1), 'COLOR_RGBA2GRAY': (4, 1),
    'COLOR_BGR2YCrCb': (3, 3), 'COLOR_RGB2YCrCb': (3, 3), 'COLOR_YCrCb2BGR': (3, 3), 'COLOR_YCrCb2RGB': (3, 3),
    'COLOR_BGR2YUV': (3, 3), 'COLOR_RGB2YUV': (3, 3), 'COLOR_YUV2BGR': (3, 3), 'COLOR_YUV2RGB': (3, 3),
    'COLOR_BGR2HSV_FULL': (3, 3), 'COLOR_RGB2HSV_FULL': (3, 3),
}


def _descale(x):
    return (x + (1 << 13)) >> 14


def _u8(x):
    return np.clip(x, 0, 255).astype(np.uint8)


def _gray15(r, g, b):
    return ((b * 3735 + g * 19235 + r * 9798 + (1 << 14)) >> 15).astype(np.uint8)


def _to_luma_chroma(r, g, b, kr, kb, crcb):
    y = _descale(r * 4899 + g * 9617 + b * 1868)
    v = _descale((r - y) * kr + (128 << 14))
    u = _descale((b - y) * kb + (128 << 14))
    return np.stack([y, v, u] if crcb else [y, u, v], -1)


def _from_luma_chroma(f, c_r, c_gv, c_gu, c_b, crcb):
    y, a, b = f[..., 0], f[..., 1] - 128, f[..., 2] - 128
    v, u = (a, b) if crcb else (b, a)
    return y + _descale(v * c_r), y + _descale(u * c_gu + v * c_gv), y + _descale(u * c_b)


def _hsv_full(r, g, b):
    i = np.arange(1, 256, dtype=np.float64)
    sdiv = np.concatenate([[0], np.rint((255 << 12) / i)]).astype(np.int64)
    hdiv = np.concatenate([[0], np.rint((256 << 12) / (6 * i))]).astype(np.int64)
    v = np.maximum(np.maximum(r, g), b)
    d = v - np.minimum(np.minimum(r, g), b)
    s = (d * sdiv[v] + (1 << 11)) >> 12
    h = np.where(v == r, g - b, np.where(v == g, b - r + 2 * d, r - g + 4 * d))
    h = (h * hdiv[d] + (1 << 11)) >> 12
    h = h + np.where(h < 0, 256, 0)
    return np.stack([_u8(h), s.astype(np.uint8), v.astype(np.uint8)], -1)


def convert(frame, conversion):
    """cv::cvtColor(frame, out, conversion) for the names in CONVERSIONS.  frame: uint8 [..., cin] (or [...] for a
    1-channel input); returns uint8 [..., cout], or [...] for a 1-channel output, as cv2 does."""
    cin, cout = CONVERSIONS[conversion]
    f = np.asarray(frame, np.uint8)
    if cin == 1 and (f.ndim < 3 or f.shape[-1] != 1):
        f = f[..., None]
    f = f.astype(np.int64)
    name = conversion[len('COLOR_'):]
    src, dst = name.split('2')
    if src == 'GRAY':
        out = np.repeat(f, cout, -1)
        if cout == 4:
            out[..., 3] = 255
        return out.astype(np.uint8)
    # the colour-space and alpha conversions read B,G,R from an input whose name starts with B
    if src.startswith(('BGR', 'RGB')):
        c0, c1, c2 = f[..., 0], f[..., 1], f[..., 2]
        r, g, b = (c2, c1, c0) if src.startswith('BGR') else (c0, c1, c2)
        if dst == 'GRAY':
            return _gray15(r, g, b)
        if dst in ('YCrCb', 'YUV'):
            crcb = dst == 'YCrCb'
            return _u8(_to_luma_chroma(r, g, b, 11682 if crcb else 14369, 9241 if crcb else 8061, crcb))
        if dst == 'HSV_FULL':
            return _hsv_full(r, g, b)
        alpha = f[..., 3] if cin == 4 else np.full_like(r, 255)
        chans = [b, g, r] if dst.startswith('BGR') else [r, g, b]
        if cout == 4:
            chans.append(alpha)
        return np.stack(chans, -1).astype(np.uint8)
    crcb = src == 'YCrCb'
    r, g, b = _from_luma_chroma(f, *((22987, -11698, -5636, 29049) if crcb else (18678, -9519, -6472, 33292)), crcb)
    return _u8(np.stack([b, g, r] if dst == 'BGR' else [r, g, b], -1))


def cube():
    """All 2^24 RGB colours as one 4096 x 4096 x 3 frame: pixel (y, x) = (y >> 4, ((y & 15) << 4) | (x >> 8), x & 255)."""
    v = np.arange(1 << 24, dtype=np.uint32)
    return np.stack([(v >> 16) & 255, (v >> 8) & 255, v & 255], -1).astype(np.uint8).reshape(4096, 4096, 3)


def cube_input(conversion):
    """The exhaustive input of one conversion: the RGB cube for 3-channel inputs; for 4-channel inputs the cube
    with alpha varying over all 256 values (alpha = (r + 7 g + 13 b) & 255, so every colour meets a different alpha
    than its neighbours); for 1-channel inputs a 4096 x 4096 ramp holding every value 65536 times."""
    cin = CONVERSIONS[conversion][0]
    c = cube()
    if cin == 3:
        return c
    if cin == 4:
        a = (c[..., 0].astype(np.uint32) + 7 * c[..., 1] + 13 * c[..., 2]) & 255
        return np.concatenate([c, a[..., None].astype(np.uint8)], -1)
    return (np.arange(1 << 24, dtype=np.uint32) & 255).astype(np.uint8).reshape(4096, 4096, 1)
