"""numpy restatement of the float32 Resize kernels (csrc/resize.cu, resize_*_f32_kernel): cv::resize's float code paths,
every product and sum rounded on its own, in OpenCV's order.  test_resize_f32_oracle.py pins it to cv2 (bit for bit
where OpenCV's order is known, within a bound where it is not); the emulator and GPU tests compare the kernels with
it bit for bit.

resize(src, dw, dh, interp) takes one H x W x C frame.  With dtype=np.float64 the same algorithm runs in double with
the same float coefficients, a reference for the error bound."""
import math

import numpy as np

f32 = np.float32
INTERP = {'INTER_LINEAR': 0, 'INTER_NEAREST': 1, 'INTER_AREA': 2, 'INTER_CUBIC': 3, 'INTER_LANCZOS4': 4}
DBL_EPSILON = 2.220446049250313e-16


def _scales(sw, sh, dw, dh):
    return 1.0 / (dw / sw), 1.0 / (dh / sh)


def path(interp, sw, sh, dw, dh):
    """The code path cv::resize takes (resize.cu plan_resize): nearest, area_fast, area, linear or taps.  At
    dsize == ssize cv::resize copies the frame in every mode: nearest at scale 1."""
    if sw == dw and sh == dh:
        return 'nearest'
    if interp in ('INTER_CUBIC', 'INTER_LANCZOS4'):
        return 'taps'
    if interp == 'INTER_NEAREST':
        return 'nearest'
    sx, sy = _scales(sw, sh, dw, dh)
    isx, isy = round(sx), round(sy)   # round half even, as saturate_cast<int>
    int_scale = abs(sx - isx) < DBL_EPSILON and abs(sy - isy) < DBL_EPSILON
    down = sx >= 1 and sy >= 1
    if interp == 'INTER_LINEAR' and sw == 2 * dw and sh == 2 * dh:
        return 'area_fast'
    if interp == 'INTER_AREA' and down and int_scale:
        return 'area_fast'
    if interp == 'INTER_AREA' and down:
        return 'area'
    return 'linear'


def _nearest(src, dw, dh):
    sh, sw = src.shape[:2]
    scx, scy = _scales(sw, sh, dw, dh)
    xs = np.minimum(np.floor(np.arange(dw) * scx).astype(np.int64), sw - 1)
    ys = np.minimum(np.floor(np.arange(dh) * scy).astype(np.int64), sh - 1)
    return src[ys][:, xs].copy()


def _linear_axis(dn, sn, scale, area_mode, clamp_frac):
    """Per destination index: first source index, second source index and the float fraction (linear_taps)."""
    s = np.empty(dn, np.int64)
    fr = np.empty(dn, f32)
    inv = dn / sn
    for d in range(dn):
        if not area_mode:
            f = f32((d + 0.5) * scale - 0.5)
            i = math.floor(f)
            f = f32(f - f32(i))
        else:
            i = math.floor(d * scale)
            f = f32((d + 1) - (i + 1) * inv)
            f = f32(0) if f <= 0 else f32(f - f32(math.floor(f)))
        s[d], fr[d] = i, f
    if clamp_frac:   # x: cv::resize clamps index and fraction; y keeps the fraction and clips the rows
        lo = s < 0
        s[lo], fr[lo] = 0, 0
        hi = s >= sn - 1
        s[hi], fr[hi] = sn - 1, 0
        return s, np.where(s + 1 < sn, s + 1, s), fr
    return np.clip(s, 0, sn - 1), np.clip(s + 1, 0, sn - 1), fr


def _linear(src, dw, dh, area_mode):
    sh, sw = src.shape[:2]
    scx, scy = _scales(sw, sh, dw, dh)
    x0, x1, fx = _linear_axis(dw, sw, scx, area_mode, True)
    y0, y1, fy = _linear_axis(dh, sh, scy, area_mode, False)
    dt = src.dtype.type
    a0, a1 = (f32(1) - fx).astype(dt)[None, :, None], fx.astype(dt)[None, :, None]
    b0, b1 = (f32(1) - fy).astype(dt)[:, None, None], fy.astype(dt)[:, None, None]
    r0, r1 = src[y0], src[y1]
    # columns clamped at the right border (x1 == x0): S * 1 without the neighbour term, OpenCV's dx >= xmax loop
    edge = (x1 == x0)[None, :, None]
    h0 = np.where(edge, r0[:, x0] * a0, r0[:, x0] * a0 + r0[:, x1] * a1)
    h1 = np.where(edge, r1[:, x0] * a0, r1[:, x0] * a0 + r1[:, x1] * a1)
    return h0 * b0 + h1 * b1


def _area_fast(src, dw, dh):
    sh, sw, cn = src.shape
    isx, isy = round(sw / dw), round(sh / dh)
    dt = src.dtype.type
    blk = src[:dh * isy, :dw * isx].reshape(dh, isy, dw, isx, cn)
    if isx == 2 and isy == 2:
        a, b, c, d = blk[:, 0, :, 0], blk[:, 0, :, 1], blk[:, 1, :, 0], blk[:, 1, :, 1]
        vec = (a + b) + (c + d)      # OpenCV's 4-float vector body
        seq = dt(0) + (((a + b) + c) + d)   # its scalar code: WT sum = 0, then the block
        if cn == 4:
            s = vec
        elif cn == 1:
            s = seq.copy()
            nv = (dw // 4) * 4
            s[:, :nv] = vec[:, :nv]
        else:
            s = seq
        return s * dt(0.25)
    area = isx * isy
    el = [blk[:, j, :, i] for j in range(isy) for i in range(isx)]   # row-major block order
    s = np.zeros_like(el[0])
    k = 0
    while k + 4 <= area:
        s = s + (((el[k] + el[k + 1]) + el[k + 2]) + el[k + 3])
        k += 4
    for k in range(k, area):
        s = s + el[k]
    return s * dt(f32(1) / f32(area))


def area_span(d, scale, ssize):
    """cv::computeResizeAreaTab for one destination index: [(source index, float weight)] in table order."""
    f1 = d * scale
    f2 = f1 + scale
    cell = min(scale, ssize - f1)
    s1, s2 = math.ceil(f1), math.floor(f2)
    s2 = min(s2, ssize - 1)
    s1 = min(s1, s2)
    taps = []
    if s1 - f1 > 1e-3:
        taps.append((s1 - 1, f32((s1 - f1) / cell)))
    for s in range(s1, s2):
        taps.append((s, f32(1.0 / cell)))
    if f2 - s2 > 1e-3:
        taps.append((s2, f32(min(min(f2 - s2, 1.0), cell) / cell)))
    return taps


def _area(src, dw, dh):
    sh, sw, cn = src.shape
    scx, scy = _scales(sw, sh, dw, dh)
    dt = src.dtype.type
    xt = [area_span(d, scx, sw) for d in range(dw)]
    n = max(len(t) for t in xt)
    xi = np.zeros((n, dw), np.int64)
    xa = np.zeros((n, dw), dt)
    live = np.zeros((n, dw), bool)
    for d, t in enumerate(xt):
        for i, (s, a) in enumerate(t):
            xi[i, d], xa[i, d], live[i, d] = s, a, True
    out = np.empty((dh, dw, cn), dt)
    for dy in range(dh):
        acc = None
        for j, (sy, beta) in enumerate(area_span(dy, scy, sh)):
            row = src[sy]
            buf = np.zeros((dw, cn), dt)
            for i in range(n):
                m = live[i]
                buf[m] = buf[m] + row[xi[i, m]] * xa[i, m][:, None]
            acc = dt(beta) * buf if acc is None else acc + dt(beta) * buf
        out[dy] = acc
    return out


def cubic_coeffs(x):
    """cv::interpolateCubic in float (resize.cu cubic_coeffs)."""
    A = f32(-0.75)
    x = f32(x)
    x1 = f32(x + f32(1))
    ox = f32(f32(1) - x)
    c0 = f32(f32(f32(f32(f32(A * x1) - f32(f32(5) * A)) * x1) + f32(f32(8) * A)) * x1) - f32(f32(4) * A)
    c1 = f32(f32(f32(f32(f32(A + f32(2)) * x) - f32(A + f32(3))) * x) * x) + f32(1)
    c2 = f32(f32(f32(f32(f32(A + f32(2)) * ox) - f32(A + f32(3))) * ox) * ox) + f32(1)
    c3 = f32(f32(f32(f32(1) - c0) - c1) - c2)
    return [f32(c0), f32(c1), f32(c2), c3]


def lanczos4_coeffs(x):
    """cv::interpolateLanczos4 (resize.cu lanczos4_coeffs): double sin / cos, float weights normalised in float."""
    x = f32(x)
    if x < f32(1.1920928955078125e-07):
        c = [f32(0)] * 8
        c[3] = f32(1)
        return c
    s45 = 0.70710678118654752440
    cs = [(1, 0), (-s45, -s45), (0, 1), (s45, -s45), (-1, 0), (s45, s45), (0, -1), (-s45, s45)]
    pi = 3.1415926535897932384626433832795
    xd = float(f32(x + f32(3)))
    y0 = -xd * pi * 0.25
    s0, c0 = math.sin(y0), math.cos(y0)
    c = []
    tot = f32(0)
    for i in range(8):
        y = -float(f32(f32(x + f32(3)) - f32(i))) * pi * 0.25
        v = f32((cs[i][0] * s0 + cs[i][1] * c0) / (y * y))
        c.append(v)
        tot = f32(tot + v)
    tot = f32(f32(1) / tot)
    return [f32(v * tot) for v in c]


def taps(dn, sn, K):
    """resize.cu build_taps: first tap index and K float coefficients per destination index."""
    scale = 1.0 / (dn / sn)
    ofs = np.empty(dn, np.int64)
    co = np.empty((dn, K), f32)
    for d in range(dn):
        f = f32((d + 0.5) * scale - 0.5)
        s0 = math.floor(f)
        f = f32(f - f32(s0))
        co[d] = cubic_coeffs(f) if K == 4 else lanczos4_coeffs(f)
        ofs[d] = s0 - (K // 2 - 1)
    return ofs, co


def _taps(src, dw, dh, K):
    sh, sw = src.shape[:2]
    dt = src.dtype.type
    xo, xa = taps(dw, sw, K)
    yo, ya = taps(dh, sh, K)
    xa, ya = xa.astype(dt), ya.astype(dt)
    cx = np.clip(xo[:, None] + np.arange(K)[None, :], 0, sw - 1)   # [dw, K]
    cy = np.clip(yo[:, None] + np.arange(K)[None, :], 0, sh - 1)   # [dh, K]
    acc = None
    for j in range(K):
        r = src[cy[:, j]]                                           # [dh, sw, C]
        h = r[:, cx[:, 0]] * xa[None, :, 0, None]
        for k in range(1, K):
            h = h + r[:, cx[:, k]] * xa[None, :, k, None]
        t = h * ya[:, j, None, None]
        acc = t if acc is None else acc + t
    return acc


def resize(src, dw, dh, interp='INTER_LINEAR', dtype=np.float32):
    """src: H x W x C; returns dh x dw x C of `dtype` (float32: the kernels' result)."""
    src = np.asarray(src)
    if src.ndim == 2:
        src = src[:, :, None]
    src = src.astype(dtype)
    sh, sw = src.shape[:2]
    p = path(interp, sw, sh, dw, dh)
    with np.errstate(over='ignore', invalid='ignore'):
        if p == 'nearest':
            return _nearest(src, dw, dh)
        if p == 'area_fast':
            return _area_fast(src, dw, dh)
        if p == 'area':
            return _area(src, dw, dh)
        if p == 'linear':
            return _linear(src, dw, dh, interp == 'INTER_AREA')
        return _taps(src, dw, dh, 4 if interp == 'INTER_CUBIC' else 8)


def bound(src):
    """The error bound of the bound tier: 8 units of 2^-23 * max|src|."""
    return 8 * 2.0 ** -23 * float(np.abs(np.asarray(src, np.float64)).max())
