"""numpy restatement of the Blur op (stb_blur_u8, ops.blur): the reference BlurKernel's box mean
(scannertools_cpp/imgproc/blur_kernel_cpu.cpp) with k = kernel_size, window rows and columns [-L, R] around the pixel,
L = ceil(k/2) - 1, R = k/2, an unsigned sum divided by k*k with truncation on interior pixels
(L <= x < W - R, L <= y < H - R) and a copy of the input everywhere else.

`blur` is built on 2-D cumulative sums; `blur_loop` is a literal transcription of the reference's quadruple loop
that test_blur_oracle.py pins it to, and `cv2_interior` is the OpenCV expression that agrees with both on the
interior.  `div_constants` / `div` restate the host-side multiply-shift division of csrc/blur.cu."""
import numpy as np


def window(k):
    return (k + 1) // 2 - 1, k // 2


def blur(x, k):
    """x: uint8 [H, W, C] -> uint8 [H, W, C]."""
    x = np.asarray(x)
    H, W, C = x.shape
    out = x.copy()
    if H < k or W < k:
        return out
    L, R = window(k)
    S = np.zeros((H + 1, W + 1, C), np.int64)
    S[1:, 1:] = x.astype(np.int64).cumsum(0).cumsum(1)
    tot = S[k:, k:] - S[:H - k + 1, k:] - S[k:, :W - k + 1] + S[:H - k + 1, :W - k + 1]
    out[L:H - R, L:W - R] = (tot // (k * k)).astype(np.uint8)
    return out


def blur_loop(x, k):
    """The reference's loop, written out: every interior pixel and channel sums its k x k window and divides; the
    other pixels keep the input value (the reference does not write them at all)."""
    x = np.asarray(x)
    H, W, C = x.shape
    L, R = window(k)
    out = x.copy()
    for y in range(L, H - R):
        for xx in range(L, W - R):
            for c in range(C):
                s = 0
                for dy in range(-L, R + 1):
                    for dx in range(-L, R + 1):
                        s += int(x[y + dy, xx + dx, c])
                out[y, xx, c] = s // (k * k)
    return out


def interior(H, W, k):
    """(rows, cols) slices of the interior, possibly empty."""
    L, R = window(k)
    return slice(L, max(H - R, L)), slice(L, max(W - R, L))


def cv2_interior(x, k):
    """cv2.boxFilter(..., CV_32S, (k, k), anchor=(L, L), normalize=False) // k^2 on the interior."""
    import cv2
    x = np.ascontiguousarray(x)
    L, _ = window(k)
    s = cv2.boxFilter(x, cv2.CV_32S, (k, k), anchor=(L, L), normalize=False)
    s = s.reshape(x.shape)
    ys, xs = interior(x.shape[0], x.shape[1], k)
    return (s[ys, xs] // (k * k)).astype(np.uint8)


def div_constants(k):
    """(m, s) with floor(n / k^2) == (n * m) >> s for 0 <= n <= 255 k^2: l = ceil(log2 k^2), s = 8 + 2l,
    m = ceil(2^s / k^2)."""
    d = k * k
    l = 0
    while (1 << l) < d:
        l += 1
    s = 8 + 2 * l
    return -(-(1 << s) // d), s


def div(n, k):
    m, s = div_constants(k)
    return (np.asarray(n, np.int64) * m) >> s
