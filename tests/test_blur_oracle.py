"""The Blur restatement of tests/blur_restate.py, pinned on the CPU: to a literal transcription of the reference's
loop, to OpenCV's unnormalised box filter on the interior for every supported kernel size, and to the input on the
border; and the multiply-shift division csrc/blur.cu uses, checked at every point where the quotient changes."""
import numpy as np
import pytest

import blur_restate as br


@pytest.mark.parametrize('k', range(1, 10))
def test_blur_restatement_equals_the_reference_loop(k):
    rng = np.random.default_rng(k)
    for (h, w) in [(k + 3, k + 5), (k, k + 1), (max(k - 1, 1), k + 2), (2 * k + 1, 3)]:
        for c in (1, 3, 4):
            x = rng.integers(0, 256, (h, w, c), dtype=np.uint8)
            assert np.array_equal(br.blur(x, k), br.blur_loop(x, k)), (k, h, w, c)
    # extreme values: every window sum at its maximum, and one bright pixel
    x = np.full((k + 4, k + 4, 3), 255, np.uint8)
    assert np.array_equal(br.blur(x, k), x)
    x[:] = 0
    x[k // 2 + 1, k // 2 + 1] = 255
    assert np.array_equal(br.blur(x, k), br.blur_loop(x, k))


@pytest.mark.parametrize('c', [1, 3, 4])
def test_blur_restatement_equals_cv2_box_filter_on_the_interior(have_cv2, c):
    if not have_cv2:
        pytest.skip('cv2 not installed')
    rng = np.random.default_rng(100 + c)
    for k in range(1, 256):
        for (h, w) in [(k + 3, k + 2), (max(k - 1, 1), k + 4), (k + 1, max(k - 1, 1))]:
            x = rng.integers(0, 256, (h, w, c), dtype=np.uint8)
            got = br.blur(x, k)
            ys, xs = br.interior(h, w, k)
            assert np.array_equal(got[ys, xs], br.cv2_interior(x, k)), (k, h, w, c)


@pytest.mark.parametrize('k', [1, 2, 3, 4, 5, 8, 16, 31, 64, 255])
def test_blur_border_is_the_input(k):
    rng = np.random.default_rng(k)
    for (h, w) in [(k + 6, k + 3), (k - 1 or 1, k + 6), (1, 1)]:
        x = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        got = br.blur(x, k)
        ys, xs = br.interior(h, w, k)
        mask = np.ones((h, w), bool)
        mask[ys, xs] = False
        assert np.array_equal(got[mask], x[mask]), (k, h, w)
        if k == 1 or h < k or w < k:
            assert np.array_equal(got, x)


def test_blur_multiply_shift_division_is_exact():
    """floor(n / k^2) == (n * m) >> s for every k in 1..255 at every breakpoint q k^2 - 1 and q k^2 (q in 0..255) and at
    255 k^2: (n * m) >> s is monotone in n, so agreeing on both sides of every step agrees everywhere between."""
    q = np.arange(256, dtype=np.int64)
    for k in range(1, 256):
        d = k * k
        m, s = br.div_constants(k)
        assert m < 1 << 32 and 255 * d * m < 1 << 63, k
        n = np.concatenate([q * d - 1, q * d, [255 * d]])
        n = n[n >= 0]
        assert np.array_equal(br.div(n, k), n // d), k
