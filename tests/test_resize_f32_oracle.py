"""Pins the float32 Resize restatement (tests/resize_f32_restate.py) to cv2's float code (cv2.ipp.setUseIPP(False)):
bit for bit where OpenCV's order of operations is reproduced (INTER_NEAREST, INTER_LINEAR with its exact-2x fast
area path, INTER_AREA up-scaling, integer factors and, on these sizes, general down-scaling), and within
8 * 2^-23 * max|src| of cv2's float64 run where it is not (INTER_CUBIC, INTER_LANCZOS4; general INTER_AREA as well)."""
import numpy as np
import pytest

import resize_f32_restate as rr

cv2 = pytest.importorskip('cv2')

# (sw, sh, dw, dh): up, down, exact 2x with dw % 4 = 0..3 (OpenCV's 1-channel vector body and scalar tail), integer
# factors 3, 4 and 5, one axis up and one down, general factors (60x45 -> 20x15 has scale 3.0000000000000004, not an
# integer), 1-pixel-wide and 1-row frames
SIZES = [(37, 29, 53, 41), (64, 48, 23, 17), (40, 30, 20, 15), (42, 30, 21, 15), (44, 30, 22, 15), (46, 30, 23, 15),
         (90, 60, 30, 20), (80, 60, 20, 15), (75, 50, 15, 10), (13, 11, 40, 29), (17, 9, 17, 30), (60, 45, 20, 15),
         (100, 37, 31, 12), (1, 7, 3, 5), (9, 1, 4, 3), (2, 2, 1, 1), (1, 1, 3, 2), (426, 240, 213, 120)]
EXACT = ('INTER_NEAREST', 'INTER_LINEAR', 'INTER_AREA')
BOUND = ('INTER_AREA', 'INTER_CUBIC', 'INTER_LANCZOS4')


def cv(src, dw, dh, interp):
    return cv2.resize(src, (dw, dh), interpolation=getattr(cv2, interp)).reshape(dh, dw, src.shape[2])


@pytest.fixture
def no_ipp():
    old = cv2.ipp.useIPP()
    cv2.ipp.setUseIPP(False)
    yield
    cv2.ipp.setUseIPP(old)


@pytest.mark.parametrize('c', [1, 2, 3, 4])
@pytest.mark.parametrize('interp', EXACT)
def test_restatement_is_cv2_bit_for_bit(no_ipp, interp, c):
    rng = np.random.default_rng(10 * c + rr.INTERP[interp])
    for sw, sh, dw, dh in SIZES:
        src = (rng.standard_normal((sh, sw, c)) * 40).astype(np.float32)
        me, ref = rr.resize(src, dw, dh, interp), cv(src, dw, dh, interp)
        assert np.array_equal(me.view(np.uint32), ref.view(np.uint32)), (interp, c, sw, sh, dw, dh, int((me != ref).sum()))


@pytest.mark.parametrize('c', [1, 2, 3, 4])
@pytest.mark.parametrize('interp', BOUND)
def test_restatement_and_cv2_within_the_bound_of_cv2_float64(no_ipp, interp, c):
    rng = np.random.default_rng(20 * c + rr.INTERP[interp])
    for sw, sh, dw, dh in SIZES + [(192, 108, 43, 24), (43, 24, 192, 108)]:
        src = (rng.standard_normal((sh, sw, c)) * 40).astype(np.float32)
        r64 = cv(src.astype(np.float64), dw, dh, interp)
        b = rr.bound(src)
        for name, got in (('restatement', rr.resize(src, dw, dh, interp)), ('cv2 float32', cv(src, dw, dh, interp))):
            err = np.abs(got.astype(np.float64) - r64).max()
            assert err <= b, (name, interp, c, sw, sh, dw, dh, err / b * 8)
        # the float64 restatement is the same algorithm in double: far inside the bound
        assert np.abs(rr.resize(src, dw, dh, interp, dtype=np.float64) - r64).max() <= b / 8


@pytest.mark.parametrize('interp', list(rr.INTERP))
def test_ipp_dispatch_stays_near_opencvs_own_code(interp):
    """Builds with IPP send float INTER_LINEAR at 1, 3 and 4 channels to it; that result moves by up to about
    2^-18.6 * max|src| and is reported, not matched."""
    old = cv2.ipp.useIPP()
    rng = np.random.default_rng(5)
    try:
        for c in (1, 2, 3, 4):
            for sw, sh, dw, dh in [(37, 29, 53, 41), (64, 48, 23, 17), (40, 30, 20, 15)]:
                src = (rng.standard_normal((sh, sw, c)) * 40).astype(np.float32)
                cv2.ipp.setUseIPP(True)
                with_ipp = cv(src, dw, dh, interp)
                cv2.ipp.setUseIPP(False)
                own = cv(src, dw, dh, interp)
                lim = 2.0 ** -16 * np.abs(src).max()
                assert np.abs(with_ipp.astype(np.float64) - own).max() <= lim, (interp, c, sw, sh, dw, dh)
    finally:
        cv2.ipp.setUseIPP(old)


def same_values(a, b):
    """Bit for bit, with NaN matched by NaN-ness (a NaN's payload is the platform's, not OpenCV's)."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint32), b[~nb].view(np.uint32))


@pytest.mark.parametrize('c', [1, 2, 3, 4])
def test_signed_zeros_in_the_exact_tier(no_ipp, c):
    """OpenCV's exact-2x scalar code starts its sum at +0, so a block of -0 gives +0 there; its vector body keeps -0.
    Frames of all -0 and of mixed +-0, exact 2x with dw % 4 = 0..3, integer factors, up- and general scales."""
    rng = np.random.default_rng(30 + c)
    for sw, sh, dw, dh in [(16, 8, 8, 4), (14, 8, 7, 4), (18, 6, 9, 3), (22, 8, 11, 4), (21, 12, 7, 4), (13, 11, 29, 17),
                           (37, 29, 11, 7), (60, 45, 20, 15)]:
        for x in (np.full((sh, sw, c), -0.0, np.float32),
                  np.where(rng.random((sh, sw, c)) < 0.5, -0.0, 0.0).astype(np.float32)):
            for interp in EXACT:
                me, ref = rr.resize(x, dw, dh, interp), cv(x, dw, dh, interp)
                assert same_values(me, ref), (interp, c, sw, sh, dw, dh)


@pytest.mark.parametrize('c', [1, 2, 3, 4])
def test_infinities_and_nans_in_the_exact_tier_and_same_size_copies(no_ipp, c):
    """+-inf, NaN and -0 among finite values: nearest, linear and the area paths follow OpenCV (the clamped right
    column of linear takes S * 1, no 0 * inf); at dsize == ssize every mode is OpenCV's copy."""
    rng = np.random.default_rng(40 + c)
    for sw, sh, dw, dh in [(16, 8, 8, 4), (14, 8, 7, 4), (21, 12, 7, 4), (13, 11, 29, 17), (9, 13, 23, 5), (13, 7, 13, 7),
                           (1, 1, 1, 1), (5, 1, 5, 1)]:
        x = (rng.standard_normal((sh, sw, c)) * 10).astype(np.float32)
        m = rng.random(x.shape)
        x[m < 0.05], x[m > 0.95], x[(m > 0.5) & (m < 0.52)], x[(m > 0.6) & (m < 0.65)] = np.inf, -np.inf, np.nan, -0.0
        for interp in rr.INTERP:
            if rr.path(interp, sw, sh, dw, dh) in ('area', 'taps'):
                continue
            me, ref = rr.resize(x, dw, dh, interp), cv(x, dw, dh, interp)
            assert same_values(me, ref), (interp, c, sw, sh, dw, dh)
        if (sw, sh) == (dw, dh):
            for interp in rr.INTERP:
                assert same_values(rr.resize(x, dw, dh, interp), x), interp
