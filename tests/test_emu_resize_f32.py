"""The float32 Resize kernels without a GPU (tests/cuda_emu): stb_resize_f32 against the restatement of
tests/resize_f32_restate.py (pinned to cv2 by test_resize_f32_oracle.py), bit for bit, in every interpolation mode at
1 to 4 channels on ragged sizes and on frame bases 4 and 8 bytes past 16-byte alignment; batches past one 64-entry
pointer table; and the C ABI's argument checks.  Every output buffer starts as bytes 0xA5, so an element the kernel
fails to write, or writes when it must not, shows."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

import resize_f32_restate as rr
from conftest import ROOT
from scannertools_b200 import _lib

sys.path.insert(0, os.path.join(ROOT, 'tests', 'cuda_emu'))

MODES = list(rr.INTERP)
SENTINEL = 0xA5


@pytest.fixture(scope='module')
def emu():
    import build_emu
    return _lib.bind(C.CDLL(build_emu.build()))


def placed(x, off):
    """A copy of x whose first element lies `off` bytes past a 16-byte boundary, inside a buffer of sentinel bytes;
    returns (buffer, address, view)."""
    nb = x.nbytes
    buf = np.full(nb + 64, SENTINEL, np.uint8)
    start = (-buf.ctypes.data) % 16 + off
    view = buf[start:start + nb].view(np.float32).reshape(x.shape)
    view[...] = x
    return buf, buf.ctypes.data + start, view


def run(emu, srcs, sw, sh, c, dw, dh, interp, outs=None):
    if outs is None:
        outs = [np.full((dh, dw, c), np.frombuffer(bytes([SENTINEL] * 4), np.float32)[0], np.float32) for _ in srcs]
    src = [s if isinstance(s, int) else s.ctypes.data for s in srcs]
    dst = [o if isinstance(o, int) else o.ctypes.data for o in outs]
    rc = emu.stb_resize_f32(_lib.ptr_table(src), len(src), sw, sh, c, _lib.ptr_table(dst), dw, dh,
                            rr.INTERP[interp] if isinstance(interp, str) else interp, None)
    return rc, outs


def same_bits(a, b):
    return np.array_equal(np.asarray(a, np.float32).view(np.uint32), np.asarray(b, np.float32).view(np.uint32))


# (sw, sh, dw, dh): up and down, exact 2x with dw % 4 = 0..3, integer factors 3 and 4, one axis up, a general
# factor, 1-pixel-wide and 1-row frames
SIZES = [(13, 11, 29, 17), (37, 29, 11, 7), (16, 10, 8, 5), (18, 6, 9, 3), (20, 4, 10, 2), (22, 8, 11, 4),
         (21, 12, 7, 4), (24, 16, 6, 4), (9, 13, 23, 5), (1, 7, 3, 5), (9, 1, 4, 3), (1, 1, 2, 3), (17, 15, 5, 6)]


@pytest.mark.parametrize('c', [1, 2, 3, 4])
@pytest.mark.parametrize('interp', MODES)
def test_emu_resize_f32_bit_exact_with_the_restatement(emu, interp, c):
    rng = np.random.default_rng(c * 10 + rr.INTERP[interp])
    for sw, sh, dw, dh in SIZES:
        x = (rng.standard_normal((sh, sw, c)) * 30).astype(np.float32)
        rc, out = run(emu, [x], sw, sh, c, dw, dh, interp)
        assert rc == 0, emu.stb_last_error()
        ref = rr.resize(x, dw, dh, interp)
        assert same_bits(out[0], ref), (interp, c, sw, sh, dw, dh, int((out[0] != ref).sum()))


@pytest.mark.parametrize('c', [1, 2, 3, 4])
@pytest.mark.parametrize('interp', MODES)
def test_emu_resize_f32_bases_off_16_byte_alignment(emu, interp, c):
    rng = np.random.default_rng(100 + c)
    for sw, sh, dw, dh in [(14, 10, 7, 5), (11, 9, 17, 6)]:   # exact 2x down, and up / down
        x = (rng.standard_normal((sh, sw, c)) * 30).astype(np.float32)
        ref = rr.resize(x, dw, dh, interp)
        for soff in (4, 8):
            for doff in (4, 8):
                sbuf, sp, _ = placed(x, soff)
                dbuf, dp, dv = placed(np.zeros((dh, dw, c), np.float32), doff)
                dbuf[:] = SENTINEL
                rc, _ = run(emu, [sp], sw, sh, c, dw, dh, interp, outs=[dp])
                assert rc == 0, emu.stb_last_error()
                assert same_bits(dv, ref), (interp, c, soff, doff)
                start = dp - dbuf.ctypes.data
                assert (dbuf[:start] == SENTINEL).all() and (dbuf[start + dv.nbytes:] == SENTINEL).all()


@pytest.mark.parametrize('interp', MODES)
def test_emu_resize_f32_batch_past_one_pointer_table(emu, interp):
    """67 frames: two launches (64 + 3 frames); every frame equals its single-frame call."""
    n, sw, sh, dw, dh, c = 67, 6, 5, 3, 4, 2
    rng = np.random.default_rng(7)
    xs = [(rng.standard_normal((sh, sw, c)) * 5).astype(np.float32) for _ in range(n)]
    rc, out = run(emu, xs, sw, sh, c, dw, dh, interp)
    assert rc == 0
    for i, x in enumerate(xs):
        assert same_bits(out[i], run(emu, [x], sw, sh, c, dw, dh, interp)[1][0]), i
        assert same_bits(out[i], rr.resize(x, dw, dh, interp)), i


def _untouched(outs):
    return all((o.view(np.uint8) == SENTINEL).all() for o in outs)


@pytest.mark.parametrize('side', ['src', 'dst'])
@pytest.mark.parametrize('interp', ['INTER_LINEAR', 'INTER_CUBIC'])
def test_emu_resize_f32_null_entry_at_65_leaves_every_output_untouched(emu, side, interp):
    n, bad = 67, 65
    src = np.random.default_rng(3).standard_normal((n, 4, 8, 2)).astype(np.float32)
    outs = [np.full((3, 5, 2), np.nan, np.float32) for _ in range(n)]
    for o in outs:
        o.view(np.uint8)[...] = SENTINEL
    st = [0 if side == 'src' and i == bad else src[i].ctypes.data for i in range(n)]
    dt = [0 if side == 'dst' and i == bad else outs[i].ctypes.data for i in range(n)]
    rc, _ = run(emu, st, 8, 4, 2, 5, 3, interp, outs=dt)
    assert rc == -1
    assert b'%s frame 65 is NULL' % (b'source' if side == 'src' else b'destination') in emu.stb_last_error()
    assert _untouched(outs)


def test_emu_resize_f32_argument_checks_write_nothing(emu):
    h, w, c = 5, 6, 2
    x = np.random.default_rng(1).standard_normal((h, w, c)).astype(np.float32)
    fresh = lambda cc=c: [np.frombuffer(bytes([SENTINEL]) * (3 * 4 * cc * 4), np.float32).reshape(3, 4, cc).copy()]
    # misaligned source or destination entry (1, 2 and 3 bytes past a float boundary), also past index 64
    for off in (1, 2, 3):
        sbuf = np.zeros(x.nbytes + 8, np.uint8)
        outs = fresh()
        rc, _ = run(emu, [sbuf.ctypes.data + off], w, h, c, 4, 3, 'INTER_LINEAR', outs=outs)
        assert rc == -1 and b'not 4-byte aligned' in emu.stb_last_error() and _untouched(outs), off
        dbuf = np.full(3 * 4 * c * 4 + 8, SENTINEL, np.uint8)
        rc, _ = run(emu, [x], w, h, c, 4, 3, 'INTER_NEAREST', outs=[dbuf.ctypes.data + off])
        assert rc == -1 and (dbuf == SENTINEL).all(), off
    xs = [x] * 67
    outs = [fresh()[0] for _ in range(67)]
    dt = [o.ctypes.data for o in outs]
    dt[65] += 2
    rc, _ = run(emu, xs, w, h, c, 4, 3, 'INTER_AREA', outs=dt)
    assert rc == -1 and b'destination frame 65 is not 4-byte aligned' in emu.stb_last_error() and _untouched(outs)
    # channels 0 and 5: unsupported; unknown interpolation codes: unsupported
    for cc in (0, 5):
        outs = fresh(max(cc, 1))
        assert run(emu, [x], w, h, cc, 4, 3, 'INTER_LINEAR', outs=outs)[0] == -4 and _untouched(outs), cc
    for interp in (-1, 5, 7):
        outs = fresh()
        assert run(emu, [x], w, h, c, 4, 3, interp, outs=outs)[0] == -4 and _untouched(outs), interp
    # bad sizes and n < 0
    for (ww, hh, dw, dh) in [(0, h, 4, 3), (w, -1, 4, 3), (w, h, 0, 3), (w, h, 4, -2)]:
        outs = fresh()
        assert run(emu, [x], ww, hh, c, dw, dh, 'INTER_LINEAR', outs=outs)[0] == -1 and _untouched(outs)
    outs = fresh()
    assert emu.stb_resize_f32(_lib.ptr_table([x.ctypes.data]), -1, w, h, c, _lib.ptr_table([outs[0].ctypes.data]), 4, 3, 0, None) == -1
    assert emu.stb_resize_f32(None, 1, w, h, c, _lib.ptr_table([outs[0].ctypes.data]), 4, 3, 0, None) == -1
    assert _untouched(outs)
    # n == 0 does nothing, even without tables or with bad arguments
    assert emu.stb_resize_f32(None, 0, w, h, c, None, 4, 3, 0, None) == 0
    assert emu.stb_resize_f32(None, 0, 0, 0, 9, None, 0, 0, 99, None) == 0
    # the 8-bit entry point still has no 2-channel kernel
    assert emu.stb_resize_u8(_lib.ptr_table([0]), 1, 4, 4, 2, _lib.ptr_table([0]), 2, 2, 0, None) == -4


def same_values(a, b):
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint32), b[~nb].view(np.uint32))


@pytest.mark.parametrize('c', [1, 2, 3, 4])
@pytest.mark.parametrize('interp', MODES)
def test_emu_resize_f32_signed_zeros_infinities_and_same_size(emu, interp, c):
    """Blocks of -0 at exact 2x with dw % 4 = 1..3 (OpenCV's scalar order turns them into +0, its vector body keeps
    -0), mixed +-0 elsewhere, and frames with +-inf / NaN resized to their own size (a copy in every mode) or, in the
    modes without taps, to other sizes."""
    rng = np.random.default_rng(50 + c)
    for sw, sh, dw, dh in [(14, 8, 7, 4), (18, 6, 9, 3), (22, 8, 11, 4), (16, 8, 8, 4), (13, 11, 29, 17), (37, 29, 11, 7)]:
        for x in (np.full((sh, sw, c), -0.0, np.float32),
                  np.where(rng.random((sh, sw, c)) < 0.5, -0.0, 0.0).astype(np.float32)):
            rc, out = run(emu, [x], sw, sh, c, dw, dh, interp)
            assert rc == 0 and same_bits(out[0], rr.resize(x, dw, dh, interp)), (interp, c, sw, sh, dw, dh)
    for sw, sh, dw, dh in [(13, 7, 13, 7), (1, 1, 1, 1), (14, 8, 7, 4), (13, 11, 29, 17)]:
        x = (rng.standard_normal((sh, sw, c)) * 10).astype(np.float32)
        m = rng.random(x.shape)
        x[m < 0.05], x[m > 0.95], x[(m > 0.5) & (m < 0.52)], x[(m > 0.6) & (m < 0.65)] = np.inf, -np.inf, np.nan, -0.0
        if (sw, sh) != (dw, dh) and rr.path(interp, sw, sh, dw, dh) in ('area', 'taps'):
            continue
        rc, out = run(emu, [x], sw, sh, c, dw, dh, interp)
        ref = rr.resize(x, dw, dh, interp)
        assert rc == 0 and same_values(out[0], ref), (interp, c, sw, sh, dw, dh)
        if (sw, sh) == (dw, dh):
            assert same_values(out[0], x)
