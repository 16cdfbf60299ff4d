"""The Blur kernel without a GPU (tests/cuda_emu): stb_blur_u8 against the restatement of tests/blur_restate.py
(pinned to the reference loop and to cv2 by test_blur_oracle.py) on ragged sizes, frames one byte or one row past a
CTA's tile or strip, unaligned bases, batches past one 64-entry pointer table, and the C ABI's argument checks.
Every output buffer starts as 0xA5, so a byte the kernel fails to write shows."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

import blur_restate as br
from conftest import ROOT
from scannertools_b200 import _lib

sys.path.insert(0, os.path.join(ROOT, 'tests', 'cuda_emu'))

KS = [1, 2, 3, 4, 5, 8, 15, 16, 31, 64, 255]
TILE_BYTES = 1024      # output bytes of a row per CTA (kBlurTileBytes)
STRIP_ROWS = 64        # rows per CTA for k <= 17 (max(64, 4 (k - 1)))


@pytest.fixture(scope='module')
def emu():
    """The emulator library, in which csrc/common.cu includes csrc/blur.cu; rebuilt when blur.cu is newer."""
    import build_emu
    blur = os.path.join(ROOT, 'scannertools_b200', 'csrc', 'blur.cu')
    stale = os.path.isfile(build_emu.OUT) and os.path.getmtime(blur) > os.path.getmtime(build_emu.OUT)
    return _lib.bind(C.CDLL(build_emu.build(force=stale)))


def run(emu, frames, k, w, h, c, out=None):
    """frames: host arrays or raw addresses; returns (status, outputs)."""
    if out is None:
        out = np.full((len(frames), h, w, c), 0xA5, np.uint8)
    src = [f if isinstance(f, int) else f.ctypes.data for f in frames]
    rc = emu.stb_blur_u8(_lib.ptr_table(src), len(frames), w, h, c, k, _lib.ptr_table([o.ctypes.data for o in out]), None)
    return rc, out


def check(emu, x, k):
    h, w, c = x.shape
    rc, out = run(emu, [x], k, w, h, c)
    assert rc == 0, (k, x.shape, emu.stb_last_error())
    ref = br.blur(x, k)
    assert np.array_equal(out[0], ref), (k, x.shape, int((out[0] != ref).sum()))


@pytest.mark.parametrize('c', [1, 3, 4])
@pytest.mark.parametrize('k', KS)
def test_emu_blur_ragged_sizes(emu, k, c):
    rng = np.random.default_rng(k * 10 + c)
    sizes = {(1, 1), (1, 37), (29, 1), (max(k - 1, 1), max(k - 1, 1)), (k, k), (k + 1, k + 1), (k + 1, k + 6),
             (k + 5, max(k - 1, 1))}
    for h, w in sorted(sizes):
        check(emu, rng.integers(0, 256, (h, w, c), dtype=np.uint8), k)


@pytest.mark.parametrize('c', [1, 3, 4])
@pytest.mark.parametrize('k', [2, 3, 15])
def test_emu_blur_one_past_a_tile_and_a_strip(emu, k, c):
    """A row one pixel past a tile of row bytes (two CTAs side by side, the second holding one pixel) and a frame
    one row past a strip (a second row of CTAs whose vertical sums start k - 1 rows above its first row)."""
    rng = np.random.default_rng(k + c)
    w = TILE_BYTES // c + 1
    for h in (STRIP_ROWS + 1, k + 2):
        check(emu, rng.integers(0, 256, (h, w, c), dtype=np.uint8), k)
    check(emu, rng.integers(0, 256, (2 * STRIP_ROWS + 1, 40 // c + 3, c), dtype=np.uint8), k)


@pytest.mark.parametrize('c', [1, 3, 4])
@pytest.mark.parametrize('k', [3, 4, 5])
def test_emu_blur_unaligned_bases(emu, k, c):
    rng = np.random.default_rng(7 * k + c)
    for h, w in [(13, 37), (9, 64)]:
        x = rng.integers(0, 256, (h, w, c), dtype=np.uint8)
        ref = br.blur(x, k)
        for off in (1, 3):
            buf = np.zeros(x.size + 8, np.uint8)
            buf[off:off + x.size] = x.reshape(-1)
            rc, out = run(emu, [buf.ctypes.data + off], k, w, h, c)
            assert rc == 0 and np.array_equal(out[0], ref), (k, c, h, w, off)
            # the destination at an odd base as well, with an aligned and with an unaligned source
            for sp in (x.ctypes.data, buf.ctypes.data + off):
                obuf = np.full(x.size + 8, 0xA5, np.uint8)
                assert emu.stb_blur_u8(_lib.ptr_table([sp]), 1, w, h, c, k, _lib.ptr_table([obuf.ctypes.data + off]), None) == 0
                assert np.array_equal(obuf[off:off + x.size], ref.reshape(-1)), (k, c, h, w, off, sp)
                assert (obuf[:off] == 0xA5).all() and (obuf[off + x.size:] == 0xA5).all()


def test_emu_blur_batch_past_one_pointer_table(emu):
    """67 frames: two launches (64 + 3 frames); every frame equals its single-frame call."""
    n, h, w, c, k = 67, 6, 7, 3, 3
    rng = np.random.default_rng(5)
    xs = [rng.integers(0, 256, (h, w, c), dtype=np.uint8) for _ in range(n)]
    rc, out = run(emu, xs, k, w, h, c)
    assert rc == 0
    for i, x in enumerate(xs):
        assert np.array_equal(out[i], run(emu, [x], k, w, h, c)[1][0]), i
        assert np.array_equal(out[i], br.blur(x, k)), i


@pytest.mark.parametrize('side', ['src', 'dst'])
def test_emu_blur_null_entry_at_65_leaves_every_output_untouched(emu, side):
    n, h, w, c, bad = 67, 4, 8, 3, 65
    src = np.random.default_rng(3).integers(0, 256, (n, h, w, c), dtype=np.uint8)
    out = np.full((n, h, w, c), 0xA5, np.uint8)
    st = _lib.ptr_table([0 if side == 'src' and i == bad else src[i].ctypes.data for i in range(n)])
    dt = _lib.ptr_table([0 if side == 'dst' and i == bad else out[i].ctypes.data for i in range(n)])
    assert emu.stb_blur_u8(st, n, w, h, c, 3, dt, None) == -1
    assert b'%s frame 65 is NULL' % (b'source' if side == 'src' else b'destination') in emu.stb_last_error()
    assert (out == 0xA5).all()


def test_emu_blur_argument_checks_write_nothing(emu):
    h, w, c = 5, 6, 3
    x = np.random.default_rng(1).integers(0, 256, (h, w, c), dtype=np.uint8)
    for k, status in [(0, -1), (-1, -1), (256, -4), (1 << 20, -4)]:
        rc, out = run(emu, [x], k, w, h, c)
        assert rc == status, (k, rc)
        assert (out == 0xA5).all(), k
    for (n, ww, hh, cc) in [(-1, w, h, c), (1, 0, h, c), (1, w, -2, c), (1, w, h, 2), (1, w, h, 0), (1, w, h, 5)]:
        out = np.full((1, h, w, c), 0xA5, np.uint8)
        rc = emu.stb_blur_u8(_lib.ptr_table([x.ctypes.data]), n, ww, hh, cc, 3, _lib.ptr_table([out.ctypes.data]), None)
        assert rc == -1, (n, ww, hh, cc)
        assert (out == 0xA5).all()
    # n == 0 is a no-op, even without tables
    assert emu.stb_blur_u8(None, 0, w, h, c, 3, None, None) == 0
    assert emu.stb_blur_u8(None, 0, w, h, c, 0, None, None) == 0


def test_emu_blur_rejects_a_destination_overlapping_its_own_source(emu):
    h, w, c = 5, 6, 3
    nb = h * w * c
    buf = np.random.default_rng(2).integers(0, 256, 3 * nb, dtype=np.uint8)
    keep = buf.copy()
    base = buf.ctypes.data
    for d in (0, 5, nb - 1, -(nb - 1), -3):
        rc = emu.stb_blur_u8(_lib.ptr_table([base + nb]), 1, w, h, c, 3, _lib.ptr_table([base + nb + d]), None)
        assert rc == -1 and b'overlaps' in emu.stb_last_error(), d
        assert np.array_equal(buf, keep), d
    # adjacent, not overlapping: allowed
    x = buf[nb:2 * nb].reshape(h, w, c).copy()
    assert emu.stb_blur_u8(_lib.ptr_table([base + nb]), 1, w, h, c, 3, _lib.ptr_table([base + 2 * nb]), None) == 0
    assert np.array_equal(buf[2 * nb:].reshape(h, w, c), br.blur(x, 3))
    # frame i overlapping frame j != i is the caller's business and is not rejected
    a = np.full((2, h, w, c), 0xA5, np.uint8)
    assert emu.stb_blur_u8(_lib.ptr_table([x.ctypes.data, a[0].ctypes.data]), 2, w, h, c, 3,
                           _lib.ptr_table([a[0].ctypes.data, a[1].ctypes.data]), None) == 0
