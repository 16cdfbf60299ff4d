"""Kernel-LOGIC tests without a GPU: the product's .cu sources are compiled with g++ against
tests/cuda_emu (a CPU emulation of blocks/threads/shared memory/warp collectives) and checked
against the oracle.  This exercises indexing, halos, tiling and the host-side level schedule;
it says nothing about performance and is not a product path (see cuda_emu.h)."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from conftest import ROOT, epe
from oracle import restate
from scannertools_b200 import _lib, synth

sys.path.insert(0, os.path.join(ROOT, 'tests', 'cuda_emu'))


@pytest.fixture(scope='module')
def emu():
    import build_emu
    return _lib.bind(C.CDLL(build_emu.build()))


def P(a):
    return C.c_void_p(a.ctypes.data)


def test_emu_histogram_ragged_and_unaligned(emu):
    for (h, w) in [(37, 53), (1, 1), (64, 64)]:
        fr = synth.noise_clip(1, 2, h, w)
        out = np.full((2, 48), -1, np.int32)
        assert emu.stb_hist_rgb16(_lib.ptr_table([f.ctypes.data for f in fr]), 2, w, h, P(out), None) == 0
        ref = np.stack([restate.histogram(f).reshape(-1) for f in fr])
        assert np.array_equal(out, ref)
        buf = np.zeros(fr[0].size + 32, np.uint8)
        for off in (1, 7):
            buf[off:off + fr[0].size] = fr[0].reshape(-1)
            o1 = np.zeros(48, np.int32)
            assert emu.stb_hist_rgb16_strided(C.c_void_p(buf.ctypes.data + off), fr[0].size, 1, w, h, P(o1), None) == 0
            assert np.array_equal(o1, ref[0])
    assert emu.stb_hist_rgb16(None, 0, 4, 4, None, None) == 0          # empty batch is a no-op
    assert emu.stb_hist_rgb16(None, 2, 4, 4, None, None) != 0          # invalid args are rejected


def test_emu_shot_scores_with_halo(emu):
    h = np.random.default_rng(0).integers(0, 100000, size=(70, 48)).astype(np.int32)
    ref = restate.shot_scores(h)
    S = np.zeros(70, np.int32)
    assert emu.stb_shot_scores(P(h), 70, None, P(S), None) == 0
    assert np.array_equal(S, ref)
    S2 = np.zeros(69, np.int32)
    assert emu.stb_shot_scores(P(h[1:]), 69, P(h[0]), P(S2), None) == 0
    assert np.array_equal(S2, ref[1:])


def test_emu_flow_histogram_edge_values(emu):
    for (h, w) in [(17, 33), (60, 107)]:
        ff = synth.textured_flow_field(3, h, w)
        out = np.zeros(128, np.int32)
        assert emu.stb_flow_hist(_lib.ptr_table([ff.ctypes.data]), 1, w, h, P(out), None) == 0
        assert np.array_equal(out.reshape(2, 64), restate.flow_histogram(ff))


def test_emu_frame_difference(emu):
    a = synth.noise_clip(2, 2, 19, 23)
    o = np.zeros_like(a[0])
    assert emu.stb_frame_diff(P(a[0]), P(a[1]), P(o), o.size, None) == 0
    assert np.array_equal(o, restate.frame_difference(a[0], a[1]))


@pytest.mark.parametrize('h,w,pairs', [(120, 160, 1), (135, 240, 2), (67, 45, 1), (64, 128, 66)])
def test_emu_farneback_vs_oracle(emu, h, w, pairs):
    """66 pairs: two pointer-table chunks per level and two slices of pyramid / expansion launches (the
    two-launch pyramid at 128x64).  Every pair must equal its single-pair run bit for bit, flow and fused
    histogram."""
    clip = synth.textured_clip(3, pairs + 1, h, w)
    hd = C.c_void_p()
    assert emu.stb_farneback_create(w, h, pairs, None, C.byref(hd)) == 0
    ws, hs = (C.c_int * 8)(), (C.c_int * 8)()
    ns = emu.stb_farneback_levels(hd, ws, hs)
    assert [(ws[k], hs[k]) for k in range(ns)] == restate.pyramid_info(w, h)
    flows = [np.zeros((h, w, 2), np.float32) for _ in range(pairs)]
    rc = emu.stb_farneback_run(hd, _lib.ptr_table([f.ctypes.data for f in clip]), pairs,
                               _lib.ptr_table([f.ctypes.data for f in flows]), None)
    assert rc == 0, emu.stb_last_error()
    fh = np.zeros((pairs, 128), np.int32)
    assert emu.stb_farneback_run_hist(hd, _lib.ptr_table([f.ctypes.data for f in clip]), pairs, None, P(fh), None) == 0
    emu.stb_farneback_destroy(hd)
    assert emu.stb_farneback_create(w, h, 1, None, C.byref(hd)) == 0
    for i in range(pairs):
        f1, fh1 = np.zeros((h, w, 2), np.float32), np.zeros(128, np.int32)
        assert emu.stb_farneback_run_hist(hd, _lib.ptr_table([clip[i].ctypes.data, clip[i + 1].ctypes.data]), 1,
                                          _lib.ptr_table([f1.ctypes.data]), P(fh1), None) == 0
        assert np.array_equal(flows[i], f1) and np.array_equal(fh[i], fh1), i
    emu.stb_farneback_destroy(hd)
    for i in range(pairs):
        e = epe(flows[i], restate.optical_flow(clip[i], clip[i + 1]))
        # north_star tolerance: mean EPE <= 1e-3 px, max <= 1e-2 px
        assert e.mean() <= 1e-3 and e.max() <= 1e-2, (i, e.mean(), e.max())
        assert e.max() < 1e-4   # in practice float32 agreement is ~1e-5 px


def test_emu_farneback_pow2_pyramid_all_levels(emu):
    """320x256 runs 4 scales whose sizes are exact powers of two: covers the merged-tap
    pyramid kernels for K = 1, 2, 3 stage by stage (I_k against the restatement)."""
    h, w = 256, 320
    clip = synth.textured_clip(6, 2, h, w)
    hd = C.c_void_p()
    assert emu.stb_farneback_create(w, h, 1, None, C.byref(hd)) == 0
    out = np.zeros((h, w, 2), np.float32)
    g0, g1 = restate.gray(clip[0]), restate.gray(clip[1])
    for k in (3, 2, 1, 0):
        lw, lh = restate.pyramid_info(w, h)[k]
        I0 = np.zeros((lh, lw), np.float32)
        R1 = np.zeros((5, lh, lw), np.float32)
        emu.stb_farneback_debug_set(hd, k, 0, P(I0), None, None, P(R1), None, None)
        assert emu.stb_farneback_run(hd, _lib.ptr_table([f.ctypes.data for f in clip]), 1,
                                     _lib.ptr_table([out.ctypes.data]), None) == 0
        _, d = restate.farneback(g0, g1, dump_level=k)
        assert np.abs(I0 - d['I0']).max() < 2e-4, k
        assert np.abs(R1 - d['R1'].transpose(2, 0, 1)).max() < 1e-4, k
    emu.stb_farneback_destroy(hd)
    e = epe(out, restate.farneback(g0, g1))
    assert e.max() < 1e-4, e.max()


def test_emu_farneback_flat_regions_next_to_edges(emu):
    """Flat background + moving square: window sums that slide over a strong edge must not
    leave rounding residue in the flat area (the reason OpenCV sums in double; box15 only adds)."""
    h, w = 120, 160
    flat = np.full((2, h, w, 3), 90, np.uint8)
    flat[0, 50:80, 50:80] = 200
    flat[1, 52:82, 53:83] = 200
    hd = C.c_void_p()
    assert emu.stb_farneback_create(w, h, 1, None, C.byref(hd)) == 0
    out = np.zeros((h, w, 2), np.float32)
    assert emu.stb_farneback_run(hd, _lib.ptr_table([f.ctypes.data for f in flat]), 1,
                                 _lib.ptr_table([out.ctypes.data]), None) == 0
    emu.stb_farneback_destroy(hd)
    e = epe(out, restate.optical_flow(flat[0], flat[1]))
    assert e.mean() <= 1e-3 and e.max() <= 1e-2, (e.mean(), e.max())


def test_emu_farneback_generic_window(emu):
    """winSize != 15 takes the generic iteration kernel."""
    h, w = 96, 128
    clip = synth.textured_clip(8, 2, h, w)
    prm = _lib.FarnebackParams(3, 0.5, 0, 9, 2, 5, 1.2, 0)
    hd = C.c_void_p()
    assert emu.stb_farneback_create(w, h, 1, C.byref(prm), C.byref(hd)) == 0
    out = np.zeros((h, w, 2), np.float32)
    assert emu.stb_farneback_run(hd, _lib.ptr_table([f.ctypes.data for f in clip]), 1,
                                 _lib.ptr_table([out.ctypes.data]), None) == 0
    emu.stb_farneback_destroy(hd)
    ref = restate.farneback(restate.gray(clip[0]), restate.gray(clip[1]), winsize=9, iters=2)
    e = epe(out, ref)
    assert e.max() < 1e-4, e.max()
    bad = _lib.FarnebackParams(3, 0.5, 0, 8, 3, 5, 1.2, 0)     # even window: rejected
    assert emu.stb_farneback_create(w, h, 1, C.byref(bad), C.byref(hd)) != 0


def test_emu_resize_bit_exact(emu):
    rng = np.random.default_rng(1)
    for (sw, sh, dw, dh, cn) in [(213, 120, 107, 60, 3), (64, 48, 32, 24, 3), (64, 48, 200, 100, 3), (101, 77, 33, 20, 1), (40, 30, 40, 30, 4)]:
        img = rng.integers(0, 256, (sh, sw, cn), dtype=np.uint8)
        out = np.zeros((dh, dw, cn), np.uint8)
        assert emu.stb_resize_bilinear_u8(_lib.ptr_table([img.ctypes.data]), 1, sw, sh, cn, _lib.ptr_table([out.ctypes.data]), dw, dh, None) == 0
        assert np.array_equal(out, restate.resize(img, dw, dh)), (sw, sh, dw, dh, cn)
    # the other interpolation names of ResizeArgs: nearest, area (integer factors, general tables,
    # up-scaled / mixed axes), 1/3/4 channels, degenerate sizes
    codes = {n: emu.stb_resize_interp_code(n.encode()) for n in ('INTER_LINEAR', 'INTER_NEAREST', 'INTER_AREA', 'INTER_CUBIC', 'INTER_LANCZOS4')}
    assert codes == {'INTER_LINEAR': 0, 'INTER_NEAREST': 1, 'INTER_AREA': 2, 'INTER_CUBIC': 3, 'INTER_LANCZOS4': 4}
    assert emu.stb_resize_interp_code(b'') == 0 and emu.stb_resize_interp_code(b'INTER_MAX') == -1
    for (sh, sw, dh, dw) in [(108, 192, 24, 43), (90, 160, 37, 71), (72, 128, 24, 43), (60, 90, 20, 30), (64, 96, 16, 24),
                             (40, 60, 20, 30), (24, 43, 108, 192), (30, 40, 60, 20), (30, 40, 15, 80), (7, 5, 31, 33),
                             (33, 47, 1, 1), (1, 1, 5, 7)]:
        for cn in (1, 3, 4):
            img = rng.integers(0, 256, (sh, sw, cn), dtype=np.uint8)
            for name, code in codes.items():
                out = np.zeros((dh, dw, cn), np.uint8)
                assert emu.stb_resize_u8(_lib.ptr_table([img.ctypes.data]), 1, sw, sh, cn, _lib.ptr_table([out.ctypes.data]),
                                         dw, dh, code, None) == 0
                assert np.array_equal(out, restate.resize(img, dw, dh, name)), (sh, sw, dh, dw, cn, name)
    img = rng.integers(0, 256, (8, 8, 3), dtype=np.uint8)
    assert emu.stb_resize_u8(_lib.ptr_table([img.ctypes.data]), 1, 8, 8, 3, _lib.ptr_table([img.ctypes.data]), 4, 4, -1, None) != 0
    w, h = C.c_int(), C.c_int()
    # ResizeArgs semantics of resize_kernel.cpp:43-61
    assert emu.stb_resize_target(1920, 1080, 426, 0, 0, 1, C.byref(w), C.byref(h)) == 0 and (w.value, h.value) == (426, 239)
    assert emu.stb_resize_target(1920, 1080, 0, 240, 0, 1, C.byref(w), C.byref(h)) == 0 and (w.value, h.value) == (426, 240)
    assert emu.stb_resize_target(320, 240, 426, 240, 1, 0, C.byref(w), C.byref(h)) == 0 and (w.value, h.value) == (320, 240)
    assert emu.stb_resize_bilinear_u8(_lib.ptr_table([0]), 1, 4, 4, 2, _lib.ptr_table([0]), 2, 2, None) != 0   # 2 channels: unsupported


def test_emu_convert_color_bit_exact(emu, golden):
    g = golden('convert_color.npz')
    img = g['in']
    h, w = img.shape[:2]
    for name in ['COLOR_RGB2HSV', 'COLOR_BGR2HSV', 'COLOR_RGB2GRAY', 'COLOR_BGR2GRAY', 'COLOR_RGB2BGR']:
        code = emu.stb_color_code(name.encode())
        oc = emu.stb_color_out_channels(code)
        out = np.zeros((h, w, oc), np.uint8)
        assert emu.stb_convert_color_u8(_lib.ptr_table([img.ctypes.data]), 1, w, h, code, _lib.ptr_table([out.ctypes.data]), None) == 0
        assert np.array_equal(out.reshape(g[name].shape), g[name]), name
    assert emu.stb_color_code(b'COLOR_BGR2XYZ') == -1
    assert emu.stb_convert_color_u8(_lib.ptr_table([img.ctypes.data]), 1, w, h, 99, _lib.ptr_table([img.ctypes.data]), None) != 0


def test_emu_fused_hsv_histogram(emu, golden):
    """stb_hist_hsv16 == Histogram(ConvertToHSV(frame)) (old/histograms.py:32-36), incl. ragged pixel
    counts, unaligned frame bases, BGR input and saturated / grey pixels."""
    rng = np.random.default_rng(21)
    rgb, bgr = emu.stb_color_code(b'COLOR_RGB2HSV'), emu.stb_color_code(b'COLOR_BGR2HSV')
    g = golden('convert_color.npz')
    cases = [np.ascontiguousarray(g['in']), rng.integers(0, 256, (21, 33, 3), dtype=np.uint8),
             rng.integers(0, 256, (1, 5, 3), dtype=np.uint8), np.full((40, 64, 3), 255, np.uint8),
             np.repeat(rng.integers(0, 256, (32, 48, 1), dtype=np.uint8), 3, axis=2)]
    for img in cases:
        h, w = img.shape[:2]
        for code, src in ((rgb, img), (bgr, np.ascontiguousarray(img[..., ::-1]))):
            out = np.zeros((1, 48), np.int32)
            assert emu.stb_hist_hsv16(_lib.ptr_table([src.ctypes.data]), 1, w, h, code, P(out), None) == 0
            ref = restate.histogram(restate.rgb2hsv(img)).reshape(-1)
            assert np.array_equal(out[0], ref), (img.shape, code)
            assert out[0].sum() == 3 * w * h and not out[0, 12:16].any()
    # two frames carved out of one buffer at a 1-byte offset: the unaligned path, strided entry point
    fr = rng.integers(0, 256, (2, 17, 23, 3), dtype=np.uint8)
    buf = np.zeros(fr.size + 16, np.uint8)
    buf[1:1 + fr.size] = fr.reshape(-1)
    out = np.zeros((2, 48), np.int32)
    assert emu.stb_hist_hsv16_strided(C.c_void_p(buf.ctypes.data + 1), fr[0].size, 2, 23, 17, rgb, P(out), None) == 0
    for i in range(2):
        assert np.array_equal(out[i], restate.histogram(restate.rgb2hsv(fr[i])).reshape(-1))
    assert emu.stb_hist_hsv16(None, 0, 4, 4, rgb, None, None) == 0
    assert emu.stb_hist_hsv16(_lib.ptr_table([fr.ctypes.data]), 1, 23, 17, emu.stb_color_code(b'COLOR_RGB2GRAY'), P(out), None) != 0


@pytest.mark.parametrize('levels,iters,win,flags,ps,pn,sig', [
    (0, 1, 15, 0, 0.5, 5, 1.2), (1, 1, 15, 0, 0.5, 5, 1.2), (2, 4, 15, 0, 0.5, 5, 1.2), (3, 3, 5, 0, 0.5, 5, 1.2),
    (3, 3, 15, 256, 0.5, 5, 1.2), (2, 2, 9, 256, 0.5, 5, 1.2), (3, 3, 15, 0, 0.75, 5, 1.2), (3, 3, 15, 0, 0.5, 7, 1.5)])
def test_emu_farneback_parameter_combinations(emu, levels, iters, win, flags, ps, pn, sig):
    """stb_farneback_params other than the reference's defaults: fewer pyramid levels, a single
    iteration (only the last-iteration kernel runs), more iterations, another window, the
    Gaussian window (flags = cv::OPTFLOW_FARNEBACK_GAUSSIAN), another pyramid scale, polyN = 7."""
    h, w = 96, 128
    clip = synth.textured_clip(9, 2, h, w)
    prm = _lib.FarnebackParams(levels, ps, 0, win, iters, pn, sig, flags)
    hd = C.c_void_p()
    assert emu.stb_farneback_create(w, h, 1, C.byref(prm), C.byref(hd)) == 0
    out = np.zeros((h, w, 2), np.float32)
    assert emu.stb_farneback_run(hd, _lib.ptr_table([f.ctypes.data for f in clip]), 1,
                                 _lib.ptr_table([out.ctypes.data]), None) == 0
    emu.stb_farneback_destroy(hd)
    ref = restate.farneback(restate.gray(clip[0]), restate.gray(clip[1]), winsize=win, iters=iters, levels=levels, flags=flags,
                            pyr_scale=ps, poly_n=pn, poly_sigma=sig)
    e = epe(out, ref)
    assert e.max() < 1e-4, (levels, iters, win, flags, ps, pn, e.max())
    if flags == 0 and (levels, iters, win) == (0, 1, 15):
        for bad in (_lib.FarnebackParams(levels, 0.5, 0, win, iters, 5, 1.2, 4),     # OPTFLOW_USE_INITIAL_FLOW
                    _lib.FarnebackParams(levels, 0.3, 0, win, iters, 5, 1.2, 0),     # pyr_scale < 0.5
                    _lib.FarnebackParams(levels, 0.5, 0, win, iters, 9, 1.5, 0)):    # polyN > 7
            assert emu.stb_farneback_create(w, h, 1, C.byref(bad), C.byref(hd)) != 0


def test_emu_pipe_host_path(emu):
    h, w = 48, 64
    clip = synth.textured_clip(5, 6, h, w)
    p = C.c_void_p()
    assert emu.stb_pipe_create(w, h, 2, 1, C.byref(p)) == 0
    hist = np.zeros((6, 48), np.int32)
    S = np.zeros(6, np.int32)
    assert emu.stb_pipe_hist(p, P(clip), 6, P(hist), P(S)) == 0
    ref = np.stack([restate.histogram(f).reshape(-1) for f in clip])
    assert np.array_equal(hist, ref) and np.array_equal(S, restate.shot_scores(ref))
    flow = np.zeros((5, h, w, 2), np.float32)
    fh = np.zeros((5, 128), np.int32)
    assert emu.stb_pipe_flow(p, P(clip), 5, P(flow), P(fh)) == 0
    for i in range(5):
        e = epe(flow[i], restate.optical_flow(clip[i], clip[i + 1]))
        assert e.max() < 1e-4, (i, e.max())
        assert np.array_equal(fh[i].reshape(2, 64), restate.flow_histogram(flow[i]))
    fh_only = np.zeros((5, 128), np.int32)            # histogram-only: flow frames are never materialised
    assert emu.stb_pipe_flow(p, P(clip), 5, None, P(fh_only)) == 0
    assert np.array_equal(fh_only, fh)
    assert emu.stb_pipe_flow(p, P(clip), 5, None, None) != 0
    # asynchronous form: two calls in flight, tickets alternate
    r0, r1 = np.zeros((5, 128), np.int32), np.zeros((5, 128), np.int32)
    t0, t1 = C.c_int(-1), C.c_int(-1)
    assert emu.stb_pipe_flow_async(p, P(clip), 5, None, P(r0), C.byref(t0)) == 0
    assert emu.stb_pipe_flow_async(p, P(clip), 5, None, P(r1), C.byref(t1)) == 0
    assert {t0.value, t1.value} == {0, 1}
    assert emu.stb_pipe_wait(p, t0.value) == 0 and emu.stb_pipe_wait(p, t1.value) == 0
    assert np.array_equal(r0, fh) and np.array_equal(r1, fh)
    assert emu.stb_pipe_wait(p, 7) != 0
    emu.stb_pipe_destroy(p)


@pytest.mark.parametrize('h,w', [(60, 100), (97, 164), (46, 80)])
def test_emu_border_tiles_ragged_sizes_and_fused_histogram(emu, h, w):
    """Sizes where every tile of the TMA iteration kernels touches the image border and the right / bottom
    tiles are ragged; the fused histogram must equal FlowHistogram of the flow the same call returns,
    with and without materialising the flow; the two-launch pyramid is off (w % 32 != 0) or on."""
    clip = synth.textured_clip(14, 3, h, w)
    hd = C.c_void_p()
    assert emu.stb_farneback_create(w, h, 2, None, C.byref(hd)) == 0
    flows = [np.zeros((h, w, 2), np.float32) for _ in range(2)]
    fh = np.zeros((2, 128), np.int32)
    ft = _lib.ptr_table([f.ctypes.data for f in clip])
    assert emu.stb_farneback_run_hist(hd, ft, 2, _lib.ptr_table([f.ctypes.data for f in flows]), P(fh), None) == 0, emu.stb_last_error()
    fh_only = np.zeros((2, 128), np.int32)
    assert emu.stb_farneback_run_hist(hd, ft, 2, None, P(fh_only), None) == 0
    plain = [np.zeros((h, w, 2), np.float32) for _ in range(2)]
    assert emu.stb_farneback_run(hd, ft, 2, _lib.ptr_table([f.ctypes.data for f in plain]), None) == 0
    emu.stb_farneback_destroy(hd)
    for i in range(2):
        e = epe(flows[i], restate.optical_flow(clip[i], clip[i + 1]))
        assert e.max() < 1e-4, (i, e.max())
        assert np.array_equal(fh[i].reshape(2, 64), restate.flow_histogram(flows[i])), i
        assert np.array_equal(plain[i], flows[i])
    assert np.array_equal(fh_only, fh)


@pytest.mark.parametrize('h,w,gen', [(120, 160, 'textured'), (97, 164, 'warped'), (76, 112, 'noise')])
def test_emu_flow_compensated_window_equals_global_gathers(emu, h, w, gen):
    """iter15_win_kernel stages the displaced R1 footprints of a tile in shared memory when their bounding box
    fits (smooth motion) and falls back to global gathers per tile when it does not (noise: incoherent flow);
    either way the flow must equal the plain iter15_tma_kernel path (STB_NO_WIN) bit for bit."""
    clip = {'textured': lambda: synth.textured_clip(5, 3, h, w), 'warped': lambda: synth.warped_clip(6, 3, h, w),
            'noise': lambda: synth.noise_clip(7, 3, h, w)}[gen]()
    ft = _lib.ptr_table([f.ctypes.data for f in clip])
    res = []
    for no_win in (False, True):
        if no_win:
            os.environ['STB_NO_WIN'] = '1'
        try:
            hd = C.c_void_p()
            assert emu.stb_farneback_create(w, h, 2, None, C.byref(hd)) == 0
        finally:
            os.environ.pop('STB_NO_WIN', None)
        flows = [np.zeros((h, w, 2), np.float32) for _ in range(2)]
        assert emu.stb_farneback_run(hd, ft, 2, _lib.ptr_table([f.ctypes.data for f in flows]), None) == 0, emu.stb_last_error()
        emu.stb_farneback_destroy(hd)
        res.append(flows)
    for i in range(2):
        assert np.array_equal(res[0][i], res[1][i]), i


@pytest.mark.parametrize('op,side', [('convert_color', 'src'), ('convert_color', 'dst'), ('resize_linear', 'src'),
                                     ('resize_linear', 'dst'), ('resize_cubic', 'src'), ('resize_cubic', 'dst'),
                                     ('hist_rgb16', 'src'), ('hist_hsv16', 'src'), ('flow_hist', 'src')])
def test_emu_null_entry_past_first_pointer_table_is_rejected_before_any_launch(emu, op, side):
    """A NULL entry at index 65 of a 67-frame batch (in the second 64-entry pointer table) is rejected with
    STB_ERR_INVALID before anything is enqueued: no output of the batch is written, not even the first chunk's."""
    n, h, w, bad = 67, 4, 8, 65
    rng = np.random.default_rng(17)
    if op == 'flow_hist':
        src = rng.standard_normal((n, h, w, 2)).astype(np.float32)
    else:
        src = rng.integers(0, 256, (n, h, w, 3), dtype=np.uint8)
    if op.startswith('hist') or op == 'flow_hist':
        out = np.full((n, 128 if op == 'flow_hist' else 48), -7, np.int32)
    else:
        out = np.full((n, 3, 5, 3) if op.startswith('resize') else (n, h, w, 3), 0xA5, np.uint8)
    srcs = [0 if side == 'src' and i == bad else src[i].ctypes.data for i in range(n)]
    dsts = [0 if side == 'dst' and i == bad else out[i].ctypes.data for i in range(n)]
    st, dt = _lib.ptr_table(srcs), _lib.ptr_table(dsts)
    rgb2hsv = emu.stb_color_code(b'COLOR_RGB2HSV')
    if op == 'convert_color':
        rc = emu.stb_convert_color_u8(st, n, w, h, rgb2hsv, dt, None)
    elif op.startswith('resize'):
        interp = emu.stb_resize_interp_code(b'INTER_CUBIC' if op == 'resize_cubic' else b'INTER_LINEAR')
        rc = emu.stb_resize_u8(st, n, w, h, 3, dt, 5, 3, interp, None)
    elif op == 'hist_rgb16':
        rc = emu.stb_hist_rgb16(st, n, w, h, P(out), None)
    elif op == 'hist_hsv16':
        rc = emu.stb_hist_hsv16(st, n, w, h, rgb2hsv, P(out), None)
    else:
        rc = emu.stb_flow_hist(st, n, w, h, P(out), None)
    assert rc == -1 and b'NULL' in emu.stb_last_error(), (rc, emu.stb_last_error())
    assert (out == (-7 if out.dtype == np.int32 else 0xA5)).all()


def test_emu_flow_histogram_fast_binning_randomised(emu):
    """flow_bins_fast (approximate location + exact path inside the guard bands, magic-number rint / floor, trash
    rows for dropped values) against the restatement on a field that mixes generic vectors, magnitudes on and next
    to integers, directions on and next to the 64 angle-bin edges, tiny, huge and non-finite values."""
    h, w = 192, 256
    ff = synth.edge_flow_field(11, h, w)
    out = np.zeros(128, np.int32)
    assert emu.stb_flow_hist(_lib.ptr_table([ff.ctypes.data]), 1, w, h, P(out), None) == 0
    assert np.array_equal(out.reshape(2, 64), restate.flow_histogram(ff))
