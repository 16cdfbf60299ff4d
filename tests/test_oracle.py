"""Pins the oracle (test infrastructure) before it is trusted:
  * the plain-C restatement (oracle/restate.c) against the committed goldens, which were
    produced by OpenCV itself through cv2 (tests/golden/make_golden.py);
  * when cv2 is importable, cv2 live against the same goldens (guards against a cv2 version
    drift between the container that made the fixtures and the box that replays them)."""
import numpy as np
import pytest

from conftest import epe
from oracle import restate

FLOW_CASES = ['160x120', '240x135', '344x260']


def test_restate_gray(golden):
    g = golden('flow_small.npz')
    for c in FLOW_CASES:
        assert np.array_equal(restate.gray(g['f0_' + c]), g['gray0_' + c])


def test_restate_histogram(golden):
    g = golden('hist_small.npz')
    names = [k[3:] for k in g.files if k.startswith('in_')]
    assert len(names) >= 5
    for nme in names:
        assert np.array_equal(restate.histogram(g['in_' + nme]), g['out_' + nme]), nme


def test_restate_shot_c1(golden):
    g = golden('shot_c1.npz')
    assert np.array_equal(restate.histogram(g['frame0']).reshape(-1), g['hists'][0].reshape(-1))
    c0 = int(g['cuts'][0])
    assert np.array_equal(restate.histogram(g['frame_first_cut']).reshape(-1), g['hists'][c0].reshape(-1))
    assert np.array_equal(restate.shot_scores(g['hists']), g['scores'])
    assert list(g['boundaries']) == list(g['cuts']) and len(g['cuts']) == 7


def test_restate_farneback(golden):
    g = golden('flow_small.npz')
    for c in FLOW_CASES:
        fl = restate.optical_flow(g['f0_' + c], g['f1_' + c])
        e = epe(fl, g['flow_' + c])
        assert e.mean() < 1e-5 and e.max() < 1e-4, (c, e.mean(), e.max())


@pytest.mark.parametrize('win,iters,levels,flags,ps,pn,sig', [(15, 3, 3, 256, 0.5, 5, 1.2), (9, 2, 2, 256, 0.5, 5, 1.2), (21, 3, 3, 0, 0.5, 5, 1.2),
                                                              (15, 3, 3, 0, 0.75, 5, 1.2), (15, 3, 3, 0, 0.5, 7, 1.5), (15, 3, 3, 0, 0.5, 3, 1.0)])
def test_restate_farneback_other_parameters_vs_cv2(win, iters, levels, flags, ps, pn, sig):
    """Window sizes / iteration counts / the Gaussian window (OPTFLOW_FARNEBACK_GAUSSIAN) of the
    restatement, checked against cv2 itself (these are not used by the reference, so no golden)."""
    cv2_ops = pytest.importorskip('oracle.cv2_ops')
    from scannertools_b200 import synth
    clip = synth.textured_clip(1, 2, 120, 160)
    ref = cv2_ops.optical_flow_params(clip[0], clip[1], num_levels=levels, win_size=win, num_iters=iters, flags=flags, pyr_scale=ps,
                                      poly_n=pn, poly_sigma=sig)
    fl = restate.farneback(restate.gray(clip[0]), restate.gray(clip[1]), winsize=win, iters=iters, levels=levels, flags=flags,
                           pyr_scale=ps, poly_n=pn, poly_sigma=sig)
    e = epe(fl, ref)
    assert e.mean() < 1e-5 and e.max() < 1e-4, (win, iters, levels, flags, ps, pn, e.mean(), e.max())


def test_restate_pyramid_geometry():
    # SURVEY Appendix A.1: round-half-even level sizes, up to 4 scales
    assert restate.pyramid_info(640, 480) == [(640, 480), (320, 240), (160, 120), (80, 60)]
    assert restate.pyramid_info(1920, 1080) == [(1920, 1080), (960, 540), (480, 270), (240, 135)]
    assert restate.pyramid_info(426, 240) == [(426, 240), (213, 120), (106, 60)]
    assert restate.pyramid_info(344, 260)[-1] == (43, 32)


def test_restate_flow_histogram(golden):
    g = golden('flowhist.npz')
    names = [k[3:] for k in g.files if k.startswith('in_')]
    for nme in names:
        assert np.array_equal(restate.flow_histogram(g['in_' + nme]), g['out_' + nme]), nme
    mag, deg = restate.polar(g['in_stress_33x17'])
    assert np.array_equal(mag, g['mag_stress_33x17'])
    assert np.array_equal(deg, g['deg_stress_33x17'])


def test_restate_frame_difference(golden):
    g = golden('framediff.npz')
    assert np.array_equal(restate.frame_difference(g['prev'], g['cur']), g['out'])


def test_shot_boundaries_against_the_reference_itself(golden, have_cv2):
    """tests/golden/shot_reference.npz was produced by the reference's OWN Python op
    (scannertools/shot_detection.py imported behind a scannerpy stub, tests/golden/ref_import.py): the
    oracle's restatement and the product's host logic must reproduce it exactly."""
    from scannertools_b200 import shot_detection, types
    g = golden('shot_reference.npz')
    names = [k[5:] for k in g.files if k.startswith('hist_')]
    assert len(names) == 7
    for nme in names:
        h, want = g['hist_' + nme], list(g['bounds_' + nme])
        elems = [types.histograms(types.histogram_bytes(x)) for x in h]
        assert shot_detection.shot_boundaries(None, elems)[0] == want, nme                 # product host logic
        assert shot_detection.shot_boundaries(None, scores=restate.shot_scores(h))[0] == want, nme   # via C scores
        if have_cv2:
            from oracle import cv2_ops
            assert cv2_ops.shot_boundaries(list(h)) == want, nme                           # oracle restatement


def test_restate_resize(golden):
    g = golden('resize.npz')
    names = [k[3:] for k in g.files if k.startswith('in_')]
    assert len(names) == 4
    for nme in names:
        out = g['out_' + nme]
        assert np.array_equal(restate.resize(g['in_' + nme], out.shape[1], out.shape[0]), out), nme


def test_restate_rgb2hsv(golden):
    g = golden('convert_color.npz')
    assert np.array_equal(restate.rgb2hsv(g['in']), g['COLOR_RGB2HSV'])
    assert np.array_equal(restate.rgb2hsv(g['in'][..., ::-1]), g['COLOR_BGR2HSV'])
    assert np.array_equal(restate.gray(g['in']), g['COLOR_BGR2GRAY'])
    # exhaustive-ish sweep against cv2 when available is in test_cv2_matches_goldens


def test_cv2_matches_goldens(golden, have_cv2):
    if not have_cv2:
        pytest.skip('cv2 not importable')
    from oracle import cv2_ops
    g = golden('flow_small.npz')
    for c in FLOW_CASES[:2]:
        e = epe(cv2_ops.optical_flow(g['f0_' + c], g['f1_' + c]), g['flow_' + c])
        assert e.max() < 1e-4, (c, e.max())
    gh = golden('hist_small.npz')
    assert np.array_equal(cv2_ops.histogram(gh['in_noise_37x53']), gh['out_noise_37x53'])
    gf = golden('flowhist.npz')
    assert np.array_equal(cv2_ops.flow_histogram(gf['in_stress_213x120']), gf['out_stress_213x120'])
    gc = golden('convert_color.npz')
    assert np.array_equal(cv2_ops.convert_color(gc['in'], 'COLOR_RGB2HSV'), gc['COLOR_RGB2HSV'])
    vals = np.arange(0, 256, 5, dtype=np.uint8)
    grid = np.stack(np.meshgrid(vals, vals, vals, indexing='ij'), -1).reshape(-1, 1, 3)
    assert np.array_equal(cv2_ops.convert_color(grid, 'COLOR_RGB2HSV'), restate.rgb2hsv(grid))
    gr = golden('resize.npz')
    assert np.array_equal(cv2_ops.resize(gr['in_up'], 200, 100), gr['out_up'])
    gs = golden('shot_c1.npz')
    assert cv2_ops.shot_boundaries(list(gs['hists'].reshape(-1, 3, 16))) == list(gs['boundaries'])


def test_restate_resize_interpolations_vs_cv2():
    """INTER_NEAREST / INTER_AREA / INTER_LINEAR of the restatement against cv2 itself on the shapes
    that reach every OpenCV branch: integer and fractional factors, 2x2, up-scaling, mixed axes,
    degenerate 1-pixel sizes; 1, 3 and 4 channels."""
    cv2 = pytest.importorskip('cv2')
    rng = np.random.default_rng(3)
    for (sh, sw, dh, dw) in [(108, 192, 24, 43), (90, 160, 37, 71), (54, 96, 50, 90), (72, 128, 24, 43), (60, 90, 20, 30),
                             (64, 96, 16, 24), (40, 60, 20, 30), (24, 43, 108, 192), (37, 71, 90, 160), (30, 40, 60, 20),
                             (30, 40, 15, 80), (270, 480, 240, 426), (7, 5, 31, 33), (50, 50, 50, 50), (33, 47, 1, 1), (1, 1, 5, 7)]:
        for cn in (1, 3, 4):
            src = rng.integers(0, 256, (sh, sw, cn), dtype=np.uint8)
            src = src[..., 0] if cn == 1 else src
            for name in ('INTER_NEAREST', 'INTER_AREA', 'INTER_LINEAR'):
                ref = cv2.resize(src, (dw, dh), interpolation=getattr(cv2, name))
                assert np.array_equal(restate.resize(src, dw, dh, name), ref), (sh, sw, dh, dw, cn, name)


def test_restate_resize_cubic_lanczos_vs_cv2():
    """INTER_CUBIC / INTER_LANCZOS4 of the restatement against OpenCV's own implementation
    (cv2.ipp.setUseIPP(False)): bit-exact, including the float vector path / integer tail split of the
    cubic vertical pass (rows whose W * cn is not a multiple of 8).  With IPP dispatch on (this wheel's
    default) 8-bit cubic comes from IPP and may differ from OpenCV's own code by one grey level; Lanczos4
    has no IPP path."""
    cv2 = pytest.importorskip('cv2')
    rng = np.random.default_rng(4)
    ipp0 = cv2.ipp.useIPP()
    try:
        for (sh, sw, dh, dw) in [(48, 64, 30, 41), (37, 53, 80, 111), (120, 160, 60, 80), (270, 480, 240, 426), (33, 47, 70, 21),
                                 (24, 43, 108, 192), (7, 5, 31, 33), (50, 50, 50, 50), (33, 47, 1, 1), (1, 1, 5, 7), (3, 2, 9, 10)]:
            for cn in (1, 3, 4):
                src = rng.integers(0, 256, (sh, sw, cn), dtype=np.uint8)
                src = src[..., 0] if cn == 1 else src
                for name in ('INTER_CUBIC', 'INTER_LANCZOS4'):
                    mine = restate.resize(src, dw, dh, name)
                    cv2.ipp.setUseIPP(False)
                    ref = cv2.resize(src, (dw, dh), interpolation=getattr(cv2, name))
                    assert np.array_equal(mine.reshape(ref.shape), ref), (sh, sw, dh, dw, cn, name)
                    cv2.ipp.setUseIPP(True)
                    ref_ipp = cv2.resize(src, (dw, dh), interpolation=getattr(cv2, name))
                    assert np.abs(mine.reshape(ref.shape).astype(int) - ref_ipp.astype(int)).max() <= 1, (sh, sw, dh, dw, cn, name)
    finally:
        cv2.ipp.setUseIPP(ipp0)


def test_restate_resize_cubic_lanczos_goldens(golden):
    g = golden('resize_taps.npz')
    for nme in [k[3:] for k in g.files if k.startswith('in_')]:
        for interp in ('INTER_CUBIC', 'INTER_LANCZOS4'):
            ref = g['out_%s_%s' % (interp, nme)]
            assert np.array_equal(restate.resize(g['in_' + nme], ref.shape[1], ref.shape[0], interp), ref), (interp, nme)


def test_cv2_fast_pyramids_is_a_no_op_on_cpu():
    """stb_farneback_params.fast_pyramids is accepted and ignored: OpenCV's CPU Farneback (the
    parity target) gives bit-identical flow with fastPyramids true or false."""
    cv2 = pytest.importorskip('cv2')
    from scannertools_b200 import synth
    clip = synth.textured_clip(1, 2, 120, 160)
    g = [cv2.cvtColor(f, cv2.COLOR_BGR2GRAY) for f in clip]
    a = cv2.FarnebackOpticalFlow_create(3, 0.5, False, 15, 3, 5, 1.2, 0).calc(g[0], g[1], None)
    b = cv2.FarnebackOpticalFlow_create(3, 0.5, True, 15, 3, 5, 1.2, 0).calc(g[0], g[1], None)
    assert np.array_equal(a, b)
