"""Parity tests proper: the CUDA path, called through the C ABI (via the ctypes wrappers in
scannertools_b200.ops), against the oracle on identical seeded inputs.

Tolerances (BASELINE.json north_star): histogram counts, scores and boundary indices bit-exact;
Farneback flow mean EPE <= 1e-3 px and max EPE <= 1e-2 px; flow histograms bit-exact on identical
flow, and per bin within the numeric bound of FLOWHIST_BIN_BOUND (see check_flow_hist_from_flow) when computed from
the GPU flow (the measured table is printed in the pytest summary).
Nothing here reads /root/reference."""
import os

import numpy as np
import pytest

from conftest import epe
from oracle import restate
from scannertools_b200 import synth

pytestmark = pytest.mark.gpu

try:
    from oracle import cv2_ops as cvo
except Exception:  # cv2 missing on the box: fall back to the pinned restatement
    cvo = None


def o_hist(f):
    return (cvo or restate).histogram(f)


def o_flow(f0, f1):
    return (cvo or restate).optical_flow(f0, f1)


def o_flow_hist(f):
    return (cvo or restate).flow_histogram(f)


@pytest.fixture(scope='module')
def torch():
    import torch
    assert torch.cuda.is_available(), 'gpu tests need a CUDA device'
    return torch


@pytest.fixture(scope='module')
def ops(torch):
    from scannertools_b200 import ops
    return ops


def dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


# ------------------------------------------------------------------ Histogram / shot scoring
def test_histogram_goldens(torch, ops, golden):
    g = golden('hist_small.npz')
    for nme in [k[3:] for k in g.files if k.startswith('in_')]:
        out = ops.histogram(dev(torch, g['in_' + nme])).cpu().numpy()
        assert np.array_equal(out[0], g['out_' + nme]), nme


@pytest.mark.parametrize('h,w', [(360, 640), (240, 426), (1080, 1920), (2160, 3840), (37, 53)])
def test_histogram_bit_exact(torch, ops, h, w):
    n = 3 if h * w > 10 ** 6 else 9
    fr = synth.noise_clip(7, n, h, w)
    fr[1] = 0           # constant frames: worst case for a shared table
    fr[2] = 255
    out = ops.histogram(dev(torch, fr)).cpu().numpy()
    ref = np.stack([np.stack([np.bincount(f[..., c].reshape(-1) >> 4, minlength=16) for c in range(3)]) for f in fr])
    assert np.array_equal(out, ref.astype(np.int32))
    assert np.array_equal(out[0], o_hist(fr[0]))
    assert (out.sum(axis=2) == h * w).all()


def test_histogram_separate_and_unaligned_buffers(torch, ops):
    h, w = 120, 213    # 3*w = 639 bytes per row: nothing is 4- or 16-byte aligned
    fr = synth.noise_clip(3, 5, h, w)
    big = torch.zeros(5 * (h * w * 3 + 64), dtype=torch.uint8, device='cuda')
    views = []
    for i in range(5):
        off = i * (h * w * 3 + 64) + (1, 3, 8, 15, 0)[i]
        v = big[off:off + h * w * 3].view(h, w, 3)
        v.copy_(dev(torch, fr[i]))
        views.append(v)
    out = ops.histogram(views).cpu().numpy()
    for i in range(5):
        assert np.array_equal(out[i], o_hist(fr[i])), i


def test_histogram_large_batch_chunks(torch, ops):
    fr = synth.noise_clip(11, 150, 36, 64)    # > 64 frames: several pointer-table launches
    out = ops.histogram([dev(torch, f) for f in fr]).cpu().numpy()
    ref = np.stack([restate.histogram(f) for f in fr])
    assert np.array_equal(out, ref)
    assert ops.histogram(torch.zeros((0, 4, 4, 3), dtype=torch.uint8, device='cuda')).shape == (0, 3, 16)


def test_shot_detection_c1_end_to_end(torch, ops, golden):
    """BASELINE configs[0]: 1000 frames 640x360, 16 bins/channel; 7 planted cuts
    (mirrors scannertools/tests/test_all.py:222-233)."""
    from scannertools_b200 import shot_detection
    g = golden('shot_c1.npz')
    clip, cuts = synth.cut_clip(5, 1000, 360, 640, n_cuts=7)
    d = dev(torch, clip)
    hist = ops.histogram(d)
    S = ops.shot_scores(hist)
    hist_h, S_h = hist.cpu().numpy(), S.cpu().numpy()
    assert np.array_equal(hist_h[0], o_hist(clip[0]))
    if np.array_equal(clip[0], g['frame0']):            # same generator output as when goldens were made
        assert np.array_equal(hist_h.reshape(1000, 48), g['hists'].reshape(1000, 48))
        assert np.array_equal(S_h, g['scores'])
    assert np.array_equal(S_h, restate.shot_scores(hist_h))
    rows = shot_detection.shot_boundaries(None, scores=S_h)
    assert rows[0] == cuts and len(rows[0]) == 7 and all(r is None for r in rows[1:])
    # frame-range shards with a one-histogram halo give the same scores
    S2 = ops.shot_scores(hist[500:], prev_hist=hist[499]).cpu().numpy()
    assert np.array_equal(S2, S_h[500:])


def test_pipeline_runners(torch, ops):
    """The shipped pipelines composed from the ops (scannertools/old/histograms.py, old/optical_flow.py,
    shot_detection.py): host frames in, chunked, results independent of the chunking."""
    from scannertools_b200 import pipelines
    clip, cuts = synth.cut_clip(5, 200, 90, 160, n_cuts=3)          # host numpy frames
    ref = np.stack([o_hist(f) for f in clip])
    assert np.array_equal(pipelines.compute_histograms(clip, batch=37), ref)
    assert np.array_equal(pipelines.compute_histograms(dev(torch, clip), batch=64), ref)
    hsv_ref = np.stack([o_hist(cvo.convert_color(f, 'COLOR_RGB2HSV') if cvo else restate.rgb2hsv(f)) for f in clip[:20]])
    assert np.array_equal(pipelines.compute_hsv_histograms(clip[:20], batch=7), hsv_ref)
    assert pipelines.detect_shots(clip, batch=33) == cuts == pipelines.detect_shots(dev(torch, clip), batch=200)
    # Resize(426x240) -> OpticalFlow -> FlowHistogram (old/histograms.py:63-79) on 7 frames of 540p
    mov = synth.textured_clip(3, 7, 540, 960)
    fh = pipelines.compute_flow_histograms(mov, batch=4)
    assert fh.shape == (6, 2, 64) and fh.dtype == np.int32
    small = ops.resize(dev(torch, mov), width=426, height=240)
    for i in range(7):
        assert np.array_equal(small[i].cpu().numpy(), (cvo or restate).resize(mov[i], 426, 240))
    of = ops.OpticalFlow(426, 240, max_batch=6)
    flow = of.execute(small)
    of.close()
    assert np.array_equal(fh, ops.flow_histogram(flow).cpu().numpy())      # chunked + fused == one batch + stand-alone op
    for i in (0, 5):
        ref_flow = o_flow(small[i].cpu().numpy(), small[i + 1].cpu().numpy())
        check_flow(flow[i].cpu().numpy(), ref_flow, ('pipeline', i))
    got = [(a, f.clone()) for a, f in pipelines.compute_flow(small, batch=4)]
    assert [a for a, _ in got] == [0, 4] and [f.shape[0] for _, f in got] == [4, 2]
    assert torch.equal(torch.cat([f for _, f in got]), flow)
    assert pipelines.compute_flow_histograms(mov[:1]).shape == (0, 2, 64) and pipelines.detect_shots(clip[:0]) == []


def test_host_pipe_histogram(torch, ops):
    clip, cuts = synth.cut_clip(9, 70, 90, 160, n_cuts=3)
    pipe = ops.Pipe(160, 90, max_batch=16)
    pinned = torch.from_numpy(clip).pin_memory()
    hist, S = pipe.histogram(pinned)
    ref = np.stack([restate.histogram(f) for f in clip])
    assert np.array_equal(hist, ref)
    assert np.array_equal(S, restate.shot_scores(ref))
    pipe.close()


# ------------------------------------------------------------------ FlowHistogram / FrameDifference
def test_flow_histogram_goldens_bit_exact(torch, ops, golden):
    g = golden('flowhist.npz')
    for nme in [k[3:] for k in g.files if k.startswith('in_')]:
        out = ops.flow_histogram(dev(torch, g['in_' + nme])).cpu().numpy()
        assert np.array_equal(out[0], g['out_' + nme]), nme


def test_flow_histogram_1080p_and_drops(torch, ops):
    f = synth.textured_flow_field(5, 1080, 1920)
    out = ops.flow_histogram(dev(torch, f)).cpu().numpy()[0]
    assert np.array_equal(out, o_flow_hist(f))
    assert out[0].sum() < 1080 * 1920 and out[1].sum() < 1080 * 1920   # >=64 px and ==360 deg are dropped


def test_flow_histogram_values_hugging_bin_edges(torch, ops):
    """The production kernel locates bins with approximate arithmetic and falls back to the
    exact IEEE path inside a guard band around every edge: fields whose magnitudes / angles sit
    within 0 .. 1e-2 of the edges (both sides) must still be bit-exact."""
    rng = np.random.default_rng(42)
    n = 1 << 18
    k = rng.integers(0, 66, n).astype(np.float64)
    dm = rng.choice([0, 1e-7, -1e-7, 1e-6, -1e-6, 1e-5, -1e-5, 1e-4, -1e-4, 3e-4, -3e-4, 1e-3, -1e-3, 1e-2, -1e-2], n)
    r = np.maximum(k + dm * np.maximum(k, 1.0), 0.0)
    e = rng.integers(0, 65, n).astype(np.float64) * (360.0 / 64.0)
    da = rng.choice([0, 1e-6, -1e-6, 1e-5, -1e-5, 1e-4, -1e-4, 5e-4, -5e-4, 2e-3, -2e-3, 1e-2, -1e-2, 0.1, -0.1], n)
    th = np.radians(e + da)
    f = np.stack([r * np.cos(th), r * np.sin(th)], axis=-1).astype(np.float32).reshape(512, 512, 2)
    # (NaN is left out: OpenCV's SIMD min/max make its NaN result unspecified)
    f[0, :8] = [[0, 0], [np.inf, 1], [1e15, -1e15], [1e-30, 1e-30], [1e20, 1e20], [-0.0, 0.0], [1, -1e-8], [64, 0]]
    out = ops.flow_histogram(dev(torch, f)).cpu().numpy()[0]
    assert np.array_equal(out, o_flow_hist(f))
    assert np.array_equal(out, restate.flow_histogram(f))


def test_frame_difference(torch, ops, golden):
    g = golden('framediff.npz')
    out = ops.frame_difference(dev(torch, g['prev']), dev(torch, g['cur'])).cpu().numpy()
    assert np.array_equal(out, g['out'])
    a = synth.noise_clip(4, 2, 1080, 1920)
    out = ops.frame_difference(dev(torch, a[0]), dev(torch, a[1])).cpu().numpy()
    assert np.array_equal(out, (a[1].astype(np.int16) - a[0].astype(np.int16)).astype(np.uint8))


# ------------------------------------------------------------------ Resize (next row, 8f rank 1)
def test_resize_goldens_and_pipeline_size(torch, ops, golden):
    g = golden('resize.npz')
    for nme in [k[3:] for k in g.files if k.startswith('in_')]:
        src, ref = g['in_' + nme], g['out_' + nme]
        if src.ndim == 2:
            src, ref = src[..., None], ref[..., None]
        out = ops.resize(dev(torch, src), width=ref.shape[1], height=ref.shape[0]).cpu().numpy()[0]
        assert np.array_equal(out, ref), nme
    # the shipped flow-histogram pipeline: Resize(426x240) -> OpticalFlow (old/histograms.py:64-68)
    fr = synth.noise_clip(9, 3, 1080, 1920)
    out = ops.resize(dev(torch, fr), width=426, height=240).cpu().numpy()
    for i in range(3):
        assert np.array_equal(out[i], (cvo or restate).resize(fr[i], 426, 240)), i
    assert ops.resize_target(1920, 1080, width=426, preserve_aspect=True) == (426, 239)
    # the other interpolation names: nearest, area (1080p -> 426x240 general tables, -> 480x270 integer
    # factor 4, -> 960x540 the 2x2 path, up-scaling and mixed axes)
    for name in ('INTER_NEAREST', 'INTER_AREA'):
        for (tw, th) in [(426, 240), (480, 270), (960, 540)]:
            out = ops.resize(dev(torch, fr[:2]), width=tw, height=th, interpolation=name).cpu().numpy()
            for i in range(2):
                assert np.array_equal(out[i], (cvo or restate).resize(fr[i], tw, th, name)), (name, tw, th, i)
    small = np.ascontiguousarray(fr[0, :97, :131])
    for name in ('INTER_NEAREST', 'INTER_AREA', 'INTER_LINEAR'):
        for (tw, th) in [(300, 200), (64, 200), (300, 31), (131, 97), (1, 1)]:
            out = ops.resize(dev(torch, small), width=tw, height=th, interpolation=name).cpu().numpy()[0]
            assert np.array_equal(out, (cvo or restate).resize(small, tw, th, name)), (name, tw, th)
    # INTER_CUBIC / INTER_LANCZOS4: host-built tap tables, bit-exact with the restatement (pinned to OpenCV's own
    # code path in tests/test_oracle.py) and with cv2 itself when its IPP dispatch is off; <= 1 grey level from IPP
    for name in ('INTER_CUBIC', 'INTER_LANCZOS4'):
        for (tw, th) in [(426, 240), (960, 540)]:
            out = ops.resize(dev(torch, fr[:1]), width=tw, height=th, interpolation=name).cpu().numpy()[0]
            assert np.array_equal(out, restate.resize(fr[0], tw, th, name)), (name, tw, th)
        for (tw, th) in [(300, 200), (64, 200), (300, 31), (131, 97), (1, 1), (43, 29)]:
            out = ops.resize(dev(torch, small), width=tw, height=th, interpolation=name).cpu().numpy()[0]
            assert np.array_equal(out, restate.resize(small, tw, th, name)), (name, tw, th)
            if cvo is not None:
                import cv2
                ipp0 = cv2.ipp.useIPP()
                try:
                    cv2.ipp.setUseIPP(False)
                    assert np.array_equal(out, cv2.resize(small, (tw, th), interpolation=getattr(cv2, name))), (name, tw, th)
                    cv2.ipp.setUseIPP(True)
                    d = np.abs(out.astype(int) - cv2.resize(small, (tw, th), interpolation=getattr(cv2, name)).astype(int))
                    assert d.max() <= 1, (name, tw, th)
                finally:
                    cv2.ipp.setUseIPP(ipp0)
    g = golden('resize_taps.npz')
    for nme in [k[3:] for k in g.files if k.startswith('in_')]:
        for name in ('INTER_CUBIC', 'INTER_LANCZOS4'):
            src, ref = g['in_' + nme], g['out_%s_%s' % (name, nme)]
            if src.ndim == 2:
                src, ref = src[..., None], ref[..., None]
            out = ops.resize(dev(torch, src), width=ref.shape[1], height=ref.shape[0], interpolation=name).cpu().numpy()[0]
            assert np.array_equal(out, ref), (name, nme)
    gray1 = np.ascontiguousarray(small[..., :1])
    for name in ('INTER_CUBIC', 'INTER_LANCZOS4'):
        out = ops.resize(dev(torch, gray1), width=77, height=50, interpolation=name).cpu().numpy()[0]
        assert np.array_equal(out[..., 0], restate.resize(gray1[..., 0], 77, 50, name).reshape(50, 77)), name
    with pytest.raises(NotImplementedError):
        ops.resize(dev(torch, fr[:1]), width=10, height=10, interpolation='INTER_MAX')


def test_convert_color_and_hsv_histogram(torch, ops, golden):
    """ConvertColor (next row, 8f rank 3) and the HSV-histogram pipeline it feeds
    (compute_hsv_histograms: ConvertToHSVCPP -> Histogram, old/histograms.py:32-36)."""
    g = golden('convert_color.npz')
    for name in ['COLOR_RGB2HSV', 'COLOR_BGR2HSV', 'COLOR_RGB2GRAY', 'COLOR_BGR2GRAY', 'COLOR_RGB2BGR']:
        out = ops.convert_color(dev(torch, g['in']), name).cpu().numpy()[0]
        assert np.array_equal(out.reshape(g[name].shape), g[name]), name
    fr = synth.noise_clip(13, 2, 1080, 1920)
    hsv = ops.convert_color(dev(torch, fr), 'COLOR_RGB2HSV')
    hsv_h = hsv.cpu().numpy()
    for i in range(2):
        assert np.array_equal(hsv_h[i], (cvo.convert_color(fr[i], 'COLOR_RGB2HSV') if cvo else restate.rgb2hsv(fr[i])))
    hist = ops.histogram(hsv).cpu().numpy()
    assert np.array_equal(hist[0], o_hist(hsv_h[0]))
    # fused ConvertToHSV -> Histogram: same counts without materialising the HSV frame
    fused = ops.histogram(dev(torch, fr), hsv='COLOR_RGB2HSV').cpu().numpy()
    assert np.array_equal(fused, hist)
    fused_list = ops.histogram([dev(torch, f) for f in fr], hsv='COLOR_RGB2HSV').cpu().numpy()
    assert np.array_equal(fused_list, hist)
    bgr = ops.histogram(dev(torch, np.ascontiguousarray(fr[..., ::-1])), hsv='COLOR_BGR2HSV').cpu().numpy()
    assert np.array_equal(bgr, hist)
    clip = synth.cut_clip(5, 70, 90, 161)[0]           # > 64 frames, odd size: unaligned frame bases
    ref = np.stack([o_hist(cvo.convert_color(f, 'COLOR_RGB2HSV') if cvo else restate.rgb2hsv(f)) for f in clip])
    assert np.array_equal(ops.histogram(dev(torch, clip), hsv='COLOR_RGB2HSV').cpu().numpy(), ref)
    assert np.array_equal(ops.histogram([dev(torch, f) for f in clip], hsv='COLOR_RGB2HSV').cpu().numpy(), ref)
    with pytest.raises(ValueError):
        ops.histogram(dev(torch, fr[:1]), hsv='COLOR_RGB2GRAY')
    with pytest.raises(NotImplementedError):
        ops.convert_color(dev(torch, fr[:1]), 'COLOR_BGR2XYZ')


# ------------------------------------------------------------------ OpticalFlow
FLOW_MEAN_TOL, FLOW_MAX_TOL = 1e-3, 1e-2   # px, north_star


def check_flow(got, ref, tag):
    e = epe(got, ref)
    assert e.mean() <= FLOW_MEAN_TOL and e.max() <= FLOW_MAX_TOL, (tag, e.mean(), e.max())
    return e


# Per-bin bound on |FlowHistogram(GPU flow) - cv2 FlowHistogram(cv2 flow)|.  north_star quotes "+-1 count per bin
# from boundary rounding".  Two independently rounded flow fields (EPE ~5e-7 px) can only differ in the bin of a pixel
# that sits within that perturbation of a bin edge, so what the bound can be depends on how many pixels the CONTENT
# puts on an edge (measured table: pytest summary / profiles/r02_flowhist_parity_table.txt / DESIGN.md section 2):
#   * generic motion (synth.warped_clip: sub-pixel translation + small rotation/zoom, a continuous spread of
#     magnitudes and directions): the +-1 of north_star holds at 426x240, 640x480 (C2) and 720p (C5); at 1080p (C3)
#     the B200 path measures 2 and at 4K 6 counts, where the oracle's own double-accumulator restatement differs
#     from cv2 by 1 and 3 (2 M / 8.3 M pixels): FLOWHIST_GENERIC_BOUND is the tightest bound measured;
#   * synth.textured_clip (blobs moving by INTEGER vectors, i.e. exactly along the axes / diagonals = exactly on the
#     0 / 45 / 90 ... degree bin edges, dy = +-5e-8): hundreds of pixels flip between the bins either side of the edge
#     (and in/out of the dropped deg == 360.0 value) in ANY two implementations -- restate vs cv2 measures up to 371
#     counts at 4K.  There the bound is relative to the oracle's own conditioning: <= 2 * (restate-vs-cv2 delta) + 2,
#     except for the two inputs of FLOWHIST_TEXTURED_MEASURED, where the B200 path's coin flips on the same on-edge
#     pixels happened to land further from cv2's than the restatement's did (measured value asserted).
FLOWHIST_GENERIC_BOUND = {(240, 426): 1, (480, 640): 1, (720, 1280): 1, (1080, 1920): 2, (2160, 3840): 6}
FLOWHIST_TEXTURED_MEASURED = {'textured 640x480 seed 1 pair 1': 21, 'textured 426x240 seed 7 pair 1': 4}


def check_flow_hist_from_flow(ops, torch, got_flow, ref_flow, tag, restate_flow=None, bound=None):
    """FlowHistogram of the GPU flow against FlowHistogram of the oracle (cv2) flow
    (scannertools/old/cpp_ops/flow_histogram_kernel_cpu.cpp:33-49).

    On IDENTICAL flow the op is bit-exact (tested separately).  On the two independently
    computed flows a pixel can change bin only through "boundary rounding": its oracle
    magnitude/angle lies within the perturbation caused by its own flow difference of a bin edge.
    Asserted: (1) per pixel, every pixel whose bin differs is such a near-edge pixel; (2) per bin,
    |count difference| <= `bound` (an absolute count, or None = 2 * the restate-vs-cv2 delta on this input + 2).
    Returns the measured row for the summary table."""
    import conftest
    gh = ops.flow_histogram(dev(torch, got_flow)).cpu().numpy()[0]
    assert np.array_equal(gh, restate.flow_histogram(got_flow)), tag       # the op itself: exact
    rh = o_flow_hist(ref_flow)
    e = epe(got_flow, ref_flow)
    mag_r, deg_r = restate.polar(ref_flow)
    mag_g, deg_g = restate.polar(got_flow)
    bm_r, bm_g = np.floor(mag_r.astype(np.float64)), np.floor(mag_g.astype(np.float64))
    ba_r = np.floor(deg_r.astype(np.float64) * (64.0 / 360.0))
    ba_g = np.floor(deg_g.astype(np.float64) * (64.0 / 360.0))
    tol_m = e * 1.01 + 1e-6
    near_m = np.abs(mag_r - np.round(mag_r)) <= tol_m
    tol_a = np.degrees(e / np.maximum(mag_r.astype(np.float64) - e, 1e-12)) * 1.01 + 0.02
    edge = 360.0 / 64.0
    dist_a = np.abs(deg_r / edge - np.round(deg_r / edge)) * edge
    near_a = (dist_a <= tol_a) | (tol_a >= edge / 2)
    assert not ((bm_r != bm_g) & ~near_m).any(), tag
    assert not ((ba_r != ba_g) & ~near_a).any(), tag
    d = np.abs(gh.astype(np.int64) - rh)
    row = {'tag': tag, 'h': got_flow.shape[0], 'w': got_flow.shape[1], 'epe_mean': float(e.mean()), 'epe_max': float(e.max()),
           'dmag': int(d[0].max()), 'dang': int(d[1].max()),
           'moved_mag': int((bm_r != bm_g).sum()), 'moved_ang': int((ba_r != ba_g).sum()),
           'r_dmag': None, 'r_dang': None}
    if restate_flow is not None:
        dr = np.abs(restate.flow_histogram(restate_flow).astype(np.int64) - rh)
        row['r_dmag'], row['r_dang'] = int(dr[0].max()), int(dr[1].max())
    conftest.FLOWHIST_ROWS.append(row)
    if bound is None:          # relative to the oracle's own conditioning on this input
        assert restate_flow is not None
        bound = max(2 * max(row['r_dmag'], row['r_dang']) + 2, FLOWHIST_TEXTURED_MEASURED.get(str(tag), 0))
    row['bound'] = bound
    if os.environ.get('STB_FLOWHIST_BOUND'):          # measurement runs: record the table without a tight bound
        bound = int(os.environ['STB_FLOWHIST_BOUND'])
    assert d.max() <= bound, (tag, 'per-bin |delta| mag %d angle %d > %d' % (row['dmag'], row['dang'], bound))
    return row


def test_farneback_goldens(torch, ops, golden):
    g = golden('flow_small.npz')
    for c in ['160x120', '240x135', '344x260']:
        f0, f1 = g['f0_' + c], g['f1_' + c]
        of = ops.OpticalFlow(f0.shape[1], f0.shape[0], max_batch=1)
        out = of.execute(dev(torch, np.stack([f0, f1]))).cpu().numpy()
        check_flow(out[0], g['flow_' + c], c)
        of.close()


def test_farneback_stage_by_stage(torch, ops):
    """I_k, R_k, M and per-level flow against the C restatement's dumps at every scale.  344x260 builds
    levels 1.. with the per-level pyramid kernels; 320x256 with pyr_h / pyr_v, whose I_k share the frame's
    I slot with level 0: the debug copy must be taken before the level-0 pyramid overwrites it."""
    for h, w in ((260, 344), (256, 320)):
        clip = synth.textured_clip(3, 2, h, w)
        of = ops.OpticalFlow(w, h, max_batch=1)
        for k in range(len(of.levels())):
            _, d = of.debug_level(dev(torch, clip), k)
            _, r = restate.farneback(restate.gray(clip[0]), restate.gray(clip[1]), dump_level=k)
            assert np.abs(d['I0'].cpu().numpy() - r['I0']).max() < 1e-3, (w, h, k)
            assert np.abs(d['I1'].cpu().numpy() - r['I1']).max() < 1e-3, (w, h, k)
            for nm in ('R0', 'R1', 'M0'):
                got = d[nm].cpu().numpy()
                ref = r[nm].transpose(2, 0, 1)
                assert np.abs(got - ref).max() <= 2e-5 * max(1.0, np.abs(ref).max()), (w, h, k, nm)
            check_flow(d['flow'].cpu().numpy(), r['flow'], 'level %d of %dx%d' % (k, w, h))
        of.close()


@pytest.mark.parametrize('h,w,seed', [(480, 640, 1), (240, 426, 7), (720, 1280, 2), (1080, 1920, 3), (2160, 3840, 4), (270, 478, 5)])
def test_farneback_parity_sizes(torch, ops, h, w, seed):
    """C2 (640x480) and the other BASELINE resolutions; 426x240 runs 3 scales only; 4K is the
    largest frame of the BASELINE configs; 478x270 has rows that are not 16-byte aligned (the LDG
    fall-back of the iteration kernel and the generic pyramid kernel)."""
    clip = synth.textured_clip(seed, 3, h, w)
    of = ops.OpticalFlow(w, h, max_batch=2)
    out = of.execute(dev(torch, clip)).cpu().numpy()
    assert out.dtype == np.float32 and out.shape == (2, h, w, 2)     # tests/test_all.py:173-177
    for i in range(2):
        ref = o_flow(clip[i], clip[i + 1])
        check_flow(out[i], ref, (h, w, i))
        # the same delta for the oracle's restatement (double accumulators, OpenCV's order) vs cv2
        rs = restate.optical_flow(clip[i], clip[i + 1])
        check_flow_hist_from_flow(ops, torch, out[i], ref, 'textured %dx%d seed %d pair %d' % (w, h, seed, i), restate_flow=rs)
    of.close()


@pytest.mark.parametrize('h,w,seed', [(240, 426, 7), (480, 640, 1), (720, 1280, 2), (1080, 1920, 3), (2160, 3840, 4)])
def test_flow_histogram_from_gpu_flow_within_one_count_per_bin(torch, ops, h, w, seed):
    """north_star: 'flow histograms must be within +-1 count per bin from boundary rounding' -- OpticalFlow ->
    FlowHistogram on the GPU against cv2 Farneback -> cv2 cartToPolar/calcHist, on generic-motion content, at the
    shipped pipeline's 426x240, C2's 640x480, C5's 720p, C3's 1080p and 4K."""
    clip = synth.warped_clip(seed, 2, h, w)
    of = ops.OpticalFlow(w, h, max_batch=1)
    flow, fh = of.execute_with_histogram(dev(torch, clip))
    flow, fh = flow.cpu().numpy()[0], fh.cpu().numpy()[0]
    of.close()
    ref = o_flow(clip[0], clip[1])
    check_flow(flow, ref, (h, w))
    rs = restate.optical_flow(clip[0], clip[1])
    check_flow_hist_from_flow(ops, torch, flow, ref, 'generic  %dx%d seed %d' % (w, h, seed), restate_flow=rs,
                              bound=FLOWHIST_GENERIC_BOUND[(h, w)])
    # the FUSED histogram (binned inside the last iteration kernel) is the one compared: same counts as the op on that flow
    assert np.array_equal(fh, restate.flow_histogram(flow))


@pytest.mark.parametrize('levels,win,iters,flags,ps,pn,sig', [
    (3, 15, 3, 256, 0.5, 5, 1.2), (2, 9, 2, 256, 0.5, 5, 1.2), (3, 21, 3, 0, 0.5, 5, 1.2), (1, 15, 1, 0, 0.5, 5, 1.2),
    (3, 7, 4, 0, 0.5, 5, 1.2), (3, 15, 3, 0, 0.75, 5, 1.2), (2, 15, 3, 256, 0.6, 5, 1.2), (3, 15, 3, 0, 0.5, 7, 1.5)])
def test_farneback_other_parameters(torch, ops, levels, win, iters, flags, ps, pn, sig):
    """FarnebackOpticalFlow arguments other than the reference's (generic kernels): the Gaussian
    window (OPTFLOW_FARNEBACK_GAUSSIAN), other windows / depths / iteration counts -- against cv2
    with the same arguments (or the pinned restatement when cv2 is missing)."""
    h, w = 270, 480
    clip = synth.textured_clip(11, 3, h, w)
    of = ops.OpticalFlow(w, h, max_batch=2, num_levels=levels, win_size=win, num_iters=iters, flags=flags, pyr_scale=ps,
                         poly_n=pn, poly_sigma=sig)
    out, fh = of.execute_with_histogram(dev(torch, clip))
    out, fh = out.cpu().numpy(), fh.cpu().numpy()
    for i in range(2):
        if cvo:
            ref = cvo.optical_flow_params(clip[i], clip[i + 1], num_levels=levels, win_size=win, num_iters=iters, flags=flags, pyr_scale=ps,
                                          poly_n=pn, poly_sigma=sig)
        else:
            ref = restate.farneback(restate.gray(clip[i]), restate.gray(clip[i + 1]), winsize=win, iters=iters, levels=levels, flags=flags,
                                    pyr_scale=ps, poly_n=pn, poly_sigma=sig)
        check_flow(out[i], ref, (levels, win, iters, flags, ps, pn, i))
        assert np.array_equal(fh[i], o_flow_hist(out[i])), i          # the (unfused here) histogram of the flow produced
    of.close()
    from scannertools_b200 import _lib
    with pytest.raises(_lib.StbError):
        ops.OpticalFlow(w, h, flags=4)                               # OPTFLOW_USE_INITIAL_FLOW


def test_farneback_batch_chunking_and_separate_buffers(torch, ops):
    """9 pairs at 160x120: several level chunks, B+1 separate frame buffers, results must not
    depend on batching (each pair equals its single-pair run bit for bit)."""
    h, w = 120, 160
    clip = synth.textured_clip(4, 10, h, w)
    frames = [dev(torch, f) for f in clip]
    of = ops.OpticalFlow(w, h, max_batch=9)
    out = of.execute(frames).cpu().numpy()
    of1 = ops.OpticalFlow(w, h, max_batch=1)
    for i in range(9):
        single = of1.execute(frames[i:i + 2]).cpu().numpy()[0]
        assert np.array_equal(out[i], single), i
        check_flow(out[i], o_flow(clip[i], clip[i + 1]), i)
    with pytest.raises(ValueError):
        of1.execute(frames[:3])
    of.close(); of1.close()


def test_farneback_content_classes(torch, ops):
    """i.i.d. noise and flat + moving square (SURVEY Appendix A sensitivity cases)."""
    h, w = 240, 320
    rng = np.random.default_rng(0)
    noise = rng.integers(0, 256, size=(2, h, w, 3), dtype=np.uint8)
    flat = np.full((2, h, w, 3), 90, np.uint8)
    flat[0, 100:140, 100:140] = 200
    flat[1, 102:142, 103:143] = 200
    of = ops.OpticalFlow(w, h, max_batch=1)
    for tag, clip in (('noise', noise), ('square', flat)):
        out = of.execute(dev(torch, clip)).cpu().numpy()[0]
        check_flow(out, o_flow(clip[0], clip[1]), tag)
    # identical frames: near-zero flow (not exactly zero: the last row/column take UpdateMatrices'
    # out-of-range branch, which leaves a non-zero h that the coarse levels spread, in OpenCV too)
    same = np.stack([noise[0], noise[0]])
    out = of.execute(dev(torch, same)).cpu().numpy()[0]
    check_flow(out, o_flow(same[0], same[1]), 'identical')
    of.close()


def test_fused_flow_histogram_and_host_pipe(torch, ops):
    h, w = 240, 426    # the shipped flow-histogram pipeline's resolution (old/histograms.py:64-68)
    clip = synth.textured_clip(7, 6, h, w)
    of = ops.OpticalFlow(w, h, max_batch=5)
    flow, fh = of.execute_with_histogram(dev(torch, clip))
    flow_h, fh_h = flow.cpu().numpy(), fh.cpu().numpy()
    _, fh_only = of.execute_with_histogram(dev(torch, clip), want_flow=False)
    assert np.array_equal(fh_only.cpu().numpy(), fh_h)
    for i in range(5):
        assert np.array_equal(fh_h[i], restate.flow_histogram(flow_h[i]))        # exact on identical flow
        check_flow_hist_from_flow(ops, torch, flow_h[i], o_flow(clip[i], clip[i + 1]), 'textured 426x240 seed 7 (6-frame clip) pair %d' % i,
                                  restate_flow=restate.optical_flow(clip[i], clip[i + 1]))
    of.close()
    pipe = ops.Pipe(w, h, max_batch=2, want_flow=True)       # batches of 2 pairs -> 3 batches with halo reuse
    pf, ph = pipe.flow(torch.from_numpy(clip).pin_memory(), want_flow=True, want_hist=True)
    assert np.array_equal(pf, flow_h) and np.array_equal(ph, fh_h)
    # asynchronous form, two calls in flight on pinned buffers
    pinned = torch.from_numpy(clip).pin_memory()
    res = [torch.zeros((5, 2, 64), dtype=torch.int32).pin_memory() for _ in range(2)]
    t0 = pipe.flow_async(pinned, res[0])
    t1 = pipe.flow_async(pinned, res[1])
    pipe.wait(t0); pipe.wait(t1)
    assert np.array_equal(res[0].numpy(), fh_h) and np.array_equal(res[1].numpy(), fh_h)
    pipe.close()


def test_c5_concurrent_streams_mixed_ops(torch, ops):
    """BASELINE configs[4] in miniature: several concurrent video streams pinned to one GPU
    (sharding.stream_assignment), each with its own OpticalFlow handle and CUDA stream, mixed
    flow + histogram work interleaved batch by batch.  Per-stream state must not leak: every
    stream's results equal those of running that stream alone, bit for bit."""
    from scannertools_b200 import sharding
    n_streams, h, w, frames_per_stream, batch = 6, 360, 640, 9, 4
    mine = sharding.stream_assignment(n_streams * 2, 2)[1]          # the streams "rank 1 of 2" owns
    assert len(mine) == n_streams
    clips = {sid: dev(torch, synth.textured_clip(50 + sid, frames_per_stream, h, w)) for sid in mine}
    # reference: one stream at a time on the default stream
    solo = ops.OpticalFlow(w, h, max_batch=frames_per_stream - 1)
    want = {}
    for sid in mine:
        flow, fh = solo.execute_with_histogram(clips[sid])
        want[sid] = (flow.clone(), fh.clone(), ops.histogram(clips[sid]).clone())
    solo.close()
    # concurrent: per-stream handles and CUDA streams, batches interleaved across streams
    handles = {sid: ops.OpticalFlow(w, h, max_batch=batch) for sid in mine}
    cstreams = {sid: torch.cuda.Stream() for sid in mine}
    got = {sid: ([], [], []) for sid in mine}
    torch.cuda.synchronize()
    for b0 in range(0, frames_per_stream - 1, batch):
        for sid in mine:
            b1 = min(b0 + batch, frames_per_stream - 1)
            with torch.cuda.stream(cstreams[sid]):
                flow, fh = handles[sid].execute_with_histogram(clips[sid][b0:b1 + 1], stream=cstreams[sid])
                hist = ops.histogram(clips[sid][b0:b1 + (1 if b1 == frames_per_stream - 1 else 0)], stream=cstreams[sid])
                got[sid][0].append(flow); got[sid][1].append(fh); got[sid][2].append(hist)
    torch.cuda.synchronize()
    for sid in mine:
        assert torch.equal(torch.cat(got[sid][0]), want[sid][0]), sid
        assert torch.equal(torch.cat(got[sid][1]), want[sid][1]), sid
        assert torch.equal(torch.cat(got[sid][2]), want[sid][2]), sid
        handles[sid].close()


def test_c_abi_error_behaviour_on_device(torch, ops):
    """Errors are status codes + stb_last_error(), never exceptions across the C boundary and
    never a silent fallback (SURVEY 8b 'Errors')."""
    import ctypes as C
    from scannertools_b200 import _lib
    lib = _lib.load()
    of = ops.OpticalFlow(160, 120, max_batch=2)
    fr = dev(torch, synth.textured_clip(1, 4, 120, 160))
    out = torch.empty((3, 120, 160, 2), dtype=torch.float32, device='cuda')
    ft = _lib.ptr_table([fr[i].data_ptr() for i in range(4)])
    ot = _lib.ptr_table([out[i].data_ptr() for i in range(3)])
    rc = lib.stb_farneback_run(of._h, ft, 3, ot, None)            # 3 pairs > max_batch 2
    assert rc == -1 and b'max_pairs' in lib.stb_last_error()
    bad = _lib.ptr_table([fr[0].data_ptr(), 0, fr[2].data_ptr()])
    assert lib.stb_farneback_run(of._h, bad, 2, ot, None) == -1 and b'NULL' in lib.stb_last_error()
    assert lib.stb_farneback_run(of._h, ft, 0, ot, None) == 0    # empty batch is a no-op
    # a NULL past the first pointer-table chunk is rejected before anything is launched
    big = ops.OpticalFlow(160, 120, max_batch=66)
    big_out = torch.empty((66, 120, 160, 2), dtype=torch.float32, device='cuda')
    bad = _lib.ptr_table([fr[i % 4].data_ptr() if i != 65 else 0 for i in range(67)])
    bot = _lib.ptr_table([big_out[i].data_ptr() for i in range(66)])
    hist = torch.empty((66, 2, 64), dtype=torch.int32, device='cuda')
    l0 = lib.stb_launch_count()
    assert lib.stb_farneback_run(big._h, bad, 66, bot, None) == -1 and b'NULL' in lib.stb_last_error()
    assert lib.stb_farneback_run_hist(big._h, bad, 66, bot, C.c_void_p(hist.data_ptr()), None) == -1 and b'NULL' in lib.stb_last_error()
    assert lib.stb_launch_count() == l0
    big.close()
    assert lib.stb_hist_rgb16_strided(C.c_void_p(fr.data_ptr()), 10, 2, 160, 120, C.c_void_p(out.data_ptr()), None) == -1  # stride < frame
    prm = _lib.FarnebackParams(3, 0.5, 0, 15, 3, 5, 1.2, 4)       # OPTFLOW_USE_INITIAL_FLOW: not implemented (the op has no flow input)
    h = C.c_void_p()
    assert lib.stb_farneback_create(160, 120, 1, C.byref(prm), C.byref(h)) == -4 and not h.value
    pipe = ops.Pipe(160, 120, max_batch=2, want_flow=False)
    with pytest.raises(_lib.StbError):
        pipe.flow(synth.textured_clip(1, 3, 120, 160), want_flow=True)
    pipe.close()
    of.close()
    with pytest.raises(TypeError):
        ops.histogram(torch.zeros((1, 4, 4, 3), dtype=torch.uint8))      # host tensor: not a device frame


def test_batched_ops_launch_counts(torch, ops):
    """Kernel launches per call of the batched entry points: one per 64-entry pointer table, one for a histogram batch
    whose frames lie at a constant stride, one per 32768 frames of a strided call, none for a rejected table."""
    import ctypes as C
    from scannertools_b200 import _lib
    lib = _lib.load()
    h, w = 8, 16
    fs, ffs = h * w * 3, h * w * 8
    src = torch.randint(0, 256, (150 * fs,), dtype=torch.uint8, device='cuda')
    dst = torch.zeros(150 * fs, dtype=torch.uint8, device='cuda')
    flow = torch.randn(150 * h * w * 2, device='cuda')
    out = torch.zeros((32769, 128), dtype=torch.int32, device='cuda')
    rgb2hsv = lib.stb_color_code(b'COLOR_RGB2HSV')

    def table(t, size, n, slot, null_at=None):
        return _lib.ptr_table([0 if i == null_at else t.data_ptr() + slot(i) * size for i in range(n)])

    def run(op, n, slot, null_src=None, null_dst=None):
        s, d = table(src, fs, n, slot, null_src), table(dst, fs, n, slot, null_dst)
        o = C.c_void_p(out.data_ptr())
        l0 = lib.stb_launch_count()
        if op == 'hist_rgb16':
            rc = lib.stb_hist_rgb16(s, n, w, h, o, None)
        elif op == 'hist_hsv16':
            rc = lib.stb_hist_hsv16(s, n, w, h, rgb2hsv, o, None)
        elif op == 'flow_hist':
            rc = lib.stb_flow_hist(table(flow, ffs, n, slot, null_src), n, w, h, o, None)
        elif op == 'convert_color':
            rc = lib.stb_convert_color_u8(s, n, w, h, rgb2hsv, d, None)
        else:
            rc = lib.stb_resize_u8(s, n, w, h, 3, d, w // 2, h // 2, 0, None)
        torch.cuda.synchronize()
        return rc, lib.stb_launch_count() - l0

    def uneven(i):                      # slots at no constant stride
        return i + i // 7

    for op in ('hist_rgb16', 'hist_hsv16', 'flow_hist', 'convert_color', 'resize'):
        for n in (1, 64, 65, 130):
            assert run(op, n, uneven) == (0, (n + 63) // 64), (op, n)
        assert run(op, 67, uneven, null_src=65) == (-1, 0), op
        if op in ('convert_color', 'resize'):
            assert run(op, 67, uneven, null_dst=65) == (-1, 0), op
    for op in ('hist_rgb16', 'hist_hsv16'):
        assert run(op, 130, lambda i: i) == (0, 1), op
    n = 32769                           # 1x1 frames, packed
    packed, packed_flow = torch.randint(0, 256, (n * 3,), dtype=torch.uint8, device='cuda'), torch.randn(n * 2, device='cuda')
    px, fl, o = C.c_void_p(packed.data_ptr()), C.c_void_p(packed_flow.data_ptr()), C.c_void_p(out.data_ptr())
    for call in (lambda: lib.stb_hist_rgb16_strided(px, 3, n, 1, 1, o, None),
                 lambda: lib.stb_hist_hsv16_strided(px, 3, n, 1, 1, rgb2hsv, o, None),
                 lambda: lib.stb_flow_hist_strided(fl, 8, n, 1, 1, o, None)):
        l0 = lib.stb_launch_count()
        assert call() == 0
        torch.cuda.synchronize()
        assert lib.stb_launch_count() - l0 == 2


def test_gray_entry_point_and_pointer_table_paths(torch, ops):
    """stb_farneback_run_gray (the cv::FarnebackOpticalFlow::calc contract on gray frames) equals
    the RGB entry point fed the same frames; FlowHistogram through the pointer-table entry point
    (separate flow buffers) equals the strided one."""
    h, w = 120, 160
    clip = synth.textured_clip(12, 4, h, w)
    of = ops.OpticalFlow(w, h, max_batch=3)
    rgb_flow = of.execute(dev(torch, clip)).cpu().numpy()
    gray = np.stack([restate.gray(f) for f in clip])[..., None]
    gray_flow = of.execute(dev(torch, gray), gray=True).cpu().numpy()
    assert np.array_equal(rgb_flow, gray_flow)
    of.close()
    flows = dev(torch, rgb_flow)
    a = ops.flow_histogram(flows).cpu().numpy()
    b = ops.flow_histogram([flows[i].clone() for i in range(3)]).cpu().numpy()
    assert np.array_equal(a, b)
    for i in range(3):
        assert np.array_equal(a[i], restate.flow_histogram(rgb_flow[i]))


def test_farneback_more_pairs_than_one_pointer_table(torch, ops):
    """More than 64 pairs in one call: the chain launches are chunked at the 64-entry pointer table and
    the pyramid / polynomial expansion is launched in slices of 65 frames on the second lane; every pair
    must equal its single-pair run, flow and fused histogram.  96x64 (2 scales) and 320x256 (4 scales)
    both take the two-launch pyramid (pyr_h / pyr_v) for levels 1.. ."""
    for h, w, n in ((64, 96, 70), (256, 320, 66)):
        clip = synth.textured_clip(21, n + 1, h, w, max_shift=1.5)
        fr = dev(torch, clip)
        of = ops.OpticalFlow(w, h, max_batch=n)
        out = of.execute(fr).cpu().numpy()
        flow_h, fh = of.execute_with_histogram(fr)
        flow_h, fh = flow_h.cpu().numpy(), fh.cpu().numpy()
        assert np.array_equal(flow_h, out)
        of1 = ops.OpticalFlow(w, h, max_batch=1)
        for i in (0, 31, 63, 64, n - 1):
            single = of1.execute(fr[i:i + 2]).cpu().numpy()[0]
            assert np.array_equal(out[i], single), (w, h, i)
            _, single_fh = of1.execute_with_histogram(fr[i:i + 2])
            assert np.array_equal(fh[i], single_fh.cpu().numpy()[0]), (w, h, i)
            check_flow(out[i], o_flow(clip[i], clip[i + 1]), (w, h, i))
        of.close(); of1.close()


def test_cuda_graph_replay_equals_direct_launches(torch, ops):
    """Batches are replayed from a cached CUDA graph whose pointer-carrying nodes (frame table, flow table,
    histogram pointer, histogram memset) are re-pointed on every call: results must equal the direct-launch path
    bit for bit across calls with DIFFERENT frame / output buffers, batch sizes and output combinations."""
    h, w = 240, 320
    clips = [dev(torch, synth.textured_clip(40 + i, 5, h, w)) for i in range(3)]
    os.environ['STB_NO_GRAPH'] = '1'
    try:
        direct = ops.OpticalFlow(w, h, max_batch=4)
    finally:
        del os.environ['STB_NO_GRAPH']
    graphed = ops.OpticalFlow(w, h, max_batch=4)
    for rep in range(2):
        for i, clip in enumerate(clips):
            n = 4 if i != 1 else 3                                   # two graph shapes
            fr = [clip[j].clone() for j in range(n + 1)]             # fresh buffers: new pointers every call
            a_flow, a_fh = direct.execute_with_histogram(fr)
            b_flow, b_fh = graphed.execute_with_histogram(fr)
            assert torch.equal(a_flow, b_flow) and torch.equal(a_fh, b_fh), (rep, i)
            _, c_fh = graphed.execute_with_histogram(fr, want_flow=False)
            assert torch.equal(c_fh, a_fh), (rep, i)
            out = torch.full((n, h, w, 2), 7.0, dtype=torch.float32, device='cuda')
            graphed.execute(fr, out=out)
            assert torch.equal(out, a_flow), (rep, i)
    direct.close(); graphed.close()


@pytest.mark.gpu
@pytest.mark.parametrize('h,w,gen', [(480, 640, 'textured'), (1080, 1920, 'warped'), (270, 480, 'noise')])
def test_flow_compensated_window_equals_global_gathers(torch, ops, h, w, gen):
    """iter15_win_kernel (R1 footprints of a tile staged in shared memory by TMA at a data-dependent origin)
    against iter15_tma_kernel (global gathers, STB_NO_WIN): bit-identical flow and fused histogram on smooth
    motion (tiles fit), blob borders (some tiles do not) and noise (incoherent flow: most tiles fall back)."""
    clip = {'textured': lambda: synth.textured_clip(5, 4, h, w), 'warped': lambda: synth.warped_clip(6, 4, h, w),
            'noise': lambda: synth.noise_clip(7, 4, h, w)}[gen]()
    fr = dev(torch, clip)
    os.environ['STB_NO_WIN'] = '1'
    try:
        plain = ops.OpticalFlow(w, h, max_batch=3)
    finally:
        del os.environ['STB_NO_WIN']
    win = ops.OpticalFlow(w, h, max_batch=3)
    a_flow, a_fh = plain.execute_with_histogram(fr)
    b_flow, b_fh = win.execute_with_histogram(fr)
    assert torch.equal(a_flow, b_flow) and torch.equal(a_fh, b_fh)
    plain.close(); win.close()


@pytest.mark.gpu
def test_flow_histogram_fast_binning_randomised(torch, ops):
    """The device's approximate bin location (MUFU.SQRT / MUFU.RCP) + exact path inside the guard bands against the
    oracle on fields dense in values on and next to bin edges, tiny / huge / non-finite values included; also
    against cv2 itself when it is importable."""
    for seed, (h, w) in ((11, (192, 256)), (12, (1080, 1920))):
        ff = synth.edge_flow_field(seed, h, w)
        out = ops.flow_histogram(dev(torch, ff)).cpu().numpy()[0]
        assert np.array_equal(out, restate.flow_histogram(ff)), seed
        if cvo is not None:
            assert np.array_equal(out, cvo.flow_histogram(ff)), seed
