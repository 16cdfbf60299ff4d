"""Generates the golden fixtures in this directory from the cv2 oracle (oracle/cv2_ops.py),
i.e. from OpenCV itself -- the library the reference's wrappers call.

Run from the repo root:  python tests/golden/make_golden.py
Inputs are stored alongside outputs (not only seeds) so the fixtures do not depend on the
generator's numpy/cv2 versions when they are replayed.  shot_reference.npz is rewritten only when
SCANNERTOOLS_REFERENCE names a checkout of the reference (ref_import.py).
"""
import glob
import os
import sys
import numpy as np

sys.path.insert(0, os.path.join(os.path.dirname(__file__), '..', '..'))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import cv2  # noqa: E402
from oracle import cv2_ops  # noqa: E402
from scannertools_b200 import synth  # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))
MAX_FILE_BYTES = 1000000
PART_ARRAY_BYTES = 960000     # raw array bytes per file, leaving room for the npz container


def save(name, **arrays):
    """np.savez_compressed of the arrays into `<name>.npz`, continued in `<name>.1.npz`, `<name>.2.npz`, ...
    where one file would pass MAX_FILE_BYTES; tests/conftest.py's `golden` fixture reads the parts as one."""
    stem = os.path.join(HERE, name)
    for old in glob.glob(glob.escape(stem) + '.[0-9]*.npz'):
        os.remove(old)
    parts, size = [{}], 0
    for k, a in arrays.items():
        nbytes = np.asarray(a).nbytes
        if parts[-1] and size + nbytes > PART_ARRAY_BYTES:
            parts.append({})
            size = 0
        parts[-1][k] = a
        size += nbytes
    for i, part in enumerate(parts):
        path = stem + ('.%d.npz' % i if i else '.npz')
        np.savez_compressed(path, **part)
        assert os.path.getsize(path) <= MAX_FILE_BYTES, (path, os.path.getsize(path))


def make_resize_taps():
    """INTER_CUBIC / INTER_LANCZOS4 goldens from OpenCV's OWN resize code: cv2.ipp.setUseIPP(False), because this
    wheel otherwise hands 8-bit cubic to IPP (a different arithmetic, +-1 grey level).  `python make_golden.py resize_taps`
    writes only this file."""
    meta = dict(cv2=cv2.__version__, numpy=np.__version__, ipp='off')
    rng = np.random.default_rng(31)
    ipp0 = cv2.ipp.useIPP()
    cv2.ipp.setUseIPP(False)
    try:
        rs = {}
        for name, (sh, sw, dh, dw, cn) in {'down_frac': (135, 240, 60, 107, 3), 'up': (37, 53, 80, 111, 3), 'half': (120, 160, 60, 80, 3),
                                           'gray_mixed': (33, 47, 70, 21, 1), 'rgba': (40, 30, 25, 64, 4), 'tiny': (3, 2, 9, 10, 3)}.items():
            img = rng.integers(0, 256, (sh, sw, cn) if cn > 1 else (sh, sw), dtype=np.uint8)
            rs['in_' + name] = img
            for interp in ('INTER_CUBIC', 'INTER_LANCZOS4'):
                rs['out_%s_%s' % (interp, name)] = cv2.resize(img, (dw, dh), interpolation=getattr(cv2, interp))
    finally:
        cv2.ipp.setUseIPP(ipp0)
    save('resize_taps', meta=str(meta), **rs)


def main():
    if sys.argv[1:] == ['resize_taps']:
        make_resize_taps()
        return
    meta = dict(cv2=cv2.__version__, numpy=np.__version__)
    make_resize_taps()

    # C1: ShotDetection clip -- 1000 frames 640x360, 7 planted cuts, seed 5 (SURVEY §8d)
    clip, cuts = synth.cut_clip(5, 1000, 360, 640, n_cuts=7)
    hists = np.stack([cv2_ops.histogram(f) for f in clip]).astype(np.int32)
    bounds = cv2_ops.shot_boundaries(list(hists))
    save('shot_c1', hists=hists, boundaries=np.array(bounds, np.int32),
         cuts=np.array(cuts, np.int32), scores=cv2_ops.shot_scores(hists),
         frame0=clip[0], frame_first_cut=clip[cuts[0]], meta=str(meta))
    print('shot_c1: boundaries', bounds, 'cuts', cuts)

    # small histogram cases incl. ragged widths (rows not 4/16-byte aligned) and constants
    hs = {}
    for name, fr in [('noise_37x53', synth.noise_clip(11, 1, 37, 53)[0]),
                     ('noise_120x213', synth.noise_clip(12, 1, 120, 213)[0]),
                     ('const0_64x64', synth.const_clip(0, 1, 64, 64)[0]),
                     ('const255_64x48', synth.const_clip(255, 1, 48, 64)[0]),
                     ('one_px', synth.noise_clip(13, 1, 1, 1)[0])]:
        hs['in_' + name] = fr
        hs['out_' + name] = cv2_ops.histogram(fr)
    save('hist_small', meta=str(meta), **hs)

    # Farneback: textured pairs at sizes covering 4 scales, 3 scales, and round-half-even
    fl = {}
    for name, seed, h, w in [('160x120', 1, 120, 160), ('240x135', 2, 135, 240), ('344x260', 3, 260, 344)]:
        c = synth.textured_clip(seed, 2, h, w)
        fl['f0_' + name] = c[0]
        fl['f1_' + name] = c[1]
        fl['gray0_' + name] = cv2_ops.gray(c[0])
        fl['flow_' + name] = cv2_ops.optical_flow(c[0], c[1])
    save('flow_small', meta=str(meta), **fl)

    # FlowHistogram: a real flow field and the stress field
    fh = {}
    real = fl['flow_240x135']
    stress = synth.textured_flow_field(3, 120, 213)
    for name, f in [('real_240x135', real), ('stress_213x120', stress),
                    ('stress_33x17', synth.textured_flow_field(4, 17, 33))]:
        fh['in_' + name] = f
        fh['out_' + name] = cv2_ops.flow_histogram(f)
        x, y = cv2.split(f)
        mag, deg = cv2.cartToPolar(x, y, angleInDegrees=True)
        if f.size < 4096:
            fh['mag_' + name] = mag
            fh['deg_' + name] = deg
    save('flowhist', meta=str(meta), **fh)

    # FrameDifference (intended semantics)
    a = synth.noise_clip(21, 2, 19, 23)
    save('framediff', prev=a[0], cur=a[1],
         out=cv2_ops.frame_difference(a[0], a[1]), meta=str(meta))
    # Resize (next row): down-scale to the shipped pipeline's 426x240, exact 2x, up-scale, gray
    rs = {}
    rng = np.random.default_rng(31)
    for name, (sw, sh, dw, dh, cn) in [('270p_to_213x120', (480, 270, 213, 120, 3)), ('half', (128, 96, 64, 48, 3)),
                                       ('up', (64, 48, 200, 100, 3)), ('gray_odd', (101, 77, 33, 20, 1))]:
        img = rng.integers(0, 256, (sh, sw, cn) if cn > 1 else (sh, sw), dtype=np.uint8)
        rs['in_' + name] = img
        rs['out_' + name] = cv2_ops.resize(img, dw, dh)
    save('resize', meta=str(meta), **rs)
    # ConvertColor (next row): the conversions the B200 build implements
    rng = np.random.default_rng(77)
    img = rng.integers(0, 256, (60, 107, 3), dtype=np.uint8)
    img[0, :6] = [[0, 0, 0], [255, 255, 255], [255, 0, 0], [0, 255, 0], [0, 0, 255], [128, 128, 127]]
    cc = {'in': img}
    for name in ['COLOR_RGB2HSV', 'COLOR_BGR2HSV', 'COLOR_RGB2GRAY', 'COLOR_BGR2GRAY', 'COLOR_RGB2BGR']:
        cc[name] = cv2_ops.convert_color(img, name)
    save('convert_color', meta=str(meta), **cc)
    # ShotBoundaries goldens from the REFERENCE ITSELF (its Python op imported from the checkout that
    # SCANNERTOOLS_REFERENCE names, behind a scannerpy stub, ref_import.py): histogram sequences -> boundary lists
    import ref_import
    if ref_import.available():
        sd, ty = ref_import.load('shot_detection'), ref_import.load('types')
        rng = np.random.default_rng(2024)

        def make(n, n_cuts, jitter):
            base = rng.integers(0, 20000, size=(n_cuts + 1, 3, 16))
            cuts_ = np.sort(rng.choice(np.arange(1, max(n, 2)), size=min(n_cuts, max(n - 1, 0)), replace=False)) if n > 1 else np.array([], int)
            seg = np.searchsorted(cuts_, np.arange(n), side='right')
            h = base[seg] + rng.integers(-jitter, jitter + 1, size=(n, 3, 16))
            return np.clip(h, 0, None).astype(np.int32)
        cases = {}
        for name, (n, k, j) in {'n1': (1, 0, 5), 'n2': (2, 1, 5), 'n40': (40, 3, 50), 'n600': (600, 5, 200),
                                'n1300': (1300, 9, 400), 'flat300': (300, 0, 0), 'noisy900': (900, 4, 6000)}.items():
            h = make(n, k, j)
            rows = sd.shot_boundaries(None, [ty.histograms(x.tobytes(), None) for x in h])
            cases['hist_' + name] = h
            cases['bounds_' + name] = np.array(rows[0], np.int32)
        save('shot_reference', meta='generated by the reference scannertools/shot_detection.py::shot_boundaries', **cases)
    for f in sorted(os.listdir(HERE)):
        if f.endswith('.npz'):
            print(f, os.path.getsize(os.path.join(HERE, f)))


if __name__ == '__main__':
    main()
