#!/usr/bin/env python
"""Times float32 Resize (stb_resize_f32) through the C ABI with CUDA events after warm-up:

  - 64 flow fields of 1920x1080x2 per call, to 426x240 (the shipped flow-histogram pipeline's size) and to 960x540
    (exact 2x), in every interpolation mode;
  - 16 frames of 3840x2160x4 per call, to 1920x1080, INTER_LINEAR and INTER_AREA.

Each call's inputs (1.06 GB and 2.12 GB) are larger than the 126 MB L2, so no pass finds its source there.  The byte
model comes from the same index tables the kernels use (tests/resize_f32_restate.py): the distinct source rows the
mode reads times the row bytes, plus the destination bytes.  Each rate is reported as a share of the copy peak that
bench.measured_peaks() returns, with the card name and power limit read in the same run.

  python tools/resize_f32_bench.py [--iters K] [--warmup W] [--json OUT]"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

MODES = ['INTER_NEAREST', 'INTER_LINEAR', 'INTER_AREA', 'INTER_CUBIC', 'INTER_LANCZOS4']
# (name, n, sw, sh, channels, dw, dh, modes)
WORKLOADS = [('flow 1080p -> 426x240', 64, 1920, 1080, 2, 426, 240, MODES),
             ('flow 1080p -> 960x540', 64, 1920, 1080, 2, 960, 540, MODES),
             ('4K x4 -> 1080p', 16, 3840, 2160, 4, 1920, 1080, ['INTER_LINEAR', 'INTER_AREA'])]


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=power.limit', '--format=csv,noheader'],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # report what could not be read rather than guess
        limit = 'unavailable (%s)' % e
    return name, limit


def source_rows(interp, sw, sh, dw, dh):
    """The distinct source rows one destination frame reads (the kernels' row index tables)."""
    import resize_f32_restate as rr
    p = rr.path(interp, sw, sh, dw, dh)
    scy = 1.0 / (dh / sh)
    if p == 'nearest':
        return len(set(min(int(np.floor(d * scy)), sh - 1) for d in range(dh)))
    if p == 'area_fast':
        return dh * round(sh / dh)
    if p == 'area':
        return len(set(s for d in range(dh) for s, _ in rr.area_span(d, scy, sh)))
    if p == 'linear':
        y0, y1, _ = rr._linear_axis(dh, sh, scy, interp == 'INTER_AREA', False)
        return len(set(y0.tolist()) | set(y1.tolist()))
    K = 4 if interp == 'INTER_CUBIC' else 8
    ofs, _ = rr.taps(dh, sh, K)
    return len(set(np.clip(ofs[:, None] + np.arange(K)[None, :], 0, sh - 1).reshape(-1).tolist()))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--json', help='also write the report here')
    a = ap.parse_args()
    import torch
    from bench import measured_peaks
    from scannertools_b200 import _lib
    lib = _lib.load()
    torch.cuda.set_device(0)
    codes = {m: lib.stb_resize_interp_code(m.encode()) for m in MODES}
    peak, peak_src = measured_peaks()
    name, limit = card()
    print('%s, power limit %s; copy peak %.0f GB/s (%s); inputs larger than L2, %d timed calls after %d warm-up calls'
          % (name, limit, peak, peak_src, a.iters, a.warmup))
    print('%-24s %-15s %9s %10s %9s %8s' % ('workload', 'mode', 'ms/call', 'model GB', 'GB/s', 'of peak'))
    gen = torch.Generator(device='cuda').manual_seed(7)
    report = {'card': name, 'power_limit': limit, 'peak_gbs': peak, 'peak_source': peak_src, 'iters': a.iters,
              'l2': 'inputs larger than L2', 'rows': []}
    s = torch.cuda.current_stream()
    for wl, n, sw, sh, c, dw, dh, modes in WORKLOADS:
        src = torch.randn((n, sh, sw, c), device='cuda', generator=gen) * 8
        dst = torch.empty((n, dh, dw, c), device='cuda')
        st = _lib.ptr_table([src[i].data_ptr() for i in range(n)])
        dt = _lib.ptr_table([dst[i].data_ptr() for i in range(n)])
        for m in modes:
            def call():
                _lib.check(lib.stb_resize_f32(st, n, sw, sh, c, dt, dw, dh, codes[m], C.c_void_p(s.cuda_stream)), lib)
            for _ in range(a.warmup):
                call()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.iters):
                call()
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / a.iters
            nbytes = n * (source_rows(m, sw, sh, dw, dh) * sw * c * 4 + dw * dh * c * 4)
            gbs = nbytes / (ms * 1e-3) / 1e9
            print('%-24s %-15s %9.3f %10.3f %9.1f %7.1f%%' % (wl, m, ms, nbytes / 1e9, gbs, 100 * gbs / peak))
            report['rows'].append({'workload': wl, 'mode': m, 'ms': ms, 'model_bytes': nbytes, 'gbs': gbs,
                                   'share_of_peak': gbs / peak})
        del src, dst
        torch.cuda.empty_cache()
    if a.json:
        with open(a.json, 'w') as f:
            json.dump(report, f, indent=1)


if __name__ == '__main__':
    main()
