#!/usr/bin/env python
"""Times every ConvertColor conversion through the C ABI with CUDA events: 1080p x 64 frames per call (1.2 to 2.1 GB
moved, well above the 126 MB L2), device-resident frames in separate buffers (one pointer table per 64 frames).
Reports per conversion the time per call, the effective rate (in + out channels) x W x H x n bytes / time and its
share of the HBM peak that bench.measured_peaks() returns (MEASURED_PEAKS.json when present, else a fallback
figure: the output says which), with the card name and power limit read in the same run.

  python tools/convert_color_bench.py [--lib PATH ...] [--rounds R] [--iters K] [--json OUT]

Several --lib arguments compare builds of libscannertools_b200.so (say the parent's and this tree's): each round
runs every library once, in that order, in a fresh process, and the report gives each conversion's median over the
rounds.  A library without stb_color_in_channels predates the 1- and 4-channel conversions, so it is given
3-channel frames, and conversions its stb_color_code does not know are skipped for it."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.abspath(os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))
sys.path.insert(0, ROOT)

# one name per conversion code
NAMES = ['COLOR_RGB2HSV', 'COLOR_BGR2HSV', 'COLOR_RGB2GRAY', 'COLOR_BGR2GRAY', 'COLOR_BGR2RGB',
         'COLOR_BGR2BGRA', 'COLOR_BGR2RGBA', 'COLOR_BGRA2BGR', 'COLOR_RGBA2BGR', 'COLOR_BGRA2RGBA',
         'COLOR_GRAY2BGR', 'COLOR_GRAY2BGRA', 'COLOR_BGRA2GRAY', 'COLOR_RGBA2GRAY',
         'COLOR_BGR2YCrCb', 'COLOR_RGB2YCrCb', 'COLOR_YCrCb2BGR', 'COLOR_YCrCb2RGB',
         'COLOR_BGR2YUV', 'COLOR_RGB2YUV', 'COLOR_YUV2BGR', 'COLOR_YUV2RGB', 'COLOR_BGR2HSV_FULL', 'COLOR_RGB2HSV_FULL']
W, H, N = 1920, 1080, 64


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(['nvidia-smi', '-i', '0', '--query-gpu=power.limit', '--format=csv,noheader'],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # report what could not be read rather than guess
        limit = 'unavailable (%s)' % e
    return name, limit


def run_one(lib_path, iters, warmup):
    """Times every conversion `lib_path` implements; returns {name: ms per call}."""
    import torch
    lib = C.CDLL(lib_path)
    lib.stb_color_code.argtypes = [C.c_char_p]
    lib.stb_convert_color_u8.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    in_channels = getattr(lib, 'stb_color_in_channels', None)
    torch.cuda.set_device(0)
    gen = torch.Generator(device='cuda').manual_seed(7)
    frames = {}
    res = {}
    for name in NAMES:
        code = lib.stb_color_code(name.encode())
        if code < 0:
            continue
        cin = in_channels(code) if in_channels else 3
        cout = lib.stb_color_out_channels(code)
        if cin not in frames:
            frames[cin] = torch.randint(0, 256, (N, H, W, cin), dtype=torch.uint8, device='cuda', generator=gen)
        src = frames[cin]
        dst = torch.empty((N, H, W, cout), dtype=torch.uint8, device='cuda')
        st = (C.c_void_p * N)(*[src[i].data_ptr() for i in range(N)])
        dt = (C.c_void_p * N)(*[dst[i].data_ptr() for i in range(N)])
        s = torch.cuda.current_stream().cuda_stream

        def call():
            rc = lib.stb_convert_color_u8(st, N, W, H, code, dt, s)
            if rc != 0:
                raise RuntimeError('%s: status %d' % (name, rc))
        for _ in range(warmup):
            call()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            call()
        b.record()
        torch.cuda.synchronize()
        res[name] = {'ms': a.elapsed_time(b) / iters, 'in': cin, 'out': cout}
        del dst
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--lib', action='append', help='libscannertools_b200.so to time (repeatable; default: this tree)')
    ap.add_argument('--rounds', type=int, default=1)
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--json', help='also write the report here')
    ap.add_argument('--child', help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.child:
        print(json.dumps(run_one(a.child, a.iters, a.warmup)))
        return
    from bench import measured_peaks
    libs = [os.path.abspath(p) for p in (a.lib or [os.path.join(ROOT, 'scannertools_b200', 'libscannertools_b200.so')])]
    runs = {p: [] for p in libs}
    for _ in range(a.rounds):
        for p in libs:
            out = subprocess.run([sys.executable, os.path.abspath(__file__), '--child', p, '--iters', str(a.iters),
                                  '--warmup', str(a.warmup)], check=True, capture_output=True, text=True).stdout
            runs[p].append(json.loads(out.strip().splitlines()[-1]))
    peak, peak_src = measured_peaks()
    name, limit = card()
    report = {'card': name, 'power_limit': limit, 'peak_gbs': peak, 'peak_source': peak_src, 'frames': [N, H, W],
              'iters': a.iters, 'rounds': a.rounds, 'libs': {}}
    print('%s, power limit %s; HBM peak %.0f GB/s (%s); %d x %dx%d frames per call, %d calls per round, %d rounds'
          % (name, limit, peak, peak_src, N, W, H, a.iters, a.rounds))
    for p in libs:
        rows = {}
        print('\n%s' % p)
        print('%-20s %5s %9s %9s %8s %9s' % ('conversion', 'in>out', 'ms/call', 'GB/s', '% peak', 'spread'))
        for nm in NAMES:
            ms = sorted(r[nm]['ms'] for r in runs[p] if nm in r)
            if not ms:
                continue
            med = ms[len(ms) // 2]
            cin, cout = runs[p][0][nm]['in'], runs[p][0][nm]['out']
            gbs = (cin + cout) * W * H * N / (med * 1e-3) / 1e9
            rows[nm] = {'ms': med, 'ms_all': ms, 'in': cin, 'out': cout, 'gbs': gbs, 'pct_peak': 100 * gbs / peak}
            print('%-20s %2d>%-2d %9.3f %9.1f %8.1f %8.1f%%' % (nm[6:], cin, cout, med, gbs, 100 * gbs / peak,
                                                              100 * (ms[-1] - ms[0]) / med))
        report['libs'][p] = rows
    if a.json:
        with open(a.json, 'w') as f:
            json.dump(report, f, indent=1)


if __name__ == '__main__':
    main()
