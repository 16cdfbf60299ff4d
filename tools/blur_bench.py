#!/usr/bin/env python
"""Times the Blur op (stb_blur_u8) through the C ABI with CUDA events: 1080p x 64 frames per call in separate
buffers (one pointer table per 64 frames; 0.13 GB for 1 channel to 0.53 GB for 4 channels each way, past the
126 MB L2), k in {3, 5, 15, 31} and C in {1, 3, 4}.  Reports per case the time per call, the effective rate
2 C x W x H x n bytes / time and its share of the HBM peak that bench.measured_peaks() returns (MEASURED_PEAKS.json
when present, else a fallback figure: the output says which), with the card name and power limit read in the same
run.

  python tools/blur_bench.py [--lib PATH ...] [--rounds R] [--iters K] [--json OUT]

Several --lib arguments compare builds of libscannertools_b200.so: each round runs every library once, in that
order, in a fresh process, and the report gives each case's median over the rounds."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.abspath(os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))
sys.path.insert(0, ROOT)

KS = [3, 5, 15, 31]
CHANNELS = [1, 3, 4]
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
    """Times every (k, C) case; returns {'k<k>c<C>': ms per call}."""
    import torch
    lib = C.CDLL(lib_path)
    lib.stb_blur_u8.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p]
    torch.cuda.set_device(0)
    gen = torch.Generator(device='cuda').manual_seed(7)
    res = {}
    for c in CHANNELS:
        src = torch.randint(0, 256, (N, H, W, c), dtype=torch.uint8, device='cuda', generator=gen)
        dst = torch.empty_like(src)
        st = (C.c_void_p * N)(*[src[i].data_ptr() for i in range(N)])
        dt = (C.c_void_p * N)(*[dst[i].data_ptr() for i in range(N)])
        s = torch.cuda.current_stream().cuda_stream
        for k in KS:
            def call():
                rc = lib.stb_blur_u8(st, N, W, H, c, k, dt, s)
                if rc != 0:
                    raise RuntimeError('k=%d C=%d: status %d' % (k, c, rc))
            for _ in range(warmup):
                call()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(iters):
                call()
            b.record()
            torch.cuda.synchronize()
            res['k%dc%d' % (k, c)] = a.elapsed_time(b) / iters
        del src, dst
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
        print('%4s %2s %9s %9s %8s %9s' % ('k', 'C', 'ms/call', 'GB/s', '% peak', 'spread'))
        for c in CHANNELS:
            for k in KS:
                key = 'k%dc%d' % (k, c)
                ms = sorted(r[key] for r in runs[p] if key in r)
                med = ms[len(ms) // 2]
                gbs = 2 * c * W * H * N / (med * 1e-3) / 1e9
                rows[key] = {'k': k, 'channels': c, 'ms': med, 'ms_all': ms, 'gbs': gbs, 'pct_peak': 100 * gbs / peak}
                print('%4d %2d %9.3f %9.1f %8.1f %8.1f%%' % (k, c, med, gbs, 100 * gbs / peak, 100 * (ms[-1] - ms[0]) / med))
        report['libs'][p] = rows
    if a.json:
        with open(a.json, 'w') as f:
            json.dump(report, f, indent=1)


if __name__ == '__main__':
    main()
