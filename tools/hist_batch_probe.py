import os, sys, torch
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), '..'))
from scannertools_b200 import ops
def timeit(fn, iters=20, warm=3):
    for _ in range(warm): fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(iters): fn()
    b.record(); torch.cuda.synchronize()
    return a.elapsed_time(b) / iters * 1e-3
big = torch.randint(0, 256, (40, 2160, 3840, 3), dtype=torch.uint8, device='cuda')
for n in (1, 2, 4, 8, 16, 32, 40):
    fr = big[:n]
    t = timeit(lambda: ops.histogram(fr))
    by = n * (3 * 2160 * 3840 + 192)
    print('4K n=%2d: %.1f us  %.1f GB/s  %.1f%%' % (n, t * 1e6, by / t / 1e9, 100 * by / t / 6514.2e9))
small = torch.randint(0, 256, (64, 1080, 1920, 3), dtype=torch.uint8, device='cuda')
for n in (1, 4, 16, 64):
    fr = small[:n]
    t = timeit(lambda: ops.histogram(fr))
    by = n * (3 * 1080 * 1920 + 192)
    print('1080p n=%2d: %.1f us  %.1f GB/s  %.1f%%' % (n, t * 1e6, by / t / 1e9, 100 * by / t / 6514.2e9))
