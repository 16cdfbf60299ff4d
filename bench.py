#!/usr/bin/env python
"""Benchmark of the per-frame analysis hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            our arm (CUDA kernels via the C ABI)
  python bench.py --impl reference ...                      reference arm: the reference's OpenCV
                                                            CPU ops on the box's host cores
  python bench.py ... --dump-outputs DIR                    our arm, and after the timed steps the
                                                            outputs of the last one as DIR/<name>.npy

Headline workload (config.workload): C3 -- 1080p Farneback OpticalFlow + FlowHistogram on ONE seeded
synthetic clip of N*pairs+1 frames, frame-range sharded over the N ranks (sharding.pair_range: rank r
owns pairs [r*pairs, (r+1)*pairs) and reads one halo frame).  A "step" is one pass of the hot path over
this rank's `--pairs` frame pairs (pairs+1 1080p RGB frames, a ring larger than L2).
`value`  = frames/s with the frames already resident in HBM (whole job, all ranks).
`e2e`    = frames/s through the host-buffer C-ABI call (stb_pipe_flow_async): pinned-host frames in,
           H2D copies inside the timed region, 512-byte flow histograms out (the shipped
           compute_flow_histograms pipeline).  `e2e_flow_frames` is the same call returning the flow
           FRAMES too (the OpticalFlow op itself, 16.6 MB/frame D2H); `e2e.copy_only` is the measured
           ceiling of the host feed: the same H2D bytes with no kernels, all ranks at once.
`roofline` = the dominant kernel (fused level-0 update iteration): algorithmic bytes per launch
           / its CUDA-event duration measured in the timed region, against MEASURED_PEAKS.json.
`extra`  = the other workloads of the metric at this N: C4 (4K RGB histogram + shot scoring on a
           frame-range-sharded clip with cuts on the shard seams), C5 (8 concurrent 720p streams
           per GPU, mixed ops), C2 (640x480 flow), the fused HSV histogram.
After the timed regions the per-frame outputs of all ranks are concatenated on the host and rank 0
re-computes the pairs / frames at every shard seam alone (`shard_check`).  Frames are independent:
no collective on the data path (scaling = weak: per-GPU work is fixed).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# algorithmic bytes (SURVEY.md §8d / DESIGN.md "Byte model")
FLOW1080_BYTES = 771768000          # canonical Farneback pass model, per 1080p frame
FLOWHIST1080_BYTES = 16589312       # 8*W*H + 512
ITER_BYTES_PER_PX = 80              # level-0 update iteration: read M, R0, R1; write M' (5 f32 each)
HIST4K_BYTES = 24883392             # 3*W*H + 192
FLOW480_BYTES = 114336000
C5_BYTES = 343008000 + 8 * 1280 * 720 + 512 + 2764992   # 720p flow + flow histogram + RGB histogram

C3_SEED, C4_SEED = 1000, 77
C4_FRAMES = 32                      # 4K frames per rank and step (796 MB > L2)
C5_STREAMS, C5_BATCH = 8, 16        # streams per GPU (64 streams on 8 GPUs), frames per stream per step

# --dump-outputs: the flow histograms of every pair in full, the flow frames (1080p x 8 bytes each) as a
# fixed seeded sample of pixels, the same for every pair, so that all files together stay within 64 MB
DUMP_MAX_BYTES = 64 << 20
DUMP_FLOW_BYTES = 48 << 20
DUMP_SEED = 2024


def dump_pixels(n_px, n_pairs):
    """Sorted flat pixel indices (into H x W) of the flow sample that --dump-outputs writes."""
    k = max(1, min(n_px, DUMP_FLOW_BYTES // (n_pairs * 8)))
    return np.sort(np.random.default_rng(DUMP_SEED).choice(n_px, size=k, replace=False))


def write_dump(out_dir, arrays):
    """One out_dir/<name>.npy per output: float32 stays float32, everything else (integer counts) is written as
    float64, which holds them exactly."""
    arrays = {k: np.ascontiguousarray(a, np.float32 if a.dtype == np.float32 else np.float64) for k, a in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    assert total <= DUMP_MAX_BYTES, ('--dump-outputs', total)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), a)


def measured_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.isfile(p):
        try:
            return float(json.load(open(p))['hbm_gbs']), 'measured'
        except Exception:
            pass
    return 6650.0, 'fallback'


def ncu_traffic():
    """dram__bytes_read.sum + dram__bytes_write.sum of the roofline kernel, per PAIR, from the
    committed `ncu --set full` capture of this round (profiles/traffic.json, written by
    tools/ncu_table.py --traffic).  None when no capture of the current kernel is committed."""
    p = os.path.join(ROOT, 'profiles', 'traffic.json')
    try:
        t = json.load(open(p))
        return float(t['bytes_per_pair']), t.get('source', 'profiles/traffic.json')
    except Exception:
        return None, None


class ClockSampler:
    """SM clock, power and clock-event (throttle) reasons sampled DURING the timed region by a thread
    polling NVML every ~5 ms (the main thread sits in C calls that release the GIL); only samples
    taken inside [t0, t1] of the timed region are kept.  Falls back to parsing `nvidia-smi -lms` when
    NVML cannot be loaded."""
    Q = ('timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index, pci_bus_id=None):
        self.idx = gpu_index
        self.pci = pci_bus_id
        self.samples = []      # (time, sm_mhz, max_mhz, power_w, reasons-set)
        self.proc = None
        self.thread = None
        self.stop_flag = False

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            h = pynvml.nvmlDeviceGetHandleByPciBusId(self.pci.encode() if hasattr(self.pci, 'encode') else self.pci) \
                if self.pci else pynvml.nvmlDeviceGetHandleByIndex(self.idx)
            mx = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            names = {'hw_slowdown': pynvml.nvmlClocksEventReasonHwSlowdown, 'hw_thermal_slowdown': pynvml.nvmlClocksEventReasonHwThermalSlowdown,
                     'sw_thermal_slowdown': pynvml.nvmlClocksEventReasonSwThermalSlowdown, 'sw_power_cap': pynvml.nvmlClocksEventReasonSwPowerCap,
                     'hw_power_brake': pynvml.nvmlClocksEventReasonHwPowerBrakeSlowdown}

            def poll():
                while not self.stop_flag:
                    try:
                        t = time.time()
                        sm = float(pynvml.nvmlDeviceGetClockInfo(h, pynvml.NVML_CLOCK_SM))
                        pw = pynvml.nvmlDeviceGetPowerUsage(h) / 1000.0
                        mask = pynvml.nvmlDeviceGetCurrentClocksEventReasons(h)
                        self.samples.append((t, sm, mx, pw, {n for n, bit in names.items() if mask & bit}))
                    except Exception:
                        pass
                    time.sleep(0.005)
            self.thread = threading.Thread(target=poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.idx), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '20'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        import datetime
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for line in self.proc.stdout:
            f = [x.strip() for x in line.strip().split(',')]
            if len(f) < 9:
                continue
            ts = time.time()
            try:
                ts = datetime.datetime.strptime(f[0], '%Y/%m/%d %H:%M:%S.%f').timestamp()
            except ValueError:
                pass
            try:
                self.samples.append((ts, float(f[1]), float(f[2]), float(f[3]),
                                     {n for n, v in zip(names, f[5:9]) if v.lower().startswith('active')}))
            except ValueError:
                continue

    def stop(self, t0=None, t1=None):
        self.stop_flag = True
        if self.thread is not None:
            self.thread.join(timeout=1)
            source = 'nvml'
        elif self.proc:
            time.sleep(0.05)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
            source = 'nvidia-smi'
        else:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['unavailable']}
        rows = [r for r in self.samples if t0 is None or (t0 - 0.02 <= r[0] <= t1 + 0.02)]
        reasons = set()
        for r in rows:
            reasons |= r[4]
        return {'sm_mhz': float(np.median([r[1] for r in rows])) if rows else None,
                'sm_min_mhz': min(r[1] for r in rows) if rows else None,
                'sm_max_mhz': max(r[2] for r in rows) if rows else None,
                'power_w_max': max(r[3] for r in rows) if rows else None, 'samples': len(rows), 'reasons': sorted(reasons),
                'source': source}


# ------------------------------------------------------------------------------ reference arm
# Each pool worker generates its clip ONCE (first call with that key) and keeps it; the timed part
# of a call is only the reference's OpenCV calls (optical_flow_kernel_cpu.cpp:36-41 +
# flow_histogram_kernel_cpu.cpp:27-54, or histogram_kernel_cpu.cpp:25-44).
_CLIPS = {}


def _cpu_worker(args):
    kind, h, w, seed, n_units = args
    import cv2
    cv2.setNumThreads(1)   # Farneback does not scale with OpenCV threads: one worker per core
    from oracle import cv2_ops
    from scannertools_b200 import synth
    key = (kind, h, w, seed, n_units)
    if key not in _CLIPS:
        _CLIPS.clear()
        _CLIPS[key] = (synth.textured_clip(seed, n_units + 1, h, w) if kind == 'flow' else synth.noise_clip(seed, 2, h, w))
    clip = _CLIPS[key]
    t0 = time.perf_counter()
    if kind == 'flow':
        for i in range(n_units):
            cv2_ops.flow_histogram(cv2_ops.optical_flow(clip[i], clip[i + 1]))
    else:
        for i in range(n_units):
            cv2_ops.histogram(clip[i & 1])
    return n_units, time.perf_counter() - t0


def cpu_pass(pool, cores, kind, h, w, units_total):
    """One step of the CPU arm: `units_total` pairs (or frames) spread over `cores` workers.
    Returns (units, wall seconds around the map, per-worker inner seconds)."""
    share = [units_total // cores + (1 if c < units_total % cores else 0) for c in range(cores)]
    jobs = [(kind, h, w, 100 + c, share[c]) for c in range(cores) if share[c] > 0]
    t0 = time.perf_counter()
    res = pool.map(_cpu_worker, jobs, chunksize=1)
    wall = time.perf_counter() - t0
    return sum(r[0] for r in res), wall, [r[1] for r in res], [r[0] for r in res]


def host_cores():
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return os.cpu_count() or 1


def run_reference(args):
    """The reference's own CPU implementation of the path: the OpenCV calls its C++ wrappers
    make (oracle/cv2_ops.py), one worker process per host core on disjoint frame pairs; a step is
    the same `--pairs` 1080p pairs as one rank's step of our arm."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import multiprocessing as mp
    cores = host_cores()
    ctx = mp.get_context('spawn')
    P = args.pairs
    # a step = the same number of pairs on every worker (no imbalance): per = round(P / cores) >= 1
    per = max(1, int(round(P / float(cores))))
    units_step = per * cores
    with ctx.Pool(cores) as pool:
        # warm-up: spawns the workers, generates each worker's clip (untimed), pages OpenCV in
        for _ in range(max(args.warmup, 1)):
            cpu_pass(pool, cores, 'flow', 1080, 1920, units_step)
        frames, wall, busy, rate_sum = 0, 0.0, 0.0, 0.0
        for _ in range(args.steps):
            f, wl, inner, units = cpu_pass(pool, cores, 'flow', 1080, 1920, units_step)
            frames += f
            wall += wl                       # around pool.map: includes IPC and the slowest worker
            busy += max(inner)               # the slowest worker's own timer around its OpenCV calls
            rate_sum += sum(u / t for u, t in zip(units, inner))
    # value: the steady-state rate of the box's cores = sum over workers of (pairs / that worker's own time around
    # its OpenCV calls), i.e. no per-step barrier and no IPC charged to the reference (the most favourable reading)
    fps = rate_sum / args.steps
    import cv2
    sample = ('%d steps x %d 1080p pairs (%d per worker) over %d worker processes (cv2 %s: 2 x cvtColor + Farneback(3,0.5,15,3,5,1.2) + '
              'cartToPolar + 2 x calcHist per pair; cv2.setNumThreads(1) per worker; clips generated once, outside the timed calls)'
              % (args.steps, units_step, per, cores, cv2.__version__))
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': fps, 'unit': 'frames/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * units_step / fps,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args),
        'cpu_baseline': {'value': fps, 'unit': 'frames/s', 'cores': cores, 'kind': 'port', 'sample': sample,
                         'pairs_per_step_run': units_step,
                         'frames_per_s_slowest_worker_bound': frames / busy, 'frames_per_s_wall_around_pool_map': frames / wall},
        'e2e': {'value': fps, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line))


METRIC = '1080p Farneback OpticalFlow + FlowHistogram throughput'


def workload_config(args):
    """Identical in both arms (the driver compares the two dicts)."""
    return {'workload': 'C3: 1080p (1920x1080) Farneback optical flow (3 levels, winsize 15, 3 iters, polyN 5) + '
                        'FlowHistogram, one synthetic textured clip, frame-range sharded (pairs_per_step pairs per GPU)',
            'pairs_per_step': args.pairs, 'batch_pairs': args.batch, 'frame': '1920x1080x3 u8',
            'l2_policy': 'inputs larger than L2: ring of %d distinct frames (%.0f MB) + %.0f MB of flow output per step'
                         % (args.pairs + 1, (args.pairs + 1) * 6.2208, args.pairs * 16.5888),
            'parallelism': 'frame-range x%d, no collective' % args.gpus}


# ------------------------------------------------------------------------------ our arm
def run_ours(args):
    import torch
    import torch.distributed as dist
    from scannertools_b200 import _lib, ops, sharding, synth
    import ctypes as C

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device; scannertools_b200 has no CPU fallback '
                         '(use --impl reference for the CPU arm)')
    torch.cuda.set_device(local)
    # feeder threads and pinned staging buffers on the GPU's own socket (no-op when the box
    # does not expose the topology); STB_NO_NUMA_BIND=1 switches it off for A/B runs
    numa_node = None if os.environ.get('STB_NO_NUMA_BIND') else sharding.bind_to_gpu_numa_node(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    lib = _lib.load()
    H, W = 1080, 1920
    P, B = args.pairs, args.batch
    assert P % B == 0, '--pairs must be a multiple of --batch'

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce_max(vals):
        t = torch.tensor(vals, dtype=torch.float64, device='cuda')
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.tolist()

    # ---- ONE seeded clip of world*P + 1 frames, frame-range sharded: this rank generates and owns
    # frames [p0, p1] (pairs [p0, p1) + the halo frame, which is also the next rank's first frame)
    n_frames = world * P + 1
    (p0, p1), (fa, fb) = sharding.pair_range(n_frames, rank, world)
    assert (p1 - p0, fb - fa) == (P, P + 1)
    clip = synth.textured_clip(C3_SEED, fb - fa, H, W, t0=fa, total=n_frames)
    host = torch.from_numpy(clip).pin_memory()
    d_frames = host.cuda(non_blocking=True)
    torch.cuda.synchronize()
    of = ops.OpticalFlow(W, H, max_batch=B)
    d_flow = torch.empty((P, H, W, 2), dtype=torch.float32, device='cuda')
    d_fh = torch.empty((P, 2, 64), dtype=torch.int32, device='cuda')
    frame_ptrs = [d_frames[i].data_ptr() for i in range(P + 1)]
    flow_ptrs = [d_flow[i].data_ptr() for i in range(P)]
    stream = torch.cuda.current_stream()
    sp = C.c_void_p(stream.cuda_stream)

    def step_device():
        for b0 in range(0, P, B):
            ft = _lib.ptr_table(frame_ptrs[b0:b0 + B + 1])
            ot = _lib.ptr_table(flow_ptrs[b0:b0 + B])
            _lib.check(lib.stb_farneback_run_hist(of._h, ft, B, ot, C.c_void_p(d_fh[b0].data_ptr()), sp), lib)

    pr = torch.cuda.get_device_properties(local)
    sampler = ClockSampler(local, '%08x:%02x:%02x.0' % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id))
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step_device()
    barrier()
    lib.stb_farneback_profile(of._h, 1)
    l0 = lib.stb_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    wall0 = time.time()
    ev0.record()
    for _ in range(args.steps):
        step_device()
    ev1.record()
    barrier()
    wall1 = time.time()
    t_dev = ev0.elapsed_time(ev1) * 1e-3
    launches = lib.stb_launch_count() - l0
    clocks = sampler.stop(wall0, wall1) if rank == 0 else None
    ms_total, nl, npi = C.c_double(), C.c_longlong(), C.c_longlong()
    _lib.check(lib.stb_farneback_profile_read(of._h, C.byref(ms_total), C.byref(nl), C.byref(npi)), lib)
    lib.stb_farneback_profile(of._h, 0)
    fh_dev = d_fh.cpu().numpy().copy()
    flow_seam = (d_flow[0].cpu().numpy().copy(), d_flow[P - 1].cpu().numpy().copy())
    if args.dump_outputs:
        pix = torch.from_numpy(dump_pixels(H * W, world * P)).cuda()
        flow_sample = d_flow.view(P, H * W, 2)[:, pix].cpu().numpy()
    del d_flow

    # ---- e2e: host frames in (pinned), flow histograms out (pinned), through the host-buffer C ABI.
    # Every step uploads its frames and reads its result back; two calls are kept in flight
    # (stb_pipe_flow_async / stb_pipe_wait: submit step i+1, then wait for and read step i), the way a
    # streaming caller drives it, so one step's uploads hide behind the previous step's kernels.
    pipe = ops.Pipe(W, H, max_batch=B, want_flow=True)
    res = [torch.empty((P, 2, 64), dtype=torch.int32).pin_memory() for _ in range(2)]

    def e2e_loop(steps, flow_bufs=None):
        chk = 0
        prev = pipe.flow_async(host, res[0], flow_out=flow_bufs[0] if flow_bufs else None)
        for i in range(1, steps):
            cur = pipe.flow_async(host, res[i & 1], flow_out=flow_bufs[i & 1] if flow_bufs else None)
            pipe.wait(prev)
            chk += int(res[(i - 1) & 1][0, 0, 0])       # the step's result is read on the host
            prev = cur
        pipe.wait(prev)
        chk += int(res[(steps - 1) & 1][0, 0, 0])
        torch.cuda.synchronize()
        return chk

    for _ in range(max(1, args.warmup // 2)):
        pipe.wait(pipe.flow_async(host, res[0]))
    fh_e2e = res[0].numpy().copy()
    barrier()
    t0 = time.perf_counter()
    e2e_loop(args.steps)
    t_e2e = time.perf_counter() - t0
    barrier()
    assert np.array_equal(fh_e2e, fh_dev), 'e2e and device-resident paths disagree'
    assert np.array_equal(res[(args.steps - 1) & 1].numpy(), fh_dev), 'asynchronous e2e result differs'

    # ---- e2e of the OpticalFlow op itself: the flow FRAMES come back too (16.6 MB per frame D2H)
    t_e2e_flow, steps_ff = float('nan'), max(2, min(args.steps, 6))
    if not args.no_flow_frames:
        fbufs = [torch.empty((P, H, W, 2), dtype=torch.float32).pin_memory() for _ in range(2)]
        e2e_loop(2, fbufs)
        barrier()
        t0 = time.perf_counter()
        e2e_loop(steps_ff, fbufs)
        t_e2e_flow = time.perf_counter() - t0
        barrier()
        last = fbufs[(steps_ff - 1) & 1]
        assert np.array_equal(last[0].numpy(), flow_seam[0]) and np.array_equal(last[P - 1].numpy(), flow_seam[1]), \
            'e2e flow frames differ from the device-resident path'
        del fbufs, last

    # ---- the ceiling of the host feed: the same H2D bytes per step with no kernels at all, every
    # rank at once (one copy stream per GPU, then split over two streams)
    copy_steps = 5
    halves = (P + 1) // 2
    s2 = [torch.cuda.Stream(), torch.cuda.Stream()]

    def copy_one():
        d_frames.copy_(host, non_blocking=True)

    def copy_two():
        cur = torch.cuda.current_stream()
        for i, (a, b) in enumerate(((0, halves), (halves, P + 1))):
            s2[i].wait_stream(cur)
            with torch.cuda.stream(s2[i]):
                d_frames[a:b].copy_(host[a:b], non_blocking=True)
        for s in s2:
            cur.wait_stream(s)

    t_copy = []
    for fn in (copy_one, copy_two):
        fn()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(copy_steps):
            fn()
        b.record()
        barrier()
        t_copy.append(a.elapsed_time(b) * 1e-3 / copy_steps)

    # ---- max over ranks (timing scalars only; no data-path collective)
    t_dev, t_e2e, t_e2e_flow, t_copy1, t_copy2 = reduce_max([t_dev, t_e2e, t_e2e_flow, t_copy[0], t_copy[1]])
    stats = torch.tensor([float(launches), ms_total.value, float(nl.value), float(npi.value)], dtype=torch.float64, device='cuda')
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)
    launches_all, ms_iter_all, nl_all, npi_all = stats.tolist()

    # ---- per-frame outputs concatenated on the host in frame order; rank 0 re-computes every pair
    # that touches a shard seam ALONE (its own handle, frames generated from the seed) and compares
    all_fh = sharding.gather_frame_outputs(fh_dev, world * P, rank, world)
    if args.dump_outputs:
        all_flow_sample = sharding.gather_frame_outputs(flow_sample, world * P, rank, world)
        if rank == 0:
            write_dump(args.dump_outputs, {'flow_hist': all_fh, 'flow_sample': all_flow_sample})
    shard_check = None
    if rank == 0:
        seams = sorted({q for r in range(1, world) for q in (r * P - 1, r * P)} | {0, world * P - 1})
        solo = ops.OpticalFlow(W, H, max_batch=1)
        for q in seams:
            fr = torch.from_numpy(synth.textured_clip(C3_SEED, 2, H, W, t0=q, total=n_frames)).cuda()
            _, fh1 = solo.execute_with_histogram(fr, want_flow=False)
            assert np.array_equal(fh1.cpu().numpy()[0], all_fh[q]), 'sharded result differs from the single-GPU result at pair %d' % q
        solo.close()
        shard_check = {'clip_frames': n_frames, 'pairs_checked_alone_on_rank0': seams, 'ok': True}
    del d_frames, host

    extra = {}
    if not args.no_extra:
        extra = extra_workloads(torch, dist, ops, lib, args, rank, world, barrier, reduce_max)
    cpu_base = None
    if rank == 0 and world == 1 and not args.no_cpu:
        cpu_base = cpu_baseline()

    if rank == 0:
        peak, peak_kind = measured_peaks()
        total_frames = world * args.steps * P
        pairs_per_launch = npi_all / nl_all if nl_all else 0.0    # one launch covers a whole batch of pairs
        iter_bytes = ITER_BYTES_PER_PX * H * W * pairs_per_launch
        avg_iter_s = (ms_iter_all / nl_all) * 1e-3 if nl_all else float('nan')
        achieved = iter_bytes / avg_iter_s / 1e9 if nl_all else None
        value = total_frames / t_dev
        traffic_pp, traffic_src = ncu_traffic()
        h2d = world * (P + 1) * H * W * 3
        line = {
            'metric': METRIC, 'value': value, 'unit': 'frames/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': 1e3 * t_dev / args.steps, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': workload_config(args),
            'host': {'numa_node_rank0': numa_node, 'cores': host_cores()},
            'hbm_roofline_frac_whole_op': (FLOW1080_BYTES + FLOWHIST1080_BYTES) * value / world / (peak * 1e9),
            'roofline': {'bound': 'hbm', 'kernel': 'iter15_win_kernel (level-0 fused box-sum / 2x2 solve / update-matrices iteration: TMA-staged M tiles, flow-compensated R1 window in shared memory)',
                         'achieved': achieved, 'peak': peak, 'peak_kind': peak_kind, 'unit': 'GB/s',
                         'frac': (achieved / peak) if achieved else None,
                         'bytes_per_launch': iter_bytes, 'pairs_per_launch': pairs_per_launch, 'avg_launch_us': avg_iter_s * 1e6,
                         'launches_timed': int(nl_all),
                         'share_of_step': (ms_iter_all * 1e-3 / world) / t_dev if t_dev else None,
                         'traffic': traffic_pp * pairs_per_launch if traffic_pp else None,
                         'traffic_source': traffic_src},
            'e2e': {'value': total_frames / t_e2e, 'unit': 'frames/s',
                    'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': world * P * 512, 'ms_per_step': 1e3 * t_e2e / args.steps,
                    'api': 'stb_pipe_flow_async + stb_pipe_wait: pinned host frames -> flow HISTOGRAMS only (the shipped '
                           'OpticalFlow -> FlowHistogram pipeline; the flow frames are not materialised -- see e2e_flow_frames), '
                           'two calls in flight',
                    'copy_only': {'what': 'the same H2D bytes per step from the same pinned buffers with no kernels, all ranks at once '
                                          '(ceiling of the host feed at this N)',
                                  'frames_per_s': world * P / t_copy1, 'gb_per_s_per_gpu': h2d / world / t_copy1 / 1e9,
                                  'two_streams_frames_per_s': world * P / t_copy2,
                                  'two_streams_gb_per_s_per_gpu': h2d / world / t_copy2 / 1e9,
                                  'e2e_over_ceiling': (total_frames / t_e2e) / (world * P / min(t_copy1, t_copy2))}},
            'e2e_flow_frames': None if args.no_flow_frames else {
                'value': world * steps_ff * P / t_e2e_flow, 'unit': 'frames/s', 'steps': steps_ff,
                'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': world * P * (H * W * 8 + 512),
                'ms_per_step': 1e3 * t_e2e_flow / steps_ff,
                'api': 'stb_pipe_flow_async with h_flow: pinned host frames -> flow frames (H x W x 2 f32) + flow histograms'},
            'gpu_launches': int(launches_all),
            'shard_check': shard_check,
            'clocks': clocks,
            'cpu_baseline': cpu_base,
            'extra': extra,
        }
        print(json.dumps(line))
    of.close()
    pipe.close()
    if world > 1:
        dist.destroy_process_group()


def extra_workloads(torch, dist, ops, lib, args, rank, world, barrier, reduce_max):
    """The other workloads of the metric, run by EVERY rank on its shard; times are max-reduced and
    values are whole-job aggregates (weak scaling: per-GPU work fixed)."""
    from scannertools_b200 import sharding, shot_detection, synth
    peak, _ = measured_peaks()
    out = {}

    def time_dev(fn, iters, warm=3):
        for _ in range(warm):
            fn()
        barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(iters):
            fn()
        b.record()
        barrier()
        return reduce_max([a.elapsed_time(b) * 1e-3 / iters])[0]

    def roof(units, bytes_per_unit, t):
        ach = units * bytes_per_unit / t / 1e9 / world
        return {'bound': 'hbm', 'achieved': ach, 'peak': peak, 'unit': 'GB/s per GPU', 'frac': ach / peak}

    # ---- C4: 4K RGB histogram + frame-difference shot scoring on ONE clip of world*32 frames, frame-range
    # sharded; hard cuts planted inside shard 0 and exactly ON every shard seam.  Each rank reads one halo
    # frame (the last frame of the previous shard) for the first score of its range.
    n4k = C4_FRAMES
    total4k = world * n4k
    cuts = sorted({11, 23} | {r * n4k for r in range(1, world)})
    f0, f1 = sharding.frame_range(total4k, rank, world)
    a0 = max(f0 - 1, 0)
    host4k = torch.from_numpy(synth.cut_clip_range(C4_SEED, total4k, 2160, 3840, a0, f1, cuts)).pin_memory()
    fr_all = host4k.cuda()
    halo = fr_all[0:1] if f0 > 0 else None
    fr = fr_all[f0 - a0:]
    state = {}

    # the halo frame (last frame of the previous shard) is needed ONCE per shard, for the first score of the range: its
    # histogram is computed before the timed loop, as a streaming run over a long shard would carry the previous
    # batch's last histogram along -- a timed step is this rank's 32 frames: histograms + scores against prev_hist
    halo_hist = ops.histogram(halo)[0] if halo is not None else None

    def c4_step():
        state['h'] = ops.histogram(fr)
        state['S'] = ops.shot_scores(state['h'], prev_hist=halo_hist)
    t = time_dev(c4_step, 20)
    S_local = state['S'].cpu().numpy()
    pipe = ops.Pipe(3840, 2160, max_batch=7)
    pipe.histogram(host4k[f0 - a0:])
    barrier()
    t0 = time.perf_counter()
    for _ in range(3):
        pipe.histogram(host4k[f0 - a0:])
    te = reduce_max([(time.perf_counter() - t0) / 3])[0]
    barrier()
    pipe.close()
    bounds, S_all = sharding.sharded_shot_detection(fr, total4k, rank, world, ops.histogram,
                                                    lambda h, p: ops.shot_scores(h, prev_hist=p).cpu().numpy(),
                                                    halo_frame=halo)
    check = None
    if rank == 0:
        assert np.array_equal(S_all[f0:f1], S_local)
        assert bounds == cuts, ('sharded shot detection', bounds, cuts)
        for c in [r * n4k for r in range(1, world)]:           # every seam frame re-scored alone on rank 0
            two = torch.from_numpy(synth.cut_clip_range(C4_SEED, total4k, 2160, 3840, c - 1, c + 1, cuts)).cuda()
            assert int(ops.shot_scores(ops.histogram(two))[1]) == int(S_all[c]), ('seam score', c)
        check = {'frames': total4k, 'planted_cuts': cuts, 'boundaries_found': bounds, 'ok': True}
    out['hist4k'] = {'workload': 'C4: 3840x2160 RGB histogram (16 bins/channel) + shot scores, one clip of %d frames '
                                 'frame-range sharded x%d (%d frames per GPU and step; the halo frame histogram of a shard is computed once, outside the timed steps), cuts on the shard seams' % (total4k, world, n4k),
                     'value': total4k / t, 'unit': 'frames/s', 'ms_per_step': t * 1e3, 'roofline': roof(total4k, HIST4K_BYTES, t),
                     'e2e': {'value': total4k / te, 'unit': 'frames/s', 'h2d_bytes_per_step': total4k * 3840 * 2160 * 3,
                             'd2h_bytes_per_step': total4k * 196},
                     'shard_check': check}
    # HSV variant of the shot-detection histogram (old/histograms.py:32-36): fused ConvertToHSV ->
    # Histogram against the two-op chain (ConvertColor writes the HSV frame, Histogram reads it back)
    th = time_dev(lambda: ops.shot_scores(ops.histogram(fr, hsv='COLOR_RGB2HSV')), 10)
    t2 = time_dev(lambda: ops.shot_scores(ops.histogram(ops.convert_color(fr, 'COLOR_RGB2HSV'))), 3, warm=1)
    out['hsvhist4k'] = {'workload': '3840x2160 fused RGB->HSV + histogram (16 bins/channel) + shot scores, %d frames per GPU and step' % n4k,
                        'value': total4k / th, 'unit': 'frames/s', 'ms_per_step': th * 1e3, 'roofline': roof(total4k, HIST4K_BYTES, th),
                        'unfused_two_op_frames_per_s': total4k / t2}
    del fr, fr_all, halo, host4k, state
    # ---- stand-alone FlowHistogram op on 1080p flow frames
    ff = torch.from_numpy(np.stack([synth.textured_flow_field(5 + i, 1080, 1920) for i in range(4)])).cuda().repeat(8, 1, 1, 1)
    tf = time_dev(lambda: ops.flow_histogram(ff), 10)
    out['flowhist1080'] = {'workload': 'FlowHistogram op alone on %d 1080p flow frames per GPU and step' % ff.shape[0],
                           'value': world * ff.shape[0] / tf, 'unit': 'frames/s', 'ms_per_step': tf * 1e3,
                           'roofline': roof(world * ff.shape[0], FLOWHIST1080_BYTES, tf)}
    del ff
    # ---- C2: 640x480 Farneback at 16 and 64 pairs per call
    out['flow480'] = {}
    for n480 in (16, 64):
        clip = synth.textured_clip(2, n480 + 1, 480, 640)
        d = torch.from_numpy(clip).cuda()
        of = ops.OpticalFlow(640, 480, max_batch=n480)
        o = torch.empty((n480, 480, 640, 2), dtype=torch.float32, device='cuda')
        t = time_dev(lambda: of.execute(d, out=o), 10)
        of.close()
        out['flow480']['pairs%d' % n480] = {
            'workload': 'C2: 640x480 Farneback (3 levels, winsize 15, 3 iters), %d pairs per call and GPU' % n480,
            'value': world * n480 / t, 'unit': 'frames/s', 'ms_per_step': t * 1e3, 'roofline': roof(world * n480, FLOW480_BYTES, t)}
        del d, o
    # ---- C5: 64 concurrent 720p streams on 8 GPUs = 8 whole streams per GPU (sharding.stream_assignment;
    # per-stream state never crosses devices), each with its own OpticalFlow handle, mixed
    # OpticalFlow+FlowHistogram and RGB Histogram work, round-robin batch by batch
    n_streams, fps_batch = C5_STREAMS, C5_BATCH
    mine = sharding.stream_assignment(n_streams * world, world)[rank]
    clips = [torch.from_numpy(synth.textured_clip(300 + sid, fps_batch + 1, 720, 1280)).cuda() for sid in mine]
    handles = [ops.OpticalFlow(1280, 720, max_batch=fps_batch) for _ in mine]

    # every video stream runs on its own CUDA stream (a 64-stream deployment has one evaluator per stream): the
    # coarse, latency-bound pyramid levels of one stream overlap the fine levels of another
    cstreams = [torch.cuda.Stream() for _ in mine]

    def c5_step():
        cur = torch.cuda.current_stream()
        for k in range(len(mine)):
            cstreams[k].wait_stream(cur)
            with torch.cuda.stream(cstreams[k]):
                handles[k].execute_with_histogram(clips[k], want_flow=False, stream=cstreams[k])
                ops.histogram(clips[k][:fps_batch], stream=cstreams[k])
        for k in range(len(mine)):
            cur.wait_stream(cstreams[k])
    t = time_dev(c5_step, 5, warm=2)

    def c5_step_serial():
        for k in range(len(mine)):
            handles[k].execute_with_histogram(clips[k], want_flow=False)
            ops.histogram(clips[k][:fps_batch])
    t_serial = time_dev(c5_step_serial, 5, warm=1)
    for hnd in handles:
        hnd.close()
    frames = world * n_streams * fps_batch
    out['c5_mixed_720p'] = {'workload': 'C5: %d concurrent 1280x720 streams (%d per GPU, whole streams pinned to GPUs), OpticalFlow+FlowHistogram '
                                        'and RGB Histogram, %d frames per stream per step' % (n_streams * world, n_streams, fps_batch),
                            'value': frames / t, 'unit': 'frames/s', 'ms_per_step': t * 1e3, 'roofline': roof(frames, C5_BYTES, t),
                            'one_cuda_stream_for_all_frames_per_s': frames / t_serial}
    return out if rank == 0 else {}


def cpu_baseline():
    """Reference CPU ops (cv2) on this box's host cores, in a child process that never touches
    CUDA (forking/spawning workers from a process with a live CUDA context is avoided)."""
    try:
        out = subprocess.run([sys.executable, os.path.abspath(__file__), '--cpu-baseline-child'], capture_output=True,
                             text=True, timeout=300)
        for line in out.stdout.splitlines():
            if line.startswith('{'):
                return json.loads(line)
        return {'error': (out.stderr or 'no output')[-300:]}
    except Exception as e:  # noqa: BLE001
        return {'error': repr(e)}


def cpu_baseline_child():
    import multiprocessing as mp
    cores = host_cores()
    ctx = mp.get_context('spawn')
    per = 2
    with ctx.Pool(cores) as pool:
        cpu_pass(pool, cores, 'flow', 1080, 1920, cores * per)       # spawn, clip generation, page-in (untimed)
        frames, wall, inner, units = cpu_pass(pool, cores, 'flow', 1080, 1920, cores * per)
        cpu_pass(pool, cores, 'hist', 2160, 3840, cores * 8)
        hframes, hwall, _, _ = cpu_pass(pool, cores, 'hist', 2160, 3840, cores * 8)
    import cv2
    print(json.dumps({'value': sum(u / t for u, t in zip(units, inner)), 'unit': 'frames/s', 'cores': cores, 'kind': 'port',
                      'sample': '%d workers x %d 1080p pairs: cv2 %s cvtColor+Farneback(3,0.5,15,3,5,1.2)+cartToPolar+2xcalcHist, '
                                'cv2.setNumThreads(1) per worker, clips generated outside the timed calls; value = sum of the '
                                "workers' own rates" % (cores, per, cv2.__version__),
                      'frames_per_s_wall_around_pool_map': frames / wall,
                      'hist4k_frames_per_s': hframes / hwall}))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=30)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--pairs', type=int, default=64, help='frame pairs per step and GPU')
    ap.add_argument('--batch', type=int, default=32, help='pairs per C-ABI batch call')
    ap.add_argument('--no-extra', action='store_true')
    ap.add_argument('--no-cpu', action='store_true')
    ap.add_argument('--no-flow-frames', action='store_true', help='skip the e2e_flow_frames figure (2 GB of pinned memory)')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='after the timed steps, write what the last one computed (flow histograms of every pair, a fixed '
                         'seeded sample of the flow frames) as DIR/<name>.npy, float32 or float64, at most 64 MB')
    ap.add_argument('--cpu-baseline-child', action='store_true', help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.cpu_baseline_child:
        cpu_baseline_child()
        return
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of our arm (--impl ours)')
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == 'reference':
        run_reference(args)
    else:
        run_ours(args)


if __name__ == '__main__':
    main()
