"""Builds scannertools_b200/libscannertools_b200.so from csrc/*.cu with nvcc for sm_100a.

In-tree on purpose: the .so is git-ignored but travels with the working tree to the GPU box.
"""
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(HERE, 'csrc')
OUT = os.path.join(HERE, 'libscannertools_b200.so')
OBJ = os.path.join(HERE, 'build')
SOURCES = ['common.cu', 'hist.cu', 'farneback.cu', 'pipe.cu', 'resize.cu', 'convert_color.cu', 'hist_hsv.cu', 'blur.cu']
NVCC_FLAGS = ['-gencode', 'arch=compute_100a,code=sm_100a', '-O3', '-lineinfo', '-std=c++17',
              '-Xcompiler', '-fPIC,-fvisibility=hidden', '-I', os.path.join(ROOT, 'include'), '-I', CSRC]


def find_nvcc():
    for c in (os.environ.get('NVCC'), shutil.which('nvcc'), '/usr/local/cuda/bin/nvcc'):
        if c and os.path.isfile(c):
            return c
    raise RuntimeError('nvcc not found: scannertools_b200 has no CPU fallback and cannot be built without CUDA')


def _newer(target, deps):
    if not os.path.isfile(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    nvcc = find_nvcc()
    os.makedirs(OBJ, exist_ok=True)
    headers = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(('.h', '.cuh'))]
    headers.append(os.path.join(ROOT, 'include', 'stb.h'))
    objs = []
    for s in SOURCES:
        src = os.path.join(CSRC, s)
        obj = os.path.join(OBJ, s[:-3] + '.o')
        objs.append(obj)
        if force or _newer(obj, [src] + headers):
            cmd = [nvcc] + NVCC_FLAGS + (['-Xptxas', '-v'] if verbose else []) + ['-c', src, '-o', obj]
            subprocess.check_call(cmd)
    if force or _newer(OUT, objs):
        subprocess.check_call([nvcc, '-shared', '-o', OUT] + objs + ['-gencode', 'arch=compute_100a,code=sm_100a'])
    return OUT


OPS_OUT = os.path.join(HERE, 'libscannertools_imgproc.so')
OPS_SOURCES = ['histogram_kernel_gpu.cpp', 'optical_flow_kernel_gpu.cpp', 'flow_histogram_kernel_gpu.cpp',
               'frame_difference_kernel_gpu.cpp', 'resize_kernel_gpu.cpp', 'convert_color_kernel_gpu.cpp', 'blur_kernel_gpu.cpp',
               'compat_runtime.cpp']


def build_scanner_ops(force=False, scanner_include=None):
    """Builds the Scanner kernel classes (csrc/scanner_ops) into libscannertools_imgproc.so -- the
    name the reference's `import scannertools.imgproc` registers.  Against the compat shim by
    default; pass the real Scanner include dir to build the drop-in (then compat_runtime.cpp,
    the shim's allocator + test harness, is left out)."""
    lib = build(force=force)
    nvcc = find_nvcc()
    cuda_home = os.path.dirname(os.path.dirname(nvcc))
    ops_dir = os.path.join(CSRC, 'scanner_ops')
    srcs = [os.path.join(ops_dir, s) for s in OPS_SOURCES if scanner_include is None or s != 'compat_runtime.cpp']
    deps = srcs + [lib] + [os.path.join(ops_dir, f) for f in os.listdir(ops_dir) if f.endswith('.h')]
    deps += [os.path.join(dp, f) for dp, _, fs in os.walk(os.path.join(CSRC, 'scanner_compat')) for f in fs]
    if not force and not _newer(OPS_OUT, deps):
        return OPS_OUT
    inc = scanner_include or os.path.join(CSRC, 'scanner_compat')
    cmd = ['g++', '-O2', '-std=c++14', '-fPIC', '-shared', '-fvisibility=hidden', '-I', inc, '-I', ops_dir,
           '-I', os.path.join(ROOT, 'include'), '-I', os.path.join(cuda_home, 'include'), '-o', OPS_OUT] + srcs + [
           '-L', HERE, '-l:libscannertools_b200.so', '-Wl,-rpath,$ORIGIN',
           '-L', os.path.join(cuda_home, 'lib64'), '-lcudart']
    if scanner_include is not None:
        cmd.insert(1, '-DSTB_SKIP_OP_DECLARATIONS')
    else:
        cmd.insert(1, '-DSTB_COMPAT_SHIM')    # the stb_shim_* test hooks exist only in the compat build
    subprocess.check_call(cmd)
    return OPS_OUT


if __name__ == '__main__':
    print(build(force='--force' in sys.argv, verbose='-v' in sys.argv))
    print(build_scanner_ops(force='--force' in sys.argv))
