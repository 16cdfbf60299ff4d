"""Scanner registration of this path's ops -- the drop-in for `import scannertools.shot_detection`
and `import scannertools.imgproc` of the reference.

Importing this module on a machine with the Scanner engine (`scannerpy`):
  * registers the Python op `ShotBoundaries(histograms: Sequence[Histogram]) -> Sequence[Any]` with
    `batch=BOUNDARY_BATCH`, exactly like /root/reference/scannertools/scannertools/shot_detection.py:11
    (`@scannerpy.register_python_op(name='ShotBoundaries', batch=BOUNDARY_BATCH)`), its body being
    scannertools_b200.shot_detection.shot_boundaries;
  * registers the kernel library `libscannertools_imgproc.so` (Histogram, OpticalFlow, FlowHistogram,
    FrameDifference, Resize, ConvertColor, Blur GPU kernels) the way scannertools/imgproc/__init__.py:1-3 does
    through scannertools_infra._register_module (scannertools_infra/__init__.py:90-100).

Without `scannerpy` the import fails loudly (there is nothing to register with); the ops themselves
stay usable through scannertools_b200.ops / .pipelines.
"""
import os
from typing import Any, Sequence

try:
    import scannerpy
    from scannerpy.types import Histogram
except ImportError as e:  # pragma: no cover - exercised through the stub in tests
    raise ImportError('scannertools_b200.scanner_register needs the Scanner engine (scannerpy); '
                      'use scannertools_b200.ops / pipelines directly without it') from e

from . import shot_detection as _sd

WINDOW_SIZE = _sd.WINDOW_SIZE
BOUNDARY_BATCH = _sd.BOUNDARY_BATCH


@scannerpy.register_python_op(name='ShotBoundaries', batch=BOUNDARY_BATCH)
def shot_boundaries(config, histograms: Sequence[Histogram]) -> Sequence[Any]:
    return _sd.shot_boundaries(config, histograms)


def register_imgproc():
    """scannertools_infra._register_module(..., 'scannertools_imgproc') for this build's library."""
    here = os.path.dirname(os.path.abspath(__file__))
    so_path = os.path.join(here, 'libscannertools_imgproc.so')
    proto_path = os.path.join(here, 'scannertools_imgproc_pb2.py')
    import scannerpy.op
    scannerpy.op.register_module(so_path, proto_path if os.path.isfile(proto_path) else None)
    return so_path


if hasattr(getattr(scannerpy, 'op', None), 'register_module') and not os.environ.get('STB_NO_IMGPROC_REGISTER'):
    register_imgproc()
