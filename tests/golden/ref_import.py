"""Imports the reference's own Python code for this path from a checkout of the reference
(scanner-research/scannertools) named by the environment variable SCANNERTOOLS_REFERENCE, behind a
minimal stub of `scannerpy`, so that goldens can be produced by the REFERENCE ITSELF where it is Python:

  * scannertools/shot_detection.py   -> shot_boundaries(config, histograms)
  * scannertools/types.py            -> histograms(buf, protobufs)

Used by make_golden.py only; the tests replay what it wrote (shot_reference.npz)."""
import importlib.util
import os
import sys
import types

REF = os.path.join(os.environ['SCANNERTOOLS_REFERENCE'], 'scannertools') if os.environ.get('SCANNERTOOLS_REFERENCE') else None


def available():
    return REF is not None and os.path.isfile(os.path.join(REF, 'shot_detection.py'))


def _stub_scannerpy():
    if 'scannerpy' in sys.modules and getattr(sys.modules['scannerpy'], '_stb_stub', False):
        return
    sp = types.ModuleType('scannerpy')
    sp._stb_stub = True

    def register_python_op(**kwargs):
        def deco(fn):
            fn._op_kwargs = kwargs
            return fn
        return deco
    sp.register_python_op = register_python_op
    st = types.ModuleType('scannerpy.types')
    st.Histogram = object
    stdlib = types.ModuleType('scannerpy.stdlib')
    poses = types.ModuleType('scannerpy.stdlib.poses')
    poses.Pose = object
    sys.modules.update({'scannerpy': sp, 'scannerpy.types': st, 'scannerpy.stdlib': stdlib, 'scannerpy.stdlib.poses': poses})


def load(name):
    _stub_scannerpy()
    spec = importlib.util.spec_from_file_location('stb_ref_' + name, os.path.join(REF, name + '.py'))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod
