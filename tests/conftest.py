import glob
import os
import sys

import numpy as np
import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), '..'))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, 'tests', 'golden')


def pytest_configure(config):
    config.addinivalue_line('markers', 'gpu: needs a CUDA device (run on the B200 box with -m gpu)')


class GoldenArrays(dict):
    """The arrays of one fixture, read from `<stem>.npz` and its parts `<stem>.<k>.npz`
    (tests/golden/make_golden.py splits a fixture so that no file exceeds 1 MB)."""

    @property
    def files(self):
        return list(self)


@pytest.fixture(scope='session')
def golden():
    def load(name):
        stem = os.path.join(GOLDEN, name[:-len('.npz')])
        out = GoldenArrays()
        for path in [stem + '.npz'] + sorted(glob.glob(glob.escape(stem) + '.[0-9]*.npz')):
            with np.load(path, allow_pickle=False) as z:
                for k in z.files:
                    assert k not in out, (path, k)
                    out[k] = z[k]
        return out
    return load


@pytest.fixture(scope='session')
def have_cv2():
    try:
        import cv2  # noqa: F401
        return True
    except Exception:
        return False


def epe(a, b):
    d = np.asarray(a, np.float64) - np.asarray(b, np.float64)
    return np.sqrt((d * d).sum(-1))


# rows appended by tests/test_gpu_parity.py::check_flow_hist_from_flow: FlowHistogram(GPU flow) vs cv2
# FlowHistogram(cv2 flow), printed as a table at the end of the run (and into gpurun_out/ when writable)
FLOWHIST_ROWS = []


def flowhist_table(rows):
    lines = ['FlowHistogram from GPU flow vs cv2 FlowHistogram of cv2 flow -- max per-bin |delta| (counts), pixels that changed bin,',
             'the bound asserted, and the same delta for the oracle restatement (restate.c, double accumulators) vs cv2',
             '%-38s %9s %9s | %5s %5s %6s | %9s %9s | %s' % ('input', 'EPE mean', 'EPE max', 'dMag', 'dAng', 'bound', 'moved mag', 'moved ang',
                                                              'restate-vs-cv2 dMag/dAng')]
    for r in rows:
        rs = '-' if r['r_dmag'] is None else '%d / %d' % (r['r_dmag'], r['r_dang'])
        lines.append('%-38s %9.2e %9.2e | %5d %5d %6s | %9d %9d | %s' % (str(r['tag']), r['epe_mean'], r['epe_max'], r['dmag'], r['dang'],
                                                                       r.get('bound', '-'), r['moved_mag'], r['moved_ang'], rs))
    return lines


def pytest_terminal_summary(terminalreporter):
    if not FLOWHIST_ROWS:
        return
    lines = flowhist_table(FLOWHIST_ROWS)
    terminalreporter.write_sep('=', 'FlowHistogram parity table')
    for ln in lines:
        terminalreporter.write_line(ln)
    try:
        out = os.path.join(ROOT, 'gpurun_out')
        if os.path.isdir(out):
            with open(os.path.join(out, 'flowhist_parity_table.txt'), 'w') as f:
                f.write('\n'.join(lines) + '\n')
    except OSError:
        pass
