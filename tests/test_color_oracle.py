"""Pins the numpy restatements of tests/color_restate.py to OpenCV: each one equals cv2.cvtColor on every 8-bit
input -- all 2^24 colours, with alpha varied over all 256 values on 4-channel inputs and every value on 1-channel
inputs.  The emulator and GPU tests of ConvertColor compare against these restatements."""
import numpy as np
import pytest

import color_restate as cr

cv2 = pytest.importorskip('cv2')


@pytest.fixture(scope='module')
def inputs():
    cache = {}

    def get(cin):
        if cin not in cache:
            cache[cin] = cr.cube_input(next(n for n, (i, _) in cr.CONVERSIONS.items() if i == cin))
        return cache[cin]
    return get


def test_cube_inputs_are_exhaustive(inputs):
    assert len(np.unique(inputs(3).reshape(-1, 3).view(np.dtype((np.void, 3))))) == 1 << 24
    c4 = inputs(4)
    assert np.array_equal(c4[..., :3], inputs(3)) and len(np.unique(c4[..., 3])) == 256
    assert np.array_equal(np.bincount(inputs(1).reshape(-1), minlength=256), np.full(256, 1 << 16))


@pytest.mark.parametrize('name', sorted(cr.CONVERSIONS))
def test_restatement_equals_cv2_on_every_input(inputs, name):
    cin, cout = cr.CONVERSIONS[name]
    x = inputs(cin)
    ref = cv2.cvtColor(x[..., 0] if cin == 1 else x, getattr(cv2, name))
    got = cr.convert(x, name)
    assert got.shape == ref.shape == (4096, 4096) + ((cout,) if cout > 1 else ())
    assert np.array_equal(got, ref), (name, int((got != ref).sum()))
