"""CPU tests of the host side of the device REPP steps (tscd_repp_prep / _tubelets / _emit): the ctypes mirrors of their
argument structs, the one Gaussian window a call uploads, and the box kind bits that stand for the dtype NumPy gives a
tubelet's boxes (the convolution keeps that dtype)."""
import ctypes
import os
import subprocess
import tempfile

import numpy as np
import pytest

from conftest import ROOT


def test_repp_struct_sizes_match_header():
    from tscd_b200 import _lib
    pairs = [("tscd_repp_prep_args", _lib.ReppPrepArgs), ("tscd_repp_tubelets_args", _lib.ReppTubeletsArgs),
             ("tscd_repp_emit_args", _lib.ReppEmitArgs)]
    body = "".join(f'printf("%zu\\n", sizeof({c}));' for c, _ in pairs)
    src = '#include <stdio.h>\n#include "tscd_b200.h"\nint main(){' + body + 'return 0;}'
    with tempfile.TemporaryDirectory() as d:
        c = os.path.join(d, "p.c")
        open(c, "w").write(src)
        exe = os.path.join(d, "p")
        subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), c, "-o", exe])
        sizes = [int(x) for x in subprocess.check_output([exe]).split()]
    assert sizes == [ctypes.sizeof(t) for _, t in pairs]


@pytest.mark.parametrize("std", [0.4 * 100 / 40, 0.9 * 100 / 40])
def test_window_slices_are_the_reference_windows(std):
    """Every tubelet length's window (recoordinate_tubelets_full: gaussian(2M-1), then w /= sum(w)) is the centred slice of the
    long window one call uploads, normalised by its own left-to-right sum."""
    from scipy.signal import windows
    from tscd_b200.repp import gaussian_window
    n = 400
    long = gaussian_window(n, std)
    for m in range(1, n + 1):
        want = windows.gaussian(2 * m - 1, std=std)
        got = long[n - m:n + m - 1]
        assert np.array_equal(got, want), m
        w = want.copy()
        w /= sum(w)
        s = 0.0
        for v in got:                                   # the device's sequential fp64 sum
            s += v
        assert np.array_equal(got / s, w), m


def test_box_kind_is_the_tubelet_dtype():
    """OR of the members' kind bits: 1 -> float32, 2 -> int64, anything else -> float64, as np.array of the boxes gives."""
    from tscd_b200.repp import box_kind
    f = np.float32
    boxes = [[f(1.5), f(2.5), f(30), f(40)], [0, f(2.5), f(30), f(40)], [f(1.5), 0, f(30), f(40)], [0, 0, 854, 480],
             [0, f(3), 854, f(20)], [1.5, 2.5, 30.0, 40.0], [np.int64(0), np.int64(0), np.int64(5), np.int64(5)],
             [np.float64(1.5), f(2.5), f(30), f(40)]]
    dt = {1: np.float32, 2: np.int64}
    for i in range(len(boxes)):
        for j in range(len(boxes)):
            members = [boxes[i], boxes[j], boxes[i]]
            k = 0
            for b in members:
                k |= box_kind(b)
            assert np.array(members).dtype == dt.get(k, np.float64), (boxes[i], boxes[j])
