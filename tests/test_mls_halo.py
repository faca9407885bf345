"""ppp_mls_halo / parallel.mls_halo (CPU, host code of the library): the float32 reach of an MLS radius plus the
margin for the exchange's double rounding (derivation in polishpathplanning_b200/csrc/mls.cu)."""
import math

import numpy as np
import pytest

from polishpathplanning_b200 import parallel

f32 = np.float32


def _sq(v):
    return f32(np.float64(v) * np.float64(v))     # exact in double, one rounding: fl32(v * v)


@pytest.mark.parametrize("radius", [15.0, 2.5, 0.1, 7.3, 1e-3, 1234.567, 3e9, 1.8e19])
@pytest.mark.parametrize("xmag", [0.0, 523.25, 1e6])
def test_reach_is_the_smallest_float_whose_square_reaches_r2(radius, xmag):
    r2 = f32(radius * radius)
    h = parallel.mls_halo(radius, xmag)
    t = f32(math.sqrt(float(r2)))
    # t: the smallest float with fl32(t * t) >= r2 (search from the halo downwards)
    margin = 2.0 ** -44 * (xmag + float(t) + 1.0)
    cand = f32(h - margin)
    for c in (np.nextafter(cand, f32(0)), cand, np.nextafter(cand, f32(np.inf))):
        if _sq(c) >= r2 and _sq(np.nextafter(c, f32(0))) < r2:
            t = c
            break
    else:
        raise AssertionError("no float reach near the halo %r" % h)
    assert h == float(t) + 2.0 ** -44 * (xmag + float(t) + 1.0)
    assert h > float(t)


def test_every_float_distance_below_the_reach_is_a_neighbour():
    """|dx| < t  <=>  fl32(dx^2) < r2 for the floats around t: a pair at dx = prev(t) is within the radius."""
    for radius in (15.0, 2.5, 0.3):
        r2 = f32(radius * radius)
        h = parallel.mls_halo(radius, 0.0)
        t = f32(h)
        while float(t) > h:
            t = np.nextafter(t, f32(0))
        t = np.nextafter(t, f32(np.inf)) if _sq(t) < r2 else t
        assert _sq(t) >= r2 and _sq(np.nextafter(t, f32(0))) < r2


@pytest.mark.parametrize("radius,xmag", [(0.0, 1.0), (-1.0, 1.0), (float("nan"), 1.0), (float("inf"), 1.0), (2e19, 1.0),
                                         (15.0, -1.0), (15.0, float("inf")), (15.0, float("nan"))])
def test_refused_arguments_give_nan(radius, xmag):
    assert math.isnan(parallel.mls_halo(radius, xmag))
