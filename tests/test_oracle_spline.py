"""CPU tests: the spline part of the semi-Lagrangian oracle (oracle/spline_oracle.c --
scipy.ndimage.map_coordinates for orders 0 and 2..5 with prefilter) is pinned bit for bit against
the scipy binary; the extrapolator with interp_order 0 / 3 against the reference's stored
outputs (tests/test_oracle_sl.py, SPLINE_CASES) and on 60 randomised calls
(tests/golden/reference_golden.npz)."""
import warnings

import fingerprint as fp
import numpy as np
import pytest
import reference_cases as rc
from conftest import assert_bits_equal
from scipy import ndimage as ndi

from oracle import semilagrangian as ora

SHAPES = [(9, 13), (1, 7), (5, 1), (2, 2), (1, 1), (3, 40), (64, 80)]


@pytest.mark.parametrize("order", [2, 3, 4, 5])
@pytest.mark.parametrize("shape", SHAPES)
def test_prefilter_matches_scipy_bitwise(shape, order):
    rng = np.random.default_rng(shape[0] * 100 + shape[1])
    a = rng.standard_normal(shape) * 10
    assert_bits_equal(ora.spline_filter(a, order, "constant"),
                      ndi.spline_filter(a, order, output=np.float64, mode="constant"), "mirror")
    # mode "nearest": 12-sample edge padding + the reflect boundary (ndimage._prepad_for_spline_filter)
    p = np.pad(a, 12, mode="edge")
    assert_bits_equal(ora.spline_filter(p, order, "nearest"),
                      ndi.spline_filter(p, order, output=np.float64, mode="nearest"), "reflect")


@pytest.mark.parametrize("order", [0, 2, 3, 4, 5])
@pytest.mark.parametrize("mode", ["constant", "nearest"])
@pytest.mark.parametrize("shape", SHAPES)
def test_samples_match_scipy_bitwise(shape, mode, order):
    m, n = shape
    rng = np.random.default_rng(m * 1000 + n * 10 + order)
    a = rng.standard_normal(shape)
    k = 1500
    cy = rng.uniform(-40, m + 40, k)
    cx = rng.uniform(-40, n + 40, k)
    cy[:300] = rng.uniform(-3, m + 2, 300)             # mostly inside / just outside
    cx[:300] = rng.uniform(-3, n + 2, 300)
    cy[300:400] = rng.integers(-2, m + 2, 100)         # exact integers and half-integers
    cx[300:400] = rng.integers(-2, n + 2, 100)
    cy[400:450] = rng.integers(-2, m + 2, 50) + 0.5
    cx[450:500] = rng.integers(-2, n + 2, 50) + 0.5
    cy[500:520], cx[520:540], cy[540:560], cx[560:580] = m - 1, n - 1, 0, 0   # the borders
    cy[580:585], cx[585:590], cy[590:595] = np.nan, np.inf, -np.inf           # non-finite
    cx[595:600] = 2.0 ** 62                                                   # huge but castable
    ref = ndi.map_coordinates(a, [cy, cx], order=order, mode=mode, cval=-7.5, prefilter=True)
    got = ora.map_coordinates_spline(a, [cy, cx], order, mode, -7.5)
    assert_bits_equal(got, ref, f"{shape} {mode} order {order}")


def test_float32_input_rounds_like_scipy():
    rng = np.random.default_rng(4)
    a = rng.standard_normal((20, 30)).astype(np.float32)
    cy, cx = rng.uniform(-2, 21, 500), rng.uniform(-2, 31, 500)
    for mode in ("constant", "nearest"):
        ref = ndi.map_coordinates(a, [cy, cx], order=3, mode=mode, cval=np.nan)
        got = ora.map_coordinates_spline(a, [cy, cx], 3, mode, np.nan)
        assert got.dtype == np.float32
        assert_bits_equal(got, ref, mode)


def test_extrapolate_spline_orders_against_live_reference(reference_golden):
    """60 small randomised calls (tests/golden/reference_cases.py) against the reference's stored
    outputs and error messages, bit for bit."""
    g = reference_golden
    warnings.simplefilter("ignore")
    for it, (P, V, ts, outval, kw) in enumerate(rc.spline_cases()):
        werr = g.get(f"spline/{it}/error")
        try:
            got, gerr = ora.extrapolate(P.copy(), V.copy(), ts, outval, **kw), None
        except ValueError as e:
            got, gerr = None, str(e)
        assert gerr == werr, (it, kw)
        if werr is None:
            got = got if isinstance(got, tuple) else (got,)
            assert f"spline/{it}/{len(got)}" not in g, (it, kw)
            for j, a in enumerate(got):
                fp.assert_same(a, g, f"spline/{it}/{j}", f"case {it} {kw}")
    with pytest.raises(RuntimeError) as e_ora:
        ora.extrapolate(np.ones((4, 4)), np.ones((2, 4, 4)), 1, interp_order=6)
    assert str(e_ora.value) == str(g["spline/order6_error"])
