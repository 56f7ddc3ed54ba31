"""CPU tests: the Proesmans oracle (oracle/proesmans_oracle.c, oracle/proesmans.py) is pinned
  * BIT FOR BIT against outputs of the reference SOURCE (pysteps/motion/proesmans.py +
    _proesmans.pyx) with the extension compiled without -ffast-math
    (tests/golden/gen_proesmans_strict_golden.py) -- ill-conditioned cases included;
  * to a tolerance against outputs of the extension compiled with the reference's own flags
    (-O3 -ffast-math, setup.py:27-28; tests/golden/gen_proesmans_golden.py): that build does not
    define its rounding, and the solver turns a flipped branch into a local change of up to a
    pixel, so only well-conditioned cases are compared closely;
  * against stored outputs of both builds on randomised calls
    (tests/golden/reference_proesmans_golden.npz, tests/golden/gen_reference_golden.py)."""
import os

import fingerprint as fp
import numpy as np
import pytest
import reference_cases as rc
from conftest import assert_bits_equal

from oracle import proesmans as ora
from proesmans_cases import CASES, STRICT_CASES, build_case

TOL = 1e-8  # px, -ffast-math build, well-conditioned cases; flows are O(1) px


@pytest.fixture(scope="module")
def golden():
    return np.load(os.path.join(os.path.dirname(__file__), "golden", "proesmans_golden.npz"))


@pytest.fixture(scope="module")
def strict_golden():
    return np.load(os.path.join(os.path.dirname(__file__), "golden", "proesmans_strict_golden.npz"))


@pytest.fixture(scope="module")
def random_golden():
    return fp.load(os.path.join(os.path.dirname(__file__), "golden", "reference_proesmans_golden.npz"))


@pytest.fixture
def raster_mean():
    ora.raster_order_mean(True)
    yield
    ora.raster_order_mean(False)


@pytest.mark.parametrize("name", STRICT_CASES)
def test_oracle_is_bit_identical_to_the_ieee_build_of_the_reference(name, strict_golden, raster_mean):
    frames, kw = build_case(name)
    adv, q = ora.proesmans(frames[-2:], full_output=True, **kw)
    assert_bits_equal(adv, strict_golden[name + "/advfield"], name + " advection fields")
    assert_bits_equal(q, strict_golden[name + "/quality"], name + " consistency maps")


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_the_fastmath_build_of_the_reference(name, golden):
    frames, kw = build_case(name)
    if frames.shape[0] != 2:
        with pytest.raises(ValueError) as e:
            ora.proesmans(frames, **kw)
        assert str(e.value) == str(golden[name + "/error"])
        frames = frames[-2:]
    adv, q = ora.proesmans(frames, full_output=True, **kw)   # default: row-wise mean, as the CUDA path
    ref_adv, ref_q = golden[name + "/advfield"], golden[name + "/quality"]
    assert adv.shape == ref_adv.shape and q.shape == ref_q.shape
    assert np.abs(adv - ref_adv).max() <= TOL and np.abs(q - ref_q).max() <= 10 * TOL
    assert np.array_equal(ora.proesmans(frames, **kw), adv[0])
    if name != "constant_32x32":
        assert np.abs(ref_adv).max() > 0.3   # the cases do exercise the solver


def test_gaussian_prefilter_against_live_reference(raster_mean, random_golden):
    frames, _ = build_case("default_96x128")
    for std in rc.PROESMANS_PREFILTER_STDS:
        b, qb = ora.proesmans(frames, filter_std=std, num_iter=10, num_levels=3, full_output=True)
        fp.assert_same(b, random_golden, f"proesmans_prefilter/{std}/advfield", f"filter_std {std}")
        fp.assert_same(qb, random_golden, f"proesmans_prefilter/{std}/quality", f"filter_std {std} quality")


def test_argument_errors():
    with pytest.raises(ValueError, match="dimension mismatch"):
        ora.proesmans(np.zeros((8, 8)))
    with pytest.raises(ValueError, match="frames 3 mismatch"):
        ora.proesmans(np.zeros((3, 8, 8)))


def test_live_ieee_build_bitwise(raster_mean, random_golden):
    for i, (fr, kw) in enumerate(rc.proesmans_random_cases(21, 25)):
        b, qb = ora.proesmans(fr, **kw)
        fp.assert_same(b, random_golden, f"proesmans_strict/{i}/advfield", f"{fr.shape} {kw}")
        fp.assert_same(qb, random_golden, f"proesmans_strict/{i}/quality", f"{fr.shape} {kw} quality")


def test_live_fastmath_build_statistically(random_golden):
    """max deviation from the -ffast-math build, over the stored sample of each field"""
    devs = []
    for i, (fr, kw) in enumerate(rc.proesmans_random_cases(22, 25)):
        b, _ = ora.proesmans(fr, **kw)
        want = random_golden[f"proesmans_fast/{i}/advfield/sample"]
        assert b.shape == fp.layout(random_golden, f"proesmans_fast/{i}/advfield")[1]
        devs.append(np.abs(fp.sample(b, random_golden, f"proesmans_fast/{i}/advfield") - want).max())
    assert np.median(devs) < 1e-9, sorted(devs)
