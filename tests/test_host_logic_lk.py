"""CPU test of the HOST logic of pysteps_b200.motion.lucaskanade.dense_lucaskanade (kwargs
plumbing, frame pairing and pooling, early-outs, masked-array handling, return conventions, the
b200_rows extension) over randomised frames and argument combinations.  The C-ABI entry points are
emulated with the oracle's stage functions (tests/cpu_abi.py), so the shim must reproduce the
oracle's dense_lucaskanade -- itself pinned to the reference -- bit for bit; errors, sparse
vectors and dense fields are also compared with the reference's stored outputs on the same calls
(tests/golden/reference_lk_host_golden.npz, tests/golden/gen_reference_golden.py)."""
import os
import warnings

import numpy as np
import pytest

import cpu_abi
import fingerprint as fp
from oracle import lucaskanade as ora
from pysteps_b200 import _synthetic as syn


@pytest.fixture(scope="module")
def golden():
    return fp.load(os.path.join(os.path.dirname(__file__), "golden", "reference_lk_host_golden.npz"))


def _error_entry(err):
    return "" if err is None else "%s: %s" % err


def _random_call(rng):
    m, n, T = int(rng.integers(40, 150)), int(rng.integers(40, 150)), int(rng.choice([1, 2, 2, 3]))
    fr = syn.rain_frames(m, n, T, int(rng.integers(0, 1000)), dx=int(rng.integers(-4, 5)), dy=int(rng.integers(-4, 5)))
    q = rng.random()
    if q < 0.25:
        fr = np.where(fr > 0.1, 10.0 * np.log10(np.maximum(fr, 0.1)), -15.0)
    elif q < 0.32:
        fr = np.zeros_like(fr)                       # nothing to track
    elif q < 0.38:
        fr = np.full_like(fr, np.nan)
    if rng.random() < 0.3:
        fr = np.stack([syn.nan_disc(f, float(rng.uniform(0.05, 0.3))) for f in fr])
    kw = {}
    if rng.random() < 0.3:
        kw["dense"] = False
    if rng.random() < 0.3:
        kw["lk_kwargs"] = dict(winsize=(int(rng.choice([15, 21, 50])),) * 2, nr_levels=int(rng.integers(0, 4)))
    if rng.random() < 0.3:
        kw["fd_kwargs"] = dict(max_corners=int(rng.choice([20, 200, 1000])), quality_level=float(rng.choice([0.01, 0.2])),
                               min_distance=int(rng.choice([3, 10, 25])), buffer_mask=int(rng.choice([0, 5, 12])))
    if rng.random() < 0.15:
        kw["fd_kwargs"] = dict(max_num_features=int(rng.choice([5, 50])))
    if rng.random() < 0.3:
        kw["interp_kwargs"] = dict(k=int(rng.choice([1, 4, 20, 30])), power=float(rng.choice([0.5, 1.0, 2.0])))
    if rng.random() < 0.2:
        kw["size_opening"] = 0
    if rng.random() < 0.2:
        kw["decl_scale"] = int(rng.choice([1, 5, 40]))
    if rng.random() < 0.2:
        kw["k_outlier"] = [5, 30, 100, None][int(rng.integers(0, 4))]
        kw["nr_std_outlier"] = float(rng.choice([1, 2, 3]))
    inp = fr
    q = rng.random()
    if q < 0.15 and np.isfinite(fr).any():
        inp = np.ma.masked_array(np.nan_to_num(fr, nan=0.0), mask=np.isnan(fr) | (rng.random(fr.shape) < 0.01))
    elif q < 0.2:
        inp = fr[0]                                  # wrong rank
    return inp, kw


def _run(fn, inp, kw):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        try:
            return fn(inp.copy(), **kw), None
        except Exception as e:  # noqa: BLE001
            return None, (type(e).__name__, str(e))


@pytest.mark.parametrize("seed", range(4))
def test_dense_lucaskanade_host_logic(seed, golden):
    from pysteps_b200.motion.lucaskanade import dense_lucaskanade
    rng = np.random.default_rng(500 + seed)
    n_ok = n_err = n_empty = 0
    with cpu_abi.emulated():
        for it in range(40):
            inp, kw = _random_call(rng)
            got, gerr = _run(dense_lucaskanade, inp, kw)
            want, werr = _run(ora.dense_lucaskanade, inp, kw)
            ctx = f"seed {seed} case {it}: shape={inp.shape} masked={isinstance(inp, np.ma.MaskedArray)} kw={kw}"
            assert gerr == werr, ctx
            assert _error_entry(gerr) == str(golden[f"host/{seed}/{it}/error"]), ctx
            if gerr is not None:
                n_err += 1
                continue
            n_ok += 1
            if kw.get("dense", True):
                assert isinstance(got, np.ndarray) and got.shape == want.shape and got.dtype == want.dtype, ctx
                assert np.array_equal(got, want), ctx
                n_empty += not got.any()
            else:
                assert isinstance(got, tuple) and len(got) == 2, ctx
                for a, b in zip(got, want):
                    assert a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a, b), ctx
                n_empty += got[0].shape[0] == 0
    assert n_ok >= 25 and n_empty >= 1, (n_ok, n_err, n_empty)


def test_row_band_fill_and_stage_mirrors():
    from pysteps_b200 import stages
    from pysteps_b200.motion.lucaskanade import dense_lucaskanade
    fr = syn.rain_frames(120, 96, 3, 5, dx=2, dy=-1)
    with cpu_abi.emulated():
        full = dense_lucaskanade(fr)
        for r0, r1 in ((0, 120), (0, 41), (41, 90), (77, 78)):
            band = dense_lucaskanade(fr, interp_kwargs={"b200_rows": (r0, r1)})
            assert band.shape == (2, r1 - r0, 96) and np.array_equal(band, full[:, r0:r1])
        with pytest.raises(ValueError):
            dense_lucaskanade(fr, interp_kwargs={"b200_rows": (5, 5)})
        assert dense_lucaskanade(fr[:1], interp_kwargs={"b200_rows": (5, 9)}).shape == (2, 4, 96)
        # the stand-alone mirrors of the helper functions (pysteps_b200.stages)
        a = np.ma.masked_invalid(fr[0]); np.ma.set_fill_value(a, a.min())
        b = np.ma.masked_invalid(fr[1]); np.ma.set_fill_value(b, b.min())
        oa, ob = ora.morph_opening(a, a.min(), 3), ora.morph_opening(b, b.min(), 3)
        ga = stages.morph_opening(a, a.min(), 3)
        assert np.array_equal(np.ma.getmaskarray(ga), np.ma.getmaskarray(oa)) and np.array_equal(ga.filled(), oa.filled())
        pts = stages.detection(oa)
        assert np.array_equal(pts, ora.detection(oa))
        xy, uv = stages.track_features(oa, ob, pts)
        oxy, ouv = ora.track_features(oa, ob, pts.astype(np.float32))
        assert np.array_equal(xy, oxy) and np.array_equal(uv, ouv)
        flags = stages.detect_outliers(uv, 3, xy, 30)
        assert np.array_equal(flags, ora.detect_outliers(uv, 3, xy, 30))
        dxy, duv = stages.decluster(xy[~flags], uv[~flags], 20, 1)
        o = ora.decluster(xy[~flags], uv[~flags], 20, 1)
        assert np.array_equal(dxy, o[0]) and np.array_equal(duv, o[1])
        g = stages.idwinterp2d(dxy, duv, np.arange(96), np.arange(120))
        assert np.array_equal(g, ora.idwinterp2d(dxy, duv, np.arange(96), np.arange(120)))
        assert np.array_equal(stages.idwinterp2d(dxy, duv, np.arange(96), np.arange(30, 70)), g[:, 30:70])


def test_sparse_vectors_equal_the_live_reference(golden):
    """The outlier stage takes neighbours in cKDTree's own order (csrc/knn.cu; emulated here by the
    kernel body compiled for the host): the sparse vectors equal the LIVE reference bit for bit --
    also on three-frame inputs whose pooled vectors coincide, where a lower-index rule would keep
    or drop a different vector (DESIGN.md section 4)."""
    from pysteps_b200.motion.lucaskanade import dense_lucaskanade
    rng = np.random.default_rng(2000)
    n = 0
    with cpu_abi.emulated():
        for it in range(60):
            inp, kw = _random_call(rng)
            kw = dict(kw, dense=False)
            got, gerr = _run(dense_lucaskanade, inp, kw)
            with ora.knn_mode("ckdtree"):
                want, werr = _run(ora.dense_lucaskanade, inp, kw)
            assert gerr == werr, (it, kw)
            assert _error_entry(gerr) == str(golden[f"sparse/{it}/error"]), (it, kw)
            if gerr is None:
                n += 1
                for a, b in zip(got, want):
                    assert a.shape == b.shape and np.array_equal(a, b), (it, kw)
                fp.assert_same(got[0], golden, f"sparse/{it}/xy", f"{it} {kw}")
                fp.assert_same(got[1], golden, f"sparse/{it}/uv", f"{it} {kw}")
    assert n >= 40


def test_dense_field_equals_the_live_reference_everywhere(golden):
    """... and the dense field equals the reference to the last bits (1e-13), pixels with a k-NN tie
    included: bit for bit against the stored digest of the reference's field or, failing that, on its
    stored sample, and at every pixel against the oracle in cKDTree mode (pinned to the reference by
    tests/test_oracle_lk.py)."""
    from pysteps_b200.motion.lucaskanade import dense_lucaskanade
    rng = np.random.default_rng(2001)
    n = 0
    with cpu_abi.emulated():
        for it in range(30):
            inp, kw = _random_call(rng)
            kw = dict(kw, dense=True)
            got, gerr = _run(dense_lucaskanade, inp, kw)
            assert _error_entry(gerr) == str(golden[f"dense/{it}/error"]), (it, kw)
            if gerr is None:
                n += 1
                fp.assert_close(got, golden, f"dense/{it}/field", 1e-13, f"case {it} {kw}")
                with ora.knn_mode("ckdtree"):
                    want = ora.dense_lucaskanade(inp.copy(), **kw)
                assert np.abs(got - want).max() <= 1e-13, (it, kw)
    assert n >= 20


def test_float32_frames_are_scaled_in_float32_like_the_reference(golden):
    """float32 frames: NumPy scales them to uint8 in float32, which moves some pixels by one grey
    level against float64 arithmetic and with them corners and vectors; the shim flags the frames
    (B200_QUANTISE_F32) and reproduces the oracle -- and, with the reference's tie order, the
    reference's stored sparse vectors."""
    from pysteps_b200.motion.lucaskanade import dense_lucaskanade
    rng = np.random.default_rng(0)
    with cpu_abi.emulated():
        for it in range(12):
            m, n = int(rng.integers(60, 160)), int(rng.integers(60, 160))
            fr = syn.rain_frames(m, n, int(rng.choice([2, 3])), int(rng.integers(0, 1000)), dx=2, dy=-1)
            if it % 2:
                fr = np.where(fr > 0.1, 10 * np.log10(np.maximum(fr, 0.1)), -15.0)
            fr = (fr + 0.37 * rng.standard_normal(fr.shape)).astype(np.float32)
            inp = fr if it % 3 else np.ma.masked_invalid(fr)
            got = dense_lucaskanade(inp.copy(), dense=False)
            want = ora.dense_lucaskanade(inp.copy(), dense=False)
            assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1]), it
            V = dense_lucaskanade(inp.copy())
            assert V.dtype == np.float64 and np.array_equal(V, ora.dense_lucaskanade(inp.copy())), it
            fp.assert_same(got[0], golden, f"float32/{it}/xy", str(it))
            fp.assert_same(got[1], golden, f"float32/{it}/uv", str(it))


def test_many_frames_pool_larger_than_the_decluster_kernel(monkeypatch):
    """The sparse pool holds max_corners vectors per frame pair; the decluster kernel's capacity is about
    the vectors that EXIST.  A long stack (pool > capacity) must work off the real count -- the reference
    has no limit -- and only a real excess is refused, by name."""
    from pysteps_b200.motion import lucaskanade as lkmod
    fr = syn.rain_frames(96, 112, 5, 3, dx=2, dy=-1)
    with cpu_abi.emulated():
        want = lkmod.dense_lucaskanade(fr)
        monkeypatch.setattr(lkmod, "_DECLUSTER_MAX", 2000)  # 4 pairs x 1000 corners = 4000 > 2000
        got = lkmod.dense_lucaskanade(fr)
        assert np.array_equal(got, want)
        monkeypatch.setattr(lkmod, "_DECLUSTER_MAX", 3)
        with pytest.raises(NotImplementedError, match="declustering more than 3"):
            lkmod.dense_lucaskanade(fr)
