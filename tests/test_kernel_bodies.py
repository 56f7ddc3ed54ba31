"""CPU execution of CUDA kernel bodies: the per-thread code of pysteps_b200/csrc/spline.cu
(spline_body.cuh, shared verbatim between the device build and tests/host_kernels/) is compiled
as host C++ and run over the whole "grid" against the oracle, bit for bit.  This pins the
arithmetic and index logic of the spline kernels without a GPU; the device build differs only
in spelling every float64 operation as a round-to-nearest intrinsic."""
import ctypes
import math
import os

import numpy as np
import pytest
from conftest import ROOT, assert_bits_equal

import fingerprint as fp
import host_kernels
import reference_cases as rc
from oracle import semilagrangian as ora

POLES = {0: (), 2: (-0.171572875253809902396622551580603843,), 3: (-0.267949192431122706472553658494127633,),
         4: (-0.361341225900220177092212841325675255, -0.013725429297339121360331226939128204),
         5: (-0.430575347099973791851434783493520110, -0.043096288203264653822712376822550182)}
F32, F64 = 0, 1
MODES = {"constant": 0, "nearest": 1}
_dp = ctypes.POINTER(ctypes.c_double)


@pytest.fixture(scope="module")
def host_golden():
    return fp.load(os.path.join(ROOT, "tests", "golden", "reference_host_golden.npz"))


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _stats(P):
    fin = np.isfinite(P)
    nn = P[~np.isnan(P)].astype(np.float64)
    return np.array([np.count_nonzero(~fin), nn.min() if nn.size else np.nan,
                     nn.max() if nn.size else np.nan, np.count_nonzero(np.isnan(P))], dtype=np.float64)


def _prepare(P, order, mode, zero_fill):
    L = host_kernels.lib()
    m, n = P.shape
    pad = L.host_spline_pad(order, MODES[mode])
    M, N = m + 2 * pad, n + 2 * pad
    reflect = mode == "nearest"
    coeffs = np.empty((M, N))
    mmin, mfin = np.full((m, n), -1.0), np.full((m, n), -1.0)
    stats = _stats(P)
    L.host_spline_prepare.restype = None
    L.host_spline_prepare.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                      ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p,
                                      ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                      ctypes.c_void_p]
    poles = np.array(POLES[order] + (0.0,))
    zp0 = np.array([math.pow(z, M if reflect else M - 1) for z in poles])
    zp1 = np.array([math.pow(z, N if reflect else N - 1) for z in poles])
    L.host_spline_prepare(_p(P), F32 if P.dtype == np.float32 else F64, m, n, order, MODES[mode], _p(stats),
                          int(zero_fill), _p(poles), _p(zp0), _p(zp1), _p(coeffs), _p(mmin), _p(mfin))
    return coeffs, mmin, mfin, stats, pad


@pytest.mark.parametrize("order", [2, 3, 4, 5])
@pytest.mark.parametrize("shape", [(9, 13), (1, 7), (5, 1), (2, 2), (1, 1), (40, 33)])
@pytest.mark.parametrize("mode", ["constant", "nearest"])
def test_prepare_and_prefilter_bodies(shape, mode, order):
    from scipy import ndimage as ndi
    rng = np.random.default_rng(shape[0] * 31 + shape[1])
    for dtype in (np.float64, np.float32):
        P = (rng.standard_normal(shape) * 5).astype(dtype)
        P[rng.random(shape) < 0.15] = np.nan
        for zero_fill in (False, True):
            if not zero_fill:
                P = np.nan_to_num(P, nan=1.5)
            coeffs, mmin, mfin, stats, pad = _prepare(P, order, mode, zero_fill)
            src = np.where(np.isfinite(P), P, 0.0).astype(np.float64) if zero_fill else P.astype(np.float64)
            padded = np.pad(src, pad, mode="edge") if pad else src
            assert_bits_equal(coeffs, ndi.spline_filter(padded, order, output=np.float64, mode=mode), "coefficients")
            assert_bits_equal(coeffs, ora.spline_filter(padded, order, mode), "coefficients vs oracle")
            minval = np.nanmin(P)
            assert_bits_equal(mmin, (P > minval).astype(float), "mask_min")      # semilagrangian.py:148
            assert_bits_equal(mfin, np.isfinite(P).astype(float) if zero_fill else np.ones(shape), "mask_finite")
    # order 0: a plain float64 copy, no masks touched
    coeffs, mmin, mfin, _, pad = _prepare(P, 0, mode, False)
    assert pad == 0 and np.array_equal(coeffs, P.astype(np.float64), equal_nan=True) and np.all(mmin == -1.0)


@pytest.mark.parametrize("order", [0, 2, 3, 4, 5])
@pytest.mark.parametrize("mode", ["constant", "nearest"])
def test_sample_body_reproduces_the_oracle_extrapolator(mode, order):
    """prepare + sample bodies, fed with per-leadtime displacements, == the oracle's (reference-
    pinned) extrapolate() with interp_order 0 / 3, incl. NaN handling, float32, bands, xy_coords."""
    L = host_kernels.lib()
    L.host_spline_sample.restype = None
    L.host_spline_sample.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                     ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                     ctypes.c_double, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                     ctypes.c_int, ctypes.c_void_p]
    rng = np.random.default_rng(10 * order + MODES[mode])
    for case in range(12):
        m, n = int(rng.integers(1, 28)), int(rng.integers(1, 28))
        dtype = rng.choice([np.float64, np.float32])
        P = (rng.standard_normal((m, n)) * 5).astype(dtype)
        allow = bool(rng.random() < 0.5)
        if allow:
            P[rng.random((m, n)) < 0.2] = np.nan
            if np.all(np.isnan(P)):
                P[0, 0] = 1.0
        V = rng.standard_normal((2, m, n)) * rng.choice([0.5, 3.0, 30.0])
        T = int(rng.integers(1, 4))
        outval = float(rng.choice([np.nan, 0.0, -15.0]))
        xy = None
        if rng.random() < 0.3:
            xx, yy = np.meshgrid(np.arange(n) + 0.25, np.arange(m) * 0.5)
            xy = np.stack([xx, yy])
        kw = dict(interp_order=order, map_coordinates_mode=mode, allow_nonfinite_values=allow, xy_coords=xy)
        want = ora.extrapolate(P, V, T, outval, **kw)
        # displacement after every leadtime: single-step calls carrying the displacement give the
        # same trajectory for equal time steps (what b200_sl_trajectories delivers in one go)
        disp = np.empty((T, 2, m, n))
        for t in range(T):
            disp[t] = ora.extrapolate(None, V, t + 1, xy_coords=xy, return_displacement=True)[1]
        coeffs, mmin, mfin, stats, _ = _prepare(P, order, mode, allow and order > 1)
        r0, r1 = (0, m) if case % 3 else (m // 3, max(m // 3 + 1, 2 * m // 3))
        band = np.ascontiguousarray(disp[:, :, r0:r1])
        out = np.empty((T, r1 - r0, n), dtype=dtype)
        L.host_spline_sample(_p(coeffs), m, n, order, MODES[mode], _p(xy), _p(band), T, r0, r1 - r0, outval,
                             _p(mmin), _p(mfin), _p(stats), F32 if dtype == np.float32 else F64, _p(out))
        assert_bits_equal(out, want[:, r0:r1], f"case {case} {(m, n)} {np.dtype(dtype).name} allow={allow}")


# ---- Proesmans (pysteps_b200/csrc/proesmans.cu / proesmans_body.cuh) -----------------------------
@pytest.mark.parametrize("case", [(64, 80, 3, 40, 50.0), (37, 53, 2, 20, 50.0), (130, 97, 4, 30, 10.0),
                                  (40, 40, 6, 10, 50.0), (5, 4, 1, 3, 50.0), (63, 95, 1, 100, 1000.0),
                                  (3, 3, 1, 5, 50.0), (2, 9, 1, 2, 50.0)])
def test_proesmans_bodies_and_wavefront_schedule(case):
    """The whole b200_proesmans_field launch sequence on the CPU: pyramid, gradients, consistency
    maps (row-wise mean), the Gauss-Seidel sweep run wavefront by wavefront (t = x + 2y) with the
    rows of a wavefront in REVERSE order and the two flow fields swapped, border fill, prolongation
    -- bit-identical to the oracle's raster-order sweep, ill-conditioned settings included."""
    from oracle import proesmans as ora_p
    from pysteps_b200 import _synthetic as syn
    m, n, levels, num_iter, lam = case
    L = host_kernels.lib()
    L.host_proesmans_field.restype = ctypes.c_int
    L.host_proesmans_scale.restype = None
    fr = syn.rain_frames(m, n, 2, 3, dx=2, dy=-1)
    lo, hi = float(fr.min()), float(fr.max())
    im = np.empty_like(fr)
    L.host_proesmans_scale(_p(np.ascontiguousarray(fr)), ctypes.c_int64(fr.size), ctypes.c_double(lo),
                           ctypes.c_double(hi), int(hi - lo > 1e-8), _p(im))
    assert_bits_equal(im, (fr - lo) / (hi - lo) * 255.0 if hi - lo > 1e-8 else fr, "scaling")
    adv, q = np.empty((2, 2, m, n)), np.empty((2, m, n))
    rc = L.host_proesmans_field(_p(im), m, n, ctypes.c_double(lam), num_iter, levels, _p(adv), _p(q))
    assert rc == 0
    want_adv, want_q = ora_p.compute_advection_field(im, lam, num_iter, levels)
    assert_bits_equal(adv, want_adv, f"{case} advection fields")
    assert_bits_equal(q, want_q, f"{case} consistency maps")
    # an empty pyramid level is refused (the reference reads out of bounds there)
    assert L.host_proesmans_field(_p(im), m, n, ctypes.c_double(lam), 1, 12, _p(adv), _p(q)) == -1


# ---- cKDTree-exact k-NN + outlier test (pysteps_b200/csrc/knn.cu / knn_body.cuh) -----------------
@pytest.mark.parametrize("kind", ["int", "half", "dup", "few_values", "real"])
@pytest.mark.parametrize("n", [1, 5, 17, 60, 400, 2000])
def test_knn_body_matches_scipy_ckdtree(kind, n):
    from scipy.spatial import cKDTree
    rng = np.random.default_rng(n * 13 + len(kind))
    W = int(rng.choice([16, 64, 300]))
    pts = np.floor(rng.uniform(0, W, (n, 2)))
    if kind == "half":
        pts = np.floor(rng.uniform(0, W, (n, 2)) * 2) / 2
    elif kind == "dup" and n >= 8:
        pts[: n // 4] = pts[n // 4: 2 * (n // 4)]
    elif kind == "few_values":
        pts = np.floor(rng.uniform(0, 4, (n, 2)))
    elif kind == "real":
        pts = rng.uniform(0, W, (n, 2))
    pts = np.ascontiguousarray(pts)
    L = host_kernels.lib()
    ref = cKDTree(pts)
    queries = np.ascontiguousarray(np.concatenate([pts[:200], np.floor(rng.uniform(-2, W + 2, (100, 2)))]))
    for k in (2, 21, 31, 101):
        k = min(k, n)
        perm = np.empty(n, np.int32)
        out = np.empty((len(queries), k), np.int32)
        L.host_kd_knn(_p(pts), n, _p(queries), len(queries), k, _p(perm), _p(out))
        assert np.array_equal(perm, ref.indices), (kind, n)
        assert np.array_equal(out, ref.query(queries, k=k)[1].reshape(len(queries), -1)), (kind, n, k)


@pytest.mark.parametrize("kind", ["int", "half", "dup", "few_values", "real", "sorted", "const_x"])
@pytest.mark.parametrize("n", [1, 17, 18, 33, 60, 400, 2000, 4096])
def test_knn_pair_formulation_build_matches_scipy_ckdtree(kind, n):
    """The build as knn.cu runs it -- libstdc++'s partition loops restated as pair swaps on
    position-aligned (x, y, index) triples (knn_body.cuh: build_pairs) -- gives scipy's own tree
    order and neighbour lists; with the introselect depth limit forced to 0..3 (heap-select branch)
    it still equals the sequential restatement given the same limit... which libstdc++ pins for the
    default limit only, so forced limits are compared on the k-NN SETS' distances."""
    from scipy.spatial import cKDTree
    rng = np.random.default_rng(n * 7 + len(kind))
    W = int(rng.choice([16, 64, 300, 2048]))
    pts = np.floor(rng.uniform(0, W, (n, 2)))
    if kind == "half":
        pts = np.floor(rng.uniform(0, W, (n, 2)) * 2) / 2
    elif kind == "dup" and n >= 8:
        pts[: n // 4] = pts[n // 4: 2 * (n // 4)]
    elif kind == "few_values":
        pts = np.floor(rng.uniform(0, 4, (n, 2)))
    elif kind == "real":
        pts = rng.uniform(0, W, (n, 2))
    elif kind == "sorted":
        pts = pts[np.lexsort((pts[:, 1], pts[:, 0]))]
    elif kind == "const_x":
        pts[:, 0] = 7.0
    pts = np.ascontiguousarray(pts)
    L = host_kernels.lib()
    L.host_kd_knn_pairs.restype = ctypes.c_int
    ref = cKDTree(pts)
    queries = np.ascontiguousarray(np.concatenate([pts[:200], np.floor(rng.uniform(-2, W + 2, (100, 2)))]))
    for k in (2, 21, 31):
        k = min(k, n)
        perm = np.empty(n, np.int32)
        out = np.empty((len(queries), k), np.int32)
        ovf = L.host_kd_knn_pairs(_p(pts), n, _p(queries), len(queries), k, -1, 0, _p(perm), _p(out))
        assert ovf == 0
        assert np.array_equal(perm, ref.indices), (kind, n)
        want_d, want_i = ref.query(queries, k=k)
        assert np.array_equal(out, want_i.reshape(len(queries), -1)), (kind, n, k)
        # the device query uses a 128-entry pending-node heap: never reached on these sets
        assert L.host_kd_knn_pairs(_p(pts), n, _p(queries), len(queries), k, -1, 128, _p(perm), _p(out)) == 0
        for depth in (0, 1, 3):  # heap-select branch: a valid tree (same neighbour distances)
            L.host_kd_knn_pairs(_p(pts), n, _p(queries), len(queries), k, depth, 0, _p(perm), _p(out))
            assert sorted(perm.tolist()) == list(range(n))
            d = np.sqrt(((pts[out] - queries[:, None, :]) ** 2).sum(-1))
            assert np.array_equal(d, want_d.reshape(len(queries), -1)), (kind, n, k, depth)


def test_outlier_body_matches_the_reference_at_ties(host_golden):
    """detect_outliers of the reference (scipy cKDTree + np.cov + np.linalg.inv) on vector sets with
    many equidistant and coincident positions: the body's flags equal the reference's stored ones
    and the oracle's in cKDTree mode."""
    from oracle import lucaskanade as ora_lk
    L = host_kernels.lib()
    L.host_detect_outliers_ckdtree.restype = None
    for it, (uv, xy, k, thr) in enumerate(rc.outlier_body_cases()):
        n = len(xy)
        flags = np.empty(n, np.uint8)
        L.host_detect_outliers_ckdtree(_p(np.ascontiguousarray(uv)), _p(np.ascontiguousarray(xy)), n,
                                       ctypes.c_double(thr), k, _p(flags))
        with ora_lk.knn_mode("ckdtree"):
            want = ora_lk.detect_outliers(uv, thr, xy, k)
        assert np.array_equal(flags.astype(bool), want), (it, n, k, thr)
        if n >= 3:
            ref = np.unpackbits(host_golden[f"outliers/{it}"], count=n).astype(bool)
            assert np.array_equal(flags.astype(bool), ref), (it, n, k, thr)


def test_exact_idw_body_matches_the_reference_at_every_grid_point(host_golden):
    """idwinterp2d with cKDTree's neighbour order, numpy's pairwise weight sum and in-order
    accumulation (knn_body.cuh: idw_point): equal to the oracle at ALL grid points and to the
    reference's stored fields (bit for bit, or within 1e-14 on a stored sample), ties and coincident
    vectors included, to the last bits of np.power vs pow."""
    from oracle import lucaskanade as ora_lk
    L = host_kernels.lib()
    L.host_idw_fill_ckdtree.restype = None
    for it, (xy, uv, W, H, k, power, off) in enumerate(rc.idw_body_cases()):
        n = len(xy)
        xg, yg = np.arange(W, dtype=float), np.arange(H, dtype=float)
        out = np.empty((2, H, W))
        L.host_idw_fill_ckdtree(_p(np.ascontiguousarray(xy)), _p(uv), n, 2, k, ctypes.c_double(power),
                                ctypes.c_double(off), ctypes.c_double(1.0), _p(xg), W, _p(yg), H, _p(out))
        with ora_lk.knn_mode("ckdtree"):
            want = ora_lk.idwinterp2d(xy, uv, np.arange(W), np.arange(H), power=power, k=k, dist_offset=off)
        assert np.abs(out - want).max() <= 1e-14, (it, n, k, power)
        fp.assert_close(out, host_golden, f"idw/{it}", 1e-14, f"case {it} {(n, k, power)}")


@pytest.mark.parametrize("shape", [(17, 23), (5, 40), (1, 9), (3, 3), (64, 80)])
@pytest.mark.parametrize("sigma", [0.5, 1.0, 2.3, 6.0])
def test_gaussian_filter_body_matches_scipy_bitwise(shape, sigma):
    from scipy import ndimage as ndi
    rng = np.random.default_rng(shape[0] + int(sigma * 10))
    a = np.ascontiguousarray(rng.standard_normal(shape) * 20)
    radius = int(4.0 * float(sigma) + 0.5)
    x = np.arange(-radius, radius + 1)
    phi = np.exp(-0.5 / (sigma * sigma) * x ** 2)
    weights = np.ascontiguousarray((phi / phi.sum())[::-1])
    out = np.empty_like(a)
    L = host_kernels.lib()
    L.host_gaussian_filter.restype = None
    L.host_gaussian_filter(_p(a), shape[0], shape[1], _p(weights), radius, _p(out))
    assert_bits_equal(out, ndi.gaussian_filter(a, sigma), f"{shape} sigma {sigma}")


def test_float32_quantise_body_matches_numpy():
    """`(x - min) / (max - min) * 255` of a float32 array (tracking/lucaskanade.py:144-160) as the
    F32 variant of the quantise kernel evaluates it."""
    L = host_kernels.lib()
    L.host_scale_f32.restype = None
    rng = np.random.default_rng(6)
    for lo, hi in ((-15.0, 43.7), (0.0, 1e-9), (3.5, 3.5), (-1e6, 2.5e6)):
        x = rng.uniform(lo, max(hi, lo + 1e-3), 5000).astype(np.float32)
        x[:2] = [lo, hi]
        mn, mx = np.float32(x.min()), np.float32(x.max())
        want = ((x - mn) / (mx - mn) * 255) if mx - mn > 1e-8 else (x - mn)
        assert want.dtype == np.float32
        got = np.empty(x.size)
        L.host_scale_f32(_p(x.astype(np.float64)), ctypes.c_int64(x.size), ctypes.c_double(float(mn)),
                         ctypes.c_double(float(mx)), _p(got))
        assert_bits_equal(got.astype(np.float32), want, f"range {lo}..{hi}")
        assert np.array_equal(got, want.astype(np.float64))


def test_float64_quantise_body_matches_numpy_at_and_around_integer_boundaries():
    """The fused LK front end scales float64 frames to uint8 with a precomputed 255 / range and evaluates the
    reference's division only near integer results (csrc/quantise_body.cuh ScaleF64).  Against NumPy's
    `((x - min) / (max - min) * 255).astype('uint8')` on random values AND on values whose scaled image
    sits exactly on, and a few ulps either side of, every integer 0..255."""
    L = host_kernels.lib()
    L.host_scale_f64.restype = None
    rng = np.random.default_rng(17)
    u8p = ctypes.POINTER(ctypes.c_uint8)
    total_fb = 0
    for lo, hi in ((0.0, 40.0), (-15.0, 43.7), (0.0, 255.0), (1.25, 1.25 + 1e-6), (-3.0e5, 7.7e6), (0.1, 0.3),
                   (0.0, 1e-9), (2.5, 2.5), (0.0, float(np.float32(37.123)))):
        rngw = hi - lo
        x = rng.uniform(lo, hi if hi > lo else lo + 1.0, 200000)
        if rngw > 1e-8:
            k = np.arange(256, dtype=np.float64)
            onb = lo + k / 255.0 * rngw                     # lands on / next to integers after scaling
            near = [onb]
            for _ in range(6):
                near.append(np.nextafter(near[-1], np.inf))
            dn = onb
            for _ in range(6):
                dn = np.nextafter(dn, -np.inf)
                near.append(dn)
            x = np.concatenate([x] + near + [np.array([lo, hi, lo - 0.37 * rngw, hi + 0.41 * rngw, np.nan, np.inf])])
        x = np.ascontiguousarray(x)
        with np.errstate(invalid="ignore", divide="ignore", over="ignore"):
            q = ((x - lo) / (hi - lo) * 255) if hi - lo > 1e-8 else (x - lo)
            want = np.trunc(np.where(np.isfinite(q) & (np.abs(q) < 2147483648.0), q, 0.0)).astype(np.int64).astype(np.uint8)
        fast = np.empty(x.size, np.uint8)
        exact = np.empty(x.size, np.uint8)
        nfb = ctypes.c_int64(0)
        L.host_scale_f64(_p(x), ctypes.c_int64(x.size), ctypes.c_double(lo), ctypes.c_double(hi),
                         fast.ctypes.data_as(u8p), exact.ctypes.data_as(u8p), ctypes.byref(nfb))
        assert np.array_equal(exact, want), f"division path, range {lo}..{hi}"
        assert np.array_equal(fast, want), f"division-free path, range {lo}..{hi}: {(fast != want).sum()} differ"
        total_fb += nfb.value
    assert total_fb > 0  # the boundary values did exercise the fallback
