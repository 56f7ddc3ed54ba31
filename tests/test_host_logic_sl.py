"""CPU test of the HOST logic of pysteps_b200.extrapolation.semilagrangian.extrapolate and of the
BPS handles: argument validation (order, types, messages), defaults, return structure, dtypes
and shapes, over randomised valid AND invalid argument combinations -- against the oracle and
the reference's stored results on the same calls (tests/golden/reference_host_golden.npz, written
by tests/golden/gen_reference_golden.py).  The C ABI is emulated by the oracle (tests/cpu_abi.py),
so numerics here say nothing about the kernels."""
import os
import warnings

import numpy as np
import pytest

import cpu_abi
import fingerprint as fp
import reference_cases as rc
from oracle import noise_motion as ora_bps
from oracle import semilagrangian as ora
from pysteps_b200 import _synthetic as syn


@pytest.fixture(scope="module")
def golden():
    return fp.load(os.path.join(os.path.dirname(__file__), "golden", "reference_host_golden.npz"))


def _bits_equal(a, b):
    return (a.shape == b.shape and a.dtype == b.dtype
            and np.array_equal(np.ascontiguousarray(a).view(np.uint8), np.ascontiguousarray(b).view(np.uint8)))


def _random_call(rng):
    m, n = int(rng.integers(1, 24)), int(rng.integers(1, 24))
    pd = rng.choice([np.float64, np.float32])
    vd = rng.choice([np.float64, np.float32])
    P = (rng.standard_normal((m, n)) * 5).astype(pd)
    scale = rng.choice([0.3, 1.0, 3.0, 15.0, 1e3])
    V = (rng.standard_normal((2, m, n)) * scale).astype(vd)
    kw = {}
    r = rng.random
    if r() < 0.25:
        P[rng.random((m, n)) < 0.3] = np.nan
    if r() < 0.05:
        P[...] = np.nan
    if r() < 0.1:
        V[:, rng.random((m, n)) < 0.2] = rng.choice([np.nan, np.inf])
    if r() < 0.03:
        V[...] = np.nan
    if r() < 0.45:
        kw["allow_nonfinite_values"] = bool(r() < 0.8)
    if r() < 0.5:
        kw["n_iter"] = int(rng.integers(0, 4))
    if r() < 0.5:
        kw["map_coordinates_mode"] = str(rng.choice(["constant", "nearest"]))
    if r() < 0.5:
        kw["return_displacement"] = bool(r() < 0.8)
    if r() < 0.3:
        kw["displacement_prev"] = rng.standard_normal((2, m, n)) * scale
    if r() < 0.2:
        xx, yy = np.meshgrid(np.arange(n) + 0.25, np.arange(m) * rng.choice([1.0, 0.5]))
        kw["xy_coords"] = np.stack([xx, yy])
    if r() < 0.1:
        kw["xy_coords"] = np.stack(np.meshgrid(np.arange(n), np.arange(m)))  # the default grid
    if r() < 0.1:
        kw["D_prev"] = None
    if r() < 0.1:
        kw["verbose"] = False
    if r() < 0.1:
        kw["interp_order"] = 1
    outval = rng.choice([np.nan, 0.0, -15.0])
    if r() < 0.2:
        outval = "min"
    q = r()
    if q < 0.4:
        ts = int(rng.integers(1, 4))
    elif q < 0.8:
        ts = sorted(set(np.round(rng.uniform(0.1, 4, int(rng.integers(1, 4))), 2).tolist()))
        kw["vel_timestep"] = float(rng.choice([1.0, 0.5, 2.0]))
    elif q < 0.87:
        ts = [2.0, 1.0]                       # not ascending
    elif q < 0.94:
        ts = np.array([1.0, 1.0, 2.0])        # ndarray with a repeated element
    else:
        ts = np.array([0.5, 1.5])
    q = r()
    if q < 0.08:
        Pin = None
    elif q < 0.12:
        Pin = P[None]                         # wrong rank
    else:
        Pin = P
    Vin = V[0] if r() < 0.04 else V
    return Pin, Vin, ts, outval, kw


def _run(fn, Pin, Vin, ts, outval, kw):
    cp = lambda v: v.copy() if isinstance(v, np.ndarray) else v  # noqa: E731
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter("always")
        try:
            res = fn(cp(Pin), cp(Vin), cp(ts), outval, **{k: cp(v) for k, v in kw.items()})
            err = None
        except Exception as e:  # noqa: BLE001
            res, err = None, (type(e).__name__, str(e))
    deprecations = sorted(str(x.message) for x in w if "D_prev" in str(x.message))
    return res, err, deprecations


@pytest.mark.parametrize("seed", range(6))
def test_extrapolate_host_logic_matches_reference(seed, golden):
    import pysteps_b200
    rng = np.random.default_rng(100 + seed)
    n_err = n_ok = 0
    with cpu_abi.emulated():
        for it in range(120):
            Pin, Vin, ts, outval, kw = _random_call(rng)
            want, werr, wdep = _run(ora.extrapolate, Pin, Vin, ts, outval, kw)
            got, gerr, gdep = _run(pysteps_b200.extrapolation.semilagrangian.extrapolate, Pin, Vin, ts, outval, kw)
            ctx = f"seed {seed} case {it}: ts={ts!r} outval={outval!r} kw={ {k: (v.shape if isinstance(v, np.ndarray) else v) for k, v in kw.items()} }"
            fp.assert_call(got, gerr, golden, f"sl/{seed}/{it}", ctx)
            assert "\n".join(gdep) == golden[f"sl/{seed}/{it}/deprecations"], ctx
            assert gerr == werr, ctx
            assert gdep == wdep, ctx
            if werr is not None:
                n_err += 1
                continue
            n_ok += 1
            assert isinstance(got, tuple) == isinstance(want, tuple), ctx
            for a, b in zip(got if isinstance(got, tuple) else (got,), want if isinstance(want, tuple) else (want,)):
                assert (a is None) == (b is None), ctx
                if a is not None:
                    assert isinstance(a, np.ndarray) and _bits_equal(a, b), ctx
    assert n_err >= 10 and n_ok >= 40, (n_err, n_ok)


def test_member_loop_with_handles_matches_reference_expression(golden):
    """nowcasts/utils.py:440-458 with lazy handles and resident displacements == the same loop
    with materialised arrays (oracle perturbator + oracle extrapolator, whose results equal the
    reference's stored ones)."""
    import pysteps_b200
    from pysteps_b200 import _device
    with cpu_abi.emulated():
        init, gen = pysteps_b200.noise.get_method("bps")
        extrap = pysteps_b200.extrapolation.get_method("semilagrangian")
        for vd, (V, P, steps) in rc.member_loop_case().items():
            pg = init(V, 0.5, 5.0, randstate=np.random.RandomState(9))
            po = ora_bps.initialize_bps(V, 0.5, 5.0, randstate=np.random.RandomState(9))
            assert pg["eps_par"] == po["eps_par"] and pg["eps_perp"] == po["eps_perp"]
            assert _bits_equal(pg["V_par"], po["V_par"]) and _bits_equal(pg["V_perp"], po["V_perp"])
            dg = dr = None
            for step in steps:
                h = V + gen(pg, step * 5.0)
                assert isinstance(h, pysteps_b200.noise.motion.PerturbedVelocity)
                out_g, dg = extrap(P, h, [1.0], displacement_prev=dg, return_displacement=True,
                                   allow_nonfinite_values=True, b200_resident=True)
                assert isinstance(dg, _device.DeviceField) and dg.shape == (2, 19, 23)
                out_r, dr = ora.extrapolate(P, V + ora_bps.generate_bps(po, step * 5.0), [1.0], displacement_prev=dr,
                                            return_displacement=True, allow_nonfinite_values=True)
                fp.assert_same(out_r, golden, f"member_loop/{vd}/{step}/out")
                fp.assert_same(dr, golden, f"member_loop/{vd}/{step}/displacement")
                assert _bits_equal(out_g, out_r) and _bits_equal(np.asarray(dg), dr)
            assert _bits_equal(np.asarray(V + gen(pg, 7.0)), V + ora_bps.generate_bps(po, 7.0))
        # non-finite perturbed field: the extrapolator's own check fires (semilagrangian.py:118-123)
        v = np.ones((2, 4, 4))
        pert = init(v, 1, 1, p_par=(1e308, 1.0, 0.0), seed=1)
        with pytest.raises(ValueError, match="velocity contains non-finite values"):
            extrap(np.ones((4, 4)), v + gen(pert, 100.0), 1)
        with pytest.raises(ValueError, match="velocity contains only non-finite values"):
            extrap(np.ones((4, 4)), v + gen(pert, 100.0), 1, allow_nonfinite_values=True)
        bad = v.copy()
        bad[0, 0, 0] = np.inf
        with pytest.raises(ValueError, match="infs or NaNs"):
            init(bad, 1, 1)


@pytest.mark.parametrize("seed", range(3))
def test_spline_orders_host_logic_and_kernel_bodies(seed, monkeypatch, golden):
    """interp_order 0, 2..5: the
    shim's branch -- trajectories per leadtime, prefilter, sampling, mask warps, outval="min" on
    the zero-filled copy, bands -- driven through the emulated C ABI, whose spline entry points
    are the CUDA kernels' own bodies compiled for the host (tests/host_kernels)."""
    import pysteps_b200
    extrap = pysteps_b200.extrapolation.semilagrangian.extrapolate
    rng = np.random.default_rng(300 + seed)
    with cpu_abi.emulated():
        with pytest.raises(RuntimeError, match="spline order not supported"):
            extrap(np.ones((4, 4)), np.ones((2, 4, 4)), 1, interp_order=6)
        n_ok = 0
        for it in range(60):
            Pin, Vin, ts, outval, kw = _random_call(rng)
            kw["interp_order"] = int(rng.choice([0, 2, 3, 3, 4, 5]))
            want, werr, wdep = _run(ora.extrapolate, Pin, Vin, ts, outval, kw)
            got, gerr, gdep = _run(extrap, Pin, Vin, ts, outval, kw)
            ctx = f"seed {seed} case {it}: ts={ts!r} outval={outval!r} kw={ {k: (v.shape if isinstance(v, np.ndarray) else v) for k, v in kw.items()} }"
            if gerr is not None and "inf in precip" in gerr[1]:
                continue
            fp.assert_call(got, gerr, golden, f"spline/{seed}/{it}", ctx)
            assert "\n".join(gdep) == golden[f"spline/{seed}/{it}/deprecations"], ctx
            assert gerr == werr and gdep == wdep, ctx
            if werr is not None:
                continue
            n_ok += 1
            for a, b in zip(got if isinstance(got, tuple) else (got,), want if isinstance(want, tuple) else (want,)):
                assert (a is None) == (b is None), ctx
                if a is not None:
                    assert _bits_equal(a, b), ctx
        assert n_ok >= 15
        # a band of output rows equals the rows of the full result
        P = rng.standard_normal((17, 21)).astype(np.float32)
        V = rng.standard_normal((2, 17, 21)) * 2
        full = extrap(P, V, 3, interp_order=3, map_coordinates_mode="nearest")
        band = extrap(P, V, 3, interp_order=3, map_coordinates_mode="nearest", b200_rows=(5, 11))
        assert _bits_equal(band, full[:, 5:11])


def test_extrapolate_members_equals_member_by_member_calls():
    """extrapolate_members (one batched launch per lead time) against the loop body of
    nowcasts/utils.py:440-458 spelled with single-member calls: same bits, float32 and float64
    precipitation, first lead time and carried displacements."""
    import pysteps_b200
    from pysteps_b200.extrapolation.semilagrangian import extrapolate, extrapolate_members
    init, gen = pysteps_b200.noise.get_method("bps")
    rng = np.random.default_rng(11)
    with cpu_abi.emulated():
        for dtype in (np.float64, np.float32):
            m, n, M = 40, 52, 3
            V = 2.0 * syn.velocity_field(m, n, 3)
            P = np.stack([syn.rain_field(m, n, 3 + j) for j in range(M)]).astype(dtype)
            perts = [init(V, 1.0, 5.0, randstate=np.random.RandomState(50 + j)) for j in range(M)]
            disp_b = None
            disp_s = [None] * M
            for t in range(3):
                Vm = [V + gen(perts[j], (t + 1) * 5.0) for j in range(M)]
                out_b, disp_b = extrapolate_members(P, Vm, displacement_prev=disp_b)
                for j in range(M):
                    o, disp_s[j] = extrapolate(P[j], Vm[j], [1.0], displacement_prev=disp_s[j], return_displacement=True)
                    assert out_b.dtype == o.dtype and np.array_equal(out_b[j], o[0], equal_nan=True), (dtype, t, j)
                    assert np.array_equal(np.asarray(disp_b)[j], np.asarray(disp_s[j])), (dtype, t, j)
            with pytest.raises(ValueError, match="same velocity"):
                V2 = V.copy()
                other = init(V2, 1.0, 5.0, randstate=np.random.RandomState(1))
                extrapolate_members(P[:2], [Vm[0], V2 + gen(other, 5.0)])
            with pytest.raises(TypeError):
                extrapolate_members(P[:1], [V])
        _ = rng


def test_float32_taps_host_logic():
    """b200_float32_taps: routed to its own C entry (emulated here by the exact loop), same return
    structure / dtypes / band shapes as the default path, and refused -- not silently recomputed some
    other way -- for what the variant does not cover."""
    from pysteps_b200.extrapolation.semilagrangian import extrapolate
    with cpu_abi.emulated():
        m, n = 30, 41
        V = 2.0 * syn.velocity_field(m, n, 3)
        for dtype in (np.float64, np.float32):
            P = syn.rain_field(m, n, 3).astype(dtype)
            want, dwant = extrapolate(P, V, 4, return_displacement=True)
            got, dgot = extrapolate(P, V, 4, return_displacement=True, b200_float32_taps=True)
            assert got.dtype == dtype and _bits_equal(got, want) and _bits_equal(dgot, dwant)
            band = extrapolate(P, V, 4, b200_float32_taps=True, b200_rows=(7, 19))
            assert _bits_equal(band, want[:, 7:19])
            o, d = extrapolate(P, V, [1.0], displacement_prev=dwant, return_displacement=True, b200_float32_taps=True)
            o2, d2 = extrapolate(P, V, [1.0], displacement_prev=dwant, return_displacement=True)
            assert _bits_equal(o, o2) and _bits_equal(d, d2)
        P = syn.rain_field(m, n, 3)
        x, y = np.meshgrid(np.arange(n, dtype=float), np.arange(m, dtype=float))
        # the default pixel grid given explicitly is still the default grid
        assert _bits_equal(extrapolate(P, V, 2, xy_coords=np.stack([x, y]), b200_float32_taps=True),
                           extrapolate(P, V, 2))
        for bad in (dict(n_iter=2), dict(n_iter=0), dict(interp_order=0), dict(interp_order=3),
                    dict(xy_coords=np.stack([x + 0.25, y]))):
            with pytest.raises(NotImplementedError, match="b200_float32_taps"):
                extrapolate(P, V, 2, b200_float32_taps=True, **bad)
        with pytest.raises(NotImplementedError, match="b200_float32_taps"):
            extrapolate(None, V, 2, return_displacement=True, b200_float32_taps=True)
        with pytest.raises(NotImplementedError, match="b200_float32_taps"):
            extrapolate(P, V, 40, b200_float32_taps=True)
        # the reference's own errors keep their precedence
        with pytest.raises(ValueError):
            extrapolate(P[0], V, 2, b200_float32_taps=True)
