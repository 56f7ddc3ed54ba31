"""The CUDA path against pysteps v1.21.3 itself, on the B200.  Stand-alone functions are compared
with the reference's stored outputs (tests/golden/reference_gpu_golden.npz, written by
tests/golden/gen_reference_golden.py); the ensemble member loop and a whole nowcasts.steps forecast
run the reference's own loop, once with its stock methods and once with the B200 methods registered
over the stock names (pysteps_b200.register(override=True)), real kernels both times, and need the
reference in compiled form (oracle/_ref, built by oracle/build_ref.py)."""
import contextlib
import io
import os
import warnings

import fingerprint as fp
import numpy as np
import pytest
import reference_cases as rc

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def golden():
    import torch
    assert torch.cuda.is_available(), "gpu-marked test needs a GPU"
    return fp.load(os.path.join(os.path.dirname(__file__), "golden", "reference_gpu_golden.npz"))


@pytest.fixture(scope="module")
def ref():
    import torch
    assert torch.cuda.is_available(), "gpu-marked test needs a GPU"
    from oracle import refimport
    if not refimport.available(extensions=True):
        pytest.skip("the reference's own nowcast loop is needed: oracle/_ref has not been built "
                    "(python oracle/build_ref.py with the pysteps v1.21.3 source tree)")
    return refimport


def _quiet(fn, *a, **k):
    with warnings.catch_warnings(), contextlib.redirect_stdout(io.StringIO()):
        warnings.simplefilter("ignore")
        return fn(*a, **k)


@pytest.mark.parametrize("shape,nframes,seed", rc.LK_GPU_CASES)
def test_dense_lucaskanade_equals_the_reference(golden, shape, nframes, seed):
    import pysteps_b200
    key = f"lk/{shape[0]}x{shape[1]}x{nframes}/{seed}"
    lk = pysteps_b200.motion.get_method("lk")
    fr = rc.lk_gpu_frames(shape, nframes, seed)
    xy, uv = lk(fr.copy(), dense=False)
    fp.assert_same(xy, golden, key + "/xy", "sparse vectors")
    fp.assert_same(uv, golden, key + "/uv", "sparse vectors")
    V = lk(fr.copy())
    fp.assert_close(V, golden, key + "/dense", 1e-12, "dense field")
    # every pixel, against the oracle (tests/test_oracle_lk.py pins it to the reference's stored fields)
    from oracle import lucaskanade as ora
    assert np.abs(V - ora.dense_lucaskanade(fr.copy())).max() <= 1e-12, "dense field at every pixel"


@pytest.mark.parametrize("case", range(6))
def test_extrapolate_equals_the_reference(golden, case):
    import pysteps_b200
    sl = pysteps_b200.extrapolation.get_method("semilagrangian")
    P, V, ts, kw = rc.sl_gpu_case(case)
    got, gd = sl(P, V, ts, return_displacement=True, **kw)
    fp.assert_same(got, golden, f"sl/{case}/fields", f"case {case} fields")
    fp.assert_same(gd, golden, f"sl/{case}/displacement", f"case {case} displacement")


def test_vet_close_to_the_reference_build(golden):
    """the reference extension is built with -ffast-math (setup.py:27-28): 1e-6 px"""
    import pysteps_b200
    vet = pysteps_b200.motion.get_method("vet")
    fp.assert_close(vet(rc.vet_gpu_frames(), verbose=False), golden, "vet/field", 1e-6)


def test_steps_forecast_with_registered_b200_methods(ref):
    """Unmodified pysteps.nowcasts.steps.forecast (cascade, AR model, noise, BPS velocity
    perturbations, AR pre-alignment through the extrapolator, member loop), 3 members on 200^2,
    seeded: stock registries, then the same call with the B200 kernels registered OVER the stock
    names -- identical output."""
    import pysteps_b200
    from pysteps_b200 import _synthetic as syn
    steps = ref.ref_module("pysteps.nowcasts.steps")
    ex_if = ref.ref_module("pysteps.extrapolation.interface")
    mo_if = ref.ref_module("pysteps.motion.interface")
    no_if = ref.ref_module("pysteps.noise.interface")
    m = n = 200
    fr = syn.rain_frames(m, n, 3, 4, dx=2, dy=-1)
    R = np.where(fr > 0.1, 10 * np.log10(np.maximum(fr, 0.1)), -15.0)
    kw = dict(timesteps=4, n_ens_members=3, n_cascade_levels=4, precip_thr=-10.0, kmperpixel=1.0, timestep=5.0,
              noise_method="nonparametric", seed=42, num_workers=1)
    saved = (dict(ex_if._extrapolation_methods), dict(mo_if._methods), dict(no_if._noise_methods))
    try:
        V_stock = _quiet(mo_if.get_method("lk"), fr)
        want = _quiet(steps.forecast, R, V_stock, **kw)
        pysteps_b200.register(override=True)
        assert ex_if.get_method("semilagrangian").__module__.startswith("pysteps_b200")
        V = _quiet(mo_if.get_method("lk"), fr)
        assert np.abs(V - V_stock).max() <= 1e-12
        got = _quiet(steps.forecast, R, V_stock, **kw)
        got_resident = _quiet(steps.forecast, R, V_stock, extrap_kwargs={"b200_resident": True}, **kw)
    finally:
        for reg, old in zip((ex_if._extrapolation_methods, mo_if._methods, no_if._noise_methods), saved):
            reg.clear()
            reg.update(old)
    assert want.shape == got.shape == (3, 4, m, n) and np.isfinite(want).any()
    assert np.array_equal(want, got, equal_nan=True)
    assert np.array_equal(want, got_resident, equal_nan=True)


def test_nowcast_main_loop_ensemble_with_b200_methods(ref):
    import pysteps_b200
    from pysteps_b200 import _synthetic as syn
    utils = ref.ref_module("pysteps.nowcasts.utils")
    noise = ref.ref_module("pysteps.noise.interface")
    pysteps_b200.register()
    m, n, members = 200, 240, 3
    precip = syn.rain_field(m, n, 5)
    velocity = 2.0 * syn.velocity_field(m, n, 5)
    params = {"decay": 0.97, "bias": np.array([0.0, 0.1, -0.05])}
    state0 = np.stack([precip * (1 + 0.05 * i) for i in range(members)])

    def model(state, params):
        fields = state["fields"] * params["decay"] + params["bias"][:, None, None]
        return fields, {"fields": fields}

    def run(noise_name, extrap_name, extrap_kwargs, timesteps):
        init, gen = noise.get_method(noise_name)
        perts = []
        for j in range(members):
            vp = init(velocity, 1.0, 5.0, randstate=np.random.RandomState(100 + j))
            perts.append(lambda t, vp=vp: gen(vp, t * 5.0))   # nowcasts/steps.py:927-929
        return utils.nowcast_main_loop(precip, velocity, {"fields": state0.copy()}, timesteps, extrap_name, model,
                                       extrap_kwargs=extrap_kwargs, velocity_pert_gen=perts, params=params,
                                       ensemble=True, num_ensemble_members=members)

    for timesteps in (3, [0.5, 1.0, 2.25, 3.0]):
        want = _quiet(run, "bps", "semilagrangian", {"allow_nonfinite_values": True}, timesteps)
        got = _quiet(run, "bps_b200", "semilagrangian_b200", {"allow_nonfinite_values": True, "b200_resident": True},
                     timesteps)
        for g_member, w_member in zip(got, want):
            for g, w in zip(g_member, w_member):
                assert np.array_equal(g, w, equal_nan=True)
