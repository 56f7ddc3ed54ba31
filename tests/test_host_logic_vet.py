"""CPU test of the HOST logic of pysteps_b200.motion.vet (argument handling, error messages,
padding / sector bookkeeping, indexing, intermediate steps, the SciPy optimiser loop) over
randomised argument combinations -- against the oracle's restatement of vet.py and the
reference's stored results and errors on the same calls (tests/golden/reference_host_golden.npz,
written by tests/golden/gen_reference_golden.py with the reference's extension built with its own
flags).  The three C-ABI entry points are emulated by the oracle (tests/cpu_abi.py): numerics here
say nothing about the kernels."""
import os
import warnings

import numpy as np
import pytest

import cpu_abi
import fingerprint as fp
from oracle import vet as ora
from pysteps_b200 import _synthetic as syn


@pytest.fixture(scope="module")
def golden():
    return fp.load(os.path.join(os.path.dirname(__file__), "golden", "reference_host_golden.npz"))


def _random_call(rng):
    m, n, T = int(rng.integers(24, 90)), int(rng.integers(24, 90)), int(rng.choice([2, 3]))
    fr = syn.rain_frames(m, n, T, int(rng.integers(0, 1000)), dx=int(rng.integers(-3, 4)), dy=int(rng.integers(-3, 4)))
    if rng.random() < 0.3:
        fr = np.stack([syn.nan_disc(f, 0.15) for f in fr])
    kw = {"options": dict(maxiter=int(rng.choice([2, 6])))}
    q = rng.random()
    if q < 0.15:
        kw["sectors"] = int(rng.choice([2, 4]))                     # scalar: rejected (vet.py:513-519)
    elif q < 0.5:
        kw["sectors"] = ((int(rng.choice([4, 8])), 2), (int(rng.choice([4, 6])), 2))
    elif q < 0.65:
        kw["sectors"] = [4, 2]
    else:
        kw["sectors"] = ((8, 4, 2), (8, 4, 2))
    if rng.random() < 0.3:
        kw["smooth_gain"] = float(rng.choice([1e3, 1e5, 1e7]))
    if rng.random() < 0.3:
        kw["padding"] = int(rng.choice([0, 3, 10]))
    if rng.random() < 0.3:
        kw["indexing"] = str(rng.choice(["yx", "xy", "ij", "zz"]))
    if rng.random() < 0.3:
        kw["intermediate_steps"] = True
    if rng.random() < 0.15:
        s = np.asarray(kw["sectors"])
        if s.ndim >= 1:
            s2 = s if s.ndim == 2 else np.stack([s, s])
            shape = (2, int(s2[0].min()), int(s2[1].min()))
            if rng.random() < 0.3:
                shape = (2, shape[1] + 1, shape[2])                 # wrong first-guess shape
            kw["first_guess"] = rng.standard_normal(shape)
    inp = fr
    q = rng.random()
    if q < 0.15:
        inp = np.ma.masked_array(np.nan_to_num(fr), mask=np.isnan(fr) | (rng.random(fr.shape) < 0.02))
    elif q < 0.2:
        inp = fr[0]
    elif q < 0.25:
        inp = np.concatenate([fr, fr])[:4]
    return inp, kw


def _run(fn, inp, kw):
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        try:
            return fn(inp.copy(), verbose=False, **{k: (v.copy() if isinstance(v, np.ndarray) else v) for k, v in kw.items()}), None
        except Exception as e:  # noqa: BLE001
            return None, (type(e).__name__, str(e))


@pytest.mark.parametrize("seed", range(3))
def test_vet_host_logic(seed, golden):
    from pysteps_b200.motion.vet import vet
    rng = np.random.default_rng(700 + seed)
    n_err = n_ok = 0
    with cpu_abi.emulated():
        for it in range(25):
            inp, kw = _random_call(rng)
            got, gerr = _run(vet, inp, kw)
            want, werr = _run(ora.vet, inp, kw)
            ctx = f"seed {seed} case {it}: shape={inp.shape} kw={ {k: (v.shape if isinstance(v, np.ndarray) else v) for k, v in kw.items()} }"
            assert gerr == werr, ctx
            assert fp._error_text(gerr) == golden[f"vet/{seed}/{it}/error"], ctx
            if gerr is not None:
                n_err += 1
                continue
            n_ok += 1
            if kw.get("intermediate_steps"):
                assert isinstance(got, tuple) and len(got[1]) == len(want[1]), ctx
                for a, b in zip(got[1], want[1]):
                    assert np.array_equal(np.asarray(a), np.asarray(b)), ctx
                got, want = got[0], want[0]
            # same cost / gradient evaluations and the same SciPy optimiser -> identical fields
            assert got.shape == want.shape and np.array_equal(got, want), ctx
            # the reference extension is built with -ffast-math
            fp.assert_close(got, golden, f"vet/{seed}/{it}/field", 1e-3, ctx)
    assert n_err >= 3 and n_ok >= 10, (n_err, n_ok)


def test_morph_and_cost_function_mirrors():
    from pysteps_b200.motion import vet as b200_vet
    rng = np.random.default_rng(3)
    img = syn.rain_field(40, 56, 1)
    disp = rng.standard_normal((2, 40, 56)) * 3
    with cpu_abi.emulated():
        w, wm, wg = b200_vet.morph(img, disp, gradient=True)
        o = ora.warp(img, np.zeros_like(img, dtype=np.int8), disp, gradient=True)
        assert np.array_equal(w, o[0]) and np.array_equal(wm, o[1]) and np.array_equal(wg, o[2])
        masked = np.ma.masked_array(img, mask=img > 5)
        w2, wm2 = b200_vet.morph(masked, disp)
        o2 = ora.warp(np.asarray(masked), np.ma.getmaskarray(masked).astype(np.int8), disp)
        assert np.array_equal(w2, o2[0]) and np.array_equal(wm2, o2[1])
        images = np.stack([img, np.roll(img, 2, axis=1), np.roll(img, 4, axis=1)])
        mask = np.zeros(img.shape, dtype=np.int8)
        sd = rng.standard_normal((2, 4, 4))
        for stack in (images, images[:2]):
            c = b200_vet.vet_cost_function(sd.ravel(), stack, (4, 4), mask, 1e5)
            g = b200_vet.vet_cost_function_gradient(sd.ravel(), stack, (4, 4), mask, 1e5)
            assert c == ora.vet_cost_function(sd.ravel(), stack, (4, 4), mask, 1e5)
            assert np.array_equal(g, ora.vet_cost_function_gradient(sd.ravel(), stack, (4, 4), mask, 1e5))
        with pytest.raises(ValueError, match="divide"):
            b200_vet.vet_cost_function(rng.standard_normal(2 * 3 * 3), images, (3, 3), mask, 1e5)
        with pytest.raises(NotImplementedError):
            b200_vet.vet_cost_function(rng.standard_normal(2), images, (1, 1), mask, 1e5)
