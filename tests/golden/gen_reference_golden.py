"""Generate reference_golden.npz, reference_proesmans_golden.npz, reference_lk_host_golden.npz,
reference_host_golden.npz (CPU tests) and reference_gpu_golden.npz (GPU tests): outputs of
pysteps v1.21.3 itself on the inputs of tests/golden/reference_cases.py.  It needs the pysteps
v1.21.3 source tree (the PYSTEPS_REFERENCE directory of oracle/build_ref.py) with its two Cython
extensions built by oracle/build_ref.py, and cv2 / scipy / Cython / gcc: the Proesmans extension is compiled
here twice more, with the reference's flags and without -ffast-math.

    python oracle/build_ref.py && python tests/golden/gen_reference_golden.py

Large arrays are stored as fingerprints (tests/golden/fingerprint.py): a digest, and a seeded sample
where a tolerance is compared.
"""
import contextlib
import importlib.util
import io
import os
import subprocess
import sys
import sysconfig
import tempfile
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

import fingerprint as fp  # noqa: E402
import reference_cases as rc  # noqa: E402
from _refimport import ref_module  # noqa: E402


def _quiet(fn, *a, **k):
    with warnings.catch_warnings(), contextlib.redirect_stdout(io.StringIO()):
        warnings.simplefilter("ignore")
        return fn(*a, **k)


def gpu_golden():
    out = {}
    lk = ref_module("pysteps.motion.lucaskanade").dense_lucaskanade
    for shape, nframes, seed in rc.LK_GPU_CASES:
        key = f"lk/{shape[0]}x{shape[1]}x{nframes}/{seed}"
        fr = rc.lk_gpu_frames(shape, nframes, seed)
        xy, uv = _quiet(lk, fr.copy(), dense=False)
        fp.store(out, key + "/xy", xy)
        fp.store(out, key + "/uv", uv)
        fp.store(out, key + "/dense", _quiet(lk, fr.copy()), count=1024)
    sl = ref_module("pysteps.extrapolation.semilagrangian").extrapolate
    for case in range(6):
        P, V, ts, kw = rc.sl_gpu_case(case)
        fields, disp = sl(P, V, ts, return_displacement=True, **kw)
        fp.store(out, f"sl/{case}/fields", fields)
        fp.store(out, f"sl/{case}/displacement", disp)
    vet = ref_module("pysteps.motion.vet").vet
    fp.store(out, "vet/field", _quiet(vet, rc.vet_gpu_frames(), verbose=False), count=1024)
    return out


def cpu_golden():
    out = {}
    lk = ref_module("pysteps.motion.lucaskanade")
    cl = ref_module("pysteps.utils.cleansing")
    for i, (fr, kw) in enumerate(rc.lk_ckdtree_cases()):
        fp.store(out, f"lk_ckdtree/{i}", _quiet(lk.dense_lucaskanade, fr.copy(), **kw))
    for i, (fr, kw) in enumerate(rc.lk_tie_cases()):
        xy, uv = _quiet(lk.dense_lucaskanade, fr.copy(), **kw)
        fp.store(out, f"lk_ties/{i}/xy", xy)
        fp.store(out, f"lk_ties/{i}/uv", uv)
        raw = dict(kw, nr_std_outlier=1e9)
        axy, auv = _quiet(lk.dense_lucaskanade, fr.copy(), **raw)
        fp.store(out, f"lk_ties/{i}/raw_xy", axy)
        fp.store(out, f"lk_ties/{i}/raw_uv", auv)
        thr, k = kw.get("nr_std_outlier", 3), kw.get("k_outlier", 30)
        out[f"lk_ties/{i}/outliers"] = np.packbits(_quiet(cl.detect_outliers, auv, thr, axy, k))
    xy, uv = lk.dense_lucaskanade(rc.lk_live_frames(), dense=False)
    fp.store(out, "lk_live/xy", xy)
    fp.store(out, "lk_live/uv", uv)

    sl = ref_module("pysteps.extrapolation.semilagrangian").extrapolate
    for i, (P, V, ts, outval, kw) in enumerate(rc.spline_cases()):
        try:
            got = _quiet(sl, P.copy(), V.copy(), ts, outval, **kw)
        except ValueError as e:
            out[f"spline/{i}/error"] = np.array(str(e))
            continue
        for j, a in enumerate(got if isinstance(got, tuple) else (got,)):
            fp.store(out, f"spline/{i}/{j}", a)
    try:
        sl(np.ones((4, 4)), np.ones((2, 4, 4)), 1, interp_order=6)
    except RuntimeError as e:
        out["spline/order6_error"] = np.array(str(e))
    P, V = rc.sl_live_case()
    a, da = sl(P, V, 6, return_displacement=True)
    fp.store(out, "sl_live/fields", a)
    fp.store(out, "sl_live/displacement", da)

    nm = ref_module("pysteps.noise.motion")
    for name, V in rc.bps_live_cases():
        a = nm.initialize_bps(V, 0.5, 10.0, p_par=(3.0, 0.4, -1.0), randstate=np.random.RandomState(5))
        for k in ("vsf", "eps_par", "eps_perp"):
            out[f"bps/{name}/{k}"] = np.asarray(a[k])
        fp.store(out, f"bps/{name}/V_par", a["V_par"])
        fp.store(out, f"bps/{name}/V_perp", a["V_perp"])
        for t in rc.BPS_LIVE_TIMES:
            fp.store(out, f"bps/{name}/pert/{t}", nm.generate_bps(a, t))
            fp.store(out, f"bps/{name}/perturbed/{t}", V + nm.generate_bps(a, t))
    bad = np.ones((2, 4, 4))
    bad[1, 0, 0] = np.inf
    try:
        nm.initialize_bps(bad, 1, 1)
    except ValueError as e:
        out["bps/nonfinite_error"] = np.array(str(e))
    return out


def _proesmans_build(tmp, flags):
    """the reference's _proesmans.pyx compiled with `flags`; returns its proesmans() (proesmans.py:73-94)"""
    import numpy
    from scipy.ndimage import gaussian_filter
    from oracle import build_ref
    src = os.path.join(build_ref.REF, "pysteps", "motion", "_proesmans.pyx")
    c_file = os.path.join(tmp, "_proesmans.c")
    so = os.path.join(tmp, "_proesmans%d%s" % (len(os.listdir(tmp)), sysconfig.get_config_var("EXT_SUFFIX")))
    subprocess.check_call([sys.executable, "-m", "cython", "-3", src, "-o", c_file])
    subprocess.check_call(["gcc", "-shared", "-fPIC", "-fopenmp", "-w"] + flags
                          + [f"-I{sysconfig.get_paths()['include']}", f"-I{numpy.get_include()}", c_file, "-o", so])
    spec = importlib.util.spec_from_file_location("pysteps.motion._proesmans", so)
    ext = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(ext)

    def proesmans(input_images, lam=50.0, num_iter=100, num_levels=6, filter_std=0.0, full_output=False):
        im = np.stack([input_images[-2, :, :].copy(), input_images[-1, :, :].copy()])
        im_min, im_max = np.min(im), np.max(im)
        if im_max - im_min > 1e-8:
            im = (im - im_min) / (im_max - im_min) * 255.0
        if filter_std > 0.0:
            im[0, :, :] = gaussian_filter(im[0, :, :], filter_std)
            im[1, :, :] = gaussian_filter(im[1, :, :], filter_std)
        advfield, quality = ext._compute_advection_field(im, lam, num_iter, num_levels)
        return (advfield, quality) if full_output else advfield[0]

    return proesmans


def proesmans_golden():
    from proesmans_cases import build_case
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        strict = _proesmans_build(tmp, ["-O2", "-fno-fast-math", "-ffp-contract=off"])
        fast = _proesmans_build(tmp, ["-O3", "-ffast-math"])   # setup.py:27-28
        frames, _ = build_case("default_96x128")
        for std in rc.PROESMANS_PREFILTER_STDS:
            a, qa = strict(frames, filter_std=std, num_iter=10, num_levels=3, full_output=True)
            fp.store(out, f"proesmans_prefilter/{std}/advfield", a)
            fp.store(out, f"proesmans_prefilter/{std}/quality", qa)
        for i, (fr, kw) in enumerate(rc.proesmans_random_cases(21, 25)):
            a, qa = strict(fr, **kw)
            fp.store(out, f"proesmans_strict/{i}/advfield", a)
            fp.store(out, f"proesmans_strict/{i}/quality", qa)
        for i, (fr, kw) in enumerate(rc.proesmans_random_cases(22, 25)):
            a, _ = fast(fr, **kw)
            fp.store(out, f"proesmans_fast/{i}/advfield", a, count=64)
    return out


def _error_entry(err):
    return np.array("" if err is None else "%s: %s" % err)


def lk_host_golden():
    """tests/test_host_logic_lk.py: the reference's errors, sparse vectors and dense fields on the
    randomised calls of that module"""
    sys.path.insert(0, os.path.dirname(HERE))
    from test_host_logic_lk import _random_call, _run
    from pysteps_b200 import _synthetic as syn
    live = ref_module("pysteps.motion.lucaskanade").dense_lucaskanade
    out = {}
    for seed in range(4):
        rng = np.random.default_rng(500 + seed)
        for it in range(40):
            inp, kw = _random_call(rng)
            out[f"host/{seed}/{it}/error"] = _error_entry(_run(live, inp, kw)[1])
    rng = np.random.default_rng(2000)
    for it in range(60):
        inp, kw = _random_call(rng)
        ref, err = _run(live, inp, dict(kw, dense=False))
        out[f"sparse/{it}/error"] = _error_entry(err)
        if err is None:
            fp.store(out, f"sparse/{it}/xy", ref[0])
            fp.store(out, f"sparse/{it}/uv", ref[1])
    rng = np.random.default_rng(2001)
    for it in range(30):
        inp, kw = _random_call(rng)
        ref, err = _run(live, inp, dict(kw, dense=True))
        out[f"dense/{it}/error"] = _error_entry(err)
        if err is None:
            fp.store(out, f"dense/{it}/field", ref, count=64)
    rng = np.random.default_rng(0)
    for it in range(12):
        m, n = int(rng.integers(60, 160)), int(rng.integers(60, 160))
        fr = syn.rain_frames(m, n, int(rng.choice([2, 3])), int(rng.integers(0, 1000)), dx=2, dy=-1)
        if it % 2:
            fr = np.where(fr > 0.1, 10 * np.log10(np.maximum(fr, 0.1)), -15.0)
        fr = (fr + 0.37 * rng.standard_normal(fr.shape)).astype(np.float32)
        inp = fr if it % 3 else np.ma.masked_invalid(fr)
        xy, uv = _quiet(live, inp.copy(), dense=False)
        fp.store(out, f"float32/{it}/xy", xy)
        fp.store(out, f"float32/{it}/uv", uv)
    return out


def host_golden():
    """tests/test_host_logic_sl.py, test_host_logic_vet.py, test_kernel_bodies.py: the reference's
    results and errors on the seeded calls of those modules"""
    sys.path.insert(0, os.path.dirname(HERE))
    import test_host_logic_sl as tsl
    import test_host_logic_vet as tvet
    out = {}
    sl = ref_module("pysteps.extrapolation.semilagrangian").extrapolate
    for seed in range(6):
        rng = np.random.default_rng(100 + seed)
        for it in range(120):
            res, err, dep = tsl._run(sl, *tsl._random_call(rng))
            fp.store_call(out, f"sl/{seed}/{it}", res, err, raw=True)
            out[f"sl/{seed}/{it}/deprecations"] = "\n".join(dep)
    for seed in range(3):
        rng = np.random.default_rng(300 + seed)
        for it in range(60):
            Pin, Vin, ts, outval, kw = tsl._random_call(rng)
            kw["interp_order"] = int(rng.choice([0, 2, 3, 3, 4, 5]))
            res, err, dep = tsl._run(sl, Pin, Vin, ts, outval, kw)
            fp.store_call(out, f"spline/{seed}/{it}", res, err, raw=True)
            out[f"spline/{seed}/{it}/deprecations"] = "\n".join(dep)
    for vd, (V, P, steps) in rc.member_loop_case().items():
        po = _oracle_bps().initialize_bps(V, 0.5, 5.0, randstate=np.random.RandomState(9))
        dr = None
        for step in steps:
            o, dr = sl(P, V + _oracle_bps().generate_bps(po, step * 5.0), [1.0], displacement_prev=dr,
                       return_displacement=True, allow_nonfinite_values=True)
            fp.store(out, f"member_loop/{vd}/{step}/out", o, raw=True)
            fp.store(out, f"member_loop/{vd}/{step}/displacement", dr, raw=True)
    vet = ref_module("pysteps.motion.vet").vet
    for seed in range(3):
        rng = np.random.default_rng(700 + seed)
        for it in range(25):
            inp, kw = tvet._random_call(rng)
            res, err = tvet._run(vet, inp, kw)
            out[f"vet/{seed}/{it}/error"] = fp._error_text(err)
            if err is None:
                fp.store(out, f"vet/{seed}/{it}/field", res[0] if kw.get("intermediate_steps") else res, count=128)
    cl = ref_module("pysteps.utils.cleansing")
    for it, (uv, xy, k, thr) in enumerate(rc.outlier_body_cases()):
        if len(xy) >= 3:
            out[f"outliers/{it}"] = np.packbits(_quiet(cl.detect_outliers, uv, thr, xy, k))
    idw = ref_module("pysteps.utils.interpolate").idwinterp2d
    for it, (xy, uv, W, H, k, power, off) in enumerate(rc.idw_body_cases()):
        fp.store(out, f"idw/{it}", idw(xy, uv, np.arange(W), np.arange(H), power=power, k=k, dist_offset=off),
                 count=256)
    return out


def _oracle_bps():
    from oracle import noise_motion
    return noise_motion


def main():
    for name, make in (("reference_gpu_golden.npz", gpu_golden), ("reference_golden.npz", cpu_golden),
                       ("reference_proesmans_golden.npz", proesmans_golden),
                       ("reference_lk_host_golden.npz", lk_host_golden),
                       ("reference_host_golden.npz", host_golden)):
        path = os.path.join(HERE, name)
        fp.save(path, make())
        print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
