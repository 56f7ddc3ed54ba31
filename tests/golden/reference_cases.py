"""Inputs of the tests that compare with stored outputs of pysteps v1.21.3 itself
(reference_golden.npz, reference_gpu_golden.npz; written by gen_reference_golden.py).  The
generator and the tests build them here, from seeds, so that both see the same arrays."""
import numpy as np

from pysteps_b200 import _synthetic as syn

# ---------------------------------------------------------------- tests/test_reference_gpu.py
LK_GPU_CASES = [((512, 512), 2, 0), ((512, 512), 3, 1), ((301, 417), 3, 2), ((1024, 1024), 2, 3)]


def lk_gpu_frames(shape, nframes, seed):
    fr = syn.rain_frames(shape[0], shape[1], nframes, seed)
    if seed == 2:
        fr = np.stack([syn.nan_disc(f, 0.1) for f in fr])
    return fr


def sl_gpu_case(case):
    """-> P, V, timesteps, kwargs of semi-Lagrangian case `case` (0..5)"""
    m, n = ((256, 320), (511, 300), (128, 128), (400, 400), (200, 256), (333, 222))[case]
    P = syn.rain_field(m, n, case)
    V = syn.velocity_field(m, n, case, ("smooth", "rotation")[case % 2]) * (1.0 + case)
    kw = [dict(), dict(n_iter=3), dict(outval="min"), dict(interp_order=3, map_coordinates_mode="nearest"),
          dict(allow_nonfinite_values=True), dict(interp_order=0)][case]
    if case == 4:
        P = syn.nan_disc(P)
    ts = [4, 3, [0.5, 1.0, 2.5], 2, 3, 3][case]
    return P, V, ts, kw


def vet_gpu_frames():
    return syn.rain_frames(256, 256, 2, 3)


# ---------------------------------------------------------------- CPU oracle tests
def lk_ckdtree_cases():
    """tests/test_oracle_lk.py::test_ckdtree_mode_against_reference: (frames, kwargs) x 30"""
    rng = np.random.default_rng(77)
    for _ in range(30):
        m, n, T = int(rng.integers(50, 200)), int(rng.integers(50, 200)), int(rng.choice([2, 3]))
        fr = syn.rain_frames(m, n, T, int(rng.integers(0, 1000)), dx=int(rng.integers(-4, 5)), dy=int(rng.integers(-4, 5)))
        kw = {}
        if rng.random() < 0.4:
            kw["k_outlier"] = int(rng.choice([5, 30, 100]))
            kw["nr_std_outlier"] = float(rng.choice([1, 2, 3]))
        if rng.random() < 0.4:
            kw["interp_kwargs"] = dict(k=int(rng.choice([1, 4, 20, 30])), power=float(rng.choice([0.5, 1.0, 2.0])))
        if rng.random() < 0.3:
            kw["decl_scale"] = int(rng.choice([1, 5, 40]))
        yield fr, kw


def lk_tie_cases():
    """tests/test_oracle_lk.py::test_outlier_decisions_differ_from_the_reference_only_at_knn_ties:
    (frames, kwargs) x 40"""
    rng = np.random.default_rng(2024)
    for _ in range(40):
        m, n, T = int(rng.integers(60, 220)), int(rng.integers(60, 220)), int(rng.choice([2, 3]))
        fr = syn.rain_frames(m, n, T, int(rng.integers(0, 1000)), dx=int(rng.integers(-4, 5)), dy=int(rng.integers(-4, 5)))
        if rng.random() < 0.3:
            fr = np.stack([syn.nan_disc(f, 0.2) for f in fr])
        kw = {"dense": False}
        if rng.random() < 0.5:
            kw["k_outlier"] = int(rng.choice([5, 30, 100]))
            kw["nr_std_outlier"] = float(rng.choice([1, 2, 3]))
        if rng.random() < 0.3:
            kw["fd_kwargs"] = dict(max_corners=int(rng.choice([50, 300])), min_distance=int(rng.choice([3, 10])))
        if rng.random() < 0.3:
            kw["lk_kwargs"] = dict(winsize=(int(rng.choice([15, 31, 50])),) * 2, nr_levels=int(rng.integers(0, 4)))
        yield fr, kw


def lk_live_frames():
    return syn.rain_frames(220, 260, 2, 11, dx=-3, dy=2)


def spline_cases():
    """tests/test_oracle_spline.py: (P, V, timesteps, outval, kwargs) x 60, small and varied"""
    rng = np.random.default_rng(77)
    for _ in range(60):
        m, n = int(rng.integers(1, 30)), int(rng.integers(1, 30))
        P = (rng.standard_normal((m, n)) * 5).astype(rng.choice([np.float64, np.float32]))
        V = (rng.standard_normal((2, m, n)) * rng.choice([0.5, 3.0, 20.0])).astype(rng.choice([np.float64, np.float32]))
        kw = {"interp_order": int(rng.choice([0, 2, 3, 3, 4, 5])), "map_coordinates_mode": str(rng.choice(["constant", "nearest"]))}
        if rng.random() < 0.4:
            P[rng.random((m, n)) < 0.2] = np.nan
            kw["allow_nonfinite_values"] = True
        if rng.random() < 0.4:
            kw["n_iter"] = int(rng.integers(0, 4))
        if rng.random() < 0.4:
            kw["return_displacement"] = True
        outval = rng.choice([np.nan, 0.0, -15.0]) if rng.random() < 0.8 else "min"
        ts = int(rng.integers(1, 4)) if rng.random() < 0.5 else [0.5, 1.25]
        yield P, V, ts, outval, kw


def sl_live_case():
    P = syn.rain_field(150, 130, 5)
    V = syn.velocity_field(150, 130, 5, "rotation") * 3
    return P, V


def bps_live_cases():
    """tests/test_oracle_bps.py: (dtype name, V) x 3 and the lead times evaluated on each"""
    rng = np.random.default_rng(3)
    for dt in (np.float64, np.float32, np.int64):
        V = (10 * rng.standard_normal((2, 33, 47))).astype(dt)
        V[:, 3:6, 4:9] = 0
        yield np.dtype(dt).name, V


BPS_LIVE_TIMES = (0.0, 10.0, 55.0)


def proesmans_random_cases(seed, count):
    """tests/test_oracle_proesmans.py: (frames, kwargs) of randomised Proesmans calls"""
    rng = np.random.default_rng(seed)
    for _ in range(count):
        m, n = int(rng.integers(8, 160)), int(rng.integers(8, 160))
        lv = int(rng.integers(1, 6))
        if (m >> (lv - 1)) < 1 or (n >> (lv - 1)) < 1:
            continue   # an empty pyramid level: the reference reads out of bounds there
        fr = syn.rain_frames(m, n, 2, int(rng.integers(0, 100)), dx=int(rng.integers(-3, 4)), dy=int(rng.integers(-3, 4)))
        yield fr, dict(lam=float(rng.choice([5.0, 50.0, 1000.0])), num_iter=int(rng.choice([1, 7, 30, 100])),
                       num_levels=lv, full_output=True)


PROESMANS_PREFILTER_STDS = (0.8, 2.5)


def outlier_body_cases():
    """tests/test_kernel_bodies.py: (uv, xy, k, threshold) x 30 with many equidistant and coincident positions"""
    rng = np.random.default_rng(31)
    for it in range(30):
        n = int(rng.choice([2, 3, 10, 40, 300, 1500]))
        xy = np.floor(rng.uniform(0, rng.choice([6, 30, 200]), (n, 2)))
        if it % 3 == 0 and n >= 8:
            xy[: n // 4] = xy[n // 4: 2 * (n // 4)]
        uv = np.stack([2 + 0.3 * rng.standard_normal(n), -1 + 0.3 * rng.standard_normal(n)], 1)
        uv[::7] += 2.0
        k = int(rng.choice([5, 30, 100]))
        thr = float(rng.choice([1, 2, 3]))
        yield uv, xy, k, thr


def idw_body_cases():
    """tests/test_kernel_bodies.py: (xy, uv, W, H, k, power, dist_offset) x 14"""
    rng = np.random.default_rng(2)
    for it in range(14):
        n = int(rng.choice([2, 30, 200, 800]))
        W, H = int(rng.choice([40, 120])), int(rng.choice([30, 90]))
        xy = np.floor(rng.uniform(0, max(W, H), (n, 2)) * 2) / 2
        if it % 3 == 0 and n >= 8:
            xy[: n // 4] = xy[n // 4: 2 * (n // 4)]
        uv = np.ascontiguousarray(rng.standard_normal((n, 2)))
        k = int(min(rng.choice([1, 4, 20, 30]), n))
        power, off = float(rng.choice([0.5, 1.0, 2.0])), float(rng.choice([0.5, 1.0]))
        yield xy, uv, W, H, k, power, off


def member_loop_case():
    """tests/test_host_logic_sl.py::test_member_loop_with_handles_matches_reference_expression:
    {velocity dtype name: (V, P, member steps)}"""
    rng = np.random.default_rng(5)
    cases = {}
    for vd in (np.float64, np.float32):
        V = (3 * rng.standard_normal((2, 19, 23))).astype(vd)
        V[:, 4:7, 5:9] = 0
        P = rng.standard_normal((19, 23))
        P[2, 3] = np.nan
        cases[np.dtype(vd).name] = (V, P, (1, 2, 3))
    return cases
