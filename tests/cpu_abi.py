"""TEST INFRASTRUCTURE: run the HOST side of pysteps_b200 (argument handling, validation order,
dtype / shape logic, lazy handles) on a machine without a GPU, by standing the oracle in for the
C-ABI entry points the semi-Lagrangian and BPS paths call.  Numerically this proves nothing about
the CUDA kernels (that is what the `-m gpu` tests are for); it lets the CPU suite compare the
host logic with the live reference on thousands of argument combinations.

    with cpu_abi.emulated():
        out = pysteps_b200.extrapolation.semilagrangian.extrapolate(P, V, 3)
"""
import contextlib
import ctypes
from unittest import mock

import numpy as np
import torch

from oracle import lib as oracle_lib
from oracle import noise_motion as ora_bps
from pysteps_b200 import _device, _lib

_NP = {_lib.F32: np.float32, _lib.F64: np.float64}
_C = {np.float32: ctypes.c_float, np.float64: ctypes.c_double, np.int8: ctypes.c_int8, np.uint8: ctypes.c_uint8,
      np.int32: ctypes.c_int32}


def _addr(p):
    if p is None:
        return None
    if isinstance(p, int):
        return p or None
    return ctypes.cast(p, ctypes.c_void_p).value


def _view(p, shape, dtype=np.float64):
    a = _addr(p)
    if a is None:
        return None
    n = int(np.prod(shape))
    buf = (_C[dtype] * n).from_address(a)
    return np.frombuffer(buf, dtype=dtype).reshape(shape)


def _field_stats(ptr, code, numel, out, stream):
    a = _view(ptr, (numel,), _NP[code])
    o = _view(out, (4,))
    fin = np.isfinite(a)
    o[0] = float(np.count_nonzero(~fin))
    nn = a[~np.isnan(a)]
    o[1] = nn.min() if nn.size else np.nan
    o[2] = nn.max() if nn.size else np.nan
    o[3] = float(np.count_nonzero(np.isnan(a)))


def _sl_rows_f32(precip, velocity, disp_prev, tdiff, T, vts, outval, mode, vdt, layout, pdt, m, n, r0, rows, out,
                 disp_out, fallback_count, stream):
    """the float32-tap entry: the emulation runs the exact loop (inside the documented tolerance)"""
    _sl_rows(precip, velocity, None, disp_prev, tdiff, T, vts, 1, outval, mode, vdt, layout, pdt, m, n, r0, rows,
             out, disp_out, stream)


def _sl_rows(precip, velocity, xy, disp_prev, tdiff, T, vts, n_iter, outval, mode, vdt, layout, pdt,
             m, n, r0, rows, out, disp_out, stream):
    vt, pt = _NP[vdt], _NP[pdt]
    if layout == _lib.LAYOUT_INTERLEAVED:
        V = np.ascontiguousarray(np.moveaxis(_view(velocity, (m, n, 2), vt), 2, 0), dtype=np.float64)
    else:
        V = np.ascontiguousarray(_view(velocity, (2, m, n), vt), dtype=np.float64)
    P = _view(precip, (m, n), pt)
    P = None if P is None else np.ascontiguousarray(P, dtype=np.float64)
    XY = _view(xy, (2, m, n))
    DP = None
    if _addr(disp_prev) is not None:
        DP = np.zeros((2, m, n))
        DP[:, r0:r0 + rows] = _view(disp_prev, (2, rows, n))
    td = np.ascontiguousarray(_view(tdiff, (T,)))
    full = None if P is None else np.empty((T, m, n))
    disp = np.empty((2, m, n))
    L = oracle_lib()
    dp = ctypes.POINTER(ctypes.c_double)
    L.ora_sl_extrapolate.restype = ctypes.c_int
    L.ora_sl_extrapolate.argtypes = [dp, dp, ctypes.c_int64, ctypes.c_int64, dp, dp, ctypes.c_int64,
                                     ctypes.c_double, ctypes.c_int, dp, ctypes.c_double, ctypes.c_int,
                                     ctypes.c_int, dp, dp]
    p = lambda a: None if a is None else a.ctypes.data_as(dp)  # noqa: E731
    rc = L.ora_sl_extrapolate(p(P), p(V), m, n, p(XY), p(td), T, vts, n_iter, p(DP), outval, mode,
                              int(vt is np.float32), p(full), p(disp))
    assert rc == 0
    if full is not None:
        _view(out, (T, rows, n), pt)[...] = full[:, r0:r0 + rows].astype(pt)
    if _addr(disp_out) is not None:
        _view(disp_out, (2, rows, n))[...] = disp[:, r0:r0 + rows]


def _sl_trajectories(velocity, xy, disp_prev, tdiff, T, vts, n_iter, vdt, layout, m, n, r0, rows, steps,
                     stream):
    """disp_steps[t] = the displacement after leadtime t: prefix runs of the oracle trajectory"""
    out = _view(steps, (T, 2, rows, n))
    tmp = np.empty((2, rows, n))
    for t in range(T):
        _sl_rows(None, velocity, xy, disp_prev, tdiff, t + 1, vts, n_iter, 0.0, 0, vdt, layout, _lib.F64,
                 m, n, r0, rows, None, tmp.ctypes.data, stream)
        out[t] = tmp


def _spline_prepare(precip, pdt, m, n, order, mode, stats, zero_fill, pole, zp0, zp1, coeffs, mmin, mfin,
                    stream):
    import host_kernels
    L = host_kernels.lib()
    L.host_spline_prepare.restype = None
    L.host_spline_prepare.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                      ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p,
                                      ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                      ctypes.c_void_p]
    L.host_spline_prepare(_addr(precip), pdt, m, n, order, mode, _addr(stats), zero_fill, _addr(pole),
                          _addr(zp0), _addr(zp1), _addr(coeffs), _addr(mmin), _addr(mfin))


def _spline_sample(coeffs, m, n, order, mode, xy, steps, T, r0, rows, outval, mmin, mfin, stats, odt, out,
                   stream):
    import host_kernels
    L = host_kernels.lib()
    L.host_spline_sample.restype = None
    L.host_spline_sample.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                     ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                     ctypes.c_double, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p,
                                     ctypes.c_int, ctypes.c_void_p]
    L.host_spline_sample(_addr(coeffs), m, n, order, mode, _addr(xy), _addr(steps), T, r0, rows, outval,
                         _addr(mmin), _addr(mfin), _addr(stats), odt, _addr(out))


def _proesmans_scale(frames, code, count, lo, hi, do_scale, out, stream):
    import host_kernels
    L = host_kernels.lib()
    src = np.ascontiguousarray(_view(frames, (count,), _NP[code]), dtype=np.float64)
    L.host_proesmans_scale.restype = None
    L.host_proesmans_scale(src.ctypes.data_as(ctypes.c_void_p), ctypes.c_int64(count), ctypes.c_double(lo),
                           ctypes.c_double(hi), int(do_scale), ctypes.c_void_p(_addr(out)))


def _gaussian_filter(src, h, w, weights, radius, out, stream):
    import host_kernels
    L = host_kernels.lib()
    L.host_gaussian_filter.restype = None
    vp = ctypes.c_void_p
    L.host_gaussian_filter(vp(_addr(src)), h, w, vp(_addr(weights)), radius, vp(_addr(out)))


def _proesmans_field(frames, m, n, lam, num_iter, num_levels, adv, quality, stream):
    import host_kernels
    L = host_kernels.lib()
    L.host_proesmans_field.restype = ctypes.c_int
    rc = L.host_proesmans_field(ctypes.c_void_p(_addr(frames)), m, n, ctypes.c_double(lam), num_iter, num_levels,
                                ctypes.c_void_p(_addr(adv)), ctypes.c_void_p(_addr(quality)))
    assert rc == 0


def _bps(velocity, code, m, n, a, b, vsf, what, out, nnf, stream):
    V = _view(velocity, (2, m, n), _NP[code])
    unit = np.zeros((2, m, n))
    with np.errstate(all="ignore"):
        speed = np.sqrt(V[0] * V[0] + V[1] * V[1])
        ok = speed > 1e-12
        for c in range(2):
            q = np.zeros((m, n), dtype=V.dtype)
            np.divide(V[c], speed, out=q, where=ok)
            unit[c] = q
        pert = (a * unit + b * np.stack([-unit[1], unit[0]])) / vsf
        res = {0: V + pert, 1: V + pert, 2: pert, 3: unit}[what]
    if what == 0:
        _view(out, (m, n, 2))[...] = np.moveaxis(res, 0, 2)
    else:
        _view(out, (2, m, n))[...] = res
    if _addr(nnf) is not None:
        _view(nnf, (1,))[0] = float(np.count_nonzero(~np.isfinite(res)))


def _sl_step_batched(velocity, vdt, m, n, members, coefs, vsf, precip, pdt, disp_prev, tdiff, vts, outval, mode,
                     out, disp_out, nnf, stream):
    """member by member: the emulated perturbation entry point, then the emulated single-step call"""
    vt, pt = _NP[vdt], _NP[pdt]
    ab = _view(coefs, (members, 2))
    tmp = np.empty((m, n, 2))
    bad = np.zeros(1)
    td = np.array([tdiff])
    N = m * n
    for j in range(members):
        _bps(velocity, vdt, m, n, float(ab[j, 0]), float(ab[j, 1]), vsf, 0, tmp.ctypes.data, bad.ctypes.data, stream)
        if _addr(nnf) is not None:
            _view(nnf, (members,))[j] = bad[0]
        dp = None if _addr(disp_prev) is None else _addr(disp_prev) + j * 2 * N * 8
        _sl_rows(_addr(precip) + j * N * np.dtype(pt).itemsize, tmp.ctypes.data, None, dp, td.ctypes.data, 1, vts, 1,
                 outval, mode, _lib.F64, _lib.LAYOUT_INTERLEAVED, pdt, m, n, 0, m,
                 _addr(out) + j * N * np.dtype(pt).itemsize, _addr(disp_out) + j * 2 * N * 8, stream)


def _vet_cost(sd, templ, inp, mask, xs, ys, nx, ny, smooth_gain, gradient, out, stream):
    from oracle import vet as ora_vet
    r = ora_vet.cost_function(_view(sd, (2, xs, ys)).copy(), _view(templ, (nx, ny)).copy(),
                              _view(inp, (nx, ny)).copy(), _view(mask, (nx, ny), np.int8).copy(),
                              smooth_gain, gradient=bool(gradient))
    if gradient:
        _view(out, (2, xs, ys))[...] = r
    else:
        _view(out, (2,))[...] = r


def _vet_value_and_gradient(x_host, images, nframes, mask, xs, ys, nx, ny, smooth_gain, work, value_host,
                            gradient_host, stream):
    """vet.py:257-293 with the oracle's _cost_function: pairs (centre, next) then (previous, centre)"""
    from oracle import vet as ora_vet
    sd = _view(x_host, (2, xs, ys)).copy()
    im = _view(images, (nframes, nx, ny))
    mk = _view(mask, (nx, ny), np.int8).copy()
    pairs = ((1, 2), (0, 1)) if nframes == 3 else ((0, 1),)
    parts = [(ora_vet.cost_function(sd, im[a].copy(), im[b].copy(), mk, smooth_gain, gradient=False),
              ora_vet.cost_function(sd, im[a].copy(), im[b].copy(), mk, smooth_gain, gradient=True))
             for a, b in pairs]
    res, smo = parts[0][0][0], parts[0][0][1]
    grad = parts[0][1]
    if nframes == 3:
        res = res + parts[1][0][0]
        smo = smo + parts[1][0][1]
        grad = grad + parts[1][1]
    _view(value_host, (2,))[...] = (res, smo)
    _view(gradient_host, (2, xs, ys))[...] = grad


def _vet_level_images(frames, umask, T, m, n, gpad, pi0, pj0, M, N, images, mask, stream):
    """vet.py:500-523 and :548-561, literally (numpy.pad), as the check of the device kernel's indexing"""
    fr = _view(frames, (T, m, n)).copy()
    bad = ~np.isfinite(fr) if _addr(umask) is None else _view(umask, (T, m, n), np.uint8).astype(bool)
    if gpad > 0:
        tup = ((0, 0), (gpad, gpad), (gpad, gpad))
        fr = np.pad(fr, tup, "constant", constant_values=np.nan)
        bad = np.pad(bad, tup, "constant", constant_values=True)
    fr[bad] = 0
    mk = np.any(bad, axis=0).astype(np.int8)
    pi1, pj1 = M - fr.shape[1] - pi0, N - fr.shape[2] - pj0
    _view(images, (T, M, N))[...] = np.pad(fr, ((0, 0), (pi0, pi1), (pj0, pj1)), "edge")
    _view(mask, (M, N), np.int8)[...] = np.pad(mk, ((pi0, pi1), (pj0, pj1)), "constant", constant_values=1)


def _vet_warp(image, mask, disp, nx, ny, out, omask, grad, stream):
    from oracle import vet as ora_vet
    g = _addr(grad) is not None
    r = ora_vet.warp(_view(image, (nx, ny)).copy(), _view(mask, (nx, ny), np.int8).copy(),
                     _view(disp, (2, nx, ny)).copy(), gradient=g)
    _view(out, (nx, ny))[...] = r[0]
    _view(omask, (nx, ny), np.int8)[...] = r[1]
    if g:
        _view(grad, (2, nx, ny))[...] = r[2]


def _zoom(a, c, h, w, oh, ow, out, stream):
    from oracle import vet as ora_vet
    _view(out, (c, oh, ow))[...] = ora_vet.zoom_o1(_view(a, (c, h, w)).copy(), oh, ow)


# ---- dense Lucas-Kanade: the entry points emulated with the oracle's stage functions -------------
# Device buffers carry their meaning between calls through this side table (pointer -> object):
# the eigenvalue map remembers the uint8 image it came from, a pyramid the image it was built of.
_side = {}


def _masked(img, mask, m, n):
    return np.ma.MaskedArray(_view(img, (m, n)).copy(), mask=_view(mask, (m, n), np.uint8).astype(bool))


def _lk_mask_invalid(img, user_mask, m, n, mask_out, stats, stream):
    a = _view(img, (m, n))
    mk = ~np.isfinite(a)
    if _addr(user_mask) is not None:
        mk |= _view(user_mask, (m, n), np.uint8).astype(bool)
    _view(mask_out, (m, n), np.uint8)[...] = mk
    good = a[~mk]
    _view(stats, (3,))[...] = [good.min() if good.size else np.nan, good.max() if good.size else np.nan, good.size]


def _lk_morph_opening(img, mask, m, n, size, thr, minv, out, stream):
    from oracle import lucaskanade as ora_lk
    ma = _masked(img, mask, m, n)
    np.ma.set_fill_value(ma, _view(minv, (1,))[0])
    r = ora_lk.morph_opening(ma, _view(thr, (1,))[0], size)
    _view(out, (m, n))[...] = np.ma.getdata(r)


def _lk_masked_minmax(img, mask, m, n, dilate, stats0, stats, stream):
    from oracle import lucaskanade as ora_lk
    a = _view(img, (m, n))
    mk = _view(mask, (m, n), np.uint8).astype(bool)
    st = _view(stats, (12,))
    st[...] = np.nan
    for s0, r0 in ((0, 0), (3, 1), (6, 2)):
        good = a[r0:][~mk[r0:]]
        st[s0:s0 + 3] = [good.min() if good.size else np.inf, good.max() if good.size else -np.inf, good.size]
    buffered = ora_lk.dilate_rect(mk.astype(np.uint8), int(dilate)) if dilate > 0 else mk.astype(np.uint8)
    st[11] = np.count_nonzero(buffered == 0)


def _lk_quantise(img, mask, m, n, mode, dilate, stats, fill, out, valid, stream):
    from oracle import lucaskanade as ora_lk
    ma = _masked(img, mask, m, n)
    if mode & 2:   # B200_QUANTISE_F32: the frames were float32 at the API
        ma = np.ma.MaskedArray(np.ma.getdata(ma).astype(np.float32), mask=np.ma.getmaskarray(ma))
    if (mode & 1) == 0:
        q = ora_lk.tracking_image(ma)
    else:
        q, v = ora_lk.detection_image(ma, dilate)
        _view(valid, (m, n), np.uint8)[...] = v
    _view(out, (m, n), np.uint8)[...] = q


def _lk_frontend(img, user_mask, m, n, size_opening, buffer_mask, flags, mask, stats0, stats, q_track, q_det,
                 valid, stream):
    """the four stage entry points in sequence, on host scratch"""
    opened = np.empty((m, n))
    op_ptr = opened.ctypes.data
    _lk_mask_invalid(img, user_mask, m, n, mask, stats0, stream)
    if size_opening > 0:
        _lk_morph_opening(img, mask, m, n, size_opening, stats0, stats0, op_ptr, stream)
    else:
        opened[...] = _view(img, (m, n))
    _lk_masked_minmax(op_ptr, mask, m, n, buffer_mask, stats0, stats, stream)
    _lk_quantise(op_ptr, mask, m, n, 0 | flags, 0, stats, stats, q_track, None, stream)
    if _addr(q_det) is not None:
        _lk_quantise(op_ptr, mask, m, n, 1 | flags, buffer_mask, stats, stats, q_det, valid, stream)


def _lk_min_eig(q, m, n, eig, stream):
    from oracle import lucaskanade as ora_lk
    img = _view(q, (m, n), np.uint8).copy()
    _view(eig, (m, n), np.float32)[...] = ora_lk.corner_min_eigen_val(img)
    _side[_addr(eig)] = img


def _lk_good_features(eig, valid, m, n, max_corners, quality, min_distance, out_xy, out_count, stream):
    from oracle import lucaskanade as ora_lk
    pts = ora_lk.good_features_to_track(_side[_addr(eig)], _view(valid, (m, n), np.uint8).copy(), max_corners,
                                        quality, min_distance)
    pts = np.asarray(pts, dtype=np.float32).reshape(-1, 2)
    _view(out_xy, (max_corners, 2), np.float32)[:len(pts)] = pts
    _view(out_count, (1,), np.int32)[0] = len(pts)


def _lk_build_pyramid(img, h, w, win_w, win_h, max_level, pyr, deriv, stream):
    if _addr(img) is not None:
        _side[_addr(pyr)] = _view(img, (h, w), np.uint8).copy()


def _lk_track(pyrI, pyrJ, derivI, h, w, win_w, win_h, max_level, max_count, eps, min_eig_thr, prev, npts, npts_dev,
              nxt, status, stream):
    from oracle import lucaskanade as ora_lk
    cnt = npts if _addr(npts_dev) is None else min(int(_view(npts_dev, (1,), np.int32)[0]), npts)
    if cnt == 0:
        return
    p0 = _view(prev, (npts, 2), np.float32)[:cnt].copy()
    p1, st = ora_lk.calc_optical_flow_pyr_lk(_side[_addr(pyrI)], _side[_addr(pyrJ)], p0, (win_w, win_h), max_level,
                                             (3, max_count, eps), min_eig_thr)
    _view(nxt, (npts, 2), np.float32)[:cnt] = p1
    _view(status, (npts,), np.uint8)[:cnt] = np.atleast_1d(np.asarray(st).squeeze())


def _lk_compact_tracks(p0, p1, status, npts_dev, cap, pool_xy, pool_uv, pool_count, pool_cap, stream):
    cnt = cap if _addr(npts_dev) is None else min(int(_view(npts_dev, (1,), np.int32)[0]), cap)
    a, b = _view(p0, (cap, 2), np.float32)[:cnt], _view(p1, (cap, 2), np.float32)[:cnt]
    keep = _view(status, (cap,), np.uint8)[:cnt] == 1
    pc = _view(pool_count, (1,), np.int32)
    k = int(keep.sum())
    _view(pool_xy, (pool_cap, 2))[pc[0]:pc[0] + k] = a[keep]
    _view(pool_uv, (pool_cap, 2))[pc[0]:pc[0] + k] = b[keep] - a[keep]   # float32 arithmetic, widened
    pc[0] += k


def _count(n_dev, cap):
    return cap if _addr(n_dev) is None else min(int(_view(n_dev, (1,), np.int32)[0]), cap)


def _lk_detect_outliers(uv, xy, n_dev, cap, thr, k, out, stream):
    """the kernel's own body (csrc/knn_body.cuh) compiled for the host"""
    import host_kernels
    cnt = _count(n_dev, cap)
    L = host_kernels.lib()
    L.host_detect_outliers_ckdtree.restype = None
    L.host_detect_outliers_ckdtree(ctypes.c_void_p(_addr(uv)), ctypes.c_void_p(_addr(xy)), cnt, ctypes.c_double(thr),
                                   int(k), ctypes.c_void_p(_addr(out)))


def _lk_detect_outliers_global(uv, n_dev, cap, thr, out, stream):
    from oracle import lucaskanade as ora_lk
    cnt = _count(n_dev, cap)
    if cnt:
        _view(out, (cap,), np.uint8)[:cnt] = ora_lk.detect_outliers(_view(uv, (cap, 2))[:cnt].copy(), thr)


def _lk_idw_fill_all(xy, vals, n_dev, cap, nvar, power, offset, mean_res, xg, nx, yg, ny, out, stream):
    _lk_idw_fill(xy, vals, n_dev, cap, nvar, None, power, offset, mean_res, xg, nx, yg, ny, 0, out, stream)


def _lk_compact_rows(xy, uv, drop, n_dev, cap, oxy, ouv, ocount, stream):
    cnt = _count(n_dev, cap)
    keep = _view(drop, (cap,), np.uint8)[:cnt] == 0
    k = int(keep.sum())
    _view(oxy, (cap, 2))[:k] = _view(xy, (cap, 2))[:cnt][keep]
    _view(ouv, (cap, 2))[:k] = _view(uv, (cap, 2))[:cnt][keep]
    _view(ocount, (1,), np.int32)[0] = k


def _lk_decluster(xy, uv, n_dev, cap, scale, min_samples, oxy, ouv, ocount, stream):
    from oracle import lucaskanade as ora_lk
    cnt = _count(n_dev, cap)
    k = 0
    if cnt:
        dxy, duv = ora_lk.decluster(_view(xy, (cap, 2))[:cnt].copy(), _view(uv, (cap, 2))[:cnt].copy(), scale,
                                    min_samples)
        k = len(dxy)
        _view(oxy, (cap, 2))[:k] = dxy
        _view(ouv, (cap, 2))[:k] = duv
    _view(ocount, (1,), np.int32)[0] = k


def _lk_idw_fill(xy, vals, n_dev, cap, nvar, k, power, offset, mean_res, xg, nx, yg, ny, on_grid, out, stream):
    from oracle import lucaskanade as ora_lk
    cnt = _count(n_dev, cap)
    gx, gy = _view(xg, (nx,)).copy(), _view(yg, (ny,)).copy()
    # the oracle derives the resolution from the grids (np.gradient needs two samples per axis);
    # the entry point is handed it (mean_res), so a one-row band is emulated on two rows
    ex = np.append(gx, gx[-1] + mean_res) if nx == 1 else gx
    ey = np.append(gy, gy[-1] + mean_res) if ny == 1 else gy
    r = ora_lk.idwinterp2d(_view(xy, (cap, 2))[:cnt].copy(), _view(vals, (cap, nvar))[:cnt].copy(),
                           ex, ey, power=power, k=k, dist_offset=offset)
    _view(out, (nvar, ny, nx))[...] = np.asarray(r).reshape(nvar, ey.size, ex.size)[:, :ny, :nx]


def _lk_idw_fill_ckdtree(xy, vals, n_dev, cap, nvar, k, power, offset, mean_res, xg, nx, yg, ny, out, stream):
    """the kernel's own body (csrc/knn_body.cuh) compiled for the host"""
    import host_kernels
    cnt = _count(n_dev, cap)
    L = host_kernels.lib()
    L.host_idw_fill_ckdtree.restype = None
    vp = ctypes.c_void_p
    L.host_idw_fill_ckdtree(vp(_addr(xy)), vp(_addr(vals)), cnt, nvar, min(k, cnt), ctypes.c_double(power),
                            ctypes.c_double(offset), ctypes.c_double(mean_res), vp(_addr(xg)), nx, vp(_addr(yg)),
                            ny, vp(_addr(out)))


def _fill_f64(ptr, count, value, stream):
    _view(ptr, (count,))[...] = value


_TABLE_LK = {"b200_mask_invalid": _lk_mask_invalid, "b200_morph_opening": _lk_morph_opening,
             "b200_masked_minmax": _lk_masked_minmax, "b200_quantise_u8": _lk_quantise,
             "b200_min_eig": _lk_min_eig, "b200_good_features": _lk_good_features,
             "b200_lk_build_pyramid": _lk_build_pyramid, "b200_lk_track": _lk_track,
             "b200_lk_compact_tracks": _lk_compact_tracks, "b200_lk_frontend": _lk_frontend,
          "b200_detect_outliers_global": _lk_detect_outliers_global, "b200_idw_fill_all": _lk_idw_fill_all, "b200_detect_outliers": _lk_detect_outliers,
             "b200_compact_rows": _lk_compact_rows, "b200_decluster": _lk_decluster,
             "b200_idw_fill": _lk_idw_fill, "b200_idw_fill_ckdtree": _lk_idw_fill_ckdtree, "b200_fill_f64": _fill_f64}

_TABLE = {"b200_vet_cost": _vet_cost, "b200_vet_value_and_gradient": _vet_value_and_gradient,
          "b200_vet_level_images": _vet_level_images, "b200_vet_warp": _vet_warp, "b200_zoom_bilinear": _zoom,
          "b200_gaussian_filter": _gaussian_filter, "b200_proesmans_scale": _proesmans_scale, "b200_proesmans_field": _proesmans_field,
          "b200_sl_trajectories": _sl_trajectories, "b200_spline_prepare": _spline_prepare,
          "b200_spline_sample": _spline_sample, "b200_field_stats": _field_stats, "b200_sl_extrapolate_rows": _sl_rows, "b200_sl_extrapolate_rows_f32": _sl_rows_f32,
          "b200_bps_perturb_velocity": _bps, "b200_sl_step_batched": _sl_step_batched}


def _call(name, *args):
    if name in _TABLE_LK:
        return _TABLE_LK[name](*args)
    if name not in _TABLE:
        raise NotImplementedError(f"cpu_abi: {name} is not emulated")
    _TABLE[name](*args)


def _to_device(a, dtype=None):
    if isinstance(a, _device.DeviceField):
        a = a.tensor
    t = a if isinstance(a, torch.Tensor) else torch.from_numpy(np.array(a, order="C"))
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    return t.contiguous()


class _Stream:
    cuda_stream = 0

    def __init__(self, *a, **k):
        pass

    def synchronize(self):
        pass

    def wait_event(self, e):
        pass

    def wait_stream(self, s):
        pass


class _Event:
    def __init__(self, *a, **k):
        pass

    def record(self, *a):
        pass

    def synchronize(self):
        pass


@contextlib.contextmanager
def emulated():
    real_empty = torch.empty

    def empty(*a, **k):
        k.pop("device", None)
        k.pop("pin_memory", None)
        return real_empty(*a, **k)

    with contextlib.ExitStack() as st:
        st.enter_context(mock.patch.object(_device, "require_cuda", lambda: None))
        st.enter_context(mock.patch.object(_device, "to_device", _to_device))
        st.enter_context(mock.patch.object(_device, "to_host", lambda t: t.clone().numpy()))
        st.enter_context(mock.patch.object(_device, "stream_ptr", lambda: 0))
        st.enter_context(mock.patch.object(_lib, "call", _call))
        st.enter_context(mock.patch.object(torch, "empty", empty))
        real_zeros = torch.zeros

        def zeros(*a, **k):
            k.pop("device", None)
            return real_zeros(*a, **k)

        st.enter_context(mock.patch.object(torch, "zeros", zeros))
        real_tensor = torch.tensor

        def tensor(*a, **k):
            k.pop("device", None)
            return real_tensor(*a, **k)

        st.enter_context(mock.patch.object(torch, "tensor", tensor))
        st.enter_context(mock.patch.object(torch.cuda, "Stream", _Stream))
        st.enter_context(mock.patch.object(torch.cuda, "Event", _Event))
        st.enter_context(mock.patch.object(torch.cuda, "stream", lambda s: contextlib.nullcontext()))
        st.enter_context(mock.patch.object(torch.cuda, "current_device", lambda: 0))
        _side.clear()
        st.enter_context(mock.patch.object(torch.cuda, "current_stream", lambda *a: _Stream()))
        # the module-level caches of streams, buffers and uploaded arrays get private, empty stand-ins:
        # on a machine with a GPU, a real stream cached by an earlier test would otherwise meet the
        # emulated events, and a host tensor cached here would later reach a real kernel as a pointer
        import threading
        from pysteps_b200.extrapolation import semilagrangian
        from pysteps_b200.motion import lucaskanade
        from pysteps_b200.noise import motion as noise_motion
        st.enter_context(mock.patch.object(lucaskanade, "_side_streams", {}))
        st.enter_context(mock.patch.object(lucaskanade, "_grids", {}))
        st.enter_context(mock.patch.object(lucaskanade, "_readback", threading.local()))
        st.enter_context(mock.patch.object(_device, "_recent", {}))
        st.enter_context(mock.patch.object(semilagrangian, "_pinned", threading.local()))
        st.enter_context(mock.patch.object(semilagrangian, "_default_grid_seen", {}))
        st.enter_context(mock.patch.object(noise_motion, "_fields", {}))
        # a device tensor's .cpu() is a fresh host copy; keep that property for the stand-ins
        st.enter_context(mock.patch.object(torch.Tensor, "cpu", lambda self, *a, **k: self.clone()))
        yield
