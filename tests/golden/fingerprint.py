"""Compact stored forms of large reference outputs, for fixtures that must stay small.

A fingerprint of an array is its dtype, shape and a SHA-256 digest of its bytes (every NaN written
as the one canonical NaN, so that NaN payloads do not count, as in conftest.bits_equal -- or, with
raw=True, the bytes as they are); the digest decides bit-identity over the WHOLE array.  Where a tolerance is compared, the values at a
seeded sample of flat positions are stored beside it, with the positions.

    store(out, "case/field", a[, count])  -> adds the entries to dict `out`
    save(path, out) / load(path)          -> .npz; every short string entry (fingerprints, error
                                             messages) is packed into two arrays
    assert_same(a, golden, "case/field")  -> bit-identical to the stored array
    assert_close(a, golden, "case/field", atol) -> bit-identical, or every sampled value within atol
    store_call / assert_call              -> the result of a call: its error, or each returned array
"""
import hashlib

import numpy as np


def _canonical(a):
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":
        a = np.where(np.isnan(a), np.array(np.nan, dtype=a.dtype), a)
    return a


def digest(a, raw=False):
    a = np.ascontiguousarray(a) if raw else _canonical(np.asarray(a))
    h = hashlib.sha256()
    h.update(f"{a.dtype.str}{a.shape}".encode())
    h.update(a.tobytes())
    return h.hexdigest()


def sample_positions(size, count):
    """flat positions sampled from an array of `size` elements (all of them when it is small)"""
    if size <= count:
        return np.arange(size)
    return np.sort(np.random.default_rng(size).choice(size, count, replace=False))


def store(out, key, a, count=0, raw=False):
    a = np.asarray(a)
    out[key] = "%s;%s;%s;%s" % (a.dtype.str, ",".join(map(str, a.shape)), digest(a, raw), "raw" if raw else "nan")
    if count:
        pos = sample_positions(a.size, count)
        out[key + "/positions"] = pos.astype(np.int32)
        out[key + "/sample"] = a.reshape(-1)[pos]


def sample(a, golden, key):
    """the values of `a` at the stored sample positions of `key`"""
    return np.asarray(a).reshape(-1)[golden[key + "/positions"]]


def save(path, out):
    text = {k: str(v) for k, v in out.items() if isinstance(v, str) or (isinstance(v, np.ndarray) and v.dtype.kind == "U")}
    arrays = {k: v for k, v in out.items() if k not in text}
    np.savez_compressed(path, _text_keys=np.array(sorted(text), dtype="S"),
                        _text_values=np.array([text[k] for k in sorted(text)], dtype="S"), **arrays)


def load(path):
    """-> dict: arrays as stored, packed strings as str"""
    with np.load(path) as z:
        d = {k: z[k] for k in z.files if not k.startswith("_text_")}
        d.update(zip((k.decode() for k in z["_text_keys"]), (v.decode() for v in z["_text_values"])))
    return d


def layout(golden, key):
    """(dtype, shape) of the stored array"""
    dt, shape = golden[key].split(";")[:2]
    return np.dtype(dt), tuple(int(s) for s in shape.split(",") if s)


def _check_layout(a, golden, key, what):
    a = np.asarray(a)
    dt, shape = layout(golden, key)
    assert a.dtype == dt, f"{what}: dtype {a.dtype} != {dt}"
    assert a.shape == shape, f"{what}: shape {a.shape} != {shape}"
    return a


def _digest_matches(a, golden, key):
    _, _, want, mode = golden[key].split(";")
    return digest(a, mode == "raw") == want


def assert_same(a, golden, key, what=""):
    a = _check_layout(a, golden, key, what or key)
    assert _digest_matches(a, golden, key), f"{what or key}: not bit-identical to the stored reference output"


def assert_close(a, golden, key, atol, what=""):
    a = _check_layout(a, golden, key, what or key)
    if _digest_matches(a, golden, key):
        return
    want = golden[key + "/sample"]
    got = sample(a, golden, key)
    assert np.array_equal(np.isnan(got), np.isnan(want)), f"{what or key}: NaN pattern"
    ok = ~np.isnan(want)
    d = np.abs(got[ok].astype(np.float64) - want[ok].astype(np.float64)).max() if ok.any() else 0.0
    assert d <= atol, f"{what or key}: max |d| = {d:.3e} > {atol:g} on {want.size} sampled values"


def _error_text(error):
    return "" if error is None else "%s: %s" % tuple(error)


def store_call(out, key, result, error, raw=False):
    """`result`: what a call returned (an array, None, or a tuple of them); `error`: None or the
    (exception type name, message) it raised instead"""
    out[key + "/error"] = _error_text(error)
    if error is None:
        items = result if isinstance(result, tuple) else (result,)
        out[key + "/returned"] = ("tuple:" if isinstance(result, tuple) else "single:") + \
            ",".join("none" if a is None else "array" for a in items)
        for j, a in enumerate(items):
            if a is not None:
                store(out, f"{key}/{j}", a, raw=raw)


def assert_call(result, error, golden, key, what=""):
    """the same error as the stored call, or the same return structure and bit-identical arrays"""
    assert _error_text(error) == golden[key + "/error"], f"{what}: error {error!r} != {golden[key + '/error']!r}"
    if error is None:
        items = result if isinstance(result, tuple) else (result,)
        returned = ("tuple:" if isinstance(result, tuple) else "single:") + \
            ",".join("none" if a is None else "array" for a in items)
        assert returned == golden[key + "/returned"], f"{what}: returned {returned} != {golden[key + '/returned']}"
        for j, a in enumerate(items):
            if a is not None:
                assert isinstance(a, np.ndarray), f"{what}: item {j} is a {type(a).__name__}"
                assert_same(a, golden, f"{key}/{j}", f"{what}: item {j}")
