"""Tolerance helper for the floating-point parity tests (north_star: "within 1e-4 rel fp32").

rel_check compares `got` with the oracle's `want` using the TRUE relative error on every element whose magnitude is
above `floor` x max|want| (default 1e-2), and an absolute bound of `small_atol` x max|want| on the elements below that
(their relative error is dominated by cancellation in the fp32 accumulation of the inputs themselves: measured on the
B200, the EXACT fp32 FMA kernel (precision 0) shows 1.35e-4 on elements between 1e-3 and 1e-2 of the maximum of a
64 -> 64 layer against the fp64-accumulating oracle, so no fp32 implementation meets 1e-4 there).  The achieved numbers are returned and, on the GPU box, appended to
gpurun_out/parity_errors.jsonl so they can be reported."""
import hashlib
import json
import os

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def rel_errors(got, want, floor=1e-2):
    got = np.asarray(got, np.float64)
    want = np.asarray(want, np.float64)
    assert got.shape == want.shape, (got.shape, want.shape)
    scale = float(np.abs(want).max()) if want.size else 0.0
    if scale == 0.0:
        return {"scale": 0.0, "max_rel": 0.0, "max_small_abs_over_scale": float(np.abs(got).max()) if got.size else 0.0,
                "n_big": 0}
    err = np.abs(got - want)
    big = np.abs(want) > floor * scale
    max_rel = float((err[big] / np.abs(want[big])).max()) if big.any() else 0.0
    small = float(err[~big].max() / scale) if (~big).any() else 0.0
    return {"scale": scale, "max_rel": max_rel, "max_small_abs_over_scale": small, "n_big": int(big.sum())}


def digest(*arrays):
    """SHA-256 over the arrays' dtypes, shapes and values: a bit-exact fingerprint of arrays too large to store as golden
    vectors.  -0.0 counts as 0.0 (as in np.array_equal / torch.equal)."""
    h = hashlib.sha256()
    for a in arrays:
        a = np.ascontiguousarray(a)
        if a.dtype.kind == "f":
            a = a + a.dtype.type(0)  # -0.0 + 0.0 == +0.0
        h.update(("%s%s" % (a.dtype.str, a.shape)).encode())
        h.update(a.tobytes())
    return h.hexdigest()


def rel_check(name, got, want, rtol=1e-4, floor=1e-2, small_atol=2e-6):
    e = rel_errors(got, want, floor)
    e.update({"name": name, "rtol": rtol, "floor": floor, "small_atol": small_atol})
    out = os.path.join(ROOT, "gpurun_out")
    if os.path.isdir(out):
        try:
            with open(os.path.join(out, "parity_errors.jsonl"), "a") as f:
                f.write(json.dumps(e) + "\n")
        except OSError:
            pass
    assert e["max_rel"] <= rtol, "%s: max relative error %.3e > %.1e (elements above %.0e x max)" % (
        name, e["max_rel"], rtol, floor)
    assert e["max_small_abs_over_scale"] <= small_atol, "%s: small-element abs error %.3e x max > %.1e" % (
        name, e["max_small_abs_over_scale"], small_atol)
    return e
