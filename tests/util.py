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


# ---- Adam: float64 references and the comparison against them (optimiser tests) -------------------------------
LR, B1, B2, EPS = 1e-3, 0.9, 0.999, 1e-8
# the optimiser kernels receive fp32 hyper-parameters; the float64 references use exactly those values
HYPER = tuple(float(np.float32(x)) for x in (LR, B1, B2, EPS))
REPLAY = 160             # exact zero-gradient steps replayed per row (adam_math.cuh kMaxReplay, DESIGN §3.2)


def adam_ref(p, m, v, g, t, hyper=HYPER):
    """torch.optim.Adam, one step at step index t (1-based), in float64 (adam_math.cuh)."""
    lr, b1, b2, eps = hyper
    p, m, v, g = (np.asarray(x, np.float64) for x in (p, m, v, g))
    m = m + (1 - b1) * (g - m)
    v = b2 * v + (1 - b2) * g * g
    p = p - lr / (1 - b1 ** t) * m / (np.sqrt(v) / np.sqrt(1 - b2 ** t) + eps)
    return p, m, v


def lazy_ref(p, m, v, g, last, t, hyper=HYPER, step=True):
    """The all-rows step t of a row last stepped at `last` (0 = never, treated as current): replay the
    min(gap, 160) zero-gradient steps last+1 .. exactly, decay m and v by beta^gap in closed form, then take
    the real step t (DESIGN §3.2).  p, m, v, g: [rows, dim]; last: [rows].  Returns (p, m, v, gap).
    step=False is the replay-only form of catch-up and flush: rows with 0 < last < t replay gap = t - last
    zero-gradient steps and take no real step; rows with last = 0 or last >= t come back unchanged (gap 0)."""
    lr, b1, b2, eps = hyper
    p, m, v = (np.asarray(x, np.float64).copy() for x in (p, m, v))
    last = np.asarray(last, np.int64)[:, None]
    if step:
        gap = np.where(last > 0, t - 1 - last, 0)
    else:
        gap = np.where((last > 0) & (last < t), t - last, 0)
    n = np.minimum(gap, REPLAY)
    for j in range(1, int(n.max(initial=0)) + 1):
        s = last + j
        term = lr / (1 - b1 ** s) * (m * b1 ** j) / (np.sqrt(v) * np.sqrt(b2) ** j / np.sqrt(1 - b2 ** s) + eps)
        p -= np.where(j <= n, term, 0.0)
    m, v = m * b1 ** gap, v * b2 ** gap
    if step:
        p, m, v = adam_ref(p, m, v, g, t, hyper)
    return p, m, v, np.broadcast_to(gap, p.shape)


def assert_adam(p, p_ref, p_before, m, m_ref, v, v_ref, what, chained=None):
    """p within one final rounding plus 1e-5 of the step; m / v within 1e-6 of each tensor's largest
    element.  `chained` (optional, per element): zero-gradient steps the kernel replayed before the real one.
    Each of them rounds p once more in fp32, so such elements get chained * 2^-24 * |p| on top."""
    p, p_ref, p_before = (np.asarray(x, np.float64) for x in (p, p_ref, p_before))
    bar = 2.0 ** -23 * np.abs(p_ref) + 1e-5 * np.abs(p_ref - p_before)
    if chained is not None:
        bar = bar + np.minimum(chained, REPLAY) * 2.0 ** -24 * np.maximum(np.abs(p_ref), np.abs(p_before))
    err = np.abs(p - p_ref)
    bad = err > bar
    assert not bad.any(), (f"{what}: p off at {int(bad.sum())}/{bad.size} elements, worst err/bar "
                           f"{float((err / np.maximum(bar, 1e-300)).max()):.3g}")
    for name, a, r in (("m", m, m_ref), ("v", v, v_ref)):
        a, r = np.asarray(a, np.float64), np.asarray(r, np.float64)
        scale = max(float(np.abs(r).max(initial=0.0)), 1e-30)
        e = float(np.abs(a - r).max(initial=0.0)) / scale
        assert e <= 1e-6, f"{what}: {name} relative error {e:.3e} > 1e-6"
