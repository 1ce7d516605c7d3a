"""The touched-row optimiser entry points, one call at a time, against float64 Adam (DESIGN §3.2).

ncf_adam_step (lazy), ncf_adam_catchup, ncf_adam_prepare, ncf_adam_flush and ncf_sgd_step each run on a seeded
state: rows last stepped at 0, 1, 2, t-161, t-160, t-159, t-1 and t plus random steps, random moments, and
gradients in some rows only.  The models reach every path of the row kernels: the NeuMF fast path at d = 32
and d = 128, the float4 general loop (d = 256), scalar rows (f = 6), GMF and MLP alone.
"""
import ctypes

import numpy as np
import pytest
import torch

from ncf_b200._lib import NcfAdamHyper
from tests.util import HYPER, adam_ref, assert_adam, lazy_ref

gpu = pytest.mark.gpu

ERR_ARG = -1
U, I, T_NOW = 300, 200, 400        # table rows; the step counter before every call
EDGE = [0, 1, 2, T_NOW - 161, T_NOW - 160, T_NOW - 159, T_NOW - 1, T_NOW]
SGD_LR = float(np.float32(1e-2))
# (model_type, f, L): NeuMF fast path d = 32 and d = 128, float4 general loop d = 256 (the `big` bench shape),
# scalar rows, GMF, MLP
MODELS = [("NeuMF-end", 8, 3), ("NeuMF-end", 32, 3), ("NeuMF-end", 64, 3), ("NeuMF-end", 6, 2), ("GMF", 16, 1),
          ("MLP", 8, 2)]
MODEL_IDS = [f"{t}-f{f}-L{L}" for t, f, L in MODELS]
SIDES = (("user", U), ("item", I))


def _dev():
    return torch.device("cuda:0")


def _lib():
    from ncf_b200 import _lib
    return _lib.load()


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _bits(a):
    a = np.asarray(a)
    return a.view(np.int32) if a.dtype == np.float32 else a


def _same(a, b, what):
    assert np.array_equal(_bits(a), _bits(b)), what


# ---- seeded states ------------------------------------------------------------------------------------------------
class Case:
    """One model with its tables, tower, gradients and Adam state on the GPU, seeded from `seed` alone (two
    Cases of the same arguments hold the same bits)."""

    def __init__(self, model_type, f, L, seed):
        from ncf_b200 import ops
        self.type, self.f, self.L = model_type, f, L
        self.d = f << (L - 1)
        self.mt = {"GMF": 0, "MLP": 1, "NeuMF-end": 2}[model_type]
        self.kinds = [k for k in ("gmf", "mlp") if not (k == "gmf" and model_type == "MLP")
                      and not (k == "mlp" and model_type == "GMF")]
        gen = torch.Generator().manual_seed(seed)
        rnd = lambda *s, sc=0.1: (torch.randn(*s, generator=gen) * sc).to(_dev())
        self.tables = {"user_gmf": rnd(U, f), "item_gmf": rnd(I, f), "user_mlp": rnd(U, self.d),
                       "item_mlp": rnd(I, self.d)}
        widths = ops.tower_widths(f, L)
        lin = [(rnd(widths[k + 1], widths[k]), rnd(widths[k + 1])) for k in range(L)]
        pred = (rnd(1, {"GMF": f, "MLP": widths[-1]}.get(model_type, f + widths[-1])), rnd(1))
        self.tower = [x.reshape(-1) for wb in lin for x in wb] + [x.reshape(-1) for x in pred]
        self.m = ops.model_struct(self.mt, f, L, U, I, tuple(self.tables.values()), lin, pred)
        self.g = ops.GradBuffers.allocate(self.mt, f, L, U, I, max(U, I), _dev())
        self.s = ops.AdamBuffers.allocate(self.mt, f, L, U, I, _dev())
        for name, n in (("user", U), ("item", I)):
            for kind in self.kinds:
                key = f"{name}_{kind}"
                shape = self.tables[key].shape
                for pre in ("m_", "v_"):
                    x = torch.randn(shape, generator=gen) * 1e-3
                    getattr(self.s, pre + key).copy_(x * x if pre == "v_" else x)
                grad = torch.randn(shape, generator=gen) * 1e-3
                grad[torch.rand(n, generator=gen) < 0.6] = 0.0      # gradients in some rows only
                getattr(self.g, "g_" + key).copy_(grad)
            last = torch.randint(1, T_NOW + 1, (n,), generator=gen, dtype=torch.int32)
            last[torch.rand(n, generator=gen) < 0.1] = 0               # never stepped
            last[torch.rand(n, generator=gen) < 0.1] = T_NOW           # current already
            last[:len(EDGE)] = torch.tensor(EDGE, dtype=torch.int32)
            getattr(self.s, name + "_last_step").copy_(last)
        for buf in (self.s.m_tower, self.s.v_tower, self.g.g_tower):
            x = torch.randn(buf.shape, generator=gen) * 1e-3
            buf.copy_(x * x if buf is self.s.v_tower else x)
        self.s.step.fill_(T_NOW)
        self.gs, self.ss = self.g.struct(), self.s.struct()
        # the tower entries a step updates: all of them, or the predict layer alone for GMF
        n_pred = pred[0].numel() + 1
        n_tower = sum(x.numel() for x in self.tower)
        self.tower_upd = slice(n_tower - n_pred, n_tower) if model_type == "GMF" else slice(0, n_tower)

    def snap(self):
        """Every buffer an optimiser entry point may write, as numpy."""
        torch.cuda.synchronize()
        out = {}
        for key, tab in self.tables.items():
            out["p_" + key] = tab
            for pre, obj in (("m_", self.s), ("v_", self.s), ("g_", self.g)):
                t = getattr(obj, pre + key)
                if t is not None:
                    out[pre + key] = t
        out["p_tower"] = torch.cat(self.tower)
        out["m_tower"], out["v_tower"], out["g_tower"] = self.s.m_tower, self.s.v_tower, self.g.g_tower
        for name, _ in SIDES:
            out[name + "_last_step"] = getattr(self.s, name + "_last_step")
            out[name + "_flag"] = getattr(self.g, name + "_flag")
            out[name + "_list"] = getattr(self.g, name + "_list")
        out["touched"] = self.g.touched_count._base     # the two counts and the ticket word behind them
        out["step"] = self.s.step
        return {k: v.detach().cpu().numpy().copy() for k, v in out.items()}


def batch(B, seed):
    """B samples with repeated ids, the EDGE rows of both tables, and out-of-range ids on either side."""
    rng = np.random.default_rng(seed)
    u, i = rng.integers(0, U, B), rng.integers(0, I, B)
    k = min(B, len(EDGE))
    u[:k], i[:k] = np.arange(k), np.arange(k)
    if B >= 40:
        u[-3:] = [-1, U, U + 7]     # out of range: the whole sample is skipped, its item too
        i[-6:-3] = [-1, I, I + 7]
    return (torch.from_numpy(u).to(_dev()), torch.from_numpy(i).to(_dev()))


# ---- the entry points, through any loaded library -----------------------------------------------------------------
def hyper(b1=HYPER[1], b2=HYPER[2], eps=HYPER[3]):
    return NcfAdamHyper(HYPER[0], b1, b2, eps)


def mark_rows(lib, c, u, i):
    return lib.ncf_mark_rows(ctypes.byref(c.m), ctypes.byref(c.gs), u.data_ptr(), i.data_ptr(), u.numel(), _stream())


def mark_rows_side(lib, c, rows, side):
    return lib.ncf_mark_rows_side(ctypes.byref(c.m), ctypes.byref(c.gs), rows.data_ptr(), rows.numel(), side,
                                  _stream())


def adam_step(lib, c, h=None):
    return lib.ncf_adam_step(ctypes.byref(c.m), ctypes.byref(c.gs), ctypes.byref(c.ss), h or hyper(), _stream())


def adam_catchup(lib, c, h=None):
    return lib.ncf_adam_catchup(ctypes.byref(c.m), ctypes.byref(c.gs), ctypes.byref(c.ss), h or hyper(), _stream())


def adam_prepare(lib, c, u, i, h=None):
    return lib.ncf_adam_prepare(ctypes.byref(c.m), ctypes.byref(c.gs), ctypes.byref(c.ss), h or hyper(),
                                u.data_ptr(), i.data_ptr(), u.numel(), _stream())


def adam_flush(lib, c, h=None):
    return lib.ncf_adam_flush(ctypes.byref(c.m), ctypes.byref(c.ss), h or hyper(), _stream())


def sgd_step(lib, c):
    return lib.ncf_sgd_step(ctypes.byref(c.m), ctypes.byref(c.gs), SGD_LR, _stream())


def ok(rc, lib=None):
    assert rc == 0, (lib or _lib()).ncf_last_error()


# ---- checks -------------------------------------------------------------------------------------------------------
def listed(snap, name, side):
    return snap[name + "_list"][:int(snap["touched"][side])].copy()


def check_replayed(c, before, after, rows_of, t, step):
    """Rows rows_of[side] of every table against lazy_ref; every other row bit-unchanged.  Returns the per-side
    stamp the rows must carry."""
    for side, (name, n) in enumerate(SIDES):
        rows = rows_of[side]
        other = np.setdiff1d(np.arange(n), rows)
        last = before[name + "_last_step"][rows]
        for kind in c.kinds:
            key = f"{name}_{kind}"
            p0, m0, v0, g0 = (before[x + key][rows] for x in ("p_", "m_", "v_", "g_"))
            pr, mr, vr, gap = lazy_ref(p0, m0, v0, g0 if step else None, last, t, step=step)
            assert_adam(after["p_" + key][rows], pr, p0, after["m_" + key][rows], mr, after["v_" + key][rows], vr,
                        key, chained=gap)
            if step:
                assert not after["g_" + key][rows].any(), f"g_{key}: listed rows not zeroed"
            else:
                _same(after["g_" + key], before["g_" + key], f"g_{key}")
            for x in ("p_", "m_", "v_", "g_"):
                _same(after[x + key][other], before[x + key][other], f"{x}{key}: a row outside the list moved")
        for x in ("p_", "m_", "v_", "g_"):     # the tables the model does not have are never touched
            for kind in {"gmf", "mlp"} - set(c.kinds):
                if x + f"{name}_{kind}" in before:
                    _same(after[x + f"{name}_{kind}"], before[x + f"{name}_{kind}"], f"{x}{name}_{kind}")
        want = before[name + "_last_step"].copy()
        want[rows] = t if step else np.where((last > 0) & (last < t), t, last)
        _same(after[name + "_last_step"], want, f"{name} last_step")


def check_unchanged(before, after, keys):
    for k in keys:
        _same(after[k], before[k], f"{k} changed")


def distinct_rows(u, i):
    u, i = u.cpu().numpy(), i.cpu().numpy()
    ok_ = (u >= 0) & (u < U) & (i >= 0) & (i < I)
    return np.unique(u[ok_]), np.unique(i[ok_])


def same_state(a, b, what):
    """Bit-equal buffers; the touched lists up to their counts, and whole, as sets (their order is that of the
    atomics, and a closed step leaves its entries behind the zeroed counts)."""
    for k in a:
        if k.endswith("_list"):
            n = int(a["touched"][0 if k.startswith("user") else 1])
            _same(np.sort(a[k][:n]), np.sort(b[k][:n]), f"{what}: {k}")
            _same(np.sort(a[k]), np.sort(b[k]), f"{what}: {k} past the count")
        else:
            _same(a[k], b[k], f"{what}: {k}")


# ---- ncf_adam_step ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("model,register", [(m, "batch") for m in MODELS] + [(MODELS[0], "items only")],
                         ids=MODEL_IDS + [MODEL_IDS[0] + "-items-only"])
def test_adam_step_matches_lazy_reference(model, register):
    """Listed rows take their replay and step t; unlisted rows keep their bits; the tower takes dense Adam; the
    step is closed (counter + 1, counts and ticket word back to 0).  `items only`: the user list is empty and
    the items were registered through ncf_mark_rows_side."""
    lib = _lib()
    c = Case(*model, seed=11)
    if register == "batch":
        ok(mark_rows(lib, c, *batch(257, seed=1)))
    else:
        ok(mark_rows_side(lib, c, batch(120, seed=2)[1], 1))
    before = c.snap()
    assert (before["touched"][0] == 0) == (register == "items only")
    rows_of = [listed(before, "user", 0), listed(before, "item", 1)]
    ok(adam_step(lib, c))
    after = c.snap()
    t = T_NOW + 1
    check_replayed(c, before, after, rows_of, t, step=True)
    for side, (name, _) in enumerate(SIDES):
        want = before[name + "_flag"].copy()
        want[rows_of[side]] = 0
        _same(after[name + "_flag"], want, f"{name} flags")
    upd = c.tower_upd
    pr, mr, vr = adam_ref(*(before[k + "_tower"][upd] for k in ("p", "m", "v", "g")), t)
    assert_adam(after["p_tower"][upd], pr, before["p_tower"][upd], after["m_tower"][upd], mr, after["v_tower"][upd],
                vr, "tower")
    assert not after["g_tower"][upd].any()
    rest = np.ones(after["p_tower"].size, bool)
    rest[upd] = False
    for k in ("p_tower", "m_tower", "v_tower", "g_tower"):
        _same(after[k][rest], before[k][rest], f"{k}: unused layers of a GMF tower")
    assert int(after["step"][0]) == t
    assert after["touched"].tolist()[:3] == [0, 0, 0]


# ---- ncf_adam_catchup ---------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("model", MODELS, ids=MODEL_IDS)
def test_adam_catchup_matches_replay_reference(model):
    lib = _lib()
    c = Case(*model, seed=12)
    ok(mark_rows(lib, c, *batch(257, seed=3)))
    before = c.snap()
    rows_of = [listed(before, "user", 0), listed(before, "item", 1)]
    ok(adam_catchup(lib, c))
    after = c.snap()
    check_replayed(c, before, after, rows_of, T_NOW, step=False)
    check_unchanged(before, after, ["user_flag", "item_flag", "user_list", "item_list", "touched", "step",
                                    "p_tower", "m_tower", "v_tower", "g_tower"])


# ---- ncf_adam_prepare ---------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("B", [300, 4096, 4097, 20000])
@pytest.mark.parametrize("model", MODELS, ids=MODEL_IDS)
def test_adam_prepare_is_mark_rows_then_catchup(model, B):
    """Both sides of the B > 4096 switch (one fused launch below, mark + catch-up above): the lists hold the
    distinct rows of the in-range samples, the replay matches the reference, and the result is bit-equal to
    ncf_mark_rows followed by ncf_adam_catchup."""
    lib = _lib()
    u, i = batch(B, seed=B)
    c = Case(*model, seed=13)
    before = c.snap()
    ok(adam_prepare(lib, c, u, i))
    after = c.snap()
    want = distinct_rows(u, i)
    rows_of = []
    for side, (name, _) in enumerate(SIDES):
        got = listed(after, name, side)
        assert len(got) == len(want[side]) and np.array_equal(np.sort(got), want[side]), f"{name} list"
        fl = np.zeros_like(before[name + "_flag"])
        fl[want[side]] = 1
        _same(after[name + "_flag"], fl, f"{name} flags")
        rows_of.append(got)
    check_replayed(c, before, after, rows_of, T_NOW, step=False)
    check_unchanged(before, after, ["step", "p_tower", "m_tower", "v_tower", "g_tower"])
    assert after["touched"][2] == 0
    c2 = Case(*model, seed=13)
    ok(mark_rows(lib, c2, u, i))
    ok(adam_catchup(lib, c2))
    same_state(after, c2.snap(), "prepare vs mark_rows + catchup")


# ---- ncf_adam_flush -----------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("model", MODELS, ids=MODEL_IDS)
def test_adam_flush_replays_every_stale_row(model):
    lib = _lib()
    c = Case(*model, seed=14)
    before = c.snap()
    ok(adam_flush(lib, c))
    after = c.snap()
    check_replayed(c, before, after, [np.arange(U), np.arange(I)], T_NOW, step=False)
    check_unchanged(before, after, ["user_flag", "item_flag", "user_list", "item_list", "touched", "step",
                                    "p_tower", "m_tower", "v_tower", "g_tower"])


# ---- ncf_sgd_step -------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("model", MODELS, ids=MODEL_IDS)
def test_sgd_step_is_p_minus_lr_g_on_listed_rows(model):
    lib = _lib()
    c = Case(*model, seed=15)
    ok(mark_rows(lib, c, *batch(257, seed=4)))
    before = c.snap()
    ok(sgd_step(lib, c))
    after = c.snap()

    def near(got, p0, g0, what):
        ref = np.asarray(p0, np.float64) - SGD_LR * np.asarray(g0, np.float64)
        err = np.abs(np.asarray(got, np.float64) - ref)
        assert (err <= 2.0 ** -24 * np.abs(ref)).all(), f"{what}: beyond one fp32 rounding"

    for side, (name, n) in enumerate(SIDES):
        rows = listed(before, name, side)
        other = np.setdiff1d(np.arange(n), rows)
        for kind in c.kinds:
            key = f"{name}_{kind}"
            near(after["p_" + key][rows], before["p_" + key][rows], before["g_" + key][rows], key)
            assert not after["g_" + key][rows].any()
            for x in ("p_", "m_", "v_", "g_"):
                _same(after[x + key][other], before[x + key][other], f"{x}{key}: a row outside the list moved")
        assert not after[name + "_flag"].any()
    upd = c.tower_upd
    near(after["p_tower"][upd], before["p_tower"][upd], before["g_tower"][upd], "tower")
    assert not after["g_tower"][upd].any()
    assert after["touched"].tolist()[:3] == [0, 0, 0]
    check_unchanged(before, after, ["step", "m_tower", "v_tower", "user_last_step", "item_last_step",
                                    "user_list", "item_list"] + [k for k in before if k[:2] in ("m_", "v_")])


# ---- bit-exact equivalences ---------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("model", MODELS, ids=MODEL_IDS)
def test_catchup_then_step_equals_the_step_alone(model):
    lib = _lib()
    u, i = batch(257, seed=5)
    a, b = Case(*model, seed=16), Case(*model, seed=16)
    for c in (a, b):
        ok(mark_rows(lib, c, u, i))
    ok(adam_catchup(lib, a))
    ok(adam_step(lib, a))
    ok(adam_step(lib, b))
    same_state(a.snap(), b.snap(), "catch-up + step vs step")


@gpu
@pytest.mark.parametrize("model", MODELS, ids=MODEL_IDS)
def test_flush_equals_catchup_of_every_row(model):
    lib = _lib()
    a, b = Case(*model, seed=17), Case(*model, seed=17)
    ok(adam_flush(lib, a))
    for side, n in ((0, U), (1, I)):
        ok(mark_rows_side(lib, b, torch.arange(n, dtype=torch.int64, device=_dev()), side))
    ok(adam_catchup(lib, b))
    sa, sb = a.snap(), b.snap()
    for k in sa:
        if k[:2] in ("p_", "m_", "v_", "g_") or k.endswith("_last_step") or k == "step":
            _same(sa[k], sb[k], f"flush vs catch-up of every row: {k}")


# ---- bad hyper-parameters -----------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("bad", [dict(b1=1.0), dict(b2=0.0), dict(eps=0.0)], ids=["beta1=1", "beta2=0", "eps=0"])
@pytest.mark.parametrize("entry", ["catchup", "prepare", "flush"])
def test_replay_entries_refuse_bad_hyper_parameters(entry, bad):
    """ncf_adam_catchup, ncf_adam_prepare and ncf_adam_flush check the hyper-parameters as ncf_adam_step does:
    NCF_ERR_ARG before any launch, every buffer bit-unchanged."""
    lib = _lib()
    c = Case(*MODELS[0], seed=18)
    u, i = batch(257, seed=6)
    ok(mark_rows(lib, c, u, i))
    before = c.snap()
    h = hyper(**bad)
    rc = {"catchup": lambda: adam_catchup(lib, c, h), "prepare": lambda: adam_prepare(lib, c, u, i, h),
          "flush": lambda: adam_flush(lib, c, h)}[entry]()
    assert rc == ERR_ARG
    assert b"hyper" in lib.ncf_last_error()
    same_state(before, c.snap(), f"{entry} with {bad}")

