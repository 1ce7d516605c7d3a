"""The kernels behind the two multi-GPU layouts (DESIGN §5), checked on ONE device with emulated ranks.

Every exchange kernel takes each rank's buffers as a plain array of device addresses, so N ranks are N
ordinary allocations on cuda:0.  Phase k of every rank is issued, in rank order, before phase k+1 of any rank;
the order of the one stream stands in for the rank barriers between phases.  Nothing here maps IPC handles
or starts a second process, and every barrier launch finds its peers already arrived (see the barrier test).

References are float64 numpy, written out in this file; the CPU-only tests at the top check them against
literal loops (step-by-step dense Adam, brute-force bucketing) so that the GPU tests compare against
something that is itself pinned.
"""
import ctypes

import numpy as np
import pytest
import torch

from oracle import ncf_numpy as onp
from tests.util import HYPER, REPLAY, adam_ref, assert_adam, assert_close, lazy_ref

gpu = pytest.mark.gpu

ERR_ARG = -1
STEPS = [0, 1, 4, 999]   # step counters before the call; at 999 an off-by-one bias correction moves p by ~3e-4


def _dev():
    return torch.device("cuda:0")


def _lib():
    from ncf_b200 import _lib
    return _lib.load()


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(_dev())


def _bits(t):
    """Bit pattern of a float tensor / array (NaN-safe exact comparison)."""
    a = t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)
    return a.view(np.int32) if a.dtype == np.float32 else a


def _same(a, b, what):
    assert np.array_equal(_bits(a), _bits(b)), what


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptrs(addresses):
    return (ctypes.c_void_p * len(addresses))(*addresses)


# ---- float64 references ----------------------------------------------------------------------------------------
def bucket_ref(item, world):
    """(owner, local index) of every sample: owner item % world, local item // world; a negative item goes
    to owner 0 with local index -1."""
    item = np.asarray(item, np.int64)
    neg = item < 0
    return np.where(neg, 0, item % world), np.where(neg, -1, item // world)


def inbox_ref(items, world, item_num):
    """Requests of every rank: {owner: {source rank: sorted list of (local row << 32) | slot}}."""
    out = {o: {r: [] for r in range(len(items))} for o in range(world)}
    for r, it in enumerate(items):
        it = np.asarray(it, np.int64)
        ok = (it >= 0) & (it < item_num)
        s = np.nonzero(ok)[0]
        for o in range(world):
            sel = s[it[s] % world == o]
            out[o][r] = sorted(((it[sel] // world) << 32 | sel).tolist())
    return out


def sum_bound(k, abs_sum):
    """fp32 summation of k terms: |error| <= k * 2^-24 * sum |terms|."""
    return k * 2.0 ** -24 * abs_sum


# ---- CPU: the references against literal loops -----------------------------------------------------------------
_LAZY_STEP = [(5, 100), (37, 198), (1, 162), (3, 400), (12, 700), (250, 500), (0, 50), (99, 100)]
_LAZY_REPLAY = _LAZY_STEP + [(100, 100), (120, 100)]


@pytest.mark.parametrize("last,t,step", [(a, b, True) for a, b in _LAZY_STEP] + [(a, b, False) for a, b in _LAZY_REPLAY],
                         ids=[f"{a}-{b}" for a, b in _LAZY_STEP] + [f"{a}-{b}-replay" for a, b in _LAZY_REPLAY])
def test_lazy_reference_matches_dense_adam_step_by_step(monkeypatch, last, t, step):
    """lazy_ref == oracle DenseAdam run step by step with zero gradients from step last+1 to t-1, then with
    the real gradient at step t.  Replay only (step=False, catch-up and flush): zero gradients from step last+1
    to t and no real step, nothing at all for last = 0 or last >= t.  DenseAdam is run in float64 (its fp32
    casts patched out) so that only the truncation of the replay remains: DESIGN §3.2 bounds the terms dropped
    beyond 160 steps, all together, by 1.4e-6 of the first replayed term (the largest ratio, 1.39e-6, is at
    last = 12; the bias corrections make early rows decay slower than (b1/sqrt(b2))^j)."""
    monkeypatch.setattr(onp, "F32", np.float64)
    rng = np.random.default_rng(last * 1000 + t)
    p0 = rng.standard_normal((4, 6)) * 0.1
    m0 = rng.standard_normal((4, 6)) * 1e-3
    v0 = (rng.standard_normal((4, 6)) * 1e-3) ** 2
    g = rng.standard_normal((4, 6)) * 1e-3
    g[1] = 0.0
    lr, b1, b2, eps = HYPER
    opt = onp.DenseAdam(lr, b1, b2, eps)
    params = {"w": p0.copy()}
    replay = last > 0 and (step or last < t)
    # last = 0 (never stepped) counts as current: the real step is step t
    opt.state["w"] = {"t": last if last > 0 else t - 1, "m": m0.copy(), "v": v0.copy()}
    if replay:
        for _ in range(last + 1, t if step else t + 1):
            opt.step(params, {"w": np.zeros_like(p0)})
    if step:
        opt.step(params, {"w": g})
    p, m, v, gap = lazy_ref(p0, m0, v0, g if step else None, np.full(4, last), t, step=step)
    want_gap = (t - 1 - last if step else t - last) if replay else 0
    assert int(gap.max()) == int(gap.min()) == want_gap
    first = lr / (1 - b1 ** (last + 1)) * np.abs(m0) * b1 / (np.sqrt(v0 * b2) / np.sqrt(1 - b2 ** (last + 1)) + eps)
    tail = 1.4e-6 * first if want_gap > REPLAY else 0.0
    assert np.all(np.abs(p - params["w"]) <= tail + 1e-12 * np.abs(p0) + 1e-15)
    assert np.allclose(m, opt.state["w"]["m"], rtol=1e-12, atol=0)
    assert np.allclose(v, opt.state["w"]["v"], rtol=1e-12, atol=0)


def test_bucket_reference_matches_brute_force():
    rng = np.random.default_rng(3)
    item = np.concatenate([rng.integers(0, 2 ** 40, 200), [-1, -1, -7, -(2 ** 40), 0, 63, 64, 65]])
    for world in (1, 2, 3, 7, 8, 64):
        owner, local = bucket_ref(item, world)
        for b, it in enumerate(item.tolist()):
            if it < 0:
                assert (owner[b], local[b]) == (0, -1)
            else:
                o = it - (it // world) * world
                assert (owner[b], local[b]) == (o, it // world) and local[b] * world + o == it


def test_inbox_reference_matches_brute_force():
    item_num, world = 50, 3
    items = [np.array([0, 5, 49, -1, 50, 5, 3]), np.array([], np.int64), np.array([2, 1, 0])]
    ref = inbox_ref(items, world, item_num)
    for o in range(world):
        for r, it in enumerate(items):
            want = []
            for s, x in enumerate(it.tolist()):
                if 0 <= x < item_num and x % world == o:
                    want.append((x // world) * 2 ** 32 + s)
            assert ref[o][r] == sorted(want)


# ---- 1. the fused step as the multi-GPU layouts call it ----------------------------------------------------------
def _near_relu_kink(params, u, i, L, tol=3e-6):
    from tests.test_gpu_umma import _near_relu_kink as kink
    return kink(params, u, i, L, tol)


def _tower_keys(L):
    """The flat tower gradient layout; a GMF model keeps the (unused) tower layers in it too."""
    keys = [f"MLP_layers.{3 * k + 1}.{s}" for k in range(L) for s in ("weight", "bias")]
    return keys + ["predict_layer.weight", "predict_layer.bias"]


def _model(model_type, f, L, U, I, seed):
    from ncf_b200.models import NCF
    torch.manual_seed(seed)
    model = NCF(U, I, f, L, 0.0, model_type).to(_dev())
    with torch.no_grad():   # the reference zero-initialises the biases; make them matter
        for lin in model.linears():
            lin.bias.uniform_(-0.1, 0.1)
    return model, {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}


def _batch(params, model_type, L, U, I, B, rng):
    u = rng.integers(0, U, B + 64)
    i = rng.integers(0, I, B + 64)
    if model_type != "GMF":
        keep = ~_near_relu_kink(params, u, i, L)
        u, i = u[keep], i[keep]
    assert u.size >= B
    return u[:B], i[:B]


def _loss_ref(logits, y, teacher, alpha, B_norm):
    """Loss and dloss/dlogit of the fused step when the mean runs over B_norm samples."""
    x, y = logits.astype(np.float64), y.astype(np.float64)
    sig = 1.0 / (1.0 + np.exp(-x))
    bce = onp.bce_with_logits(logits, y)
    if teacher is None:
        return bce.sum() / B_norm, (sig - y) / B_norm
    t = teacher.astype(np.float64)
    return ((alpha * bce + (1 - alpha) * (x - t) ** 2).sum() / B_norm,
            (alpha * (sig - y) + (1 - alpha) * 2.0 * (x - t)) / B_norm)


def _step_norm(m, g, ud, idd, yd, teacher, alpha, B_norm):
    from ncf_b200 import ops
    B = ud.numel()
    ws = torch.empty(ops.train_workspace_bytes(m, B), dtype=torch.uint8, device=_dev())
    loss = torch.zeros(1, dtype=torch.float64, device=_dev())
    logits = torch.empty(B, device=_dev())
    ops.mark_rows(m, g.struct(), ud, idd)
    rc = _lib().ncf_train_step_grads_norm(
        ctypes.byref(m), ctypes.byref(g.struct()), ud.data_ptr(), idd.data_ptr(), yd.data_ptr(),
        teacher.data_ptr() if teacher is not None else None, alpha, B, B_norm, loss.data_ptr(), logits.data_ptr(),
        ws.data_ptr(), ws.numel(), _stream())
    assert rc == 0, _lib().ncf_last_error()
    torch.cuda.synchronize()
    return float(loss.item()), logits.cpu().numpy()


def _check_tower(g, ref, params, L):
    flat, off = g.g_tower.cpu().numpy(), 0
    for k in _tower_keys(L):
        n = params[k].size
        if k in ref:
            assert_close(flat[off:off + n].reshape(ref[k].shape), ref[k], f"grad {k}")
        else:   # GMF: the tower takes no gradient
            assert not flat[off:off + n].any(), f"grad {k} of a GMF model"
        off += n
    assert off == flat.size


# (model_type, f, L, B, tile path): 4 = thread per sample (f = 8), 2 = mma.sync with 32-row tiles (B = 300) and
# 64-row tiles (B = 6000, more 64-row tiles than the 148 SMs take twice), 1 = generic FMA, 3 = tcgen05
NORM_CASES = [("NeuMF-end", 8, 3, 700, 4), ("NeuMF-end", 16, 2, 300, 2), ("NeuMF-end", 16, 2, 6000, 2),
              ("NeuMF-end", 6, 2, 500, 1), ("GMF", 8, 1, 500, 1), ("NeuMF-end", 32, 3, 1500, 3),
              ("NeuMF-end", 64, 3, 1500, 3)]


@gpu
@pytest.mark.parametrize("teacher", [False, True], ids=["bce", "kd"])
@pytest.mark.parametrize("norm", ["B", "3B+7"])
@pytest.mark.parametrize("model_type,f,L,B,path", NORM_CASES)
def test_step_norm_matches_oracle(monkeypatch, model_type, f, L, B, path, norm, teacher):
    """ncf_train_step_grads_norm: logits, loss and every gradient buffer == the oracle with the loss mean over
    B_norm (the oracle's loss and dlogit scaled by B / B_norm)."""
    from ncf_b200 import ops
    if path == 3:
        monkeypatch.setenv("NCF_UMMA_MIN_B", "1")
    U, I = 700, 500
    rng = np.random.default_rng(f * 100 + L + B)
    model, params = _model(model_type, f, L, U, I, seed=f + B)
    u, i = _batch(params, model_type, L, U, I, B, rng)
    y = (rng.random(B) < 0.3).astype(np.float32)
    t = rng.standard_normal(B).astype(np.float32) if teacher else None
    alpha = 0.4 if teacher else 1.0
    B_norm = B if norm == "B" else 3 * B + 7
    g = ops.GradBuffers.allocate(model.abi_type(), f, L, U, I, B, _dev())
    loss, logits = _step_norm(model.abi_struct(), g, _cuda(u), _cuda(i), _cuda(y),
                              _cuda(t) if teacher else None, alpha, B_norm)
    assert _lib().ncf_last_tile_path() == path
    ref_logits = onp.forward(params, u, i, model_type)
    ref_loss, dl = _loss_ref(ref_logits, y, t, alpha, B_norm)
    assert_close(logits, ref_logits, "logits")
    assert abs(loss - ref_loss) <= 5e-6 * abs(ref_loss), (loss, ref_loss)
    ref = onp.backward(params, u, i, model_type, dl)
    for key, buf in (("embed_user_GMF.weight", g.g_user_gmf), ("embed_item_GMF.weight", g.g_item_gmf),
                     ("embed_user_MLP.weight", g.g_user_mlp), ("embed_item_MLP.weight", g.g_item_mlp)):
        if key in ref:
            assert_close(buf.cpu().numpy(), ref[key], f"grad {key}")
    _check_tower(g, ref, params, L)


@gpu
@pytest.mark.parametrize("norm", ["B", "3B+7"])
@pytest.mark.parametrize("model_type,f,L,B,path", [("NeuMF-end", 8, 3, 700, 4), ("NeuMF-end", 16, 2, 6000, 2),
                                                   ("NeuMF-end", 64, 3, 1500, 3)])
def test_row_sharded_call_form_gives_per_sample_item_gradients(monkeypatch, model_type, f, L, B, path, norm):
    """The call of RowShardedTrainer (both transports): item tables = the [b, f] / [b, d] receive buffers with
    item_num = b, item ids = positions 0..b-1, g_item_* = per-sample buffers.  Every sample's item gradient
    must be the oracle's per-sample gradient (no two samples share a row)."""
    from ncf_b200 import ops
    if path == 3:
        monkeypatch.setenv("NCF_UMMA_MIN_B", "1")
    U, I = 700, 500
    rng = np.random.default_rng(B + f)
    model, params = _model(model_type, f, L, U, I, seed=B)
    u, i = _batch(params, model_type, L, U, I, B, rng)
    y = (rng.random(B) < 0.3).astype(np.float32)
    B_norm = B if norm == "B" else 3 * B + 7
    recv = dict(params)
    recv["embed_item_GMF.weight"] = params["embed_item_GMF.weight"][i]
    recv["embed_item_MLP.weight"] = params["embed_item_MLP.weight"][i]
    pos = np.arange(B, dtype=np.int64)
    rows_gmf, rows_mlp = _cuda(recv["embed_item_GMF.weight"]), _cuda(recv["embed_item_MLP.weight"])
    m = ops.model_struct(model.abi_type(), f, L, U, B,
                         (model.embed_user_GMF.weight.detach(), rows_gmf, model.embed_user_MLP.weight.detach(), rows_mlp),
                         [(l.weight.detach(), l.bias.detach()) for l in model.linears()],
                         (model.predict_layer.weight.detach(), model.predict_layer.bias.detach()))
    g = ops.GradBuffers.allocate(model.abi_type(), f, L, U, B, B, _dev())   # g_item_* = [B, f] / [B, d]
    loss, logits = _step_norm(m, g, _cuda(u), _cuda(pos), _cuda(y), None, 1.0, B_norm)
    assert _lib().ncf_last_tile_path() == path
    ref_logits = onp.forward(recv, u, pos, model_type)
    ref_loss, dl = _loss_ref(ref_logits, y, None, 1.0, B_norm)
    assert_close(logits, ref_logits, "logits")
    assert abs(loss - ref_loss) <= 5e-6 * abs(ref_loss)
    ref = onp.backward(recv, u, pos, model_type, dl)
    assert_close(g.g_item_gmf.cpu().numpy(), ref["embed_item_GMF.weight"], "per-sample item GMF gradient")
    assert_close(g.g_item_mlp.cpu().numpy(), ref["embed_item_MLP.weight"], "per-sample item MLP gradient")
    assert_close(g.g_user_gmf.cpu().numpy(), ref["embed_user_GMF.weight"], "user GMF gradient")
    assert_close(g.g_user_mlp.cpu().numpy(), ref["embed_user_MLP.weight"], "user MLP gradient")
    _check_tower(g, ref, params, L)


@gpu
def test_step_norm_below_the_batch_is_refused():
    from ncf_b200 import ops
    U, I, f, L, B = 50, 40, 8, 2, 32
    model, _ = _model("NeuMF-end", f, L, U, I, seed=0)
    g = ops.GradBuffers.allocate(model.abi_type(), f, L, U, I, B, _dev())
    m = model.abi_struct()
    u = torch.zeros(B, dtype=torch.int64, device=_dev())
    y = torch.zeros(B, device=_dev())
    ws = torch.empty(ops.train_workspace_bytes(m, B), dtype=torch.uint8, device=_dev())
    loss = torch.zeros(1, dtype=torch.float64, device=_dev())
    rc = _lib().ncf_train_step_grads_norm(ctypes.byref(m), ctypes.byref(g.struct()), u.data_ptr(), u.data_ptr(),
                                          y.data_ptr(), None, 1.0, B, B - 1, loss.data_ptr(), None, ws.data_ptr(),
                                          ws.numel(), _stream())
    assert rc == ERR_ARG
    torch.cuda.synchronize()
    assert float(loss.item()) == 0.0 and not g.g_tower.any()


# ---- 2. optimiser kernels against float64 Adam -------------------------------------------------------------------
def _adam_inputs(n, rng):
    p = (rng.standard_normal(n) * 0.1).astype(np.float32)
    m = (rng.standard_normal(n) * 1e-3).astype(np.float32)
    v = ((rng.standard_normal(n) * 1e-3) ** 2).astype(np.float32)
    g = (rng.standard_normal(n) * 1e-3).astype(np.float32)
    k = rng.integers(0, 5, n)           # exact zeros, +-1e-9, +-1e3 among ordinary gradients
    g[k == 1] = 0.0
    g[k == 2] = np.float32(1e-9) * np.sign(rng.standard_normal(int((k == 2).sum())))
    g[k == 3] = np.float32(1e3) * np.sign(rng.standard_normal(int((k == 3).sum())))
    return p, m, v, g


@gpu
@pytest.mark.parametrize("step", STEPS)
@pytest.mark.parametrize("n", [0, 4, 4 * 300007])
def test_adam_range_matches_float64_adam(n, step):
    rng = np.random.default_rng(n + step)
    pad = 8    # the call sees [0, n) of buffers of n + pad: the tail must not move
    host = _adam_inputs(n + pad, rng)
    p, m, v, g = (_cuda(a) for a in host)
    st = torch.tensor([step], dtype=torch.int64, device=_dev())
    rc = _lib().ncf_adam_range(p.data_ptr(), m.data_ptr(), v.data_ptr(), g.data_ptr(), n, st.data_ptr(),
                               _lib_hyper(), _stream())
    assert rc == 0
    torch.cuda.synchronize()
    assert int(st.item()) == step
    assert not g[:n].any()
    for name, a, h in (("p", p, host[0]), ("m", m, host[1]), ("v", v, host[2]), ("g", g, host[3])):
        _same(a[n:], h[n:], f"{name} beyond n")
    if n:
        pr, mr, vr = adam_ref(*(h[:n] for h in host), step + 1)
        assert_adam(p[:n].cpu().numpy(), pr, host[0][:n], m[:n].cpu().numpy(), mr, v[:n].cpu().numpy(), vr, "adam_range")


def _p2p_slices(n, W):
    per = -(-n // (4 * W)) * 4          # ncf_b200/dist.py: per = ceil(n / 4W) * 4
    return [(min(r * per, n), min((r + 1) * per, n)) for r in range(W)]


@gpu
@pytest.mark.parametrize("scale", ["1/W", "1"])
@pytest.mark.parametrize("W", [1, 2, 3, 5, 8])
def test_adam_p2p_matches_float64_adam_on_the_rank_sum(W, scale):
    """Every emulated rank updates its slice from every rank's gradients and stores the new parameters into
    every rank's buffer.  The gradient is the kernel's fp32 sum in rank order times grad_scale, which numpy
    reproduces bit for bit; the update is then held to float64 Adam on it."""
    from ncf_b200 import ops
    n = 4 * 1001 + 4 * W                 # the last slice is shorter than the others
    slices = _p2p_slices(n, W)
    assert len({b - a for a, b in slices}) > 1 or W == 1
    gs = np.float32(1.0 / W) if scale == "1/W" else np.float32(1.0)
    for step in STEPS:
        rng = np.random.default_rng(W * 10 + step)
        p0, _, _, _ = _adam_inputs(n, rng)
        grads = [_adam_inputs(n, rng)[3] for _ in range(W)]
        mv = [(_adam_inputs(b - a, rng)[1], _adam_inputs(b - a, rng)[2]) for a, b in slices]
        P = [_cuda(p0) for _ in range(W)]
        G = [_cuda(x) for x in grads]
        M = [_cuda(a) for a, _ in mv]
        V = [_cuda(b) for _, b in mv]
        st = torch.tensor([step], dtype=torch.int64, device=_dev())
        gp, pp = [t.data_ptr() for t in G], [t.data_ptr() for t in P]
        for r, (a, b) in enumerate(slices):
            before = [t.cpu().numpy() for t in P]
            ops.adam_p2p(gp, pp, M[r], V[r], a, r, st, *HYPER, grad_scale=float(gs))
            torch.cuda.synchronize()
            for q in range(W):   # outside slice r nothing moved, in any rank's buffer
                now = P[q].cpu().numpy()
                _same(np.concatenate([now[:a], now[b:]]), np.concatenate([before[q][:a], before[q][b:]]),
                      f"step {step}: rank {r}'s call wrote outside its slice of rank {q}'s parameters")
        got = [t.cpu().numpy() for t in P]
        for q in range(1, W):
            _same(got[q], got[0], f"step {step}: parameters of rank {q} differ from rank 0")
        gsum = grads[0].copy()
        for x in grads[1:]:
            gsum = (gsum + x).astype(np.float32)
        gsum = (gsum * gs).astype(np.float32)
        for r, (a, b) in enumerate(slices):
            pr, mr, vr = adam_ref(p0[a:b], mv[r][0], mv[r][1], gsum[a:b], step + 1)
            assert_adam(got[0][a:b], pr, p0[a:b], M[r].cpu().numpy(), mr, V[r].cpu().numpy(), vr,
                        f"W={W} step {step} slice {r}")
        for q in range(W):
            _same(G[q], grads[q], "gradients are read only")
        assert int(st.item()) == step


@gpu
def test_adam_p2p_with_an_empty_slice_changes_nothing():
    W, n = 3, 64
    P = [torch.randn(n, device=_dev()) for _ in range(W)]
    G = [torch.randn(n, device=_dev()) for _ in range(W)]
    m, v = torch.randn(n, device=_dev()), torch.rand(n, device=_dev())
    st = torch.zeros(1, dtype=torch.int64, device=_dev())
    before = [t.clone() for t in P + G + [m, v]]
    rc = _lib().ncf_adam_p2p(_ptrs([t.data_ptr() for t in G]), _ptrs([t.data_ptr() for t in P]), m.data_ptr(),
                             v.data_ptr(), 16, 0, W, 1, 1.0 / W, st.data_ptr(),
                             _lib_hyper(), _stream())
    assert rc == 0
    torch.cuda.synchronize()
    for a, b in zip(P + G + [m, v], before):
        _same(a, b, "an empty slice must not write")


def _lib_hyper():
    from ncf_b200._lib import NcfAdamHyper
    return NcfAdamHyper(*HYPER)


def _flat_model(model_type, f, L, U, I, seed):
    """Tables, tower and the optimiser state of one model as torch tensors + the ABI structs."""
    from ncf_b200 import ops
    gen = torch.Generator().manual_seed(seed)
    d = f << (L - 1)
    rnd = lambda *s, sc=0.1: (torch.randn(*s, generator=gen) * sc).to(_dev())
    tables = (rnd(U, f), rnd(I, f), rnd(U, d), rnd(I, d))
    widths = ops.tower_widths(f, L)
    lin = [(rnd(widths[k + 1], widths[k]), rnd(widths[k + 1])) for k in range(L)]
    pred_w = rnd(1, f + widths[-1] if model_type == "NeuMF-end" else (f if model_type == "GMF" else widths[-1]))
    pred = (pred_w, rnd(1))
    mt = {"GMF": 0, "MLP": 1, "NeuMF-end": 2}[model_type]
    m = ops.model_struct(mt, f, L, U, I, tables, lin, pred)
    return mt, tables, lin, pred, m


def _tower_params(lin, pred):
    return [x.reshape(-1) for x in [x for wb in lin for x in wb] + list(pred)]


@gpu
@pytest.mark.parametrize("f", [8, 16])
@pytest.mark.parametrize("parts", [0, 1, 2, 4, 5, 6, 7])
@pytest.mark.parametrize("rng_kind", ["all", "inner", "empty"])
def test_adam_step_dense_range_matches_lazy_reference(f, parts, rng_kind):
    _dense_range_case("NeuMF-end", f, 2, parts, rng_kind)


@gpu
@pytest.mark.parametrize("rng_kind", ["all", "inner"])
def test_adam_step_dense_range_scalar_rows(rng_kind):
    """f = 6: rows are not float4-wide, the per-row kernel runs; only parts = 7 is accepted there."""
    _dense_range_case("NeuMF-end", 6, 2, 7, rng_kind)
    from ncf_b200 import ops
    mt, tables, lin, pred, m = _flat_model("NeuMF-end", 6, 2, 40, 30, 1)
    g = ops.GradBuffers.allocate(mt, 6, 2, 40, 30, 40, _dev())
    s = ops.AdamBuffers.allocate(mt, 6, 2, 40, 30, _dev())
    for parts in (1, 2, 3, 4, 5, 6):
        rc = _lib().ncf_adam_step_dense_range(ctypes.byref(m), ctypes.byref(g.struct()), ctypes.byref(s.struct()),
                                              _lib_hyper(), 0, 40, parts, _stream())
        assert rc == ERR_ARG
    torch.cuda.synchronize()
    assert int(s.step.item()) == 0


def _dense_range_case(model_type, f, L, parts, rng_kind):
    from ncf_b200 import ops
    U, I, t_now = 300, 200, 400
    lo, hi = {"all": (0, U), "inner": (17, U - 5), "empty": (123, 123)}[rng_kind]
    mt, tables, lin, pred, m = _flat_model(model_type, f, L, U, I, seed=f * 10 + parts)
    g = ops.GradBuffers.allocate(mt, f, L, U, I, U, _dev())
    s = ops.AdamBuffers.allocate(mt, f, L, U, I, _dev())
    gen = torch.Generator().manual_seed(parts * 7 + f)
    names = ("user_gmf", "item_gmf", "user_mlp", "item_mlp")
    for name, tab in zip(names, tables):
        for pre in ("m_", "v_"):
            x = torch.randn(tab.shape, generator=gen) * 1e-3
            getattr(s, pre + name).copy_(x * x if pre == "v_" else x)
        grad = torch.randn(tab.shape, generator=gen) * 1e-3
        grad[torch.rand(tab.shape[0], generator=gen) < 0.6] = 0.0     # gradients in some rows only
        getattr(g, "g_" + name).copy_(grad)
    for buf in (s.m_tower, s.v_tower, g.g_tower):
        x = torch.randn(buf.shape, generator=gen) * 1e-3
        buf.copy_(x * x if buf is s.v_tower else x)
    for name, n in (("user_last_step", U), ("item_last_step", I)):
        last = torch.randint(1, t_now + 1, (n,), generator=gen, dtype=torch.int32)
        last[torch.rand(n, generator=gen) < 0.1] = 0             # never stepped
        last[torch.rand(n, generator=gen) < 0.1] = t_now         # current already
        last[:8] = torch.tensor([1, 2, t_now - 161, t_now - 160, t_now - 159, t_now - 1, t_now, 0], dtype=torch.int32)
        getattr(s, name).copy_(last)
    g.user_flag.copy_(torch.randint(0, 2, (U,), generator=gen, dtype=torch.int32))
    g.item_flag.copy_(torch.randint(0, 2, (I,), generator=gen, dtype=torch.int32))
    g.touched_count.copy_(torch.tensor([5, 9], dtype=torch.int32))
    s.step.fill_(t_now)
    tower = _tower_params(lin, pred)

    snap = lambda: {k: v.cpu().numpy().copy() for k, v in _state_tensors(g, s, tables, tower).items()}
    before = snap()
    ops.adam_step_dense_range(m, g.struct(), s.struct(), lo, hi, *HYPER, parts=parts)
    torch.cuda.synchronize()
    after = snap()
    t = t_now + 1

    assert int(s.step.item()) == t and g.touched_count.tolist() == [0, 0]
    # stamps: user rows in [lo, hi) and every item row, whatever parts is; user rows outside keep theirs
    want_last_u = before["user_last_step"].copy()
    want_last_u[lo:hi] = t
    want_flag_u = before["user_flag"].copy()
    want_flag_u[lo:hi] = 0
    _same(after["user_last_step"], want_last_u, "user last_step")
    _same(after["user_flag"], want_flag_u, "user flags")
    assert (after["item_last_step"] == t).all() and (after["item_flag"] == 0).all()

    for side, rows in ((0, slice(lo, hi)), (1, slice(0, I))):
        upd = bool(parts & (1 if side == 0 else 2))
        last = before["user_last_step" if side == 0 else "item_last_step"][rows]
        for kind in ("gmf", "mlp"):
            name = ("user_" if side == 0 else "item_") + kind
            keys = ("p_" + name, "m_" + name, "v_" + name, "g_" + name)
            if side == 0:   # user rows outside the range are never touched
                for k in keys:
                    _same(np.concatenate([after[k][:lo], after[k][hi:]]),
                          np.concatenate([before[k][:lo], before[k][hi:]]), f"{k} outside [lo, hi)")
            if not upd:
                for k in keys:
                    _same(after[k], before[k], f"{k}: part {parts} does not include it")
                continue
            p0, m0, v0, g0 = (before[k][rows] for k in keys)
            pr, mr, vr, gap = lazy_ref(p0, m0, v0, g0, last, t)
            assert_adam(after[keys[0]][rows], pr, p0, after[keys[1]][rows], mr, after[keys[2]][rows], vr,
                        f"{name} parts={parts}", chained=gap)
            assert not after[keys[3]][rows].any(), f"{keys[3]} not zeroed"
    k_t = ("p_tower", "m_tower", "v_tower", "g_tower")
    if parts & 4:
        pr, mr, vr = adam_ref(before["p_tower"], before["m_tower"], before["v_tower"], before["g_tower"], t)
        assert_adam(after["p_tower"], pr, before["p_tower"], after["m_tower"], mr, after["v_tower"], vr, "tower")
        assert not after["g_tower"].any()
    else:
        for k in k_t:
            _same(after[k], before[k], f"{k}: part {parts} does not include it")


def _state_tensors(g, s, tables, tower):
    out = {}
    for name, tab in zip(("user_gmf", "item_gmf", "user_mlp", "item_mlp"), tables):
        out["p_" + name] = tab
        out["m_" + name], out["v_" + name] = getattr(s, "m_" + name), getattr(s, "v_" + name)
        out["g_" + name] = getattr(g, "g_" + name)
    out["p_tower"] = torch.cat(tower)
    out["m_tower"], out["v_tower"], out["g_tower"] = s.m_tower, s.v_tower, g.g_tower
    out["user_last_step"], out["item_last_step"] = s.user_last_step, s.item_last_step
    out["user_flag"], out["item_flag"] = g.user_flag, g.item_flag
    out["user_list"], out["item_list"] = g.user_list, g.item_list
    return out


@gpu
def test_adam_finish_dense_stamps_and_closes_the_step_only():
    from ncf_b200 import ops
    U, I, f, L = 130, 70, 8, 2
    mt, tables, lin, pred, m = _flat_model("NeuMF-end", f, L, U, I, seed=3)
    g = ops.GradBuffers.allocate(mt, f, L, U, I, U, _dev())
    s = ops.AdamBuffers.allocate(mt, f, L, U, I, _dev())
    gen = torch.Generator().manual_seed(4)
    for name in ("m_user_gmf", "v_item_gmf", "m_item_mlp", "v_user_mlp", "m_tower"):
        getattr(s, name).copy_(torch.rand(getattr(s, name).shape, generator=gen))
    g.g_item_gmf.copy_(torch.randn(I, f, generator=gen))
    s.user_last_step.copy_(torch.randint(0, 50, (U,), generator=gen, dtype=torch.int32))
    s.item_last_step.copy_(torch.randint(0, 50, (I,), generator=gen, dtype=torch.int32))
    g.user_flag.copy_(torch.randint(0, 2, (U,), generator=gen, dtype=torch.int32))
    g.item_flag.copy_(torch.randint(0, 2, (I,), generator=gen, dtype=torch.int32))
    g.touched_count.copy_(torch.tensor([3, 4], dtype=torch.int32))
    s.step.fill_(49)
    tower = _tower_params(lin, pred)
    before = {k: v.cpu().numpy().copy() for k, v in _state_tensors(g, s, tables, tower).items()}
    ops.adam_finish_dense(m, g.struct(), s.struct())
    torch.cuda.synchronize()
    after = {k: v.cpu().numpy().copy() for k, v in _state_tensors(g, s, tables, tower).items()}
    assert int(s.step.item()) == 50 and g.touched_count.tolist() == [0, 0]
    assert (after["user_last_step"] == 50).all() and (after["item_last_step"] == 50).all()
    assert not after["user_flag"].any() and not after["item_flag"].any()
    for k in before:
        if k not in ("user_last_step", "item_last_step", "user_flag", "item_flag"):
            _same(after[k], before[k], k)


@gpu
@pytest.mark.parametrize("side", [0, 1])
def test_mark_rows_side_appends_distinct_rows(side):
    from ncf_b200 import ops
    U, I, f, L = 300, 200, 8, 2
    mt, tables, lin, pred, m = _flat_model("NeuMF-end", f, L, U, I, seed=5)
    g = ops.GradBuffers.allocate(mt, f, L, U, I, max(U, I), _dev())
    limit = U if side == 0 else I
    rng = np.random.default_rng(side)
    first = rng.integers(0, limit, 40)
    second = np.concatenate([rng.integers(0, limit, 500), first[:10], [-1, limit, -1, limit, 0, limit - 1]])
    ops.mark_rows_side(m, g.struct(), _cuda(first), side)
    torch.cuda.synchronize()
    lst = g.user_list if side == 0 else g.item_list
    flag = g.user_flag if side == 0 else g.item_flag
    n1 = int(g.touched_count[side].item())
    head = lst[:n1].cpu().numpy().copy()
    assert n1 == len(set(first.tolist())) and set(head.tolist()) == set(first.tolist())
    ops.mark_rows_side(m, g.struct(), _cuda(second), side)
    torch.cuda.synchronize()
    n2 = int(g.touched_count[side].item())
    want = set(first.tolist()) | {x for x in second.tolist() if 0 <= x < limit}
    got = lst[:n2].cpu().numpy()
    assert n2 == len(want) and len(set(got.tolist())) == n2 and set(got.tolist()) == want
    _same(got[:n1], head, "the rows already listed stay in place")
    fl = np.zeros(limit, np.int32)
    fl[list(want)] = 1
    _same(flag, fl, "flags")
    other = 1 - side
    assert int(g.touched_count[other].item()) == 0
    assert not (g.item_flag if side == 0 else g.user_flag).any()


# ---- 3. row exchange, NCCL transport ------------------------------------------------------------------------
def _items(kind, n, world, rng):
    if kind == "uniform":
        return rng.integers(0, 10_000, n)
    if kind == "one_owner":
        return rng.integers(0, 10_000, n) * world + (world - 1)
    if kind == "big":
        return rng.integers(0, 2 ** 40, n)
    it = rng.integers(0, 10_000, n)            # "negative": ids a sampler without a legal negative writes
    neg = rng.random(n) < 0.2
    it[neg] = -1
    it[neg & (rng.random(n) < 0.3)] = -(2 ** 35) - 3
    return it


@gpu
@pytest.mark.parametrize("kind", ["uniform", "one_owner", "big", "negative"])
@pytest.mark.parametrize("n", [0, 1, 100_003])
@pytest.mark.parametrize("W", [1, 2, 3, 7, 8, 64])
def test_bucket_by_owner_groups_by_owner(W, n, kind):
    from ncf_b200 import ops
    rng = np.random.default_rng(W * 7 + n)
    item = _items(kind, n, W, rng).astype(np.int64)
    perm, local, counts = ops.bucket_by_owner(_cuda(item), W)
    torch.cuda.synchronize()
    perm, local, counts = perm.cpu().numpy(), local.cpu().numpy(), counts.cpu().numpy()
    owner, local_ref = bucket_ref(item, W)
    assert np.array_equal(counts, np.bincount(owner, minlength=W)) and counts.sum() == n
    assert np.array_equal(np.sort(perm), np.arange(n))
    edges = np.concatenate([[0], np.cumsum(counts)])
    for w in range(W):   # group w holds exactly the samples owned by w (order inside a group is free)
        grp = perm[edges[w]:edges[w + 1]]
        assert (owner[grp] == w).all()
    assert np.array_equal(local, local_ref[perm])


@gpu
def test_bucket_by_owner_refuses_more_than_64_ranks():
    item = torch.zeros(4, dtype=torch.int64, device=_dev())
    scratch = torch.zeros(80, dtype=torch.int64, device=_dev())
    c = torch.zeros(80, dtype=torch.int32, device=_dev())
    rc = _lib().ncf_bucket_by_owner(item.data_ptr(), 4, 65, scratch.data_ptr(), scratch.data_ptr(), c.data_ptr(),
                                    c.data_ptr(), _stream())
    assert rc == ERR_ARG


@gpu
@pytest.mark.parametrize("n", [0, 1, 100_003])
def test_permute_is_a_gather(n):
    from ncf_b200 import ops
    rng = np.random.default_rng(n)
    perm = np.concatenate([rng.permutation(n)[: n // 2], rng.integers(0, max(n, 1), n - n // 2)]).astype(np.int64)
    a = rng.integers(-2 ** 62, 2 ** 62, n).astype(np.int64)
    b = rng.standard_normal(n).astype(np.float32)
    ga, gb = ops.permute(_cuda(a), _cuda(perm)), ops.permute(_cuda(b), _cuda(perm))
    torch.cuda.synchronize()
    _same(ga, a[perm], "permute_i64")
    _same(gb, b[perm], "permute_f32")


DIMS = [1, 3, 4, 8, 33, 132, 256]   # scalar path, float4 path, lanes that loop more than once


def _row_ids(rows, n, rng):
    idx = rng.integers(0, rows, n)
    idx[rng.random(n) < 0.3] = 7        # duplicates
    bad = rng.choice(n, 12, replace=False)
    idx[bad[:6]] = -1
    idx[bad[6:]] = rows
    return idx.astype(np.int64)


@gpu
@pytest.mark.parametrize("dim", DIMS)
def test_gather_rows_is_exact_and_zero_fills_invalid_ids(dim):
    from ncf_b200 import ops
    rng = np.random.default_rng(dim)
    rows, n = 700, 3001
    table = rng.standard_normal((rows, dim)).astype(np.float32)
    idx = _row_ids(rows, n, rng)
    out = ops.gather_rows(_cuda(table), _cuda(idx))
    torch.cuda.synchronize()
    ok = (idx >= 0) & (idx < rows)
    want = np.zeros((n, dim), np.float32)
    want[ok] = table[idx[ok]]
    _same(out, want, "gathered rows")


@gpu
@pytest.mark.parametrize("dim", DIMS)
def test_scatter_add_rows_matches_float64_sum(dim):
    from ncf_b200 import ops
    rng = np.random.default_rng(100 + dim)
    rows = 700
    idx = np.concatenate([_row_ids(rows, 3001, rng), np.full(10_000, 11)])   # row 11 takes 10 000 adds
    rng.shuffle(idx)
    table = rng.standard_normal((rows, dim)).astype(np.float32)
    vals = rng.standard_normal((idx.size, dim)).astype(np.float32)
    t = _cuda(table)
    ops.scatter_add_rows(t, _cuda(idx), _cuda(vals))
    torch.cuda.synchronize()
    got = t.cpu().numpy()
    ok = (idx >= 0) & (idx < rows)
    ref = table.astype(np.float64)
    np.add.at(ref, idx[ok], vals[ok].astype(np.float64))
    absum = np.abs(table).astype(np.float64)
    np.add.at(absum, idx[ok], np.abs(vals[ok]).astype(np.float64))
    k = 1 + np.bincount(idx[ok], minlength=rows)[:, None]
    assert (np.abs(got - ref) <= sum_bound(k, absum)).all()
    named = np.zeros(rows, bool)
    named[idx[ok]] = True
    _same(got[~named], table[~named], "rows no id names")


# ---- 4. row exchange, peer-memory transport (ncf_shard_*) ---------------------------------------------------------
CAP = 4096
SIZES = {1: [CAP], 2: [CAP, 517], 3: [1234, 0, CAP], 8: [CAP, 0, 1234, 77, 4000, 3, 2048, 999]}
SENTINEL = np.int32(0x7FC0DEAD)   # a NaN pattern: receive slots that nobody pushes into keep it


def _shard_rows(n, W, r):
    return (n - r + W - 1) // W


def _rank_items(W, item_num, sizes, rng):
    out = []
    for r, n in enumerate(sizes):
        it = rng.integers(0, item_num, n)
        k = rng.random(n)
        it[k < 0.15] = 13                                     # one hot item
        own = k > 0.85                                        # items this requester owns itself
        it[own] = (rng.integers(0, item_num // W, int(own.sum())) * W + r) % item_num
        if n > 4:
            it[1], it[n - 2], it[n // 2] = -1, item_num, -1    # dropped: no request, no row, no gradient
        out.append(it.astype(np.int64))
    return out


SHARD_MODELS = [("NeuMF-end", 8, 1), ("NeuMF-end", 8, 3), ("NeuMF-end", 32, 1), ("NeuMF-end", 32, 3),
                ("GMF", 8, 1), ("MLP", 32, 3)]


@gpu
@pytest.mark.parametrize("model_type,f,L", SHARD_MODELS)
@pytest.mark.parametrize("W", [1, 2, 3, 8])
def test_peer_exchange_phase_by_phase(W, model_type, f, L):
    from ncf_b200 import ops
    d = f << (L - 1)
    gmf, mlp = model_type != "MLP", model_type != "GMF"
    item_num, U = 3001, 50
    rng = np.random.default_rng(W * 100 + f + L)
    sizes = SIZES[W]
    items = _rank_items(W, item_num, sizes, rng)
    glob_gmf = rng.standard_normal((item_num, f)).astype(np.float32)
    glob_mlp = rng.standard_normal((item_num, d)).astype(np.float32)
    shards, inbox, count, cursor = [], [], [], []
    for o in range(W):
        rows = _shard_rows(item_num, W, o)
        mt, tables, lin, pred, _ = _flat_model(model_type, f, L, U, rows, seed=o)
        tables[1].copy_(_cuda(glob_gmf[o::W]))
        tables[3].copy_(_cuda(glob_mlp[o::W]))
        m = ops.model_struct(mt, f, L, U, rows, tables, lin, pred)
        if not gmf:
            m.embed_user_gmf = m.embed_item_gmf = None
        if not mlp:
            m.embed_user_mlp = m.embed_item_mlp = None
        g = ops.GradBuffers.allocate(mt, f, L, U, rows, rows, _dev())
        shards.append((m, g, tables))
        inbox.append(torch.full((W * CAP,), -5, dtype=torch.int64, device=_dev()))
        count.append(torch.full((W,), -5, dtype=torch.int32, device=_dev()))
        cursor.append(torch.zeros(W, dtype=torch.int32, device=_dev()))
    ib, ic = [t.data_ptr() for t in inbox], [t.data_ptr() for t in count]
    it_d = [_cuda(x) for x in items]

    # request
    for r in range(W):
        ops.shard_request(it_d[r], W, r, CAP, item_num, ib, ic, cursor[r])
    torch.cuda.synchronize()
    ref = inbox_ref(items, W, item_num)
    for o in range(W):
        cnt = count[o].cpu().numpy()
        box = inbox[o].cpu().numpy()
        for r in range(W):
            assert cnt[r] == len(ref[o][r]), (o, r)
            assert sorted(box[r * CAP: r * CAP + cnt[r]].tolist()) == ref[o][r], (o, r)

    # mark
    for o, (m, g, _) in enumerate(shards):
        ops.shard_mark_requests(m, g.struct(), inbox[o], count[o], W, CAP)
    torch.cuda.synchronize()
    for o, (m, g, _) in enumerate(shards):
        want = {e >> 32 for r in range(W) for e in ref[o][r]}
        n = int(g.touched_count[1].item())
        got = g.item_list[:n].cpu().numpy().tolist()
        assert n == len(want) and set(got) == want and len(set(got)) == n
        fl = np.zeros(m.item_num, np.int32)
        fl[list(want)] = 1
        _same(g.item_flag, fl, "item flags")
        assert int(g.touched_count[0].item()) == 0

    # push rows
    recv_gmf = [torch.full((CAP * f,), int(SENTINEL), dtype=torch.int32, device=_dev()).view(torch.float32)
                for _ in range(W)]
    recv_mlp = [torch.full((CAP * d,), int(SENTINEL), dtype=torch.int32, device=_dev()).view(torch.float32)
                for _ in range(W)]
    for o, (m, _, _) in enumerate(shards):
        ops.shard_push_rows(m, inbox[o], count[o], W, CAP, [t.data_ptr() for t in recv_gmf] if gmf else None,
                            [t.data_ptr() for t in recv_mlp] if mlp else None)
    torch.cuda.synchronize()
    for r, it in enumerate(items):
        ok = (it >= 0) & (it < item_num)
        for on, glob, recv, w in ((gmf, glob_gmf, recv_gmf, f), (mlp, glob_mlp, recv_mlp, d)):
            got = _bits(recv[r]).reshape(CAP, w)
            want = np.full((CAP, w), SENTINEL, np.int32)
            if on:
                want[np.nonzero(ok)[0]] = glob[it[ok]].view(np.int32)
            assert np.array_equal(got, want), f"receive slots of rank {r}"

    # push grads
    gbuf_gmf, gbuf_mlp = [], []
    for o, (m, g, _) in enumerate(shards):
        if gmf:
            g.g_item_gmf.copy_(torch.randn(g.g_item_gmf.shape, generator=torch.Generator().manual_seed(o)))
        if mlp:
            g.g_item_mlp.copy_(torch.randn(g.g_item_mlp.shape, generator=torch.Generator().manual_seed(50 + o)))
        gbuf_gmf.append(g.g_item_gmf.cpu().numpy().copy() if gmf else None)
        gbuf_mlp.append(g.g_item_mlp.cpu().numpy().copy() if mlp else None)
    per_gmf = [rng.standard_normal((n, f)).astype(np.float32) for n in sizes]
    per_mlp = [rng.standard_normal((n, d)).astype(np.float32) for n in sizes]
    for r in range(W):
        ops.shard_push_grads(it_d[r], W, item_num, _cuda(per_gmf[r]) if gmf else None,
                             _cuda(per_mlp[r]) if mlp else None, f, d,
                             [sh[1].g_item_gmf.data_ptr() for sh in shards] if gmf else None,
                             [sh[1].g_item_mlp.data_ptr() for sh in shards] if mlp else None)
    torch.cuda.synchronize()
    all_items = np.concatenate(items)
    ok = (all_items >= 0) & (all_items < item_num)
    for on, per, before, attr, w in ((gmf, per_gmf, gbuf_gmf, "g_item_gmf", f), (mlp, per_mlp, gbuf_mlp, "g_item_mlp", d)):
        if not on:
            continue
        vals = np.concatenate(per)[ok].astype(np.float64)
        glob_ref = np.zeros((item_num, w))
        glob_abs = np.zeros((item_num, w))
        glob_before = np.zeros((item_num, w), np.float32)
        for o in range(W):
            glob_ref[o::W] = before[o]
            glob_before[o::W] = before[o]
        glob_abs[:] = np.abs(glob_ref)
        np.add.at(glob_ref, all_items[ok], vals)
        np.add.at(glob_abs, all_items[ok], np.abs(vals))
        k = 1 + np.bincount(all_items[ok], minlength=item_num)[:, None]
        for o, (_, g, _) in enumerate(shards):
            got = getattr(g, attr).cpu().numpy()
            assert (np.abs(got - glob_ref[o::W]) <= sum_bound(k[o::W], glob_abs[o::W])).all(), f"{attr} of rank {o}"
            untouched = k[o::W, 0] == 1
            _same(got[untouched], glob_before[o::W][untouched], f"{attr} rows nobody pushed to")


@gpu
def test_peer_exchange_refuses_bad_arguments_before_any_launch():
    from ncf_b200 import ops
    lib, W, cap = _lib(), 2, 64
    item = torch.zeros(cap + 1, dtype=torch.int64, device=_dev())
    inbox = [torch.zeros(W * cap, dtype=torch.int64, device=_dev()) for _ in range(W)]
    count = [torch.zeros(8, dtype=torch.int32, device=_dev()) for _ in range(W)]
    cursor = torch.zeros(8, dtype=torch.int32, device=_dev())
    ib, ic = _ptrs([t.data_ptr() for t in inbox]), _ptrs([t.data_ptr() for t in count])
    off = _ptrs([inbox[0].data_ptr(), inbox[1].data_ptr() + 4])
    s = _stream()
    torch.cuda.synchronize()
    assert lib.ncf_shard_request(item.data_ptr(), cap + 1, W, 0, cap, 10, ib, ic, cursor.data_ptr(), s) == ERR_ARG
    for world in (0, 9):
        assert lib.ncf_shard_request(item.data_ptr(), 4, world, 0, cap, 10, ib, ic, cursor.data_ptr(), s) == ERR_ARG
    assert lib.ncf_shard_request(item.data_ptr(), 4, W, 0, cap, 10, off, ic, cursor.data_ptr(), s) == ERR_ARG
    rows = [torch.zeros(cap * 8, device=_dev()) for _ in range(W)]
    rp = _ptrs([t.data_ptr() for t in rows])
    roff = _ptrs([rows[0].data_ptr(), rows[1].data_ptr() + 4])
    mt, tables, lin, pred, m6 = _flat_model("NeuMF-end", 6, 1, 10, 10, 0)
    assert lib.ncf_shard_push_rows(ctypes.byref(m6), inbox[0].data_ptr(), count[0].data_ptr(), W, cap, rp, rp, s) == ERR_ARG
    _, _, _, _, m8 = _flat_model("NeuMF-end", 8, 1, 10, 10, 0)
    for world in (0, 9):
        assert lib.ncf_shard_push_rows(ctypes.byref(m8), inbox[0].data_ptr(), count[0].data_ptr(), world, cap, rp, rp,
                                       s) == ERR_ARG
    assert lib.ncf_shard_push_rows(ctypes.byref(m8), inbox[0].data_ptr(), count[0].data_ptr(), W, cap, roff, rp, s) == ERR_ARG
    gsrc = torch.zeros(cap * 8, device=_dev())
    assert lib.ncf_shard_push_grads(item.data_ptr(), 4, W, 10, gsrc.data_ptr(), None, 6, 8, rp, None, s) == ERR_ARG
    assert lib.ncf_shard_push_grads(item.data_ptr(), 4, W, 10, gsrc.data_ptr(), None, 8, 8, roff, None, s) == ERR_ARG
    for world in (0, 9):
        assert lib.ncf_shard_push_grads(item.data_ptr(), 4, world, 10, gsrc.data_ptr(), None, 8, 8, rp, None, s) == ERR_ARG
    g = ops.GradBuffers.allocate(mt, 8, 1, 10, 10, 10, _dev())
    for world in (0, 9):
        assert lib.ncf_shard_mark_requests(ctypes.byref(m8), ctypes.byref(g.struct()), inbox[0].data_ptr(),
                                           count[0].data_ptr(), world, cap, s) == ERR_ARG
    torch.cuda.synchronize()
    assert not cursor.any() and all(not t.any() for t in inbox + count + rows)


# ---- 5. the peer barrier, with every peer already arrived ----------------------------------------------------------
def _arm(flags, rank, value, own=0):
    """Every slot of every rank's flag array = value, slot `rank` = own: whatever slot the kernel waits on is
    satisfied at once."""
    for f in flags:
        f.fill_(value)
        f[rank] = own


def _barrier(flags, W, rank, counter):
    rc = _lib().ncf_peer_barrier(_ptrs([f.data_ptr() for f in flags]), W, rank, counter.data_ptr(), _stream())
    assert rc == 0


def _check_arrival(flags, rank, epoch, armed):
    for r, f in enumerate(flags):
        a = f.cpu().numpy().view(np.uint32)
        assert a[rank] == np.uint32(epoch), (r, a[rank], epoch)
        assert (np.delete(a, rank) == np.delete(armed[r], rank)).all(), f"flag array {r}: other slots changed"


@gpu
@pytest.mark.parametrize("W,rank", [(1, 0), (2, 0), (2, 1), (8, 0), (8, 7)])
def test_peer_barrier_publishes_the_epoch_and_counts(W, rank):
    flags = [torch.zeros(8, dtype=torch.int32, device=_dev()) for _ in range(W)]
    counter = torch.zeros(1, dtype=torch.int32, device=_dev())
    for e in (1, 2, 3):                              # eager
        _arm(flags, rank, e + 100)
        armed = [f.cpu().numpy().view(np.uint32).copy() for f in flags]
        _barrier(flags, W, rank, counter)
        torch.cuda.synchronize()
        assert int(counter.item()) == e
        _check_arrival(flags, rank, e, armed)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    _arm(flags, rank, 10_000)
    torch.cuda.synchronize()
    with torch.cuda.graph(graph, stream=s):
        _barrier(flags, W, rank, counter)
    torch.cuda.synchronize()
    assert int(counter.item()) == 3                  # capturing ran nothing
    for e in (4, 5, 6):                              # replayed
        _arm(flags, rank, e + 100)
        armed = [f.cpu().numpy().view(np.uint32).copy() for f in flags]
        torch.cuda.synchronize()
        graph.replay()
        torch.cuda.synchronize()
        assert int(counter.item()) == e
        _check_arrival(flags, rank, e, armed)


@gpu
@pytest.mark.parametrize("W,rank", [(2, 1), (8, 3)])
def test_peer_barrier_counter_wraps(W, rank):
    flags = [torch.zeros(8, dtype=torch.int32, device=_dev()) for _ in range(W)]
    for r, f in enumerate(flags):
        f.copy_(torch.tensor([0, 5, 0, 5, 0, 5, 0, 5], dtype=torch.int32))
        f[rank] = 0
    armed = [f.cpu().numpy().view(np.uint32).copy() for f in flags]
    counter = torch.tensor([-1], dtype=torch.int32, device=_dev())   # 2^32 - 1: the next epoch is 0
    _barrier(flags, W, rank, counter)
    torch.cuda.synchronize()
    assert int(counter.item()) == 0
    _check_arrival(flags, rank, 0, armed)
