"""Leave-one-out ranking (ncf_eval_rank) and evaluation (ncf_eval_users) against references.

Ranking is checked bit for bit against the numpy restatement below.  End to end, the ranking of the
device's own scores is checked exactly, and only the scores are compared with the oracle within a
tolerance; the oracle's ranking is compared only for rows whose held-out score is clear of every other
candidate.  So no check depends on how near-ties fall.

Order: larger score first; equal scores (-0.0 == +0.0) go to the lower column; NaN is not a candidate.
Rows with fewer than k numbers pad topk with -1; a NaN held-out score is a miss.
"""
import ctypes

import numpy as np
import pytest
import torch

from oracle import ncf_numpy as onp
from tests.test_recommend import _quantised_rows
from tests.util import assert_close

gpu = pytest.mark.gpu


def _dev():
    return torch.device("cuda:0")


# ---- numpy restatement of ncf_eval_rank (the reference of the GPU tests below) -----------------------------
def rank_rows(scores, k):
    """-> (hit uint8 [n], rank int32 [n], ndcg float64 [n], topk int32 [n, k]) of scores [n, C]: topk = the k
    best non-NaN columns, larger score first, equal scores (-0.0 == +0.0) to the lower column, padded with
    -1; rank = position of column 0 in that order, -1 when it is NaN or not among the first k."""
    s = np.asarray(scores, dtype=np.float32)
    n, C = s.shape
    nan = np.isnan(s)
    neg = np.where(nan, 0.0, -(s.astype(np.float64) + 0.0))
    cols = np.broadcast_to(np.arange(C), (n, C))
    order = np.lexsort((cols, neg, nan), axis=-1)          # last key first: numbers before NaN
    valid = np.take_along_axis(~nan, order, axis=1)
    topk = np.where(valid[:, :k], order[:, :k], -1).astype(np.int32)
    pos = np.argmax(order == 0, axis=1)
    rank = np.where(~nan[:, 0] & (pos < k), pos, -1).astype(np.int32)
    ndcg = np.where(rank >= 0, 1.0 / np.log2(np.maximum(rank, 0) + 2.0), 0.0)
    return (rank >= 0).astype(np.uint8), rank, ndcg, topk


SPECIALS = np.array([0.0, -0.0, np.inf, -np.inf, 1e-45, -1e-45, 1e-40, -3e-39, 1.0, -1.0, 2.0], dtype=np.float32)
LEVELS = np.array([-1.0, 0.0, 0.5, 1.0], dtype=np.float32)


def _rows(rng, n, C):
    """n rows of C scores; row r is of kind r % 12: distinct values, a few levels (ties decide most places),
    all equal, +-0 / +-inf / subnormals, NaN held-out score, NaN in a lane's first slot (column < 32), NaN
    in a later slot (column >= 32), NaN in the last column, all NaN, fewer than 12 numbers, scattered NaN
    among ties, specials with scattered NaN.  Where a NaN sits elsewhere, column 0 gets one of the row's
    larger values, so that its rank depends on how the NaN is treated."""
    s = rng.standard_normal((n, C)).astype(np.float32)
    for r in range(n):
        kind = r % 12
        if kind == 1:
            s[r] = LEVELS[rng.integers(0, LEVELS.size, C)]
        elif kind == 2:
            s[r] = 0.25
        elif kind == 3:
            s[r] = SPECIALS[rng.integers(0, SPECIALS.size, C)]
        elif kind == 4:
            s[r] = LEVELS[rng.integers(0, LEVELS.size, C)]
            s[r, 0] = np.nan
        elif kind in (5, 6, 7) and C > 1:
            s[r] = np.round(s[r] * 2) / 2                  # ties as well
            if kind == 5:
                c = rng.integers(1, min(C, 32)) if C > 2 else 1
            elif kind == 6:
                c = rng.integers(32, C) if C > 32 else C - 1
            else:
                c = C - 1
            s[r, 0] = np.sort(s[r])[-rng.integers(1, min(C, 12) + 1)]
            s[r, c] = np.nan
        elif kind == 8:
            s[r] = np.nan
        elif kind == 9:
            m = rng.integers(1, min(C, 12) + 1)
            keep = rng.choice(C, m, replace=False)
            vals = LEVELS[rng.integers(0, LEVELS.size, m)]
            s[r] = np.nan
            s[r, keep] = vals
        elif kind == 10:
            s[r] = LEVELS[rng.integers(0, LEVELS.size, C)]
            s[r, rng.random(C) < 0.2] = np.nan
        elif kind == 11:
            s[r] = SPECIALS[rng.integers(0, SPECIALS.size, C)]
            s[r, rng.random(C) < 0.3] = np.nan
    return s


def _ks(C):
    return sorted({k for k in (1, 10, C) if k <= C})


def _sorted_ranking(row, k):
    """One row by brute force: (rank, topk list)."""
    cand = [(c, float(v) + 0.0) for c, v in enumerate(row) if not np.isnan(v)]
    order = [c for c, _ in sorted(cand, key=lambda cv: (-cv[1], cv[0]))]
    top = (order + [-1] * k)[:k]
    return (top.index(0) if 0 in top else -1), top


# ---- CPU: the restatement against brute force ---------------------------------------------------------------
@pytest.mark.parametrize("C,k", [(1, 1), (2, 2), (31, 10), (33, 33), (64, 1), (100, 10), (1024, 1024)])
def test_numpy_rank_rows_matches_sorted(C, k):
    rng = np.random.default_rng(C * 31 + k)
    s = np.concatenate([_rows(rng, 36, C), _quantised_rows(rng, 12, C)])
    hit, rank, ndcg, topk = rank_rows(s, k)
    for r in range(s.shape[0]):
        want_rank, want_top = _sorted_ranking(s[r], k)
        assert topk[r].tolist() == want_top, f"row {r}"
        assert rank[r] == want_rank and hit[r] == (want_rank >= 0), f"row {r}"
        assert ndcg[r] == (0.0 if want_rank < 0 else 1.0 / np.log2(want_rank + 2)), f"row {r}"
    nan0 = np.isnan(s[:, 0])
    assert nan0.any() and (rank[nan0] == -1).all()         # the rows cover a NaN held-out score
    assert (np.isnan(s).all(1) & (topk == -1).all(1)).any()


# ---- CPU: bad arguments --------------------------------------------------------------------------------------
def test_bad_arguments_are_reported_and_empty_input_is_a_no_op():
    """Every check comes before any CUDA call: the non-NULL pointers below are never dereferenced."""
    from ncf_b200 import _lib
    from tests.test_recommend import _fake_model
    lib = _lib.load()
    P = 4096   # stands for a device address
    rank = lambda n, C, k, s=P: lib.ncf_eval_rank(s, n, C, k, P, P, P, P, None)
    assert rank(4, 1025, 1) == -1 and b"C=1025" in lib.ncf_last_error()
    assert rank(4, 0, 1) == -1 and b"C=0" in lib.ncf_last_error()
    assert rank(4, 5, 6) == -1 and b"k=6" in lib.ncf_last_error()
    assert rank(4, 5, 0) == -1 and b"k=0" in lib.ncf_last_error()
    assert rank(-1, 5, 1) == -1 and b"negative n" in lib.ncf_last_error()
    assert rank(4, 5, 2, s=None) == -1 and b"NULL" in lib.ncf_last_error()
    assert rank(0, 1024, 1024, s=None) == 0                                  # n = 0: nothing to do
    m = _fake_model()
    users = lambda n, C, k, ws=P, wsb=1 << 40: lib.ncf_eval_users(ctypes.byref(m), P, P, n, C, k, P, P, P, P, P,
                                                                  ws, wsb, None)
    assert users(4, 1025, 1) == -1 and b"C=1025" in lib.ncf_last_error()
    assert users(4, 50, 51) == -1 and b"k=51" in lib.ncf_last_error()
    assert users(0, 100, 10, ws=None, wsb=0) == 0
    assert users(4, 100, 10, ws=None) == -3 and b"workspace too small" in lib.ncf_last_error()
    assert lib.ncf_eval_users(ctypes.byref(m), None, P, 4, 100, 10, P, P, P, P, P, P, 1 << 40, None) == -1


# ---- GPU: ncf_eval_rank on given scores is exact ---------------------------------------------------------------
def _check_ranking(scores, k, hit, rank, ndcg, topk, what=""):
    """Device outputs (tensors) == rank_rows(scores): hit, rank and topk exactly, ndcg within 1 ulp of the
    float32 of the float64 value."""
    w_hit, w_rank, w_ndcg, w_topk = rank_rows(scores, k)
    got_rank, got_topk = rank.cpu().numpy(), topk.cpu().numpy()
    for name, got, want in (("rank", got_rank, w_rank), ("topk", got_topk, w_topk)):
        bad = np.flatnonzero((got != want).reshape(got.shape[0], -1).any(1))
        assert bad.size == 0, f"{what} k={k}: {name} differs in {bad.size} rows, first {bad[0]}: " \
                              f"{got[bad[0]]} vs {want[bad[0]]}, scores {scores[bad[0], :12]}"
    assert np.array_equal(hit.cpu().numpy(), w_hit), f"{what} k={k}: hit"
    got_nd = ndcg.cpu().numpy().view(np.int32).astype(np.int64)
    want_nd = w_ndcg.astype(np.float32).view(np.int32).astype(np.int64)
    assert np.abs(got_nd - want_nd).max() <= 1, f"{what} k={k}: ndcg beyond 1 ulp"


EVAL_C = [1, 2, 31, 32, 33, 64, 100, 101, 1000, 1023, 1024]


@gpu
@pytest.mark.parametrize("C", EVAL_C)
def test_eval_rank_matches_restatement(C):
    from ncf_b200 import ops
    s = _rows(np.random.default_rng(C), 240, C)
    st = torch.from_numpy(s).to(_dev())
    for k in _ks(C):
        _check_ranking(s, k, *ops.eval_rank(st, k), what=f"C={C}")


@gpu
@pytest.mark.parametrize("C", EVAL_C)
def test_eval_rank_agrees_with_topk_rows(C):
    """ncf_topk_rows(target = column 0) on the same rows: the same order, so the same first k columns, and
    its full target rank equals the eval rank where that is >= 0 and is >= k (or -1 for a NaN column 0)
    where the eval rank is -1."""
    from ncf_b200 import ops
    s = _rows(np.random.default_rng(C + 1), 240, C)
    st = torch.from_numpy(s).to(_dev())
    target = torch.zeros(s.shape[0], dtype=torch.int64, device=_dev())
    nan0 = np.isnan(s[:, 0])
    for k in _ks(C):
        _, rank, _, topk = ops.eval_rank(st, k)
        items, _, full = ops.topk_rows(st, k, target)
        rank, full = rank.cpu().numpy(), full.cpu().numpy()
        assert np.array_equal(items.cpu().numpy(), topk.cpu().numpy().astype(np.int64)), f"k={k}: top k differs"
        inside = rank >= 0
        assert np.array_equal(full[inside], rank[inside]), f"k={k}"
        assert np.all(np.where(nan0, full == -1, full >= k)[~inside]), f"k={k}"


@gpu
def test_eval_rank_with_several_rows_per_warp():
    """The grid is capped at num_sms * 8 blocks of 8 warps; 30 000 rows give every warp several."""
    from ncf_b200 import ops
    n, C, k = 30000, 100, 10
    assert n >= 3 * torch.cuda.get_device_properties(0).multi_processor_count * 8 * 8
    s = _rows(np.random.default_rng(5), n, C)
    _check_ranking(s, k, *ops.eval_rank(torch.from_numpy(s).to(_dev()), k))


@gpu
def test_eval_rank_outputs_may_be_null():
    """Each of hit / rank / ndcg / topk_idx passed as NULL in turn: the other outputs do not change."""
    from ncf_b200 import _lib, ops
    from ncf_b200._lib import check, current_stream, ptr
    lib = _lib.load()
    n, C, k = 500, 100, 10
    s = _rows(np.random.default_rng(6), n, C)
    st = torch.from_numpy(s).to(_dev())
    full = ops.eval_rank(st, k)
    _check_ranking(s, k, *full)
    for drop in range(4):
        outs = [torch.full_like(t, 7) for t in full]
        args = [None if j == drop else ptr(o) for j, o in enumerate(outs)]
        check(lib.ncf_eval_rank(ptr(st), n, C, k, *args, current_stream()), "ncf_eval_rank")
        for j in range(4):
            want = full[j] if j != drop else torch.full_like(full[j], 7)
            assert torch.equal(outs[j].view(torch.uint8), want.view(torch.uint8)), f"NULL output {drop}: output {j}"


@gpu
def test_eval_rank_of_no_rows():
    from ncf_b200 import ops
    hit, rank, ndcg, topk = ops.eval_rank(torch.empty(0, 100, device=_dev()), 10)
    assert hit.numel() == rank.numel() == ndcg.numel() == topk.numel() == 0


# ---- GPU: ncf_eval_users end to end on every tile path --------------------------------------------------------
U, I = 400, 1200


def _model(model_type, f, L, seed):
    """Embeddings scaled as the metrics goldens do (x60) so that near-ties are rare; non-zero biases."""
    from ncf_b200.models import NCF
    torch.manual_seed(seed)
    model = NCF(U, I, f, L, 0.0, model_type)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if name.startswith("embed_"):
                p.mul_(60.0)
        for lin in model.linears():
            lin.bias.uniform_(-0.1, 0.1)
    return model.to(_dev()).eval()


def _inputs(rng, n, C):
    """users [n], cands [n, C] (distinct items per row, as the test sets have) with out-of-range ids: a bad
    candidate in row 1, a bad held-out item in row 2, a bad user in row 3."""
    users = rng.integers(0, U, n)
    cands = np.stack([rng.choice(I, C, replace=False) for _ in range(n)])
    cands[1, C // 2] = I
    cands[2, 0] = -1
    users[3] = U
    return users, cands


def _device_users(users, pad):
    """users on the device, followed in the same allocation by `pad` valid ids: a kernel that indexed the
    users wrongly (by row instead of row / C) would read wrong values, not memory outside the buffer."""
    buf = torch.zeros(users.size + pad, dtype=torch.int64, device=_dev())
    buf[:users.size] = torch.from_numpy(users).to(_dev())
    return buf[:users.size]


def _oracle_scores(model, users, cands):
    """oracle forward of every (user, candidate) pair; NaN where an id is outside the tables."""
    n, C = cands.shape
    bad = (cands < 0) | (cands >= I) | ((users < 0) | (users >= U))[:, None]
    params = {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}
    u = np.where(bad, 0, np.repeat(users, C).reshape(n, C)).reshape(-1)
    i = np.where(bad, 0, cands).reshape(-1)
    ref = onp.forward(params, u, i, model.model_type).reshape(n, C)
    ref[bad] = np.nan
    return ref, bad


def _check_scores(got, ref, bad, math, what):
    """NaN exactly at the out-of-range pairs; the rest within the fp32 bar, or the TF32 bound."""
    assert np.array_equal(np.isnan(got), bad), f"{what}: NaN scores are not exactly the out-of-range pairs"
    if math == "tf32":
        assert np.max(np.abs(got[~bad] - ref[~bad])) <= 5e-3 * np.max(np.abs(ref[~bad])), f"{what}: tf32 scores"
    else:
        assert_close(got[~bad], ref[~bad], f"{what}: candidate scores")


# (model_type, f, L, n, C, tile path, tower_math, NCF_UMMA_FUSED)
E2E = [
    ("GMF", 8, 1, 64, 100, 1, "fp32", None),
    ("NeuMF-end", 6, 2, 64, 100, 1, "fp32", None),
    ("NeuMF-end", 12, 2, 40, 100, 1, "fp32", None),
    ("NeuMF-end", 64, 4, 30, 100, 1, "fp32", None),         # too wide for tcgen05 and the mma.sync smem
    ("NeuMF-end", 8, 1, 64, 100, 4, "fp32", None),
    ("NeuMF-end", 8, 2, 64, 100, 4, "fp32", None),
    ("NeuMF-end", 8, 3, 64, 100, 4, "fp32", None),
    ("MLP", 8, 1, 64, 100, 4, "fp32", None),
    ("MLP", 8, 3, 64, 100, 4, "fp32", None),
    ("NeuMF-end", 32, 2, 20, 100, 5, "fp32", None),         # n*C <= 2048: the layer-per-launch forward
    ("NeuMF-end", 16, 1, 30, 67, 5, "fp32", None),          # C not a multiple of 32
    ("NeuMF-end", 16, 2, 30, 100, 2, "fp32", None),         # 32-row mma.sync tiles
    ("NeuMF-end", 16, 2, 60, 100, 2, "fp32", None),         # 64-row tiles
    ("NeuMF-end", 32, 3, 50, 100, 2, "fp32", None),         # below the tcgen05 threshold
    ("NeuMF-end", 32, 3, 50, 100, 2, "tf32", None),
    ("NeuMF-end", 32, 3, 100, 100, 3, "fp32", None),        # fused tcgen05 tower kernel
    ("NeuMF-end", 64, 2, 90, 100, 3, "fp32", None),
    ("NeuMF-end", 32, 3, 100, 100, 3, "tf32", None),
    ("NeuMF-end", 128, 1, 300, 999, 3, "fp32", None),       # per-layer GEMMs; the 2nd sub-batch starts at user 262
    ("NeuMF-end", 32, 3, 300, 999, 3, "fp32", "0"),
]


def _e2e_id(case):
    mt, f, L, n, C, path, math, fused = case
    return f"path{path}-{mt}-f{f}-L{L}-{n}x{C}" + ("-tf32" if math == "tf32" else "") + \
        ("-perlayer" if fused == "0" else "")


@gpu
@pytest.mark.parametrize("case", E2E, ids=[_e2e_id(c) for c in E2E])
def test_eval_users_on_every_tile_path(case, monkeypatch):
    from ncf_b200 import _lib
    from ncf_b200._lib import check, current_stream, ptr
    from ncf_b200.metrics import evaluate
    model_type, f, L, n, C, path, math, fused = case
    k = 10
    for var in ("NCF_UMMA_MIN_B", "NCF_UMMA_DISABLE", "NCF_UMMA_FUSED"):
        monkeypatch.delenv(var, raising=False)
    if fused is not None:
        monkeypatch.setenv("NCF_UMMA_FUSED", fused)
    lib = _lib.load()
    model = _model(model_type, f, L, seed=n * C + f)
    model.tower_math = math
    users, cands = _inputs(np.random.default_rng(f * 1000 + n), n, C)
    ud, cd = _device_users(users, n * C), torch.from_numpy(cands).to(_dev())
    with torch.no_grad():
        res = evaluate(model, ud, cd, k)
    assert lib.ncf_last_tile_path() == path, f"ran on tile path {lib.ncf_last_tile_path()}"
    got = res.scores.cpu().numpy()
    ref, bad = _oracle_scores(model, users, cands)

    # (a) scoring against the oracle; out-of-range ids give NaN
    _check_scores(got, ref, bad, math, "scores_out")
    # (b) ranking of the device's own scores, exactly
    _check_ranking(got, k, res.hit, res.rank, res.ndcg, res.topk, what=_e2e_id(case))
    topk = res.topk.cpu().numpy()
    assert C // 2 not in topk[1] and res.rank[2].item() == -1 and res.rank[3].item() == -1
    assert (topk[3] == -1).all()
    # (c) ranking of the oracle's scores where the held-out score is clear of every other candidate: by more
    # than twice the largest deviation of any device score, so that no comparison with it can flip
    if math == "fp32":
        tol = 2 * np.max(np.abs(got[~bad] - ref[~bad]))
        gap = np.abs(ref - ref[:, :1])
        gap[:, 0] = np.inf
        clear = np.where(np.isnan(gap), np.inf, gap).min(1) > tol
        w_hit, w_rank, _, _ = rank_rows(ref, k)
        assert clear.mean() >= 0.75, f"only {clear.sum()} of {n} rows are clear of near-ties"
        assert np.array_equal(res.rank.cpu().numpy()[clear], w_rank[clear])
        assert np.array_equal(res.hit.cpu().numpy()[clear], w_hit[clear])

    # scores_out = NULL: the scores stay at the start of the workspace (eval.cu), which starts filled with NaN
    # (0xFF bytes), so a read of a score that was never written is a miss and shows up below
    m = model.abi_struct()
    nbytes = int(lib.ncf_eval_workspace_bytes(ctypes.byref(m), n, C))
    ws = torch.full((nbytes,), 0xFF, dtype=torch.uint8, device=_dev())
    outs = [torch.empty_like(t) for t in (res.hit, res.rank, res.ndcg, res.topk)]
    check(lib.ncf_eval_users(ctypes.byref(m), ptr(ud), ptr(cd), n, C, k, *map(ptr, outs), None, ptr(ws), nbytes,
                             current_stream()), "ncf_eval_users")
    assert lib.ncf_last_tile_path() == path
    ws_scores = ws[:n * C * 4].view(torch.float32).reshape(n, C).cpu().numpy()
    _check_scores(ws_scores, ref, bad, math, "scores_out = NULL")
    _check_ranking(ws_scores, k, *outs, what="scores_out = NULL")
    # the tcgen05 kernels may round differently from run to run: rows of bitwise-equal scores rank equally
    same = (ws_scores.view(np.uint32) == got.view(np.uint32)).all(1)
    for name, a, b in zip(("hit", "rank", "ndcg", "topk"), outs, (res.hit, res.rank, res.ndcg, res.topk)):
        assert np.array_equal(a.cpu().numpy()[same], b.cpu().numpy()[same]), f"scores_out = NULL: {name} differs"


# ---- GPU: what a user sees from a model that gives NaN ------------------------------------------------------
@gpu
def test_nan_model_scores_zero_not_one():
    """A model whose every score is NaN (here: predict_layer.bias = NaN) is a miss for every user in
    evaluate, metrics() and evaluate_top_k, not a perfect HR = 1."""
    import torch.utils.data as data
    from ncf_b200.datasets import NCFData
    from ncf_b200.metrics import evaluate, evaluate_top_k, metrics
    model = _model("NeuMF-end", 8, 3, seed=1)
    with torch.no_grad():
        model.predict_layer.bias.fill_(float("nan"))
    rng = np.random.default_rng(1)
    n, C = 50, 100
    users, cands = rng.integers(0, U, n), rng.integers(0, I, (n, C))
    ud, cd = torch.from_numpy(users).to(_dev()), torch.from_numpy(cands).to(_dev())
    with torch.no_grad():
        res = evaluate(model, ud, cd, 10)
        hr_at_k, ndcg_at_k = evaluate_top_k(model, ud, cd, 10)
    assert torch.isnan(res.scores).all()
    assert (res.hit == 0).all() and (res.rank == -1).all() and (res.ndcg == 0).all() and (res.topk == -1).all()
    HR, NDCG = res.lists()
    assert HR == [0] * n and NDCG == [0.0] * n
    assert set(hr_at_k.values()) == {0.0} and set(ndcg_at_k.values()) == {0.0}
    pairs = np.stack([np.repeat(users, C), cands.reshape(-1)], 1)
    loader = data.DataLoader(NCFData(pairs, I, None, 0, False), batch_size=C, shuffle=False)
    HR, NDCG = metrics(model, loader, 10)
    assert HR == [0] * n and NDCG == [0.0] * n
