"""Full-catalog top-K recommendation and full-ranking evaluation (ncf_mask_items, ncf_topk_rows,
ncf_recommend and their Python layers).

Selection on given score matrices is exact: items, score bits and target ranks equal the numpy restatement
below.  Where the model scores the catalog, the tcgen05 path may differ in the last bit from run to run, so those
comparisons are tie-aware: scores within 1e-5 * max|score| of each other may trade places.
"""
import ctypes
import functools

import numpy as np
import pytest
import torch

from oracle import ncf_numpy as onp

gpu = pytest.mark.gpu


# ---- fixtures ------------------------------------------------------------------------------------------
def _dev():
    return torch.device("cuda:0")


def _quantised_rows(rng, n, C):
    """Rows of a handful of distinct values (ties decide most positions) incl. +-0.0, +-inf and NaN, rows of
    distinct values, rows whose values share their leading bits, short rows and an all-NaN row."""
    vals = np.array([-3.0, -1.0, -0.0, 0.0, 0.5, 1.0, 2.0, np.inf, -np.inf, np.nan], dtype=np.float32)
    s = vals[rng.integers(0, vals.size, (n, C))]
    if n > 1:
        s[1] = rng.standard_normal(C).astype(np.float32)                       # distinct values
    if n > 2:
        s[2] = np.float32(1.0) + np.float32(2.0 ** -23) * rng.integers(0, 4096, C).astype(np.float32)
    if n > 3:
        s[3] = np.nan                                                          # no candidate at all
    if n > 4:
        s[4] = np.nan
        s[4, rng.choice(C, min(C, 3), replace=False)] = vals[rng.integers(0, 8, min(C, 3))]   # short row
    if n > 5:
        s[5] = np.where(rng.random(C) < 0.5, np.float32(-0.0), np.float32(0.0))
    return s


def _targets(rng, scores):
    n, C = scores.shape
    t = rng.integers(0, C, n).astype(np.int64)
    t[0] = -1
    if n > 1:
        t[1] = C
    if n > 3:
        t[3] = C - 1                                                           # NaN column
    return t


# ---- numpy restatement of masking and selection (the reference of the GPU tests below) ----------------------
def mask_items(scores, users, rowptr, col):
    """ncf_mask_items: a copy of scores [n, C] with scores[r, c] = NaN for every item c in [0, C) of user
    users[r]'s CSR row; rows of users outside [0, len(rowptr) - 1) are all NaN."""
    out = np.array(scores, dtype=np.float32, copy=True)
    n, C = out.shape
    user_num = len(rowptr) - 1
    for r in range(n):
        u = int(users[r])
        if u < 0 or u >= user_num:
            out[r, :] = np.nan
            continue
        c = np.asarray(col[rowptr[u]:rowptr[u + 1]], dtype=np.int64)
        out[r, c[(c >= 0) & (c < C)]] = np.nan
    return out


def topk_rows(scores, k, target=None):
    """ncf_topk_rows: the k best non-NaN columns of every row, larger score first, equal scores (-0.0 == +0.0)
    to the lower column; padding -1 / NaN.  Returns (items int64 [n, k], scores float32 [n, k] as stored in
    the row, target_rank int32 [n]: candidates before column target[r], -1 when that column is out of range or
    NaN, or when target is None)."""
    s = np.asarray(scores, dtype=np.float32)
    n, C = s.shape
    items = np.full((n, k), -1, dtype=np.int64)
    top = np.full((n, k), np.nan, dtype=np.float32)
    rank = np.full(n, -1, dtype=np.int32)
    for r in range(n):
        col = np.flatnonzero(~np.isnan(s[r]))
        v = s[r, col].astype(np.float64) + 0.0          # -0.0 -> +0.0
        order = col[np.lexsort((col, -v))]
        m = min(k, order.size)
        items[r, :m] = order[:m]
        top[r, :m] = s[r, order[:m]]
        if target is not None:
            t = int(target[r])
            if 0 <= t < C and not np.isnan(s[r, t]):
                rank[r] = int(np.flatnonzero(order == t)[0])
    return items, top, rank


def _bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _csr(pairs_u, pairs_i, user_num):
    order = np.lexsort((pairs_i, pairs_u))
    u, i = pairs_u[order], pairs_i[order]
    rowptr = np.zeros(user_num + 1, dtype=np.int64)
    np.add.at(rowptr, u + 1, 1)
    return np.cumsum(rowptr), i.astype(np.int32)


def _check_tie_aware(items, scores, rank, ref, k, target=None):
    """items/scores/rank of our call against the oracle ranking of `ref` [n, C] (NaN = excluded)."""
    tol = 1e-5 * float(np.nanmax(np.abs(np.where(np.isinf(ref), np.nan, ref))))
    oi, osc, orank = topk_rows(ref, min(k + 1, ref.shape[1]), target)
    for r in range(ref.shape[0]):
        valid = items[r] >= 0
        assert np.array_equal(valid, oi[r, :k] >= 0), f"row {r}: candidate count differs"
        got = items[r, valid]
        assert not np.isnan(ref[r, got]).any(), f"row {r}: an excluded item was returned"
        assert len(set(got.tolist())) == got.size, f"row {r}: an item was returned twice"
        assert np.all(np.abs(scores[r, valid] - ref[r, got]) <= tol), f"row {r}: returned scores differ"
        os_r = osc[r].astype(np.float64)
        for j in np.flatnonzero(items[r] != oi[r, :k]):
            near = (j > 0 and abs(os_r[j] - os_r[j - 1]) <= tol) or \
                   (j + 1 < os_r.size and abs(os_r[j] - os_r[j + 1]) <= tol)
            assert near, f"row {r}: item {j} differs from the oracle outside the tie tolerance"
        if target is not None:
            if orank[r] < 0:
                assert rank[r] == -1, f"row {r}: rank of an excluded target"
            else:
                t = ref[r, target[r]]
                slack = int(np.sum(np.abs(ref[r][~np.isnan(ref[r])] - t) <= tol))
                assert abs(int(rank[r]) - int(orank[r])) <= slack, f"row {r}: rank {rank[r]} vs {orank[r]}"


# ---- CPU: the numpy restatement against brute force --------------------------------------------------
@pytest.mark.parametrize("C,k", [(1, 1), (7, 3), (31, 10), (200, 50), (50, 64)])
def test_numpy_topk_rows_matches_sorted(C, k):
    rng = np.random.default_rng(C * 131 + k)
    s = _quantised_rows(rng, 12, C)
    t = _targets(rng, s)
    items, top, rank = topk_rows(s, k, t)
    for r in range(s.shape[0]):
        cand = [(c, float(v) + 0.0) for c, v in enumerate(s[r]) if not np.isnan(v)]
        order = [c for c, _ in sorted(cand, key=lambda cv: (-cv[1], cv[0]))]
        want = (order + [-1] * k)[:k]
        assert items[r].tolist() == want
        want_top = np.array([s[r, c] if c >= 0 else np.nan for c in want], dtype=np.float32)
        assert np.array_equal(_bits(top[r]), _bits(want_top))
        want_rank = order.index(t[r]) if 0 <= t[r] < C and t[r] in order else -1
        assert rank[r] == want_rank


def test_numpy_mask_items():
    s = np.arange(12, dtype=np.float32).reshape(3, 4)
    rowptr, col = np.array([0, 2, 2, 5]), np.array([1, 1, 0, 3, 9], dtype=np.int32)
    got = mask_items(s, np.array([0, 1, 5]), rowptr, col)
    assert np.isnan(got[0, 1]) and np.isnan(got[2]).all()
    assert np.array_equal(got[0, [0, 2, 3]], s[0, [0, 2, 3]]) and np.array_equal(got[1], s[1])


# ---- CPU: bad arguments -------------------------------------------------------------------------------
def _fake_model():
    from ncf_b200 import _lib
    m = _lib.NcfModel()
    m.model_type, m.factor_num, m.num_layers, m.mlp_dim = 2, 8, 3, 32
    m.user_num, m.item_num = 100, 50
    m.embed_user_gmf = m.embed_item_gmf = m.embed_user_mlp = m.embed_item_mlp = 256
    for j in range(3):
        m.mlp_w[j] = m.mlp_b[j] = 256
    m.predict_w = m.predict_b = 256
    return m


def test_bad_arguments_are_reported_not_crashed():
    """Every check comes before any CUDA call: the non-NULL pointers below are never dereferenced."""
    from ncf_b200 import _lib
    lib = _lib.load()
    P = 4096   # stands for a device address
    topk = lambda n, C, k, item=P, score=P, ws=0: lib.ncf_topk_rows(P, n, C, k, None, item, score, None, None, ws, None)
    assert topk(4, 5, 0) == -1 and b"k=0" in lib.ncf_last_error()
    assert topk(4, 2000, 1025) == -1 and b"k=1025" in lib.ncf_last_error()
    assert topk(4, 5, 6) == -1 and b"k=6" in lib.ncf_last_error()
    assert topk(4, 0, 1) == -1 and b"C=0" in lib.ncf_last_error()
    assert topk(4, 5, 2, item=None) == -1 and b"null" in lib.ncf_last_error()
    assert topk(4, 5, 2, score=None) == -1
    assert lib.ncf_topk_rows(P, 4, 5, 2, P, P, P, None, None, 0, None) == -1   # target without target_rank
    assert lib.ncf_topk_rows_workspace_bytes(4, 5, 6) == -1
    assert lib.ncf_mask_items(None, 4, 5, P, 10, P, P, None) == -1 and b"null" in lib.ncf_last_error()
    assert lib.ncf_mask_items(P, 4, 0, P, 10, P, P, None) == -1

    m = _fake_model()
    rec = lambda k, chunk=8, item=P, ws=P, wsb=1 << 40, rowptr=None, col=None: lib.ncf_recommend(
        ctypes.byref(m), P, 10, k, rowptr, col, None, chunk, item, P, None, ws, wsb, None)
    assert rec(0) == -1 and b"k=0" in lib.ncf_last_error()
    assert rec(1025) == -1 and b"k=1025" in lib.ncf_last_error()
    assert rec(51) == -1 and b"k=51" in lib.ncf_last_error()                  # k > item_num
    assert rec(5, chunk=0) == -1
    assert rec(5, item=None) == -1 and b"null" in lib.ncf_last_error()
    assert rec(5, rowptr=P) == -1                                             # rowptr without col
    need = lib.ncf_recommend_workspace_bytes(ctypes.byref(m), 8, 5)
    assert need >= 8 * 50 * (4 + 8)
    assert rec(5, wsb=need - 1) == -3 and b"workspace too small" in lib.ncf_last_error()
    assert rec(5, ws=None) == -3
    assert lib.ncf_recommend_workspace_bytes(ctypes.byref(m), 0, 5) == -1
    assert lib.ncf_recommend_workspace_bytes(ctypes.byref(m), 8, 0) == -1
    bad = _fake_model()
    bad.predict_w = None
    assert lib.ncf_recommend(ctypes.byref(bad), P, 10, 5, None, None, None, 8, P, P, None, P, 1 << 40, None) == -1


# ---- GPU: selection and masking are exact ------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("C", [1, 7, 31, 1000, 3706, 26744, 1000003])
def test_topk_rows_is_exact(C):
    from ncf_b200 import ops
    rng = np.random.default_rng(C)
    n = 3 if C > 100000 else (8 if C > 10000 else 40)
    s = _quantised_rows(rng, n, C)
    t = _targets(rng, s)
    st, tt = torch.from_numpy(s).to(_dev()), torch.from_numpy(t).to(_dev())
    for k in [k for k in (1, 10, 100, 1024) if k <= C]:
        items, top, rank = ops.topk_rows(st, k, tt)
        oi, otop, orank = topk_rows(s, k, t)
        assert np.array_equal(items.cpu().numpy(), oi), f"k={k}: items differ"
        assert np.array_equal(_bits(top.cpu().numpy()), _bits(otop)), f"k={k}: score bits differ"
        assert np.array_equal(rank.cpu().numpy(), orank), f"k={k}: target ranks differ"
    items, _, rank = ops.topk_rows(st, 1)
    assert rank is None and np.array_equal(items.cpu().numpy(), topk_rows(s, 1)[0])


@gpu
def test_mask_items_matches_oracle():
    from ncf_b200 import ops
    rng = np.random.default_rng(7)
    U, C, n = 50, 300, 40
    pu = rng.integers(0, U - 10, 2000)                      # users U-10.. have empty rows
    pi = rng.integers(0, C + 20, 2000)                      # some columns >= C
    pu = np.concatenate([pu, pu[:300]])                     # duplicate pairs
    pi = np.concatenate([pi, pi[:300]])
    rowptr, col = ops.csr_build(torch.from_numpy(pu).to(_dev()), torch.from_numpy(pi).to(_dev()), U)
    users = rng.integers(0, U, n)
    users[:3] = [-1, U, U - 1]
    s = rng.standard_normal((n, C)).astype(np.float32)
    got = ops.mask_items(torch.from_numpy(s).to(_dev()), torch.from_numpy(users).to(_dev()), rowptr, col)
    want = mask_items(s, users, *_csr(pu, pi, U))
    assert np.array_equal(_bits(got.cpu().numpy()), _bits(want))


# ---- GPU: recommend end to end ------------------------------------------------------------------------------
def _model(model_type, f, L, U, I, seed=0):
    from ncf_b200.models import NCF
    torch.manual_seed(seed)
    model = NCF(U, I, f, L, 0.0, model_type)
    with torch.no_grad():
        for p in model.parameters():        # spread the scores: the default init leaves them near-equal
            p.mul_(4.0)
    return model.to(_dev()).eval()


@functools.lru_cache(maxsize=None)
def _case(seed, U, I, n_pairs):
    rng = np.random.default_rng(seed)
    pu, pi = rng.integers(0, U, n_pairs), rng.integers(0, I, n_pairs)
    return pu, pi, _csr(pu, pi, U)


def _oracle_scores(model, users, I, pu, pi):
    params = {k: v.detach().cpu().numpy() for k, v in model.state_dict().items()}
    ref = onp.forward(params, np.repeat(users, I), np.tile(np.arange(I), users.size), model.model_type)
    return mask_items(ref.reshape(users.size, I), users, *_csr(pu, pi, model.user_num))


PATHS = [("GMF", 8, 1, 1), ("NeuMF-end", 8, 3, 4), ("MLP", 16, 2, 2), ("NeuMF-end", 6, 2, 1), ("NeuMF-end", 32, 3, 3)]


@gpu
@pytest.mark.parametrize("model_type,f,L,path", PATHS, ids=[f"{m}-f{f}-L{L}" for m, f, L, _ in PATHS])
def test_recommend_matches_oracle_on_every_tile_path(model_type, f, L, path):
    from ncf_b200 import _lib, ops
    U, I, k, chunk = 200, 700, 10, 20                        # 14 000 pairs per chunk: tcgen05 for f = 32
    model = _model(model_type, f, L, U, I)
    pu, pi, _ = _case(1, U, I, 30000)
    rowptr, col = ops.csr_build(torch.from_numpy(pu).to(_dev()), torch.from_numpy(pi).to(_dev()), U)
    rng = np.random.default_rng(2)
    users = rng.permutation(U)[:160]
    target = rng.integers(0, I, users.size)
    items, scores, rank = ops.recommend(model.abi_struct(), torch.from_numpy(users).to(_dev()), k, chunk, rowptr, col,
                                        torch.from_numpy(target).to(_dev()))
    assert _lib.load().ncf_last_tile_path() == path
    ref = _oracle_scores(model, users, I, pu, pi)
    _check_tie_aware(items.cpu().numpy(), scores.cpu().numpy(), rank.cpu().numpy(), ref, k, target)
    excluded = set(zip(pu.tolist(), pi.tolist()))
    assert not any((int(u), int(i)) in excluded for u, row in zip(users, items.cpu().numpy()) for i in row)


@gpu
def test_chunk_size_does_not_change_results():
    from ncf_b200.recommend import recommend_ranked
    U, I, k = 60, 700, 25
    model = _model("NeuMF-end", 32, 3, U, I, seed=3)
    pu, pi, _ = _case(4, U, I, 8000)
    from ncf_b200 import ops
    exclude = ops.csr_build(torch.from_numpy(pu).to(_dev()), torch.from_numpy(pi).to(_dev()), U)
    users = np.arange(U)
    target = np.random.default_rng(5).integers(0, I, U)
    ref = _oracle_scores(model, users, I, pu, pi)
    for chunk in (1, 7, U):
        items, scores, rank = recommend_ranked(model, torch.from_numpy(users).to(_dev()), k, exclude, chunk,
                                               torch.from_numpy(target).to(_dev()))
        _check_tie_aware(items.cpu().numpy(), scores.cpu().numpy(), rank.cpu().numpy(), ref, k, target)


@gpu
def test_full_ranking_restricted_to_candidates_equals_sampled_evaluation():
    """Excluding every item but a user's 100 test candidates turns the full ranking into the sampled one."""
    from ncf_b200 import ops
    from ncf_b200.metrics import evaluate, evaluate_full_ranking
    from ncf_b200.synth import make_interactions
    d = make_interactions("tiny", device=_dev())
    model = _model("NeuMF-end", 8, 3, d.user_num, d.item_num, seed=6)
    cands = d.test_cands.cpu().numpy()
    keep = np.zeros((cands.shape[0], d.item_num), dtype=bool)
    keep[np.arange(cands.shape[0])[:, None], cands] = True
    users = d.test_users.cpu().numpy()
    ex_u, ex_i = np.nonzero(~keep)
    exclude = ops.csr_build(torch.from_numpy(users[ex_u]).to(_dev()), torch.from_numpy(ex_i).to(_dev()), d.user_num)
    rank, hr, ndcg = evaluate_full_ranking(model, d.test_users, d.test_cands[:, 0].contiguous(), exclude, ks=(1, 10))
    res = evaluate(model, d.test_users, d.test_cands, 10)
    full, sampled, s = rank.cpu().numpy(), res.rank.cpu().numpy(), res.scores.cpu().numpy()
    tol = 1e-5 * float(np.abs(s).max())
    within = sampled >= 0
    assert within.any()
    for r in np.flatnonzero(within):
        slack = int(np.sum(np.abs(s[r] - s[r, 0]) <= tol)) - 1
        assert abs(int(full[r]) - int(sampled[r])) <= slack, f"user {r}: full {full[r]} vs sampled {sampled[r]}"
    assert (full[~within] >= 10 - 1).all()
    assert abs(hr[10] - float(np.mean(within))) <= 2.0 / len(sampled)
    HR, NDCG = res.lists()
    assert abs(ndcg[10] - float(np.mean(NDCG))) <= 2.0 / len(sampled)


@gpu
def test_recommend_replays_in_a_cuda_graph():
    from ncf_b200 import ops
    U, I, k, chunk = 64, 3000, 20, 16
    model = _model("NeuMF-end", 32, 3, U, I, seed=8)
    pu, pi, _ = _case(9, U, I, 20000)
    rowptr, col = ops.csr_build(torch.from_numpy(pu).to(_dev()), torch.from_numpy(pi).to(_dev()), U)
    users = torch.arange(U, device=_dev())
    target = torch.from_numpy(np.random.default_rng(10).integers(0, I, U)).to(_dev())
    m = model.abi_struct()
    ws = torch.empty(ops.recommend_workspace_bytes(m, chunk, k), dtype=torch.uint8, device=_dev())
    eager = ops.recommend(m, users, k, chunk, rowptr, col, target, workspace=ws)
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            captured = ops.recommend(m, users, k, chunk, rowptr, col, target, workspace=ws)
    for t in captured:
        t.fill_(-7)
    g.replay()
    torch.cuda.synchronize()
    ref = _oracle_scores(model, users.cpu().numpy(), I, pu, pi)
    for items, scores, rank in (eager, captured):
        _check_tie_aware(items.cpu().numpy(), scores.cpu().numpy(), rank.cpu().numpy(), ref, k, target.cpu().numpy())


@gpu
def test_million_item_catalog_in_chunks():
    from ncf_b200 import ops
    U, I, k, chunk = 8, 1_000_000, 100, 2
    model = _model("NeuMF-end", 32, 3, U, I, seed=11)
    rng = np.random.default_rng(12)
    pu, pi = rng.integers(0, U, 50000), rng.integers(0, I, 50000)
    rowptr, col = ops.csr_build(torch.from_numpy(pu).to(_dev()), torch.from_numpy(pi).to(_dev()), U)
    users = np.array([3, 0, 7, 5, 6], dtype=np.int64)
    target = rng.integers(0, I, users.size)
    m = model.abi_struct()
    need = ops.recommend_workspace_bytes(m, chunk, k)
    assert need < 2**30                                             # two users: scores, ids, forward scratch
    ws = torch.empty(need, dtype=torch.uint8, device=_dev())
    items, scores, rank = ops.recommend(m, torch.from_numpy(users).to(_dev()), k, chunk, rowptr, col,
                                        torch.from_numpy(target).to(_dev()), workspace=ws)
    ut = torch.from_numpy(np.repeat(users, I)).to(_dev())
    it = torch.arange(I, device=_dev()).repeat(users.size)
    with torch.no_grad():
        ref = ops.forward(m, ut, it).cpu().numpy().reshape(users.size, I)
    ref = mask_items(ref, users, *_csr(pu, pi, U))
    _check_tie_aware(items.cpu().numpy(), scores.cpu().numpy(), rank.cpu().numpy(), ref, k, target)


# ---- GPU: quality and the command line -----------------------------------------------------------------------
def _train_tiny(epochs):
    from ncf_b200.models import NCF
    from ncf_b200.synth import make_interactions
    from ncf_b200.train_loop import fit
    d = make_interactions("tiny", device=_dev())
    torch.manual_seed(0)
    model = NCF(d.user_num, d.item_num, 8, 3, 0.0, "NeuMF-end").to(_dev())
    train = torch.stack([d.pos_user, d.pos_item], 1)
    if epochs:
        fit(model, train, d.test_users, d.test_cands, epochs=epochs, batch_size=256, lr=1e-3, num_ng=4, top_k=10)
    return d, model.eval()


@gpu
def test_trained_model_ranks_held_out_items_well_above_chance():
    from ncf_b200 import ops
    from ncf_b200.metrics import evaluate_full_ranking
    d, untrained = _train_tiny(0)
    untrained = {k: v.clone() for k, v in untrained.state_dict().items()}
    d, model = _train_tiny(5)
    exclude = ops.csr_build(d.pos_user, d.pos_item, d.user_num)
    targets = d.test_cands[:, 0].contiguous()
    _, hr, ndcg = evaluate_full_ranking(model, d.test_users, targets, exclude)
    unseen = d.item_num - torch.bincount(d.pos_user, minlength=d.user_num).cpu().numpy()
    chance = float(np.mean(10.0 / unseen))
    model.load_state_dict(untrained)
    _, hr0, _ = evaluate_full_ranking(model, d.test_users, targets, exclude)
    assert hr[10] >= 3 * chance, (hr[10], chance)
    assert hr[10] > hr0[10] + 0.05, (hr[10], hr0[10])
    assert hr[1] <= hr[5] <= hr[10] <= hr[20] and ndcg[10] <= hr[10]


@gpu
def test_command_line_writes_unseen_top_k(tmp_path, capsys):
    import importlib.util
    from pathlib import Path
    root = Path(__file__).resolve().parent.parent
    spec = importlib.util.spec_from_file_location("recommend_cli", root / "scripts" / "recommend.py")
    cli = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(cli)
    d, model = _train_tiny(1)
    ckpt, out = tmp_path / "model.pth", tmp_path / "recs.tsv"
    torch.save(model.state_dict(), ckpt)
    k = 15
    res = cli.main(["--checkpoint", str(ckpt), "--model", "NeuMF-end", "--factor_num", "8", "--num_layers", "3",
                    "--synthetic", "tiny", "--top_k", str(k), "--out", str(out)])
    text = capsys.readouterr().out
    assert "--- RESULTS ---" in text and f"HR@{k}:" in text and f"NDCG@{k}:" in text
    assert f"Users: {d.user_num}" in text and f"Items: {d.item_num}" in text
    seen = {}
    for u, i in zip(d.pos_user.tolist(), d.pos_item.tolist()):
        seen.setdefault(u, set()).add(i)
    lines = out.read_text().splitlines()
    assert len(lines) == d.user_num
    for line in lines:
        fields = [int(x) for x in line.split("\t")]
        u, items = fields[0], fields[1:]
        assert len(items) == k and len(set(items)) == k and min(items) >= 0
        assert not (set(items) & seen.get(u, set())), f"user {u}: a training item was recommended"
    assert 0.0 <= res["hr"] <= 1.0
