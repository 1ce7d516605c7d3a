"""ORACLE tooling — generates tests/golden/*.npz by running the UNMODIFIED reference.

Runs only in the build container (it imports /root/reference, which does not exist on the GPU
box).  The reference needs two accommodations to import here (SURVEY.md §8c): `matplotlib` is
missing (stubbed with empty modules; only plotting uses it) and `src.utils.config` reads a
CWD-relative YAML and mkdirs `results/` on import (we chdir to a scratch copy of the YAML).

    python oracle/make_golden.py            # rewrites tests/golden/
    python oracle/make_golden.py --sweep-only   # only the SWEEP_CASES fixtures

Every fixture records the inputs (initial state_dict, index/label batches) and what the reference
computed from them (logits, losses, autograd gradients, weights after optimiser steps, HR/NDCG).
"""
from __future__ import annotations

import json
import os
import shutil
import sys
import tempfile
import types
from pathlib import Path

import numpy as np
import torch

REPO = Path(__file__).resolve().parent.parent
OUT = REPO / "tests" / "golden"
REF = Path("/root/reference")


def import_reference():
    for m in ("matplotlib", "matplotlib.pyplot"):
        sys.modules.setdefault(m, types.ModuleType(m))
    scratch = tempfile.mkdtemp(prefix="ncf_ref_")
    os.makedirs(scratch + "/configs/experiments")
    shutil.copy(REF / "configs/experiments/neumf.yaml", scratch + "/configs/experiments/")
    os.chdir(scratch)
    sys.path.insert(0, str(REF))
    from src.ncf.models import NCF
    from src.training.metrics import metrics
    from src.distillation import ResponseDistillation
    from src.data.datasets import NCFData
    return NCF, metrics, ResponseDistillation, NCFData


def sd_np(model, prefix):
    return {f"{prefix}/{k}": v.detach().cpu().numpy().copy() for k, v in model.state_dict().items()}


def grads_np(model, prefix):
    out = {}
    for k, p in model.named_parameters():
        if p.grad is not None:
            out[f"{prefix}/{k}"] = p.grad.detach().cpu().numpy().copy()
    return out


def make_batches(rng, U, I, B, T, hot_users=None):
    """Random (user, item, label) batches; a few 'hot' users/items repeat inside a batch and a
    good share of rows is absent from some steps, which is what exercises the lazy Adam."""
    user = rng.integers(0, U, size=(T, B))
    item = rng.integers(0, I, size=(T, B))
    if hot_users:
        user[:, : B // 4] = rng.integers(0, hot_users, size=(T, B // 4))
        item[:, : B // 4] = rng.integers(0, hot_users, size=(T, B // 4))
    label = (rng.random((T, B)) < 0.3).astype(np.float32)
    return user.astype(np.int64), item.astype(np.int64), label


THIN_BLOCK = 16


def thin_outputs(data, L, seed):
    """Keeps a fixture with a wide tower under 1 MB: of each tower weight matrix in the output groups
    (grad0, after1, final) one row per block of THIN_BLOCK rows is kept, at a seeded offset inside the
    block, and the others are stored as NaN (tests/util.py:group masks them out of the comparisons).
    The inputs stay whole; after2, which no test reads, is dropped."""
    rng = np.random.default_rng(seed)
    for k in range(L):
        key = f"MLP_layers.{3 * k + 1}.weight"
        rows = data[f"init/{key}"].shape[0]
        keep = np.arange(0, rows, THIN_BLOCK) + rng.integers(0, THIN_BLOCK, -(-rows // THIN_BLOCK))
        drop = np.ones(rows, dtype=bool)
        drop[keep[keep < rows]] = False
        for prefix in ("grad0", "after1", "final"):
            a = data[f"{prefix}/{key}"].copy()
            a[drop] = np.nan
            data[f"{prefix}/{key}"] = a
    for k in [k for k in data if k.startswith("after2/")]:
        del data[k]


def train_case(NCF, name, model_type, U, I, f, L, B, T, optimizer, lr, seed, short_last=0, thin=False):
    torch.manual_seed(seed)
    rng = np.random.default_rng(seed)
    model = NCF(U, I, f, L, 0.0, model_type)
    data = sd_np(model, "init")
    user, item, label = make_batches(rng, U, I, B, T, hot_users=max(2, U // 10))
    data.update(user=user, item=item, label=label)
    crit = torch.nn.BCEWithLogitsLoss()
    opt = (torch.optim.Adam(model.parameters(), lr=lr) if optimizer == "adam"
           else torch.optim.SGD(model.parameters(), lr=lr))
    losses = []
    for t in range(T):
        n = B - short_last if (short_last and t == T - 1) else B  # drop_last=False tail batch
        u, i, y = (torch.from_numpy(a[t, :n]) for a in (user, item, label))
        opt.zero_grad()
        pred = model(u, i)
        loss = crit(pred, y)
        loss.backward()
        if t == 0:
            data["logits0"] = pred.detach().numpy().copy()
            data.update(grads_np(model, "grad0"))
        opt.step()
        losses.append(loss.item())
        if t == 0:
            data.update(sd_np(model, "after1"))
        if t == 1:
            data.update(sd_np(model, "after2"))
    data.update(sd_np(model, "final"))
    data["loss"] = np.array(losses, dtype=np.float64)
    if thin:
        thin_outputs(data, L, seed)
    meta = dict(model_type=model_type, U=U, I=I, f=f, L=L, B=B, T=T, optimizer=optimizer, lr=lr,
                short_last=short_last, torch=torch.__version__)
    np.savez_compressed(OUT / f"{name}.npz", meta=json.dumps(meta), **data)
    print(name, "loss", losses[0], "->", losses[-1])


def kd_case(NCF, ResponseDistillation, name, seed):
    torch.manual_seed(seed)
    rng = np.random.default_rng(seed)
    U, I, B, T = 48, 36, 40, 5
    tf, tL, sf, sL = 16, 3, 8, 2  # reference rule: teacher = (2f, L+1) of the student (train_student.py:86)
    teacher = NCF(U, I, tf, tL, 0.0, "NeuMF-end")
    student = NCF(U, I, sf, sL, 0.0, "NeuMF-end")
    # make the teacher non-trivial: larger embeddings so its logits are not ~0
    with torch.no_grad():
        for k, p in teacher.named_parameters():
            if k.startswith("embed_"):
                p.mul_(30.0)
    data = {}
    data.update(sd_np(teacher, "teacher"))
    data.update(sd_np(student, "init"))
    user, item, label = make_batches(rng, U, I, B, T, hot_users=5)
    data.update(user=user, item=item, label=label)
    alpha = 0.5
    dist = ResponseDistillation(teacher, student, temperature=2.0, alpha=alpha)
    opt = torch.optim.Adam(student.parameters(), lr=1e-3)
    losses = []
    for t in range(T):
        dist.train()
        u, i, y = (torch.from_numpy(a[t]) for a in (user, item, label))
        opt.zero_grad()
        loss = dist(u, i, y)
        loss.backward()
        if t == 0:
            data.update(grads_np(student, "grad0"))
            with torch.no_grad():
                data["teacher_logits0"] = teacher(u, i).numpy().copy()
                data["student_logits0"] = student(u, i).numpy().copy()
        opt.step()
        losses.append(loss.item())
    data.update(sd_np(student, "final"))
    data["loss"] = np.array(losses, dtype=np.float64)
    meta = dict(U=U, I=I, B=B, T=T, teacher=dict(f=tf, L=tL), student=dict(f=sf, L=sL), alpha=alpha,
                lr=1e-3, model_type="NeuMF-end", torch=torch.__version__)
    np.savez_compressed(OUT / f"{name}.npz", meta=json.dumps(meta), **data)
    print(name, "loss", losses[0], "->", losses[-1])


def pretrain_case(NCF, name, seed):
    """NeuMF-pre: load_pretrain_weights from a GMF and an MLP state dict, then SGD(lr*10)
    (reference scripts/train_neumf.py:62-70,87-88; models.py:48-95)."""
    torch.manual_seed(seed)
    rng = np.random.default_rng(seed)
    U, I, f, L, B, T = 40, 30, 8, 3, 32, 4
    gmf = NCF(U, I, f, L, 0.0, "GMF")
    mlp = NCF(U, I, f, L, 0.0, "MLP")
    model = NCF(U, I, f, L, 0.0, "NeuMF-pre")
    data = {}
    data.update(sd_np(gmf, "gmf"))
    data.update(sd_np(mlp, "mlp"))
    torch.manual_seed(seed + 1)  # the predict layer is re-drawn inside load_pretrain_weights
    model.load_pretrain_weights(gmf.state_dict(), mlp.state_dict())
    data.update(sd_np(model, "init"))
    user, item, label = make_batches(rng, U, I, B, T, hot_users=4)
    data.update(user=user, item=item, label=label)
    crit = torch.nn.BCEWithLogitsLoss()
    opt = torch.optim.SGD(model.parameters(), lr=0.01)
    losses = []
    for t in range(T):
        u, i, y = (torch.from_numpy(a[t]) for a in (user, item, label))
        opt.zero_grad()
        loss = crit(model(u, i), y)
        loss.backward()
        opt.step()
        losses.append(loss.item())
    data.update(sd_np(model, "final"))
    data["loss"] = np.array(losses, dtype=np.float64)
    meta = dict(U=U, I=I, f=f, L=L, B=B, T=T, lr=0.01, optimizer="sgd", model_type="NeuMF-pre",
                reseed=seed + 1, torch=torch.__version__)
    np.savez_compressed(OUT / f"{name}.npz", meta=json.dumps(meta), **data)
    print(name, "loss", losses)


def metrics_case(NCF, metrics, NCFData, name, model_type, f, L, seed):
    """metrics() over a small leave-one-out test set (reference src/training/metrics.py:4-25 via
    DataLoader(batch_size=100, shuffle=False), scripts/train_neumf.py:56,125)."""
    torch.manual_seed(seed)
    rng = np.random.default_rng(seed)
    U, I, n, C, k = 64, 400, 64, 100, 10
    model = NCF(U, I, f, L, 0.0, model_type)
    with torch.no_grad():
        for pname, p in model.named_parameters():
            if pname.startswith("embed_"):
                p.mul_(60.0)  # spread the scores so that near-ties are rare
    users = np.arange(n, dtype=np.int64)
    cands = np.stack([rng.choice(I, size=C, replace=False) for _ in range(n)]).astype(np.int64)
    test_data = [[int(u), int(c)] for u, row in zip(users, cands) for c in row]
    ds = NCFData(test_data, I, None, 0, False)
    loader = torch.utils.data.DataLoader(ds, batch_size=C, shuffle=False, num_workers=0)
    model.eval()
    with torch.no_grad():
        HR, NDCG = metrics(model, loader, k)
        scores = model(torch.from_numpy(np.repeat(users, C)), torch.from_numpy(cands.reshape(-1)))
    scores = scores.numpy().reshape(n, C)
    # tie-freeness margin of the reference scores (so rankings are well defined, SURVEY.md §0.6)
    srt = -np.sort(-scores, axis=1)
    gap = np.min(srt[:, :-1] - srt[:, 1:])
    data = sd_np(model, "init")
    data.update(users=users, cands=cands, HR=np.array(HR, dtype=np.int64),
                NDCG=np.array(NDCG, dtype=np.float64), scores=scores)
    meta = dict(model_type=model_type, U=U, I=I, f=f, L=L, n=n, C=C, k=k, min_gap=float(gap),
                torch=torch.__version__)
    np.savez_compressed(OUT / f"{name}.npz", meta=json.dumps(meta), **data)
    print(name, "HR", np.mean(HR), "NDCG", np.mean(NDCG), "min gap", gap)


def init_case(NCF, name):
    """Same seed => same initial weights as the reference (models.py:38-46)."""
    torch.manual_seed(2025)
    model = NCF(37, 29, 8, 3, 0.0, "NeuMF-end")
    data = sd_np(model, "init")
    meta = dict(seed=2025, U=37, I=29, f=8, L=3, model_type="NeuMF-end", torch=torch.__version__)
    np.savez_compressed(OUT / f"{name}.npz", meta=json.dumps(meta), **data)


def sampler_stats_case(NCFData, name):
    """Distribution of the reference ng_sample (datasets.py:53-69) on a tiny problem: per-user
    histogram of drawn items, for a statistical comparison with the Philox sampler."""
    import scipy.sparse as sp
    rng = np.random.default_rng(7)
    U, I, num_ng = 6, 12, 4
    pairs = sorted({(int(u), int(i)) for u, i in zip(rng.integers(0, U, 30), rng.integers(0, I, 30))})
    mat = sp.dok_matrix((U, I), dtype=np.float32)
    for u, i in pairs:
        mat[u, i] = 1.0
    ds = NCFData([list(p) for p in pairs], I, mat, num_ng, True)
    np.random.seed(11)
    hist = np.zeros((U, I), dtype=np.int64)
    reps = 400
    for _ in range(reps):
        ds.ng_sample()
        for u, j in ds.features_ng:
            hist[u, j] += 1
    labels = np.array(ds.labels_fill)
    feats = np.array(ds.features_fill)
    meta = dict(U=U, I=I, num_ng=num_ng, reps=reps)
    np.savez_compressed(OUT / f"{name}.npz", meta=json.dumps(meta), pairs=np.array(pairs, dtype=np.int64),
                        hist=hist, last_labels=labels, last_features=feats)
    print(name, "collisions", int(sum(hist[u, i] for u, i in pairs)))


# Tower shapes the tcgen05 path accepts beyond the ones above (tests: the opt-in shape sweep)
SWEEP_CASES = [
    ("train_neumf_f32_l1", "NeuMF-end", 40, 30, 32, 1, 48, 3, "adam", 1e-3, 21),
    ("train_mlp_f32_l3", "MLP", 30, 24, 32, 3, 40, 3, "adam", 1e-3, 22),
    ("train_neumf_f64_l1", "NeuMF-end", 24, 18, 64, 1, 40, 3, "adam", 1e-3, 23),
    ("train_neumf_f64_l2", "NeuMF-end", 24, 18, 64, 2, 40, 3, "adam", 1e-3, 24),
]


def main():
    OUT.mkdir(parents=True, exist_ok=True)
    NCF, metrics, ResponseDistillation, NCFData = import_reference()
    torch.set_num_threads(1)
    for case in SWEEP_CASES:
        train_case(NCF, *case)
    if "--sweep-only" in sys.argv:  # leave the other fixtures untouched
        return
    train_case(NCF, "train_gmf_f8", "GMF", 60, 40, 8, 3, 32, 8, "adam", 1e-3, 1)
    train_case(NCF, "train_mlp_f8_l3", "MLP", 60, 40, 8, 3, 32, 8, "adam", 1e-3, 2)
    train_case(NCF, "train_neumf_f8_l3", "NeuMF-end", 60, 40, 8, 3, 32, 8, "adam", 1e-3, 3, short_last=5)
    train_case(NCF, "train_neumf_f32_l2", "NeuMF-end", 50, 30, 32, 2, 48, 6, "adam", 1e-3, 4)
    train_case(NCF, "train_neumf_f6_l2", "NeuMF-end", 33, 21, 6, 2, 20, 6, "adam", 1e-3, 5)
    train_case(NCF, "train_neumf_f5_l1", "NeuMF-end", 33, 21, 5, 1, 20, 5, "adam", 2e-3, 6)
    train_case(NCF, "train_neumf_f64_l3", "NeuMF-end", 24, 18, 64, 3, 40, 3, "adam", 1e-3, 7, thin=True)
    train_case(NCF, "train_neumf_f8_l3_sgd", "NeuMF-end", 60, 40, 8, 3, 32, 5, "sgd", 0.01, 8)
    kd_case(NCF, ResponseDistillation, "kd_response", 9)
    pretrain_case(NCF, "neumf_pre_sgd", 10)
    metrics_case(NCF, metrics, NCFData, "metrics_neumf_f8_l3", "NeuMF-end", 8, 3, 11)
    metrics_case(NCF, metrics, NCFData, "metrics_gmf_f8", "GMF", 8, 3, 12)
    init_case(NCF, "init_seed2025")
    sampler_stats_case(NCFData, "sampler_stats")


if __name__ == "__main__":
    main()
