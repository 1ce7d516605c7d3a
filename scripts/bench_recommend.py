#!/usr/bin/env python3
"""Benchmark of full-catalog top-K recommendation (ncf_recommend): one JSON line per workload.

    python scripts/bench_recommend.py [--workloads ml1m_f8,ml1m_f32,ml20m_f32] [--repeats 3] [--k 10]

Every workload scores all users of a synthetic MovieLens shape against every item with a NeuMF model
(seeded random weights: the work does not depend on training), leaves out each user's synthetic training
pairs and keeps the 10 best items per user:
  ml1m_f8    6 040 x 3 706,    NeuMF f=8  L=3 (thread-per-sample forward kernel)
  ml1m_f32   6 040 x 3 706,    NeuMF f=32 L=3 (tcgen05 forward kernel)
  ml20m_f32  138 493 x 26 744, NeuMF f=32 L=3 (3.7 G scored pairs)

Each line reports
  e2e_ms          one ncf_recommend call over all users (CUDA events; median/min/max of --repeats runs after
                  a warm-up run), users/s and scored pairs/s from the median;
  stages_ms       in a separate run, the three stages chunk by chunk through their public entry points with
                  CUDA events around each: scoring (ops.forward on the chunk's pair list), masking
                  (ops.mask_items), selection (ops.topk_rows);
  select_GBps     score bytes the selection kernel reads (4 reads of every score) / its time;
  torch           the same-GPU composition: ops.forward on the pair list + masked_fill + torch.topk, same
                  model, data and chunks, and its agreement with ours (items equal except where adjacent
                  scores lie within 1e-5 * max|score|; largest score difference);
  gpu, power_limit_w  read (never set) in the same process.
Chunks: the default of ncf_b200.recommend (workspace <= 1 GiB).  Nothing is written to the repository.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))

from ncf_b200 import ops
from ncf_b200.models import NCF
from ncf_b200.recommend import default_chunk_users
from ncf_b200.synth import make_interactions

WORKLOADS = {"ml1m_f8": ("ml1m", 8, 3), "ml1m_f32": ("ml1m", 32, 3), "ml20m_f32": ("ml20m", 32, 3)}


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits",
                              "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        name, power = [x.strip() for x in out.stdout.strip().splitlines()[0].split(",")]
        return name, float(power)
    except Exception:
        return torch.cuda.get_device_name(), None


def spread(ms):
    s = sorted(ms)
    return {"median": s[len(s) // 2], "min": s[0], "max": s[-1], "runs": [round(x, 3) for x in ms]}


class Timer:
    def __init__(self):
        self.total = 0.0

    def __enter__(self):
        self.a, self.b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        self.a.record()
        return self

    def __exit__(self, *exc):
        self.b.record()
        self.b.synchronize()
        self.total += self.a.elapsed_time(self.b)


def chunk_pairs(users, I):
    return users.repeat_interleave(I), torch.arange(I, device=users.device).repeat(users.numel())


def stages(m, users, I, k, chunk, rowptr, col):
    t_score, t_mask, t_sel = Timer(), Timer(), Timer()
    fws = torch.empty(ops.forward_workspace_bytes(m, chunk * I), dtype=torch.uint8, device=users.device)
    for lo in range(0, users.numel(), chunk):
        u = users[lo:lo + chunk]
        pu, pi = chunk_pairs(u, I)
        scores = torch.empty(u.numel(), I, dtype=torch.float32, device=users.device)
        with t_score:
            ops.forward(m, pu, pi, out=scores.view(-1), workspace=fws)
        with t_mask:
            ops.mask_items(scores, u, rowptr, col)
        with t_sel:
            ops.topk_rows(scores, k)
    return t_score.total, t_mask.total, t_sel.total


def torch_composition(m, users, I, k, chunk, rowptr, col):
    """ops.forward on the pair list + masked_fill(-inf) + torch.topk, chunk by chunk (the workaround the
    project offered before ncf_recommend).  -> (items, scores)"""
    items, top = [], []
    for lo in range(0, users.numel(), chunk):
        u = users[lo:lo + chunk]
        pu, pi = chunk_pairs(u, I)
        scores = ops.forward(m, pu, pi).view(u.numel(), I)
        beg, end = rowptr[u], rowptr[u + 1]
        cnt = end - beg
        rows = torch.arange(u.numel(), device=u.device).repeat_interleave(cnt)
        pos = torch.arange(int(cnt.sum()), device=u.device) - (cnt.cumsum(0) - cnt).repeat_interleave(cnt)
        cols = col[(beg.repeat_interleave(cnt) + pos)].long()
        mask = torch.zeros(u.numel(), I, dtype=torch.bool, device=u.device)
        mask[rows, cols] = True
        v, i = torch.topk(scores.masked_fill_(mask, float("-inf")), k + 1, dim=1)
        items.append(i)
        top.append(v)
    return torch.cat(items), torch.cat(top)


def agreement(ours_items, ours_scores, t_items, t_scores, k):
    tol = 1e-5 * float(t_scores[:, :k].abs().max())
    diff = ours_items != t_items[:, :k]
    gap = (t_scores[:, 1:] - t_scores[:, :-1]).abs() <= tol          # [n, k]: positions j, j+1 within tol
    near = torch.zeros_like(diff)
    near[:, 1:] |= gap[:, :k - 1]
    near |= gap[:, :k]
    ok = (~diff | near).all(dim=1)
    return {"rows_equal_tie_aware": float(ok.float().mean()),
            "rows_identical": float((~diff).all(dim=1).float().mean()),
            "max_abs_score_diff": float((ours_scores - t_scores[:, :k]).abs().max()), "tolerance": tol}


def run(name, k, repeats):
    shape, f, L = WORKLOADS[name]
    dev = torch.device("cuda")
    d = make_interactions(shape, device=dev)
    U, I = d.user_num, d.item_num
    torch.manual_seed(0)
    model = NCF(U, I, f, L, 0.0, "NeuMF-end").to(dev).eval()
    m = model.abi_struct()
    rowptr, col = ops.csr_build(d.pos_user, d.pos_item, U)
    users = torch.arange(U, device=dev)
    chunk = default_chunk_users(m, U, k)
    ws = torch.empty(ops.recommend_workspace_bytes(m, chunk, k), dtype=torch.uint8, device=dev)

    ops.recommend(m, users, k, chunk, rowptr, col, workspace=ws)              # warm-up
    e2e = []
    for _ in range(repeats):
        with Timer() as t:
            items, scores, _ = ops.recommend(m, users, k, chunk, rowptr, col, workspace=ws)
        e2e.append(t.total)
    stages(m, users, I, k, chunk, rowptr, col)                                # warm-up
    st = [stages(m, users, I, k, chunk, rowptr, col) for _ in range(repeats)]
    with torch.no_grad():
        torch_composition(m, users, I, k, chunk, rowptr, col)                # warm-up
        tt = []
        for _ in range(repeats):
            with Timer() as t:
                t_items, t_scores = torch_composition(m, users, I, k, chunk, rowptr, col)
            tt.append(t.total)
    pairs = U * I
    med = spread(e2e)["median"]
    score_ms, mask_ms, sel_ms = (spread([s[j] for s in st]) for j in range(3))
    name_gpu, power = gpu_info()
    return {
        "workload": name, "users": U, "items": I, "factor_num": f, "num_layers": L, "k": k,
        "excluded_pairs": int(d.pos_user.numel()), "chunk_users": chunk, "workspace_bytes": ws.numel(),
        "e2e_ms": spread(e2e), "users_per_s": U / med * 1e3, "pairs_per_s": pairs / med * 1e3,
        "stages_ms": {"score": score_ms, "mask": mask_ms, "select": sel_ms},
        "mask_plus_select_over_score": (mask_ms["median"] + sel_ms["median"]) / score_ms["median"],
        "select_bytes_read": 4 * 4 * pairs, "select_GBps": 4 * 4 * pairs / sel_ms["median"] / 1e6,
        "torch": {"ms": spread(tt), "ours_speedup": spread(tt)["median"] / med,
                  "agreement": agreement(items, scores, t_items, t_scores, k)},
        "gpu": name_gpu, "power_limit_w": power, "repeats": repeats,
    }


def main(argv=None):
    p = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    p.add_argument("--workloads", default=",".join(WORKLOADS))
    p.add_argument("--repeats", type=int, default=3)
    p.add_argument("--k", type=int, default=10)
    args = p.parse_args(argv)
    if not torch.cuda.is_available():
        raise SystemExit("bench_recommend needs a CUDA device")
    for name in args.workloads.split(","):
        print(json.dumps(run(name, args.k, max(1, args.repeats))), flush=True)


if __name__ == "__main__":
    main()
