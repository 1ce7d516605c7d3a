#!/usr/bin/env python3
"""Top-K recommendations over the whole catalog from a trained checkpoint, and the full-ranking HR@K /
NDCG@K of the held-out items.

Loads a state_dict written by the training scripts (--model/--factor_num/--num_layers as in
train_neumf.py), leaves out each user's training items, writes one line per user to --out:

    user<TAB>item1<TAB>...<TAB>itemK          (best first; -1 pads a user with fewer than K unseen items)

and prints a --- RESULTS --- block.  The held-out item of a test user is column 0 of its test candidates;
its full rank is taken against every item the user has not trained on.

    python scripts/recommend.py --checkpoint results/models/NeuMF_end_3l_8f_best.pth --out recs.tsv
    python scripts/recommend.py --synthetic ml1m --checkpoint ckpt.pth --out recs.tsv --top_k 20
"""
import argparse
import os
import sys

import torch

sys.path.append(os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))

from ncf_b200 import ops
from ncf_b200.config import config
from ncf_b200.metrics import evaluate_full_ranking
from ncf_b200.models import NCF
from ncf_b200.recommend import recommend
from ncf_b200.train_loop import load_dataset


def run(args, device):
    train, test_users, test_cands, user_num, item_num, _ = load_dataset(device, args.synthetic)
    model = NCF(user_num, item_num, args.factor_num, args.num_layers, 0.0, args.model)
    model.load_state_dict(torch.load(args.checkpoint, map_location="cpu"))
    model.to(device).eval()
    exclude = ops.csr_build(train[:, 0].contiguous(), train[:, 1].contiguous(), user_num)
    users = torch.arange(user_num, dtype=torch.int64, device=device)
    items, _ = recommend(model, users, args.top_k, exclude, args.chunk_users)
    with open(args.out, "w") as f:
        for u, row in zip(range(user_num), items.cpu().numpy()):
            f.write(str(u) + "\t" + "\t".join(map(str, row.tolist())) + "\n")
    _, hr, ndcg = evaluate_full_ranking(model, test_users, test_cands[:, 0].contiguous(), exclude, ks=(args.top_k,))
    print("\n--- RESULTS ---")
    print(f"Model: {args.model}")
    print(f"Users: {user_num}")
    print(f"Items: {item_num}")
    print(f"HR@{args.top_k}: {hr[args.top_k]}")
    print(f"NDCG@{args.top_k}: {ndcg[args.top_k]}")
    print("--- END RESULTS ---")
    return {"users": user_num, "items": item_num, "hr": hr[args.top_k], "ndcg": ndcg[args.top_k]}


def main(argv=None):
    p = argparse.ArgumentParser(description="Full-catalog top-K recommendation")
    p.add_argument("--checkpoint", type=str, required=True, help="state_dict written by a training script")
    p.add_argument("--model", type=str, default="NeuMF-end", choices=["GMF", "MLP", "NeuMF-end", "NeuMF-pre"])
    p.add_argument("--factor_num", type=int, default=config.factor_num)
    p.add_argument("--num_layers", type=int, default=config.num_layers)
    p.add_argument("--top_k", type=int, default=config.top_k)
    p.add_argument("--out", type=str, required=True, help="TSV file: user, then its top_k items")
    p.add_argument("--chunk_users", type=int, default=None, help="users per forward (default: 1 GiB workspace)")
    p.add_argument("--synthetic", type=str, default=None, help="synthetic shape (tiny|ml100k|ml1m|ml20m) instead of data files")
    p.add_argument("--gpu", type=str, default="0")
    args = p.parse_args(argv)
    os.environ.setdefault("CUDA_VISIBLE_DEVICES", args.gpu)
    if not torch.cuda.is_available():
        raise SystemExit("ncf_b200 needs a CUDA device: there is no CPU fallback")
    return run(args, torch.device("cuda"))


if __name__ == "__main__":
    main()
