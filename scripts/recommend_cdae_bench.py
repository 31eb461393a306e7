"""CDAE top-K recommendation at Yelp2018 shape: CDAERecommender (list encoder + biased retrieval kernel) against the ways to
get the same ranking without it.

Workload: syn.make_interactions() (31,668 users x 38,048 items), the seen lists of the train split, a CDAETrainer with the
given hidden size (freshly initialised: the timings do not depend on the parameter values), a seeded batch of user ids.

Arms per configuration (h, B, K):
  recommender  trainer.recommender(seen).recommend(uid, k)
  dense        what a caller does today: the dense multi-hot x on the device, model.eval()(uid, x) (the dense prediction),
               pred * (1 - x) as cdae_trainer.py masks, torch.topk
  augmented    the evaluation's workaround for the output bias: z = [z | 1 | 0...] from the dense x (yr_cdae_hidden_ex),
               [W_o | b_o | 0...] copied, the unbiased ops.recommend_topk with per-row seen lists; not available when
               h + 1 rounds past 1024 (h = 1024)
The median and min of CUDA-event timings and the peak memory above the baseline per call, as scripts/recommend_bench.py.
id_agreement: the share of ids equal to the recommender arm's; max_score_diff: the largest difference of the returned scores
(dense: sigmoid of the recommender's logits against the predictions). One JSON line per configuration, the GPU's name and
power limit first.

    python scripts/recommend_cdae_bench.py [--hs 64,256,1024] [--batches 256,4096] [--ks 20,100] [--out file.jsonl]
"""
import argparse
import json
import os
import sys
import tempfile
from types import SimpleNamespace

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from recommend_bench import gpu_info, measure  # noqa: E402


def multi_hot(ptr, idx, uid, nI):
    """Dense [B x nI] fp32 multi-hot of the users' seen lists, built on the device."""
    p = ptr.to(torch.int64)
    start, cnt = p[uid], p[uid + 1] - p[uid]
    row = torch.repeat_interleave(torch.arange(uid.numel(), device=uid.device), cnt)
    first = torch.repeat_interleave(torch.cumsum(cnt, 0) - cnt, cnt)
    pos = torch.arange(row.numel(), device=uid.device) - first + torch.repeat_interleave(start, cnt)
    x = torch.zeros(uid.numel(), nI, device=uid.device)
    x[row, idx[pos].to(torch.int64)] = 1.0
    return x, row, idx[pos]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--hs", default="64,256,1024")
    ap.add_argument("--batches", default="256,4096")
    ap.add_argument("--ks", default="20,100")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("recommend_cdae_bench.py measures on a CUDA device; none is visible")

    from yelprecommendation_b200 import ops
    from yelprecommendation_b200.data import synthetic as syn
    from yelprecommendation_b200.retrieval import SeenItems
    from yelprecommendation_b200.trainers import CDAETrainer

    dev = torch.device("cuda", 0)
    inter = syn.make_interactions()                      # Yelp2018 shape: 31,668 users x 38,048 items
    split = syn.split_per_user(inter, seed=42)
    seen = SeenItems.from_split(split, inter.num_items)
    nU, nI = inter.num_users, inter.num_items
    ptr, idx = seen.on(dev)
    rng = np.random.default_rng(0)
    head = dict(gpu_info(), users=nU, items=nI, seen_nnz=int(seen.idx.numel()), warmup=args.warmup, iters=args.iters)
    lines = [head]
    print(json.dumps(head), flush=True)
    for h in (int(x) for x in args.hs.split(",")):
        torch.manual_seed(h)
        cfg = SimpleNamespace(device="cuda", model_dir=tempfile.mkdtemp(), hidden_size=h, corruption_level=0.0,
                              hidden_activation="sigmoid", output_activation="sigmoid", optimizer="adam", lr=1e-3,
                              weight_decay=0.0, top_n=20, wandb=False, epochs=1, patience=1, best_metric="loss",
                              negative_sampling=True, loss_name="bce", batch_size=256)
        tr = CDAETrainer(cfg, nI, nU)
        model = tr.model.eval()
        rec = tr.recommender(seen)
        ldz = (h + 1 + 7) // 8 * 8
        for B in (int(x) for x in args.batches.split(",")):
            uid = torch.from_numpy(rng.integers(0, nU, size=B)).to(dev)
            for k in (int(x) for x in args.ks.split(",")):
                def recommender():
                    return rec.recommend(uid, k)

                def dense():
                    x, _, _ = multi_hot(ptr, idx, uid, nI)
                    pred = model(uid, x) * (1 - x)
                    sc, ids = torch.topk(pred, k, dim=1)
                    return ids, sc

                def augmented():
                    x, row, item = multi_hot(ptr, idx, uid, nI)
                    z = model.hidden(uid, x, ldz=ldz)
                    Va = torch.zeros(nI, ldz, device=dev)
                    Va[:, :h] = model.output_layer.weight.data
                    Va[:, h] = model.output_layer.bias.data
                    bptr = torch.zeros(B + 1, dtype=torch.int64, device=dev)
                    bptr[1:] = torch.cumsum(torch.bincount(row, minlength=B), 0)
                    return ops.recommend_topk(z, Va, torch.arange(B, device=dev), k, bptr.to(torch.int32),
                                              item.to(torch.int32))

                ai, asc = recommender()
                di, dsc = dense()
                t_a, t_a_min, m_a = measure(recommender, args.warmup, args.iters)
                t_d, t_d_min, m_d = measure(dense, args.warmup, args.iters)
                line = dict(h=h, batch=B, k=k, recommender_ms=round(t_a, 4), recommender_min_ms=round(t_a_min, 4),
                            recommender_peak_mb=round(m_a / 2 ** 20, 2),
                            dense_ms=round(t_d, 4), dense_min_ms=round(t_d_min, 4), dense_peak_mb=round(m_d / 2 ** 20, 2),
                            dense_id_agreement=float((di == ai).float().mean().item()),
                            dense_max_score_diff=float((dsc - torch.sigmoid(asc)).abs().max().item()),
                            vs_dense=round(t_d / t_a, 3))
                if ldz <= ops.RECOMMEND_MAX_D:
                    xi, xsc = augmented()
                    t_x, t_x_min, m_x = measure(augmented, args.warmup, args.iters)
                    line.update(augmented_ms=round(t_x, 4), augmented_min_ms=round(t_x_min, 4),
                                augmented_peak_mb=round(m_x / 2 ** 20, 2),
                                augmented_id_agreement=float((xi == ai).float().mean().item()),
                                augmented_max_score_diff=float((xsc - asc).abs().max().item()),
                                vs_augmented=round(t_x / t_a, 3))
                    del xi, xsc
                else:
                    line.update(augmented_ms=None, augmented_note=f"[z|1] is {ldz} wide, above {ops.RECOMMEND_MAX_D}")
                lines.append(line)
                print(json.dumps(line), flush=True)
                del ai, asc, di, dsc
                torch.cuda.empty_cache()
        del tr, model, rec
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()
