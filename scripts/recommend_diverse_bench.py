"""Diverse retrieval at Yelp2018 shape: Maximal Marginal Relevance re-ranking of a top-N pool, the kernel
(ops.recommend_mmr, yr_recommend_mmr) against the plain PyTorch way to do it, on tables with visible taste clusters.

Tables: 16 cluster centres (unit Gaussian / sqrt(d)); every item is a centre plus noise of half its scale, every user
c1 + 0.8 c2 + 0.6 c3 of three random centres plus the same noise, so a user's best items come from three tastes and the
top of a plain top-k list is crowded with the strongest one, as on the synthetic interactions (n_clusters = 16). Seen items:
SeenItems.from_split of the synthetic Yelp2018 split (31,668 users x 38,048 items).

Arms per configuration (d, B, k, N), lam = 0.5:
  pool     rec.recommend(user_ids, N)                        the pool the re-ranking starts from
  mmr      ops.recommend_mmr(item_emb, pool ids, pool scores, k, lam)
  diverse  rec.recommend_diverse(user_ids, k, lam, pool=N)   the whole call: pool + mmr
  torch    gather the pool rows [B x N x d], normalise, bmm Gram [B x N x N], k steps of elementwise ops + argmax
The median of CUDA-event timings and the peak memory per call, as scripts/recommend_bench.py. torch_id_agreement: the
share of ids the torch arm returns in the mmr arm's place (fp32 rounding of its Gram can flip near-ties). lam1_equal:
recommend_diverse with lam = 1 equals recommend(user_ids, k) bit for bit. Diversity of the returned lists, lam = 1 against
lam = 0.5: mean pairwise cosine of the items of a list (in item_emb) and mean number of distinct clusters. One JSON line
per configuration, the GPU's name and power limit first.

    python scripts/recommend_diverse_bench.py [--ds 64,256] [--batches 256,4096] [--pools 20:200,50:500] [--out f.jsonl]
"""
import argparse
import json
import os
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from recommend_bench import gpu_info, measure  # noqa: E402

N_CLUSTERS = 16


def torch_mmr(V, pool_ids, pool_scores, k, a, c):
    """What the re-ranking costs without the kernel: dense per-row Gram matrix and k launches of elementwise ops."""
    B, N = pool_ids.shape
    valid = pool_ids >= 0
    X = V[pool_ids.clamp(min=0)] * valid[..., None]
    X = X * torch.nan_to_num(X.norm(dim=-1, keepdim=True).reciprocal(), posinf=0.0)
    S = torch.bmm(X, X.transpose(1, 2))
    ar = a * pool_scores
    pen = torch.zeros(B, N, device=V.device)
    avail = valid.clone()
    rows = torch.arange(B, device=V.device)
    out_ids = torch.full((B, k), -1, dtype=torch.int64, device=V.device)
    out_sc = torch.full((B, k), float("-inf"), device=V.device)
    for t in range(k):
        m = (ar - c * pen).masked_fill(~avail, float("-inf"))
        s = m.argmax(1)
        has = avail[rows, s]
        out_ids[:, t] = torch.where(has, pool_ids[rows, s], -1)
        out_sc[:, t] = torch.where(has, pool_scores[rows, s], float("-inf"))
        avail[rows, s] = False
        pen = S[rows, :, s] if t == 0 else torch.maximum(pen, S[rows, :, s])
    return out_ids, out_sc


def diversity(V, cluster, ids):
    """(mean pairwise cosine within a list, mean number of distinct clusters in a list) over rows."""
    X = torch.nn.functional.normalize(V[ids.clamp(min=0)], dim=-1)
    k = ids.shape[1]
    G = torch.bmm(X, X.transpose(1, 2))
    cos = ((G.sum((1, 2)) - G.diagonal(dim1=1, dim2=2).sum(1)) / (k * (k - 1))).mean().item()
    cl = cluster[ids.clamp(min=0)]
    distinct = torch.zeros(cl.shape[0], N_CLUSTERS, device=ids.device).scatter_(1, cl, 1.0).sum(1).mean().item()
    return round(cos, 4), round(distinct, 3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ds", default="64,256")
    ap.add_argument("--batches", default="256,4096")
    ap.add_argument("--pools", default="20:200,50:500")
    ap.add_argument("--lam", type=float, default=0.5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("recommend_diverse_bench.py measures on a CUDA device; none is visible")

    from yelprecommendation_b200 import ops
    from yelprecommendation_b200.data import synthetic as syn
    from yelprecommendation_b200.retrieval import Recommender, SeenItems

    dev = torch.device("cuda", 0)
    inter = syn.make_interactions()                      # Yelp2018 shape: 31,668 users x 38,048 items
    split = syn.split_per_user(inter, seed=42)
    seen = SeenItems.from_split(split, inter.num_items)
    nU, nI = inter.num_users, inter.num_items
    head = dict(gpu_info(), users=nU, items=nI, seen_nnz=int(seen.idx.numel()), clusters=N_CLUSTERS, lam=args.lam,
                warmup=args.warmup, iters=args.iters)
    lines = [head]
    print(json.dumps(head), flush=True)
    rng = np.random.default_rng(0)
    a, c = ops.mmr_weights(args.lam)
    for d in (int(x) for x in args.ds.split(",")):
        g = torch.Generator(device=dev).manual_seed(d)
        C = torch.randn(N_CLUSTERS, d, device=dev, generator=g) * d ** -0.5
        icl = torch.randint(0, N_CLUSTERS, (nI,), device=dev, generator=g)
        V = C[icl] + 0.5 * torch.randn(nI, d, device=dev, generator=g) * d ** -0.5
        ucl = torch.randint(0, N_CLUSTERS, (nU, 3), device=dev, generator=g)
        U = C[ucl[:, 0]] + 0.8 * C[ucl[:, 1]] + 0.6 * C[ucl[:, 2]] + \
            0.5 * torch.randn(nU, d, device=dev, generator=g) * d ** -0.5
        rec = Recommender(U, V, seen)
        for B in (int(x) for x in args.batches.split(",")):
            uid = torch.from_numpy(rng.integers(0, nU, size=B)).to(dev)
            for kn in args.pools.split(","):
                k, N = (int(x) for x in kn.split(":"))
                pids, psc = rec.recommend(uid, N)
                pool = lambda: rec.recommend(uid, N)
                mmr = lambda: ops.recommend_mmr(V, pids, psc, k, args.lam)
                diverse = lambda: rec.recommend_diverse(uid, k, lam=args.lam, pool=N)
                tarm = lambda: torch_mmr(V, pids, psc, k, a, c)
                mi, ms = mmr()
                ti, ts = tarm()
                di, ds = diverse()
                l1i, l1s = rec.recommend_diverse(uid, k, lam=1.0, pool=N)
                ki, ks = rec.recommend(uid, k)
                tp, tp_min, mp = measure(pool, args.warmup, args.iters)
                tm, tm_min, mm = measure(mmr, args.warmup, args.iters)
                td, td_min, md = measure(diverse, args.warmup, args.iters)
                tt, tt_min, mt = measure(tarm, args.warmup, args.iters)
                cos1, cl1 = diversity(V, icl, l1i)
                cos5, cl5 = diversity(V, icl, mi)
                line = dict(d=d, batch=B, k=k, pool=N,
                            pool_ms=round(tp, 4), mmr_ms=round(tm, 4), mmr_min_ms=round(tm_min, 4),
                            diverse_ms=round(td, 4), torch_ms=round(tt, 4),
                            mmr_over_pool=round(tm / tp, 4), mmr_vs_torch=round(tt / tm, 3),
                            pool_peak_mb=round(mp / 2 ** 20, 2), mmr_peak_mb=round(mm / 2 ** 20, 2),
                            diverse_peak_mb=round(md / 2 ** 20, 2), torch_peak_mb=round(mt / 2 ** 20, 2),
                            gram_mb=round(B * N * N * 4 / 2 ** 20, 2),
                            torch_id_agreement=round(float((ti == mi).float().mean().item()), 6),
                            diverse_equals_mmr=bool(torch.equal(di, mi) and torch.equal(ds, ms)),
                            lam1_equal=bool(torch.equal(l1i, ki) and torch.equal(l1s, ks)),
                            cos_lam1=cos1, cos_lam=cos5, clusters_lam1=cl1, clusters_lam=cl5)
                lines.append(line)
                print(json.dumps(line), flush=True)
                del pids, psc, mi, ms, ti, ts, di, ds, l1i, l1s, ki, ks
                torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()
