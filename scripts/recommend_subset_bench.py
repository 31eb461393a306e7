"""Subset-restricted top-K retrieval at Yelp2018 shape: the subset kernel (yr_recommend_subset_topk) against the ways to get
the same answer without it, on seeded synthetic subsets.

Subsets: 100 disjoint "cities" with Zipf sizes (the largest ~10 % of the catalog, the smallest ~50 items) and 20
overlapping "categories" of 1-5 % of the catalog each. Request mixes: (a) every row draws a city by size, (b) every row in
the largest city, (c) every row in a city of ~1 % of the catalog, (d) every row -1 (whole catalog).

Arms per configuration (d, B, K, mix):
  subset     ops.recommend_subset_topk, subset ids on the device, max_len from the requested subsets
  exclusion  the unrestricted kernel with a per-row exclusion CSR (seen items + everything outside the subset,
             seen_by_row); the CSR's size and the time to build it on the device are reported, not timed in the arm
  dense      B x items scores, seen and outside-subset items masked, torch.topk
  unrestricted  recommend(user_ids, k) on the same batch, ignoring the subsets (the reference point)
The median of CUDA-event timings and the peak memory per call, as scripts/recommend_bench.py. id_agreement and
score_equal compare the subset arm with the exclusion arm (bit-identical by construction). One JSON line per
configuration, the GPU's name and power limit first.

    python scripts/recommend_subset_bench.py [--ds 64,256] [--batches 256,4096] [--ks 20,100] [--out file.jsonl]
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


def make_subsets(nI, rng):
    """(cities, categories) as lists of ascending item-id arrays."""
    n_city = 100
    w = 1.0 / np.arange(1, n_city + 1) ** 1.2
    sizes = np.maximum(50, np.round(w / w[0] * 0.10 * nI)).astype(np.int64)
    perm = rng.permutation(nI)
    cities, at = [], 0
    for s in sizes:
        cities.append(np.sort(perm[at:at + s]))
        at += s
    cats = [np.sort(rng.choice(nI, int(rng.uniform(0.01, 0.05) * nI), replace=False)) for _ in range(20)]
    return cities, cats


def exclusion_csr(seen_ptr, seen_idx, sub_mask, uid, sid):
    """Per batch row: seen items of uid[b] + items outside subset sid[b] (sub_mask [G x nI] bool, True = member), on the
    device. Returns (ptr int32 [B + 1], idx int32)."""
    B, nI = uid.numel(), sub_mask.shape[1]
    drop = ~sub_mask[sid.clamp(min=0)]
    drop[sid < 0] = False
    ptr = seen_ptr.to(torch.int64)
    start, cnt = ptr[uid], ptr[uid + 1] - ptr[uid]
    row = torch.repeat_interleave(torch.arange(B, device=uid.device), cnt)
    first = torch.repeat_interleave(torch.cumsum(cnt, 0) - cnt, cnt)
    pos = torch.arange(row.numel(), device=uid.device) - first + torch.repeat_interleave(start, cnt)
    drop[row, seen_idx[pos].to(torch.int64)] = True
    counts = drop.sum(1)
    out_ptr = torch.zeros(B + 1, dtype=torch.int64, device=uid.device)
    out_ptr[1:] = torch.cumsum(counts, 0)
    idx = drop.nonzero()[:, 1].to(torch.int32)               # row-major: ascending per row
    return out_ptr.to(torch.int32), idx


def dense_subset_topk(U, V, uid, k, seen_ptr, seen_idx, sub_mask, sid):
    scores = U[uid] @ V.T
    outside = ~sub_mask[sid.clamp(min=0)]
    outside[sid < 0] = False
    scores.masked_fill_(outside, float("-inf"))
    ptr = seen_ptr.to(torch.int64)
    start, cnt = ptr[uid], ptr[uid + 1] - ptr[uid]
    row = torch.repeat_interleave(torch.arange(uid.numel(), device=uid.device), cnt)
    first = torch.repeat_interleave(torch.cumsum(cnt, 0) - cnt, cnt)
    pos = torch.arange(row.numel(), device=uid.device) - first + torch.repeat_interleave(start, cnt)
    scores[row, seen_idx[pos].to(torch.int64)] = float("-inf")
    sc, ids = torch.topk(scores, k, dim=1)
    return ids, sc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ds", default="64,256")
    ap.add_argument("--batches", default="256,4096")
    ap.add_argument("--ks", default="20,100")
    ap.add_argument("--mixes", default="a,b,c,d")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("recommend_subset_bench.py measures on a CUDA device; none is visible")

    from yelprecommendation_b200 import ops
    from yelprecommendation_b200.data import synthetic as syn
    from yelprecommendation_b200.retrieval import ItemSubsets, Recommender, SeenItems

    dev = torch.device("cuda", 0)
    inter = syn.make_interactions()                      # Yelp2018 shape: 31,668 users x 38,048 items
    split = syn.split_per_user(inter, seed=42)
    seen = SeenItems.from_split(split, inter.num_items)
    nU, nI = inter.num_users, inter.num_items
    rng = np.random.default_rng(0)
    cities, cats = make_subsets(nI, rng)
    lists = cities + cats
    subsets = ItemSubsets.from_pairs(np.concatenate([np.full(len(x), g) for g, x in enumerate(lists)]),
                                     np.concatenate(lists), len(lists), nI)
    sptr, sidx = subsets.on(dev)
    ptr, idx = seen.on(dev)
    sub_mask = torch.zeros(len(lists), nI, dtype=torch.bool, device=dev)
    for g, x in enumerate(lists):
        sub_mask[g, torch.from_numpy(x).to(dev)] = True
    city_len = np.array([len(c) for c in cities])
    one_pct = int(np.argmin(np.abs(city_len - 0.01 * nI)))
    head = dict(gpu_info(), users=nU, items=nI, seen_nnz=int(seen.idx.numel()), cities=len(cities),
                city_sizes=[int(city_len.max()), int(city_len[one_pct]), int(city_len.min())], categories=len(cats),
                category_sizes=[int(min(map(len, cats))), int(max(map(len, cats)))], warmup=args.warmup, iters=args.iters)
    lines = [head]
    print(json.dumps(head), flush=True)
    for d in (int(x) for x in args.ds.split(",")):
        g = torch.Generator(device=dev).manual_seed(d)
        U = torch.randn(nU, d, device=dev, generator=g) * d ** -0.5
        V = torch.randn(nI, d, device=dev, generator=g) * d ** -0.5
        rec = Recommender(U, V, seen, subsets=subsets)
        for B in (int(x) for x in args.batches.split(",")):
            uid = torch.from_numpy(rng.integers(0, nU, size=B)).to(dev)
            mixes = {"a": rng.choice(len(cities), size=B, p=city_len / city_len.sum()),
                     "b": np.full(B, int(np.argmax(city_len))), "c": np.full(B, one_pct), "d": np.full(B, -1)}
            for mix in args.mixes.split(","):
                s = mixes[mix]
                max_len = nI if (s < 0).any() else int(subsets.lengths[s[s >= 0]].max())
                sid = torch.from_numpy(s).to(dev)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                xptr, xidx = exclusion_csr(ptr, idx, sub_mask, uid, sid)
                e1.record()
                e1.synchronize()
                csr_ms = e0.elapsed_time(e1)
                for k in (int(x) for x in args.ks.split(",")):
                    sub = lambda: ops.recommend_subset_topk(U, V, uid, k, sptr, sidx, sid, max_len, ptr, idx)
                    exc = lambda: ops.recommend_topk(U, V, uid, k, xptr, xidx, seen_by_row=True)
                    dense = lambda: dense_subset_topk(U, V, uid, k, ptr, idx, sub_mask, sid)
                    full = lambda: rec.recommend(uid, k)
                    si, ss = sub()
                    xi, xs = exc()
                    ts, ts_min, ms = measure(sub, args.warmup, args.iters)
                    tx, tx_min, mx = measure(exc, args.warmup, args.iters)
                    td, td_min, md = measure(dense, args.warmup, args.iters)
                    tf, tf_min, mf = measure(full, args.warmup, args.iters)
                    line = dict(d=d, batch=B, k=k, mix=mix, max_len=max_len,
                                subset_ms=round(ts, 4), subset_min_ms=round(ts_min, 4),
                                exclusion_ms=round(tx, 4), dense_ms=round(td, 4), unrestricted_ms=round(tf, 4),
                                vs_exclusion=round(tx / ts, 3), vs_dense=round(td / ts, 3), vs_unrestricted=round(tf / ts, 3),
                                subset_peak_mb=round(ms / 2 ** 20, 2), exclusion_peak_mb=round(mx / 2 ** 20, 2),
                                dense_peak_mb=round(md / 2 ** 20, 2), unrestricted_peak_mb=round(mf / 2 ** 20, 2),
                                exclusion_csr_mb=round((xptr.numel() + xidx.numel()) * 4 / 2 ** 20, 2),
                                exclusion_csr_build_ms=round(csr_ms, 4),
                                id_agreement=float((si == xi).float().mean().item()),
                                score_equal=bool(torch.equal(ss, xs)))
                    lines.append(line)
                    print(json.dumps(line), flush=True)
                    del si, ss, xi, xs
                del xptr, xidx
                torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()
