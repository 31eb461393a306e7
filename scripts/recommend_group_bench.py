"""Group retrieval at Yelp2018 shape: least-misery and average top-K for groups of users, the kernel
(Recommender.recommend_group, yr_recommend_group_topk) against the ways to get the same lists without it.

Tables: Gaussian user / item tables scaled by 1 / sqrt(d). Seen items: SeenItems.from_split of the synthetic Yelp2018 split
(31,668 users x 38,048 items). Groups: G groups of m distinct random users, m in {2, 4, 8}, or "mix" (m uniform in 2..8).

Arms per configuration (d, G, m, K, agg):
  group    rec.recommend_group(groups, K, agg)
  members  rec.recommend(all G * m member users, K): the same fma work, one list per member (the yardstick)
  dense    member by member U[u_j] @ V^T into one G x nI fold (torch.minimum, or adds then a division), the union of the
           members' seen items set to -inf, torch.topk. Member index lists and seen entries are prepared outside the timing
  meanvec  (mean only) the members' mean user vector per group through ops.recommend_topk with the union of their seen
           lists by row (prepared outside the timing): 1 / m of the fma work, equal only up to rounding
The median of CUDA-event timings and the peak memory per call, as scripts/recommend_bench.py. group_of_one_equal:
recommend_group of G groups of one equals recommend of the same users bit for bit. dense_id_agreement /
meanvec_id_agreement: the share of the group arm's ids each returns in the same row (any position). One JSON line per
configuration, the GPU's name, power limit and SM clock first.

    python scripts/recommend_group_bench.py [--ds 64,256] [--groups 256,4096] [--out f.jsonl]
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


def dense_group(U, V, steps, m, k, agg, seen_rows, seen_items):
    """The fold without the kernel: steps[j] = (rows with more than j members, their j-th member), G x nI scores."""
    A = None
    for rows, uid in steps:
        s = U[uid] @ V.T
        if A is None:
            A = s
        elif agg == "min":
            A[rows] = torch.minimum(A[rows], s)
        else:
            A[rows] += s
    if agg == "mean":
        A /= m[:, None]
    A[seen_rows, seen_items] = float("-inf")
    sc, ids = torch.topk(A, k, dim=1)
    return ids, sc


def agreement(a, b):
    """Mean over rows of |ids of a in row r that b also returns in row r| / k."""
    k = a.shape[1]
    hit = (a[:, :, None] == b[:, None, :]).any(2) & (a >= 0)
    return round(float(hit.float().sum(1).mean().item() / k), 6)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ds", default="64,256")
    ap.add_argument("--groups", default="256,4096")
    ap.add_argument("--sizes", default="2:20,4:20,8:20,mix:20,4:100")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("recommend_group_bench.py measures on a CUDA device; none is visible")

    from yelprecommendation_b200 import ops
    from yelprecommendation_b200.data import synthetic as syn
    from yelprecommendation_b200.retrieval import Recommender, SeenItems, UserGroups, _list_entries

    dev = torch.device("cuda", 0)
    inter = syn.make_interactions()                      # Yelp2018 shape: 31,668 users x 38,048 items
    split = syn.split_per_user(inter, seed=42)
    seen = SeenItems.from_split(split, inter.num_items)
    nU, nI = inter.num_users, inter.num_items
    head = dict(gpu_info(), users=nU, items=nI, seen_nnz=int(seen.idx.numel()), warmup=args.warmup, iters=args.iters)
    lines = [head]
    print(json.dumps(head), flush=True)
    for d in (int(x) for x in args.ds.split(",")):
        g = torch.Generator(device=dev).manual_seed(d)
        U = torch.randn(nU, d, device=dev, generator=g) * d ** -0.5
        V = torch.randn(nI, d, device=dev, generator=g) * d ** -0.5
        rec = Recommender(U, V, seen)
        for G in (int(x) for x in args.groups.split(",")):
            for mk in args.sizes.split(","):
                ms, k = mk.split(":")
                k = int(k)
                rng = np.random.default_rng(G * 1000 + d + k)
                sizes = rng.integers(2, 9, G) if ms == "mix" else np.full(G, int(ms))
                groups = UserGroups.from_lists([rng.choice(nU, s, replace=False) for s in sizes], nU)
                gptr, mem = groups.on(dev)
                ptr64 = gptr.to(torch.int64)
                m = (ptr64[1:] - ptr64[:-1]).to(torch.float32)
                steps = []
                for j in range(int(sizes.max())):
                    rows = (m > j).nonzero().reshape(-1)
                    steps.append((rows, mem[ptr64[rows] + j]))
                grow = torch.repeat_interleave(torch.arange(G, device=dev), (ptr64[1:] - ptr64[:-1]))
                er, ei = _list_entries(seen, mem, dev)
                seen_rows, seen_items = grow[er], ei
                union = SeenItems.from_pairs(seen_rows.cpu(), seen_items.cpu(), G, nI)
                uptr, uidx = union.on(dev)
                members = lambda: rec.recommend(mem, k)
                tmem, _, pmem = measure(members, args.warmup, args.iters)
                ones = mem[:G]                                   # G groups of one
                singles = UserGroups(torch.arange(G + 1, dtype=torch.int32), ones.cpu(), G, nU)
                ri, rsc = rec.recommend(ones, k)
                for agg in ("min", "mean"):
                    grp = lambda: rec.recommend_group(groups, k, agg)
                    dense = lambda: dense_group(U, V, steps, m, k, agg, seen_rows, seen_items)
                    gi, gs = grp()
                    di, _ = dense()
                    oi, osc = rec.recommend_group(singles, k, agg)
                    one_equal = bool(torch.equal(oi, ri) and torch.equal(osc, rsc))
                    tg, tg_min, pg = measure(grp, args.warmup, args.iters)
                    td, _, pd = measure(dense, args.warmup, args.iters)
                    line = dict(d=d, groups=G, members=ms, k=k, agg=agg, member_users=int(mem.numel()),
                                group_ms=round(tg, 4), group_min_ms=round(tg_min, 4), members_ms=round(tmem, 4),
                                dense_ms=round(td, 4), group_over_members=round(tg / tmem, 4),
                                dense_over_group=round(td / tg, 3), group_peak_mb=round(pg / 2 ** 20, 2),
                                members_peak_mb=round(pmem / 2 ** 20, 2), dense_peak_mb=round(pd / 2 ** 20, 2),
                                dense_id_agreement=agreement(gi, di), group_of_one_equal=one_equal)
                    if agg == "mean":
                        Um = torch.zeros(G, d, device=dev).index_add_(0, grow, U[mem]) / m[:, None]
                        meanvec = lambda: ops.recommend_topk(Um, V, torch.arange(G, device=dev), k, uptr, uidx,
                                                             seen_by_row=True)
                        vi, _ = meanvec()
                        tv, _, pv = measure(meanvec, args.warmup, args.iters)
                        line.update(meanvec_ms=round(tv, 4), meanvec_peak_mb=round(pv / 2 ** 20, 2),
                                    meanvec_id_agreement=agreement(gi, vi))
                    lines.append(line)
                    print(json.dumps(line), flush=True)
                    del gi, gs, di
                    torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()
