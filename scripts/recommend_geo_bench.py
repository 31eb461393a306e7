"""Radius-restricted top-K retrieval at Yelp2018 shape: the geo kernel (yr_recommend_geo_topk) against the ways to get the
same answer without it, on a seeded synthetic map.

Items: 100 "cities" with Zipf sizes (city k holds a share proportional to 1 / k: the largest ~19 % of the catalog, the
smallest ~0.2 %), each a Gaussian of 3 km spread around a centre
drawn over North America (lat 25..50, lon -125..-70). Requests: a city drawn by size, the centre within ~1 km of the city
centre, and a radius of 1, 5 or 25 km (mixes r1, r5, r25), or the whole Earth (mix earth). Item grid cells: --cell-km.

Arms per configuration (d, B, K, mix):
  geo        ops.recommend_geo_topk with the requests' (c, t) on the device
  exclusion  the unrestricted kernel with a per-row exclusion CSR (seen items + every item outside the radius,
             seen_by_row); the CSR's size and the time to build it on the device are reported, not timed in the arm
  dense      B x items scores, seen and outside-radius items masked, torch.topk
  unrestricted  recommend(user_ids, k) on the same batch, ignoring the radius (the reference point)
The median of CUDA-event timings and the peak memory per call, as scripts/recommend_bench.py. id_agreement and
score_equal compare the geo arm with the exclusion arm (bit-identical by construction); in_radius_mean is the mean number
of items inside a row's radius. One JSON line per configuration, the GPU's name and power limit first.

    python scripts/recommend_geo_bench.py [--ds 64,256] [--batches 256,4096] [--ks 20,100] [--out file.jsonl]
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


def make_map(nI, rng, n_city=100, spread_km=3.0):
    """(lat, lon) of every item, (lat, lon) of the city centres and the city sizes."""
    w = 1.0 / np.arange(1, n_city + 1)                       # Zipf: city k holds a share proportional to 1 / k
    sizes = np.floor(w / w.sum() * nI).astype(np.int64)
    sizes[: nI - sizes.sum()] += 1                           # the rounding remainder, one item each to the largest
    clat, clon = rng.uniform(25, 50, n_city), rng.uniform(-125, -70, n_city)
    city = rng.permutation(np.repeat(np.arange(n_city), sizes))
    deg = spread_km / 111.2
    lat = clat[city] + rng.normal(0, deg, nI)
    lon = clon[city] + rng.normal(0, deg, nI) / np.cos(np.radians(clat[city]))
    return lat, lon, clat, clon, sizes


def seen_rows(seen_ptr, seen_idx, uid):
    ptr = seen_ptr.to(torch.int64)
    start, cnt = ptr[uid], ptr[uid + 1] - ptr[uid]
    row = torch.repeat_interleave(torch.arange(uid.numel(), device=uid.device), cnt)
    first = torch.repeat_interleave(torch.cumsum(cnt, 0) - cnt, cnt)
    pos = torch.arange(row.numel(), device=uid.device) - first + torch.repeat_interleave(start, cnt)
    return row, seen_idx[pos].to(torch.int64)


def exclusion_csr(seen_ptr, seen_idx, inside, uid):
    """Per batch row: seen items of uid[b] + items outside the radius (inside [B x nI] bool), on the device."""
    drop = ~inside
    row, item = seen_rows(seen_ptr, seen_idx, uid)
    drop[row, item] = True
    out_ptr = torch.zeros(uid.numel() + 1, dtype=torch.int64, device=uid.device)
    out_ptr[1:] = torch.cumsum(drop.sum(1), 0)
    idx = drop.nonzero()[:, 1].to(torch.int32)               # row-major: ascending per row
    return out_ptr.to(torch.int32), idx


def dense_geo_topk(U, V, uid, k, seen_ptr, seen_idx, P, c, t):
    from yelprecommendation_b200.retrieval import _geo_inside
    scores = U[uid] @ V.T
    scores.masked_fill_(~_geo_inside(P, c, t), float("-inf"))
    row, item = seen_rows(seen_ptr, seen_idx, uid)
    scores[row, item] = float("-inf")
    sc, ids = torch.topk(scores, k, dim=1)
    return ids, sc


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--ds", default="64,256")
    ap.add_argument("--batches", default="256,4096")
    ap.add_argument("--ks", default="20,100")
    ap.add_argument("--mixes", default="r1,r5,r25,earth")
    ap.add_argument("--cell-km", type=float, default=2.0)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("recommend_geo_bench.py measures on a CUDA device; none is visible")

    from yelprecommendation_b200 import ops
    from yelprecommendation_b200.data import synthetic as syn
    from yelprecommendation_b200.retrieval import (EARTH_RADIUS_KM, ItemLocations, Recommender, SeenItems, _geo_inside,
                                                   geo_query)

    dev = torch.device("cuda", 0)
    inter = syn.make_interactions()                      # Yelp2018 shape: 31,668 users x 38,048 items
    split = syn.split_per_user(inter, seed=42)
    seen = SeenItems.from_split(split, inter.num_items)
    nU, nI = inter.num_users, inter.num_items
    rng = np.random.default_rng(0)
    lat, lon, clat, clon, sizes = make_map(nI, rng)
    loc = ItemLocations.from_degrees(lat, lon, cell_km=args.cell_km)
    keys, cptr, citems, P = loc.on(dev)
    ptr, idx = seen.on(dev)
    head = dict(gpu_info(), users=nU, items=nI, seen_nnz=int(seen.idx.numel()), cities=len(sizes),
                city_sizes=[int(sizes.max()), int(np.median(sizes)), int(sizes.min())], cell_km=args.cell_km,
                nonempty_cells=int(keys.numel()), warmup=args.warmup, iters=args.iters)
    lines = [head]
    print(json.dumps(head), flush=True)
    radius = {"r1": 1.0, "r5": 5.0, "r25": 25.0, "earth": np.pi * EARTH_RADIUS_KM}
    for d in (int(x) for x in args.ds.split(",")):
        g = torch.Generator(device=dev).manual_seed(d)
        U = torch.randn(nU, d, device=dev, generator=g) * d ** -0.5
        V = torch.randn(nI, d, device=dev, generator=g) * d ** -0.5
        rec = Recommender(U, V, seen)
        for B in (int(x) for x in args.batches.split(",")):
            uid = torch.from_numpy(rng.integers(0, nU, size=B)).to(dev)
            j = rng.choice(len(sizes), size=B, p=sizes / sizes.sum())
            qlat = clat[j] + rng.normal(0, 1.0 / 111.2, B)
            qlon = clon[j] + rng.normal(0, 1.0 / 111.2, B) / np.cos(np.radians(clat[j]))
            for mix in args.mixes.split(","):
                c, t = geo_query((qlat, qlon), radius[mix], B)
                c, t = torch.from_numpy(c).to(dev), torch.from_numpy(t).to(dev)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                inside = _geo_inside(P, c, t)
                xptr, xidx = exclusion_csr(ptr, idx, inside, uid)
                e1.record()
                e1.synchronize()
                csr_ms = e0.elapsed_time(e1)
                in_mean = float(inside.sum(1).double().mean().item())
                del inside
                for k in (int(x) for x in args.ks.split(",")):
                    geo = lambda: ops.recommend_geo_topk(U, V, uid, k, keys, cptr, citems, P, loc.cell_deg, c, t, ptr,
                                                         idx)
                    exc = lambda: ops.recommend_topk(U, V, uid, k, xptr, xidx, seen_by_row=True)
                    dense = lambda: dense_geo_topk(U, V, uid, k, ptr, idx, P, c, t)
                    full = lambda: rec.recommend(uid, k)
                    gi, gs = geo()
                    xi, xs = exc()
                    tg, tg_min, mg = measure(geo, args.warmup, args.iters)
                    tx, tx_min, mx = measure(exc, args.warmup, args.iters)
                    td, td_min, md = measure(dense, args.warmup, args.iters)
                    tf, tf_min, mf = measure(full, args.warmup, args.iters)
                    line = dict(d=d, batch=B, k=k, mix=mix, radius_km=round(float(radius[mix]), 3),
                                in_radius_mean=round(in_mean, 1), in_radius_frac=round(in_mean / nI, 4),
                                geo_ms=round(tg, 4), geo_min_ms=round(tg_min, 4),
                                exclusion_ms=round(tx, 4), dense_ms=round(td, 4), unrestricted_ms=round(tf, 4),
                                vs_exclusion=round(tx / tg, 3), vs_dense=round(td / tg, 3),
                                vs_unrestricted=round(tf / tg, 3),
                                geo_peak_mb=round(mg / 2 ** 20, 2), exclusion_peak_mb=round(mx / 2 ** 20, 2),
                                dense_peak_mb=round(md / 2 ** 20, 2), unrestricted_peak_mb=round(mf / 2 ** 20, 2),
                                exclusion_csr_mb=round((xptr.numel() + xidx.numel()) * 4 / 2 ** 20, 2),
                                exclusion_csr_build_ms=round(csr_ms, 4),
                                id_agreement=float((gi == xi).float().mean().item()),
                                score_equal=bool(torch.equal(gs, xs)))
                    lines.append(line)
                    print(json.dumps(line), flush=True)
                    del gi, gs, xi, xs
                del xptr, xidx
                torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()
