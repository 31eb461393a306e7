"""Top-K retrieval at Yelp2018 shape: the fused kernel (retrieval.Recommender on CUDA, yr_recommend_topk) against the
dense PyTorch path (B x num_items scores, seen items masked by index_put, torch.topk), for several batch sizes and K.

Per configuration: warm-up calls, then `--iters` calls each timed with CUDA events; the median is reported, with the peak
memory allocated during one call above what was allocated before it (torch.cuda.max_memory_allocated). The item table
(38,048 x d fp32 = 9.7 MB at d = 64) fits in L2, as it does in real use. One JSON line per configuration, the GPU's name
and power limit first.

    python scripts/recommend_bench.py [--batches 256,1024,4096,16384] [--ks 20,100,1000] [--d 64] [--out file.jsonl]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, sm = (x.strip() for x in out.split(","))
        return {"gpu": name, "power_limit": power, "sm_max_clock": sm}
    except Exception as e:  # noqa: BLE001
        return {"gpu": torch.cuda.get_device_name(), "power_limit": f"unknown ({e.__class__.__name__})"}


def dense_topk(U, V, uid, k, seen_ptr, seen_idx):
    """What retrieval costs without the kernel: the whole score block, masked, then torch.topk."""
    scores = U[uid] @ V.T
    ptr = seen_ptr.to(torch.int64)
    start, cnt = ptr[uid], ptr[uid + 1] - ptr[uid]
    row = torch.repeat_interleave(torch.arange(uid.numel(), device=uid.device), cnt)
    first = torch.repeat_interleave(torch.cumsum(cnt, 0) - cnt, cnt)
    pos = torch.arange(row.numel(), device=uid.device) - first + torch.repeat_interleave(start, cnt)
    scores[row, seen_idx[pos].to(torch.int64)] = float("-inf")
    sc, ids = torch.topk(scores, k, dim=1)
    return ids, sc


def measure(fn, warmup, iters):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    fn()
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    times = []
    for _ in range(iters):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        times.append(e0.elapsed_time(e1))
    return statistics.median(times), min(times), peak


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="256,1024,4096,16384")
    ap.add_argument("--ks", default="20,100,1000")
    ap.add_argument("--d", type=int, default=64)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("recommend_bench.py measures on a CUDA device; none is visible")

    from yelprecommendation_b200.data import synthetic as syn
    from yelprecommendation_b200.retrieval import Recommender, SeenItems

    dev = torch.device("cuda", 0)
    inter = syn.make_interactions()                      # Yelp2018 shape: 31,668 users x 38,048 items
    split = syn.split_per_user(inter, seed=42)
    seen = SeenItems.from_split(split, inter.num_items)
    nU, nI, d = inter.num_users, inter.num_items, args.d
    g = torch.Generator(device=dev).manual_seed(0)
    U = torch.randn(nU, d, device=dev, generator=g) * d ** -0.5
    V = torch.randn(nI, d, device=dev, generator=g) * d ** -0.5
    rec = Recommender(U, V, seen)
    ptr, idx = seen.on(dev)
    lines = [dict(gpu_info(), users=nU, items=nI, d=d, seen_nnz=int(seen.idx.numel()), warmup=args.warmup, iters=args.iters)]
    print(json.dumps(lines[0]), flush=True)
    rng = np.random.default_rng(0)
    for B in (int(x) for x in args.batches.split(",")):
        uid = torch.from_numpy(rng.choice(nU, size=min(B, nU), replace=B > nU)).to(dev) if B <= nU else \
            torch.from_numpy(rng.integers(0, nU, size=B)).to(dev)
        for k in (int(x) for x in args.ks.split(",")):
            fused = lambda: rec.recommend(uid, k)
            dense = lambda: dense_topk(U, V, uid, k, ptr, idx)
            fi, fs = fused()
            di, ds = dense()
            agree = float((fi == di).float().mean().item())
            max_sc = float((fs - ds).abs().max().item())
            tf, tf_min, mf = measure(fused, args.warmup, args.iters)
            td, td_min, md = measure(dense, args.warmup, args.iters)
            line = dict(batch=B, k=k, fused_ms=round(tf, 4), fused_min_ms=round(tf_min, 4), dense_ms=round(td, 4),
                        dense_min_ms=round(td_min, 4), speedup=round(td / tf, 3), fused_peak_mb=round(mf / 2 ** 20, 2),
                        dense_peak_mb=round(md / 2 ** 20, 2), score_matrix_mb=round(B * nI * 4 / 2 ** 20, 2),
                        id_agreement=round(agree, 6), max_score_diff=max_sc)
            lines.append(line)
            print(json.dumps(line), flush=True)
            del fi, fs, di, ds
            torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(json.dumps(x) for x in lines) + "\n")


if __name__ == "__main__":
    main()
