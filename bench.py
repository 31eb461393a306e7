#!/usr/bin/env python
"""bench.py — headline benchmark of the BPR-MF / NGCF train + full-catalog eval hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

Headline (BASELINE.json configs[1]): NGCF 3-layer d=64 BPR training on the synthetic Yelp2018-shape graph
(31,668 users x 38,048 items, 1,561,406 interactions), batch 2048, Adam lr 1e-4 — `value` = training triples/s
with every input resident in HBM; `e2e` = the same metric through NGCFTrainer.train() with HOST batches (pinned
H2D of the ids and a D2H read of the loss every step). The JSON line also carries, under "extra", the two other
rows of the metric: BPR-MF training triples/s (configs[0]) and full-catalog top-10 eval users/s for the MF and
NGCF embeddings (configs[2]), each with its own roofline fraction.

N > 1 (one process per GPU under torchrun): NGCF/MF training at Yelp shape does not shard (17.8 MB of parameters,
sequential step semantics — DESIGN.md "replicas only"), so every rank trains an independent replica and `value`
is the sum over replicas (weak scaling); evaluation shards its rows across ranks with no data-path collective.

`--impl reference`: the reference's own CPU implementation of the same step (oracle/torch_port.py, the torch-CPU
restatement pinned to the real reference by tests/golden — /root/reference does not exist on the GPU box), on all
host threads, rank 0 only.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time
from types import SimpleNamespace

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True       # the benchmark may run from a read-only tree: it leaves no bytecode caches there

METRIC = "ngcf_bpr_train_triples_per_sec"
UNIT = "triples/s"
B = 2048
D = 64
LAYERS = 3
M_BYTES = (31_668 + 38_048) * D * 4            # one N x d fp32 row matrix = 17.85 MB
WORKLOAD = ("NGCF 3-layer d=64 BPR train step, Yelp2018-shape graph (31,668u x 38,048i, 1,561,406 interactions), "
            "batch 2048, Adam lr 1e-4 (BASELINE.json configs[1])")
NCU_SPMM_DRAM_BYTES = 45_472_000               # ncu --set full, spmm_chunk_kernel<64,0> (full graph): dram read 44.07 MB + write 1.40 MB (profiles/r01_ncu_full_summary_final.txt)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return dict(hbm=float(j["hbm_gbs"]), bf16=float(j["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, bf16=1590.0, src="fallback")


class ClockSampler:
    """SM clock + clock-event (throttle) reasons sampled DURING the timed region. The region is tens of ms, so this polls
    NVML in-process every ~2 ms (the `nvidia-smi -lms` recipe of B200_PROFILING.md cannot start that fast); the same
    counters nvidia-smi prints: clocks.sm, clocks.max.sm, clocks_event_reasons.*"""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, gpu_index):
        self.sm, self.mask, self.max_mhz, self.h, self.nv = [], 0, None, None, None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml
            pynvml.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            ids = [x for x in vis.split(",") if x.strip()]
            phys = int(ids[gpu_index]) if ids and all(x.strip().isdigit() for x in ids) else gpu_index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nv = pynvml
        except Exception:
            self.h = None

    def _sample(self):
        nv = self.nv
        self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
        try:
            self.mask |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
        except Exception:
            self.mask |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))

    def _pump(self):
        while not self._stop.is_set():
            try:
                self._sample()
            except Exception:
                return
            time.sleep(0.002)

    def start(self):
        if self.h is not None:
            self._thr = threading.Thread(target=self._pump, daemon=True)
            self._thr.start()

    def stop(self):
        self._stop.set()
        if self._thr is not None:
            self._thr.join(timeout=1.0)
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(v for k, v in self.REASONS.items() if self.mask & k), "samples": len(self.sm),
                "source": "NVML polled every 2 ms inside the timed region"}


def build_workload(seed=2018):
    from yelprecommendation_b200.data import synthetic as syn
    from yelprecommendation_b200.data.graph import build_eval_csr, build_laplacian
    inter = syn.make_interactions(seed=seed)
    split = syn.split_per_user(inter, seed=42)
    tu, tp_, tn = syn.sample_triples(split, inter.num_items, seed=42)
    L = build_laplacian(inter.user, inter.item, inter.rating, inter.num_users, inter.num_items)
    uid, pos, mask = syn.eval_lists(split, "valid")
    ecsr = build_eval_csr(uid, pos, mask, inter.num_items)
    return SimpleNamespace(inter=inter, split=split, tri=(tu, tp_, tn), L=L, ecsr=ecsr)


def cfg(**kw):
    base = dict(device="cuda", model_dir=tempfile.mkdtemp(), embed_size=D, optimizer="adam", lr=1e-4, weight_decay=0.0,
                top_n=10, wandb=False, num_orders=LAYERS, epochs=1, patience=1, best_metric="loss", batch_size=B)
    base.update(kw)
    return SimpleNamespace(**base)


def timed(fn, n, stream_sync=True):
    """ms for n calls of fn, CUDA events on the current stream, synchronised on both sides."""
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(n):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def dump_outputs(out_dir, ntr, step_losses):
    """What the timed NGCF step hands its caller after the last timed step: that step's batch-mean BPR loss and the
    parameters it updated (state_dict names), one float32 .npy each (17.9 MB in all at the Yelp shape)."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"loss": step_losses[-1:], **ntr.model.state_dict()}
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().to(torch.float32).cpu().numpy())


# ---------------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle.torch_port import NGCFPort
    from yelprecommendation_b200.data import synthetic as syn
    w = build_workload()
    torch.manual_seed(42)
    n = w.inter.num_users + w.inter.num_items
    emb = torch.randn(n, D)
    lin = lambda: torch.nn.Linear(D, D, bias=False).weight.detach()
    port = NGCFPort(emb, [lin() for _ in range(LAYERS)], [lin() for _ in range(LAYERS)], w.inter.num_users, w.L,
                    "adam", 1e-4, 0.0)
    batches = syn.to_batches(*[a[: B * (args.steps + args.warmup)] for a in w.tri], B)
    budget_s = float(os.environ.get("YR_REF_BUDGET_S", "170"))
    t0 = time.perf_counter()
    port.train(batches[:1])
    t_first = time.perf_counter() - t0
    warm = max(0, min(args.warmup - 1, int(budget_s * 0.2 / max(t_first, 1e-6))))
    if warm:
        port.train(batches[1:1 + warm])
    steps = max(1, min(args.steps, int(budget_s * 0.8 / max(t_first, 1e-6))))
    use = batches[1 + warm:1 + warm + steps]
    t0 = time.perf_counter()
    port.train(use)
    dt = time.perf_counter() - t0
    val = steps * B / dt
    cores = torch.get_num_threads()
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "steps_requested": args.steps, "warmup": warm + 1, "ms_per_step": 1e3 * dt / steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": "port",
                             "sample": f"{steps} full train steps of oracle/torch_port.NGCFPort (torch CPU ops of the "
                                       "reference, N x N identity hoisted: (L+I)E = LE + E)"},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "host": {"cpu_count": os.cpu_count(), "torch_threads": cores}}
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------------------------------------
def config5_extras(extra, dev, rank, world, barrier, max_over_ranks, pk, args):
    """BASELINE config 5: scaled synthetic BPR-MF + NGCF, 10 M users x 2 M items, ~500 M interactions, d = 128, tables and SpMM
    row-sharded over the N ranks of this run (strong scaling: the problem is fixed, N = 1 runs it on one GPU)."""
    import torch.distributed as dist
    from yelprecommendation_b200.data.scaled import make_scaled_graph
    from yelprecommendation_b200.trainers.sharded_mf_trainer import ShardedMFTrainer
    from yelprecommendation_b200.trainers.sharded_ngcf_trainer import ShardedNGCFTrainer
    sc = float(args.c5_scale)
    nU5, nI5, nnz5, d5, B5 = int(10_000_000 * sc), int(2_000_000 * sc), int(500_000_000 * sc), 128, 65_536
    ref_path = os.path.join(ROOT, "profiles", "r02_c5_n1.json")
    ref1 = json.load(open(ref_path)) if (os.path.exists(ref_path) and sc == 1.0) else {}

    def eff(key, value):
        """strong-scaling efficiency against the committed 1-GPU run of the same build (profiles/r02_c5_n1.json)"""
        base = ref1.get(key, {}).get("value")
        return (value / base / world) if base else None

    torch.cuda.empty_cache()
    g5 = torch.Generator(device=dev).manual_seed(5)              # same triples on every rank
    n_mf = 12
    skip_mf = os.environ.get("YR_C5_SKIP_MF", "0") == "1"          # experiments on the NGCF exchange only
    su5 = torch.randint(0, nU5, (n_mf + 3, B5), device=dev, generator=g5)
    sp5 = torch.randint(0, nI5, (n_mf + 3, B5), device=dev, generator=g5)
    sn5 = torch.randint(0, nI5, (n_mf + 3, B5), device=dev, generator=g5)
    # ---- row-sharded BPR-MF
    for oname in (() if skip_mf else ("sgd", "adam")):
        try:
            tr = ShardedMFTrainer(cfg(embed_size=d5, optimizer=oname), nI5, nU5)
            acc = torch.zeros(1, device=dev, dtype=torch.float64)
            for i in range(3):
                tr.train_step(su5[i], sp5[i], sn5[i], acc)
            barrier()
            ms5 = max_over_ranks(timed(lambda i: tr.train_step(su5[3 + i], sp5[3 + i], sn5[3 + i], acc), n_mf)) / n_mf
            val = B5 / (ms5 * 1e-3)
            rec = {"value": val, "unit": UNIT, "ms_per_step": ms5, "scaling": "strong", "batch": B5,
                   "tables": f"{nU5:,}u x {nI5:,}i x d{d5} row-sharded over {world} GPU(s)",
                   "efficiency_vs_n1": eff(f"c5_mf_{oname}", val)}
            tm = tr.traffic_model(B5)
            rec.update(tm)
            # every GPU moves alg_bytes_per_triple * B / world through its HBM per step; the exchange moves nvlink_bytes over
            # NVLink 5 (900 GB/s per direction per GPU): whichever fraction is larger is what bounds the step
            rec["hbm_frac"] = tm["alg_bytes_per_triple"] * B5 / world / (ms5 * 1e-3) / 1e9 / pk["hbm"]
            rec["nvlink_frac_of_900GBps"] = tm["nvlink_bytes_per_step_per_gpu"] / 2 / (ms5 * 1e-3) / 900e9 if world > 1 else None
            extra[f"c5_mf_{oname}"] = rec
            del tr
        except Exception as ex:
            extra[f"c5_mf_{oname}"] = {"error": repr(ex)}
        torch.cuda.empty_cache()
    del su5, sp5, sn5
    # ---- row-sharded NGCF, 3 layers, d = 128, Adam
    t0 = time.perf_counter()
    graph = make_scaled_graph(nU5, nI5, nnz5, seed=5, device=dev)
    torch.cuda.synchronize()
    t_gen = time.perf_counter() - t0
    n_ng = 2
    su = torch.randint(0, nU5, (n_ng + 1, B5), device=dev, generator=g5)
    sp = torch.randint(0, nI5, (n_ng + 1, B5), device=dev, generator=g5)
    sn_ = torch.randint(0, nI5, (n_ng + 1, B5), device=dev, generator=g5)
    t0 = time.perf_counter()
    tr = ShardedNGCFTrainer(cfg(seed=42, embed_size=d5, num_orders=3, optimizer="adam", lr=1e-4), nI5, nU5, graph)
    nnz_graph = graph.nnz
    del graph
    torch.cuda.empty_cache()
    torch.cuda.synchronize()
    t_build = time.perf_counter() - t0
    acc = torch.zeros(1, device=dev, dtype=torch.float64)
    tr.train_step(su[0], sp[0], sn_[0], acc)                     # warm-up: NCCL pair connections, kernel attributes
    barrier()
    ms_ng = max_over_ranks(timed(lambda i: tr.train_step(su[1 + i], sp[1 + i], sn_[1 + i], acc), n_ng)) / n_ng
    # pieces, timed alone on this rank (CUDA events): one panel-less SpMM over the local block and the exposed exchange
    X = tr.X[0] if world > 1 else tr.E[0]
    ms_spmm = timed(lambda i: [tr.k.spmm(Ap, X, tr.LE[0][a:b], False) for a, b, Ap in tr.panels], 2) / 2
    ms_dfw = timed(lambda i: [tr.k.dense_fwd(tr.E[0][a:b], tr.LE[0][a:b], tr.W1[0], tr.W2[0], tr.E[1][a:b]) for a, b, _ in tr.panels], 2) / 2
    def dense_bwd_all(i):                       # dense backward of one layer over the local rows (T, G += ..., dW partials)
        for pi, (a, b, _) in enumerate(tr.panels):
            tr.k.dense_bwd(tr.E[0][a:b], tr.LE[0][a:b], tr.E[1][a:b], tr.G[1][a:b], tr.W1[0], tr.W2[0], tr.G[0][a:b], tr.T[a:b],
                           tr.dWp[pi, 0], tr.dWp[pi, 1])
    ms_dbw = timed(dense_bwd_all, 2) / 2
    ms_xchg = None
    if world > 1:
        def xchg(i):
            tr._exchange_all(tr.E[0], 0)
            tr._wait(0)
        xchg(0)
        barrier()
        ms_xchg = max_over_ranks(timed(xchg, 2) / 2)
    val = B5 / (ms_ng * 1e-3)
    gather_bytes = tr.nnz_local * d5 * 4
    extra["c5_ngcf"] = {
        "value": val, "unit": UNIT, "ms_per_step": ms_ng, "scaling": "strong", "batch": B5, "layers": 3, "embed_size": d5,
        "graph": f"{nU5:,}u x {nI5:,}i, {nnz_graph:,} interactions (Philox seed 5, device-generated), Laplacian nnz {2 * nnz_graph:,}",
        "rows_per_gpu": tr.per, "nnz_per_gpu": tr.nnz_local, "row_panels": len(tr.panels),
        "graph_gen_s": t_gen, "shard_build_s": t_build,
        "efficiency_vs_n1": eff("c5_ngcf", val),
        "spmm_ms_per_layer": ms_spmm, "spmm_gather_TBps": gather_bytes / (ms_spmm * 1e-3) / 1e12,
        "dense_fwd_ms_per_layer": ms_dfw, "dense_bwd_ms_per_layer": ms_dbw,
        "dense_kernels": "tcgen05 3xTF32 ring kernels at d = 128 (csrc/ngcf_tc.cu, csrc/ngcf_tc_bwd.cu), yr_dense_mode 2",
        "exchange_ms_per_layer_alone": ms_xchg,
        "exchange_bytes_per_layer_per_gpu": (world - 1) * tr.per * d5 * 4 if world > 1 else 0,
        "exchange": None if world == 1 else tr._xmode,
        "collectives": "none (1 GPU)" if world == 1 else
        f"per layer fwd and bwd: {len(tr.panels)} panel rounds ({(world - 1) * tr.per * d5 * 4 / 1e9:.2f} GB received per GPU per layer) "
        + ("pushed into the peers' symmetric-memory buffers by the copy engines (one stream per peer, one signal per peer and layer)"
           if tr._xmode == "symm" else "as grouped NCCL send/recv") +
        " underneath the next panel's SpMM/transform; all_reduce(tail rows 3B x 512 floats) + all_reduce(dW) per step",
        "loss_mean": float(acc.item()) / ((n_ng + 1) * B5)}
    del tr
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-extra", action="store_true", help="skip the MF-train / eval sub-benchmarks")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-c5", action="store_true", help="skip the scaled config-5 runs (10 M x 2 M, 500 M interactions)")
    ap.add_argument("--c5-scale", type=float, default=1.0, help="shrink config 5 (users, items, interactions) by this factor")
    ap.add_argument("--only-c5", action="store_true", help="profiling aid: only the config-5 runs, no JSON contract")
    ap.add_argument("--only", default="", help="profiling aid: run only 'ngcf' | 'mf' | 'eval' steps, no JSON contract")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the loss and parameters of the last timed NGCF step (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl == "reference" or args.only_c5 or args.only in ("mf", "eval")):
        ap.error("--dump-outputs writes the timed NGCF step's outputs: not with --impl reference, --only-c5 or --only mf|eval")
    args.warmup = max(args.warmup, 3) if not args.only else args.warmup
    if args.impl == "reference":
        return run_reference(args)

    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    import __graft_entry__ as ge
    from yelprecommendation_b200 import _cabi, ops, parallel
    if not os.path.exists(_cabi.lib_path()):
        ge.build()
    lib = _cabi.load()
    from yelprecommendation_b200.data import synthetic as syn
    from yelprecommendation_b200.trainers import MFTrainer, NGCFTrainer

    pk = peaks()
    if args.only_c5:
        def _barrier():
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()

        def _max(ms):
            if world > 1:
                t = torch.tensor([ms], device=dev, dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                return float(t.item())
            return ms
        extra = {}
        config5_extras(extra, dev, rank, world, _barrier, _max, pk, args)
        if rank == 0:
            print(json.dumps({"n_gpus": world, "extra": extra}))
        if world > 1:
            dist.destroy_process_group()
        return 0
    w = build_workload()
    K, W = args.steps, args.warmup
    tu, tp_, tn = w.tri
    n_need = B * (K + W)
    reps = (n_need + len(tu) - 1) // len(tu)
    # each replica (rank) walks the pre-sampled triples from a different offset
    off = (rank * 7919 * B) % len(tu)
    take = lambda a: np.roll(np.tile(a, reps), -off)[:n_need]
    hu, hp, hn = take(tu), take(tp_), take(tn)
    du, dp, dn = (torch.from_numpy(a).to(dev) for a in (hu, hp, hn))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev, dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    if args.only == "eval":      # profiling aid: K fused evaluations of the planted MF tables, nothing else
        decsr = ops.DeviceEvalCSR(w.ecsr, dev, 10)
        Up, Vp = syn.planted_embeddings(w.inter)
        Ud, Vd = torch.from_numpy(Up).to(dev), torch.from_numpy(Vp).to(dev)
        Vt, _ = ops.transpose_items(Vd)
        for _ in range(W):
            ops.eval_topk_metrics(Ud, Vd, decsr, Vt)
        ms = timed(lambda i: ops.eval_topk_metrics(Ud, Vd, decsr, Vt), K)
        fb = getattr(ops.eval_topk_metrics, "last_fallback_rows", None)
        print(f"eval only: {ms / K:.3f} ms/eval  {w.ecsr.n_eval / (ms / K * 1e-3):.0f} users/s  "
              f"fallback_rows={int(fb.item()) if fb is not None else 'n/a'}", flush=True)
        rng = np.random.default_rng(0)
        Ur = torch.from_numpy(rng.standard_normal(Up.shape).astype(np.float32)).to(dev)
        Vr = torch.from_numpy(rng.standard_normal(Vp.shape).astype(np.float32)).to(dev)
        Vtr, _ = ops.transpose_items(Vr)
        ops.eval_topk_metrics(Ur, Vr, decsr, Vtr)
        ms = timed(lambda i: ops.eval_topk_metrics(Ur, Vr, decsr, Vtr), K)
        fb = getattr(ops.eval_topk_metrics, "last_fallback_rows", None)
        print(f"eval only (random N(0,1) tables): {ms / K:.3f} ms/eval  fallback_rows={int(fb.item()) if fb is not None else 'n/a'}",
              flush=True)
        return 0
    if args.only == "mf":        # profiling aid: one persistent launch of K SGD steps
        torch.manual_seed(42)
        mtr = MFTrainer(cfg(optimizer=os.environ.get("YR_BENCH_MF_OPT", "sgd"),
                            deterministic=os.environ.get("YR_BENCH_MF_DET", "0") == "1"), w.inter.num_items, w.inter.num_users)
        mtr.train_on_device(du[: B * W], dp[: B * W], dn[: B * W], B)
        ms = timed(lambda i: mtr.train_on_device(du[: B * K], dp[: B * K], dn[: B * K], B), 1)
        ms2 = timed(lambda i: mtr.train_on_device(du[: B * K], dp[: B * K], dn[: B * K], B), 1)
        print(f"mf only ({mtr.optimizer.name}, deterministic={getattr(mtr.cfg, 'deterministic', False)}): "
              f"{1e3 * ms / K:.2f} us/step first timed launch, {1e3 * ms2 / K:.2f} us/step second", flush=True)
        return 0

    # ------------------------------------------------------------------ NGCF training (headline)
    torch.manual_seed(42)
    ntr = NGCFTrainer(cfg(), w.inter.num_items, w.inter.num_users, w.L)
    st, _ = ntr._state()
    sl = torch.zeros(K + W, device=dev)

    def ngcf_step(i):
        s = i * B
        ntr.train_step_on_device(du[s:s + B], dp[s:s + B], dn[s:s + B], sl[i:i + 1], st)

    for i in range(W):
        ngcf_step(i)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    ms = timed(lambda i: ngcf_step(W + i), K)
    clocks = sampler.stop()
    barrier()
    ms = max_over_ranks(ms)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ntr, sl)
    ngcf_loss = ntr.loss_sum()
    value = world * K * B / (ms * 1e-3)
    if args.only == "ngcf":
        print(f"ngcf only: {ms / K:.3f} ms/step", flush=True)
        return 0

    # per-kernel timing of the step's pieces, each through its own C-ABI entry (same stream, CUDA events)
    import ctypes as C
    csr = ntr.model.csr(w.L)
    n = w.inter.num_users + w.inter.num_items
    E0 = ntr.model.embedding.weight.data
    X, Y, G, T = (torch.randn(n, D, device=dev) for _ in range(4))
    W1, W2 = ntr.model.W1[0].weight.data, ntr.model.W2[0].weight.data
    nnzL = csr.nnz
    csr_bytes = nnzL * 8 + (n + 1) * 4
    reps_k = 20
    pieces = {}

    def piece(name, fn, alg_bytes):
        for _ in range(3):
            fn(0)
        t = timed(fn, reps_k) / reps_k
        pieces[name] = {"ms": t, "alg_bytes": alg_bytes, "gbs": alg_bytes / (t * 1e-3) / 1e9}

    piece("spmm_csr", lambda i: ops.spmm_csr(csr.fwd, X, out=Y), csr_bytes + 2 * M_BYTES)
    piece("layer_fwd(spmm+dense)", lambda i: ops.ngcf_layer_fwd(csr, X, W1, W2), csr_bytes + 3 * M_BYTES)
    piece("layer_bwd(dense+reduce+spmmT)", lambda i: ops.ngcf_layer_bwd(csr, X, Y, T, G, W1, W2, torch.zeros_like(X)),
          csr_bytes + 7 * M_BYTES)
    optst = _cabi.make_opt("adam", 1e-4, 0.0, 5)
    m1, v1 = torch.zeros_like(X), torch.zeros_like(X)
    piece("dense_adam", lambda i: ops.dense_opt_step(X, G, m1, v1, optst), 6 * M_BYTES)
    step_alg_bytes = LAYERS * (csr_bytes + 3 * M_BYTES) + LAYERS * (csr_bytes + 7 * M_BYTES) + \
        3 * B * (LAYERS + 1) * D * 4 * 2 + 6 * M_BYTES
    # dominant kernel of the step: spmm_chunk_kernel<64> (2 x LAYERS launches per step, ~half of the step time —
    # profiles/ launch list). Its algorithmic HBM bytes are CSR + read X + write Y; what it actually lives on is the
    # L2->SM gather traffic nnz * d * 4 (X is L2-resident), reported next to it.
    dom = "spmm_csr"
    # per step: 2 (LAYERS - 1) full SpMMs (forward + backward of every layer but the last) + the last layer's forward
    # on the batch rows and its backward as a scatter from them (both ~half the non-zeros: popular positives)
    n_full_spmm = 2 * (LAYERS - 1)
    spmm_share = n_full_spmm * pieces[dom]["ms"] / (ms / K)
    gather_bytes = nnzL * D * 4
    roofline = {"bound": "hbm", "kernel": "spmm_chunk_kernel<64> (yr_spmm_csr)", "achieved": pieces[dom]["gbs"],
                "peak": pk["hbm"], "unit": "GB/s", "frac": pieces[dom]["gbs"] / pk["hbm"],
                # dram__bytes_read.sum + dram__bytes_write.sum of one launch, ncu --set full (profiles/): see DESIGN.md
                "traffic": NCU_SPMM_DRAM_BYTES, "peak_source": pk["src"],
                "launch_ms": pieces[dom]["ms"], "alg_bytes_per_launch": pieces[dom]["alg_bytes"],
                "launches_per_step": n_full_spmm, "share_of_step": spmm_share,
                "l2_gather": {"bytes_per_launch": gather_bytes, "achieved_GBps": gather_bytes / (pieces[dom]["ms"] * 1e-3) / 1e9,
                              "note": "every non-zero gathers one 256 B row of the L2-resident operand; this, not HBM, bounds the kernel"},
                "step": {"alg_bytes": step_alg_bytes, "achieved": step_alg_bytes / (ms / K * 1e-3) / 1e9,
                         "frac": step_alg_bytes / (ms / K * 1e-3) / 1e9 / pk["hbm"]},
                "pieces": {k: {"ms": round(v["ms"], 4), "GBps": round(v["gbs"], 1)} for k, v in pieces.items()}}
    del X, Y, G, T, m1, v1

    # ------------------------------------------------------------------ e2e through the public trainer API
    host_batches = syn.to_batches(hu, hp, hn, B)
    for b in host_batches[:W]:
        ntr.train([b])
    barrier()
    t0 = time.perf_counter()
    ms_e2e = timed(lambda i: ntr.train([host_batches[W + i]]), K)      # H2D ids + step + D2H loss, every step
    ms_e2e = max_over_ranks(max(ms_e2e, (time.perf_counter() - t0) * 1e3))
    e2e = {"value": world * K * B / (ms_e2e * 1e-3), "unit": UNIT, "h2d_bytes_per_step": 3 * B * 8,
           "d2h_bytes_per_step": 8 + 4, "api": "NGCFTrainer.train([batch]) per step (host int64 batches in, float loss out)"}

    extra = {}
    if not args.no_extra:
        # -------------------------------------------------------------- BPR-MF training (configs[0])
        torch.manual_seed(42)
        mtr = MFTrainer(cfg(), w.inter.num_items, w.inter.num_users)
        for name, okw, bpt in (("adam", dict(optimizer="adam"), None), ("sgd", dict(optimizer="sgd"), 1560)):
            torch.manual_seed(42)
            mtr = MFTrainer(cfg(**okw), w.inter.num_items, w.inter.num_users)
            steps_mf = max(K, 200)
            nt = B * steps_mf
            rp = (nt + len(tu) - 1) // len(tu)
            mu, mp, mn = (torch.from_numpy(np.tile(a, rp)[:nt]).to(dev) for a in (tu, tp_, tn))
            mtr.train_on_device(mu[: B * 8], mp[: B * 8], mn[: B * 8], B)
            barrier()
            ms_mf = max_over_ranks(timed(lambda i: mtr.train_on_device(mu, mp, mn, B), 1))
            mtr.loss_sum()
            tps = world * nt / (ms_mf * 1e-3)
            alg = (107.1e6 / B + 792) if name == "adam" else 1560.0
            extra[f"mf_train_{name}"] = {"value": tps, "unit": UNIT, "us_per_step": 1e3 * ms_mf / steps_mf,
                                         "alg_bytes_per_triple": alg, "hbm_frac": tps / world * alg / 1e9 / pk["hbm"],
                                         "note": "one persistent cooperative launch for all steps; tables (17.8 MB) are L2-resident"}
            if name == "sgd":
                hb = syn.to_batches(*[np.tile(a, rp)[:nt] for a in (tu, tp_, tn)], B)
                mtr.train(hb)                                   # first pass touches the pinned staging pages
                barrier()
                best = None
                for _ in range(3):
                    t0 = time.perf_counter()
                    mtr.train(hb)
                    torch.cuda.synchronize()
                    dt = time.perf_counter() - t0
                    best = dt if best is None else min(best, dt)
                extra["mf_train_sgd"]["e2e_value"] = world * nt / best
                extra["mf_train_sgd"]["e2e_note"] = "MFTrainer.train(host batches): best of 3 passes over 200 batches, wall clock"
            # CPU baseline of this leg (SURVEY 8(d)): the reference's MFTrainer.train loop (trainers/mf_trainer.py:100-116) as
            # oracle/torch_port.MFPort — same ATen CPU ops, dense embedding gradients, dense optimizer — 5 warm-up + 50 steps
            if rank == 0 and world == 1 and not args.no_cpu_baseline:
                from oracle.torch_port import MFPort
                torch.manual_seed(42)
                ref_m = MFTrainer(cfg(**okw), w.inter.num_items, w.inter.num_users).model
                port = MFPort(ref_m.user_embedding.weight.detach().cpu(), ref_m.item_embedding.weight.detach().cpu(),
                              optimizer=name, lr=1e-4, weight_decay=0.0)
                cb = syn.to_batches(*[a[: B * 55] for a in (tu, tp_, tn)], B)
                port.train(cb[:5])
                t0 = time.perf_counter()
                port.train(cb[5:55])
                dt = time.perf_counter() - t0
                extra[f"mf_train_{name}"]["cpu_baseline"] = {
                    "value": 50 * B / dt, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port", "ms_per_step": 1e3 * dt / 50,
                    "sample": "5 warm-up + 50 timed steps (batch 2048) of oracle/torch_port.MFPort.train on the host"}
                del port, ref_m
        # -------------------------------------------------------------- TF32 tensor peak of this GPU, measured here
        # (SURVEY 8(d): MEASURED_PEAKS.json has no TF32 figure). Library GEMM used as a yardstick only.
        tf32_peak = None
        try:
            old_tf32 = torch.backends.cuda.matmul.allow_tf32
            torch.backends.cuda.matmul.allow_tf32 = True
            ma = torch.randn(8192, 8192, device=dev)
            mb = torch.randn(8192, 8192, device=dev)
            for _ in range(2):
                torch.matmul(ma, mb)
            ms_mm = min(timed(lambda i: torch.matmul(ma, mb), 3) / 3 for _ in range(3))
            tf32_peak = 2.0 * 8192 ** 3 / (ms_mm * 1e-3) / 1e12
            torch.backends.cuda.matmul.allow_tf32 = old_tf32
            del ma, mb
            extra["tf32_matmul_peak"] = {"value": tf32_peak, "unit": "TFLOP/s", "how": "torch.matmul fp32 with TF32 on, 8192^3, best of 3 x 3"}
        except Exception as ex:
            extra["tf32_matmul_peak"] = {"error": repr(ex)}
        # -------------------------------------------------------------- full-catalog evaluation (configs[2])
        lo, hi = parallel.shard_range(w.ecsr.n_eval, rank, world)
        decsr_full = ops.DeviceEvalCSR(w.ecsr, dev, 10)
        decsr = decsr_full.slice(lo, hi) if world > 1 else decsr_full
        Up, Vp = syn.planted_embeddings(w.inter)
        Ud, Vd = torch.from_numpy(Up).to(dev), torch.from_numpy(Vp).to(dev)
        layers, _, _ = ntr.propagate()
        cat = ops.ngcf_concat(layers)
        for name, (Ue, Ve) in (("mf", (Ud, Vd)), ("ngcf", (cat[: w.inter.num_users], cat[w.inter.num_users:]))):
            Vt, _ = ops.transpose_items(Ve.contiguous())
            for _ in range(5):
                ops.eval_topk_metrics(Ue, Ve, decsr, Vt)
            barrier()
            reps_e = 10
            res = [None]
            calls = []
            for _ in range(reps_e):                           # per-call CUDA events; median reported, every call kept
                calls.append(timed(lambda i: res.__setitem__(0, ops.eval_topk_metrics(Ue, Ve, decsr, Vt)), 1))
            ms_ev = max_over_ranks(float(np.median(calls)))
            sums = parallel.all_reduce_sums(res[0][3])
            d_eff = Ue.shape[1]
            flops = 2.0 * w.ecsr.n_eval * w.inter.num_items * d_eff
            ups = w.ecsr.n_eval / (ms_ev * 1e-3)
            extra[f"eval_{name}"] = {"value": ups, "unit": "users/s", "ms": ms_ev, "d_eff": d_eff,
                                     "ms_calls": [round(x, 3) for x in calls],
                                     "tflops": flops / (ms_ev * 1e-3) / 1e12,
                                     "tensor_frac_vs_bf16_peak": flops / (ms_ev * 1e-3) / 1e12 / pk["bf16"],
                                     "tensor_frac_vs_tf32_measured": (flops / (ms_ev * 1e-3) / 1e12 / tf32_peak) if tf32_peak else None,
                                     "metrics": [round(x, 6) for x in ops.metrics_from_sums(sums.cpu(), w.ecsr.n_eval)],
                                     "fallback_rows": int(ops.eval_topk_metrics.last_fallback_rows.item())
                                     if hasattr(ops.eval_topk_metrics, "last_fallback_rows") else None,
                                     "item_slices": int(getattr(ops.eval_topk_metrics, "last_slices", 1)),
                                     "note": "tcgen05 TF32 filter + exact fp32 fma-chain re-score (bit-identical top-K to the "
                                             "FP32-pipe kernel); rows sharded over ranks, no data-path collective; a shard too small to "
                                             "fill the SMs is cut into item_slices concurrent launches that share their thresholds"}
            # e2e: host lists -> CSR upload -> kernel -> metrics back
        # CPU baselines of the evaluation leg (SURVEY 8(d)): the reference's per-user loop (trainers/mf_trainer.py:134-161:
        # score every item, mask, argpartition, metric.py) on the first 512 evaluation rows, for MF and — with the
        # propagate-once restatement — for NGCF
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            try:
                from oracle.torch_port import MFPort, NGCFPort
                n_cpu_ev = 512
                ev_uid = w.ecsr.eval_uid[:n_cpu_ev]
                mrows = [w.ecsr.mask_idx[w.ecsr.mask_ptr[e]:w.ecsr.mask_ptr[e + 1]] for e in range(n_cpu_ev)]
                arows = [w.ecsr.act_idx[w.ecsr.act_ptr[e]:w.ecsr.act_ptr[e + 1]].tolist() for e in range(n_cpu_ev)]
                port = MFPort(torch.from_numpy(Up), torch.from_numpy(Vp))
                port.evaluate(ev_uid[:16], mrows[:16], arows[:16])
                t0 = time.perf_counter()
                port.evaluate(ev_uid, mrows, arows)
                dt = time.perf_counter() - t0
                extra["eval_mf"]["cpu_baseline"] = {"value": n_cpu_ev / dt, "unit": "users/s", "cores": torch.get_num_threads(),
                                                    "kind": "port", "sample": f"first {n_cpu_ev} evaluation rows through "
                                                    "oracle/torch_port.MFPort.evaluate (per-user loop of the reference) on the host"}
                sdn = {k: v.detach().cpu().clone() for k, v in ntr.model.state_dict().items()}
                nport = NGCFPort(sdn["embedding.weight"], [sdn[f"W1.{l}.weight"] for l in range(LAYERS)],
                                 [sdn[f"W2.{l}.weight"] for l in range(LAYERS)], w.inter.num_users, w.L)
                t0 = time.perf_counter()
                nport.evaluate(ev_uid, mrows, arows)
                dt = time.perf_counter() - t0
                extra["eval_ngcf"]["cpu_baseline"] = {"value": n_cpu_ev / dt, "unit": "users/s", "cores": torch.get_num_threads(),
                                                      "kind": "port", "sample": f"one propagation + first {n_cpu_ev} evaluation rows "
                                                      "through oracle/torch_port.NGCFPort.evaluate on the host (the reference "
                                                      "re-propagates per user: ~20 s/user, Q12)"}
                del port, nport
            except Exception as ex:
                extra["eval_cpu_baseline"] = {"error": repr(ex)}
        t0 = time.perf_counter()
        mtr.evaluate(w.ecsr)
        extra["eval_mf"]["e2e_users_per_s_first_call"] = w.ecsr.n_eval / (time.perf_counter() - t0)
        t0 = time.perf_counter()
        mtr.evaluate(w.ecsr)
        extra["eval_mf"]["e2e_users_per_s"] = w.ecsr.n_eval / (time.perf_counter() - t0)

        # -------------------------------------------------------------- CDAE training (configs[3]), B = 32
        try:
            from yelprecommendation_b200.trainers import CDAETrainer
            nI, Bc, n_b = w.inter.num_items, 32, 48
            rng = np.random.default_rng(4 + rank)
            users = rng.choice(w.inter.num_users, Bc * n_b, replace=False)
            xin = np.zeros((Bc * n_b, nI), np.float32)
            neg = np.zeros_like(xin)
            for r, u in enumerate(users):
                items = w.split.train_items[w.split.train_ptr[u]:w.split.train_ptr[u + 1]]
                xin[r, items] = 1.0
                cand = rng.integers(0, nI, size=5 * len(items) + 8)
                cand = cand[xin[r, cand] == 0][: 5 * len(items)]
                neg[r, cand] = 1.0
            ccfg = cfg(hidden_size=64, corruption_level=0.6, hidden_activation="sigmoid", output_activation="sigmoid",
                       negative_sampling=True, loss_name="bce", lr=1e-4, optimizer="adam")
            torch.manual_seed(42)
            ctr = CDAETrainer(ccfg, nI, w.inter.num_users)
            hb = [{"user_id": torch.from_numpy(users[s:s + Bc].copy()), "input_mask": torch.from_numpy(xin[s:s + Bc]),
                   "negative_mask": torch.from_numpy(neg[s:s + Bc])} for s in range(0, Bc * n_b, Bc)]
            db = [{k: v.to(dev) for k, v in b.items()} for b in hb]
            ctr.train(db[:4])
            barrier()
            ms_c = max_over_ranks(timed(lambda i: ctr.train(db), 1))
            t0 = time.perf_counter()
            ctr.train(hb)                                   # host tensors: H2D of the dense masks every step
            torch.cuda.synchronize()
            e2e_c = time.perf_counter() - t0
            # the same batches as index lists (data/cdae_sparse.py, what a list-holding dataset yields): host -> device per step
            from yelprecommendation_b200.data.cdae_sparse import sparse_cdae_batch
            sbatches = [sparse_cdae_batch(b_) for b_ in hb]
            ctr.train(sbatches[:4])
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ctr.train(sbatches)
            torch.cuda.synchronize()
            e2e_s = time.perf_counter() - t0
            h2d_s = sum(sum(v.numel() * v.element_size() for v in b_.values()) for b_ in sbatches) / len(sbatches)
            extra["cdae_train"] = {"value": world * Bc * n_b / (ms_c * 1e-3), "unit": "users/s", "ms_per_step": ms_c / n_b,
                                   "batch": Bc, "e2e_value": world * Bc * n_b / e2e_c,
                                   "h2d_bytes_per_step": 2 * Bc * nI * 4,
                                   "e2e_value_index_lists": world * Bc * n_b / e2e_s, "h2d_bytes_per_step_index_lists": h2d_s,
                                   "note": "masks resident in HBM for `value`; e2e ships the dense [32 x 38,048] input/negative "
                                           "masks the reference's CDAEDataset yields; e2e_value_index_lists ships the same batches "
                                           "as item lists (yr_cdae_step_idx)"}
            if rank == 0 and world == 1 and not args.no_cpu_baseline:
                from oracle.torch_port import CDAEPort
                port = CDAEPort({k: v.detach().cpu() for k, v in ctr.model.state_dict().items()}, "adam", 1e-4)
                keeps = [(torch.rand(Bc, nI) >= 0.6).float() / 0.4 for _ in range(12)]
                port.train(hb[:2], keeps[:2])
                t0 = time.perf_counter()
                port.train(hb[2:12], keeps[2:12])
                extra["cdae_train"]["cpu_port_users_per_s"] = 10 * Bc / (time.perf_counter() - t0)
            del xin, neg, hb, db
        except Exception as ex:   # the CDAE row must not take the headline down
            extra["cdae_train"] = {"error": repr(ex)}

        # -------------------------------------------------------------- device-side input builders (SURVEY 8(f) 2-3)
        try:
            from yelprecommendation_b200.data.graph import build_laplacian, build_laplacian_csr_device
            from yelprecommendation_b200.data.sampler import DeviceTripleLoader
            iu, ii, ir = (torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in
                          (w.inter.user.astype(np.int64), w.inter.item.astype(np.int64), w.inter.rating.astype(np.float32)))
            build_laplacian_csr_device(iu, ii, ir, w.inter.num_users, w.inter.num_items)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            build_laplacian_csr_device(iu, ii, ir, w.inter.num_users, w.inter.num_items)
            torch.cuda.synchronize()
            t_dev = time.perf_counter() - t0
            extra["laplacian_build"] = {"value": len(w.inter.user) / t_dev, "unit": "interactions/s", "ms": 1e3 * t_dev,
                                        "note": "COO -> normalised CSR + SpMM plan, device kernels + host plan (wall clock)"}
            if rank == 0 and world == 1 and not args.no_cpu_baseline:
                t0 = time.perf_counter()
                build_laplacian(w.inter.user, w.inter.item, w.inter.rating, w.inter.num_users, w.inter.num_items)
                extra["laplacian_build"]["cpu_port_ms"] = 1e3 * (time.perf_counter() - t0)
            ld = DeviceTripleLoader.from_split(w.split, w.inter.num_items, batch_size=B, device=dev, seed=42)
            ld.epoch_triples()
            ms_s = timed(lambda i: ld.epoch_triples(), 5) / 5
            extra["negative_sampling"] = {"value": ld.user.numel() / (ms_s * 1e-3), "unit": "triples/s", "ms_per_epoch": ms_s,
                                          "note": "one epoch of (user, pos, fresh negative) triples sampled + shuffled in HBM"}
            # one whole epoch the way train.py drives it: fresh negatives + shuffle + every batch, nothing leaves HBM
            for oname in ("sgd", "adam"):
                torch.manual_seed(42)
                etr = MFTrainer(cfg(optimizer=oname), w.inter.num_items, w.inter.num_users)
                etr.train(ld)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                etr.train(ld)
                torch.cuda.synchronize()
                dt = time.perf_counter() - t0
                extra[f"mf_epoch_device_loader_{oname}"] = {
                    "value": ld.user.numel() / dt, "unit": UNIT, "ms_per_epoch": 1e3 * dt, "steps": len(ld),
                    "note": "MFTrainer.train(DeviceTripleLoader): sampling + shuffle + all steps of an epoch (wall clock)"}
            if rank == 0 and world == 1 and not args.no_cpu_baseline:
                t0 = time.perf_counter()
                syn.sample_triples(w.split, w.inter.num_items, seed=1)
                extra["negative_sampling"]["cpu_port_triples_per_s"] = ld.user.numel() / (time.perf_counter() - t0)
        except Exception as ex:
            extra["builders"] = {"error": repr(ex)}

        # -------------------------------------------------------------- BASELINE config 5 at its stated scale (configs[4])
        if not args.no_c5:
            try:
                config5_extras(extra, dev, rank, world, barrier, max_over_ranks, pk, args)
            except Exception as ex:
                extra["c5"] = {"error": repr(ex)}

    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        from oracle.torch_port import NGCFPort
        sd = {k: v.detach().cpu().clone() for k, v in ntr.model.state_dict().items()}
        port = NGCFPort(sd["embedding.weight"], [sd[f"W1.{l}.weight"] for l in range(LAYERS)],
                        [sd[f"W2.{l}.weight"] for l in range(LAYERS)], w.inter.num_users, w.L, "adam", 1e-4, 0.0)
        port.train(host_batches[:1])
        t0 = time.perf_counter()
        n_cpu = 0
        while n_cpu < 3 or (time.perf_counter() - t0 < 12 and n_cpu < 10):
            port.train(host_batches[1 + n_cpu:2 + n_cpu])
            n_cpu += 1
        dt = time.perf_counter() - t0
        cpu_baseline = {"value": n_cpu * B / dt, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                        "sample": f"{n_cpu} full NGCF train steps (batch 2048) of oracle/torch_port.NGCFPort on the host",
                        "ms_per_step": 1e3 * dt / n_cpu}
        # the reference VERBATIM (models/ngcf.py:61: a dense N x N torch.eye per layer per step, 19.4 GB each) — one step, only
        # when the host has the memory for it; reported next to the identity-hoisted port above, labelled
        try:
            import psutil
            if os.environ.get("YR_BENCH_VERBATIM", "1") == "1" and psutil.virtual_memory().available > 80e9:
                vport = NGCFPort(sd["embedding.weight"], [sd[f"W1.{l}.weight"] for l in range(LAYERS)],
                                 [sd[f"W2.{l}.weight"] for l in range(LAYERS)], w.inter.num_users, w.L, "adam", 1e-4, 0.0,
                                 verbatim_eye=True)
                t0 = time.perf_counter()
                vport.train(host_batches[:1])
                dtv = time.perf_counter() - t0
                cpu_baseline["verbatim_eye"] = {"value": B / dtv, "unit": UNIT, "s_per_step": dtv, "steps": 1,
                                                "note": "NGCFPort(verbatim_eye=True): the N x N identity built per layer per step"}
                del vport
        except Exception as ex:
            cpu_baseline["verbatim_eye"] = {"skipped": repr(ex)}

    if rank == 0:
        # kernels of one yr_ngcf_train_step (profiles/r02_launches_ngcf_step.csv): touched rows 1, forward 2 per layer, tail 2,
        # backward: last layer 4 (dense-on-rows, reduce, scatter, clear) + 4 per other layer (weight split, tensor-core
        # backward, reduce, transposed SpMM), optimizer 1
        launches_per_step = 1 + 2 * LAYERS + 2 + 4 + 4 * (LAYERS - 1) + 1
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W,
                "ms_per_step": ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic",
                "config": {"workload": WORKLOAD,
                           "parallelism": "1 GPU" if world == 1 else f"{world} independent replicas (replicas only)",
                           "l2": "per-step working set (~0.4 GB of E/LE/G/T/CSR/Adam state) exceeds the 126 MB L2; no flush"},
                "clocks": clocks, "e2e": e2e, "gpu_launches": launches_per_step * K, "roofline": roofline,
                "cpu_baseline": cpu_baseline, "extra": extra, "loss_sum": ngcf_loss,
                "lib": os.path.relpath(_cabi.lib_path(), ROOT)}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
