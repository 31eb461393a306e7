"""Top-K retrieval: the fused kernel (yr_recommend_topk) against the PyTorch reference, the reference against a brute-force
restatement, input checks, and evaluation through the retrieval kernel against the default evaluation.

Exactness: tables drawn from multiples of 1/4 in [-2, 2] make every dot product exact in fp32 (and bf16 holds the
values exactly), so any summation order gives the same scores — ids and scores must then match bit for bit, and the
many equal scores exercise the tie rule (lower item id first)."""
import os
import re
import subprocess

import numpy as np
import pytest
import torch

from util import cfg

I32, I64, F32 = torch.int32, torch.int64, torch.float32


def quarter_table(rng, n, d):
    return torch.from_numpy((rng.integers(-8, 9, size=(n, d)) / 4.0).astype(np.float32))


def seen_lists(rng, nU, nI, heavy=(), empty=()):
    """Random seen items; users in `heavy` have seen all but 5 items, users in `empty` nothing."""
    from yelprecommendation_b200.retrieval import SeenItems
    us, its = [], []
    for u in range(nU):
        if u in empty:
            continue
        if u in heavy:
            keep = rng.choice(nI, 5, replace=False)
            items = np.setdiff1d(np.arange(nI), keep)
        else:
            items = rng.choice(nI, int(rng.integers(1, min(nI, 200))), replace=False)
        us.append(np.full(items.size, u))
        its.append(items)
    return SeenItems.from_pairs(np.concatenate(us), np.concatenate(its), nU, nI)


def brute_force(U, V, uids, k, seen):
    """Per user: sorted((-score, id)) over the unseen items, padded — the definition, one Python sort per row."""
    S = U.double().numpy() @ V.double().numpy().T
    ids = np.full((len(uids), k), -1, np.int64)
    sc = np.full((len(uids), k), -np.inf, np.float32)
    for r, u in enumerate(uids):
        drop = set() if seen is None else set(seen.idx[seen.ptr[u]:seen.ptr[u + 1]].tolist())
        cand = sorted((-S[u, i], i) for i in range(V.shape[0]) if i not in drop)[:k]
        ids[r, :len(cand)] = [i for _, i in cand]
        sc[r, :len(cand)] = [-s for s, _ in cand]
    return ids, sc


# ------------------------------------------------------------------------------------------------------------------
# CPU: the reference path, the seen-items builder, input checks
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 7, 50])
def test_reference_matches_brute_force(k):
    from yelprecommendation_b200.retrieval import recommend_reference
    rng = np.random.default_rng(k)
    nU, nI, d = 12, 45, 8
    U, V = quarter_table(rng, nU, d), quarter_table(rng, nI, d)
    seen = seen_lists(rng, nU, nI, heavy={3}, empty={5})
    uids = np.array([0, 3, 5, 11, 3])
    ids, sc = recommend_reference(U, V, torch.from_numpy(uids), k, seen)
    bids, bsc = brute_force(U, V, uids, k, seen)
    assert np.array_equal(ids.numpy(), bids)
    assert np.array_equal(sc.numpy(), bsc)
    ids0, _ = recommend_reference(U, V, torch.from_numpy(uids), k, None)
    assert np.array_equal(ids0.numpy(), brute_force(U, V, uids, k, None)[0])


def test_seen_items_from_pairs():
    from yelprecommendation_b200.retrieval import SeenItems
    s = SeenItems.from_pairs([2, 0, 2, 2, 0], [5, 1, 3, 5, 0], num_users=4, num_items=6)
    assert s.ptr.tolist() == [0, 2, 2, 4, 4]
    assert s.idx.tolist() == [0, 1, 3, 5]
    with pytest.raises(IndexError):
        SeenItems.from_pairs([0], [6], num_users=4, num_items=6)
    with pytest.raises(IndexError):
        SeenItems.from_pairs([4], [0], num_users=4, num_items=6)


def test_recommender_on_cpu_tables_uses_the_reference():
    from yelprecommendation_b200.retrieval import Recommender, recommend_reference
    rng = np.random.default_rng(1)
    U, V = quarter_table(rng, 6, 8), quarter_table(rng, 30, 8)
    seen = seen_lists(rng, 6, 30)
    ids, sc = Recommender(U, V, seen).recommend([1, 4], 5)
    rids, rsc = recommend_reference(U, V, [1, 4], 5, seen)
    assert torch.equal(ids, rids) and torch.equal(sc, rsc)
    with pytest.raises(ValueError, match="exclude_seen"):
        Recommender(U, V).recommend([1], 5)
    with pytest.raises(ValueError, match="k must be"):
        Recommender(U, V, seen).recommend([1], 0)
    with pytest.raises(IndexError):
        Recommender(U, V, seen).recommend([6], 3)


def test_kernel_rejects_cpu_tensors():
    from yelprecommendation_b200 import _cabi, ops
    U, V = torch.zeros(4, 8), torch.zeros(9, 8)
    with pytest.raises(_cabi.YelprecError, match="CUDA"):
        ops.recommend_topk(U, V, torch.zeros(2, dtype=I64), 3)


def test_kernel_instances_are_built_for_sm100a():
    """The retrieval kernels are in the library as sm_100a SASS (one instance per table dtype, users-per-block and bias)."""
    from yelprecommendation_b200 import _cabi
    import __graft_entry__ as ge
    if not os.path.exists(_cabi.lib_path()):
        ge.build()
    out = subprocess.run(["cuobjdump", "-sass", _cabi.lib_path()], capture_output=True, text=True).stdout
    names = set(re.findall(r"Function : (\S*recommend\S*)", out))
    assert len([n for n in names if "recommend_topk_kernel" in n]) == 12, names   # fp32 / bf16 x TU x bias
    assert not any("_bias_kernel" in n for n in names), names
    assert any("recommend_merge_kernel" in n for n in names), names
    lib = _cabi.load()
    assert lib.yr_recommend_ws_bytes(0, 10, 5) == 0


# ------------------------------------------------------------------------------------------------------------------
# GPU: fused kernel == reference
# ------------------------------------------------------------------------------------------------------------------
# (nU, nI, d, B): item counts off the 256-item tile; 20,011 items are cut into several item splits and merged
SIZES = [(40, 1000, 8, 40), (300, 5003, 64, 300), (64, 20011, 32, 7), (600, 20011, 128, 600)]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("k", [1, 20, 100, 300, 1000])
def test_fused_equals_reference_exact(size, k, dtype):
    from yelprecommendation_b200.retrieval import Recommender, recommend_reference
    nU, nI, d, B = size
    rng = np.random.default_rng(nI + k + d)
    U, V = quarter_table(rng, nU, d), quarter_table(rng, nI, d)
    seen = seen_lists(rng, nU, nI, heavy={1, nU - 1}, empty={0, 2})
    uids = rng.integers(0, nU, size=B)
    uids[:4] = [0, 1, 2, nU - 1]
    Ud, Vd = U.cuda().to(dtype), V.cuda().to(dtype)
    uid = torch.from_numpy(uids).cuda()
    for exclude in (True, False):
        ids, sc = Recommender(Ud, Vd, seen).recommend(uid, k, exclude_seen=exclude)
        rids, rsc = recommend_reference(U, V, torch.from_numpy(uids), k, seen if exclude else None)
        assert ids.shape == (B, k) and ids.dtype == I64 and sc.dtype == F32
        assert torch.equal(ids.cpu(), rids), (exclude, (ids.cpu() != rids).nonzero()[:5])
        assert torch.equal(sc.cpu(), rsc)
    # user 1 has seen all but 5 items: 5 real entries, then padding
    ids, sc = Recommender(Ud, Vd, seen).recommend(uid[1:2], k)
    n = min(k, 5)
    assert (ids[0, :n] >= 0).all() and (ids[0, n:] == -1).all() and torch.isinf(sc[0, n:]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("k", [20, 100])
def test_fused_gaussian_tables(k):
    """Gaussian fp32 tables: the kernel's fma chain and the reference's matmul round differently in the last bits, so scores
    agree to 1e-5 relative and ids wherever the reference's scores are not within that of a neighbour."""
    from yelprecommendation_b200.retrieval import Recommender, recommend_reference
    g = torch.Generator().manual_seed(k)
    nU, nI, d = 500, 38048, 64
    U, V = torch.randn(nU, d, generator=g), torch.randn(nI, d, generator=g)
    seen = seen_lists(np.random.default_rng(k), nU, nI)
    uids = torch.arange(0, nU, 3)
    ids, sc = Recommender(U.cuda(), V.cuda(), seen).recommend(uids.cuda(), k)
    rids, rsc = recommend_reference(U.double(), V.double(), uids, k, seen)
    scale = rsc.abs().max().item()
    assert (sc.cpu().double() - rsc).abs().max().item() <= 1e-5 * scale
    r = rsc.numpy()
    gap = np.minimum(np.abs(np.diff(r, axis=1, prepend=np.inf)), np.abs(np.diff(r, axis=1, append=-np.inf)))
    clear = gap > 1e-5 * scale
    assert np.array_equal(ids.cpu().numpy()[clear], rids.numpy()[clear])
    assert clear.mean() > 0.9


@pytest.mark.gpu
def test_k_beyond_catalog_pads():
    from yelprecommendation_b200.retrieval import Recommender
    rng = np.random.default_rng(3)
    U, V = quarter_table(rng, 5, 16).cuda(), quarter_table(rng, 30, 16).cuda()
    seen = seen_lists(rng, 5, 30, empty={0})
    ids, sc = Recommender(U, V, seen).recommend([0, 1], 40)
    assert (ids[0, :30] >= 0).all() and (ids[0, 30:] == -1).all()
    assert torch.isinf(sc[0, 30:]).all() and (sc[0, 30:] < 0).all()
    n_unseen = 30 - int(seen.ptr[2] - seen.ptr[1])
    assert (ids[1, :n_unseen] >= 0).all() and (ids[1, n_unseen:] == -1).all()


@pytest.mark.gpu
def test_exclude_seen_false_is_plain_topk():
    from yelprecommendation_b200.retrieval import Recommender
    g = torch.Generator().manual_seed(0)
    U, V = torch.randn(64, 32, generator=g).cuda(), torch.randn(9000, 32, generator=g).cuda()
    seen = seen_lists(np.random.default_rng(0), 64, 9000)
    uids = torch.arange(64, device="cuda")
    ids, sc = Recommender(U, V, seen).recommend(uids, 50, exclude_seen=False)
    tv, ti = torch.topk(U @ V.T, 50, dim=1)
    assert torch.allclose(sc, tv, rtol=1e-5, atol=1e-5)
    assert (ids == ti).float().mean().item() > 0.99     # ids differ only where two scores are within rounding


@pytest.mark.gpu
def test_bad_inputs_raise():
    from yelprecommendation_b200 import _cabi, ops
    U, V = torch.zeros(4, 8, device="cuda"), torch.zeros(9, 8, device="cuda")
    u = torch.tensor([0, 3], device="cuda")
    with pytest.raises(_cabi.YelprecError, match="CUDA"):
        ops.recommend_topk(U, V, u.cpu(), 3)
    for k in (0, -1, 1025, 2.5):
        with pytest.raises(ValueError, match="k must be"):
            ops.recommend_topk(U, V, u, k)
    with pytest.raises(IndexError, match="out of range"):
        ops.recommend_topk(U, V, torch.tensor([0, 4], device="cuda"), 3)
    with pytest.raises(IndexError, match="out of range"):
        ops.recommend_topk(U, V, torch.tensor([-1], device="cuda"), 3)
    with pytest.raises(TypeError):
        ops.recommend_topk(U.double(), V.double(), u, 3)
    with pytest.raises(TypeError):
        ops.recommend_topk(U, V.bfloat16(), u, 3)
    with pytest.raises(ValueError, match="multiple of 8"):
        ops.recommend_topk(torch.zeros(4, 12, device="cuda"), torch.zeros(9, 12, device="cuda"), u, 3)
    with pytest.raises(ValueError, match="offsets"):
        ops.recommend_topk(U, V, u, 3, torch.zeros(3, dtype=I32, device="cuda"), torch.zeros(1, dtype=I32, device="cuda"))
    ids, sc = ops.recommend_topk(U, V, torch.zeros(0, dtype=I64, device="cuda"), 3)
    assert ids.shape == (0, 3)


# ------------------------------------------------------------------------------------------------------------------
# GPU: evaluation through the retrieval kernel
# ------------------------------------------------------------------------------------------------------------------
def _fixture():
    from yelprecommendation_b200.data import synthetic as syn
    from yelprecommendation_b200.data.graph import build_eval_csr, build_laplacian
    inter = syn.make_interactions(num_users=300, num_items=400, nnz=6000, seed=3, n_clusters=4)
    split = syn.split_per_user(inter, seed=42)
    tu, tp, tn = syn.sample_triples(split, inter.num_items, seed=42)
    batches = syn.to_batches(tu, tp, tn, 256)[:4]
    csrs = {m: build_eval_csr(*syn.eval_lists(split, m), inter.num_items) for m in ("valid", "test")}
    L = build_laplacian(inter.user, inter.item, inter.rating, inter.num_users, inter.num_items)
    return inter, split, batches, csrs, L


@pytest.mark.gpu
@pytest.mark.parametrize("top_n", [10, 20])
def test_mf_metrics_through_retrieval_equal_default(top_n):
    from yelprecommendation_b200.trainers import MFTrainer
    inter, split, batches, csrs, _ = _fixture()
    torch.manual_seed(0)
    tr = MFTrainer(cfg(optimizer="adam", top_n=top_n), inter.num_items, inter.num_users)
    tr.train(batches)
    for mode, csr in csrs.items():
        tr.cfg.eval_mode = None
        want = tr.evaluate(csr, mode)
        want_topk = tr.last_topk.clone()
        tr.cfg.eval_mode = "retrieval"
        got = tr.evaluate(csr, mode)
        assert got == want, (mode, got, want)
        assert torch.equal(tr.last_topk, want_topk)


@pytest.mark.gpu
def test_ngcf_metrics_through_retrieval_equal_default():
    from yelprecommendation_b200.retrieval import SeenItems, recommend_reference
    from yelprecommendation_b200.trainers import NGCFTrainer
    inter, split, batches, csrs, L = _fixture()
    torch.manual_seed(1)
    tr = NGCFTrainer(cfg(optimizer="adam"), inter.num_items, inter.num_users, L)
    tr.train(batches[:2])
    want = tr.evaluate(csrs["valid"])
    tr.cfg.eval_mode = "retrieval"
    assert tr.evaluate(csrs["valid"]) == want
    # the trainer's recommender ranks with the same tables
    seen = SeenItems.from_split(split, inter.num_items)
    rec = tr.recommender(seen)
    uids = torch.arange(0, inter.num_users, 7, device="cuda")
    ids, sc = rec.recommend(uids, 20)
    rids, rsc = recommend_reference(rec.user_emb.double(), rec.item_emb.double(), uids, 20, seen)
    assert (sc.double() - rsc).abs().max().item() <= 1e-5 * rsc.abs().max().item()
    assert (ids == rids).float().mean().item() > 0.99
