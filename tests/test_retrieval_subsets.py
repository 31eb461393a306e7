"""Subset-restricted top-K retrieval: the subset kernel (yr_recommend_subset_topk) against the PyTorch reference and against
the unrestricted kernel with the items outside each row's subset excluded, the reference against a brute-force
restatement, the subset builder and input checks. Exactness as in test_retrieval: quarter tables make every score exact."""
import os
import re
import subprocess

import numpy as np
import pytest
import torch

from test_retrieval import SIZES, brute_force, quarter_table, seen_lists

I32, I64, F32 = torch.int32, torch.int64, torch.float32


def subsets_of(lists, nI):
    from yelprecommendation_b200.retrieval import ItemSubsets
    s = np.concatenate([np.full(len(x), g) for g, x in enumerate(lists)] + [np.zeros(0, np.int64)]).astype(np.int64)
    i = np.concatenate([np.asarray(x, np.int64) for x in lists] + [np.zeros(0, np.int64)])
    return ItemSubsets.from_pairs(s, i, len(lists), nI)


def brute_force_subset(U, V, uids, k, seen, subsets, sub):
    """Per row: brute_force over the row's subset (all items for -1), the items outside it treated as seen."""
    from yelprecommendation_b200.retrieval import SeenItems
    nI = V.shape[0]
    ids = np.full((len(uids), k), -1, np.int64)
    sc = np.full((len(uids), k), -np.inf, np.float32)
    for r, (u, g) in enumerate(zip(uids, sub)):
        drop = set() if seen is None else set(seen.idx[seen.ptr[u]:seen.ptr[u + 1]].tolist())
        if g >= 0:
            drop |= set(range(nI)) - set(subsets.idx[subsets.ptr[g]:subsets.ptr[g + 1]].tolist())
        one = SeenItems.from_pairs(np.full(len(drop), u, np.int64), np.array(sorted(drop), np.int64), U.shape[0], nI)
        ids[r:r + 1], sc[r:r + 1] = brute_force(U, V, [u], k, one)
    return ids, sc


def exclusion_csr(seen, subsets, uids, sub, nI, dev):
    """Per batch row: the seen items plus every item outside the row's subset (the seen_by_row workaround)."""
    rows = []
    for u, g in zip(uids, sub):
        drop = set(seen.idx[seen.ptr[u]:seen.ptr[u + 1]].tolist()) if seen is not None else set()
        if g >= 0:
            drop |= set(range(nI)) - set(subsets.idx[subsets.ptr[g]:subsets.ptr[g + 1]].tolist())
        rows.append(np.array(sorted(drop), np.int32))
    ptr = np.zeros(len(rows) + 1, np.int64)
    ptr[1:] = np.cumsum([len(x) for x in rows])
    idx = np.concatenate(rows + [np.zeros(0, np.int32)])
    return torch.from_numpy(ptr.astype(np.int32)).to(dev), torch.from_numpy(idx).to(dev)


# ------------------------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------------------------
def test_item_subsets_from_pairs():
    from yelprecommendation_b200.retrieval import ItemSubsets
    s = ItemSubsets.from_pairs([2, 0, 2, 2, 0, 3], [5, 1, 3, 5, 0, 2], num_subsets=5, num_items=6)
    assert s.ptr.tolist() == [0, 2, 2, 4, 5, 5]
    assert s.idx.tolist() == [0, 1, 3, 5, 2]
    assert s.num_subsets == 5 and s.num_items == 6 and s.max_len == 2
    e = ItemSubsets.from_pairs([], [], num_subsets=3, num_items=6)
    assert e.ptr.tolist() == [0, 0, 0, 0] and e.max_len == 0
    with pytest.raises(IndexError, match="item id"):
        ItemSubsets.from_pairs([0], [6], num_subsets=4, num_items=6)
    with pytest.raises(IndexError, match="subset id"):
        ItemSubsets.from_pairs([4], [0], num_subsets=4, num_items=6)
    with pytest.raises(IndexError):
        ItemSubsets.from_pairs([-1], [0], num_subsets=4, num_items=6)


@pytest.mark.parametrize("k", [1, 7, 50])
def test_reference_with_subsets_matches_brute_force(k):
    from yelprecommendation_b200.retrieval import recommend_reference
    rng = np.random.default_rng(10 + k)
    nU, nI, d = 12, 45, 8
    U, V = quarter_table(rng, nU, d), quarter_table(rng, nI, d)
    seen = seen_lists(rng, nU, nI, heavy={3}, empty={5})
    # overlapping subsets, an empty one, one smaller than k, the whole catalog
    subsets = subsets_of([np.arange(0, 30), np.arange(20, 45, 2), [], [4, 9, 11], np.arange(nI)], nI)
    uids = np.array([0, 3, 5, 11, 3, 7, 8, 0])
    sub = np.array([0, 1, -1, 2, 3, 4, -1, 1])
    for s in (seen, None):
        ids, sc = recommend_reference(U, V, torch.from_numpy(uids), k, s, subsets, torch.from_numpy(sub))
        bids, bsc = brute_force_subset(U, V, uids, k, s, subsets, sub)
        assert np.array_equal(ids.numpy(), bids)
        assert np.array_equal(sc.numpy(), bsc)
    # a single int applies to every row
    ids, _ = recommend_reference(U, V, uids, k, seen, subsets, 1)
    assert np.array_equal(ids.numpy(), brute_force_subset(U, V, uids, k, seen, subsets, [1] * len(uids))[0])


def test_recommender_on_cpu_tables_with_subsets():
    from yelprecommendation_b200.retrieval import ItemSubsets, Recommender, recommend_reference
    rng = np.random.default_rng(2)
    U, V = quarter_table(rng, 6, 8), quarter_table(rng, 30, 8)
    seen = seen_lists(rng, 6, 30)
    subsets = subsets_of([np.arange(10), np.arange(5, 30, 3)], 30)
    rec = Recommender(U, V, seen, subsets=subsets)
    ids, sc = rec.recommend([1, 4, 2], 5, subset=[1, -1, 0])
    rids, rsc = recommend_reference(U, V, [1, 4, 2], 5, seen, subsets, [1, -1, 0])
    assert torch.equal(ids, rids) and torch.equal(sc, rsc)
    # subset=None is the unrestricted call
    assert torch.equal(rec.recommend([1, 4], 5)[0], recommend_reference(U, V, [1, 4], 5, seen)[0])
    with pytest.raises(ValueError, match="subsets"):
        Recommender(U, V, seen).recommend([1], 5, subset=0)
    with pytest.raises(ValueError, match="items"):
        Recommender(U, V, seen, subsets=ItemSubsets.from_pairs([0], [1], 1, 31))
    with pytest.raises(IndexError, match="subset id"):
        rec.recommend([1, 2], 5, subset=[0, 2])
    with pytest.raises(IndexError, match="subset id"):
        rec.recommend([1, 2], 5, subset=-2)
    with pytest.raises(ValueError, match="subset ids for"):
        rec.recommend([1, 2], 5, subset=[0, 1, 0])


def test_subset_kernel_rejects_cpu_tensors():
    from yelprecommendation_b200 import _cabi, ops
    U, V = torch.zeros(4, 8), torch.zeros(9, 8)
    z = torch.zeros(2, dtype=I64)
    with pytest.raises(_cabi.YelprecError, match="CUDA"):
        ops.recommend_subset_topk(U, V, z, 3, torch.zeros(2, dtype=I32), torch.zeros(1, dtype=I32), z, 9)


def test_subset_kernel_is_built_for_sm100a():
    """One subset kernel instance per table dtype and users-per-block, next to the 6 unrestricted ones."""
    from yelprecommendation_b200 import _cabi
    import __graft_entry__ as ge
    if not os.path.exists(_cabi.lib_path()):
        ge.build()
    out = subprocess.run(["cuobjdump", "-sass", _cabi.lib_path()], capture_output=True, text=True).stdout
    names = set(re.findall(r"Function : (\S*recommend\S*)", out))
    assert len([n for n in names if "recommend_subset_kernel" in n]) == 6, names
    assert len([n for n in names if "recommend_topk_kernel" in n]) == 6, names
    assert any("recommend_subset_plan_kernel" in n for n in names), names
    assert _cabi.load().yr_recommend_subset_ws_bytes(0, 3, 10, 5) == 0


# ------------------------------------------------------------------------------------------------------------------
# GPU: subset kernel == reference (quarter tables, exact)
# ------------------------------------------------------------------------------------------------------------------
def _subset_lists(rng, nI):
    """Sizes 0, 1, 255, 256, 257, 7 (below most k), ~15,000 (several splits, when the catalog has it), the whole
    catalog, and two overlapping ones."""
    def pick(n):
        return np.sort(rng.choice(nI, min(n, nI), replace=False))
    half = pick(nI // 2)
    return [pick(0), pick(1), pick(255), pick(256), pick(257), pick(7), pick(15000), np.arange(nI),
            half, np.union1d(half[: len(half) // 2], pick(nI // 3))]


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("k", [1, 20, 100, 1000])
def test_subset_equals_reference_exact(size, k, dtype):
    from yelprecommendation_b200.retrieval import Recommender, recommend_reference
    nU, nI, d, B = size
    rng = np.random.default_rng(nI + k + d + 1)
    U, V = quarter_table(rng, nU, d), quarter_table(rng, nI, d)
    lists = _subset_lists(rng, nI)
    subsets = subsets_of(lists, nI)
    G = len(lists)
    # user 1 has seen all but 5 items of subset 9 (and nothing else); users 0 and 2 have no history
    heavy = np.setdiff1d(lists[9], rng.choice(lists[9], min(5, len(lists[9])), replace=False))
    base = seen_lists(rng, nU, nI, empty={0, 1, 2})
    us = np.concatenate([np.repeat(np.arange(nU), np.diff(base.ptr.numpy())), np.full(len(heavy), 1)])
    its = np.concatenate([base.idx.numpy(), heavy])
    from yelprecommendation_b200.retrieval import SeenItems
    seen = SeenItems.from_pairs(us, its, nU, nI)
    n = max(B, 2 * G + 4)
    uids = rng.integers(0, nU, size=n)
    sub = rng.integers(-1, G, size=n)
    uids[:4], sub[:4] = [0, 1, 2, 1], [3, 9, -1, 0]          # user 1 twice, in two groups
    Ud, Vd = U.cuda().to(dtype), V.cuda().to(dtype)
    rec = Recommender(Ud, Vd, seen, subsets=subsets)
    mixes = {"mixed": sub, "one group": np.full(n, 6), "all different": np.arange(n) % (G + 1) - 1}
    for name, s in mixes.items():
        perm = rng.permutation(n)                            # shuffled rows: results follow request order
        u, s = uids[perm], s[perm]
        for exclude in (True, False):
            for arg in (s, torch.from_numpy(s).cuda()):      # host ids (exact split count) and device ids
                ids, sc = rec.recommend(torch.from_numpy(u).cuda(), k, exclude_seen=exclude, subset=arg)
                rids, rsc = recommend_reference(U, V, torch.from_numpy(u), k, seen if exclude else None, subsets, s)
                assert ids.shape == (n, k) and ids.dtype == I64 and sc.dtype == F32
                assert torch.equal(ids.cpu(), rids), (name, exclude, (ids.cpu() != rids).nonzero()[:5])
                assert torch.equal(sc.cpu(), rsc), (name, exclude)
    # user 1 in subset 9: 5 real entries, then padding
    ids, sc = rec.recommend([1], k, subset=9)
    m = min(k, 5, len(lists[9]))
    assert (ids[0, :m] >= 0).all() and (ids[0, m:] == -1).all() and torch.isinf(sc[0, m:]).all()


# ------------------------------------------------------------------------------------------------------------------
# GPU: bit-identical to the unrestricted kernel with the exclusion CSR, on Gaussian tables
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("d", [64, 256])
@pytest.mark.parametrize("k", [20, 100])
def test_subset_bit_identical_to_exclusion_csr(d, k):
    from yelprecommendation_b200 import ops
    from yelprecommendation_b200.retrieval import Recommender
    g = torch.Generator().manual_seed(d + k)
    nU, nI = 400, 38048
    U, V = torch.randn(nU, d, generator=g).cuda(), torch.randn(nI, d, generator=g).cuda()
    rng = np.random.default_rng(d)
    seen = seen_lists(rng, nU, nI)
    lists = [np.sort(rng.choice(nI, n, replace=False)) for n in (50, 380, 1500, 3800, 12000, 0, 30)]
    subsets = subsets_of(lists, nI)
    B = 300
    uids = rng.integers(0, nU, size=B)
    sub = rng.integers(-1, len(lists), size=B)
    rec = Recommender(U, V, seen, subsets=subsets)
    ids, sc = rec.recommend(torch.from_numpy(uids).cuda(), k, subset=sub)
    ptr, idx = exclusion_csr(seen, subsets, uids, sub, nI, "cuda")
    xids, xsc = ops.recommend_topk(U, V, torch.from_numpy(uids).cuda(), k, ptr, idx, seen_by_row=True)
    assert torch.equal(ids, xids), (ids != xids).nonzero()[:5]
    assert torch.equal(sc, xsc)
    whole = torch.from_numpy(sub == -1).cuda()
    uids_whole = torch.from_numpy(uids).cuda()[whole]
    wids, wsc = rec.recommend(uids_whole, k)
    assert torch.equal(ids[whole], wids) and torch.equal(sc[whole], wsc)
    aids, asc = rec.recommend(uids_whole, k, subset=-1)
    assert torch.equal(aids, wids) and torch.equal(asc, wsc)


@pytest.mark.gpu
def test_subset_bad_inputs_raise():
    from yelprecommendation_b200 import ops
    U, V = torch.zeros(4, 8, device="cuda"), torch.zeros(9, 8, device="cuda")
    sptr = torch.tensor([0, 2, 5], dtype=I32, device="cuda")
    sidx = torch.tensor([1, 3, 0, 4, 8], dtype=I32, device="cuda")
    u = torch.tensor([0, 3], device="cuda")
    s = torch.tensor([1, -1], device="cuda")
    ids, sc = ops.recommend_subset_topk(U, V, u, 3, sptr, sidx, s, 9)
    assert ids.shape == (2, 3)
    with pytest.raises(IndexError, match="user id"):
        ops.recommend_subset_topk(U, V, torch.tensor([0, 4], device="cuda"), 3, sptr, sidx, s, 9)
    with pytest.raises(IndexError, match="subset id"):
        ops.recommend_subset_topk(U, V, u, 3, sptr, sidx, torch.tensor([2, 0], device="cuda"), 9)
    with pytest.raises(IndexError, match="subset id"):
        ops.recommend_subset_topk(U, V, u, 3, sptr, sidx, torch.tensor([0, -2], device="cuda"), 9)
    with pytest.raises(ValueError, match="subset ids for"):
        ops.recommend_subset_topk(U, V, u, 3, sptr, sidx, s[:1], 9)
    with pytest.raises(TypeError):
        ops.recommend_subset_topk(U, V, u, 3, sptr, sidx, s.float(), 9)
    with pytest.raises(ValueError, match="int32 CSR"):
        ops.recommend_subset_topk(U, V, u, 3, sptr.long(), sidx, s, 9)
    with pytest.raises(ValueError, match="k must be"):
        ops.recommend_subset_topk(U, V, u, 0, sptr, sidx, s, 9)
    ids, sc = ops.recommend_subset_topk(U, V, torch.zeros(0, dtype=I64, device="cuda"), 3, sptr, sidx,
                                        torch.zeros(0, dtype=I64, device="cuda"), 9)
    assert ids.shape == (0, 3) and sc.shape == (0, 3)


@pytest.mark.gpu
def test_trainer_recommenders_with_subsets():
    from util import cfg
    from test_retrieval import _fixture
    from yelprecommendation_b200.retrieval import Recommender, SeenItems
    from yelprecommendation_b200.trainers import MFTrainer, NGCFTrainer
    inter, split, batches, _, L = _fixture()
    seen = SeenItems.from_split(split, inter.num_items)
    rng = np.random.default_rng(4)
    subsets = subsets_of([np.sort(rng.choice(inter.num_items, n, replace=False)) for n in (30, 120, 5)], inter.num_items)
    uids = torch.arange(0, inter.num_users, 5, device="cuda")
    sub = rng.integers(-1, 3, size=uids.numel())
    torch.manual_seed(0)
    mf = MFTrainer(cfg(optimizer="adam"), inter.num_items, inter.num_users)
    mf.train(batches[:2])
    torch.manual_seed(1)
    ngcf = NGCFTrainer(cfg(optimizer="adam"), inter.num_items, inter.num_users, L)
    ngcf.train(batches[:1])
    for tr in (mf, ngcf):
        rec = tr.recommender(seen, subsets)
        ids, sc = rec.recommend(uids, 10, subset=sub)
        want = Recommender(rec.user_emb, rec.item_emb, seen, subsets).recommend(uids, 10, subset=sub)
        assert torch.equal(ids, want[0]) and torch.equal(sc, want[1])
