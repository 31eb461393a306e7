"""Group retrieval: least-misery and average top-K for groups of users (yr_recommend_group_topk,
recommend_group_reference, Recommender.recommend_group, CDAERecommender.recommend_group).

The reference is checked against a brute-force restatement, one numpy float32 scalar operation at a time. On
quarter-valued tables (multiples of 1/4 in [-2, 2], exact in bf16 too) every member score is exact in any summation
order, and the fold (min, or adds in member order and one division) is the same sequence of correctly rounded fp32
operations in the kernel and the reference: ids and scores must agree bit for bit. A group of one must be recommend's
row bit for bit on any table."""
import copy
import os
import re
import subprocess

import numpy as np
import pytest
import torch

from test_retrieval import _fixture, quarter_table, seen_lists
from test_retrieval_cdae import cdae_model, quarter_params
from util import cfg

I32, I64, F32 = torch.int32, torch.int64, torch.float32


def random_groups(rng, G, nU, sizes=(1, 2, 31, 32)):
    """G groups as lists of user ids in random order: the given sizes first, then random sizes 1 to 32 (capped by nU)."""
    out = []
    for g in range(G):
        m = sizes[g] if g < len(sizes) else int(rng.integers(1, 33))
        out.append(rng.choice(nU, min(m, nU), replace=False).tolist())
    return out


def brute_group(U, V, groups, k, agg, seen=None, subsets=None, subset=None, bias=None):
    """The definition, one numpy float32 scalar operation at a time: per item, each member's score (a float64 dot product,
    exact on quarter tables, rounded to float32, then + bias in float32), folded by min (NaN-propagating) or by adds in
    ascending member order and one division; the returnable items sorted by (-score, id)."""
    f = np.float32
    U64, V64 = U.double().numpy(), V.double().numpy()
    nI = V.shape[0]
    ids = np.full((len(groups), k), -1, np.int64)
    sc = np.full((len(groups), k), -np.inf, np.float32)
    for r, grp in enumerate(groups):
        mem = sorted(set(grp))
        drop = set()
        if seen is not None:
            for u in mem:
                drop |= set(seen.idx[seen.ptr[u]:seen.ptr[u + 1]].tolist())
        s_id = None if subset is None else (subset if np.ndim(subset) == 0 else subset[r])
        allowed = range(nI) if s_id is None or s_id == -1 else \
            subsets.idx[subsets.ptr[s_id]:subsets.ptr[s_id + 1]].tolist()
        cand = []
        for i in allowed:
            if i in drop:
                continue
            a = None
            for u in mem:
                s = f(U64[u] @ V64[i])
                if bias is not None:
                    s = f(s + f(bias[i]))
                if a is None:
                    a = s
                elif agg == "min":
                    a = s if (np.isnan(s) or s < a) and not np.isnan(a) else a
                else:
                    a = f(a + s)
            if agg == "mean":
                a = f(a / f(len(mem)))
            if np.isnan(a) or a == -np.inf:
                continue
            cand.append((-float(a), i, a))
        cand.sort()
        cand = cand[:k]
        ids[r, :len(cand)] = [i for _, i, _ in cand]
        sc[r, :len(cand)] = [a for _, _, a in cand]
    return ids, sc


def city_subsets(rng, nI, n=6):
    """n subsets of the catalog; subset 2 is empty."""
    from yelprecommendation_b200.retrieval import ItemSubsets
    city = rng.integers(0, n, nI)
    city[city == 2] = 3
    return ItemSubsets.from_pairs(city, np.arange(nI), n, nI)


# ------------------------------------------------------------------------------------------------------------------
# CPU: the reference against the brute force, the builders, the CPU path of Recommender
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("agg", ["min", "mean"])
@pytest.mark.parametrize("k", [1, 7, 50])
def test_reference_matches_brute_force(agg, k):
    from yelprecommendation_b200.retrieval import recommend_group_reference
    rng = np.random.default_rng(k + len(agg))
    nU, nI, d = 40, 45, 8
    U, V = quarter_table(rng, nU, d), quarter_table(rng, nI, d)
    b = quarter_table(rng, nI, 1)[:, 0]
    seen = seen_lists(rng, nU, nI, heavy={3}, empty={5})
    subsets = city_subsets(rng, nI)
    groups = random_groups(rng, 9, nU, sizes=(1, 2, 3, 31, 32)) + [[5], [3, 5]]
    sub = rng.integers(-1, 6, len(groups))
    sub[:3] = [-1, 2, 4]
    for use_seen in (False, True):
        for bias in (None, b):
            for subset in (None, 4, sub):
                kw = dict(seen=seen if use_seen else None, subsets=subsets, subset=subset, item_bias=bias)
                ids, sc = recommend_group_reference(U, V, groups, k, agg, **kw)
                bids, bsc = brute_group(U, V, groups, k, agg, seen if use_seen else None, subsets, subset,
                                        None if bias is None else bias.numpy())
                assert np.array_equal(ids.numpy(), bids), (use_seen, bias is None, subset)
                assert np.array_equal(sc.numpy(), bsc)


def test_reference_nan_and_mean_rounding():
    """A NaN member score makes the least-misery score NaN (never returned); the mean divides once, correctly rounded."""
    from yelprecommendation_b200.retrieval import recommend_group_reference
    U = torch.zeros(4, 8)
    U[0, 0] = float("inf")                                     # user 0: +inf, or NaN where v_0 = 0 (item 1)
    U[1, 1] = U[2, 2] = U[3, 3] = 1.0
    V = torch.zeros(4, 8)
    V[0, :4] = torch.tensor([1.0, 1.0, 0.0, 0.0])
    V[1, :4] = torch.tensor([0.0, 3.0, 3.0, 3.0])
    V[2, :4] = 2.0
    V[3, :4] = torch.tensor([1.0, 0.5, 0.25, 0.25])
    ids, sc = recommend_group_reference(U, V, [[0, 1, 2], [1, 2]], 4, "min")
    assert ids[0].tolist() == [2, 3, 0, -1] and sc[0].tolist()[:3] == [2.0, 0.25, 0.0]
    assert ids[1].tolist() == [1, 2, 3, 0]                     # user 0's NaN is not in group 1
    ids, sc = recommend_group_reference(U, V, [[1, 2, 3]], 4, "mean")
    assert ids[0].tolist() == [1, 2, 0, 3]                     # items 0 and 3 tie at 1 / 3: the lower id first
    assert sc[0, 2].item() == sc[0, 3].item() == float(np.float32(1.0) / np.float32(3.0))


def test_user_groups_builders():
    from yelprecommendation_b200.retrieval import UserGroups
    g = UserGroups.from_lists([[42, 3, 17, 3], [9, 8], [5]], 50)
    assert g.ptr.tolist() == [0, 3, 5, 6] and g.members.tolist() == [3, 17, 42, 8, 9, 5]
    assert g.ptr.dtype == I32 and g.members.dtype == I64 and g.num_groups == 3 and g.num_users == 50
    p = UserGroups.from_pairs([1, 0, 1, 0, 0], [9, 42, 8, 3, 17], 2, 50)
    assert p.ptr.tolist() == [0, 3, 5] and p.members.tolist() == [3, 17, 42, 8, 9]
    assert UserGroups.from_lists([list(range(32))], 32).members.tolist() == list(range(32))
    assert UserGroups.from_lists([[7] * 40], 8).members.tolist() == [7]       # duplicates dropped before the cap
    with pytest.raises(ValueError, match="1 to 32"):
        UserGroups.from_lists([[1, 2], []], 50)
    with pytest.raises(ValueError, match="1 to 32"):
        UserGroups.from_lists([list(range(33))], 50)
    with pytest.raises(ValueError, match="1 to 32"):
        UserGroups.from_pairs([0, 0], [1, 2], 2, 50)           # group 1 has no members
    with pytest.raises(IndexError, match="user id"):
        UserGroups.from_lists([[1, 50]], 50)
    with pytest.raises(IndexError, match="user id"):
        UserGroups.from_lists([[-1]], 50)
    with pytest.raises(IndexError, match="group id"):
        UserGroups.from_pairs([2], [1], 2, 50)


def test_recommender_on_cpu_tables_uses_the_reference():
    from yelprecommendation_b200.retrieval import (ItemLocations, Recommender, UserGroups, recommend_group_reference,
                                                   recommend_reference)
    rng = np.random.default_rng(3)
    nU, nI = 40, 60
    U, V = quarter_table(rng, nU, 16), quarter_table(rng, nI, 16)
    seen = seen_lists(rng, nU, nI)
    subsets = city_subsets(rng, nI)
    loc = ItemLocations.from_degrees(rng.uniform(40, 41, nI), rng.uniform(-75, -74, nI))
    rec = Recommender(U, V, seen, subsets=subsets, locations=loc)
    groups = random_groups(rng, 6, nU)
    for agg in ("min", "mean"):
        for kw in ({}, {"subset": 1}, {"exclude_seen": False}):
            ids, sc = rec.recommend_group(groups, 9, agg, **kw)
            excl = kw.get("exclude_seen", True)
            rids, rsc = recommend_group_reference(U, V, groups, 9, agg, seen if excl else None, subsets,
                                                  kw.get("subset"))
            assert torch.equal(ids, rids) and torch.equal(sc, rsc), (agg, kw)
        for u in (0, 7, 39):                                   # a group of one is recommend
            ids, sc = rec.recommend_group(UserGroups.from_lists([[u]], nU), 9, agg, subset=3)
            kids, ksc = recommend_reference(U, V, [u], 9, seen, subsets, 3)
            assert torch.equal(ids, kids) and torch.equal(sc, ksc)
    shuffled = [list(reversed(g)) for g in groups]
    assert all(torch.equal(a, b) for a, b in zip(rec.recommend_group(groups, 9, "min"),
                                                 rec.recommend_group(shuffled, 9, "min")))
    with pytest.raises(ValueError, match="near is not supported"):
        rec.recommend_group(groups, 5, near=(40.5, -74.5), radius_km=3.0)
    with pytest.raises(ValueError, match="near is not supported"):
        rec.recommend_group(groups, 5, radius_km=3.0)
    with pytest.raises(ValueError, match="agg"):
        rec.recommend_group(groups, 5, agg="max")
    with pytest.raises(ValueError, match="k must be"):
        rec.recommend_group(groups, 0)
    with pytest.raises(ValueError, match="exclude_seen"):
        Recommender(U, V).recommend_group(groups, 5)
    with pytest.raises(ValueError, match="covers|cover"):
        rec.recommend_group(UserGroups.from_lists([[1]], nU + 1), 5)
    with pytest.raises(IndexError, match="user id"):
        rec.recommend_group([[1, nU]], 5)
    with pytest.raises(IndexError, match="subset id"):
        rec.recommend_group(groups, 5, subset=6)


def test_ops_reject_cpu_tensors_and_bad_agg():
    from yelprecommendation_b200 import _cabi, ops
    U, V = torch.zeros(4, 8), torch.zeros(9, 8)
    with pytest.raises(_cabi.YelprecError, match="CUDA"):
        ops.recommend_group_topk(U, V, torch.tensor([0, 1], dtype=I32), torch.zeros(1, dtype=I64), 3, "mean")
    with pytest.raises(ValueError, match="agg"):
        ops.group_agg("median")
    assert ops.RECOMMEND_GROUP_MAX_MEMBERS == 32


def test_kernel_instances_are_built_for_sm100a():
    """fp32 / bf16 x groups per block 16 / 8 / 4 x bias, agg a runtime argument: 12 instances of sm_100a SASS, with no
    stack and no spills."""
    from yelprecommendation_b200 import _cabi
    import __graft_entry__ as ge
    if not os.path.exists(_cabi.lib_path()):
        ge.build()
    out = subprocess.run(["cuobjdump", "-sass", _cabi.lib_path()], capture_output=True, text=True).stdout
    names = set(re.findall(r"Function : (\S*recommend_group_kernel\S*)", out))
    assert len(names) == 12, names
    lib = _cabi.load()
    assert lib.yr_recommend_group_ws_bytes(0, 0, 10, 5) == 0
    log = os.path.join(os.path.dirname(_cabi.lib_path()), "..", "csrc", "build", "retrieval.ptxas.log")
    if os.path.exists(log):
        entries = [e for e in re.split(r"Compiling entry function ", open(log).read())[1:]
                   if "recommend_group_kernel" in e.split("'")[1]]
        assert len(entries) == 12
        for e in entries:
            assert re.search(r"0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads", e), e[:300]


# ------------------------------------------------------------------------------------------------------------------
# GPU: the kernel against the reference
# ------------------------------------------------------------------------------------------------------------------
# (nU, nI, d, G): test_retrieval's SIZES (item counts off the tile; 20,011 items take several splits) and d = 1024
SIZES = [(40, 1000, 8, 40), (300, 5003, 64, 300), (64, 20011, 32, 7), (600, 20011, 128, 600), (50, 5003, 1024, 20)]


def _check(rec, Uref, Vref, groups, k, agg, seen, subsets=None, subset=None, bias=None):
    """Kernel (rec on the device) == reference (Uref, Vref: fp32 tables on the device), ids and scores bit for bit."""
    from yelprecommendation_b200.retrieval import recommend_group_reference
    ids, sc = rec(groups, k, agg)
    rids, rsc = recommend_group_reference(Uref, Vref, groups, k, agg, seen, subsets, subset, item_bias=bias)
    assert ids.shape == (len(groups) if isinstance(groups, list) else groups.num_groups, k) and ids.dtype == I64
    assert torch.equal(ids, rids), (agg, (ids != rids).nonzero()[:5])
    assert torch.equal(sc, rsc), agg


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("k", [1, 20, 100, 300, 1000])
def test_kernel_equals_reference_exact(size, k, dtype):
    from yelprecommendation_b200 import ops
    from yelprecommendation_b200.retrieval import UserGroups
    nU, nI, d, G = size
    rng = np.random.default_rng(nI + k + d)
    U, V = quarter_table(rng, nU, d).cuda(), quarter_table(rng, nI, d).cuda()
    b = quarter_table(rng, nI, 1)[:, 0].cuda()
    seen = seen_lists(rng, nU, nI, heavy={1, nU - 1}, empty={0, 2})
    groups = UserGroups.from_lists([[0], [1], [2, 1]] + random_groups(rng, G, nU), nU)   # sizes 1, 2, 31, 32, mixed
    Ud, Vd = U.to(dtype), V.to(dtype)
    gptr, mem = groups.on("cuda")
    sptr, sidx = seen.on("cuda")
    for agg in ("min", "mean"):
        for with_seen in (True, False):
            for bias in (None, b):
                sp, si = (sptr, sidx) if with_seen else (None, None)
                _check(lambda g, kk, a: ops.recommend_group_topk(Ud, Vd, gptr, mem, kk, a, sp, si, item_bias=bias),
                       U, V, groups, k, agg, seen if with_seen else None, bias=bias)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("k", [5, 300])
def test_subsets_equal_reference_exact(k, dtype):
    """Subset ids -1, an empty subset and mixed ids in one call (host and device ids), and one id for every group."""
    from yelprecommendation_b200.retrieval import Recommender
    rng = np.random.default_rng(k)
    nU, nI, d = 200, 20011, 64
    U, V = quarter_table(rng, nU, d).cuda(), quarter_table(rng, nI, d).cuda()
    seen = seen_lists(rng, nU, nI, heavy={1})
    subsets = city_subsets(rng, nI)
    groups = random_groups(rng, 150, nU) + [[1], [1, 2]]
    rec = Recommender(U.to(dtype), V.to(dtype), seen, subsets=subsets)
    sub = rng.integers(-1, 6, len(groups))
    sub[:4] = [-1, 2, 0, 5]
    for subset in (sub, torch.from_numpy(sub).cuda(), 2, -1, 4):
        for agg in ("min", "mean"):
            _check(lambda g, kk, a: rec.recommend_group(g, kk, a, subset=subset), U, V, groups, k, agg, seen, subsets,
                   subset.cpu() if torch.is_tensor(subset) else subset)
    ids, _ = rec.recommend_group(groups, k, subset=2)
    assert (ids == -1).all()                                  # the empty subset: all padding


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_group_of_one_equals_recommend(dtype):
    """Gaussian tables, where summation order matters: a group of one is recommend's row bit for bit, with and without
    seen lists, with a subset, and with a per-item bias (recommend_topk_ex)."""
    from yelprecommendation_b200 import ops
    from yelprecommendation_b200.retrieval import Recommender, UserGroups
    g = torch.Generator().manual_seed(1)
    nU, nI, d = 500, 30011, 64
    U, V = torch.randn(nU, d, generator=g).cuda().to(dtype), torch.randn(nI, d, generator=g).cuda().to(dtype)
    bias = torch.randn(nI, generator=g).cuda()
    rng = np.random.default_rng(1)
    seen = seen_lists(rng, nU, nI)
    subsets = city_subsets(rng, nI)
    rec = Recommender(U, V, seen, subsets=subsets)
    uid = torch.arange(0, nU, 3)
    ones = UserGroups.from_lists([[u] for u in uid.tolist()], nU)
    for agg in ("min", "mean"):
        for kw in ({}, {"exclude_seen": False}, {"subset": 3}):
            for k in (20, 100):
                ids, sc = rec.recommend_group(ones, k, agg, **kw)
                kids, ksc = rec.recommend(uid, k, **kw)
                assert torch.equal(ids, kids) and torch.equal(sc, ksc), (agg, kw, k)
        gptr, mem = ones.on("cuda")
        sptr, sidx = seen.on("cuda")
        ids, sc = ops.recommend_group_topk(U, V, gptr, mem, 20, agg, sptr, sidx, item_bias=bias)
        kids, ksc = ops.recommend_topk(U, V, uid.cuda(), 20, sptr, sidx, item_bias=bias)
        assert torch.equal(ids, kids) and torch.equal(sc, ksc), agg


@pytest.mark.gpu
def test_member_order_does_not_matter():
    from yelprecommendation_b200.retrieval import Recommender, UserGroups
    g = torch.Generator().manual_seed(2)
    nU, nI, d = 300, 9000, 32
    U, V = torch.randn(nU, d, generator=g).cuda(), torch.randn(nI, d, generator=g).cuda()
    rng = np.random.default_rng(2)
    rec = Recommender(U, V, seen_lists(rng, nU, nI))
    groups = random_groups(rng, 64, nU)
    shuffled = [rng.permutation(x).tolist() for x in groups]
    pairs = UserGroups.from_pairs(np.repeat(np.arange(64), [len(x) for x in groups])[::-1],
                                  np.concatenate(groups)[::-1], 64, nU)
    for agg in ("min", "mean"):
        ids, sc = rec.recommend_group(groups, 30, agg)
        for other in (shuffled, pairs):
            oids, osc = rec.recommend_group(other, 30, agg)
            assert torch.equal(ids, oids) and torch.equal(sc, osc), agg


@pytest.mark.gpu
def test_nan_rows_are_never_returned():
    """A NaN user row makes every least-misery and mean score of its groups NaN: all padding. A NaN item row is never
    returned to any group."""
    from yelprecommendation_b200.retrieval import Recommender
    rng = np.random.default_rng(4)
    nU, nI, d = 50, 1000, 16
    U, V = quarter_table(rng, nU, d), quarter_table(rng, nI, d)
    U[7] = float("nan")
    V[[3, 600, 999]] = float("nan")
    V[5, 0] = float("nan")
    rec = Recommender(U.cuda(), V.cuda())
    groups = [[7], [7, 8, 9], [8, 9], [1, 2, 3, 4]]
    for agg in ("min", "mean"):
        ids, sc = rec.recommend_group(groups, 1000, agg, exclude_seen=False)
        assert (ids[:2] == -1).all() and torch.isinf(sc[:2]).all(), agg
        for r in (2, 3):
            row = ids[r][ids[r] >= 0].cpu().numpy()
            assert len(row) == nI - 4 and not set(row.tolist()) & {3, 5, 600, 999}, agg
            assert not torch.isnan(sc[r]).any()


def _group_call(lib, U, V, gptr, mem, K, agg, err, sub=None):
    from yelprecommendation_b200 import _cabi
    from yelprecommendation_b200._cabi import dptr, stream_ptr
    G = gptr.numel() - 1
    nI = V.shape[0]
    ids = torch.empty(G, K, dtype=I64, device="cuda")
    sc = torch.empty(G, K, dtype=F32, device="cuda")
    sptr, sidx, sid = sub if sub is not None else (None, None, None)
    NS = sptr.numel() - 1 if sub is not None else 0
    nbytes = lib.yr_recommend_group_ws_bytes(G, NS, nI, K)
    ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device="cuda")
    rc = lib.yr_recommend_group_topk(U.data_ptr(), U.shape[0], V.data_ptr(), nI, V.shape[1], _cabi.YR_DTYPE_F32,
                                     dptr(gptr), G, dptr(mem), mem.numel(), agg, dptr(sptr), dptr(sidx), NS, nI,
                                     dptr(sid), None, None, K, dptr(ids), dptr(sc), dptr(ws), nbytes, dptr(err),
                                     stream_ptr(), None)
    torch.cuda.synchronize()
    return rc, ids, sc


@pytest.mark.gpu
def test_bad_inputs_raise_and_the_error_word():
    """Bad member ids, subset ids and group sizes set their bits and pad their rows only; good calls leave the word 0."""
    from yelprecommendation_b200 import _cabi, ops
    from yelprecommendation_b200.retrieval import Recommender
    lib = _cabi.load()
    rng = np.random.default_rng(5)
    U, V = quarter_table(rng, 20, 8).cuda(), quarter_table(rng, 5000, 8).cuda()
    err = torch.zeros(1, dtype=I32, device="cuda")
    i32 = lambda x: torch.tensor(x, dtype=I32, device="cuda")
    i64 = lambda x: torch.tensor(x, dtype=I64, device="cuda")
    good_ptr, good_mem = i32([0, 2, 3]), i64([1, 5, 7])
    for agg in (_cabi.YR_GROUP_MIN, _cabi.YR_GROUP_MEAN):
        rc, ids, _ = _group_call(lib, U, V, good_ptr, good_mem, 10, agg, err)
        assert rc == 0 and int(err.item()) == 0 and (ids >= 0).all()
    rc, ids, _ = _group_call(lib, U, V, good_ptr, i64([1, 20, 7]), 10, 1, err)     # member 20 of 20 users
    assert rc == 0 and int(err.item()) == 1 and (ids[0] == -1).all() and (ids[1] >= 0).all()
    err.zero_()
    rc, ids, _ = _group_call(lib, U, V, i32([0, 0, 33, 34]), i64(list(range(20)) * 2), 10, 0, err)   # 0 and 33
    assert rc == 0 and int(err.item()) == 4 and (ids[:2] == -1).all() and (ids[2] >= 0).all()
    err.zero_()
    sub = (i32([0, 2, 4]), i32([1, 2, 3, 4]), i64([0, 2]))                            # subset 2 of 2
    rc, ids, _ = _group_call(lib, U, V, good_ptr, good_mem, 10, 0, err, sub)
    assert rc == 0 and int(err.item()) == 2 and (ids[1] == -1).all() and sorted(ids[0, :2].tolist()) == [1, 2]
    assert (ids[0, 2:] == -1).all()
    err.zero_()
    rc, ids, _ = _group_call(lib, U, V, good_ptr, good_mem, 10, 2, err)               # no such aggregation
    assert rc == 1000 and int(err.item()) == 0
    rc, _, _ = _group_call(lib, U, V, good_ptr, good_mem, 10, 0, err, (i32([0, 2, 4]), i32([1, 2, 3, 4]), i64([0, -1])))
    assert rc == 0 and int(err.item()) == 0

    with pytest.raises(IndexError, match="member id"):
        ops.recommend_group_topk(U, V, good_ptr, i64([1, 20, 7]), 5, "min")
    with pytest.raises(ValueError, match="1 to 32"):
        ops.recommend_group_topk(U, V, i32([0, 0, 3]), good_mem, 5, "mean")
    with pytest.raises(IndexError, match="subset id"):
        ops.recommend_group_topk(U, V, good_ptr, good_mem, 5, "mean", subset_ptr=sub[0], subset_idx=sub[1],
                                 subset_ids=sub[2])
    with pytest.raises(ValueError, match="agg"):
        ops.recommend_group_topk(U, V, good_ptr, good_mem, 5, "max")
    with pytest.raises(ValueError, match="go together"):
        ops.recommend_group_topk(U, V, good_ptr, good_mem, 5, "min", subset_ids=sub[2])
    rec = Recommender(U, V)
    with pytest.raises(IndexError, match="user id"):
        rec.recommend_group([[1, 20]], 5, exclude_seen=False)
    with pytest.raises(ValueError, match="near is not supported"):
        rec.recommend_group([[1, 2]], 5, exclude_seen=False, near=(0.0, 0.0), radius_km=1.0)
    ids, sc = ops.recommend_group_topk(U, V, i32([0]), i64([]), 5, "min")
    assert ids.shape == (0, 5) and sc.shape == (0, 5)


# ------------------------------------------------------------------------------------------------------------------
# GPU: the CDAE and the trainers
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("h", [64, 1024])
@pytest.mark.parametrize("k", [1, 20, 300])
def test_cdae_recommend_group_equals_reference_exact(h, k):
    from yelprecommendation_b200.retrieval import CDAERecommender, cdae_recommend_group_reference
    rng = np.random.default_rng(h + k)
    nU, nI = 40, 300
    model = cdae_model(nU, nI, h, "identity")
    quarter_params(model, rng)
    seen = seen_lists(rng, nU, nI, heavy={1}, empty={2})
    subsets = city_subsets(rng, nI)
    groups = random_groups(rng, 12, nU) + [[2], [1, 2], [5, 6, 5]]
    cpu = copy.deepcopy(model).cpu()
    rec = CDAERecommender(model, seen, subsets=subsets)
    for agg in ("min", "mean"):
        for excl in (True, False):
            for subset in (None, 3):
                ids, sc = rec.recommend_group(groups, k, agg, exclude_seen=excl, subset=subset)
                rids, rsc = cdae_recommend_group_reference(cpu, groups, k, seen, agg, excl, subsets, subset)
                assert torch.equal(ids.cpu(), rids) and torch.equal(sc.cpu(), rsc), (agg, excl, subset)


@pytest.mark.gpu
def test_trainers_recommend_group():
    """MF, NGCF (concatenated width 256) and CDAE recommenders: a group of one is recommend, and groups never get an item
    any member has seen."""
    from yelprecommendation_b200.retrieval import SeenItems
    from yelprecommendation_b200.trainers import CDAETrainer, MFTrainer, NGCFTrainer
    inter, split, batches, csrs, L = _fixture()
    seen = SeenItems.from_split(split, inter.num_items)
    torch.manual_seed(0)
    mf = MFTrainer(cfg(optimizer="adam"), inter.num_items, inter.num_users)
    mf.train(batches)
    ngcf = NGCFTrainer(cfg(optimizer="adam"), inter.num_items, inter.num_users, L)
    ngcf.train(batches[:2])
    cdae = CDAETrainer(cfg(optimizer="adam", hidden_size=64, corruption_level=0.0, hidden_activation="sigmoid",
                           output_activation="sigmoid", negative_sampling=True, loss_name="bce"),
                       inter.num_items, inter.num_users)
    rng = np.random.default_rng(6)
    uid = list(range(0, inter.num_users, 7))
    groups = [rng.choice(inter.num_users, int(rng.integers(2, 9)), replace=False).tolist() for _ in range(40)]
    for name, tr in (("mf", mf), ("ngcf", ngcf), ("cdae", cdae)):
        rec = tr.recommender(seen)
        for agg in ("min", "mean"):
            ids1, sc1 = rec.recommend_group([[u] for u in uid], 10, agg)
            kids, ksc = rec.recommend(uid, 10)
            assert torch.equal(ids1, kids) and torch.equal(sc1, ksc), (name, agg)
            ids, sc = rec.recommend_group(groups, 10, agg)
            h = ids.cpu().numpy()
            for r, grp in enumerate(groups):
                row = h[r][h[r] >= 0]
                assert len(row) == 10 and len(set(row.tolist())) == 10, name
                for u in grp:
                    assert not set(row.tolist()) & set(seen.idx[seen.ptr[u]:seen.ptr[u + 1]].tolist()), (name, agg)
