"""Diverse retrieval: Maximal Marginal Relevance re-ranking of a top-K pool (yr_recommend_mmr, mmr_reference,
recommend_diverse).

The reference is checked against a brute-force restatement in numpy float32 scalars. On quarter-valued tables (multiples
of 1/4 in [-2, 2], exact in bf16 too) every dot product and every sum of squares is exact in any summation order, so the
kernel and the reference agree bit for bit for every lam. On Gaussian tables the kernel's picks are checked against a
float64 greedy wherever its best and second-best marginal relevances are clearly apart."""
import os
import re
import subprocess

import numpy as np
import pytest
import torch

from test_retrieval import _fixture, quarter_table, seen_lists
from util import cfg

I32, I64, F32 = torch.int32, torch.int64, torch.float32


def quarter_pool(rng, B, N, nI, pad_frac=0.15, sort=True):
    """Pools of B rows x N positions: random item ids (duplicates allowed), -1 in the middle and at the end of rows,
    quarter-valued scores with many ties; sorted by (score desc, id asc) like recommend's output when `sort`."""
    ids = rng.integers(0, nI, size=(B, N)).astype(np.int64)
    ids[rng.random((B, N)) < pad_frac] = -1
    if N > 2:
        ids[:, -1] = -1
    if B > 2:
        ids[1] = -1                                            # an all-padding row
    sc = (rng.integers(-12, 13, size=(B, N)) / 4.0).astype(np.float32)
    sc[ids < 0] = -np.inf
    if sort:
        for b in range(B):
            o = sorted(range(N), key=lambda j: (ids[b, j] < 0, -sc[b, j], ids[b, j]))
            ids[b], sc[b] = ids[b, o], sc[b, o]
    return torch.from_numpy(ids), torch.from_numpy(sc)


def brute_mmr(V, ids, sc, k, lam):
    """The definition, one numpy float32 scalar operation at a time."""
    f = np.float32
    V = V.numpy().astype(np.float32)
    ids, sc = ids.numpy(), sc.numpy()
    a = f(lam)
    c = f(1) - a
    B, N = ids.shape
    out_ids = np.full((B, k), -1, np.int64)
    out_sc = np.full((B, k), -np.inf, np.float32)

    def nrm(i):
        ss = f(sum(float(x) * float(x) for x in V[i]))        # exact on quarter tables
        return f(0) if ss == 0 else f(1) / np.sqrt(ss)

    for b in range(B):
        p, r = ids[b], sc[b]
        n = [nrm(i) if i >= 0 else f(0) for i in p]

        def sim(i, j):
            return f(float(V[p[i]].astype(np.float64) @ V[p[j]].astype(np.float64))) * (n[i] * n[j])

        picked = []
        for t in range(k):
            cand = [j for j in range(N) if p[j] >= 0 and j not in picked]
            if not cand:
                break

            def m(j):
                pen = max(sim(j, s) for s in picked) if picked else f(0)
                v = a * r[j] - c * pen
                return f(-np.inf) if np.isnan(v) else (f(0) if v == 0 else v)

            s = max(cand, key=lambda j: (m(j), -j))
            picked.append(s)
            out_ids[b, t], out_sc[b, t] = p[s], r[s]
    return out_ids, out_sc


# ------------------------------------------------------------------------------------------------------------------
# CPU: the reference against the brute force, input checks, the CPU path of Recommender
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("lam", [0.0, 0.3, 0.5, 1.0])
@pytest.mark.parametrize("N,k", [(12, 5), (9, 9), (16, 14)])
def test_reference_matches_brute_force(lam, N, k):
    from yelprecommendation_b200.retrieval import mmr_reference
    rng = np.random.default_rng(int(lam * 10) + N)
    nI, d = 20, 8
    V = quarter_table(rng, nI, d)
    V[3] = 0                                                   # zero-norm items
    V[7] = 0
    V[5] = V[4]                                                # two items, one direction
    for sort in (True, False):
        ids, sc = quarter_pool(rng, 6, N, nI, pad_frac=0.3, sort=sort)
        ids[0, :4] = torch.tensor([3, 3, 7, 5])                # duplicate ids, zero rows
        ids[2, 1] = -1                                         # a hole in the middle
        sc[0, :4] = 1.0                                        # equal relevance
        sc[2, 1] = float("-inf")
        got_ids, got_sc = mmr_reference(V, ids, sc, k, lam)
        want_ids, want_sc = brute_mmr(V, ids, sc, k, lam)
        assert np.array_equal(got_ids.numpy(), want_ids), (lam, sort, got_ids, want_ids)
        assert np.array_equal(got_sc.numpy(), want_sc)
        assert (got_ids[1] == -1).all() and torch.isinf(got_sc[1]).all()   # all padding
    if lam == 1.0:                                             # pure relevance: the first k entries of a sorted pool
        ids, sc = quarter_pool(rng, 6, N, nI, sort=True)
        got_ids, got_sc = mmr_reference(V, ids, sc, k, lam)
        assert torch.equal(got_ids, ids[:, :k]) and torch.equal(got_sc, sc[:, :k])


def test_reference_pads_short_rows():
    from yelprecommendation_b200.retrieval import mmr_reference
    V = quarter_table(np.random.default_rng(0), 10, 8)
    ids = torch.tensor([[4, -1, 2, -1, -1], [-1, -1, -1, -1, -1]])
    sc = torch.tensor([[1.0, float("-inf"), 0.5, float("-inf"), float("-inf")], [float("-inf")] * 5])
    got_ids, got_sc = mmr_reference(V, ids, sc, 4, 0.5)
    assert got_ids[0, 2:].tolist() == [-1, -1] and sorted(got_ids[0, :2].tolist()) == [2, 4]
    assert (got_ids[1] == -1).all() and torch.isinf(got_sc).sum() == 6
    ids0, sc0 = mmr_reference(V, torch.zeros(0, 5, dtype=I64), torch.zeros(0, 5), 3, 0.5)
    assert ids0.shape == (0, 3) and sc0.shape == (0, 3)


def test_bad_inputs_raise_on_cpu():
    from yelprecommendation_b200 import _cabi, ops
    from yelprecommendation_b200.retrieval import Recommender, mmr_reference
    rng = np.random.default_rng(2)
    U, V = quarter_table(rng, 6, 8), quarter_table(rng, 30, 8)
    seen = seen_lists(rng, 6, 30)
    rec = Recommender(U, V, seen)
    ids, sc = quarter_pool(rng, 3, 10, 30)
    for lam in (-0.1, 1.5, float("nan"), None, "0.5", True):
        with pytest.raises(ValueError, match="lam"):
            mmr_reference(V, ids, sc, 3, lam)
        with pytest.raises(ValueError, match="lam"):
            rec.recommend_diverse([1, 2], 3, lam=lam)
    for k in (0, 11, 2.5, -1):
        with pytest.raises(ValueError, match="k must be"):
            mmr_reference(V, ids, sc, k, 0.5)
    with pytest.raises(ValueError, match="k must be"):
        rec.recommend_diverse([1], 0)
    for pool in (2, 1025, 3.5):
        with pytest.raises(ValueError, match="pool"):
            rec.recommend_diverse([1], 3, pool=pool)
    with pytest.raises(ValueError, match="pool must hold"):
        mmr_reference(V, torch.zeros(2, 1025, dtype=I64), torch.zeros(2, 1025), 3, 0.5)
    with pytest.raises(ValueError, match="exclude_seen"):
        Recommender(U, V).recommend_diverse([1], 3)
    with pytest.raises(IndexError, match="pool id"):
        mmr_reference(V, torch.tensor([[0, 30]]), torch.zeros(1, 2), 1, 0.5)
    with pytest.raises(IndexError, match="pool id"):
        mmr_reference(V, torch.tensor([[-2, 0]]), torch.zeros(1, 2), 1, 0.5)
    with pytest.raises(_cabi.YelprecError, match="CUDA"):
        ops.recommend_mmr(V, ids, sc, 3, 0.5)
    assert ops.mmr_weights(0.3) == (float(np.float32(0.3)), float(np.float32(1) - np.float32(0.3)))


def test_recommender_on_cpu_tables_uses_the_reference():
    from yelprecommendation_b200.retrieval import Recommender, recommend_diverse_reference
    rng = np.random.default_rng(4)
    U, V = quarter_table(rng, 8, 16), quarter_table(rng, 60, 16)
    seen = seen_lists(rng, 8, 60)
    rec = Recommender(U, V, seen)
    for lam, pool in ((0.5, None), (0.2, 12), (1.0, 40)):
        ids, sc = rec.recommend_diverse([1, 4, 7], 6, lam=lam, pool=pool)
        rids, rsc = recommend_diverse_reference(U, V, [1, 4, 7], 6, lam=lam, pool=pool, seen=seen)
        assert torch.equal(ids, rids) and torch.equal(sc, rsc)
    ids, sc = rec.recommend_diverse([1, 4, 7], 6, lam=1.0)
    kids, ksc = rec.recommend([1, 4, 7], 6)
    assert torch.equal(ids, kids) and torch.equal(sc, ksc)


def test_kernel_instances_are_built_for_sm100a():
    """fp32 / bf16 x staged / not staged, as sm_100a SASS, with no stack and no spills."""
    from yelprecommendation_b200 import _cabi
    import __graft_entry__ as ge
    if not os.path.exists(_cabi.lib_path()):
        ge.build()
    out = subprocess.run(["cuobjdump", "-sass", _cabi.lib_path()], capture_output=True, text=True).stdout
    names = set(re.findall(r"Function : (\S*recommend_mmr_kernel\S*)", out))
    assert len(names) == 4, names
    log = os.path.join(os.path.dirname(_cabi.lib_path()), "..", "csrc", "build", "retrieval.ptxas.log")
    if os.path.exists(log):
        entries = [e for e in re.split(r"Compiling entry function ", open(log).read())[1:]
                   if "recommend_mmr_kernel" in e.split("'")[1]]
        assert len(entries) == 4
        for e in entries:
            assert re.search(r"0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads", e), e[:300]


# ------------------------------------------------------------------------------------------------------------------
# GPU: the kernel against the reference
# ------------------------------------------------------------------------------------------------------------------
# Rows are staged in shared memory while N * d * sizeof(T) (plus 17 bytes a position) fit in 113 KB: in fp32 (256, 64),
# (1024, 8) and (20, 1024) are staged, (37, 1024), (256, 256) and (1024, 64) are read from global memory; bf16 halves
# the rows, so (37, 1024) is staged there.
POOLS = [(1, 1), (20, 20), (100, 100), (37, 1), (37, 20), (256, 1), (256, 20), (256, 100), (1024, 20), (1024, 100)]


def _kernel_vs_reference(V, B, N, k, dtype, seed, lam_list=(0.0, 0.3, 0.5, 1.0)):
    from yelprecommendation_b200 import ops
    from yelprecommendation_b200.retrieval import mmr_reference
    rng = np.random.default_rng(seed)
    ids, sc = quarter_pool(rng, B, N, V.shape[0], sort=bool(seed % 2))
    Vd = V.cuda().to(dtype)
    for lam in lam_list:
        got_ids, got_sc = ops.recommend_mmr(Vd, ids.cuda(), sc.cuda(), k, lam)
        want_ids, want_sc = mmr_reference(V, ids, sc, k, lam)
        assert got_ids.shape == (B, k) and got_ids.dtype == I64 and got_sc.dtype == F32
        assert torch.equal(got_ids.cpu(), want_ids), (lam, (got_ids.cpu() != want_ids).nonzero()[:5])
        assert torch.equal(got_sc.cpu(), want_sc), lam


def _quarter_items(rng, nI, d):
    V = quarter_table(rng, nI, d)
    V[::17] = 0                                                # zero-norm items
    pair = torch.arange(1, nI - 1, 17)
    V[pair] = V[pair + 1]                                      # pairs with one direction
    return V


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("d", [8, 64, 256, 1024])
@pytest.mark.parametrize("N,k", POOLS)
def test_kernel_equals_reference_exact(N, k, d, dtype):
    rng = np.random.default_rng(N * 7 + k + d)
    V = _quarter_items(rng, 3000, d)
    _kernel_vs_reference(V, 7, N, k, dtype, N + k + d, lam_list=(0.0, 0.3, 0.5, 1.0) if d <= 256 else (0.0, 0.5))


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
def test_kernel_equals_reference_batches(dtype):
    rng = np.random.default_rng(11)
    V = _quarter_items(rng, 5000, 64)
    _kernel_vs_reference(V, 4096, 37, 20, dtype, 1, lam_list=(0.0, 0.5, 1.0))
    _kernel_vs_reference(V, 1, 256, 100, dtype, 2)
    _kernel_vs_reference(V, 3, 1024, 1024, dtype, 3, lam_list=(0.5,))   # k = N = 1024
    from yelprecommendation_b200 import ops
    ids, sc = ops.recommend_mmr(V.cuda().to(dtype), torch.zeros(0, 40, dtype=I64, device="cuda"),
                                torch.zeros(0, 40, device="cuda"), 10, 0.5)
    assert ids.shape == (0, 10) and sc.shape == (0, 10)


@pytest.mark.gpu
def test_kernel_gaussian_tables_against_float64():
    """Gaussian fp32 tables: the kernel's picks against a float64 greedy, row by row up to the first step whose best and
    second-best float64 marginal relevances are within 1e-5 * scale of each other."""
    from yelprecommendation_b200 import ops
    g = torch.Generator().manual_seed(5)
    nI, d, B, N, k = 20000, 64, 256, 200, 20
    V = torch.randn(nI, d, generator=g)
    ids = torch.stack([torch.randperm(nI, generator=g)[:N] for _ in range(B)])
    sc = torch.sort(torch.randn(B, N, generator=g) * 2, dim=1, descending=True).values
    V64 = V.double().numpy()
    full = 0
    for lam in (0.3, 0.7):
        got, _ = ops.recommend_mmr(V.cuda(), ids.cuda(), sc.cuda(), k, lam)
        got = got.cpu().numpy()
        a, c = ops.mmr_weights(lam)
        for b in range(B):
            X = V64[ids[b].numpy()]
            X = X / np.linalg.norm(X, axis=1, keepdims=True)
            S = X @ X.T
            r = sc[b].double().numpy()
            scale = np.abs(a * r).max() + c
            pos = {int(i): j for j, i in enumerate(ids[b].tolist())}
            pen = np.zeros(N)
            avail = np.ones(N, bool)
            ok = True
            for t in range(k):
                m = np.where(avail, a * r - c * pen, -np.inf)
                o = np.argsort(-m, kind="stable")
                if m[o[0]] - m[o[1]] <= 1e-5 * scale:
                    ok = False
                    break
                assert got[b, t] == ids[b, o[0]].item(), (lam, b, t)
                s = pos[int(got[b, t])]
                avail[s] = False
                pen = S[:, s] if t == 0 else np.maximum(pen, S[:, s])
            full += ok
    assert full >= 0.9 * 2 * B, full


@pytest.mark.gpu
def test_error_word_raises():
    from yelprecommendation_b200 import _cabi, ops
    V = torch.zeros(10, 8, device="cuda")
    sc = torch.zeros(2, 3, device="cuda")
    for bad in (10, -2):
        ids = torch.tensor([[0, 1, 2], [3, bad, 4]], device="cuda")
        with pytest.raises(IndexError, match="pool id"):
            ops.recommend_mmr(V, ids, sc, 2, 0.5)
    ids = torch.tensor([[0, 1, 2], [3, 5, 4]], device="cuda")
    with pytest.raises(ValueError, match="k must be"):
        ops.recommend_mmr(V, ids, sc, 4, 0.5)
    with pytest.raises(ValueError, match="lam"):
        ops.recommend_mmr(V, ids, sc, 2, 1.01)
    with pytest.raises(TypeError):
        ops.recommend_mmr(V, ids.to(I32), sc, 2, 0.5)
    with pytest.raises(ValueError, match="multiple of 8"):
        ops.recommend_mmr(torch.zeros(10, 12, device="cuda"), ids, sc, 2, 0.5)
    with pytest.raises(_cabi.YelprecError, match="CUDA"):
        ops.recommend_mmr(V, ids.cpu(), sc, 2, 0.5)


# ------------------------------------------------------------------------------------------------------------------
# GPU: recommend_diverse
# ------------------------------------------------------------------------------------------------------------------
def _restricted_recommender():
    from yelprecommendation_b200.retrieval import ItemLocations, ItemSubsets, Recommender
    g = torch.Generator().manual_seed(9)
    nU, nI, d = 200, 3000, 32
    U, V = torch.randn(nU, d, generator=g), torch.randn(nI, d, generator=g)
    rng = np.random.default_rng(9)
    seen = seen_lists(rng, nU, nI)
    city = rng.integers(0, 12, nI)
    subsets = ItemSubsets.from_pairs(city, np.arange(nI), 12, nI)
    lat, lon = rng.uniform(40, 41, nI), rng.uniform(-75, -74, nI)
    loc = ItemLocations.from_degrees(lat, lon)
    return Recommender(U.cuda(), V.cuda(), seen, subsets=subsets, locations=loc), seen, subsets, loc, city, lat, lon


@pytest.mark.gpu
def test_lam_one_equals_recommend():
    rec, seen, subsets, loc, city, lat, lon = _restricted_recommender()
    uid = torch.arange(0, 200, 3, device="cuda")
    for kw in ({}, {"subset": 4}, {"near": (40.5, -74.5), "radius_km": 20.0}):
        for k, pool in ((20, None), (7, 300)):
            ids, sc = rec.recommend_diverse(uid, k, lam=1.0, pool=pool, **kw)
            kids, ksc = rec.recommend(uid, k, **kw)
            assert torch.equal(ids, kids) and torch.equal(sc, ksc), kw


@pytest.mark.gpu
def test_composition_and_restrictions():
    from yelprecommendation_b200 import ops
    from yelprecommendation_b200.retrieval import EARTH_RADIUS_KM
    rec, seen, subsets, loc, city, lat, lon = _restricted_recommender()
    uid = torch.arange(0, 200, 2, device="cuda")
    k, N = 20, 80
    for kw in ({}, {"subset": 4}, {"near": (40.5, -74.5), "radius_km": 20.0}):
        ids, sc = rec.recommend_diverse(uid, k, lam=0.5, pool=N, **kw)
        pids, psc = rec.recommend(uid, N, **kw)
        cids, csc = ops.recommend_mmr(rec.item_emb, pids, psc, k, 0.5)
        assert torch.equal(ids, cids) and torch.equal(sc, csc), kw
        assert not torch.equal(ids, pids[:, :k])               # the re-ranking changes the lists
        h = ids.cpu().numpy()
        for b, u in enumerate(uid.tolist()):
            row = h[b][h[b] >= 0]
            assert len(set(row.tolist())) == len(row)
            assert not set(row.tolist()) & set(seen.idx[seen.ptr[u]:seen.ptr[u + 1]].tolist())
            if "subset" in kw:
                assert (city[row] == 4).all()
            if "near" in kw:
                p, q = np.radians(lat[row]), np.radians(lon[row])
                cosd = np.sin(p) * np.sin(np.radians(40.5)) + np.cos(p) * np.cos(np.radians(40.5)) * \
                    np.cos(q - np.radians(-74.5))
                assert (np.arccos(np.clip(cosd, -1, 1)) * EARTH_RADIUS_KM <= 20.0 + 1e-3).all()


@pytest.mark.gpu
def test_trainers_recommend_diverse():
    """MF, NGCF (concatenated width 256) and CDAE recommenders: lam = 1 is recommend, lam = 0.5 is the kernel on
    recommend's pool, unseen and unique, and agrees with the reference re-ranking of the same pool."""
    from yelprecommendation_b200 import ops
    from yelprecommendation_b200.retrieval import SeenItems, mmr_reference
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
    uid = torch.arange(0, inter.num_users, 5, device="cuda")
    for name, tr in (("mf", mf), ("ngcf", ngcf), ("cdae", cdae)):
        rec = tr.recommender(seen)
        V = rec.item_emb if name != "cdae" else cdae.model.output_layer.weight.data
        if name == "ngcf":
            assert V.shape[1] == 256
        ids1, sc1 = rec.recommend_diverse(uid, 10, lam=1.0)
        kids, ksc = rec.recommend(uid, 10)
        assert torch.equal(ids1, kids) and torch.equal(sc1, ksc), name
        ids, sc = rec.recommend_diverse(uid, 10, lam=0.5)
        pids, psc = rec.recommend(uid, 40)
        cids, _ = ops.recommend_mmr(V, pids, psc, 10, 0.5)
        assert torch.equal(ids, cids), name
        rids, _ = mmr_reference(V.cpu(), pids.cpu(), psc.cpu(), 10, 0.5)
        assert (ids.cpu() == rids).float().mean().item() > 0.9, name
        h = ids.cpu().numpy()
        for b, u in enumerate(uid.tolist()):
            row = h[b][h[b] >= 0]
            assert len(row) == 10 and len(set(row.tolist())) == 10, name
            assert not set(row.tolist()) & set(seen.idx[seen.ptr[u]:seen.ptr[u + 1]].tolist()), name
