"""Radius-restricted top-K retrieval: the geo kernel (yr_recommend_geo_topk) against the PyTorch reference and against the
unrestricted kernel with the items outside each row's radius excluded, the reference predicate against a brute-force
numpy restatement, the item index and the input checks. Exactness as in test_retrieval: quarter tables make every score
exact, so ids and scores must match bit for bit."""
import copy
import os
import re
import subprocess

import numpy as np
import pytest
import torch

from test_retrieval import quarter_table, seen_lists

I32, I64, F32, F64 = torch.int32, torch.int64, torch.float32, torch.float64
R_KM = 6371.0088


def places(rng, nI, n_clusters=12, spread_km=3.0):
    """Items in Gaussian clusters around random centres, plus items on the antimeridian (both signs), at both poles and
    one isolated item at (0, 0)."""
    lat0 = rng.uniform(-60, 60, n_clusters)
    lon0 = rng.uniform(-180, 180, n_clusters)
    lon0[0], lat0[0] = 179.99, 10.0                               # a cluster straddling the antimeridian
    c = rng.integers(0, n_clusters, nI)
    lat = lat0[c] + rng.normal(0, spread_km / 111.2, nI)
    lon = lon0[c] + rng.normal(0, spread_km / 111.2, nI) / np.cos(np.radians(lat0[c]))
    lon = (lon + 180.0) % 360.0 - 180.0
    lat = np.clip(lat, -90, 90)
    special = [(10.0, 180.0), (10.0, -180.0), (10.01, 179.995), (90.0, 0.0), (90.0, 123.0), (-90.0, -45.0),
               (89.999, 17.0), (0.0, 0.0)]
    for j, (a, o) in enumerate(special):
        lat[j], lon[j] = a, o
    return lat, lon, (lat0, lon0)


def requests(rng, B, lat, lon, centres):
    """Mixed centres and radii: cluster centres at 1 / 5 / 25 km, nowhere (0 items), one isolated item, the antimeridian
    from both sides, both poles, whole Earth."""
    lat0, lon0 = centres
    j = rng.integers(0, len(lat0), B)
    qlat, qlon = lat0[j] + rng.normal(0, 0.01, B), lon0[j].copy()
    qlat = np.clip(qlat, -90, 90)
    r = rng.choice([1.0, 5.0, 25.0], B)
    fixed = [(0.0, 0.0, 0.001),        # exactly one item (the isolated one)
             (-45.0, 100.0, 0.5),      # no item
             (10.0, 180.0, 2.0), (10.0, -180.0, 2.0), (10.0, 179.999, 30.0),
             (90.0, 0.0, 5.0), (-90.0, 0.0, 5.0), (89.99, -170.0, 50.0),
             (0.0, 0.0, np.inf), (33.0, -100.0, 2.1e4)]              # whole Earth
    for i, (a, o, rr) in enumerate(fixed[:B]):
        qlat[i], qlon[i], r[i] = a, o, rr
    return qlat, qlon, r


def predicate_numpy(P, c, t):
    """bool [B x nI] by the definition, in numpy float64, one rounded operation at a time."""
    out = np.zeros((c.shape[0], P.shape[0]), bool)
    for b in range(c.shape[0]):
        x = np.multiply(c[b, 0], P[:, 0])
        y = np.multiply(c[b, 1], P[:, 1])
        z = np.multiply(c[b, 2], P[:, 2])
        out[b] = np.add(np.add(x, y), z) >= t[b]
    return out


def exclusion_csr_geo(seen, uids, inside, dev):
    """Per batch row: the seen items plus every item outside the row's radius."""
    rows = []
    nI = inside.shape[1]
    for b, u in enumerate(uids):
        drop = np.flatnonzero(~inside[b])
        if seen is not None:
            drop = np.union1d(drop, seen.idx[seen.ptr[u]:seen.ptr[u + 1]].numpy())
        rows.append(np.asarray(drop, np.int32))
    ptr = np.zeros(len(rows) + 1, np.int64)
    ptr[1:] = np.cumsum([len(x) for x in rows])
    idx = np.concatenate(rows + [np.zeros(0, np.int32)])
    assert idx.size == 0 or idx.max() < nI
    return torch.from_numpy(ptr.astype(np.int32)).to(dev), torch.from_numpy(idx).to(dev)


# ------------------------------------------------------------------------------------------------------------------
# CPU
# ------------------------------------------------------------------------------------------------------------------
def test_item_locations_index_and_validation():
    from yelprecommendation_b200.retrieval import ItemLocations
    rng = np.random.default_rng(0)
    lat, lon, _ = places(rng, 500)
    loc = ItemLocations.from_degrees(lat, lon, cell_km=5.0)
    P = loc.P.numpy()
    phi, lam = np.radians(lat), np.radians(lon)
    assert P.dtype == np.float64 and np.array_equal(P[:, 2], np.sin(phi))
    assert np.array_equal(P[:, 0], np.cos(phi) * np.cos(lam))
    w = loc.cell_deg
    key = (np.clip(np.floor((lat + 90) / w), 0, loc.num_lat - 1).astype(np.int64) * loc.num_lon
           + np.clip(np.floor((lon + 180) / w), 0, loc.num_lon - 1).astype(np.int64))
    items = loc.cell_items.numpy()
    assert sorted(items.tolist()) == list(range(500))
    assert [(key[i], i) for i in items] == sorted((key[i], i) for i in range(500))
    keys, ptr = loc.cell_keys.numpy(), loc.cell_ptr.numpy()
    assert np.all(np.diff(keys) > 0) and ptr[0] == 0 and ptr[-1] == 500
    for j in range(keys.size):
        assert np.all(key[items[ptr[j]:ptr[j + 1]]] == keys[j])
    big = ItemLocations.from_degrees(lat, lon, cell_km=1e5)          # one cell larger than the Earth
    assert big.num_lat == 1 and big.num_lon == 1 and big.cell_keys.tolist() == [0]
    for bad_lat, bad_lon in [([91.0], [0.0]), ([-90.5], [0.0]), ([0.0], [180.01]), ([np.nan], [0.0]),
                             ([0.0], [np.inf])]:
        with pytest.raises(ValueError):
            ItemLocations.from_degrees(bad_lat, bad_lon)
    with pytest.raises(ValueError):
        ItemLocations.from_degrees([0.0, 1.0], [0.0])
    with pytest.raises(ValueError, match="cell_km"):
        ItemLocations.from_degrees([0.0], [0.0], cell_km=0.0)


def test_geo_query_and_reference_predicate_match_numpy():
    from yelprecommendation_b200.retrieval import ItemLocations, _geo_inside, geo_query
    rng = np.random.default_rng(1)
    lat, lon, centres = places(rng, 3000)
    loc = ItemLocations.from_degrees(lat, lon)
    qlat, qlon, r = requests(rng, 60, lat, lon, centres)
    c, t = geo_query((qlat, qlon), r, 60)
    assert c.dtype == np.float64 and t.dtype == np.float64
    assert np.isneginf(t[8]) and np.isneginf(t[9])
    assert t[2] == np.cos(2.0 / R_KM)
    want = predicate_numpy(loc.P.numpy(), c, t)
    got = _geo_inside(loc.P, torch.from_numpy(c), torch.from_numpy(t)).numpy()
    assert np.array_equal(got, want)
    assert want[0].sum() == 1 and want[0, 7] and want[1].sum() == 0 and want[8].all()
    assert want[2, 0] and want[2, 1] and want[3, 0] and want[3, 1]            # both sides of the antimeridian
    assert want[5, 3] and want[5, 4] and not want[5, 5] and want[6, 5]          # poles
    one_c, one_t = geo_query((12.5, -3.0), 7.0, 4)
    assert one_c.shape == (4, 3) and np.all(one_t == np.cos(7.0 / R_KM))


@pytest.mark.parametrize("k", [1, 7, 50])
def test_cpu_recommender_near_equals_reference_and_brute_force(k):
    from yelprecommendation_b200.retrieval import ItemLocations, Recommender, geo_query, recommend_reference
    from test_retrieval import brute_force
    from yelprecommendation_b200.retrieval import SeenItems
    rng = np.random.default_rng(k)
    nU, nI, d, B = 40, 700, 8, 30
    lat, lon, centres = places(rng, nI, n_clusters=5)
    loc = ItemLocations.from_degrees(lat, lon, cell_km=3.0)
    U, V = quarter_table(rng, nU, d), quarter_table(rng, nI, d)
    seen = seen_lists(rng, nU, nI)
    uids = rng.integers(0, nU, B)
    qlat, qlon, r = requests(rng, B, lat, lon, centres)
    rec = Recommender(U, V, seen, locations=loc)
    ids, sc = rec.recommend(uids, k, near=(qlat, qlon), radius_km=r)
    rids, rsc = recommend_reference(U, V, uids, k, seen, locations=loc, near=(qlat, qlon), radius_km=r)
    assert torch.equal(ids, rids) and torch.equal(sc, rsc)
    inside = predicate_numpy(loc.P.numpy(), *geo_query((qlat, qlon), r, B))
    for b in range(B):
        drop = np.union1d(np.flatnonzero(~inside[b]), seen.idx[seen.ptr[uids[b]]:seen.ptr[uids[b] + 1]].numpy())
        one = SeenItems.from_pairs(np.full(drop.size, uids[b]), drop, nU, nI)
        bi, bs = brute_force(U, V, [uids[b]], k, one)
        assert np.array_equal(ids[b].numpy(), bi[0]) and np.array_equal(sc[b].numpy(), bs[0])


def test_bad_near_and_radius_raise():
    from yelprecommendation_b200.retrieval import ItemLocations, ItemSubsets, Recommender
    rng = np.random.default_rng(3)
    U, V = quarter_table(rng, 5, 8), quarter_table(rng, 20, 8)
    loc = ItemLocations.from_degrees(rng.uniform(-80, 80, 20), rng.uniform(-170, 170, 20))
    subsets = ItemSubsets.from_pairs([0, 0], [1, 2], 1, 20)
    rec = Recommender(U, V, locations=loc, subsets=subsets)
    u = [0, 1, 2]
    ok = rec.recommend(u, 3, exclude_seen=False, near=(1.0, 2.0), radius_km=1e4)
    assert ok[0].shape == (3, 3)
    for near, r in [((1.0, 2.0), 0.0), ((1.0, 2.0), -1.0), ((1.0, 2.0), np.nan), ((1.0, 2.0), [1.0, 2.0]),
                    (([1.0, 2.0], [1.0, 2.0]), 1.0), ((95.0, 0.0), 1.0), ((0.0, -181.0), 1.0), ((np.nan, 0.0), 1.0),
                    ((1.0,), 1.0), (5.0, 1.0), ((1.0, 2.0), None), (None, 1.0)]:
        with pytest.raises(ValueError):
            rec.recommend(u, 3, exclude_seen=False, near=near, radius_km=r)
    with pytest.raises(ValueError, match="subset and near"):
        rec.recommend(u, 3, exclude_seen=False, subset=0, near=(1.0, 2.0), radius_km=1.0)
    with pytest.raises(ValueError, match="locations"):
        Recommender(U, V).recommend(u, 3, exclude_seen=False, near=(1.0, 2.0), radius_km=1.0)
    with pytest.raises(ValueError, match="locations cover"):
        Recommender(U, V[:10], locations=loc)


def test_geo_kernel_rejects_cpu_tensors_and_is_built_without_spills():
    from yelprecommendation_b200 import _cabi, ops
    import __graft_entry__ as ge
    z = torch.zeros(2, dtype=I64)
    with pytest.raises(_cabi.YelprecError, match="CUDA"):
        ops.recommend_geo_topk(torch.zeros(4, 8), torch.zeros(9, 8), z, 3, z, torch.zeros(3, dtype=I32),
                               torch.zeros(9, dtype=I32), torch.zeros(9, 3, dtype=F64), 1.0,
                               torch.zeros(2, 3, dtype=F64), torch.zeros(2, dtype=F64))
    if not os.path.exists(_cabi.lib_path()):
        ge.build()
    out = subprocess.run(["cuobjdump", "-sass", _cabi.lib_path()], capture_output=True, text=True).stdout
    names = set(re.findall(r"Function : (\S*recommend_geo\S*)", out))
    assert len([n for n in names if "recommend_geo_kernel" in n]) == 12, names      # fp32 / bf16 x TU x bias
    assert any("recommend_geo_window_kernel" in n for n in names), names
    log = os.path.join(os.path.dirname(_cabi.lib_path()), "..", "csrc", "build", "retrieval.ptxas.log")
    if os.path.exists(log):
        text = open(log).read()
        for entry in re.split(r"Compiling entry function ", text)[1:]:
            if "recommend_geo" in entry.split("'")[1] or "recommend_subset_kernel" in entry.split("'")[1]:
                assert re.search(r"0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads", entry), entry[:300]
    assert _cabi.load().yr_recommend_geo_ws_bytes(0, 10, 5) == 0


# ------------------------------------------------------------------------------------------------------------------
# GPU
# ------------------------------------------------------------------------------------------------------------------
def _geo_call(U, V, uids, k, loc, c, t, seen=None, bias=None):
    from yelprecommendation_b200 import ops
    keys, ptr, items, P = loc.on(U.device)
    sp, si = seen.on(U.device) if seen is not None else (None, None)
    return ops.recommend_geo_topk(U, V, uids, k, keys, ptr, items, P, loc.cell_deg, torch.from_numpy(c).to(U.device),
                                  torch.from_numpy(t).to(U.device), sp, si, item_bias=bias)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("d", [8, 64, 520, 1024])
@pytest.mark.parametrize("k", [1, 20, 1000])
def test_geo_bit_identical_to_exclusion_csr(d, k, dtype):
    from yelprecommendation_b200 import ops
    from yelprecommendation_b200.retrieval import ItemLocations, geo_query
    g = torch.Generator().manual_seed(d + k)
    nU, nI, B = 300, 12000, 96
    U = torch.randn(nU, d, generator=g).cuda().to(dtype)
    V = torch.randn(nI, d, generator=g).cuda().to(dtype)
    rng = np.random.default_rng(d * 7 + k)
    lat, lon, centres = places(rng, nI, n_clusters=8, spread_km=20.0)
    loc = ItemLocations.from_degrees(lat, lon, cell_km=4.0)
    seen = seen_lists(rng, nU, nI)
    uids = rng.integers(0, nU, B)
    qlat, qlon, r = requests(rng, B, lat, lon, centres)
    c, t = geo_query((qlat, qlon), r, B)
    ud = torch.from_numpy(uids).cuda()
    ids, sc = _geo_call(U, V, ud, k, loc, c, t, seen)
    ptr, idx = exclusion_csr_geo(seen, uids, predicate_numpy(loc.P.numpy(), c, t), "cuda")
    xids, xsc = ops.recommend_topk(U, V, ud, k, ptr, idx, seen_by_row=True)
    assert torch.equal(ids, xids), (ids != xids).nonzero()[:5]
    assert torch.equal(sc, xsc)


@pytest.mark.gpu
@pytest.mark.parametrize("cell_km", [0.5, 5.0, 60.0, 1e5])
@pytest.mark.parametrize("k", [1, 20, 300])
def test_geo_equals_reference_exact(cell_km, k):
    from yelprecommendation_b200.retrieval import ItemLocations, Recommender, geo_query, recommend_reference
    rng = np.random.default_rng(k + int(cell_km))
    nU, nI, d, B = 80, 5000, 32, 64
    U, V = quarter_table(rng, nU, d), quarter_table(rng, nI, d)
    bias = torch.from_numpy((rng.integers(-8, 9, nI) / 4.0).astype(np.float32))
    lat, lon, centres = places(rng, nI)
    loc = ItemLocations.from_degrees(lat, lon, cell_km=cell_km)
    seen = seen_lists(rng, nU, nI, empty={0})
    uids = rng.integers(0, nU, B)
    qlat, qlon, r = requests(rng, B, lat, lon, centres)
    near = (qlat, qlon)
    rec = Recommender(U.cuda(), V.cuda(), seen, locations=loc)
    perm = rng.permutation(B)                                    # results follow request order
    for rows in (np.arange(B), perm):
        for exclude in (True, False):
            nr = (qlat[rows], qlon[rows])
            ids, sc = rec.recommend(torch.from_numpy(uids[rows]).cuda(), k, exclude_seen=exclude, near=nr,
                                    radius_km=r[rows])
            rids, rsc = recommend_reference(U, V, uids[rows], k, seen if exclude else None, locations=loc, near=nr,
                                            radius_km=r[rows])
            assert torch.equal(ids.cpu(), rids), (exclude, (ids.cpu() != rids).nonzero()[:5])
            assert torch.equal(sc.cpu(), rsc)
    c, t = geo_query(near, r, B)
    for exclude in (True, False):
        ids, sc = _geo_call(U.cuda(), V.cuda(), torch.from_numpy(uids).cuda(), k, loc, c, t,
                            seen if exclude else None, bias.cuda())
        rids, rsc = recommend_reference(U, V, uids, k, seen if exclude else None, item_bias=bias, locations=loc,
                                        near=near, radius_km=r)
        assert torch.equal(ids.cpu(), rids) and torch.equal(sc.cpu(), rsc)
    # one item in range (row 0), none (row 1): the rest is padding
    ids, sc = rec.recommend(torch.from_numpy(uids[:2]).cuda(), k, exclude_seen=False, near=(qlat[:2], qlon[:2]),
                            radius_km=r[:2])
    assert ids[0, 0].item() == 7 and (ids[0, 1:] == -1).all() and (ids[1] == -1).all() and torch.isinf(sc[1]).all()
    # the same requests give the same results at every cell size
    other = ItemLocations.from_degrees(lat, lon, cell_km=1.0)
    a = Recommender(U.cuda(), V.cuda(), seen, locations=other).recommend(uids, k, near=near, radius_km=r)
    b = rec.recommend(uids, k, near=near, radius_km=r)
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])


@pytest.mark.gpu
def test_geo_boundary_is_exact():
    """t equal to an item's exact dot product includes the item; the next float64 above excludes it."""
    from yelprecommendation_b200.retrieval import ItemLocations, geo_query
    rng = np.random.default_rng(11)
    nI = 2000
    lat, lon, centres = places(rng, nI)
    loc = ItemLocations.from_degrees(lat, lon, cell_km=2.0)
    U, V = quarter_table(rng, 4, 8).cuda(), quarter_table(rng, nI, 8).cuda()
    P = loc.P.numpy()
    for item in (100, 7, 0, 3):
        c, _ = geo_query((lat[item] - 0.01 if lat[item] > 0 else lat[item] + 0.01, lon[item]), 5.0, 1)
        dot = np.add(np.add(np.multiply(c[0, 0], P[item, 0]), np.multiply(c[0, 1], P[item, 1])),
                     np.multiply(c[0, 2], P[item, 2]))
        inside = predicate_numpy(P, c, np.array([dot]))[0]
        assert inside[item] and inside.sum() < 1000
        for t, want in ((dot, True), (np.nextafter(dot, np.inf), False)):
            ids, _ = _geo_call(U, V, torch.zeros(1, dtype=I64, device="cuda"), 1000, loc, c, np.array([t]))
            got = set(ids[0][ids[0] >= 0].tolist())
            assert (item in got) == want, (item, t)
            assert got == set(np.flatnonzero(predicate_numpy(P, c, np.array([t]))[0]).tolist())


@pytest.mark.gpu
def test_geo_bad_inputs():
    from yelprecommendation_b200 import ops
    from yelprecommendation_b200.retrieval import ItemLocations, geo_query
    rng = np.random.default_rng(5)
    lat, lon, _ = places(rng, 300)
    loc = ItemLocations.from_degrees(lat, lon)
    U, V = quarter_table(rng, 4, 8).cuda(), quarter_table(rng, 300, 8).cuda()
    c, t = geo_query((lat[20], lon[20]), 50.0, 2)
    ids, sc = _geo_call(U, V, torch.tensor([0, 3], device="cuda"), 5, loc, c, t)
    assert ids.shape == (2, 5) and (ids[:, 0] >= 0).all()
    with pytest.raises(IndexError, match="user id"):
        _geo_call(U, V, torch.tensor([0, 4], device="cuda"), 5, loc, c, t)
    with pytest.raises(IndexError, match="user id"):
        _geo_call(U, V, torch.tensor([-1, 0], device="cuda"), 5, loc, c, t)
    for cc, tt in ((np.array([[np.nan, 0, 1], c[1]]), t), (c, np.array([t[0], np.nan])), (c, np.array([np.inf, t[1]])),
                   (np.array([c[0], [np.inf, 0, 0]]), t)):
        with pytest.raises(ValueError, match="not finite"):
            _geo_call(U, V, torch.tensor([0, 1], device="cuda"), 5, loc, cc, tt)
    keys, ptr, items, P = loc.on("cuda")
    with pytest.raises(ValueError, match="threshold"):
        ops.recommend_geo_topk(U, V, torch.tensor([0, 1], device="cuda"), 5, keys, ptr, items, P, loc.cell_deg,
                               torch.from_numpy(c).cuda(), torch.from_numpy(t[:1]).cuda())
    with pytest.raises(TypeError):
        ops.recommend_geo_topk(U, V, torch.tensor([0, 1], device="cuda"), 5, keys, ptr, items, P, loc.cell_deg,
                               torch.from_numpy(c).cuda().float(), torch.from_numpy(t).cuda())
    with pytest.raises(ValueError, match="k must be"):
        _geo_call(U, V, torch.tensor([0, 1], device="cuda"), 0, loc, c, t)
    e = torch.zeros(0, dtype=I64, device="cuda")
    ids, sc = ops.recommend_geo_topk(U, V, e, 5, keys, ptr, items, P, loc.cell_deg, torch.zeros(0, 3, dtype=F64,
                                     device="cuda"), torch.zeros(0, dtype=F64, device="cuda"))
    assert ids.shape == (0, 5) and sc.shape == (0, 5)


@pytest.mark.gpu
@pytest.mark.parametrize("h", [64, 1024])
def test_cdae_recommender_near_equals_reference(h):
    from test_retrieval_cdae import cdae_model, quarter_params
    from yelprecommendation_b200.retrieval import CDAERecommender, ItemLocations, cdae_recommend_reference
    rng = np.random.default_rng(h)
    nU, nI, B = 30, 3000, 40
    model = cdae_model(nU, nI, h, "identity")
    quarter_params(model, rng)
    seen = seen_lists(rng, nU, nI, heavy={1}, empty={2})
    lat, lon, centres = places(rng, nI)
    loc = ItemLocations.from_degrees(lat, lon, cell_km=3.0)
    uids = rng.integers(0, nU, B)
    uids[:3] = [1, 2, 2]
    qlat, qlon, r = requests(rng, B, lat, lon, centres)
    cpu = copy.deepcopy(model).cpu()
    rec = CDAERecommender(model, seen, locations=loc)
    for excl in (True, False):
        ids, sc = rec.recommend(uids, 20, exclude_seen=excl, near=(qlat, qlon), radius_km=r)
        rids, rsc = cdae_recommend_reference(cpu, uids, 20, seen, exclude_seen=excl, locations=loc, near=(qlat, qlon),
                                             radius_km=r)
        assert torch.equal(ids.cpu(), rids) and torch.equal(sc.cpu(), rsc)
    with pytest.raises(ValueError, match="subset"):
        rec.recommend(uids, 5, subset=0, near=(0.0, 0.0), radius_km=1.0)


@pytest.mark.gpu
def test_trainer_recommenders_with_locations():
    from util import cfg
    from test_retrieval import _fixture
    from yelprecommendation_b200.retrieval import ItemLocations, Recommender, SeenItems
    from yelprecommendation_b200.trainers import MFTrainer
    inter, split, batches, _, L = _fixture()
    seen = SeenItems.from_split(split, inter.num_items)
    rng = np.random.default_rng(4)
    lat, lon, centres = places(rng, inter.num_items, n_clusters=3, spread_km=50.0)
    loc = ItemLocations.from_degrees(lat, lon)
    uids = torch.arange(0, inter.num_users, 5, device="cuda")
    qlat, qlon, r = requests(rng, uids.numel(), lat, lon, centres)
    torch.manual_seed(0)
    mf = MFTrainer(cfg(optimizer="adam"), inter.num_items, inter.num_users)
    mf.train(batches[:2])
    rec = mf.recommender(seen, locations=loc)
    ids, sc = rec.recommend(uids, 10, near=(qlat, qlon), radius_km=r * 10)
    want = Recommender(rec.user_emb, rec.item_emb, seen, locations=loc).recommend(uids, 10, near=(qlat, qlon),
                                                                                 radius_km=r * 10)
    assert torch.equal(ids, want[0]) and torch.equal(sc, want[1])
