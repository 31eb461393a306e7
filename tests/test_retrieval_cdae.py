"""CDAE recommendation: the list encoder (yr_cdae_encode) against the dense hidden layer, the per-item bias of the retrieval
kernels against the unbiased kernels on augmented tables, tables up to 1024 wide, and CDAERecommender against the
trainer's evaluation and against cdae_recommend_reference. Exactness as in test_retrieval: quarter-valued tables make every
score exact, so ids and scores must match bit for bit."""
import copy

import numpy as np
import pytest
import torch

from test_retrieval import brute_force, quarter_table, seen_lists
from test_retrieval_subsets import exclusion_csr, subsets_of
from util import cfg, load_npz

I32, I64, F32 = torch.int32, torch.int64, torch.float32


def augment(U, V, b):
    """[U | 1 | 0...], [V | b | 0...], padded to a multiple of 8: their plain dot products are the biased scores."""
    pad = 8
    Ua = torch.zeros(U.shape[0], U.shape[1] + pad, dtype=U.dtype, device=U.device)
    Va = torch.zeros(V.shape[0], V.shape[1] + pad, dtype=V.dtype, device=V.device)
    Ua[:, :U.shape[1]], Ua[:, U.shape[1]] = U, 1
    Va[:, :V.shape[1]], Va[:, V.shape[1]] = V, b.to(V.dtype)
    return Ua, Va


def cdae_model(nU, nI, h, act="sigmoid", device="cuda", seed=0):
    from yelprecommendation_b200.models.cdae import CDAE
    torch.manual_seed(seed)
    c = cfg(hidden_size=h, corruption_level=0.0, hidden_activation=act, output_activation="sigmoid")
    return CDAE(c, nI, nU).to(device).eval()


def quarter_params(model, rng):
    """Every parameter a multiple of 1/4 in [-2, 2]: with the identity activation every logit is exact in fp32."""
    for p in model.parameters():
        p.data.copy_(torch.from_numpy((rng.integers(-8, 9, size=tuple(p.shape)) / 4.0).astype(np.float32)))


def multi_hot(seen, uids, nI):
    x = torch.zeros(len(uids), nI)
    for r, u in enumerate(uids):
        x[r, seen.idx[seen.ptr[u]:seen.ptr[u + 1]].long()] = 1
    return x


def brute_force_cdae(model, seen, uids, k, exclude_seen=True):
    """The definition in float64: z = act(Wh . x + bh + Vu[u]), logits = Wo . z + bo, unseen items sorted (-logit, id)."""
    p = {n: t.detach().cpu().double() for n, t in model.named_parameters()}
    x = multi_hot(seen, uids, model.num_items).double()
    pre = x @ p["hidden_layer.weight"].T + p["hidden_layer.bias"] + p["user_nodes.weight"][torch.as_tensor(uids)]
    z = pre if model.hidden_act == 1 else torch.sigmoid(pre)
    B = len(uids)
    Za, Va = torch.cat([z, torch.ones(B, 1, dtype=z.dtype)], 1), torch.cat(
        [p["output_layer.weight"], p["output_layer.bias"][:, None]], 1)
    from yelprecommendation_b200.retrieval import SeenItems
    rows = SeenItems.from_pairs(*np.nonzero(multi_hot(seen, uids, model.num_items).numpy()), B, model.num_items)
    return brute_force(Za, Va, range(B), k, rows if exclude_seen else None)


# ------------------------------------------------------------------------------------------------------------------
# CPU: the references against brute force, input checks
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("k", [1, 7, 50])
def test_reference_with_bias_matches_brute_force(k):
    from yelprecommendation_b200.retrieval import recommend_reference
    rng = np.random.default_rng(k)
    nU, nI, d = 12, 45, 8
    U, V = quarter_table(rng, nU, d), quarter_table(rng, nI, d)
    b = quarter_table(rng, nI, 1)[:, 0]
    seen = seen_lists(rng, nU, nI, heavy={3}, empty={5})
    uids = np.array([0, 3, 5, 11, 3])
    ids, sc = recommend_reference(U, V, torch.from_numpy(uids), k, seen, item_bias=b)
    Ua, Va = augment(U.double(), V.double(), b.double())
    bids, bsc = brute_force(Ua, Va, uids, k, seen)
    assert np.array_equal(ids.numpy(), bids)
    assert np.array_equal(sc.numpy(), bsc)


@pytest.mark.parametrize("act", ["identity", "sigmoid"])
@pytest.mark.parametrize("k", [1, 10, 60])
def test_cdae_reference_matches_brute_force(act, k):
    from yelprecommendation_b200.retrieval import cdae_recommend_reference
    rng = np.random.default_rng(k)
    nU, nI = 9, 60
    model = cdae_model(nU, nI, 32, act, device="cpu")
    quarter_params(model, rng)
    seen = seen_lists(rng, nU, nI, heavy={2}, empty={4})
    uids = [0, 2, 4, 8, 2]
    for excl in (True, False):
        ids, sc = cdae_recommend_reference(model, uids, k, seen, exclude_seen=excl)
        bids, bsc = brute_force_cdae(model, seen, uids, k, excl)
        if act == "identity":
            assert np.array_equal(ids.numpy(), bids) and np.array_equal(sc.numpy(), bsc)
        else:
            fin = np.isfinite(bsc)
            assert np.array_equal(np.isfinite(sc.numpy()), fin)
            assert np.allclose(sc.numpy()[fin], bsc[fin], rtol=0, atol=1e-5)


def test_cdae_recommender_rejects_bad_setups_on_cpu():
    from yelprecommendation_b200 import _cabi
    from yelprecommendation_b200.retrieval import CDAERecommender, cdae_recommend_reference
    rng = np.random.default_rng(0)
    model = cdae_model(6, 30, 32, device="cpu")
    seen = seen_lists(rng, 6, 30)
    with pytest.raises(_cabi.YelprecError):
        CDAERecommender(model, seen)
    with pytest.raises(ValueError, match="seen"):
        CDAERecommender(model, None)
    with pytest.raises(ValueError, match="seen items cover"):
        CDAERecommender(model, seen_lists(rng, 7, 30))
    with pytest.raises(ValueError, match="subsets cover"):
        CDAERecommender(model, seen, subsets=subsets_of([[1, 2]], 31))
    with pytest.raises(ValueError, match="k must be"):
        cdae_recommend_reference(model, [1], 0, seen)
    with pytest.raises(IndexError):
        cdae_recommend_reference(model, [6], 3, seen)


# ------------------------------------------------------------------------------------------------------------------
# GPU: the encoder
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("act", ["sigmoid", "identity"])
@pytest.mark.parametrize("h", [32, 64, 128, 256, 512, 1024])
def test_encoder_equals_dense_hidden(h, act):
    from yelprecommendation_b200.retrieval import SeenItems
    rng = np.random.default_rng(h)
    nU, nI = 40, 700
    model = cdae_model(nU, nI, h, act, seed=h)
    us, its = [], []
    for u in range(nU):
        n = 0 if u == 3 else nI - 50 if u == 5 else int(rng.integers(1, 60))   # empty, > half the catalog, typical
        items = rng.choice(nI, n, replace=False)
        us.append(np.full(n, u)), its.append(items)
    seen = SeenItems.from_pairs(np.concatenate(us), np.concatenate(its), nU, nI)
    uids = np.concatenate([[3, 5, 5, 0], rng.integers(0, nU, 33)])       # repeated ids, B = 37
    ptr, idx = seen.on("cuda")
    z = model.hidden_from_lists(torch.from_numpy(uids).cuda(), ptr, idx)
    want = model.hidden(torch.from_numpy(uids).cuda(), multi_hot(seen, uids, nI).cuda())
    assert z.shape == (len(uids), h)
    assert torch.equal(z, want)


@pytest.mark.gpu
def test_encoder_bad_ids_raise():
    rng = np.random.default_rng(0)
    model = cdae_model(5, 50, 64)
    seen = seen_lists(rng, 5, 50)
    ptr, idx = seen.on("cuda")
    with pytest.raises(IndexError, match="user id"):
        model.hidden_from_lists(torch.tensor([1, 5]).cuda(), ptr, idx)
    bad = idx.clone()
    bad[int(seen.ptr[2])] = 50
    with pytest.raises(IndexError, match="item id"):
        model.hidden_from_lists(torch.tensor([2]).cuda(), ptr, bad)
    back = ptr.clone()
    back[3] = back[2] - 1                                                  # decreasing offsets
    with pytest.raises(IndexError, match="item id"):
        model.hidden_from_lists(torch.tensor([2]).cuda(), back, idx)
    # the rows around the bad ones are still right
    z = model.hidden_from_lists(torch.tensor([0, 1]).cuda(), ptr, idx)
    assert torch.equal(z, model.hidden(torch.tensor([0, 1]).cuda(), multi_hot(seen, [0, 1], 50).cuda()))


# ------------------------------------------------------------------------------------------------------------------
# GPU: per-item bias, wide tables
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("with_seen", [True, False])
@pytest.mark.parametrize("k", [1, 20, 1000])
@pytest.mark.parametrize("d", [64, 256])
def test_bias_bit_identical_to_augmented_tables(d, k, with_seen):
    from yelprecommendation_b200 import ops
    rng = np.random.default_rng(d + k)
    nU, nI = 300, 20011                                                      # several item splits
    g = torch.Generator().manual_seed(d * 7 + k)
    U, V = torch.randn(nU, d, generator=g).cuda(), torch.randn(nI, d, generator=g).cuda()
    b = torch.randn(nI, generator=g).cuda()
    Ua, Va = augment(U, V, b)
    seen = seen_lists(rng, nU, nI, heavy={7}, empty={9})
    ptr, idx = seen.on("cuda") if with_seen else (None, None)
    uids = torch.from_numpy(np.concatenate([[7, 9], rng.integers(0, nU, 298)])).cuda()
    got = ops.recommend_topk(U, V, uids, k, ptr, idx, item_bias=b)
    want = ops.recommend_topk(Ua, Va, uids, k, ptr, idx)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])
    subsets = subsets_of([np.sort(rng.choice(nI, n, replace=False)) for n in (0, 5, 3000, 15000)], nI)
    sptr, sidx = subsets.on("cuda")
    sid = torch.from_numpy(rng.integers(-1, 4, uids.numel())).cuda()
    got = ops.recommend_subset_topk(U, V, uids, k, sptr, sidx, sid, nI, ptr, idx, item_bias=b)
    want = ops.recommend_subset_topk(Ua, Va, uids, k, sptr, sidx, sid, nI, ptr, idx)
    assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1])


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.bfloat16])
@pytest.mark.parametrize("bias", [False, True])
@pytest.mark.parametrize("d,k", [(64, 20), (520, 1), (520, 300), (1024, 20), (1024, 1000)])
def test_wide_and_biased_equal_reference_exact(d, k, bias, dtype):
    from yelprecommendation_b200 import ops
    from yelprecommendation_b200.retrieval import recommend_reference
    rng = np.random.default_rng(d + k)
    nU, nI = 200, 9001
    U, V = quarter_table(rng, nU, d).cuda().to(dtype), quarter_table(rng, nI, d).cuda().to(dtype)
    b = quarter_table(rng, nI, 1)[:, 0].cuda() if bias else None
    seen = seen_lists(rng, nU, nI, heavy={4}, empty={6})
    ptr, idx = seen.on("cuda")
    uids = torch.from_numpy(np.concatenate([[4, 6], rng.integers(0, nU, 150)])).cuda()
    ids, sc = ops.recommend_topk(U, V, uids, k, ptr, idx, item_bias=b)
    rids, rsc = recommend_reference(U, V, uids, k, seen, item_bias=b)
    assert torch.equal(ids, rids) and torch.equal(sc, rsc)
    subsets = subsets_of([np.sort(rng.choice(nI, n, replace=False)) for n in (0, 40, 2000, 8000)], nI)
    sub = rng.integers(-1, 4, uids.numel())
    sptr, sidx = subsets.on("cuda")
    ids, sc = ops.recommend_subset_topk(U, V, uids, k, sptr, sidx, torch.from_numpy(sub).cuda(), nI, ptr, idx,
                                        item_bias=b)
    rids, rsc = recommend_reference(U, V, uids, k, seen, subsets, sub, item_bias=b)
    assert torch.equal(ids, rids) and torch.equal(sc, rsc)


@pytest.mark.gpu
@pytest.mark.parametrize("k", [1, 20, 256, 300, 1000])
@pytest.mark.parametrize("B", [1, 700, 2048, 4096])
def test_workspace_queries_cover_wide_launches(B, k):
    """The workspace queries do not know d and assume the users per block of d <= 512; d > 512 launches take at most 8,
    which must never mean more item splits. The library refuses a workspace smaller than the launch needs
    (YR_ERR_WORKSPACE), so calls sized by the queries must go through, including those where the users per block drop."""
    from yelprecommendation_b200 import ops
    nI, d = 60000, 1024
    U = torch.zeros(B, d, device="cuda")
    V = torch.zeros(nI, d, device="cuda")
    uids = torch.arange(B, device="cuda")
    ids, _ = ops.recommend_topk(U, V, uids, k, item_bias=torch.zeros(nI, device="cuda"))
    assert torch.equal(ids[:, 0], torch.zeros(B, dtype=I64, device="cuda"))    # all scores 0: ties to the lowest id
    subsets = subsets_of([np.arange(0, nI, 2)], nI)
    sptr, sidx = subsets.on("cuda")
    ids, _ = ops.recommend_subset_topk(U, V, uids, k, sptr, sidx, torch.zeros(B, dtype=I64, device="cuda"), nI // 2)
    assert torch.equal(ids[:, 0], torch.zeros(B, dtype=I64, device="cuda"))


@pytest.mark.gpu
def test_mf_recommender_at_width_1024():
    from yelprecommendation_b200.retrieval import SeenItems, recommend_reference
    from yelprecommendation_b200.trainers import MFTrainer
    from test_retrieval import _fixture
    inter, split, batches, _, _ = _fixture()
    torch.manual_seed(0)
    tr = MFTrainer(cfg(embed_size=1024), inter.num_items, inter.num_users)
    tr.train(batches[:2])
    seen = SeenItems.from_split(split, inter.num_items)
    uids = torch.arange(inter.num_users, device="cuda")
    ids, sc = tr.recommender(seen).recommend(uids, 20)
    U, V = tr.model.user_embedding.weight.data, tr.model.item_embedding.weight.data
    rids, rsc = recommend_reference(U, V, uids, 20, seen)
    assert (ids == rids).float().mean() > 0.99
    assert torch.allclose(sc, rsc, rtol=0, atol=1e-4)


@pytest.mark.gpu
def test_bias_input_checks():
    from yelprecommendation_b200 import ops
    U, V = torch.zeros(4, 8, device="cuda"), torch.zeros(10, 8, device="cuda")
    uids = torch.arange(4, device="cuda")
    for b in (torch.zeros(9, device="cuda"), torch.zeros(10, device="cuda", dtype=torch.float64), torch.zeros(10)):
        with pytest.raises(ValueError, match="item_bias"):
            ops.recommend_topk(U, V, uids, 3, item_bias=b)
    with pytest.raises(ValueError, match="multiple of 8"):
        ops.recommend_topk(torch.zeros(4, 12, device="cuda"), torch.zeros(10, 12, device="cuda"), uids, 3)
    with pytest.raises(ValueError, match="at most 1024"):
        ops.recommend_topk(torch.zeros(4, 1032, device="cuda"), torch.zeros(10, 1032, device="cuda"), uids, 3)


# ------------------------------------------------------------------------------------------------------------------
# GPU: CDAERecommender
# ------------------------------------------------------------------------------------------------------------------
def _cdae_trainer(h):
    """cdae_small.npz after the training batches of test_cdae (h = 64: the fixture's initial parameters)."""
    from test_cdae import _fixture, _trainer
    from yelprecommendation_b200.retrieval import SeenItems
    from yelprecommendation_b200.trainers import CDAETrainer
    g, nU, nI, B, tb, vb, eb, keeps, init = _fixture()
    if h == 64:
        tr = _trainer(g, nU, nI, init, "adam", 1e-2)
    else:
        torch.manual_seed(h)
        tr = CDAETrainer(cfg(optimizer="adam", lr=1e-2, hidden_size=h, corruption_level=0.6, hidden_activation="sigmoid",
                             output_activation="sigmoid", negative_sampling=True, loss_name="bce"), nI, nU)
    tr.train(tb, keeps=keeps)
    m = g["train_mask"] + g["valid_mask"]
    seen = SeenItems.from_pairs(*np.nonzero(m), nU, nI)
    return tr, seen, eb, m, nU, nI


@pytest.mark.gpu
@pytest.mark.parametrize("h", [64, 512])
def test_cdae_recommender_equals_evaluation_ranking(h):
    tr, seen, eb, m, nU, nI = _cdae_trainer(h)
    tr.evaluate(eb)
    K = int(tr.cfg.top_n)
    ids, sc = tr.recommender(seen).recommend(torch.arange(nU), K)
    full = (nI - (m != 0).sum(1)) >= K
    assert full.sum() > nU // 2
    assert torch.equal(ids[torch.from_numpy(full).cuda()], tr.last_topk[torch.from_numpy(full).cuda()])
    assert torch.isfinite(sc[torch.from_numpy(full).cuda()]).all()


@pytest.mark.gpu
@pytest.mark.parametrize("h", [64, 1024])
@pytest.mark.parametrize("k", [1, 20, 300])
def test_cdae_recommender_equals_reference_exact(h, k):
    from yelprecommendation_b200.retrieval import CDAERecommender, cdae_recommend_reference
    rng = np.random.default_rng(h + k)
    nU, nI = 30, 300
    model = cdae_model(nU, nI, h, "identity")
    quarter_params(model, rng)
    seen = seen_lists(rng, nU, nI, heavy={1}, empty={2})
    uids = np.concatenate([[1, 2, 2], rng.integers(0, nU, 20)])
    cpu = copy.deepcopy(model).cpu()
    rec = CDAERecommender(model, seen)
    for excl in (True, False):
        ids, sc = rec.recommend(uids, k, exclude_seen=excl)
        rids, rsc = cdae_recommend_reference(cpu, uids, k, seen, exclude_seen=excl)
        assert torch.equal(ids.cpu(), rids) and torch.equal(sc.cpu(), rsc)


@pytest.mark.gpu
def test_cdae_recommender_close_to_reference_trained():
    from yelprecommendation_b200.retrieval import cdae_recommend_reference
    tr, seen, eb, m, nU, nI = _cdae_trainer(64)
    ids, sc = tr.recommender(seen).recommend(np.arange(nU), 20)
    rids, rsc = cdae_recommend_reference(copy.deepcopy(tr.model).cpu(), np.arange(nU), 20, seen)
    fin = torch.isfinite(rsc)
    assert torch.equal(torch.isfinite(sc.cpu()), fin)
    assert (sc.cpu()[fin] - rsc[fin]).abs().max() <= 1e-5
    assert (ids.cpu() == rids).float().mean() > 0.98


@pytest.mark.gpu
def test_cdae_recommender_subsets_equal_exclusion():
    from yelprecommendation_b200 import ops
    tr, seen, eb, m, nU, nI = _cdae_trainer(64)
    rng = np.random.default_rng(3)
    subsets = subsets_of([[], rng.choice(nI, 3, replace=False), rng.choice(nI, nI // 3, replace=False), np.arange(nI)],
                         nI)
    rec = tr.recommender(seen, subsets)
    uids = np.concatenate([[0, 0, 5], rng.integers(0, nU, 40)])
    sub = np.concatenate([[0, 1, -1], rng.integers(-1, 4, 40)])
    ids, sc = rec.recommend(uids, 20, subset=sub)
    mdl = tr.model
    ptr, idx = seen.on("cuda")
    z = mdl.hidden_from_lists(torch.from_numpy(uids).cuda(), ptr, idx)
    eptr, eidx = exclusion_csr(seen, subsets, uids, sub, nI, "cuda")
    want = ops.recommend_topk(z, mdl.output_layer.weight.data, torch.arange(len(uids), device="cuda"), 20, eptr, eidx,
                              seen_by_row=True, item_bias=mdl.output_layer.bias.data)
    assert torch.equal(ids, want[0]) and torch.equal(sc, want[1])
    assert (ids[0] == -1).all()                                            # the empty subset: all padding
    ids1, _ = rec.recommend(uids, 20, subset=2)
    assert ids1.shape == (len(uids), 20)


@pytest.mark.gpu
def test_cdae_recommender_sees_live_weights():
    tr, seen, eb, m, nU, nI = _cdae_trainer(64)
    from test_cdae import _fixture
    tb = _fixture()[4]
    rec = tr.recommender(seen)
    before = rec.recommend(np.arange(nU), 20)
    tr.train(tb[:1])
    after = rec.recommend(np.arange(nU), 20)
    fresh = tr.recommender(seen).recommend(np.arange(nU), 20)
    assert torch.equal(after[0], fresh[0]) and torch.equal(after[1], fresh[1])
    assert not torch.equal(before[1], after[1])


@pytest.mark.gpu
def test_cdae_recommender_bad_inputs_raise():
    tr, seen, eb, m, nU, nI = _cdae_trainer(64)
    rec = tr.recommender(seen)
    with pytest.raises(ValueError, match="seen"):
        tr.recommender(None)
    with pytest.raises(ValueError, match="k must be"):
        rec.recommend([0], 0)
    with pytest.raises(ValueError, match="k must be"):
        rec.recommend([0], 1025)
    with pytest.raises(ValueError, match="subset"):
        rec.recommend([0], 5, subset=0)
    with pytest.raises(IndexError, match="user id"):
        rec.recommend([nU], 5)
    with pytest.raises(IndexError):
        tr.recommender(seen, subsets_of([[1]], nI)).recommend([0], 5, subset=1)
    ids, sc = rec.recommend([], 5)
    assert ids.shape == (0, 5) and sc.shape == (0, 5)
