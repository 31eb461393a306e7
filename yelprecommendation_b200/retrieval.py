"""Top-K recommendation retrieval: each user's K best unseen items from trained user / item embeddings.

    seen = SeenItems.from_split(split, num_items)              # what every user already interacted with
    rec = Recommender(user_emb, item_emb, seen)                # or trainer.recommender(seen)
    ids, scores = rec.recommend(user_ids, k=20)                # int64 [B x k], float32 [B x k]

    cities = ItemSubsets.from_pairs(city_of_item, item, num_cities, num_items)
    rec = Recommender(user_emb, item_emb, seen, subsets=cities)
    ids, scores = rec.recommend(user_ids, k=20, subset=city)   # row b: only items of city[b] (-1 = whole catalog)

Ranking: score = u . v (fp32 accumulation; fp32 or bf16 tables), best first, ties broken by the lower item id. With
exclude_seen the user's seen items are never returned; a user with fewer than k returnable items gets the row padded with
id -1 and score -inf. Items scoring -inf or NaN are never returned.

On CUDA tables `recommend` runs one fused kernel (yr_recommend_topk): scores, seen-item masking and the running top-K stay
on chip, so the B x num_items score matrix is never materialised. On CPU tables it runs `recommend_reference`, the plain
PyTorch restatement (dense scores, masked, stably sorted) that also serves as the kernel's oracle. With `subset`, the
kernel is yr_recommend_subset_topk: rows are grouped by subset on the device and each streams only its subset's items;
ids and scores equal what the unrestricted kernel returns with every item outside the subset excluded.

    rec = CDAERecommender(cdae_model, seen)                    # or cdae_trainer.recommender(seen)
    ids, logits = rec.recommend(user_ids, k=20)                # same contract; the scores are CDAE output logits

A CDAE user is encoded from their interaction list (yr_cdae_encode), and the output bias enters the retrieval kernels as a
per-item bias added after the dot product.
"""
from __future__ import annotations

from typing import Optional, Tuple

import numpy as np
import torch

from . import ops

I32, I64, F32 = torch.int32, torch.int64, torch.float32


class ItemLists:
    """Item lists as CSR: ptr int32 [num_rows + 1], idx int32 ascending and unique inside a row; max_len = the longest."""
    _row = "row"

    def __init__(self, ptr, idx, num_rows: int, num_items: int):
        self.ptr = torch.as_tensor(ptr, dtype=I32)
        self.idx = torch.as_tensor(idx, dtype=I32)
        self.num_items = int(num_items)
        self._rows = int(num_rows)
        if self.ptr.numel() != self._rows + 1:
            raise ValueError(f"{type(self).__name__}: {self.ptr.numel()} offsets for {self._rows} {self._row}s")
        self.lengths = np.diff(self.ptr.cpu().numpy().astype(np.int64))
        self.max_len = int(self.lengths.max()) if self._rows else 0
        self._on = {self.ptr.device: (self.ptr, self.idx)}

    @classmethod
    def _from_pairs(cls, rows, items, num_rows: int, num_items: int) -> "ItemLists":
        r = np.asarray(rows.cpu() if torch.is_tensor(rows) else rows, dtype=np.int64).reshape(-1)
        i = np.asarray(items.cpu() if torch.is_tensor(items) else items, dtype=np.int64).reshape(-1)
        name = f"{cls.__name__}.from_pairs"
        if r.shape != i.shape:
            raise ValueError(f"{name}: {r.size} {cls._row}s but {i.size} items")
        if r.size and (r.min() < 0 or r.max() >= num_rows):
            raise IndexError(f"{name}: {cls._row} id out of range [0, {num_rows})")
        if i.size and (i.min() < 0 or i.max() >= num_items):
            raise IndexError(f"{name}: item id out of range [0, {num_items})")
        key = np.unique(r * num_items + i)
        ptr = np.zeros(num_rows + 1, dtype=np.int64)
        ptr[1:] = np.cumsum(np.bincount(key // num_items, minlength=num_rows))
        return cls(ptr.astype(np.int32), (key % num_items).astype(np.int32), num_rows, num_items)

    def on(self, device) -> Tuple[torch.Tensor, torch.Tensor]:
        """(ptr, idx) on `device`, copied once per device."""
        device = torch.device(device)
        if device.type == "cuda" and device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        if device not in self._on:
            self._on[device] = (self.ptr.to(device), self.idx.to(device))
        return self._on[device]


class SeenItems(ItemLists):
    """Per-user seen items as CSR: ptr int32 [num_users + 1], idx int32 ascending and unique inside a row."""
    _row = "user"

    def __init__(self, ptr, idx, num_users: int, num_items: int):
        super().__init__(ptr, idx, num_users, num_items)

    @property
    def num_users(self) -> int:
        return self._rows

    @classmethod
    def from_pairs(cls, users, items, num_users: int, num_items: int) -> "SeenItems":
        """From (user, item) interaction pairs; duplicates are dropped."""
        return cls._from_pairs(users, items, num_users, num_items)

    @classmethod
    def from_split(cls, split, num_items: int, parts=("train",)) -> "SeenItems":
        """From a data.synthetic.Split: the union of the named parts (("train", "valid") before a test evaluation)."""
        users, items = [], []
        for part in parts:
            ptr, it = getattr(split, f"{part}_ptr"), getattr(split, f"{part}_items")
            users.append(np.repeat(np.arange(len(ptr) - 1, dtype=np.int64), np.diff(ptr)))
            items.append(np.asarray(it, dtype=np.int64))
        return cls.from_pairs(np.concatenate(users), np.concatenate(items), len(split.train_ptr) - 1, num_items)


class ItemSubsets(ItemLists):
    """Named subsets of the catalog (cities, categories, ...) as CSR: ptr int32 [num_subsets + 1], idx int32 ascending and
    unique inside a subset. Subsets may overlap or be empty."""
    _row = "subset"

    def __init__(self, ptr, idx, num_subsets: int, num_items: int):
        super().__init__(ptr, idx, num_subsets, num_items)

    @property
    def num_subsets(self) -> int:
        return self._rows

    @classmethod
    def from_pairs(cls, subset, item, num_subsets: int, num_items: int) -> "ItemSubsets":
        """From (subset, item) membership pairs; duplicates are dropped."""
        return cls._from_pairs(subset, item, num_subsets, num_items)


def _check_k(k) -> int:
    if isinstance(k, bool) or int(k) != k or not 1 <= int(k) <= ops.RECOMMEND_MAX_K:
        raise ValueError(f"recommend: k must be an integer in [1, {ops.RECOMMEND_MAX_K}], got {k}")
    return int(k)


def _list_entries(lists: ItemLists, rows: torch.Tensor, dev):
    """(batch row, item id) of every entry of lists[rows[b]], for all b: the CSR rows gathered per batch row."""
    ptr, idx = lists.on(dev)
    ptr = ptr.to(I64)
    start, cnt = ptr[rows], ptr[rows + 1] - ptr[rows]
    row = torch.repeat_interleave(torch.arange(rows.numel(), device=dev), cnt)
    first = torch.repeat_interleave(torch.cumsum(cnt, 0) - cnt, cnt)
    pos = torch.arange(row.numel(), device=dev) - first + torch.repeat_interleave(start, cnt)
    return row, idx[pos].to(I64)


def _subset_rows(subset, B: int, subsets: Optional[ItemSubsets]):
    """`subset` (an int for every row, or B ints; -1 = whole catalog) as int64 [B], range-checked when on the host."""
    if subsets is None:
        raise ValueError("recommend: subset needs the item subsets (Recommender(..., subsets=ItemSubsets...))")
    if torch.is_tensor(subset) and subset.is_cuda:
        sid = subset.reshape(-1)
        if sid.dtype not in (I32, I64):
            raise TypeError(f"recommend: subset must hold integers, got {sid.dtype}")
    else:
        a = np.asarray(subset.cpu() if torch.is_tensor(subset) else subset)
        if a.size and not np.issubdtype(a.dtype, np.integer):
            raise TypeError(f"recommend: subset must hold integers, got {a.dtype}")
        a = a.astype(np.int64)
        if a.ndim == 0:
            a = np.full(B, int(a), dtype=np.int64)
        sid = torch.from_numpy(a.reshape(-1))
        if sid.numel() == B and B and (int(sid.min()) < -1 or int(sid.max()) >= subsets.num_subsets):
            raise IndexError(f"recommend: subset id out of range [-1, {subsets.num_subsets})")
    if sid.numel() != B:
        raise ValueError(f"recommend: {sid.numel()} subset ids for {B} users")
    return sid


def recommend_reference(user_emb: torch.Tensor, item_emb: torch.Tensor, user_ids, k: int,
                        seen: Optional[SeenItems] = None, subsets: Optional[ItemSubsets] = None,
                        subset=None, item_bias: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Plain PyTorch on the tables' device: dense [B x num_items] scores (+ item_bias [num_items], fp32), seen items and
    items outside the row's subset (subsets[subset[b]]; -1 = whole catalog) set to -inf, a stable descending sort
    (torch.topk does not fix the order of ties), and slots holding -inf turned into padding (id -1)."""
    k = _check_k(k)
    dev = user_emb.device
    uid = torch.as_tensor(user_ids).to(device=dev, dtype=I64).reshape(-1)
    nU, nI = user_emb.shape[0], item_emb.shape[0]
    if uid.numel() and (int(uid.min()) < 0 or int(uid.max()) >= nU):
        raise IndexError(f"recommend: user id out of range [0, {nU})")
    B = uid.numel()
    scores = user_emb[uid].to(F32) @ item_emb.to(F32).T
    if item_bias is not None:
        scores = scores + item_bias.to(device=dev, dtype=F32)[None, :]
    scores = torch.where(torch.isnan(scores), torch.full_like(scores, float("-inf")), scores)
    if seen is not None:
        row, item = _list_entries(seen, uid, dev)
        scores[row, item] = float("-inf")
    if subset is not None:
        sid = _subset_rows(subset, B, subsets).to(dev)
        if B and (int(sid.min()) < -1 or int(sid.max()) >= subsets.num_subsets):
            raise IndexError(f"recommend: subset id out of range [-1, {subsets.num_subsets})")
        if subsets.num_items != nI:
            raise ValueError(f"recommend: subsets cover {subsets.num_items} items, the item table {nI}")
        outside = (sid >= 0)[:, None].expand(B, nI).clone()
        limited = (sid >= 0).nonzero().reshape(-1)
        row, item = _list_entries(subsets, sid[limited], dev)
        outside[limited[row], item] = False
        scores[outside] = float("-inf")
    kk = min(k, nI)
    sc, order = torch.sort(scores, dim=1, descending=True, stable=True)
    sc, order = sc[:, :kk].contiguous(), order[:, :kk].contiguous()
    order[sc == float("-inf")] = -1
    ids = torch.full((B, k), -1, dtype=I64, device=dev)
    out = torch.full((B, k), float("-inf"), dtype=F32, device=dev)
    ids[:, :kk], out[:, :kk] = order, sc
    return ids, out


class Recommender:
    """Top-K retrieval over fixed user / item tables ([num_users x d], [num_items x d], fp32 or bf16, same device),
    optionally restricted per request to one of the item subsets."""

    def __init__(self, user_emb: torch.Tensor, item_emb: torch.Tensor, seen: Optional[SeenItems] = None,
                 subsets: Optional[ItemSubsets] = None):
        if user_emb.device != item_emb.device:
            raise ValueError(f"Recommender: user and item tables on different devices ({user_emb.device}, {item_emb.device})")
        if seen is not None and (seen.num_users != user_emb.shape[0] or seen.num_items != item_emb.shape[0]):
            raise ValueError(f"Recommender: seen items cover {seen.num_users} users x {seen.num_items} items, the tables "
                             f"{user_emb.shape[0]} x {item_emb.shape[0]}")
        if subsets is not None and subsets.num_items != item_emb.shape[0]:
            raise ValueError(f"Recommender: subsets cover {subsets.num_items} items, the item table {item_emb.shape[0]}")
        self.user_emb, self.item_emb, self.seen, self.subsets = user_emb.detach(), item_emb.detach(), seen, subsets

    def recommend(self, user_ids, k: int, exclude_seen: bool = True, subset=None) -> Tuple[torch.Tensor, torch.Tensor]:
        """(item ids int64 [B x k], scores float32 [B x k]) on the tables' device, best first. subset: None (the whole
        catalog), an int for every row, or B ints (-1 = whole catalog for that row): row b then ranks only the items of
        subsets[subset[b]]. Host-side subset ids let the number of item splits follow the requested subsets; on a CUDA
        tensor it follows the whole catalog (no device read)."""
        if exclude_seen and self.seen is None:
            raise ValueError("recommend: exclude_seen=True needs the seen items (Recommender(..., seen=SeenItems...))")
        seen = self.seen if exclude_seen else None
        dev = self.user_emb.device
        if subset is not None and self.subsets is None:
            raise ValueError("recommend: subset needs the item subsets (Recommender(..., subsets=ItemSubsets...))")
        if dev.type != "cuda":
            return recommend_reference(self.user_emb, self.item_emb, user_ids, k, seen, self.subsets, subset)
        uid = user_ids if torch.is_tensor(user_ids) else torch.as_tensor(np.asarray(user_ids, dtype=np.int64))
        uid = uid.to(dev).reshape(-1)
        ptr, idx = seen.on(dev) if seen is not None else (None, None)
        return _recommend_kernel(self.user_emb, self.item_emb, uid, k, ptr, idx, self.subsets, subset)


def _recommend_kernel(U, V, uid, k, seen_ptr, seen_idx, subsets: Optional[ItemSubsets], subset, item_bias=None):
    """ops.recommend_topk, or with `subset` ops.recommend_subset_topk: seen lists indexed by uid, which is on U's device.
    Host-side subset ids let the number of item splits follow the requested subsets; on a CUDA tensor it follows the whole
    catalog (no device read)."""
    if subset is None:
        return ops.recommend_topk(U, V, uid, k, seen_ptr, seen_idx, item_bias=item_bias)
    sid = _subset_rows(subset, uid.numel(), subsets)
    nI = V.shape[0]
    if sid.is_cuda:
        max_len = nI
    else:
        h = sid.numpy()
        max_len = int(subsets.lengths[h[h >= 0]].max(initial=0))
        if (h == -1).any():
            max_len = nI
    sptr, sidx = subsets.on(U.device)
    return ops.recommend_subset_topk(U, V, uid, k, sptr, sidx, sid.to(U.device), max_len, seen_ptr, seen_idx,
                                     item_bias=item_bias)


def _cdae_check(model, seen: Optional[SeenItems], subsets: Optional[ItemSubsets], what: str) -> None:
    if seen is None:
        raise ValueError(f"{what}: CDAE needs the seen items even with exclude_seen=False: they are the model's input")
    if seen.num_users != model.num_users or seen.num_items != model.num_items:
        raise ValueError(f"{what}: seen items cover {seen.num_users} users x {seen.num_items} items, the model "
                         f"{model.num_users} x {model.num_items}")
    if subsets is not None and subsets.num_items != model.num_items:
        raise ValueError(f"{what}: subsets cover {subsets.num_items} items, the model {model.num_items}")


def cdae_recommend_reference(model, user_ids, k: int, seen: SeenItems, exclude_seen: bool = True,
                             subsets: Optional[ItemSubsets] = None, subset=None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Plain PyTorch restatement of CDAERecommender.recommend on the model's device: the dense multi-hot x of the users'
    seen items, z = act(x @ W_h^T + b_h + V_u[u]), then recommend_reference over the logits z . W_o[i] + b_o[i]."""
    _cdae_check(model, seen, subsets, "cdae_recommend_reference")
    dev = model.hidden_layer.weight.device
    uid = torch.as_tensor(user_ids).to(device=dev, dtype=I64).reshape(-1)
    if uid.numel() and (int(uid.min()) < 0 or int(uid.max()) >= model.num_users):
        raise IndexError(f"recommend: user id out of range [0, {model.num_users})")
    B = uid.numel()
    x = torch.zeros(B, model.num_items, device=dev, dtype=F32)
    row, item = _list_entries(seen, uid, dev)
    x[row, item] = 1.0
    Wh, bh = model.hidden_layer.weight.data, model.hidden_layer.bias.data
    pre = x @ Wh.T + bh + model.user_nodes.weight.data[uid]
    z = pre if model.hidden_act == 1 else torch.sigmoid(pre)
    rows = SeenItems(*_batch_lists(seen, uid), B, model.num_items) if exclude_seen else None
    return recommend_reference(z, model.output_layer.weight.data, torch.arange(B, device=dev), k, rows, subsets, subset,
                               item_bias=model.output_layer.bias.data)


def _batch_lists(seen: SeenItems, uid: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """(ptr int32 [B + 1], idx int32): seen[uid[b]] for every batch row b, a CSR indexed by the batch row (uid's device)."""
    dev = uid.device
    ptr = seen.on(dev)[0].to(I64)
    bptr = torch.zeros(uid.numel() + 1, device=dev, dtype=I64)
    bptr[1:] = torch.cumsum(ptr[uid + 1] - ptr[uid], 0)
    return bptr.to(I32), _list_entries(seen, uid, dev)[1].to(I32)


class CDAERecommender:
    """Top-K retrieval for a CDAE model (models/cdae.py) on the device, through its live parameters: training between
    calls is reflected. The user side is encoded from the user's interaction list (seen, which is the model's input and is
    therefore required even with exclude_seen=False, as CDAETrainer.evaluate feeds and masks the same input), without a
    B x num_items input or output: z = act(W_h[:, seen[u]].sum(1) + b_h + V_u[u]) (yr_cdae_encode), then the fused
    retrieval kernel ranks the logits z . W_o[i] + b_o[i] (b_o as the per-item bias).

    recommend(user_ids, k, exclude_seen=True, subset=None) has Recommender.recommend's contract: (item ids int64 [B x k],
    scores float32 [B x k]), best first, ties to the lower id, short rows padded with -1 / -inf, the same subset semantics.
    The scores are logits, the values CDAETrainer.evaluate ranks by; sigmoid(score) is the model's predicted probability.
    """

    def __init__(self, model, seen: SeenItems, subsets: Optional[ItemSubsets] = None):
        _cdae_check(model, seen, subsets, "CDAERecommender")
        if model.hidden_layer.weight.device.type != "cuda":
            raise ops.YelprecError("CDAERecommender: the model must be on a CUDA device (the reference path is "
                                   "retrieval.cdae_recommend_reference)")
        self.model, self.seen, self.subsets = model, seen, subsets

    def recommend(self, user_ids, k: int, exclude_seen: bool = True, subset=None) -> Tuple[torch.Tensor, torch.Tensor]:
        """(item ids int64 [B x k], logits float32 [B x k]) on the model's device, best first; see the class docstring."""
        m = self.model
        dev = m.hidden_layer.weight.device
        if subset is not None and self.subsets is None:
            raise ValueError("recommend: subset needs the item subsets (CDAERecommender(..., subsets=ItemSubsets...))")
        k = _check_k(k)
        uid = user_ids if torch.is_tensor(user_ids) else torch.as_tensor(np.asarray(user_ids, dtype=np.int64))
        uid = uid.to(device=dev, dtype=I64).reshape(-1)
        B = uid.numel()
        if subset is not None:
            _subset_rows(subset, B, self.subsets)
        if B == 0:
            return torch.empty(0, k, device=dev, dtype=I64), torch.empty(0, k, device=dev, dtype=F32)
        ptr, idx = self.seen.on(dev)
        z = m.hidden_from_lists(uid, ptr, idx)
        rows = torch.arange(B, device=dev, dtype=I64)
        bptr, bidx = _batch_lists(self.seen, uid) if exclude_seen else (None, None)
        return _recommend_kernel(z, m.output_layer.weight.data, rows, k, bptr, bidx, self.subsets, subset,
                                 item_bias=m.output_layer.bias.data)
