"""Top-K recommendation retrieval: each user's K best unseen items from trained user / item embeddings.

    seen = SeenItems.from_split(split, num_items)              # what every user already interacted with
    rec = Recommender(user_emb, item_emb, seen)                # or trainer.recommender(seen)
    ids, scores = rec.recommend(user_ids, k=20)                # int64 [B x k], float32 [B x k]

Ranking: score = u . v (fp32 accumulation; fp32 or bf16 tables), best first, ties broken by the lower item id. With
exclude_seen the user's seen items are never returned; a user with fewer than k returnable items gets the row padded with
id -1 and score -inf. Items scoring -inf or NaN are never returned.

On CUDA tables `recommend` runs one fused kernel (yr_recommend_topk): scores, seen-item masking and the running top-K stay
on chip, so the B x num_items score matrix is never materialised. On CPU tables it runs `recommend_reference`, the plain
PyTorch restatement (dense scores, masked, stably sorted) that also serves as the kernel's oracle.
"""
from __future__ import annotations

from typing import Optional, Tuple

import numpy as np
import torch

from . import ops

I32, I64, F32 = torch.int32, torch.int64, torch.float32


class SeenItems:
    """Per-user seen items as CSR: ptr int32 [num_users + 1], idx int32 ascending and unique inside a row."""

    def __init__(self, ptr, idx, num_users: int, num_items: int):
        self.ptr = torch.as_tensor(ptr, dtype=I32)
        self.idx = torch.as_tensor(idx, dtype=I32)
        self.num_users, self.num_items = int(num_users), int(num_items)
        if self.ptr.numel() != self.num_users + 1:
            raise ValueError(f"SeenItems: {self.ptr.numel()} offsets for {self.num_users} users")
        self._on = {self.ptr.device: (self.ptr, self.idx)}

    @classmethod
    def from_pairs(cls, users, items, num_users: int, num_items: int) -> "SeenItems":
        """From (user, item) interaction pairs; duplicates are dropped."""
        u = np.asarray(users.cpu() if torch.is_tensor(users) else users, dtype=np.int64).reshape(-1)
        i = np.asarray(items.cpu() if torch.is_tensor(items) else items, dtype=np.int64).reshape(-1)
        if u.shape != i.shape:
            raise ValueError(f"SeenItems.from_pairs: {u.size} users but {i.size} items")
        if u.size and (u.min() < 0 or u.max() >= num_users):
            raise IndexError(f"SeenItems.from_pairs: user id out of range [0, {num_users})")
        if i.size and (i.min() < 0 or i.max() >= num_items):
            raise IndexError(f"SeenItems.from_pairs: item id out of range [0, {num_items})")
        key = np.unique(u * num_items + i)
        ptr = np.zeros(num_users + 1, dtype=np.int64)
        ptr[1:] = np.cumsum(np.bincount(key // num_items, minlength=num_users))
        return cls(ptr.astype(np.int32), (key % num_items).astype(np.int32), num_users, num_items)

    @classmethod
    def from_split(cls, split, num_items: int, parts=("train",)) -> "SeenItems":
        """From a data.synthetic.Split: the union of the named parts (("train", "valid") before a test evaluation)."""
        users, items = [], []
        for part in parts:
            ptr, it = getattr(split, f"{part}_ptr"), getattr(split, f"{part}_items")
            users.append(np.repeat(np.arange(len(ptr) - 1, dtype=np.int64), np.diff(ptr)))
            items.append(np.asarray(it, dtype=np.int64))
        return cls.from_pairs(np.concatenate(users), np.concatenate(items), len(split.train_ptr) - 1, num_items)

    def on(self, device) -> Tuple[torch.Tensor, torch.Tensor]:
        """(ptr, idx) on `device`, copied once per device."""
        device = torch.device(device)
        if device.type == "cuda" and device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        if device not in self._on:
            self._on[device] = (self.ptr.to(device), self.idx.to(device))
        return self._on[device]


def _check_k(k) -> int:
    if isinstance(k, bool) or int(k) != k or not 1 <= int(k) <= ops.RECOMMEND_MAX_K:
        raise ValueError(f"recommend: k must be an integer in [1, {ops.RECOMMEND_MAX_K}], got {k}")
    return int(k)


def recommend_reference(user_emb: torch.Tensor, item_emb: torch.Tensor, user_ids, k: int,
                        seen: Optional[SeenItems] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Plain PyTorch on the tables' device: dense [B x num_items] scores, seen items set to -inf, a stable descending sort
    (torch.topk does not fix the order of ties), and slots holding -inf turned into padding (id -1)."""
    k = _check_k(k)
    dev = user_emb.device
    uid = torch.as_tensor(user_ids).to(device=dev, dtype=I64).reshape(-1)
    nU, nI = user_emb.shape[0], item_emb.shape[0]
    if uid.numel() and (int(uid.min()) < 0 or int(uid.max()) >= nU):
        raise IndexError(f"recommend: user id out of range [0, {nU})")
    B = uid.numel()
    scores = user_emb[uid].to(F32) @ item_emb.to(F32).T
    scores = torch.where(torch.isnan(scores), torch.full_like(scores, float("-inf")), scores)
    if seen is not None:
        ptr, idx = seen.on(dev)
        ptr = ptr.to(I64)
        start, cnt = ptr[uid], ptr[uid + 1] - ptr[uid]
        row = torch.repeat_interleave(torch.arange(B, device=dev), cnt)
        first = torch.repeat_interleave(torch.cumsum(cnt, 0) - cnt, cnt)
        pos = torch.arange(row.numel(), device=dev) - first + torch.repeat_interleave(start, cnt)
        scores[row, idx[pos].to(I64)] = float("-inf")
    kk = min(k, nI)
    sc, order = torch.sort(scores, dim=1, descending=True, stable=True)
    sc, order = sc[:, :kk].contiguous(), order[:, :kk].contiguous()
    order[sc == float("-inf")] = -1
    ids = torch.full((B, k), -1, dtype=I64, device=dev)
    out = torch.full((B, k), float("-inf"), dtype=F32, device=dev)
    ids[:, :kk], out[:, :kk] = order, sc
    return ids, out


class Recommender:
    """Top-K retrieval over fixed user / item tables ([num_users x d], [num_items x d], fp32 or bf16, same device)."""

    def __init__(self, user_emb: torch.Tensor, item_emb: torch.Tensor, seen: Optional[SeenItems] = None):
        if user_emb.device != item_emb.device:
            raise ValueError(f"Recommender: user and item tables on different devices ({user_emb.device}, {item_emb.device})")
        if seen is not None and (seen.num_users != user_emb.shape[0] or seen.num_items != item_emb.shape[0]):
            raise ValueError(f"Recommender: seen items cover {seen.num_users} users x {seen.num_items} items, the tables "
                             f"{user_emb.shape[0]} x {item_emb.shape[0]}")
        self.user_emb, self.item_emb, self.seen = user_emb.detach(), item_emb.detach(), seen

    def recommend(self, user_ids, k: int, exclude_seen: bool = True) -> Tuple[torch.Tensor, torch.Tensor]:
        """(item ids int64 [B x k], scores float32 [B x k]) on the tables' device, best first."""
        if exclude_seen and self.seen is None:
            raise ValueError("recommend: exclude_seen=True needs the seen items (Recommender(..., seen=SeenItems...))")
        seen = self.seen if exclude_seen else None
        dev = self.user_emb.device
        if dev.type != "cuda":
            return recommend_reference(self.user_emb, self.item_emb, user_ids, k, seen)
        uid = user_ids if torch.is_tensor(user_ids) else torch.as_tensor(np.asarray(user_ids, dtype=np.int64))
        uid = uid.to(dev).reshape(-1)
        ptr, idx = seen.on(dev) if seen is not None else (None, None)
        return ops.recommend_topk(self.user_emb, self.item_emb, uid, k, ptr, idx)
