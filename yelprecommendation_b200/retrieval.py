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

    places = ItemLocations.from_degrees(item_lat, item_lon)    # where each item is
    rec = Recommender(user_emb, item_emb, seen, locations=places)
    ids, scores = rec.recommend(user_ids, k=20, near=(lat, lon), radius_km=5)   # only items within 5 km

With `near`, row b ranks only the items inside its radius, decided by one exact float64 predicate shared by the kernel
(yr_recommend_geo_topk) and the reference: item i is inside iff ((c_x * p_x) + (c_y * p_y)) + (c_z * p_z) >= t, each
product and sum rounded on its own, with p = ItemLocations.P[i], c the centre's unit vector and t = cos(radius_km /
EARTH_RADIUS_KM) (-inf from half the Earth's circumference on), all computed on the host by geo_query. The kernel reads
only the items of the grid cells around each centre; ids and scores equal what the unrestricted kernel returns with every
item outside the radius excluded.
"""
from __future__ import annotations

from typing import Optional, Tuple

import numpy as np
import torch

from . import ops

I32, I64, F32 = torch.int32, torch.int64, torch.float32


EARTH_RADIUS_KM = 6371.0088          # mean Earth radius (IUGG)
GEO_MIN_CELL_KM = 0.01               # grid cells at least 10 m wide: the window's one-cell margin covers float64 rounding


def _unit_xyz(lat: np.ndarray, lon: np.ndarray) -> np.ndarray:
    """float64 [n x 3] unit vectors (cos(phi) cos(lam), cos(phi) sin(lam), sin(phi)) of (lat, lon) in degrees."""
    phi, lam = np.radians(lat), np.radians(lon)
    return np.stack([np.cos(phi) * np.cos(lam), np.cos(phi) * np.sin(lam), np.sin(phi)], axis=1)


def _check_degrees(lat: np.ndarray, lon: np.ndarray, what: str) -> None:
    if not (np.isfinite(lat).all() and np.isfinite(lon).all()):
        raise ValueError(f"{what}: coordinates must be finite")
    if lat.size and np.abs(lat).max() > 90.0:
        raise ValueError(f"{what}: latitude outside [-90, 90]")
    if lon.size and np.abs(lon).max() > 180.0:
        raise ValueError(f"{what}: longitude outside [-180, 180]")


def _as_f64(x) -> np.ndarray:
    return np.asarray(x.detach().cpu().numpy() if torch.is_tensor(x) else x, dtype=np.float64)


class ItemLocations:
    """Item positions on the sphere and a grid index over them, for radius-restricted retrieval.

    P: float64 [num_items x 3], the unit vector of each item's (lat, lon). The grid: cells of cell_deg degrees of latitude
    and longitude (cell_km of arc along a meridian); an item is in lat band floor((lat + 90) / cell_deg) and lon band
    floor((lon + 180) / cell_deg), each clamped to the grid, cell key = lat band * num_lon + lon band. cell_items int32
    [num_items] holds the item ids sorted by (key, id), cell_keys int64 the ascending keys of the non-empty cells and
    cell_ptr int32 their offsets into cell_items. The cell size sets how many items a request reads, never its result."""

    def __init__(self, lat, lon, cell_km: float = 2.0):
        lat, lon = _as_f64(lat).reshape(-1), _as_f64(lon).reshape(-1)
        if lat.shape != lon.shape:
            raise ValueError(f"ItemLocations: {lat.size} latitudes but {lon.size} longitudes")
        _check_degrees(lat, lon, "ItemLocations")
        cell_km = float(cell_km)
        if not cell_km >= GEO_MIN_CELL_KM or not np.isfinite(cell_km):
            raise ValueError(f"ItemLocations: cell_km must be finite and at least {GEO_MIN_CELL_KM}, got {cell_km}")
        n = lat.size
        self.num_items, self.cell_km = n, cell_km
        self.cell_deg = min(float(np.degrees(cell_km / EARTH_RADIUS_KM)), 360.0)
        self.num_lat, self.num_lon = ops.geo_grid_shape(self.cell_deg)
        self.P = torch.from_numpy(_unit_xyz(lat, lon))
        lat_band = np.clip(np.floor((lat + 90.0) / self.cell_deg), 0, self.num_lat - 1).astype(np.int64)
        lon_band = np.clip(np.floor((lon + 180.0) / self.cell_deg), 0, self.num_lon - 1).astype(np.int64)
        key = lat_band * self.num_lon + lon_band
        order = np.lexsort((np.arange(n), key))
        keys, first = np.unique(key[order], return_index=True)
        self.cell_items = torch.from_numpy(order.astype(np.int32))
        self.cell_keys = torch.from_numpy(keys.astype(np.int64))
        self.cell_ptr = torch.from_numpy(np.append(first, n).astype(np.int32))
        self._on = {}

    @classmethod
    def from_degrees(cls, lat, lon, cell_km: float = 2.0) -> "ItemLocations":
        """From each item's latitude and longitude in degrees (item i at (lat[i], lon[i])). ValueError on non-finite
        coordinates, |lat| > 90 or |lon| > 180."""
        return cls(lat, lon, cell_km)

    def on(self, device) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor, torch.Tensor]:
        """(cell_keys, cell_ptr, cell_items, P) on `device`, copied once per device."""
        device = torch.device(device)
        if device.type == "cuda" and device.index is None:
            device = torch.device("cuda", torch.cuda.current_device())
        if device not in self._on:
            self._on[device] = tuple(x.to(device) for x in (self.cell_keys, self.cell_ptr, self.cell_items, self.P))
        return self._on[device]


def geo_query(near, radius_km, B: int) -> Tuple[np.ndarray, np.ndarray]:
    """(c float64 [B x 3], t float64 [B]) of B radius requests: near = one (lat, lon) pair in degrees for every row, or
    two length-B sequences; radius_km = one value or B values, each > 0. c is the centre's unit vector, t =
    cos(radius_km / EARTH_RADIUS_KM), or -inf when radius_km >= pi * EARTH_RADIUS_KM (every item). The one place where
    requests become the predicate's operands, for the kernel and the reference alike."""
    if near is None or radius_km is None:
        raise ValueError("recommend: near and radius_km go together")
    try:
        lat, lon = near
    except (TypeError, ValueError):
        raise ValueError("recommend: near must be a (lat, lon) pair, or two sequences of B values") from None
    lat, lon = _as_f64(lat), _as_f64(lon)
    if lat.ndim == 0 and lon.ndim == 0:
        lat, lon = np.full(B, float(lat)), np.full(B, float(lon))
    elif lat.shape != (B,) or lon.shape != (B,):
        raise ValueError(f"recommend: near must be one (lat, lon) pair or two sequences of {B} values, got shapes "
                         f"{lat.shape} and {lon.shape}")
    _check_degrees(lat, lon, "recommend")
    r = _as_f64(radius_km)
    if r.ndim == 0:
        r = np.full(B, float(r))
    elif r.shape != (B,):
        raise ValueError(f"recommend: radius_km must be one value or {B} values, got shape {r.shape}")
    if np.isnan(r).any() or (r <= 0).any():
        raise ValueError("recommend: radius_km must be > 0")
    whole = r >= np.pi * EARTH_RADIUS_KM
    t = np.where(whole, -np.inf, np.cos(np.where(whole, 0.0, r) / EARTH_RADIUS_KM))
    return _unit_xyz(lat, lon).reshape(B, 3), t


def _geo_inside(P: torch.Tensor, c: torch.Tensor, t: torch.Tensor) -> torch.Tensor:
    """bool [B x nI]: ((c_x * p_x) + (c_y * p_y)) + (c_z * p_z) >= t_b, float64, one rounded operation at a time."""
    return ((c[:, 0:1] * P[None, :, 0]) + (c[:, 1:2] * P[None, :, 1])) + (c[:, 2:3] * P[None, :, 2]) >= t[:, None]


def _geo_args(subset, near, radius_km, locations: Optional[ItemLocations], nI: int, what: str) -> bool:
    """Whether a request is radius-restricted, after checking that it can be."""
    if near is None and radius_km is None:
        return False
    if subset is not None:
        raise ValueError("recommend: subset and near cannot be combined")
    if locations is None:
        raise ValueError(f"recommend: near needs the item locations ({what}(..., locations=ItemLocations...))")
    if locations.num_items != nI:
        raise ValueError(f"recommend: locations cover {locations.num_items} items, the item table {nI}")
    return True


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
                        subset=None, item_bias: Optional[torch.Tensor] = None,
                        locations: Optional[ItemLocations] = None, near=None,
                        radius_km=None) -> Tuple[torch.Tensor, torch.Tensor]:
    """Plain PyTorch on the tables' device: dense [B x num_items] scores (+ item_bias [num_items], fp32), seen items,
    items outside the row's subset (subsets[subset[b]]; -1 = whole catalog) and items outside the row's radius (near,
    radius_km: geo_query's predicate over locations.P) set to -inf, a stable descending sort (torch.topk does not fix the
    order of ties), and slots holding -inf turned into padding (id -1)."""
    k = _check_k(k)
    dev = user_emb.device
    uid = torch.as_tensor(user_ids).to(device=dev, dtype=I64).reshape(-1)
    nU, nI = user_emb.shape[0], item_emb.shape[0]
    if uid.numel() and (int(uid.min()) < 0 or int(uid.max()) >= nU):
        raise IndexError(f"recommend: user id out of range [0, {nU})")
    B = uid.numel()
    geo = _geo_args(subset, near, radius_km, locations, nI, "Recommender")
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
    if geo:
        c, t = geo_query(near, radius_km, B)
        P = locations.P.to(dev)
        inside = _geo_inside(P, torch.from_numpy(c).to(dev), torch.from_numpy(t).to(dev))
        scores[~inside] = float("-inf")
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
    optionally restricted per request to one of the item subsets or to the items within a radius (locations)."""

    def __init__(self, user_emb: torch.Tensor, item_emb: torch.Tensor, seen: Optional[SeenItems] = None,
                 subsets: Optional[ItemSubsets] = None, locations: Optional[ItemLocations] = None):
        if user_emb.device != item_emb.device:
            raise ValueError(f"Recommender: user and item tables on different devices ({user_emb.device}, {item_emb.device})")
        if seen is not None and (seen.num_users != user_emb.shape[0] or seen.num_items != item_emb.shape[0]):
            raise ValueError(f"Recommender: seen items cover {seen.num_users} users x {seen.num_items} items, the tables "
                             f"{user_emb.shape[0]} x {item_emb.shape[0]}")
        if subsets is not None and subsets.num_items != item_emb.shape[0]:
            raise ValueError(f"Recommender: subsets cover {subsets.num_items} items, the item table {item_emb.shape[0]}")
        if locations is not None and locations.num_items != item_emb.shape[0]:
            raise ValueError(f"Recommender: locations cover {locations.num_items} items, the item table "
                             f"{item_emb.shape[0]}")
        self.user_emb, self.item_emb, self.seen, self.subsets = user_emb.detach(), item_emb.detach(), seen, subsets
        self.locations = locations

    def recommend(self, user_ids, k: int, exclude_seen: bool = True, subset=None, near=None,
                  radius_km=None) -> Tuple[torch.Tensor, torch.Tensor]:
        """(item ids int64 [B x k], scores float32 [B x k]) on the tables' device, best first. subset: None (the whole
        catalog), an int for every row, or B ints (-1 = whole catalog for that row): row b then ranks only the items of
        subsets[subset[b]]. Host-side subset ids let the number of item splits follow the requested subsets; on a CUDA
        tensor it follows the whole catalog (no device read). near = (lat, lon) in degrees (one pair, or two sequences
        of B values) with radius_km (one value or B values, > 0): row b ranks only the items within radius_km[b] of
        near[b] (geo_query); not combined with subset."""
        if exclude_seen and self.seen is None:
            raise ValueError("recommend: exclude_seen=True needs the seen items (Recommender(..., seen=SeenItems...))")
        seen = self.seen if exclude_seen else None
        dev = self.user_emb.device
        if subset is not None and self.subsets is None:
            raise ValueError("recommend: subset needs the item subsets (Recommender(..., subsets=ItemSubsets...))")
        _geo_args(subset, near, radius_km, self.locations, self.item_emb.shape[0], "Recommender")
        if dev.type != "cuda":
            return recommend_reference(self.user_emb, self.item_emb, user_ids, k, seen, self.subsets, subset,
                                       locations=self.locations, near=near, radius_km=radius_km)
        uid = user_ids if torch.is_tensor(user_ids) else torch.as_tensor(np.asarray(user_ids, dtype=np.int64))
        uid = uid.to(dev).reshape(-1)
        ptr, idx = seen.on(dev) if seen is not None else (None, None)
        return _recommend_kernel(self.user_emb, self.item_emb, uid, k, ptr, idx, self.subsets, subset,
                                 locations=self.locations, near=near, radius_km=radius_km)


def _recommend_kernel(U, V, uid, k, seen_ptr, seen_idx, subsets: Optional[ItemSubsets], subset, item_bias=None,
                      locations: Optional[ItemLocations] = None, near=None, radius_km=None):
    """ops.recommend_topk, with `subset` ops.recommend_subset_topk, with `near` ops.recommend_geo_topk: seen lists indexed
    by uid, which is on U's device. Host-side subset ids let the number of item splits follow the requested subsets; on a
    CUDA tensor it follows the whole catalog (no device read)."""
    if _geo_args(subset, near, radius_km, locations, V.shape[0], "Recommender"):
        c, t = geo_query(near, radius_km, uid.numel())
        keys, cptr, items, P = locations.on(U.device)
        return ops.recommend_geo_topk(U, V, uid, k, keys, cptr, items, P, locations.cell_deg,
                                      torch.from_numpy(c).to(U.device), torch.from_numpy(t).to(U.device), seen_ptr,
                                      seen_idx, item_bias=item_bias)
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
                             subsets: Optional[ItemSubsets] = None, subset=None,
                             locations: Optional[ItemLocations] = None, near=None,
                             radius_km=None) -> Tuple[torch.Tensor, torch.Tensor]:
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
                               item_bias=model.output_layer.bias.data, locations=locations, near=near,
                               radius_km=radius_km)


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

    recommend(user_ids, k, exclude_seen=True, subset=None, near=None, radius_km=None) has Recommender.recommend's
    contract: (item ids int64 [B x k], scores float32 [B x k]), best first, ties to the lower id, short rows padded with
    -1 / -inf, the same subset and radius semantics.
    The scores are logits, the values CDAETrainer.evaluate ranks by; sigmoid(score) is the model's predicted probability.
    """

    def __init__(self, model, seen: SeenItems, subsets: Optional[ItemSubsets] = None,
                 locations: Optional[ItemLocations] = None):
        _cdae_check(model, seen, subsets, "CDAERecommender")
        if locations is not None and locations.num_items != model.num_items:
            raise ValueError(f"CDAERecommender: locations cover {locations.num_items} items, the model {model.num_items}")
        if model.hidden_layer.weight.device.type != "cuda":
            raise ops.YelprecError("CDAERecommender: the model must be on a CUDA device (the reference path is "
                                   "retrieval.cdae_recommend_reference)")
        self.model, self.seen, self.subsets, self.locations = model, seen, subsets, locations

    def recommend(self, user_ids, k: int, exclude_seen: bool = True, subset=None, near=None,
                  radius_km=None) -> Tuple[torch.Tensor, torch.Tensor]:
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
        if _geo_args(subset, near, radius_km, self.locations, m.num_items, "CDAERecommender"):
            geo_query(near, radius_km, B)
        if B == 0:
            return torch.empty(0, k, device=dev, dtype=I64), torch.empty(0, k, device=dev, dtype=F32)
        ptr, idx = self.seen.on(dev)
        z = m.hidden_from_lists(uid, ptr, idx)
        rows = torch.arange(B, device=dev, dtype=I64)
        bptr, bidx = _batch_lists(self.seen, uid) if exclude_seen else (None, None)
        return _recommend_kernel(z, m.output_layer.weight.data, rows, k, bptr, bidx, self.subsets, subset,
                                 item_bias=m.output_layer.bias.data, locations=self.locations, near=near,
                                 radius_km=radius_km)
