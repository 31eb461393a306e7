"""Drop-in for the reference's trainers/cdae_trainer.py:22-144 on the sm_100a kernels (BASELINE config 4).

`train` runs one yr_cdae_step per DataLoader batch: the dense `input_mask` / `negative_mask` rows the reference's
CDAEDataset yields are compacted on the device (or, for index-list batches — data/cdae_sparse.py — shipped as a few hundred
bytes per user through yr_cdae_step_idx), the loss and its gradient are evaluated only at the loss positions, and
every parameter gets torch's dense optimizer step. `validate` returns the reference's 5-tuple (loss, P, R, MAP, NDCG),
`evaluate` the 4 metrics; both rank with the fused full-catalog kernels on the output LOGITS: sigmoid is monotone, so
top-K by logit equals top-K by prediction except where the float sigmoid saturates into ties — which the reference
orders arbitrarily (NumPy argpartition). Masking by `pred * logical_not(input_mask)` (cdae_trainer.py:132) puts the
train items at 0, below every unmasked prediction: the same order as masking logits to -3.40282e+38.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from .. import _cabi, ops
from ..loss import NSBCELoss
from ..models.cdae import CDAE
from .base_trainer import BaseTrainer, FusedOptimizer, logger

I32, I64, F32, F64 = torch.int32, torch.int64, torch.float32, torch.float64
def _ldz(h: int) -> int:
    """Width of [z (h) | 1 | 0...]: logits = [z|1].[Wo|bo]^T, padded to what the evaluation kernels like (d % 32 == 0)."""
    return (h + 1 + 31) // 32 * 32


class CDAETrainer(BaseTrainer):
    def __init__(self, cfg, num_items: int, num_users: int) -> None:
        super().__init__(cfg)
        self.num_items, self.num_users = num_items, num_users
        self.model = CDAE(self.cfg, num_items, num_users).to(self.device)
        self.optimizer: FusedOptimizer = self._optimizer(self.cfg.optimizer, self.model, self.cfg.lr)   # wd = 0, as the reference
        self.loss = self._loss()
        self._bufs = None
        self.last_step_losses = None
        self.last_topk = None

    def _loss(self):
        if self.cfg.loss_name.lower() == "bce" and self.cfg.negative_sampling:
            return NSBCELoss()
        if self.cfg.loss_name.lower() == "bce":
            raise NotImplementedError("the B200 CDAE path implements the reference's negative_sampling=True loss")
        logger.error(f"Loss Not Exists: {self.cfg.loss_name} when negative_sampling == {self.cfg.negative_sampling}")
        raise NotImplementedError(f"Loss Not Exists: {self.cfg.loss_name}")

    # ------------------------------------------------------------------------------------------
    def _state(self):
        m = self.model
        if self._bufs is None:
            params = [m.hidden_layer.weight, m.hidden_layer.bias, m.user_nodes.weight, m.output_layer.weight,
                      m.output_layer.bias]
            z = lambda t: torch.zeros_like(t.data)
            b = {"grads": [z(t) for t in params], "loss": torch.zeros(2, device=self.device, dtype=F64),
                 "err": torch.zeros(1, device=self.device, dtype=I32)}
            if self.optimizer.needs_moments:
                b["m"], b["v"] = [z(t) for t in params], [z(t) for t in params]
            self._bufs = b
        b = self._bufs
        pack = lambda ts: _cabi.YrCdaeTensors(*[_cabi.dptr(t, F32) for t in ts])
        return b, pack(b["grads"]), (pack(b["m"]) if "m" in b else None), (pack(b["v"]) if "v" in b else None)

    def _step(self, user_id, x, keep, target, negative_mask, train: bool, step_loss=None):
        lib = _cabi.load()
        m = self.model
        b, g, mo, vo = self._state()
        dev = self.device
        user_id = user_id.to(device=dev, dtype=I64, non_blocking=True).contiguous()
        x, target, negative_mask = (t.to(device=dev, dtype=F32, non_blocking=True).contiguous()
                                    for t in (x, target, negative_mask))
        B = x.shape[0]
        ws = m.workspace(B)
        P = m.tensors()
        opt = self.optimizer.opt_struct(self.optimizer.step_count + 1) if train else None
        _cabi.check(lib.yr_cdae_step_ex(C.byref(P), C.byref(g) if train else None,
                                     C.byref(mo) if (train and mo is not None) else None,
                                     C.byref(vo) if (train and vo is not None) else None,
                                     C.byref(opt) if train else None, self.num_users, self.num_items, m.hidden_size,
                                     m.hidden_act,
                                     _cabi.dptr(user_id), _cabi.dptr(x), _cabi.dptr(keep) if keep is not None else None,
                                     _cabi.dptr(target), _cabi.dptr(negative_mask), B, _cabi.dptr(b["loss"]),
                                     _cabi.dptr(step_loss) if step_loss is not None else None, _cabi.dptr(ws), ws.numel(),
                                     _cabi.dptr(b["err"]), _cabi.stream_ptr(dev)), "yr_cdae_step_ex")
        if train:
            self.optimizer.step_count += 1

    def _step_idx(self, data, train: bool, step_loss=None, keep_vals=None):
        """One step from an index-list batch (data/cdae_sparse.py): nothing of size B x num_items crosses PCIe or exists in HBM."""
        lib = _cabi.load()
        m = self.model
        b, g, mo, vo = self._state()
        dev = self.device
        mv = lambda k, dt: data[k].to(device=dev, dtype=dt, non_blocking=True).contiguous()
        uid, in_ptr, in_idx = mv("user_id", I64), mv("input_ptr", I32), mv("input_idx", I32)
        ls_ptr, ls_idx, ls_val = mv("loss_ptr", I32), mv("loss_idx", I32), mv("loss_val", F32)
        B = int(uid.numel())
        in_val = None
        if train:
            if keep_vals is not None:
                in_val = keep_vals.to(device=dev, dtype=F32).contiguous()
            else:
                p_drop = float(m.corruption_level)
                in_val = ((torch.rand(in_idx.numel(), device=dev) >= p_drop).to(F32) / (1.0 - p_drop)) if p_drop > 0 else None
        ws = m.workspace(B)
        P = m.tensors()
        opt = self.optimizer.opt_struct(self.optimizer.step_count + 1) if train else None
        _cabi.check(lib.yr_cdae_step_idx(C.byref(P), C.byref(g) if train else None,
                                         C.byref(mo) if (train and mo is not None) else None,
                                         C.byref(vo) if (train and vo is not None) else None,
                                         C.byref(opt) if train else None, self.num_users, self.num_items, m.hidden_size,
                                         m.hidden_act, _cabi.dptr(uid), _cabi.dptr(in_ptr), _cabi.dptr(in_idx),
                                         _cabi.dptr(in_val) if in_val is not None else None, _cabi.dptr(ls_ptr),
                                         _cabi.dptr(ls_idx), _cabi.dptr(ls_val), B, _cabi.dptr(b["loss"]),
                                         _cabi.dptr(step_loss) if step_loss is not None else None, _cabi.dptr(ws), ws.numel(),
                                         _cabi.dptr(b["err"]), _cabi.stream_ptr(dev)), "yr_cdae_step_idx")
        if train:
            self.optimizer.step_count += 1

    def _loss_sum(self) -> float:
        b = self._bufs
        v = float(b["loss"][0].item())
        ops._raise_if_err(b["err"], "CDAETrainer")
        b["loss"].zero_()
        return v

    def train(self, train_dataloader, keeps=None) -> float:
        """`keeps`: optional iterable of dropout multipliers (one [B x num_items] tensor per batch) to replay a run with
        the masks another implementation drew; by default they are drawn on the device like nn.Dropout does."""
        if not self.model.training:
            self.model.train()
        self._state()[0]["loss"].zero_()
        keeps = iter(keeps) if keeps is not None else None
        losses = []
        for data in train_dataloader:
            sl = torch.empty(1, device=self.device, dtype=F32)
            if "input_idx" in data:                         # index-list batch (data/cdae_sparse.py): `keeps` = values per listed input
                self._step_idx(data, True, sl, next(keeps) if keeps is not None else None)
                losses.append(sl)
                continue
            x = data["input_mask"].to(self.device, dtype=F32)
            keep = next(keeps).to(self.device, dtype=F32).contiguous() if keeps is not None else self.model.draw_keep(x)
            self._step(data["user_id"], x, keep, x, data["negative_mask"], True, sl)
            losses.append(sl)
        if not losses:
            return 0
        self.last_step_losses = torch.cat(losses)
        return self._loss_sum()

    # ------------------------------------------------------------------------------------------
    # ---- ranking: streamed batch by batch (the reference streams too, cdae_trainer.py:123-144) -----------------------
    def _rank_begin(self):
        return {"z": [], "mask": [], "act": [], "n": 0}

    @staticmethod
    def _rows_of(mask: torch.Tensor):
        """Dense multi-hot [B x nI] (already on the device) -> (count per row [B] int64, column ids int32, row-major)."""
        nz = mask != 0
        return nz.sum(dim=1), nz.nonzero(as_tuple=False)[:, 1].to(I32)

    def _rank_add(self, acc, user_id, x_dev: torch.Tensor, actual_dev: torch.Tensor) -> None:
        """Hidden activations of one batch + the CSR pieces of its mask / ground-truth rows; nothing of size
        B x num_items outlives the batch."""
        m = self.model
        acc["z"].append(m.hidden(user_id, x_dev, None, ldz=_ldz(m.hidden_size)))
        acc["mask"].append(self._rows_of(x_dev))
        acc["act"].append(self._rows_of(actual_dev))
        acc["n"] += int(x_dev.shape[0])

    def _rank_finish(self, acc):
        """One fused top-K + metrics pass over every accumulated row."""
        m, n, dev = self.model, acc["n"], self.device
        if n == 0:
            raise ZeroDivisionError("division by zero")       # what metric.py does on an empty evaluation set
        Z = torch.cat(acc["z"])
        V = torch.zeros(self.num_items, _ldz(m.hidden_size), device=dev, dtype=F32)
        V[:, : m.hidden_size] = m.output_layer.weight.data
        V[:, m.hidden_size] = m.output_layer.bias.data

        def csr(parts):
            cnt = torch.cat([c for c, _ in parts])
            idx = torch.cat([i for _, i in parts])
            ptr = torch.zeros(n + 1, device=dev, dtype=I64)
            ptr[1:] = torch.cumsum(cnt, 0)
            return ptr.to(I32), idx, cnt.to(I32)

        mask_ptr, mask_idx, _ = csr(acc["mask"])
        act_ptr, act_idx, act_cnt = csr(acc["act"])
        ecsr = ops.DeviceEvalCSR.from_device(torch.arange(n, device=dev, dtype=I64), mask_ptr, mask_idx, act_ptr, act_idx,
                                             act_cnt, int(self.cfg.top_n))
        topk, _, _, sums, err = ops.eval_topk_metrics(Z, V, ecsr)
        self.last_topk = topk
        sums_h = sums.cpu()
        return ops.metrics_from_sums(sums_h, n)

    def validate(self, valid_dataloader) -> tuple:
        self.model.eval()
        self._state()[0]["loss"].zero_()
        acc = self._rank_begin()
        for data in valid_dataloader:                         # one pass: loss step + hidden activations per batch
            x = data["input_mask"].to(self.device, dtype=F32)
            vm = data["valid_mask"].to(self.device, dtype=F32)
            self._step(data["user_id"], x, None, x + vm, data["negative_mask"], False)   # train + valid 1 (cdae_trainer.py:67)
            self._rank_add(acc, data["user_id"], x, vm)
        valid_loss = self._loss_sum() if acc["n"] else 0
        p, r, mp, nd = self._rank_finish(acc)
        return (valid_loss, p, r, mp, nd)

    def evaluate(self, test_dataloader) -> tuple:
        self.model.eval()
        acc = self._rank_begin()
        for data in test_dataloader:
            x = data["input_mask"].to(self.device, dtype=F32)
            self._rank_add(acc, data["user_id"], x, data["test_mask"].to(self.device, dtype=F32))
        result = self._rank_finish(acc)
        k = self.cfg.top_n
        logger.info(f"[Trainer] Test > precision@{k} : {result[0]:.4f} / Recall@{k}: {result[1]:.4f} / "
                    f"MAP@{k}: {result[2]:.4f} / NDCG@{k}: {result[3]:.4f}")
        return result

    def recommender(self, seen=None, subsets=None, locations=None):
        """retrieval.CDAERecommender over the model's live parameters (recommend(user_ids, k, exclude_seen=True,
        subset=None, near=None, radius_km=None); scores are output logits). `seen` is required: it is the users' input as
        well as what is excluded."""
        from ..retrieval import CDAERecommender
        return CDAERecommender(self.model, seen, subsets, locations)

    def run(self, train_dataloader, valid_dataloader):
        """Epoch loop of trainers/base_trainer.py:49-115 (validate returns the 5-tuple for CDAE)."""
        best = (1e+6, .0, .0, .0, .0)
        endurance = 0
        for epoch in range(self.cfg.epochs):
            train_loss = self.train(train_dataloader)
            current = self.validate(valid_dataloader)
            logger.info(f"[Trainer] epoch: {epoch} > train loss: {train_loss:.4f} / valid loss: {current[0]:.4f} / "
                        f"precision@K : {current[1]:.4f} / Recall@K: {current[2]:.4f} / MAP@K: {current[3]:.4f} / "
                        f"NDCG@K: {current[4]:.4f}")
            if self._is_surpass_best_metric(current=current, best=best):
                best, endurance = current, 0
                torch.save(self.model.state_dict(), f"{self.cfg.model_dir}/best_model.pt")
            else:
                endurance += 1
                if endurance > self.cfg.patience:
                    break
