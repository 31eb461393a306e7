"""Drop-in for the reference's trainers/mf_trainer.py:22-178 on the sm_100a kernels.

Same constructor order `(cfg, num_items, num_users)` (quirk Q17) and the same methods. `train` feeds the
persistent fused kernel (yr_bpr_mf_train): per batch forward x2 + BPR loss + sparse gradient accumulate + one
optimizer update per row, no autograd, no dense gradient, `loss.item()` replaced by one device-side running sum
read back once per call (the returned value is still the SUM of batch-mean losses, quirk Q1).
`evaluate` runs the fused score+mask+top-K+metrics kernel (yr_eval_topk_metrics) over all eval rows at once.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from .. import _cabi, ops
from ..data.graph import eval_csr_from_frame
from ..loss import BPRLoss
from ..models.mf import MatrixFactorization
from .base_trainer import BaseTrainer, BatchStager, FusedOptimizer, logger

I32, I64, F32, F64 = torch.int32, torch.int64, torch.float32, torch.float64


class MFTrainer(BaseTrainer):
    def __init__(self, cfg, num_items: int, num_users: int) -> None:
        super().__init__(cfg)
        self.num_items = num_items
        self.num_users = num_users
        if self.cfg.embed_size not in (32, 64, 128, 256, 512, 1024):
            raise _cabi.YelprecError(f"MF embed_size {self.cfg.embed_size}: the fused trainer takes 32, 64, 128, 256, 512, 1024 "
                                     "(the values of the reference's mf_sweep_config.yaml)")
        self.model = MatrixFactorization(self.cfg, num_users, num_items).to(self.device)
        self.optimizer: FusedOptimizer = self._optimizer(self.cfg.optimizer, self.model, self.cfg.lr,
                                                         self.cfg.weight_decay)
        self.loss = self._loss()
        self._scratch = None
        self._stager = None
        self._eval_cache = {}
        self.last_step_losses = None
        self.last_topk = None

    def _loss(self):
        return BPRLoss()

    # ------------------------------------------------------------------------------------------
    def _state(self, batch_cap: int, n_triples: int = 0):
        """Device scratch of the fused kernel (allocated once; the flags' all-zero invariant is kept by the kernel)."""
        U, V = self.model.user_embedding.weight, self.model.item_embedding.weight
        dev = self.device
        if self._scratch is None or self._scratch["cap"] < batch_cap or self._scratch["U_ptr"] != U.data_ptr():
            z = lambda *s, dt=F32: torch.zeros(*s, device=dev, dtype=dt)
            sc = {"cap": batch_cap, "U_ptr": U.data_ptr(),
                  "flagU": z(U.shape[0], dt=I32), "flagV": z(V.shape[0], dt=I32), "counters": z(16, dt=I32),
                  "err": z(1, dt=I32), "loss_sum": z(1, dt=F64), "ws": None}
            if self.optimizer.needs_moments and "U" not in self.optimizer.state:
                self.optimizer.state["U"] = (z(*U.shape), z(*U.shape))
                self.optimizer.state["V"] = (z(*V.shape), z(*V.shape))
            self._scratch = sc
        sc = self._scratch
        need = _cabi.load().yr_bpr_mf_train_ws_bytes(max(int(n_triples), 1), int(batch_cap), int(U.shape[1]))
        if sc["ws"] is None or sc["ws"].numel() < need:
            sc["ws"] = torch.empty(need, device=dev, dtype=torch.uint8)
        mU = vU = mV = vV = None
        if self.optimizer.needs_moments:
            (mU, vU), (mV, vV) = self.optimizer.state["U"], self.optimizer.state["V"]
        p = _cabi.dptr
        st = _cabi.YrMfState(p(U.data, F32), p(V.data, F32), p(mU), p(vU), p(mV), p(vV),
                             p(sc["flagU"]), p(sc["flagV"]), p(sc["counters"]), p(sc["err"]),
                             p(sc["ws"]), sc["ws"].numel(), U.shape[0], V.shape[0], U.shape[1],
                             1 if getattr(self.cfg, "deterministic", False) else 0)
        return st, sc

    def _get_stager(self, dataloader) -> BatchStager:
        cap = int(getattr(dataloader, "batch_size", None) or 0)
        if cap <= 0:
            try:
                cap = max(int(b["user_id"].numel()) for b in dataloader)
            except TypeError:
                cap = int(getattr(self.cfg, "batch_size", 2048))
        cap = max(cap, 1)
        if self._stager is None or self._stager.cap < cap:
            chunk = int(getattr(self.cfg, "steps_per_launch", 64))
            self._stager = BatchStager(self.device, cap, chunk)
        return self._stager

    def train_on_device(self, uid: torch.Tensor, pos: torch.Tensor, neg: torch.Tensor, batch_size: int,
                        step_loss: torch.Tensor = None) -> None:
        """Hot loop with the triples already resident in HBM: ONE launch for all batches. The running loss sum
        stays on the device (read it with `.loss_sum()`)."""
        lib = _cabi.load()
        n = int(uid.numel())
        st, sc = self._state(batch_size, n)
        n_steps = (n + batch_size - 1) // batch_size
        opt = self.optimizer.opt_struct(self.optimizer.step_count + 1)
        _cabi.check(lib.yr_bpr_mf_train(C.byref(st), C.byref(opt), _cabi.dptr(uid, I64), _cabi.dptr(pos, I64),
                                        _cabi.dptr(neg, I64), n, batch_size, _cabi.dptr(sc["loss_sum"]),
                                        _cabi.dptr(step_loss) if step_loss is not None else None,
                                        _cabi.stream_ptr(self.device)), "yr_bpr_mf_train")
        self.optimizer.step_count += n_steps

    def loss_sum(self, reset=True) -> float:
        sc = self._scratch
        v = float(sc["loss_sum"].item())
        ops._raise_if_err(sc["err"], "MFTrainer.train")
        if reset:
            sc["loss_sum"].zero_()
        return v

    def train(self, train_dataloader) -> float:
        if not self.model.training:
            self.model.train()
        if hasattr(train_dataloader, "epoch_triples"):        # data.sampler.DeviceTripleLoader: epoch resident in HBM
            uid, pos, neg = train_dataloader.epoch_triples()
            B = int(train_dataloader.batch_size)
            self._state(B)[1]["loss_sum"].zero_()
            if uid.numel() == 0:
                return 0
            sl = torch.empty((uid.numel() + B - 1) // B, device=self.device, dtype=F32)
            self.train_on_device(uid, pos, neg, B, sl)
            self.last_step_losses = sl
            return self.loss_sum()
        stager = self._get_stager(train_dataloader)
        self._state(stager.cap)[1]["loss_sum"].zero_()
        step_losses = []
        for uid, pos, neg, n, B in stager.chunks(train_dataloader):
            sl = torch.empty((n + B - 1) // B, device=self.device, dtype=F32)
            self.train_on_device(uid, pos, neg, B, sl)
            step_losses.append(sl)
        if not step_losses:
            return 0
        total = self.loss_sum()
        self.last_step_losses = torch.cat(step_losses)
        return total

    def validate(self, valid_dataloader) -> float:
        self.model.eval()
        lib = _cabi.load()
        stager = self._get_stager(valid_dataloader)
        U, V = self.model.user_embedding.weight.data, self.model.item_embedding.weight.data
        loss_sum = torch.zeros(1, device=self.device, dtype=F64)
        err = torch.zeros(1, device=self.device, dtype=I32)
        for uid, pos, neg, n, B in stager.chunks(valid_dataloader):
            _cabi.check(lib.yr_bpr_mf_validate(_cabi.dptr(U, F32), _cabi.dptr(V, F32), U.shape[0], V.shape[0], U.shape[1],
                                               _cabi.dptr(uid, I64), _cabi.dptr(pos, I64), _cabi.dptr(neg, I64), n, B,
                                               _cabi.dptr(loss_sum), None, _cabi.dptr(err),
                                               _cabi.stream_ptr(self.device)), "yr_bpr_mf_validate")
        total = float(loss_sum.item())
        ops._raise_if_err(err, "MFTrainer.validate")
        return total

    # ------------------------------------------------------------------------------------------
    def _eval_csr(self, eval_data) -> ops.DeviceEvalCSR:
        # the cache entry holds the frame itself and is compared by identity (an id() alone can be recycled); a frame
        # that is mutated in place between calls must be passed as a new object
        hit = self._eval_cache.get("entry")
        if hit is None or hit[0] is not eval_data or hit[1] != int(self.cfg.top_n):
            csr = eval_data if hasattr(eval_data, "eval_uid") else eval_csr_from_frame(eval_data, self.num_items)
            hit = (eval_data, int(self.cfg.top_n), ops.DeviceEvalCSR(csr, self.device, int(self.cfg.top_n)))
            self._eval_cache = {"entry": hit}
        return hit[2]

    def evaluate(self, eval_data, mode="valid") -> tuple:
        """eval_data: the reference's DataFrame (index user_id, list columns pos_items / mask_items) or a prebuilt
        data.graph.EvalCSR. Returns (precision@K, recall@K, map@K, ndcg@K) as Python floats."""
        self.model.eval()
        ecsr = self._eval_csr(eval_data)
        U, V = self.model.user_embedding.weight.data, self.model.item_embedding.weight.data
        topk, _, _, sums, err = ops.eval_topk_metrics(U, V, ecsr, mode=getattr(self.cfg, "eval_mode", None))
        self.last_topk = topk
        sums_h = sums.cpu()
        ops._raise_if_err(err, "MFTrainer.evaluate")
        result = ops.metrics_from_sums(sums_h, ecsr.n_eval)
        if mode == "test":
            k = self.cfg.top_n
            logger.info(f"[Trainer] Test > precision@{k} : {result[0]:.4f} / Recall@{k}: {result[1]:.4f} / "
                        f"MAP@{k}: {result[2]:.4f} / NDCG@{k}: {result[3]:.4f}")
        return result

    def recommender(self, seen=None, subsets=None, locations=None):
        """retrieval.Recommender over the current user / item tables (recommend(user_ids, k, exclude_seen=True, subset=None,
        near=None, radius_km=None), recommend_diverse(user_ids, k, lam=0.5, pool=None, ...) for a diverse list re-ranked
        from a pool of recommend's best, and recommend_group(groups, k, agg="mean", ...) for one list per group of users
        ranked by the members' least-misery or mean score)."""
        from ..retrieval import Recommender
        return Recommender(self.model.user_embedding.weight.data, self.model.item_embedding.weight.data, seen, subsets,
                           locations)

    def _generate_top_k_recommendation(self, pred: torch.Tensor, mask_items) -> np.ndarray:
        """One score row -> top-K item ids, best first (mf_trainer.py:163-178). Ties: (score desc, id asc)."""
        if not pred.is_cuda:
            raise _cabi.YelprecError("expected a CUDA score tensor (no CPU fallback)")
        return ops.topk_masked_row(pred, mask_items, int(self.cfg.top_n)).cpu().numpy()
