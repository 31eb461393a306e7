"""Drop-in for the reference's trainers/ngcf_trainer.py:22-182 on the sm_100a kernels.

`train` runs one yr_ngcf_train_step per batch (3 fused layer forwards, gather/dot/BPR tail, 3 layer backwards,
dense optimizer over embedding + W1/W2) with no autograd graph and no N x N identity; `validate` propagates ONCE
per call and scores every batch on the resulting layer outputs (parameters do not change inside validate);
`evaluate` propagates once, concatenates the layer outputs and runs the same fused top-K/metrics kernel as MF.

Quirk Q12: the reference evaluates 100 rows drawn with np.random.randint (with replacement) and re-propagates the
whole graph for each. `cfg.ngcf_eval_mode = 'sample100'` reproduces that row draw (same global NumPy RNG call);
the default 'full' evaluates every row of eval_data, which is what BASELINE.json config 3 asks for.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from .. import _cabi, ops
from ..data.graph import EvalCSR, eval_csr_from_frame
from ..loss import BPRLoss
from ..models.ngcf import NGCF, _LEAKY_SLOPE
from .base_trainer import BaseTrainer, BatchStager, FusedOptimizer, logger

I32, I64, F32, F64 = torch.int32, torch.int64, torch.float32, torch.float64


class NGCFTrainer(BaseTrainer):
    def __init__(self, cfg, num_items: int, num_users: int, laplacian_matrix) -> None:
        super().__init__(cfg)
        logger.info(f"[DEVICE] device = {self.device}")
        self.num_items = num_items
        self.num_users = num_users
        self.model = NGCF(self.cfg, num_users, num_items).to(self.device)
        self.optimizer: FusedOptimizer = self._optimizer(self.cfg.optimizer, self.model, self.cfg.lr,
                                                         self.cfg.weight_decay)
        self.loss = self._loss()
        self.laplacian_matrix = laplacian_matrix
        self._bufs = None
        # batches up to this many triples use the row-sparse top-layer backward (larger ones run it densely)
        self._row_cap = max(int(getattr(cfg, "batch_size", 0) or 0), 4096)
        self._stager = None
        self._eval_cache = {}
        self.last_step_losses = None
        self.last_topk = None

    def _loss(self):
        return BPRLoss()

    # ------------------------------------------------------------------------------------------
    def _state(self):
        m = self.model
        dev = self.device
        # the ctypes struct only holds pointers: rebuild it when one of them changed (load_state_dict, new optimizer state)
        key = (m.embedding.weight.data_ptr(), tuple(w.weight.data_ptr() for w in m.W1), tuple(w.weight.data_ptr() for w in m.W2),
               id(self.laplacian_matrix), self._bufs is not None and self._bufs["E0_ptr"],
               int(m.dense_mode), int(getattr(self.cfg, "ngcf_top_rows_mode", 1)))
        hit = getattr(self, "_st_cache", None)
        if hit is not None and hit[0] == key:
            return hit[1], self._bufs
        st, b = self._build_state()
        key = key[:4] + (b["E0_ptr"],) + key[5:]
        self._st_cache = (key, st)
        return st, b

    def _build_state(self):
        m = self.model
        dev = self.device
        csr = m.csr(self.laplacian_matrix)
        E0 = m.embedding.weight.data
        n, d = E0.shape
        L = len(m.W1)
        if L > _cabi.YR_NGCF_MAX_LAYERS:
            raise _cabi.YelprecError(f"num_orders={L} exceeds {_cabi.YR_NGCF_MAX_LAYERS}")
        b = self._bufs
        if b is None or b["E0_ptr"] != E0.data_ptr():
            lib = _cabi.load()
            z = lambda *s, dt=F32: torch.zeros(*s, device=dev, dtype=dt)
            b = {"E0_ptr": E0.data_ptr(),
                 "E": [z(n, d) for _ in range(L)], "LE": [z(n, d) for _ in range(L)],
                 "G": [z(n, d) for _ in range(L + 1)], "T": z(n, d),
                 "dW1": [z(d, d) for _ in range(L)], "dW2": [z(d, d) for _ in range(L)],
                 "loss": z(2, dt=F64), "err": z(1, dt=I32),
                 # row scratch of the row-sparse top-layer backward (flags / count stay zero between steps)
                 "row_flag": z(n, dt=I32), "row_list": z(3 * self._row_cap, dt=I32), "row_count": z(1, dt=I32)}
            nbytes = lib.yr_ngcf_layer_bwd_ws_bytes(d)
            b["ws"] = torch.empty(nbytes, device=dev, dtype=torch.uint8)
            b["E_dev"] = ops.device_ptr_array([E0] + b["E"])
            b["G_dev"] = ops.device_ptr_array(b["G"])
            if self.optimizer.needs_moments and "E" not in self.optimizer.state:
                self.optimizer.state["E"] = (z(n, d), z(n, d))
                self.optimizer.state["W1"] = [(z(d, d), z(d, d)) for _ in range(L)]
                self.optimizer.state["W2"] = [(z(d, d), z(d, d)) for _ in range(L)]
            self._bufs = b
        st = _cabi.YrNgcfState()
        st.nU, st.nI, st.d, st.n_layers = self.num_users, self.num_items, d, L
        p = _cabi.dptr
        st.L, st.LT = csr.fwd.struct(d), csr.bwd.struct(d)
        st.E[0] = p(E0, F32)
        st.G[0] = p(b["G"][0])
        for l in range(L):
            st.E[l + 1], st.LE[l], st.G[l + 1] = p(b["E"][l]), p(b["LE"][l]), p(b["G"][l + 1])
            st.W1[l], st.W2[l] = p(m.W1[l].weight.data, F32), p(m.W2[l].weight.data, F32)
            st.dW1[l], st.dW2[l] = p(b["dW1"][l]), p(b["dW2"][l])
            if self.optimizer.needs_moments:
                st.mW1[l], st.vW1[l] = map(p, self.optimizer.state["W1"][l])
                st.mW2[l], st.vW2[l] = map(p, self.optimizer.state["W2"][l])
        if self.optimizer.needs_moments:
            st.mE, st.vE = map(p, self.optimizer.state["E"])
        st.T = p(b["T"])
        st.E_dev, st.G_dev = p(b["E_dev"]), p(b["G_dev"])
        st.ws, st.ws_bytes = p(b["ws"]), b["ws"].numel()
        st.loss, st.err = p(b["loss"]), p(b["err"])
        st.row_flag, st.row_list, st.row_count = p(b["row_flag"]), p(b["row_list"]), p(b["row_count"])
        st.row_list_cap = b["row_list"].numel()
        st.dense_mode = int(m.dense_mode)
        st.top_rows_mode = int(getattr(self.cfg, "ngcf_top_rows_mode", 1))
        return st, b

    def _get_stager(self, dataloader) -> BatchStager:
        cap = int(getattr(dataloader, "batch_size", None) or 0)
        if cap <= 0:
            try:
                cap = max(int(x["user_id"].numel()) for x in dataloader)
            except TypeError:
                cap = int(getattr(self.cfg, "batch_size", 2048))
        if self._stager is None or self._stager.cap < cap:
            self._stager = BatchStager(self.device, max(cap, 1), int(getattr(self.cfg, "steps_per_launch", 16)))
        return self._stager

    def train_step_on_device(self, uid, pos, neg, step_loss=None, _st=None) -> None:
        """One optimizer step on a batch already resident in HBM."""
        lib = _cabi.load()
        st = _st if _st is not None else self._state()[0]
        opt = self.optimizer.opt_struct(self.optimizer.step_count + 1)
        prefix = self._take_prefix()
        _cabi.check(lib.yr_ngcf_train_step_ex(C.byref(st), C.byref(opt), _LEAKY_SLOPE, _cabi.dptr(uid, I64),
                                              _cabi.dptr(pos, I64), _cabi.dptr(neg, I64), int(uid.numel()),
                                              _cabi.dptr(step_loss) if step_loss is not None else None, prefix,
                                              _cabi.stream_ptr(self.device)), "yr_ngcf_train_step_ex")
        self.optimizer.step_count += 1

    # ---- batch-independent part of the next step, enqueued while the host reads the loss back -----------------
    def _param_versions(self):
        m = self.model
        return (m.embedding.weight._version, m.embedding.weight.data_ptr(), tuple(w.weight._version for w in m.W1),
                tuple(w.weight._version for w in m.W2), self.optimizer.step_count, id(self.laplacian_matrix))

    def _take_prefix(self) -> int:
        """Number of leading layers already propagated for the CURRENT parameters (0 unless _prepropagate ran and nothing
        touched the parameters since — Python-side writes bump the tensors' versions, our steps bump step_count)."""
        tag = getattr(self, "_prefix_tag", None)
        self._prefix_tag = None
        if tag is not None and tag[0] == self._param_versions():
            return tag[1]
        return 0

    def _prepropagate(self, st) -> None:
        n_prefix = int(st.n_layers) - 1            # the last layer depends on the batch rows (row-sparse), the others do not
        if n_prefix <= 0:
            return
        lib = _cabi.load()
        _cabi.check(lib.yr_ngcf_propagate_prefix(C.byref(st), _LEAKY_SLOPE, n_prefix, _cabi.stream_ptr(self.device)),
                    "yr_ngcf_propagate_prefix")
        self._prefix_tag = (self._param_versions(), n_prefix)

    def loss_sum(self, reset=True, prepropagate_state=None) -> float:
        """Running sum of batch-mean losses; one event synchronisation brings the loss and the bad-id flag back. With
        `prepropagate_state` the batch-independent layers of the NEXT step are enqueued behind the copies, so the GPU
        is busy while the host returns the loss and stages the next batch (include/yelprec_b200.h)."""
        b = self._bufs
        h = b.get("host_out")
        if h is None:
            h = b["host_out"] = (torch.empty(2, dtype=F64).pin_memory(), torch.empty(1, dtype=I32).pin_memory(),
                                 torch.cuda.Event())
        h[0].copy_(b["loss"], non_blocking=True)
        h[1].copy_(b["err"], non_blocking=True)
        h[2].record(torch.cuda.current_stream(self.device))
        if reset:
            b["loss"].zero_()                      # stream-ordered after the copy
        if prepropagate_state is not None and self.model.training:
            self._prepropagate(prepropagate_state)
        h[2].synchronize()
        v = float(h[0][0])
        if int(h[1][0]) != 0:
            # like the other fused trainers, the step that saw the bad id has already been applied (the reference raises
            # before its update); INTEGRATION.md states this difference
            ops._raise_if_err(b["err"], "NGCFTrainer")
        return v

    def train(self, train_dataloader) -> float:
        if not self.model.training:
            self.model.train()
        st, b = self._state()
        b["loss"].zero_()
        if hasattr(train_dataloader, "epoch_triples"):        # data.sampler.DeviceTripleLoader: epoch resident in HBM
            uid, pos, neg = train_dataloader.epoch_triples()
            B, n = int(train_dataloader.batch_size), int(uid.numel())
            if n == 0:
                return 0
            sl = torch.empty((n + B - 1) // B, device=self.device, dtype=F32)
            for k, s in enumerate(range(0, n, B)):
                self.train_step_on_device(uid[s:s + B], pos[s:s + B], neg[s:s + B], sl[k:k + 1], st)
            self.last_step_losses = sl
            return self.loss_sum(prepropagate_state=st)
        stager = self._get_stager(train_dataloader)
        losses = []
        for uid, pos, neg, n, B in stager.chunks(train_dataloader):
            sl = torch.empty((n + B - 1) // B, device=self.device, dtype=F32)
            for k, s in enumerate(range(0, n, B)):
                self.train_step_on_device(uid[s:s + B], pos[s:s + B], neg[s:s + B], sl[k:k + 1], st)
            losses.append(sl)
        if not losses:
            return 0
        self.last_step_losses = torch.cat(losses) if len(losses) > 1 else losses[0]
        return self.loss_sum(prepropagate_state=st)

    def propagate(self):
        """E_0..E_L after one propagation of the current parameters (device tensors, not copies)."""
        lib = _cabi.load()
        st, b = self._state()
        _cabi.check(lib.yr_ngcf_propagate(C.byref(st), _LEAKY_SLOPE, _cabi.stream_ptr(self.device)), "yr_ngcf_propagate")
        return [self.model.embedding.weight.data] + b["E"], st, b

    def validate(self, valid_dataloader) -> float:
        self.model.eval()
        lib = _cabi.load()
        _, st, b = self.propagate()
        b["loss"].zero_()
        stager = self._get_stager(valid_dataloader)
        d, L = st.d, st.n_layers
        for uid, pos, neg, n, B in stager.chunks(valid_dataloader):
            for s in range(0, n, B):
                u, p, q = uid[s:s + B], pos[s:s + B], neg[s:s + B]
                _cabi.check(lib.yr_ngcf_tail(st.E_dev, None, L, self.num_users, self.num_items, d, _cabi.dptr(u, I64),
                                             _cabi.dptr(p, I64), _cabi.dptr(q, I64), int(u.numel()), None, None, st.loss,
                                             None, st.err, _cabi.stream_ptr(self.device)), "yr_ngcf_tail")
        return self.loss_sum()

    # ------------------------------------------------------------------------------------------
    def _eval_csr(self, eval_data) -> ops.DeviceEvalCSR:
        mode = getattr(self.cfg, "ngcf_eval_mode", "full")
        if mode == "sample100" and not isinstance(eval_data, EvalCSR):
            # same global-RNG draw as trainers/ngcf_trainer.py:140 (rows, with replacement)
            rows = np.random.randint(eval_data.shape[0], size=100)
            sub = eval_data.iloc[rows, :]
            return ops.DeviceEvalCSR(eval_csr_from_frame(sub, self.num_items), self.device, int(self.cfg.top_n))
        # the cache entry holds the frame itself and is compared by identity (an id() alone can be recycled)
        hit = self._eval_cache.get("entry")
        if hit is None or hit[0] is not eval_data or hit[1] != int(self.cfg.top_n):
            csr = eval_data if isinstance(eval_data, EvalCSR) else eval_csr_from_frame(eval_data, self.num_items)
            hit = (eval_data, int(self.cfg.top_n), ops.DeviceEvalCSR(csr, self.device, int(self.cfg.top_n)))
            self._eval_cache = {"entry": hit}
        return hit[2]

    def evaluate(self, eval_data, mode="valid") -> tuple:
        self.model.eval()
        ecsr = self._eval_csr(eval_data)
        layers, _, _ = self.propagate()
        cat = ops.ngcf_concat(layers)
        users, items = cat[: self.num_users], cat[self.num_users:]
        topk, _, _, sums, err = ops.eval_topk_metrics(users, items, ecsr, mode=getattr(self.cfg, "eval_mode", None))
        self.last_topk = topk
        sums_h = sums.cpu()
        ops._raise_if_err(err, "NGCFTrainer.evaluate")
        result = ops.metrics_from_sums(sums_h, ecsr.n_eval)
        if mode == "test":
            k = self.cfg.top_n
            logger.info(f"[Trainer] Test > precision@{k} : {result[0]:.4f} / Recall@{k}: {result[1]:.4f} / "
                        f"MAP@{k}: {result[2]:.4f} / NDCG@{k}: {result[3]:.4f}")
        return result

    def recommender(self, seen=None, subsets=None, locations=None):
        """retrieval.Recommender over the propagated, layer-concatenated user / item embeddings that evaluate() ranks with;
        recommend_diverse measures similarity in the concatenated item rows, and recommend_group aggregates the members'
        scores over the same rows."""
        from ..retrieval import Recommender
        cat = ops.ngcf_concat(self.propagate()[0])
        return Recommender(cat[: self.num_users], cat[self.num_users:], seen, subsets, locations)

    def _generate_top_k_recommendation(self, pred: torch.Tensor, mask_items) -> np.ndarray:
        if not pred.is_cuda:
            raise _cabi.YelprecError("expected a CUDA score tensor (no CPU fallback)")
        return ops.topk_masked_row(pred, mask_items, int(self.cfg.top_n)).cpu().numpy()
