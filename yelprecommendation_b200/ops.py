"""Tensor-level wrappers over the C ABI (include/yelprec_b200.h) + autograd glue.

Every function here launches hand-written sm_100a kernels from libyelprec_b200.so on the current CUDA
stream. CPU tensors are rejected: the product has no CPU path (the CPU restatement lives in oracle/ and is
test infrastructure only).
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch
from torch.library import custom_op

from . import _cabi
from ._cabi import YelprecError, check, dptr, stream_ptr

F32, I64, I32, F64 = torch.float32, torch.int64, torch.int32, torch.float64


def _ids(t: torch.Tensor, device) -> torch.Tensor:
    if not torch.is_tensor(t):
        t = torch.as_tensor(t)
    t = t.to(device=device, dtype=I64, non_blocking=True)
    return t.contiguous()


def _raise_if_err(err: torch.Tensor, what: str) -> None:
    """reference behaviour: nn.Embedding raises IndexError on an out-of-range id."""
    if int(err.item()) != 0:
        err.zero_()
        raise IndexError(f"{what}: index out of range in self")


# ----------------------------------------------------------------------------------------------------
# MF score / BPR loss (autograd-capable, so an unmodified reference trainer can call loss.backward())
# ----------------------------------------------------------------------------------------------------
# Registered as PyTorch custom ops (torch.ops.yelprec.*): each op body is one call into the C ABI; the backward formulas
# are custom ops as well, attached with register_autograd.
@custom_op("yelprec::mf_score", mutates_args=(), device_types="cuda")
def _op_mf_score(U: torch.Tensor, V: torch.Tensor, uid: torch.Tensor, iid: torch.Tensor) -> torch.Tensor:
    """MatrixFactorization.forward (models/mf.py:20-23) -> yr_mf_score."""
    lib = _cabi.load()
    Uc, Vc = U.detach().contiguous(), V.detach().contiguous()
    uid, iid = uid.contiguous(), iid.contiguous()
    out = torch.empty(uid.numel(), device=U.device, dtype=F32)
    err = torch.zeros(1, device=U.device, dtype=I32)
    check(lib.yr_mf_score(dptr(Uc, F32), dptr(Vc, F32), Uc.shape[0], Vc.shape[0], Uc.shape[1],
                          dptr(uid, I64), dptr(iid, I64), uid.numel(), dptr(out), dptr(err),
                          stream_ptr(U.device)), "yr_mf_score")
    _raise_if_err(err, "MatrixFactorization.forward")
    return out


@_op_mf_score.register_fake
def _(U, V, uid, iid):
    return U.new_empty((uid.numel(),), dtype=F32)


@custom_op("yelprec::mf_score_bwd", mutates_args=(), device_types="cuda")
def _op_mf_score_bwd(U: torch.Tensor, V: torch.Tensor, uid: torch.Tensor, iid: torch.Tensor,
                     gout: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    lib = _cabi.load()
    U, V = U.detach().contiguous(), V.detach().contiguous()
    uid, iid = uid.contiguous(), iid.contiguous()
    gU, gV = torch.zeros_like(U), torch.zeros_like(V)
    gout = gout.contiguous().to(F32)
    check(lib.yr_mf_score_bwd(dptr(U, F32), dptr(V, F32), U.shape[0], V.shape[0], U.shape[1], dptr(uid, I64), dptr(iid, I64),
                              uid.numel(), dptr(gout), dptr(gU), dptr(gV), stream_ptr(U.device)),
          "yr_mf_score_bwd")
    return gU, gV


@_op_mf_score_bwd.register_fake
def _(U, V, uid, iid, gout):
    return torch.empty_like(U), torch.empty_like(V)


def _mf_score_setup(ctx, inputs, output):
    ctx.save_for_backward(*inputs)


def _mf_score_backward(ctx, gout):
    U, V, uid, iid = ctx.saved_tensors
    gU, gV = _op_mf_score_bwd(U, V, uid, iid, gout)
    return gU, gV, None, None


_op_mf_score.register_autograd(_mf_score_backward, setup_context=_mf_score_setup)


def mf_score(U: torch.Tensor, V: torch.Tensor, uid: torch.Tensor, iid: torch.Tensor) -> torch.Tensor:
    uid, iid = _ids(uid, U.device), _ids(iid, U.device)
    if uid.numel() != iid.numel():
        raise RuntimeError(f"The size of tensor a ({uid.numel()}) must match the size of tensor b ({iid.numel()})")
    if not U.is_cuda:
        raise YelprecError("MatrixFactorization.forward: expected CUDA tensors (no CPU fallback)")
    return _op_mf_score(U, V, uid, iid)


@custom_op("yelprec::bpr_loss", mutates_args=(), device_types="cuda")
def _op_bpr_loss(pos: torch.Tensor, neg: torch.Tensor) -> torch.Tensor:
    """BPRLoss.forward (loss.py:25-27) -> yr_bpr_loss_fwd."""
    lib = _cabi.load()
    pos, neg = pos.detach().contiguous().to(F32), neg.detach().contiguous().to(F32)
    loss = torch.empty((), device=pos.device, dtype=F32)
    check(lib.yr_bpr_loss_fwd(dptr(pos), dptr(neg), pos.numel(), dptr(loss), stream_ptr(pos.device)),
          "yr_bpr_loss_fwd")
    return loss


@_op_bpr_loss.register_fake
def _(pos, neg):
    return pos.new_empty((), dtype=F32)


@custom_op("yelprec::bpr_loss_bwd", mutates_args=(), device_types="cuda")
def _op_bpr_loss_bwd(pos: torch.Tensor, neg: torch.Tensor, gloss: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    lib = _cabi.load()
    pos, neg = pos.detach().contiguous().to(F32), neg.detach().contiguous().to(F32)
    gpos, gneg = torch.empty_like(pos), torch.empty_like(neg)
    gloss = gloss.contiguous().to(F32)
    check(lib.yr_bpr_loss_bwd(dptr(pos), dptr(neg), pos.numel(), dptr(gloss), dptr(gpos), dptr(gneg),
                              stream_ptr(pos.device)), "yr_bpr_loss_bwd")
    return gpos, gneg


@_op_bpr_loss_bwd.register_fake
def _(pos, neg, gloss):
    return torch.empty_like(pos, dtype=F32), torch.empty_like(neg, dtype=F32)


def _bpr_loss_setup(ctx, inputs, output):
    ctx.save_for_backward(*inputs)


def _bpr_loss_backward(ctx, gloss):
    pos, neg = ctx.saved_tensors
    return _op_bpr_loss_bwd(pos, neg, gloss)


_op_bpr_loss.register_autograd(_bpr_loss_backward, setup_context=_bpr_loss_setup)


def bpr_loss(pos: torch.Tensor, neg: torch.Tensor) -> torch.Tensor:
    if not pos.is_cuda:
        raise YelprecError("BPRLoss: expected CUDA tensors (no CPU fallback)")
    return _op_bpr_loss(pos, neg)


# ----------------------------------------------------------------------------------------------------
# SpMM / NGCF layer (autograd-capable)
# ----------------------------------------------------------------------------------------------------
def spmm_csr(A, X: torch.Tensor, out: Optional[torch.Tensor] = None, accumulate=False):
    """A: data.graph.CSRMatrix. Returns A @ X (or out += A @ X)."""
    lib = _cabi.load()
    X = X.contiguous()
    if out is None:
        out = torch.empty_like(X)
        accumulate = False
    st = A.struct(X.shape[1])
    check(lib.yr_spmm_csr(C.byref(st), X.shape[1], dptr(X, F32), dptr(out, F32), 1 if accumulate else 0,
                          stream_ptr(X.device)), "yr_spmm_csr")
    return out


def ngcf_layer_fwd(csr, E, W1, W2, slope=0.01, dense_mode: int = _cabi.YR_DENSE_TC_FWD):
    """csr: data.graph.LaplacianCSR. dense_mode: yr_dense_mode (include/yelprec_b200.h)."""
    lib = _cabi.load()
    E, W1, W2 = E.contiguous(), W1.contiguous(), W2.contiguous()
    En, LE = torch.empty_like(E), torch.empty_like(E)
    st = csr.fwd.struct(E.shape[1])
    check(lib.yr_ngcf_layer_fwd(C.byref(st), E.shape[1], dptr(E, F32), dptr(W1, F32), dptr(W2, F32), float(slope),
                                dptr(En), dptr(LE), int(dense_mode), stream_ptr(E.device)), "yr_ngcf_layer_fwd")
    return En, LE


def ngcf_layer_bwd(csr, E, LE, En, Gn, W1, W2, G, slope=0.01, dense_mode: int = _cabi.YR_DENSE_TC_FWD):
    """G (accumulated in place) += dLoss/dE; returns (dW1, dW2)."""
    lib = _cabi.load()
    d = E.shape[1]
    T = torch.empty_like(E)
    dW1, dW2 = torch.empty_like(W1), torch.empty_like(W2)
    nbytes = lib.yr_ngcf_layer_bwd_ws_bytes(d)
    ws = torch.empty(nbytes, device=E.device, dtype=torch.uint8)
    st = csr.bwd.struct(d)
    check(lib.yr_ngcf_layer_bwd(C.byref(st), d, dptr(E.contiguous(), F32), dptr(LE, F32), dptr(En, F32),
                                dptr(Gn.contiguous(), F32), dptr(W1.contiguous(), F32), dptr(W2.contiguous(), F32),
                                float(slope), dptr(G, F32), dptr(T), dptr(dW1), dptr(dW2), dptr(ws), nbytes, int(dense_mode),
                                stream_ptr(E.device)), "yr_ngcf_layer_bwd")
    return dW1, dW2


# The graph travels as an integer handle (custom ops take tensors and scalars only): data.graph.LaplacianCSR objects are
# registered by identity and live as long as the model that owns them.
import weakref

_CSR_REGISTRY = weakref.WeakValueDictionary()      # the owning model keeps the CSR alive; the registry never does


def _csr_handle(csr) -> int:
    h = id(csr)
    _CSR_REGISTRY[h] = csr
    return h


@custom_op("yelprec::ngcf_layer", mutates_args=(), device_types="cuda")
def _op_ngcf_layer(E: torch.Tensor, W1: torch.Tensor, W2: torch.Tensor, csr_handle: int,
                   slope: float, dense_mode: int) -> Tuple[torch.Tensor, torch.Tensor]:
    """NGCF.embedding_propagation (models/ngcf.py:60-72) -> yr_ngcf_layer_fwd. Returns (E_next, L E)."""
    Ed, W1d, W2d = E.detach().contiguous(), W1.detach().contiguous(), W2.detach().contiguous()
    return ngcf_layer_fwd(_CSR_REGISTRY[csr_handle], Ed, W1d, W2d, slope, dense_mode)


@_op_ngcf_layer.register_fake
def _(E, W1, W2, csr_handle, slope, dense_mode):
    return torch.empty_like(E), torch.empty_like(E)


@custom_op("yelprec::ngcf_layer_bwd", mutates_args=(), device_types="cuda")
def _op_ngcf_layer_bwd(E: torch.Tensor, LE: torch.Tensor, En: torch.Tensor, Gn: torch.Tensor, W1: torch.Tensor,
                       W2: torch.Tensor, csr_handle: int, slope: float,
                       dense_mode: int) -> Tuple[torch.Tensor, torch.Tensor, torch.Tensor]:
    E, W1, W2 = E.detach().contiguous(), W1.detach().contiguous(), W2.detach().contiguous()
    G = torch.zeros_like(E)
    dW1, dW2 = ngcf_layer_bwd(_CSR_REGISTRY[csr_handle], E, LE.contiguous(), En.contiguous(), Gn.contiguous(), W1, W2, G, slope,
                              dense_mode)
    return G, dW1, dW2


@_op_ngcf_layer_bwd.register_fake
def _(E, LE, En, Gn, W1, W2, csr_handle, slope, dense_mode):
    return torch.empty_like(E), torch.empty_like(W1), torch.empty_like(W2)


def _ngcf_layer_setup(ctx, inputs, output):
    E, W1, W2, csr_handle, slope, dense_mode = inputs
    En, LE = output
    ctx.save_for_backward(E, LE, En, W1, W2)
    ctx.csr_handle, ctx.slope, ctx.dense_mode = csr_handle, slope, dense_mode


def _ngcf_layer_backward(ctx, gEn, gLE):
    E, LE, En, W1, W2 = ctx.saved_tensors
    G, dW1, dW2 = _op_ngcf_layer_bwd(E, LE, En, gEn, W1, W2, ctx.csr_handle, ctx.slope, ctx.dense_mode)
    return G, dW1, dW2, None, None, None


_op_ngcf_layer.register_autograd(_ngcf_layer_backward, setup_context=_ngcf_layer_setup)


def ngcf_layer(E, W1, W2, csr, slope=0.01, dense_mode: int = _cabi.YR_DENSE_TC_FWD):
    if not E.is_cuda:
        raise YelprecError("NGCF.embedding_propagation: expected CUDA tensors (no CPU fallback)")
    return _op_ngcf_layer(E, W1, W2, _csr_handle(csr), float(slope), int(dense_mode))[0]


def dense_opt_step(p, g, m, v, opt: _cabi.YrOpt):
    lib = _cabi.load()
    check(lib.yr_dense_opt_step(dptr(p, F32), dptr(g.contiguous(), F32), dptr(m), dptr(v), p.numel(), C.byref(opt),
                                stream_ptr(p.device)), "yr_dense_opt_step")


def sample_negatives(uid: torch.Tensor, pos_ptr: torch.Tensor, pos_idx: torch.Tensor, num_users: int, num_items: int,
                     seed: int, offset: int = 0, max_blocks: int = 64, err: Optional[torch.Tensor] = None) -> torch.Tensor:
    """One negative per entry of `uid` (int64, device), uniform over the items outside the user's sorted positive list
    (CSR int32 pos_ptr / pos_idx) — MFDataset._negative_sampling (data/datasets/mf_dataset.py:18-22) on the device."""
    lib = _cabi.load()
    uid = uid.contiguous()
    neg = torch.empty_like(uid)
    if uid.numel() == 0:
        return neg
    own_err = err is None
    if own_err:
        err = torch.zeros(1, dtype=I32, device=uid.device)
    check(lib.yr_sample_negatives(dptr(uid, I64), uid.numel(), dptr(pos_ptr, I32), dptr(pos_idx, I32), int(num_users),
                                  int(num_items), int(seed) & (2 ** 64 - 1), int(offset) & (2 ** 64 - 1), int(max_blocks),
                                  dptr(neg, I64), dptr(err, I32), stream_ptr(uid.device)), "yr_sample_negatives")
    if own_err:
        code = int(err.item())
        if code == 1:
            raise IndexError("sample_negatives: index out of range in self")
        if code == 2:
            raise RuntimeError("sample_negatives: no item outside a user's positives")
    return neg


def device_ptr_array(tensors: Sequence[torch.Tensor]) -> torch.Tensor:
    """int64 device tensor holding the data pointers of `tensors` (a `float* const*` for the kernels)."""
    dev = tensors[0].device
    return torch.tensor([t.data_ptr() for t in tensors], dtype=I64).to(dev)


def ngcf_concat(E_layers: Sequence[torch.Tensor]) -> torch.Tensor:
    lib = _cabi.load()
    n, d = E_layers[0].shape
    L = len(E_layers) - 1
    ptrs = device_ptr_array([e.contiguous() for e in E_layers])
    out = torch.empty(n, (L + 1) * d, device=E_layers[0].device, dtype=F32)
    check(lib.yr_ngcf_concat(dptr(ptrs), L, n, d, dptr(out), stream_ptr(out.device)), "yr_ngcf_concat")
    return out


# ----------------------------------------------------------------------------------------------------
# evaluation
# ----------------------------------------------------------------------------------------------------
class DeviceEvalCSR:
    """EvalCSR (data/graph.py) uploaded once; reused across epochs."""

    def __init__(self, csr, device, K: int):
        from .data.graph import inv_log2_table
        t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(device)
        self.n_eval = csr.n_eval
        self.eval_uid = t(csr.eval_uid)
        self.mask_ptr, self.mask_idx = t(csr.mask_ptr), t(csr.mask_idx if csr.mask_idx.size else np.zeros(1, np.int32))
        self.act_ptr, self.act_idx = t(csr.act_ptr), t(csr.act_idx if csr.act_idx.size else np.zeros(1, np.int32))
        self.act_nuniq = t(csr.act_nuniq if csr.act_nuniq.size else np.zeros(1, np.int32))
        self.inv_log2 = t(inv_log2_table(K))
        self.K = K

    @classmethod
    def from_device(cls, eval_uid, mask_ptr, mask_idx, act_ptr, act_idx, act_nuniq, K: int) -> "DeviceEvalCSR":
        """Built from tensors that already live on the device (int64 uid, int32 CSR pieces; mask ids ascending per row,
        act ids in their original order, act_nuniq = |set(row)|)."""
        from .data.graph import inv_log2_table
        out = object.__new__(cls)
        dev = eval_uid.device
        pad = lambda t: t.contiguous() if t.numel() else torch.zeros(1, dtype=I32, device=dev)
        out.n_eval = int(eval_uid.numel())
        out.eval_uid = eval_uid.to(I64).contiguous()
        out.mask_ptr, out.mask_idx = mask_ptr.to(I32).contiguous(), pad(mask_idx.to(I32))
        out.act_ptr, out.act_idx = act_ptr.to(I32).contiguous(), pad(act_idx.to(I32))
        out.act_nuniq = pad(act_nuniq.to(I32))
        out.inv_log2 = torch.from_numpy(np.ascontiguousarray(inv_log2_table(K))).to(dev)
        out.K = K
        return out

    def slice(self, lo: int, hi: int) -> "DeviceEvalCSR":
        """Rows [lo, hi) — user sharding across GPUs (no communication until the metric sums)."""
        out = object.__new__(DeviceEvalCSR)
        out.n_eval = hi - lo
        out.eval_uid = self.eval_uid[lo:hi].contiguous()
        for name in ("mask", "act"):
            ptr = getattr(self, f"{name}_ptr")
            idx = getattr(self, f"{name}_idx")
            base, end = int(ptr[lo].item()), int(ptr[hi].item())
            setattr(out, f"{name}_ptr", (ptr[lo:hi + 1] - base).contiguous())
            sl = idx[base:end]
            setattr(out, f"{name}_idx", sl.contiguous() if sl.numel() else torch.zeros(1, dtype=I32, device=idx.device))
        nu = self.act_nuniq[lo:hi]
        out.act_nuniq = nu.contiguous() if nu.numel() else torch.zeros(1, dtype=I32, device=nu.device)
        out.inv_log2, out.K = self.inv_log2, self.K
        return out


def transpose_items(V: torch.Tensor) -> Tuple[torch.Tensor, int]:
    """[nI x d] -> ([pad32(d) x ldt], ldt) with ldt = nI rounded up to the 128-item tile."""
    lib = _cabi.load()
    V = V.detach().contiguous()
    nI, d = V.shape
    ldt = (nI + 127) // 128 * 128
    d_pad = (d + 31) // 32 * 32
    Vt = torch.empty(d_pad, ldt, device=V.device, dtype=F32)
    check(lib.yr_transpose_items(dptr(V, F32), nI, d, dptr(Vt), ldt, stream_ptr(V.device)), "yr_transpose_items")
    return Vt, ldt


_SM_COUNT = {}
_SLICE_STREAMS = {}


def _sm_count(dev) -> int:
    i = dev.index if dev.index is not None else torch.cuda.current_device()
    if i not in _SM_COUNT:
        _SM_COUNT[i] = torch.cuda.get_device_properties(i).multi_processor_count
    return _SM_COUNT[i]


def eval_item_slices(n_eval: int, nI: int, K: int, dev) -> int:
    """How many item slices a full-catalog evaluation of n_eval rows is cut into. The tensor-core kernel runs one CTA per SM
    over 128-row user tiles, each streaming the whole catalog: a row shard of 31 tiles (8 ranks at Yelp shape) leaves 117 of
    148 SMs idle. Cut into S item slices evaluated by S concurrent launches, S x tiles CTAs are busy and a tile's stream is S
    times shorter. YR_EVAL_SLICES overrides (1 = never slice)."""
    import os
    env = os.environ.get("YR_EVAL_SLICES")
    return slices_for(n_eval, nI, K, _sm_count(dev), int(env) if env else None)


def slices_for(n_eval: int, nI: int, K: int, sm_count: int, forced: int = None) -> int:
    """The rule behind eval_item_slices (host arithmetic only): as many slices as it takes for tiles x slices CTAs to fill the SMs,
    at most 8 and at most 64 // K (yr_topk_merge keeps S * K <= 64 candidates per row), each slice at least 2,048 items long."""
    tiles = max(1, (n_eval + 127) // 128)
    S = forced if forced is not None else sm_count // tiles
    S = max(1, min(S, 8, 64 // max(K, 1)))
    while S > 1 and -(-nI // S) < 2048:          # keep slices long enough for the running threshold to settle
        S -= 1
    return S


def _sliced_masks(ecsr: DeviceEvalCSR, S: int, per: int, nI: int):
    """Per item slice s: the mask CSR restricted to items [s * per, (s + 1) * per), ids re-based to the slice (ascending per
    row, like the original). Index plumbing with torch ops, once per (evaluation set, S); cached on the DeviceEvalCSR.
    Returns None when some row has fewer than K unmasked items inside a slice (the unsliced path handles such rows)."""
    cache = ecsr.__dict__.setdefault("_slice_cache", {})
    key = (S, per, nI)
    if key in cache:
        return cache[key]
    n, dev = ecsr.n_eval, ecsr.eval_uid.device
    ptr = ecsr.mask_ptr.to(I64)
    nnz = int(ptr[n].item())
    idx = ecsr.mask_idx[:nnz].to(I64)
    row = torch.repeat_interleave(torch.arange(n, device=dev), ptr[1:n + 1] - ptr[:n])
    sl = torch.div(idx, per, rounding_mode="floor")
    out, ok = [], True
    for s_ in range(S):
        sel = sl == s_
        cnt = torch.bincount(row[sel], minlength=n)
        size = min(per, nI - s_ * per)
        if n and int(cnt.max().item()) > size - ecsr.K:
            ok = False
            break
        p_s = torch.zeros(n + 1, device=dev, dtype=I64)
        p_s[1:] = torch.cumsum(cnt, 0)
        i_s = (idx[sel] - s_ * per).to(I32)
        out.append((p_s.to(I32).contiguous(), i_s.contiguous() if i_s.numel() else torch.zeros(1, dtype=I32, device=dev)))
    cache[key] = out if ok else None
    return cache[key]


def _eval_tc_call(lib, Uemb, Vemb, Vt, ldt, nI, d, ecsr, mask_ptr, mask_idx, topk, tsc, um, sums, ws, err, slice_, n_slices, xchg,
                  stream):
    n, K = ecsr.n_eval, ecsr.K
    check(lib.yr_eval_topk_metrics_tc_slice(dptr(Uemb, F32), Uemb.shape[0], Vemb.data_ptr(), Vt.data_ptr(), ldt, nI, d,
                                            dptr(ecsr.eval_uid, I64), n, dptr(mask_ptr, I32), dptr(mask_idx, I32),
                                            dptr(ecsr.act_ptr, I32), dptr(ecsr.act_idx, I32), dptr(ecsr.act_nuniq, I32),
                                            dptr(ecsr.inv_log2, F64), K, dptr(topk), dptr(tsc), dptr(um), dptr(sums),
                                            dptr(ws), ws.numel(), dptr(err), slice_, n_slices, dptr(xchg, F32), stream),
          "yr_eval_topk_metrics_tc_slice")


def _eval_tc_sliced(lib, Uemb, Vemb, Vt, ldt, ecsr, S: int):
    """S concurrent tensor-core evaluations on disjoint item slices, then yr_topk_merge + yr_topk_metrics: the same top-K
    lists (ids, order, exact scores) and metrics as the unsliced call."""
    dev = Uemb.device
    nI, d = Vemb.shape
    n, K = ecsr.n_eval, ecsr.K
    per = (-(-nI // S) + 127) // 128 * 128
    S = -(-nI // per)
    masks = _sliced_masks(ecsr, S, per, nI) if S > 1 else None
    if masks is None:
        return None
    # buffers, streams and events of the sliced call are kept with the evaluation set: the S launches are short, so the host
    # side (allocations, event creation) would otherwise show up between them
    wsb = lib.yr_eval_tc_ws_bytes(n)
    wkey = ("ws", S, per, K)
    cache = ecsr.__dict__.setdefault("_slice_cache", {})
    if wkey not in cache:
        cache[wkey] = dict(ids=torch.empty(S, n, K, device=dev, dtype=I64), scs=torch.empty(S, n, K, device=dev, dtype=F32),
                           um=torch.zeros(S, n, 4, device=dev, dtype=F64), sums=torch.zeros(S, 6, device=dev, dtype=F64),
                           errs=torch.zeros(S, device=dev, dtype=I32), wss=torch.empty(S, wsb, device=dev, dtype=torch.uint8),
                           xchg=torch.empty(S, max(n, 1), device=dev, dtype=F32),
                           off=torch.arange(S, device=dev, dtype=I64) * per,
                           ready=torch.cuda.Event(), done=[torch.cuda.Event() for _ in range(S)])
    c = cache[wkey]
    ids, scs, um_s, sums_s, errs, wss, xchg = c["ids"], c["scs"], c["um"], c["sums"], c["errs"], c["wss"], c["xchg"]
    xchg.fill_(float("-inf"))                                       # the slices' shared thresholds
    key = (dev.index, S)
    if key not in _SLICE_STREAMS:
        _SLICE_STREAMS[key] = [torch.cuda.Stream(device=dev) for _ in range(S)]
    cur = torch.cuda.current_stream(dev)
    ready = c["ready"]
    ready.record(cur)
    esz = Vemb.element_size()
    for s_, st in enumerate(_SLICE_STREAMS[key]):
        i0 = s_ * per
        n_s = min(per, nI - i0)
        st.wait_event(ready)
        mp, mi = masks[s_]
        # item slice = rows [i0, i0 + n_s) of V (row-major) and columns [i0, ...) of the transposed copy
        _eval_tc_call(lib, Uemb, _PtrView(Vemb.data_ptr() + i0 * d * esz), _PtrView(Vt.data_ptr() + i0 * esz), ldt, n_s, d, ecsr,
                      mp, mi, ids[s_], scs[s_], um_s[s_], sums_s[s_], wss[s_], errs[s_:s_ + 1], s_, S, xchg, st.cuda_stream)
        c["done"][s_].record(st)
    for ev in c["done"]:
        cur.wait_event(ev)
    off = c["off"]
    topk = torch.empty(max(n, 1), K, device=dev, dtype=I64)
    tsc = torch.empty(max(n, 1), K, device=dev, dtype=F32)
    check(lib.yr_topk_merge(dptr(ids, I64), dptr(scs, F32), S, n, K, dptr(off, I64), dptr(topk), dptr(tsc), stream_ptr(dev)),
          "yr_topk_merge")
    um, sums = topk_metrics(topk[:n], ecsr)
    err = errs.max().reshape(1)
    eval_topk_metrics.last_fallback_rows = wss[:, 4:8].contiguous().view(I32).sum().reshape(1)
    eval_topk_metrics.last_slices = S
    return topk[:n], tsc[:n], um, sums, err


class _PtrView:
    """A device address handed to the C ABI in place of a tensor (an item-table slice that starts inside a tensor)."""

    def __init__(self, ptr: int):
        self._ptr = ptr

    def data_ptr(self) -> int:
        return self._ptr


def eval_topk_metrics(Uemb: torch.Tensor, Vemb: torch.Tensor, ecsr: DeviceEvalCSR, Vt=None, mode: str = None,
                      slices: int = None):
    """Returns (topk [n_eval x K] int64, topk_score, user_metrics [n_eval x 4] f64, sums [6] f64, err) on device.

    mode 'tc'    : tensor-core filter + exact re-score (yr_eval_topk_metrics_tc) — bit-identical outputs;
    mode 'exact' : FP32-pipe kernel (yr_eval_topk_metrics);
    mode 'retrieval': top-K retrieval kernel (yr_recommend_topk, masked items score -3.40282e+38 as in the other modes)
                   + yr_topk_metrics — the same scores, lists and metrics;
    mode None    : env YR_EVAL_MODE, else 'tc' whenever the library supports (d, K), 'exact' otherwise.
    slices       : item slices for small row sets (tensor-core mode only; None = eval_item_slices()); identical outputs."""
    import os
    lib = _cabi.load()
    Uemb = Uemb.detach().contiguous()
    Vemb = Vemb.detach().contiguous()
    dev = Uemb.device
    nI, d = Vemb.shape
    mode = mode or os.environ.get("YR_EVAL_MODE") or "auto"
    if mode == "retrieval":
        eval_topk_metrics.last_slices = 1
        topk, tsc = recommend_topk(Uemb, Vemb, ecsr.eval_uid, ecsr.K, ecsr.mask_ptr, ecsr.mask_idx, seen_by_row=True,
                                   masked_score=EVAL_MASK_VALUE)
        um, sums = topk_metrics(topk, ecsr)
        return topk, tsc, um, sums, torch.zeros(1, device=dev, dtype=I32)
    use_tc = mode == "tc" or (mode == "auto" and lib.yr_eval_tc_supported(d, ecsr.K) != 0)
    eval_topk_metrics.last_slices = 1
    if use_tc and ecsr.n_eval > 0:
        S = int(slices) if slices is not None else eval_item_slices(ecsr.n_eval, nI, ecsr.K, dev)
        if S > 1:
            if Vt is None:
                Vt, ldt = transpose_items(Vemb)
            else:
                ldt = Vt.shape[1]
            res = _eval_tc_sliced(lib, Uemb, Vemb, Vt, ldt, ecsr, S)
            if res is not None:
                return res
    if use_tc:
        if Vt is None:
            Vt, ldt = transpose_items(Vemb)
        else:
            ldt = Vt.shape[1]
        n, K = ecsr.n_eval, ecsr.K
        topk = torch.empty(max(n, 1), K, device=dev, dtype=I64)
        tsc = torch.empty(max(n, 1), K, device=dev, dtype=F32)
        um = torch.zeros(max(n, 1), 4, device=dev, dtype=F64)
        sums = torch.zeros(6, device=dev, dtype=F64)
        err = torch.zeros(1, device=dev, dtype=I32)
        ws = torch.empty(lib.yr_eval_tc_ws_bytes(n), device=dev, dtype=torch.uint8)
        check(lib.yr_eval_topk_metrics_tc(dptr(Uemb, F32), Uemb.shape[0], dptr(Vemb, F32), dptr(Vt, F32), ldt, nI, d,
                                          dptr(ecsr.eval_uid, I64), n, dptr(ecsr.mask_ptr, I32), dptr(ecsr.mask_idx, I32),
                                          dptr(ecsr.act_ptr, I32), dptr(ecsr.act_idx, I32), dptr(ecsr.act_nuniq, I32),
                                          dptr(ecsr.inv_log2, F64), K, dptr(topk), dptr(tsc), dptr(um), dptr(sums),
                                          dptr(ws), ws.numel(), dptr(err), stream_ptr(dev)), "yr_eval_topk_metrics_tc")
        eval_topk_metrics.last_fallback_rows = ws[4:8].view(I32)      # device int32[1]: rows sent to the exact kernel
        return topk[:n], tsc[:n], um[:n], sums, err
    if d % 4 != 0:
        raise NotImplementedError(f"full-catalog evaluation: embedding width {d} is not a multiple of 4")
    if Vt is None:
        Vt, ldt = transpose_items(Vemb)
    else:
        ldt = Vt.shape[1]
    n, K = ecsr.n_eval, ecsr.K
    topk = torch.empty(max(n, 1), K, device=dev, dtype=I64)
    tsc = torch.empty(max(n, 1), K, device=dev, dtype=F32)
    um = torch.zeros(max(n, 1), 4, device=dev, dtype=F64)
    sums = torch.zeros(6, device=dev, dtype=F64)
    err = torch.zeros(1, device=dev, dtype=I32)
    ws = torch.empty(lib.yr_eval_ws_bytes(n, d, K), device=dev, dtype=torch.uint8)
    check(lib.yr_eval_topk_metrics(dptr(Uemb, F32), Uemb.shape[0], dptr(Vt, F32), ldt, nI, d, dptr(ecsr.eval_uid, I64), n,
                                   dptr(ecsr.mask_ptr, I32), dptr(ecsr.mask_idx, I32), dptr(ecsr.act_ptr, I32),
                                   dptr(ecsr.act_idx, I32), dptr(ecsr.act_nuniq, I32), dptr(ecsr.inv_log2, F64), K,
                                   dptr(topk), dptr(tsc), dptr(um), dptr(sums), dptr(ws), ws.numel(), dptr(err),
                                   stream_ptr(dev)), "yr_eval_topk_metrics")
    return topk[:n], tsc[:n], um[:n], sums, err


EVAL_MASK_VALUE = -3.40282e+38     # score of a masked (train) item in evaluation (trainers/mf_trainer.py:167)


def metrics_from_sums(sums, n_eval: int):
    """(precision, recall, map, ndcg) with the reference's divisors (metric.py:24,47,70,104 — quirk Q6)."""
    s = [float(x) for x in sums]
    if n_eval == 0:
        raise ZeroDivisionError("division by zero")        # what metric.py does on an empty eval set
    return (s[0] / n_eval, s[1] / s[4], s[2] / s[5], s[3] / s[4])


def topk_masked_row(pred: torch.Tensor, mask_items, K: int) -> torch.Tensor:
    lib = _cabi.load()
    pred = pred.detach().contiguous().to(F32)
    mask = torch.as_tensor(np.asarray(mask_items, dtype=np.int64).reshape(-1)).to(pred.device)
    out = torch.empty(K, device=pred.device, dtype=I64)
    check(lib.yr_topk_masked_row(dptr(pred), pred.numel(), dptr(mask) if mask.numel() else None, mask.numel(), K,
                                 dptr(out), stream_ptr(pred.device)), "yr_topk_masked_row")
    return out


def topk_metrics(predicted: torch.Tensor, ecsr: DeviceEvalCSR):
    lib = _cabi.load()
    predicted = predicted.contiguous()
    n = predicted.shape[0]
    um = torch.zeros(max(n, 1), 4, device=predicted.device, dtype=F64)
    sums = torch.zeros(6, device=predicted.device, dtype=F64)
    check(lib.yr_topk_metrics(dptr(predicted, I64), predicted.shape[1], n, dptr(ecsr.act_ptr, I32),
                              dptr(ecsr.act_idx, I32), dptr(ecsr.act_nuniq, I32), dptr(ecsr.inv_log2, F64), ecsr.K,
                              dptr(um), dptr(sums), stream_ptr(predicted.device)), "yr_topk_metrics")
    return um[:n], sums


# ----------------------------------------------------------------------------------------------------
# top-K retrieval
# ----------------------------------------------------------------------------------------------------
RECOMMEND_MAX_K = 1024
RECOMMEND_MAX_D = 1024
_RT_DTYPES = {F32: _cabi.YR_DTYPE_F32, torch.bfloat16: _cabi.YR_DTYPE_BF16}


def _item_bias(item_bias: Optional[torch.Tensor], nI: int, dev, what: str) -> Optional[torch.Tensor]:
    """item_bias as a contiguous fp32 [nI] tensor on `dev` (None passes through)."""
    if item_bias is None:
        return None
    if not torch.is_tensor(item_bias) or item_bias.dtype != F32 or item_bias.dim() != 1 or item_bias.numel() != nI:
        raise ValueError(f"{what}: item_bias must be a float32 tensor of shape [{nI}]")
    if item_bias.device != dev:
        raise ValueError(f"{what}: item_bias must live on the device of the embeddings ({dev}), got {item_bias.device}")
    return item_bias.detach().contiguous()


def _rt_tables(what: str, U, V, user_ids, K):
    """The checks of the embedding tables, k and user_ids every retrieval entry makes: (device, d, nU, nI, K, B)."""
    if not (torch.is_tensor(U) and torch.is_tensor(V) and torch.is_tensor(user_ids)):
        raise TypeError(f"{what}: U, V and user_ids must be tensors")
    if not (U.is_cuda and V.is_cuda and user_ids.is_cuda):
        raise YelprecError(f"{what}: U, V and user_ids must be CUDA tensors (the reference path is "
                           "retrieval.recommend_reference)")
    dev = U.device
    if V.device != dev or user_ids.device != dev:
        raise ValueError(f"{what}: tensors on different devices ({U.device}, {V.device}, {user_ids.device})")
    if U.dtype not in _RT_DTYPES or V.dtype != U.dtype:
        raise TypeError(f"{what}: U and V must both be float32 or both bfloat16, got {U.dtype} and {V.dtype}")
    if U.dim() != 2 or V.dim() != 2 or U.shape[1] != V.shape[1]:
        raise ValueError(f"{what}: U [nU x d] and V [nI x d] expected, got {tuple(U.shape)} and {tuple(V.shape)}")
    d = int(U.shape[1])
    if d % 8 != 0 or d > RECOMMEND_MAX_D:
        raise ValueError(f"{what}: embedding width {d} must be a multiple of 8 and at most {RECOMMEND_MAX_D}")
    nU, nI = int(U.shape[0]), int(V.shape[0])
    if nU == 0 or nI == 0 or nI >= 2 ** 31 - 1:
        raise ValueError(f"{what}: {nU} users x {nI} items is not a valid catalog")
    if isinstance(K, bool) or int(K) != K or not 1 <= int(K) <= RECOMMEND_MAX_K:
        raise ValueError(f"{what}: k must be an integer in [1, {RECOMMEND_MAX_K}], got {K}")
    if user_ids.dtype not in (I64, I32) or user_ids.dim() != 1:
        raise TypeError(f"{what}: user_ids must be a 1-D int64 or int32 tensor, got {user_ids.dtype} "
                        f"{tuple(user_ids.shape)}")
    return dev, d, nU, nI, int(K), int(user_ids.numel())


def _rt_seen_and_bias(what: str, seen_ptr, seen_idx, rows: int, item_bias, nI: int, dev):
    """The seen lists (int32 CSR over `rows` rows) and item_bias, checked and made contiguous: (ptr, idx, bias)."""
    if (seen_ptr is None) != (seen_idx is None):
        raise ValueError(f"{what}: seen_ptr and seen_idx go together")
    bias = _item_bias(item_bias, nI, dev, what)
    if seen_ptr is not None:
        if seen_ptr.dtype != I32 or seen_idx.dtype != I32 or seen_ptr.numel() != rows + 1:
            raise ValueError(f"{what}: seen lists must be int32 CSR with {rows + 1} offsets")
        if seen_ptr.device != dev or seen_idx.device != dev:
            raise ValueError(f"{what}: seen lists must live on the device of the embeddings")
        seen_ptr = seen_ptr.contiguous()
        seen_idx = seen_idx.contiguous() if seen_idx.numel() else torch.zeros(1, dtype=I32, device=dev)
    return seen_ptr, seen_idx, bias


def _rt_run(U, V, B: int, K: int, dev, ws_bytes, launch):
    """Allocates the outputs, the workspace (ws_bytes(lib) bytes) and the error word, and calls
    launch(lib, Uc, Vc, ids, scores, ws, nbytes, err): (ids, scores, error word), the error word 0 when B == 0."""
    lib = _cabi.load()
    Uc, Vc = U.detach().contiguous(), V.detach().contiguous()
    ids = torch.empty(B, K, device=dev, dtype=I64)
    scores = torch.empty(B, K, device=dev, dtype=F32)
    if B == 0:
        return ids, scores, 0
    err = torch.zeros(1, device=dev, dtype=I32)
    nbytes = ws_bytes(lib)
    ws = torch.empty(max(nbytes, 1), device=dev, dtype=torch.uint8)
    launch(lib, Uc, Vc, ids, scores, ws, nbytes, err)
    return ids, scores, int(err.item())


def recommend_topk(U: torch.Tensor, V: torch.Tensor, user_ids: torch.Tensor, K: int, seen_ptr: Optional[torch.Tensor] = None,
                   seen_idx: Optional[torch.Tensor] = None, seen_by_row: bool = False,
                   masked_score: float = float("-inf"),
                   item_bias: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """yr_recommend_topk_ex: (ids int64 [B x K], scores float32 [B x K]) of the K best items per user by (score desc, id
    asc), score = U[uid] . V[item] (+ item_bias[item]) in fp32 (fp32 or bf16 tables, fp32 bias). Seen items (CSR int32,
    ascending per row, rows = user ids, or batch rows with seen_by_row) score `masked_score`; -inf drops them. Short rows
    are padded with id -1 / score -inf."""
    what = "recommend_topk"
    dev, d, nU, nI, K, B = _rt_tables(what, U, V, user_ids, K)
    seen_ptr, seen_idx, bias = _rt_seen_and_bias(what, seen_ptr, seen_idx, B if seen_by_row else nU, item_bias, nI, dev)
    uid = user_ids.to(I64).contiguous()

    def launch(lib, Uc, Vc, ids, scores, ws, nbytes, err):
        check(lib.yr_recommend_topk_ex(Uc.data_ptr(), nU, Vc.data_ptr(), nI, d, _RT_DTYPES[U.dtype], dptr(uid, I64), B,
                                       dptr(seen_ptr), dptr(seen_idx), 1 if seen_by_row else 0, float(masked_score), K,
                                       dptr(ids), dptr(scores), dptr(ws), nbytes, dptr(err), stream_ptr(dev),
                                       dptr(bias)), "yr_recommend_topk_ex")

    ids, scores, e = _rt_run(U, V, B, K, dev, lambda lib: lib.yr_recommend_ws_bytes(B, nI, K), launch)
    if e != 0:
        raise IndexError(f"{what}: user id out of range [0, {nU})")
    return ids, scores


def recommend_subset_topk(U: torch.Tensor, V: torch.Tensor, user_ids: torch.Tensor, K: int, subset_ptr: torch.Tensor,
                          subset_idx: torch.Tensor, subset_ids: torch.Tensor, max_len: int,
                          seen_ptr: Optional[torch.Tensor] = None,
                          seen_idx: Optional[torch.Tensor] = None,
                          item_bias: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """yr_recommend_subset_topk_ex: recommend_topk with row b restricted to the items of subset subset_ids[b] (-1 = the whole
    catalog). Subsets: CSR int32 (subset_ptr [G + 1], subset_idx ascending per subset). max_len: the longest list a row
    streams (the longest subset, num_items if a row is -1); it sets only the number of item splits. Seen lists are indexed
    by user id. (ids int64 [B x K], scores float32 [B x K]), identical to recommend_topk with the items outside each row's
    subset excluded."""
    what = "recommend_subset_topk"
    if not (torch.is_tensor(subset_ptr) and torch.is_tensor(subset_idx) and torch.is_tensor(subset_ids)):
        raise TypeError(f"{what}: subset_ptr, subset_idx and subset_ids must be tensors")
    dev, d, nU, nI, K, B = _rt_tables(what, U, V, user_ids, K)
    if subset_ids.dtype not in (I64, I32) or subset_ids.dim() != 1:
        raise TypeError(f"{what}: subset_ids must be a 1-D int64 or int32 tensor, got {subset_ids.dtype} "
                        f"{tuple(subset_ids.shape)}")
    if subset_ids.numel() != B:
        raise ValueError(f"{what}: {subset_ids.numel()} subset ids for {B} users")
    if subset_ptr.dtype != I32 or subset_idx.dtype != I32 or subset_ptr.dim() != 1 or subset_ptr.numel() < 1:
        raise ValueError(f"{what}: subsets must be an int32 CSR (subset_ptr [G + 1], subset_idx)")
    if subset_ptr.device != dev or subset_idx.device != dev or subset_ids.device != dev:
        raise ValueError(f"{what}: subsets and subset ids must live on the device of the embeddings")
    G = int(subset_ptr.numel()) - 1
    if isinstance(max_len, bool) or int(max_len) != max_len or int(max_len) < 0:
        raise ValueError(f"{what}: max_len must be a non-negative integer, got {max_len}")
    seen_ptr, seen_idx, bias = _rt_seen_and_bias(what, seen_ptr, seen_idx, nU, item_bias, nI, dev)
    uid = user_ids.to(I64).contiguous()
    sid = subset_ids.to(I64).contiguous()
    sptr = subset_ptr.contiguous()
    sidx = subset_idx.contiguous() if subset_idx.numel() else torch.zeros(1, dtype=I32, device=dev)

    def launch(lib, Uc, Vc, ids, scores, ws, nbytes, err):
        check(lib.yr_recommend_subset_topk_ex(Uc.data_ptr(), nU, Vc.data_ptr(), nI, d, _RT_DTYPES[U.dtype],
                                              dptr(uid, I64), B, dptr(sptr, I32), dptr(sidx, I32), G, int(max_len),
                                              dptr(sid, I64), dptr(seen_ptr), dptr(seen_idx), K, dptr(ids), dptr(scores),
                                              dptr(ws), nbytes, dptr(err), stream_ptr(dev), dptr(bias)),
              "yr_recommend_subset_topk_ex")

    ids, scores, e = _rt_run(U, V, B, K, dev, lambda lib: lib.yr_recommend_subset_ws_bytes(B, G, int(max_len), K),
                             launch)
    if e & 1:
        raise IndexError(f"{what}: user id out of range [0, {nU})")
    if e & 2:
        raise IndexError(f"{what}: subset id out of range [-1, {G})")
    return ids, scores


def geo_grid_shape(cell_deg: float) -> Tuple[int, int]:
    """(lat bands, lon bands) of the item grid with cells of cell_deg degrees: ceil(180 / w), ceil(360 / w)."""
    import math
    return int(math.ceil(180.0 / cell_deg)), int(math.ceil(360.0 / cell_deg))


def recommend_geo_topk(U: torch.Tensor, V: torch.Tensor, user_ids: torch.Tensor, K: int, cell_keys: torch.Tensor,
                       cell_ptr: torch.Tensor, cell_items: torch.Tensor, item_xyz: torch.Tensor, cell_deg: float,
                       centre_xyz: torch.Tensor, threshold: torch.Tensor, seen_ptr: Optional[torch.Tensor] = None,
                       seen_idx: Optional[torch.Tensor] = None,
                       item_bias: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """yr_recommend_geo_topk: recommend_topk with row b restricted to the items i inside its radius,
    ((c_x * p_x) + (c_y * p_y)) + (c_z * p_z) >= threshold[b] in float64 with c = centre_xyz[b] and p = item_xyz[i] (unit
    vectors, float64 [B x 3] and [nI x 3]); threshold = cos(radius / Earth radius), -inf for every item. The item grid
    (cell_keys int64, cell_ptr int32, cell_items int32 and cells of cell_deg degrees) is retrieval.ItemLocations'; it
    bounds which items are read, never the result. Seen lists are indexed by user id. (ids int64 [B x K], scores float32
    [B x K]), identical to recommend_topk with the items outside each row's radius excluded. A user id out of range
    raises IndexError, a non-finite centre or a NaN / +inf threshold ValueError (both after the launch, from the error
    word: one scalar read per call)."""
    what = "recommend_geo_topk"
    if not all(torch.is_tensor(x) for x in (cell_keys, cell_ptr, cell_items, item_xyz, centre_xyz, threshold)):
        raise TypeError(f"{what}: the item grid, item_xyz, centre_xyz and threshold must be tensors")
    dev, d, nU, nI, K, B = _rt_tables(what, U, V, user_ids, K)
    if centre_xyz.dtype != F64 or threshold.dtype != F64:
        raise TypeError(f"{what}: centre_xyz and threshold must be float64, got {centre_xyz.dtype} and "
                        f"{threshold.dtype}")
    if tuple(centre_xyz.shape) != (B, 3) or tuple(threshold.shape) != (B,):
        raise ValueError(f"{what}: centre_xyz [{B} x 3] and threshold [{B}] expected, got "
                         f"{tuple(centre_xyz.shape)} and {tuple(threshold.shape)}")
    if item_xyz.dtype != F64 or tuple(item_xyz.shape) != (nI, 3):
        raise ValueError(f"{what}: item_xyz must be float64 [{nI} x 3]")
    if cell_keys.dtype != I64 or cell_ptr.dtype != I32 or cell_items.dtype != I32 or cell_keys.dim() != 1 or \
            cell_ptr.numel() != cell_keys.numel() + 1 or cell_items.numel() != nI:
        raise ValueError(f"{what}: the item grid must be cell_keys int64 [C], cell_ptr int32 [C + 1] and "
                         f"cell_items int32 [{nI}]")
    if any(x.device != dev for x in (cell_keys, cell_ptr, cell_items, item_xyz, centre_xyz, threshold)):
        raise ValueError(f"{what}: the item grid, item_xyz, centre_xyz and threshold must live on the device "
                         "of the embeddings")
    cell_deg = float(cell_deg)
    if not 0.0 < cell_deg <= 360.0:
        raise ValueError(f"{what}: cell_deg must be in (0, 360], got {cell_deg}")
    nlat, nlon = geo_grid_shape(cell_deg)
    seen_ptr, seen_idx, bias = _rt_seen_and_bias(what, seen_ptr, seen_idx, nU, item_bias, nI, dev)
    uid = user_ids.to(I64).contiguous()
    keys = cell_keys.contiguous() if cell_keys.numel() else torch.zeros(1, dtype=I64, device=dev)
    cptr, citems, P = cell_ptr.contiguous(), cell_items.contiguous(), item_xyz.contiguous()
    c, t = centre_xyz.contiguous(), threshold.contiguous()

    def launch(lib, Uc, Vc, ids, scores, ws, nbytes, err):
        check(lib.yr_recommend_geo_topk(Uc.data_ptr(), nU, Vc.data_ptr(), nI, d, _RT_DTYPES[U.dtype], dptr(uid, I64), B,
                                        dptr(keys, I64), dptr(cptr, I32), int(cell_keys.numel()), dptr(citems, I32),
                                        dptr(P, F64), cell_deg, nlat, nlon, dptr(c, F64), dptr(t, F64), dptr(seen_ptr),
                                        dptr(seen_idx), K, dptr(ids), dptr(scores), dptr(ws), nbytes, dptr(err),
                                        stream_ptr(dev), dptr(bias)), "yr_recommend_geo_topk")

    ids, scores, e = _rt_run(U, V, B, K, dev, lambda lib: lib.yr_recommend_geo_ws_bytes(B, nI, K), launch)
    if e & 1:
        raise IndexError(f"{what}: user id out of range [0, {nU})")
    if e & 2:
        raise ValueError(f"{what}: a centre is not finite or a threshold is NaN or +inf")
    return ids, scores


RECOMMEND_MMR_MAX_POOL = 1024


def mmr_weights(lam) -> Tuple[float, float]:
    """(a, c) of a diversity re-ranking with trade-off lam in [0, 1]: a = fp32(lam), c = fp32(1 - a) computed in fp32.
    The one place both weights are made, for the kernel and the reference alike."""
    if isinstance(lam, bool) or not isinstance(lam, (int, float, np.floating, np.integer)) or not 0.0 <= float(lam) <= 1.0:
        raise ValueError(f"recommend_mmr: lam must be a number in [0, 1], got {lam}")
    a = np.float32(lam)
    return float(a), float(np.float32(1.0) - a)


def mmr_sizes(what: str, K, N: int) -> int:
    """K checked against a pool of N (1 <= K <= N <= RECOMMEND_MMR_MAX_POOL)."""
    if not 1 <= N <= RECOMMEND_MMR_MAX_POOL:
        raise ValueError(f"{what}: the pool must hold 1 to {RECOMMEND_MMR_MAX_POOL} entries a row, got {N}")
    if isinstance(K, bool) or int(K) != K or not 1 <= int(K) <= N:
        raise ValueError(f"{what}: k must be an integer in [1, {N}] (the pool size), got {K}")
    return int(K)


def recommend_mmr(V: torch.Tensor, pool_ids: torch.Tensor, pool_scores: torch.Tensor, K: int,
                  lam: float) -> Tuple[torch.Tensor, torch.Tensor]:
    """yr_recommend_mmr: diversity re-ranking (Maximal Marginal Relevance) of each row's pool (ids int64 [B x N], -1 =
    empty; scores float32 [B x N], e.g. recommend_topk's output with K = N). Step t picks the unpicked entry with the
    largest lam * score - (1 - lam) * (its largest cosine similarity in V to the entries already picked), ties to the
    earlier entry. (ids int64 [B x K], scores float32 [B x K]) in pick order, the scores the pool's; rows that run out of
    entries are padded with -1 / -inf. V: the item table [nI x d] (fp32 or bf16) the similarity is measured in. A pool id
    outside [-1, nI) raises IndexError (after the launch, from the error word)."""
    what = "recommend_mmr"
    if not (torch.is_tensor(V) and torch.is_tensor(pool_ids) and torch.is_tensor(pool_scores)):
        raise TypeError(f"{what}: V, pool_ids and pool_scores must be tensors")
    if not (V.is_cuda and pool_ids.is_cuda and pool_scores.is_cuda):
        raise YelprecError(f"{what}: V, pool_ids and pool_scores must be CUDA tensors (the reference path is "
                           "retrieval.mmr_reference)")
    dev = V.device
    if pool_ids.device != dev or pool_scores.device != dev:
        raise ValueError(f"{what}: tensors on different devices ({V.device}, {pool_ids.device}, {pool_scores.device})")
    if V.dtype not in _RT_DTYPES or V.dim() != 2:
        raise TypeError(f"{what}: V must be a float32 or bfloat16 [nI x d] table, got {V.dtype} {tuple(V.shape)}")
    nI, d = int(V.shape[0]), int(V.shape[1])
    if d % 8 != 0 or d > RECOMMEND_MAX_D:
        raise ValueError(f"{what}: embedding width {d} must be a multiple of 8 and at most {RECOMMEND_MAX_D}")
    if nI == 0 or nI >= 2 ** 31 - 1:
        raise ValueError(f"{what}: {nI} items is not a valid catalog")
    if pool_ids.dtype != I64 or pool_scores.dtype != F32 or pool_ids.dim() != 2 or \
            pool_scores.shape != pool_ids.shape:
        raise TypeError(f"{what}: pool_ids int64 [B x N] and pool_scores float32 [B x N] expected, got "
                        f"{pool_ids.dtype} {tuple(pool_ids.shape)} and {pool_scores.dtype} {tuple(pool_scores.shape)}")
    B, N = int(pool_ids.shape[0]), int(pool_ids.shape[1])
    K = mmr_sizes(what, K, N)
    a, c = mmr_weights(lam)
    ids = torch.empty(B, K, device=dev, dtype=I64)
    scores = torch.empty(B, K, device=dev, dtype=F32)
    if B == 0:
        return ids, scores
    lib = _cabi.load()
    Vc, pid, psc = V.detach().contiguous(), pool_ids.contiguous(), pool_scores.contiguous()
    err = torch.zeros(1, device=dev, dtype=I32)
    check(lib.yr_recommend_mmr(Vc.data_ptr(), nI, d, _RT_DTYPES[V.dtype], dptr(pid, I64), dptr(psc, F32), B, N, K, a, c,
                               dptr(ids), dptr(scores), dptr(err), stream_ptr(dev)), "yr_recommend_mmr")
    if int(err.item()) != 0:
        raise IndexError(f"{what}: pool id out of range [-1, {nI})")
    return ids, scores


RECOMMEND_GROUP_MAX_MEMBERS = _cabi.YR_GROUP_MAX_MEMBERS
_GROUP_AGGS = {"min": _cabi.YR_GROUP_MIN, "mean": _cabi.YR_GROUP_MEAN}


def group_agg(agg) -> int:
    """The C ABI code of a group aggregation: "min" (least misery) or "mean"."""
    if not isinstance(agg, str) or agg not in _GROUP_AGGS:
        raise ValueError(f"recommend_group: agg must be 'min' or 'mean', got {agg!r}")
    return _GROUP_AGGS[agg]


def recommend_group_topk(U: torch.Tensor, V: torch.Tensor, group_ptr: torch.Tensor, members: torch.Tensor, K: int,
                         agg: str, seen_ptr: Optional[torch.Tensor] = None, seen_idx: Optional[torch.Tensor] = None,
                         subset_ptr: Optional[torch.Tensor] = None, subset_idx: Optional[torch.Tensor] = None,
                         subset_ids: Optional[torch.Tensor] = None, max_len: Optional[int] = None,
                         item_bias: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """yr_recommend_group_topk: (ids int64 [G x K], scores float32 [G x K]) of the K best items per group of users, group
    g = members[group_ptr[g] .. group_ptr[g + 1]) (rows of U, 1 to RECOMMEND_GROUP_MAX_MEMBERS, ascending), by the
    aggregate of the members' scores U[u] . V[i] (+ item_bias[i]): agg = "min" (least misery) or "mean" (summed in member
    order, then divided by the member count). Items in any member's seen list (CSR int32 indexed by the row of U) are
    never returned. subset_ids (int64 [G], -1 = whole catalog; None = every group ranks the whole catalog) restricts
    group g to subset subset_ids[g] of the subset CSR, as recommend_subset_topk; max_len as there (None: num_items).
    A member out of range raises IndexError, a subset id out of range IndexError and a group size outside
    [1, RECOMMEND_GROUP_MAX_MEMBERS] ValueError, all after the launch, from the error word (one scalar read per call)."""
    what = "recommend_group_topk"
    if not (torch.is_tensor(group_ptr) and torch.is_tensor(members)):
        raise TypeError(f"{what}: group_ptr and members must be tensors")
    dev, d, nU, nI, K, M = _rt_tables(what, U, V, members, K)
    code = group_agg(agg)
    if group_ptr.dtype != I32 or group_ptr.dim() != 1 or group_ptr.numel() < 1:
        raise ValueError(f"{what}: group_ptr must be int32 [G + 1]")
    if members.dtype != I64 or group_ptr.device != dev:
        raise ValueError(f"{what}: members must be int64 and group_ptr on the device of the embeddings")
    G = int(group_ptr.numel()) - 1
    if (subset_ids is None) != (subset_ptr is None) or (subset_ptr is None) != (subset_idx is None):
        raise ValueError(f"{what}: subset_ptr, subset_idx and subset_ids go together")
    NS, sptr, sidx, sid = 0, None, None, None
    if subset_ids is not None:
        if not (torch.is_tensor(subset_ptr) and torch.is_tensor(subset_idx) and torch.is_tensor(subset_ids)):
            raise TypeError(f"{what}: subset_ptr, subset_idx and subset_ids must be tensors")
        if subset_ids.dtype not in (I64, I32) or subset_ids.dim() != 1 or subset_ids.numel() != G:
            raise ValueError(f"{what}: subset_ids must be a 1-D int64 or int32 tensor of {G} ids, got "
                             f"{subset_ids.dtype} {tuple(subset_ids.shape)}")
        if subset_ptr.dtype != I32 or subset_idx.dtype != I32 or subset_ptr.dim() != 1 or subset_ptr.numel() < 1:
            raise ValueError(f"{what}: subsets must be an int32 CSR (subset_ptr [G + 1], subset_idx)")
        if subset_ptr.device != dev or subset_idx.device != dev or subset_ids.device != dev:
            raise ValueError(f"{what}: subsets and subset ids must live on the device of the embeddings")
        NS = int(subset_ptr.numel()) - 1
        sid, sptr = subset_ids.to(I64).contiguous(), subset_ptr.contiguous()
        sidx = subset_idx.contiguous() if subset_idx.numel() else torch.zeros(1, dtype=I32, device=dev)
    max_len = nI if max_len is None or subset_ids is None else max_len
    if isinstance(max_len, bool) or int(max_len) != max_len or int(max_len) < 0:
        raise ValueError(f"{what}: max_len must be a non-negative integer, got {max_len}")
    seen_ptr, seen_idx, bias = _rt_seen_and_bias(what, seen_ptr, seen_idx, nU, item_bias, nI, dev)
    gptr, mem = group_ptr.contiguous(), members.contiguous()
    if M == 0:
        mem = torch.zeros(1, dtype=I64, device=dev)

    def launch(lib, Uc, Vc, ids, scores, ws, nbytes, err):
        check(lib.yr_recommend_group_topk(Uc.data_ptr(), nU, Vc.data_ptr(), nI, d, _RT_DTYPES[U.dtype], dptr(gptr, I32),
                                          G, dptr(mem, I64), M, code, dptr(sptr), dptr(sidx), NS, int(max_len),
                                          dptr(sid), dptr(seen_ptr), dptr(seen_idx), K, dptr(ids), dptr(scores),
                                          dptr(ws), nbytes, dptr(err), stream_ptr(dev), dptr(bias)),
              "yr_recommend_group_topk")

    ids, scores, e = _rt_run(U, V, G, K, dev, lambda lib: lib.yr_recommend_group_ws_bytes(G, NS, int(max_len), K),
                             launch)
    if e & 1:
        raise IndexError(f"{what}: member id out of range [0, {nU})")
    if e & 2:
        raise IndexError(f"{what}: subset id out of range [-1, {NS})")
    if e & 4:
        raise ValueError(f"{what}: a group must have 1 to {RECOMMEND_GROUP_MAX_MEMBERS} members")
    return ids, scores
