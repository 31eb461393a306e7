"""Drop-in for the reference's loss.py:19-27 (BPRLoss) on the sm_100a kernels (yr_bpr_loss_fwd/_bwd)."""
import torch.nn as nn

from . import ops


class BPRLoss(nn.Module):
    def __init__(self):
        super().__init__()

    def forward(self, positive_preds, negative_preds):
        return ops.bpr_loss(positive_preds, negative_preds)


class NSBCELoss(nn.Module):
    """Drop-in for the reference's loss.py:7-16: BCE (mean) over the positions where target + negative_mask != 0,
    on dense tensors (yr_nsbce_loss). Inference-style (no autograd): the fused CDAE trainer computes the same loss at the
    compacted positions without ever building the dense prediction, and its gradient the way torch's autograd takes it
    through sigmoid and binary_cross_entropy, (p - t) / max((1 - p) p, 1e-12) * (1 - p) p, so a saturated p gives
    torch's gradient rather than p - t."""

    def __init__(self, weight=None, size_average=None, reduce=None, reduction: str = "mean") -> None:
        super().__init__()
        if weight is not None or reduction != "mean":
            raise NotImplementedError("NSBCELoss on the B200 path supports the reference's defaults (no weight, mean)")

    def forward(self, input, target, negative_mask):
        import torch
        from . import _cabi
        lib = _cabi.load()
        if not input.is_cuda:
            raise _cabi.YelprecError("NSBCELoss: expected CUDA tensors (no CPU fallback)")
        inp, tgt, neg = (t.detach().contiguous().float() for t in (input, target, negative_mask))
        out = torch.empty((), device=inp.device, dtype=torch.float32)
        ws = torch.empty(64, device=inp.device, dtype=torch.uint8)
        _cabi.check(lib.yr_nsbce_loss(_cabi.dptr(inp), _cabi.dptr(tgt), _cabi.dptr(neg), inp.numel(), _cabi.dptr(out),
                                      _cabi.dptr(ws), ws.numel(), _cabi.stream_ptr(inp.device)), "yr_nsbce_loss")
        return out
