"""Drop-in for the reference's models/cdae.py:7-52 on the sm_100a kernels (BASELINE config 4).

Same constructor `(cfg, num_items, num_users)` (items first, as the reference has it), same parameters / state_dict
keys (`hidden_layer.{weight,bias}`, `user_nodes.weight`, `output_layer.{weight,bias}`), same init. `forward(user_id, x)`
returns the dense [B x num_items] prediction like the reference (yr_cdae_hidden + yr_cdae_output); it is an inference
path (no autograd graph) — training goes through trainers/cdae_trainer.py, which never materialises the dense output.

Dropout (models/cdae.py:43-48, quirk Q16: `if self.train:` is always true, the layer itself obeys .train()/.eval()):
in training mode a keep-multiplier tensor (0 or 1/(1-p)) is drawn with torch's generator on the device, or supplied by
the caller through `keep=` so that a run can be replayed against the CPU reference with the same mask.
"""
import ctypes as C

import torch
import torch.nn as nn

from .. import _cabi
from .base_model import BaseModel

F32, I64, I32 = torch.float32, torch.int64, torch.int32


class CDAE(BaseModel):
    def __init__(self, cfg, num_items, num_users):
        super().__init__()
        self.num_items = num_items
        self.num_users = num_users
        self.hidden_size = cfg.hidden_size
        self.device = cfg.device
        self.corruption_level = cfg.corruption_level
        self.dropout_layer = nn.Dropout(p=self.corruption_level)
        self.hidden_layer = nn.Linear(self.num_items, self.hidden_size, bias=True, dtype=torch.float32)
        self.user_nodes = nn.Embedding(self.num_users, self.hidden_size, dtype=torch.float32)
        self.output_layer = nn.Linear(self.hidden_size, self.num_items, bias=True, dtype=torch.float32)
        if cfg.hidden_activation not in ("sigmoid", "identity"):
            raise _cabi.YelprecError(f"hidden_activation {cfg.hidden_activation!r}: the reference knows 'sigmoid' and 'identity'")
        if cfg.output_activation != "sigmoid":
            # NSBCELoss is a BCE on the output (loss.py:12-16): torch rejects anything that is not a probability
            raise _cabi.YelprecError("the B200 CDAE kernels keep the reference's sigmoid output activation")
        if cfg.hidden_size not in (32, 64, 128, 256, 512, 1024):
            raise _cabi.YelprecError(f"hidden_size {cfg.hidden_size}: the CDAE kernels take 32, 64, 128, 256, 512, 1024 "
                                     "(the values of the reference's cdae_sweep_config.yaml)")
        self.hidden_act = 0 if cfg.hidden_activation == "sigmoid" else 1          # enum yr_activation
        self.hidden_activation = self._activation_module(cfg.hidden_activation)
        self.output_activation = self._activation_module(cfg.output_activation)
        self._init_weights()
        self._ws = None

    def _init_weights(self):
        for child in self.children():
            if isinstance(child, nn.Linear):
                nn.init.xavier_uniform_(child.weight)
                nn.init.uniform_(child.bias)
            elif isinstance(child, nn.Embedding):
                nn.init.uniform_(child.weight)

    # ------------------------------------------------------------------------------------------
    def tensors(self) -> _cabi.YrCdaeTensors:
        p = _cabi.dptr
        return _cabi.YrCdaeTensors(p(self.hidden_layer.weight.data, F32), p(self.hidden_layer.bias.data, F32),
                                   p(self.user_nodes.weight.data, F32), p(self.output_layer.weight.data, F32),
                                   p(self.output_layer.bias.data, F32))

    def workspace(self, B: int) -> torch.Tensor:
        lib = _cabi.load()
        need = lib.yr_cdae_ws_bytes(B, self.num_items)
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, device=self.hidden_layer.weight.device, dtype=torch.uint8)
        return self._ws

    def draw_keep(self, x: torch.Tensor) -> torch.Tensor:
        """nn.Dropout's multiplier for x: Bernoulli(1-p) / (1-p)."""
        p = float(self.corruption_level)
        if p <= 0.0:
            return torch.ones_like(x)
        return (torch.rand_like(x) >= p).to(x.dtype) / (1.0 - p)

    def hidden(self, user_id, x, keep=None, ldz=None):
        """[B x ldz] hidden activations, columns h.. = 1, 0, 0, ... (so [z|1].[Wo|bo]^T is the output logit)."""
        lib = _cabi.load()
        dev = self.hidden_layer.weight.device
        user_id = user_id.to(device=dev, dtype=I64).contiguous()
        x = x.to(device=dev, dtype=F32).contiguous()
        B = x.shape[0]
        ldz = ldz or self.hidden_size
        z = torch.empty(B, ldz, device=dev, dtype=F32)
        err = torch.zeros(1, device=dev, dtype=I32)
        ws = self.workspace(B)
        st = self.tensors()
        _cabi.check(lib.yr_cdae_hidden_ex(C.byref(st), self.num_users, self.num_items, self.hidden_size, self.hidden_act,
                                       _cabi.dptr(user_id), _cabi.dptr(x), _cabi.dptr(keep) if keep is not None else None,
                                       B, _cabi.dptr(z), ldz, _cabi.dptr(ws), ws.numel(), _cabi.dptr(err),
                                       _cabi.stream_ptr(dev)), "yr_cdae_hidden_ex")
        if int(err.item()):
            raise IndexError("CDAE.forward: index out of range in self")
        return z

    def hidden_from_lists(self, user_id, ptr, idx) -> torch.Tensor:
        """[B x h] hidden activations of the evaluation-mode model (no dropout) from interaction lists instead of a dense
        multi-hot: ptr int32 [num_users + 1] / idx int32 is a CSR indexed by user id with ascending unique item ids per row
        (retrieval.SeenItems). Equal, bit for bit, to hidden(user_id, x)[:, :h] with x the multi-hot of the same lists;
        nothing of size B x num_items is allocated."""
        lib = _cabi.load()
        dev = self.hidden_layer.weight.device
        user_id = user_id.to(device=dev, dtype=I64).reshape(-1).contiguous()
        if ptr.dtype != I32 or idx.dtype != I32 or ptr.numel() != self.num_users + 1:
            raise ValueError(f"CDAE.hidden_from_lists: lists must be an int32 CSR with {self.num_users + 1} offsets")
        if ptr.device != dev or idx.device != dev:
            raise ValueError(f"CDAE.hidden_from_lists: lists must live on the model's device ({dev})")
        ptr = ptr.contiguous()
        idx = idx.contiguous() if idx.numel() else torch.zeros(1, device=dev, dtype=I32)
        B = user_id.numel()
        z = torch.empty(B, self.hidden_size, device=dev, dtype=F32)
        err = torch.zeros(1, device=dev, dtype=I32)
        st = self.tensors()
        _cabi.check(lib.yr_cdae_encode(C.byref(st), self.num_users, self.num_items, self.hidden_size, self.hidden_act,
                                       _cabi.dptr(user_id), B, _cabi.dptr(ptr), _cabi.dptr(idx), _cabi.dptr(z),
                                       self.hidden_size, _cabi.dptr(err), _cabi.stream_ptr(dev)), "yr_cdae_encode")
        e = int(err.item())
        if e & 1:
            raise IndexError(f"CDAE.hidden_from_lists: user id out of range [0, {self.num_users})")
        if e & 2:
            raise IndexError(f"CDAE.hidden_from_lists: item id out of range [0, {self.num_items}) "
                             "(or malformed list offsets)")
        return z

    def forward(self, user_id, x, keep=None):
        lib = _cabi.load()
        x = x.to(device=self.hidden_layer.weight.device, dtype=F32).contiguous()
        if keep is None and self.training:
            keep = self.draw_keep(x)
        z = self.hidden(user_id, x, keep)
        pred = torch.empty(x.shape[0], self.num_items, device=z.device, dtype=F32)
        st = self.tensors()
        _cabi.check(lib.yr_cdae_output(C.byref(st), self.num_items, self.hidden_size, _cabi.dptr(z), z.shape[1],
                                       x.shape[0], _cabi.dptr(pred), _cabi.stream_ptr(z.device)), "yr_cdae_output")
        return pred
