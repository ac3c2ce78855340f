"""In-batch sampled-softmax (InfoNCE) loss over a batch's positives and negatives, as one fused tensor-core call
(``ngcf_softmax_loss``): the alternative to ``BPR`` that scores each row against every positive and negative row of
the batch (2B - 1 negatives instead of 1) at no extra propagation cost."""
from __future__ import annotations

import ctypes as C

import torch
import torch.nn as nn

from . import _lib

MAX_BATCH = 4096
MAX_DIM = 1152          # the model's largest d0 + sum(d_k): nine blocks of 128


class _SoftmaxFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, u, p, n, pos_ids, neg_ids, weight_decay, batch_size, temperature):
        lib = _lib.load()
        B, D = u.shape
        has_n = n.numel() > 0
        ws_bytes = C.c_size_t()
        _lib.check(lib.ngcf_softmax_loss_workspace(B, 2 * B if has_n else B, D, C.byref(ws_bytes)),
                   "softmax_loss_workspace")
        ws = torch.empty(ws_bytes.value, dtype=torch.uint8, device=u.device)
        loss = torch.empty((), dtype=torch.float32, device=u.device)
        if any(ctx.needs_input_grad[:3]):
            gu, gp = torch.empty_like(u), torch.empty_like(p)
            gn = torch.empty_like(n) if has_n else None
        else:
            gu = gp = gn = None
        _lib.check(lib.ngcf_softmax_loss(u.data_ptr(), p.data_ptr(), n.data_ptr() if has_n else None, B, D,
                                         _lib.ptr(pos_ids), _lib.ptr(neg_ids), float(temperature),
                                         float(weight_decay), float(batch_size), loss.data_ptr(), _lib.ptr(gu),
                                         _lib.ptr(gp), _lib.ptr(gn), ws.data_ptr(), ws_bytes.value,
                                         _lib.current_stream()), "softmax_loss")
        ctx.grads = (gu, gp, gn)
        return loss

    @staticmethod
    def backward(ctx, gloss):
        gu, gp, gn = ctx.grads
        return (gu * gloss, gp * gloss, None if gn is None else gn * gloss, None, None, None, None, None)


class SoftmaxLoss(nn.Module):
    """``SoftmaxLoss(weight_decay, batch_size, temperature)(u, p, n, pos_ids=None, neg_ids=None)``.

    Row i of ``u`` is scored against every column c = (p rows, then n rows; ``n`` may be empty): s_ij = u_i.c_j / tau,
    and the loss is ``(1/batch_size) sum_i [logsumexp_j s_ij - s_ii + weight_decay (|u_i|^2 + |p_i|^2 + |n_i|^2)]``,
    the divisor the constructor's ``batch_size`` as in ``BPR``.  With the batch's item ids (``pos_ids``, and
    ``neg_ids`` when ``n`` is given), a column holding row i's own positive item elsewhere in the batch is not a
    negative for row i: it is left out of the sum.  ``GraphedStep`` and ``Experiment.train`` pass the ids."""

    def __init__(self, weight_decay, batch_size, temperature: float = 0.2):
        super().__init__()
        if not temperature > 0:
            raise ValueError(f"SoftmaxLoss: temperature {temperature} is not > 0")
        if not weight_decay >= 0:
            raise ValueError(f"SoftmaxLoss: weight_decay {weight_decay} is not >= 0")
        if not batch_size > 0:
            raise ValueError(f"SoftmaxLoss: batch_size {batch_size} is not > 0")
        self.weight_decay = weight_decay
        self.batch_size = batch_size
        self.temperature = temperature

    @_lib.on_device
    def forward(self, u, p, n, pos_ids=None, neg_ids=None):
        for name, t in (("u", u), ("p", p), ("n", n)):
            if name == "n" and t.numel() == 0:              # no negatives (NGCF returns a host torch.empty(0))
                continue
            if t.device.type != "cuda":
                raise RuntimeError("SoftmaxLoss (B200) runs on CUDA tensors only; there is no CPU fallback")
            if t.dtype != torch.float32:
                raise TypeError(f"SoftmaxLoss: {name} is {t.dtype}, not torch.float32")
        if u.dim() != 2 or p.shape != u.shape:
            raise ValueError(f"SoftmaxLoss: u {tuple(u.shape)} and p {tuple(p.shape)} must be the same [B, D]")
        B, D = u.shape
        has_n = n.numel() > 0
        if has_n and n.shape != u.shape:
            raise ValueError(f"SoftmaxLoss: n {tuple(n.shape)} must be empty or [B, D] = {tuple(u.shape)}")
        if not 1 <= B <= MAX_BATCH or not 1 <= D <= MAX_DIM:
            raise ValueError(f"SoftmaxLoss: [B, D] = [{B}, {D}] outside [1, {MAX_BATCH}] x [1, {MAX_DIM}]")
        if any(t.device != u.device for t in (p, n) if t.numel()):
            raise RuntimeError("SoftmaxLoss: u, p and n are on different devices")
        if neg_ids is not None and pos_ids is None:
            raise ValueError("SoftmaxLoss: neg_ids without pos_ids")
        if neg_ids is not None and not has_n:
            raise ValueError("SoftmaxLoss: neg_ids without negatives")
        if pos_ids is not None and has_n and neg_ids is None:
            raise ValueError("SoftmaxLoss: with negatives, pass neg_ids along with pos_ids")
        for name, t in (("pos_ids", pos_ids), ("neg_ids", neg_ids)):
            if t is None:
                continue
            if t.dtype != torch.int64 or t.shape != (B,):
                raise ValueError(f"SoftmaxLoss: {name} must be int64 [{B}], got {t.dtype} {tuple(t.shape)}")
            if t.device != u.device:
                raise RuntimeError(f"SoftmaxLoss: {name} is on {t.device}, the rows on {u.device}")
        ids = [None if t is None else t.contiguous() for t in (pos_ids, neg_ids)]
        return _SoftmaxFn.apply(u.contiguous(), p.contiguous(), n.contiguous() if has_n else n, ids[0], ids[1],
                                self.weight_decay, self.batch_size, self.temperature)
