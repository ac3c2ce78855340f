"""Fused scoring + top-k: the ``torch.mm(u, all_i_emb.T)`` + ``torch.topk`` pair of demo.py:234-235 and
experiment.py:93,104,109 without materialising the score matrix.

Full-ranking evaluation (the protocol of the NGCF paper's Gowalla / Yelp2018 / Amazon-Book numbers) on top of it: every
item is scored for every test user, the user's training items are dropped (``score_topk(..., exclude=train)``), and
Recall / Precision / NDCG / Hit at K are computed against the held-out items on the device (``full_rank_eval``)."""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib

MAX_CUTOFFS = 8           # ngcf_rank_metrics: at most 8 cut-offs K ...
MAX_K = 128               # ... each <= 128 (the longest list ngcf_score_topk returns)


class Interactions:
    """Per-row item sets as a CSR: ``ptr`` int64 [n_rows + 1], ``idx`` int32; row r's items ``idx[ptr[r]:ptr[r+1]]``
    are ascending and unique (the kernels rely on that).  Build it with :meth:`from_pairs`, which establishes it."""

    def __init__(self, ptr: torch.Tensor, idx: torch.Tensor, n_rows: int, n_items: int):
        self.ptr, self.idx, self.n_rows, self.n_items = ptr, idx, int(n_rows), int(n_items)

    @classmethod
    def from_pairs(cls, user, item, n_items: int, rows=None) -> "Interactions":
        """(user, item) pairs -> per-row sorted, de-duplicated item lists, on the device of ``user``.

        ``rows=None``: row r holds user r's items, for r in ``0 .. max(user)``.  Otherwise row r holds the items of user
        ``rows[r]`` (unique ids, any order; e.g. ``test_users.unique()``) and pairs of other users are left out.  Item
        ids outside ``[0, n_items)`` and negative user ids raise ``ValueError``."""
        user = torch.as_tensor(user).reshape(-1).to(torch.int64)
        item = torch.as_tensor(item).reshape(-1).to(device=user.device, dtype=torch.int64)
        n_items = int(n_items)
        if not 0 < n_items <= 0x7fffffff:
            raise ValueError(f"Interactions: n_items {n_items} not in [1, 2^31-1]")
        if user.numel() != item.numel():
            raise ValueError(f"Interactions: {user.numel()} users but {item.numel()} items")
        if item.numel() and (int(item.min()) < 0 or int(item.max()) >= n_items):
            raise ValueError(f"Interactions: item ids must lie in [0, {n_items})")
        if user.numel() and int(user.min()) < 0:
            raise ValueError("Interactions: negative user id")
        if rows is None:
            n_rows = int(user.max()) + 1 if user.numel() else 0
            row = user
        else:
            rows = torch.as_tensor(rows).reshape(-1).to(device=user.device, dtype=torch.int64)
            n_rows = rows.numel()
            srt, order = torch.sort(rows)
            if n_rows > 1 and bool((srt[1:] == srt[:-1]).any()):
                raise ValueError("Interactions: rows must be unique user ids")
            pos = torch.searchsorted(srt, user).clamp_(max=max(n_rows - 1, 0))
            keep = srt[pos] == user if n_rows else torch.zeros_like(user, dtype=torch.bool)
            row, item = order[pos[keep]], item[keep]
        key = torch.unique(row * n_items + item)                          # sorted: by row, then item; duplicates gone
        row = torch.div(key, n_items, rounding_mode="floor")
        counts = torch.bincount(row, minlength=n_rows)
        ptr = torch.cat((counts.new_zeros(1), counts.cumsum(0)))
        return cls(ptr, (key - row * n_items).to(torch.int32), n_rows, n_items)

    def to(self, device) -> "Interactions":
        ptr = self.ptr.to(device)
        if ptr is self.ptr:
            return self
        return Interactions(ptr, self.idx.to(device), self.n_rows, self.n_items)

    def __repr__(self):
        return f"Interactions(n_rows={self.n_rows}, n_items={self.n_items}, nnz={self.idx.numel()})"


def _check_interactions(x, what: str, n_rows: int, n_items: int) -> None:
    if not isinstance(x, Interactions):
        raise TypeError(f"{what} must be an Interactions (Interactions.from_pairs)")
    if x.n_rows != n_rows or x.n_items != n_items:
        raise ValueError(f"{what} has {x.n_rows} rows over {x.n_items} items; the embeddings have {n_rows} users and "
                         f"{n_items} items")


def _check_cutoffs(Ks) -> list:
    Ks = [int(K) for K in Ks]
    if not 1 <= len(Ks) <= MAX_CUTOFFS:
        raise ValueError(f"Ks: 1 to {MAX_CUTOFFS} cut-offs, got {len(Ks)}")
    if Ks[0] < 1 or any(b <= a for a, b in zip(Ks, Ks[1:])):
        raise ValueError(f"Ks must be strictly ascending and >= 1, got {Ks}")
    if Ks[-1] > MAX_K:
        raise ValueError(f"Ks: the largest cut-off is {MAX_K}, got {Ks[-1]}")
    return Ks


@_lib.on_device
def score_topk(u_embeds: torch.Tensor, item_embeds: torch.Tensor, k: int, exclude: Interactions | None = None):
    """Returns (values [U,k] fp32, indices [U,k] int64), descending, like ``torch.topk(u @ items.T, k)``.

    ``exclude``: an :class:`Interactions` with one row per user row of ``u_embeds``; user r's listed items are never
    ranked (a user's training items in full-ranking evaluation).  A row with fewer than k items left ends in slots
    with index -1 and value ``-FLT_MAX``.  k <= 32 runs on the tensor cores (n_items >= 1024, D a multiple of 4); k > 32
    runs a much slower CUDA-core kernel (~8 ms per 1 024 users at Gowalla shape)."""
    if u_embeds.device.type != "cuda" or item_embeds.device.type != "cuda":
        raise RuntimeError("score_topk (B200) runs on CUDA tensors only; there is no CPU fallback")
    lib = _lib.load()
    u = u_embeds.detach().to(torch.float32).contiguous()
    it = item_embeds.detach().to(torch.float32).contiguous()
    if u.dim() != 2 or it.dim() != 2 or u.shape[1] != it.shape[1]:
        raise RuntimeError(f"mat1 and mat2 shapes cannot be multiplied ({tuple(u.shape)} and {tuple(it.T.shape)})")
    U, D = u.shape
    n_items = it.shape[0]
    if k > n_items:
        raise RuntimeError("selected index k out of range")          # what torch.topk raises
    if exclude is not None:
        _check_interactions(exclude, "exclude", U, n_items)
        exclude = exclude.to(u.device)
    need = C.c_size_t(0)
    _lib.check(lib.ngcf_score_topk_workspace(U, n_items, D, k, C.byref(need)), "score_topk_workspace")
    ws = torch.empty(need.value, dtype=torch.uint8, device=u.device)
    val = torch.empty(U, k, dtype=torch.float32, device=u.device)
    idx = torch.empty(U, k, dtype=torch.int64, device=u.device)
    if exclude is None:
        _lib.check(lib.ngcf_score_topk(u.data_ptr(), U, it.data_ptr(), n_items, D, k, val.data_ptr(), idx.data_ptr(),
                                       ws.data_ptr(), need.value, _lib.current_stream()), "score_topk")
    else:
        _lib.check(lib.ngcf_score_topk_excluding(u.data_ptr(), U, it.data_ptr(), n_items, D, k, exclude.ptr.data_ptr(),
                                                 _lib.ptr(exclude.idx), val.data_ptr(), idx.data_ptr(), ws.data_ptr(),
                                                 need.value, _lib.current_stream()), "score_topk_excluding")
    return val, idx


@_lib.on_device
def rank_metrics(topk_idx: torch.Tensor, truth: Interactions, Ks=(20,)):
    """Recall / Precision / NDCG / Hit at each K of ranked lists ``topk_idx`` [U, k] int64 (-1 = empty slot) against
    ``truth`` (one row per list).  Returns CUDA tensors, without synchronising: ``totals`` [len(Ks)*4 + 1] = per K the
    means (recall, precision, ndcg, hit) over the users with a non-empty truth row, then their number; ``per_user``
    [U, len(Ks), 4] (zeros for users without truth items).  Capturable in a CUDA graph once ``truth`` is on the device."""
    Ks = _check_cutoffs(Ks)
    if topk_idx.dim() != 2:
        raise ValueError("rank_metrics: topk_idx must be [users, k]")
    U, k = topk_idx.shape
    if not isinstance(truth, Interactions) or truth.n_rows != U:
        raise ValueError(f"rank_metrics: truth must be an Interactions with {U} rows")
    if Ks[-1] > k:
        raise ValueError(f"rank_metrics: cut-off {Ks[-1]} > list length {k}")
    if topk_idx.device.type != "cuda":
        raise RuntimeError("rank_metrics (B200) runs on CUDA tensors only; there is no CPU fallback")
    lib = _lib.load()
    idx = topk_idx.to(torch.int64).contiguous()
    truth = truth.to(idx.device)
    per = torch.empty(U, len(Ks), 4, dtype=torch.float32, device=idx.device)
    totals = torch.empty(len(Ks) * 4 + 1, dtype=torch.float32, device=idx.device)
    _lib.check(lib.ngcf_rank_metrics(idx.data_ptr(), U, k, truth.ptr.data_ptr(), _lib.ptr(truth.idx), _lib.int_array(Ks),
                                     len(Ks), per.data_ptr(), totals.data_ptr(), _lib.current_stream()), "rank_metrics")
    return totals, per


@_lib.on_device
def full_rank_eval(user_embeds: torch.Tensor, item_embeds: torch.Tensor, *, train: Interactions, test: Interactions,
                   Ks=(20,), return_per_user: bool = False):
    """Full-ranking evaluation: every item scored for every row of ``user_embeds``, the row's ``train`` items dropped,
    the top ``max(Ks)`` kept and compared with its ``test`` items.  Returns ``{"recall@K", "precision@K", "ndcg@K",
    "hit@K" for each K, "n_users"}`` (means over the rows with test items; one device-to-host read), and with
    ``return_per_user`` also the [rows, len(Ks), 4] per-row (recall, precision, ndcg, hit) tensor.  ``max(Ks)`` <= 32 runs
    on the tensor cores; larger cut-offs take the slow CUDA-core ranking (see :func:`score_topk`)."""
    Ks = _check_cutoffs(Ks)
    U, n_items = user_embeds.shape[0], item_embeds.shape[0]
    _check_interactions(train, "train", U, n_items)
    _check_interactions(test, "test", U, n_items)
    if user_embeds.device.type != "cuda" or item_embeds.device.type != "cuda":
        raise RuntimeError("full_rank_eval (B200) runs on CUDA tensors only; there is no CPU fallback")
    _, idx = score_topk(user_embeds, item_embeds, Ks[-1], exclude=train)
    totals, per = rank_metrics(idx, test, Ks)
    vals = totals.tolist()
    out = {}
    for j, K in enumerate(Ks):
        for m, name in enumerate(("recall", "precision", "ndcg", "hit")):
            out[f"{name}@{K}"] = vals[4 * j + m]
    out["n_users"] = int(vals[-1])
    return (out, per) if return_per_user else out
