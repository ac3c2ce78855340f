"""Triple sampler on the device (SURVEY.md section 8(f) #3): the reference's ``TourDataset`` (model/utils.py:168-275).

The reference builds its (positive, negative) rows with a Python loop over users that re-scans the frame per user
(``df.loc[df['userid'].isin([userid])]``, utils.py:236) and calls ``np.random.choice(neg_items, ng_ratio,
replace=False)`` per positive row (utils.py:258) — O(users x rows) pandas work before the first training step.
Here the frame is indexed once on the host (vectorised numpy: first-seen user order, per-user sorted positive lists)
and ``ngcf_sample_negatives`` draws every row's negatives in one launch.

Same outputs (``users`` / ``items`` LongTensors in the reference's row order and layout, ``__len__``, ``__getitem__``)
and the same distribution: per positive row an ordered uniform sample, without replacement, of the items the user has
no positive feedback for.  The random STREAM differs (counter-based device RNG keyed on (seed, row, draw) instead of
numpy's global MT19937), so parity is distributional and structural, not bit-wise; ``tests/`` pin the row layout
against the reference's own output and check the draws' support, distinctness and uniformity.
"""
from __future__ import annotations

import numpy as np
import torch

from . import _lib

CONTEXT_COLS = ("year", "userid", "age", "sex", "month", "day", "dayofweek")      # utils.py:242-248


@_lib.on_device
def sample_negatives(pos_ptr, pos_idx, row_user, candidates, ng_ratio: int, seed: int):
    """out[r, :] = ng_ratio distinct entries of ``candidates`` outside user row_user[r]'s positive list
    (pos_idx[pos_ptr[u]:pos_ptr[u+1]] = ascending unique candidate indices).  CUDA tensors in, CUDA int64 [R, ng] out."""
    if row_user.device.type != "cuda":
        raise RuntimeError("sample_negatives (B200) runs on CUDA tensors only; there is no CPU fallback")
    lib = _lib.load()
    dev = row_user.device
    pos_ptr = pos_ptr.to(device=dev, dtype=torch.int32).contiguous()
    pos_idx = pos_idx.to(device=dev, dtype=torch.int32).contiguous()
    row_user = row_user.to(torch.int64).contiguous()
    candidates = candidates.to(device=dev, dtype=torch.int64).contiguous()
    R = row_user.numel()
    out = torch.empty(R, ng_ratio, dtype=torch.int64, device=dev)
    n_short = torch.zeros(1, dtype=torch.int32, device=dev)
    _lib.check(lib.ngcf_sample_negatives(pos_ptr.data_ptr(), _lib.ptr(pos_idx) if pos_idx.numel() else None,
                                         row_user.data_ptr(), R, candidates.data_ptr(), candidates.numel(),
                                         int(ng_ratio), int(seed) & (2 ** 64 - 1), out.data_ptr(), n_short.data_ptr(),
                                         _lib.current_stream()), "sample_negatives")
    if int(n_short) > 0:
        raise ValueError("Cannot take a larger sample than population when 'replace=False'")   # numpy's, utils.py:258
    return out


def index_frame(cols: dict, total_items, rating_col: str = "rating"):
    """Host index of the frame (O(rows log rows), no per-user scans): the reference's row order — users in first-seen
    order, each user's positive rows in frame order (utils.py:235-238,251) — and the per-user positive lists.
    Returns dict(rows, row_user, pos_ptr, pos_idx, candidates)."""
    uid = np.asarray(cols["userid"])
    rating = np.asarray(cols[rating_col])
    item = np.asarray(cols["itemid"])
    cand = np.unique(np.asarray(total_items))                                   # utils.py:224; np.setxor1d sorts
    _, first, inv = np.unique(uid, return_index=True, return_inverse=True)
    rank = np.empty(first.size, dtype=np.int64)
    rank[np.argsort(first, kind="stable")] = np.arange(first.size)
    code = rank[inv.reshape(-1)]                                                # user -> first-seen rank
    rows = np.flatnonzero(rating > 0)                                           # utils.py:238
    rows = rows[np.argsort(code[rows], kind="stable")]
    cidx = np.searchsorted(cand, item[rows])
    if rows.size and (cidx.max() >= cand.size or not np.array_equal(cand[cidx], item[rows])):
        raise ValueError("df holds item ids that total_df does not")
    pairs = np.unique(code[rows] * np.int64(cand.size) + cidx)                  # unique (user, item), ascending
    pu, pi = pairs // cand.size, pairs % cand.size
    pos_ptr = np.zeros(first.size + 1, dtype=np.int64)
    np.cumsum(np.bincount(pu, minlength=first.size), out=pos_ptr[1:])
    return dict(rows=rows, row_user=code[rows], pos_ptr=pos_ptr.astype(np.int32), pos_idx=pi.astype(np.int32),
                candidates=cand.astype(np.int64))


class TourDataset(torch.utils.data.Dataset):
    """``TourDataset(df, total_df, train, rating_col)`` of utils.py:168-211 (pandas frames or dicts of columns).
    ``seed``: device-RNG key (default: drawn from torch's CPU generator, so ``torch.manual_seed`` reproduces it)."""

    def __init__(self, df, total_df, train: bool, rating_col: str, device="cuda", seed: int | None = None):
        super().__init__()
        self.df, self.total_df, self.train, self.rating_col = df, total_df, train, rating_col
        self.device = torch.device(device)
        self.seed = int(torch.randint(0, 2 ** 62, (1,)).item()) if seed is None else int(seed)
        self.users, self.items = self._negative_sampling()

    def __len__(self) -> int:
        return len(self.users)

    def __getitem__(self, index):
        u = self.users[index]
        if self.train:                       # year, uid, a, s, m, d, dow, pos, neg (utils.py:201-204)
            return u[0], u[1], u[2], u[3], u[4], u[5], u[6], self.items[index][0], self.items[index][1]
        return u[0], u[1], u[2], u[3], u[4], u[5], u[6], u[7], self.items[index]      # utils.py:206-209

    def _negative_sampling(self):
        if self.device.type != "cuda":
            raise RuntimeError("TourDataset (B200) samples on a CUDA device only; there is no CPU fallback")
        col = (lambda f, c: f[c].to_numpy()) if hasattr(self.df, "columns") else (lambda f, c: np.asarray(f[c]))
        cols = {c: col(self.df, c) for c in CONTEXT_COLS + ("itemid", self.rating_col)}
        ix = index_frame(cols, col(self.total_df, "itemid"), self.rating_col)
        ng_ratio = 1 if self.train else 24                                       # utils.py:227-230
        dev = self.device
        rows = ix["rows"]
        neg = sample_negatives(torch.from_numpy(ix["pos_ptr"]).to(dev), torch.from_numpy(ix["pos_idx"]).to(dev),
                               torch.from_numpy(ix["row_user"]).to(dev), torch.from_numpy(ix["candidates"]).to(dev),
                               ng_ratio, self.seed).cpu()
        ctx = [cols[c][rows] for c in CONTEXT_COLS]
        pos = torch.from_numpy(cols["itemid"][rows].astype(np.int64))
        if self.train:
            users = np.stack(ctx, axis=1).astype(np.int64)                       # [R, 7]
            items = torch.cat((pos[:, None], neg), dim=1)                        # [R, 2]: positive, negative
        else:
            users = np.stack(ctx + [cols[self.rating_col][rows]], axis=1).astype(np.int64)    # LongTensor truncates
            users = np.repeat(users, ng_ratio + 1, axis=0)                       # [R*25, 8] (utils.py:249-266)
            items = torch.cat((pos[:, None], neg), dim=1).reshape(-1)            # [R*25]: positive, then its negatives
        return torch.from_numpy(users).reshape(-1, 7 if self.train else 8), items


class HardNegatives:
    """Dynamic hard-negative sampling (DNS): pass as ``neg_item=`` to ``NGCF.forward`` (or ``negatives=`` to
    ``GraphedStep``) and each batch row's negative is chosen on the device, inside the step, from ``n_candidates``
    items drawn uniformly (with replacement) among those the user has no ``train`` interaction with: the candidate
    whose final embedding row has the largest |dot product| with the user's, under the layer outputs of that same
    forward.  ``train``: an :class:`Interactions` with one row per user, e.g. ``Interactions.from_pairs(users, items,
    n_item, rows=torch.arange(n_user))``.  After each forward ``chosen`` (int64 [B], item ids) holds the picks; with
    ``debug=True`` also ``cand`` (int64 [B, n_candidates]) and ``score`` (fp32 [B, n_candidates]).

    ``signed=True`` picks the candidate of largest signed score instead, for :class:`SoftmaxLoss`: there a large
    negative score is an easy negative, while BPR's loss compares |u.p| with |u.n|."""

    MAX_CANDIDATES = 64                  # ngcf_hard_negatives: M <= 64

    def __init__(self, train, n_candidates: int = 32, *, signed: bool = False, debug: bool = False):
        from .scoring import Interactions
        if not isinstance(train, Interactions):
            raise TypeError("HardNegatives: train must be an Interactions (Interactions.from_pairs)")
        n_candidates = int(n_candidates)
        if not 1 <= n_candidates <= self.MAX_CANDIDATES:
            raise ValueError(f"HardNegatives: n_candidates {n_candidates} not in [1, {self.MAX_CANDIDATES}]")
        deg = train.ptr.detach().cpu().diff()
        if deg.numel() and int(deg.max()) >= train.n_items:
            # the kernel draws from the items outside the row's list and has no way to report an empty set
            u = int(torch.nonzero(deg >= train.n_items)[0])
            raise ValueError(f"HardNegatives: row {u} lists all {train.n_items} items; it has no negative to draw")
        self.train, self.n_candidates, self.signed, self.debug = train, n_candidates, bool(signed), bool(debug)
        self.chosen = self.cand = self.score = None
        self._dev = {}

    def _on(self, device):
        """``train`` on ``device``, copied once (a forward under CUDA-graph capture must not copy from the host)."""
        t = self._dev.get(device)
        if t is None:
            t = self._dev[device] = self.train.to(device)
        return t

    def __repr__(self):
        return f"HardNegatives({self.train!r}, n_candidates={self.n_candidates})"
