"""Drop-in ``NGCF`` module (reference: model/NGCF.py:7-156) over the B200 C-ABI kernels.

Same constructor, ``forward`` signature, attributes (``all_users_emb`` / ``all_items_emb``), parameter
names/order/shapes (``state_dict`` compatible both ways with the reference's ``.pth`` files) and the same
initialisation stream, so ``main.py`` / ``demo.py`` run unchanged with this module on ``sys.path`` first.
Everything numerical runs in libngcf_b200.so; there is no PyTorch/CPU fallback.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np
import torch
import torch.nn as nn

import torch.distributed as dist

from . import _lib
from .plan import LaplacianPlan, NodeDropout, spmm
from .sampler import HardNegatives
from .sharded import RowShards, all_gather_rows

LEAKY_SLOPE = 0.2   # NGCF.py:140


class _Ctx:
    """Per-forward state shared by an autograd node and its module (NGCF or LightGCN): plan, layer outputs, RNG key,
    node dropout, batch rows.  LightGCN leaves the NGCF-only fields (dims, S, W1, W2, vals_*, mess_*, last_partial,
    fm_stream) unset."""
    __slots__ = ("plan", "E", "seed", "seed_dev", "drop_p", "dropout", "rows", "offsets", "fresh_key", "hneg",
                 "dims", "S", "W1", "W2", "vals_f", "vals_b", "mess_mult", "mess_p", "mess_bits", "last_partial",
                 "fm_stream")

    @property
    def node_mode(self) -> str:
        return self.dropout.mode


class _RowGrads:
    """A backward's output-row gradients summed per distinct row (ngcf_rowgrad_scatter): row r's sum is gsum[slot[r]],
    slot[r] = -1 for rows without one.  ``reset()`` puts those slots back to -1 at the end of the backward."""

    def __init__(self, mod, st: _Ctx, gouts, n_sets: int, width: int, n_rows: int):
        dev = st.E[0].device
        g = [(go.contiguous() if go is not None else torch.zeros(st.rows[j].numel(), width, device=dev))
             for j, go in enumerate(gouts)]
        batch = [r.numel() for r in st.rows[:n_sets]]
        self.n_sets, self.rows, self.offs = n_sets, _lib.ptr_array(st.rows[:n_sets]), _lib.i64_array(st.offsets[:n_sets])
        self.batch = _lib.i64_array(batch)
        self.slot = mod._slot_map(n_rows, dev)
        self.gsum = torch.empty(max(sum(batch), 1), width, dtype=torch.float32, device=dev)
        _lib.check(_lib.load().ngcf_rowgrad_scatter(self.rows, self.offs, _lib.ptr_array(g), self.batch, n_sets, width,
                                                    self.slot.data_ptr(), self.gsum.data_ptr(), _lib.current_stream()),
                   "rowgrad_scatter")

    def reset(self):
        _lib.check(_lib.load().ngcf_rowgrad_reset(self.rows, self.offs, self.batch, self.n_sets, self.slot.data_ptr(),
                                                  _lib.current_stream()), "rowgrad_reset")


def _index(t, dev) -> torch.Tensor:
    return t.to(device=dev, dtype=torch.int64).contiguous()


def _capturing() -> bool:
    return torch.cuda.is_current_stream_capturing()


def _join_feature_mix(st):
    """The feature mix of this forward ran on a second stream (NGCF.forward): whatever reads the table next waits for it."""
    if st.fm_stream is not None:
        torch.cuda.current_stream().wait_stream(st.fm_stream)
        st.fm_stream = None


class _Propagate(torch.autograd.Function):
    """K-layer propagation + output-row gather (NGCF.py:120-156) and its hand-written backward.

    With ``mod._shard`` set (row-sharded multi-GPU run, sharded.py) every per-layer tensor below holds this rank's
    row block only and ``st.E[k]`` is the full ``[N_pad, d_k]`` layer input, assembled by one exchange per layer and
    direction plus one for the table gradient and one for the W/b gradients: peer-memory stores over NVLink
    (sharded.PeerExchange; the last layer's output travels for the batch rows only) or, without symmetric memory, NCCL
    all-gathers / an all-reduce.  Without a shard ``st.E[k]`` is simply E_k and nothing is communicated."""

    @staticmethod
    def forward(ctx, mod, st: _Ctx, n_sets, user_w, item_w, *wb):
        lib = _lib.load()
        K = mod.n_layer
        W1, b1, W2, b2 = wb[0:K], wb[K:2 * K], wb[2 * K:3 * K], wb[3 * K:4 * K]
        dev = user_w.device
        sh = mod._shard
        N = mod.n_user + mod.n_item
        r0, nloc, nv = (sh.r0, sh.rows, sh.valid) if sh is not None else (0, N, N)
        X0 = mod._packed_table()                                       # [N(_pad), d0] = cat(user, item), NGCF.py:120
        if mod._snapshot:                                              # the reference's cat() is a copy: opt-in here
            _join_feature_mix(st)
            X0 = X0.clone()
        st.E, st.S, st.W1, st.W2 = [X0], [], list(W1), list(W2)
        side = st.plan.fwd
        st.last_partial = None
        # the reference's own width 65 runs the row-per-warp kernel from per-step decision bytes (NodeDropout)
        st.dropout = NodeDropout(st.plan, mod._node_mode, st.drop_p, st.seed, st.seed_dev, K, r0, st.dims)
        # message dropout (NGCF.py:142): optionally this step's decisions for every layer, one bit per element, drawn
        # by a full-GPU pass instead of inside the dense kernels (measured slower at Gowalla shape: off by default)
        self_uses_mess_bits = mod._mess_bits
        st.mess_bits = [None] * K
        for k in range(K):
            if self_uses_mess_bits and st.mess_mult is None and st.mess_p[k] > 0 and st.dims[k + 1] % 4 == 0:
                bits = torch.empty(nloc * ((st.dims[k + 1] + 31) // 32), dtype=torch.int32, device=dev)
                _lib.check(lib.ngcf_mess_dropout_bits(nv, st.dims[k + 1], float(st.mess_p[k]), st.seed,
                                                      _lib.ptr(st.seed_dev), k, r0, bits.data_ptr(),
                                                      _lib.current_stream()),
                           "mess_dropout_bits")
                st.mess_bits[k] = bits
        # [W1^T ; W2^T] and 2 b1 + b2 of every layer: one launch (NGCF.py:131-136 applies w1_list[i] twice)
        wcats = [torch.empty(2 * st.dims[k] * st.dims[k + 1], dtype=torch.float32, device=dev) for k in range(K)]
        biases = [torch.empty(st.dims[k + 1], dtype=torch.float32, device=dev) for k in range(K)]
        _lib.check(lib.ngcf_pack_weights_all(_lib.ptr_array(W1), _lib.ptr_array(b1), _lib.ptr_array(W2), _lib.ptr_array(b2),
                                             _lib.int_array(st.dims[:K]), _lib.int_array(st.dims[1:]), K,
                                             _lib.ptr_array(wcats), _lib.ptr_array(biases), _lib.current_stream()),
                   "pack_weights_all")
        _join_feature_mix(st)                                          # the first product reads the mixed user rows
        for k in range(K):
            d_in, d_out = st.dims[k], st.dims[k + 1]
            vals = st.vals_f[k] if st.vals_f is not None else None
            S = spmm(side, vals, st.E[k], d_in, **st.dropout.args(k))                           # NGCF.py:124-130
            wcat, bias = wcats[k], biases[k]
            xkey = None
            if sh is None:
                Xn = En = torch.empty(N, d_out, dtype=torch.float32, device=dev)
            elif mod._xchg is not None and d_out % 4 == 0:
                xkey = ("E", k + 1)                                    # persistent symmetric matrix: this rank's rows are
                Xn = mod._xchg.matrix(xkey, sh.N_pad, d_out)           # written in place, then pushed to the peers
                En = Xn[r0:r0 + nloc]
            else:
                Xn = torch.empty(sh.N_pad, d_out, dtype=torch.float32, device=dev)
                En = torch.zeros(nloc, d_out, dtype=torch.float32, device=dev) if nv < nloc else \
                    torch.empty(nloc, d_out, dtype=torch.float32, device=dev)
            mm = st.mess_mult[k] if st.mess_mult is not None else None
            E_loc = st.E[k][r0:r0 + nloc]
            _lib.check(lib.ngcf_dense_fwd(S.data_ptr(), E_loc.data_ptr(), nv, d_in, d_out, wcat.data_ptr(),
                                          bias.data_ptr(), LEAKY_SLOPE, _lib.ptr(mm[r0:r0 + nloc] if mm is not None else None),
                                          _lib.ptr(st.mess_bits[k]), float(st.mess_p[k]), st.seed, _lib.ptr(st.seed_dev), k, r0, En.data_ptr(),
                                          _lib.current_stream()),
                       "dense_fwd")                                                          # NGCF.py:131-142
            if xkey is not None and k == K - 1:
                # nothing downstream gathers from the LAST layer's output: other ranks need it for the <= 3 B batch rows only
                # (NGCF.py:151-155); all_users_emb / all_items_emb complete it on first read (_materialize)
                mod._xchg.push_selected(xkey, r0, nloc, st.rows[:n_sets], st.offsets[:n_sets])
                st.last_partial = xkey
            elif xkey is not None:
                mod._xchg.push(xkey, r0, nloc)                         # every rank needs all of E_{k+1}
            elif sh is not None:
                all_gather_rows(Xn, En, mod._group)
            st.S.append(S)
            st.E.append(Xn)
        D = sum(st.dims)
        layers, dims = _lib.ptr_array(st.E), _lib.int_array(st.dims)
        if st.hneg is not None:                                        # dynamic hard negatives: fills st.rows[2]
            hn, train, chosen, cand, score = st.hneg
            pick = lib.ngcf_hard_negatives_signed if hn.signed else lib.ngcf_hard_negatives
            _lib.check(pick(layers, dims, K + 1, mod.n_user, st.rows[0].data_ptr(),
                            st.rows[0].numel(), train.ptr.data_ptr(), _lib.ptr(train.idx),
                            mod.n_item, hn.n_candidates, st.seed, _lib.ptr(st.seed_dev),
                            chosen.data_ptr(), _lib.ptr(cand), _lib.ptr(score), _lib.current_stream()),
                       "hard_negatives")
        outs =[torch.empty(st.rows[j].numel(), D, dtype=torch.float32, device=dev) for j in range(n_sets)]
        _lib.check(lib.ngcf_gather_concat_sets(layers, dims, K + 1, _lib.ptr_array(st.rows[:n_sets]),
                                               _lib.i64_array(st.offsets[:n_sets]),
                                               _lib.i64_array([r.numel() for r in st.rows[:n_sets]]), _lib.ptr_array(outs),
                                               n_sets, D, _lib.current_stream()), "gather_concat_sets")   # NGCF.py:144-155
        ctx.st, ctx.mod, ctx.n_sets = st, mod, n_sets
        return tuple(outs)

    @staticmethod
    def backward(ctx, *gouts):
        lib = _lib.load()
        st, mod, n_sets = ctx.st, ctx.mod, ctx.n_sets
        mod._check_fresh(st, "loss.backward()")
        K, dims = mod.n_layer, st.dims
        dev = st.E[0].device
        sh = mod._shard
        N = mod.n_user + mod.n_item
        r0, nloc, nv, N_all = (sh.r0, sh.rows, sh.valid, sh.N_pad) if sh is not None else (0, N, N, N)
        D = sum(dims)
        rg = _RowGrads(mod, st, gouts, n_sets, D, N_all)
        slot, gsum = rg.slot, rg.gsum
        # F.normalize's backward (NGCF.py:144) for the <= 3B rows that carry an output-row gradient, once, in place
        _lib.check(lib.ngcf_rowgrad_normalize(rg.rows, rg.offs, rg.batch, n_sets, _lib.ptr_array(st.E),
                                              _lib.int_array(dims), K + 1, slot.data_ptr(), gsum.data_ptr(), D,
                                              _lib.current_stream()), "rowgrad_normalize")
        slot_loc = slot[r0:r0 + nloc]
        sizes = [dims[k + 1] * dims[k] for k in range(K)]
        n_flat = 2 * sum(sizes) + 2 * sum(dims[1:])
        if sh is not None and mod._xchg is not None:
            # W/b gradients of all ranks side by side in one symmetric [world, F] matrix: this rank accumulates into its own
            # row, pushes it, and every rank adds the rows up in rank order (same bits everywhere, no NCCL launch)
            f_pad = (n_flat + 3) // 4 * 4
            wg_all = mod._xchg.matrix(("wgrad", f_pad), sh.world, f_pad)
            flat = wg_all[sh.rank, :n_flat]
            flat.zero_()
        else:
            wg_all = None
            flat = torch.zeros(n_flat, dtype=torch.float32, device=dev)
        gW1, gW2, gb1, gb2, o = [], [], [], [], 0
        for k in range(K):
            gW1.append(flat[o:o + sizes[k]].view(dims[k + 1], dims[k])); o += sizes[k]
            gW2.append(flat[o:o + sizes[k]].view(dims[k + 1], dims[k])); o += sizes[k]
            gb1.append(flat[o:o + dims[k + 1]]); o += dims[k + 1]
            gb2.append(flat[o:o + dims[k + 1]]); o += dims[k + 1]
        # explicit (COO-order) masks need the separately sorted L^T; in-kernel device-RNG dropout is keyed on the
        # entry's coordinates, so a symmetric L keeps sharing its forward arrays (transposed=1 swaps the key)
        side = st.plan.side(True, st.vals_b is not None)
        st.dropout.draw_transposed()
        gE_next = None
        col_off = D
        # the weight-gradient kernels need gM only: beside the transposed product (and the gS exchange queued behind the
        # backward kernel in row-sharded runs) they run on a second stream; each layer then keeps its own gM until the
        # join below.  0.508 -> 0.494 ms per step on one B200 (GraphedStep), 0.611 -> 0.594 ms at 2 ranks.
        # (second streams cost the HOST two event calls per fork and join: they pay under CUDA-graph capture, where the
        # step is replayed without host work, and in row-sharded runs; the eager single-GPU step is host-bound already)
        overlap = _capturing() or (sh is not None and mod._xchg is not None)
        if overlap:
            if mod._side_stream is None:
                mod._side_stream = torch.cuda.Stream(device=dev)
            _lib.check(lib.ngcf_set_wgrad_stream(mod._side_stream.cuda_stream), "set_wgrad_stream")
            lib.ngcf_wgrad_stream_forked()                            # clear the flag
            gM_keep = []
        else:
            gM_scratch = torch.empty(nloc, max(dims[1:]), dtype=torch.float32, device=dev)
        for k in range(K - 1, -1, -1):
            d_in, d_out = dims[k], dims[k + 1]
            col_off -= d_out
            peer = sh is not None and mod._xchg is not None and d_in % 4 == 0
            if peer:                                                  # gS rows in place in the symmetric matrix
                gS_all = mod._xchg.matrix(("gS", d_in), N_all, d_in)
                gS = gS_all[r0:r0 + nloc]
            else:
                gS = torch.empty(nloc, d_in, dtype=torch.float32, device=dev)
            if peer and k == 0:                                       # gE_0 = gEl + L^T gS accumulates in place in ITS matrix
                gE0_all = mod._xchg.matrix(("gE0", d_in), N_all, d_in)
                gEl = gE0_all[r0:r0 + nloc]
            else:
                gEl = torch.empty(nloc, d_in, dtype=torch.float32, device=dev)
            mm = st.mess_mult[k] if st.mess_mult is not None else None
            if overlap:
                gM_scratch = torch.empty(nloc, dims[k + 1], dtype=torch.float32, device=dev)
                gM_keep.append(gM_scratch)
            _lib.check(lib.ngcf_dense_bwd(_lib.ptr(gE_next), slot_loc.data_ptr(), gsum.data_ptr(), D, col_off,
                                          st.E[k + 1][r0:r0 + nloc].data_ptr(), st.S[k].data_ptr(),
                                          st.E[k][r0:r0 + nloc].data_ptr(), nv, d_in, d_out,
                                          st.W1[k].data_ptr(), st.W2[k].data_ptr(), LEAKY_SLOPE,
                                          _lib.ptr(mm[r0:r0 + nloc] if mm is not None else None),
                                          _lib.ptr(st.mess_bits[k]), float(st.mess_p[k]), st.seed,
                                          _lib.ptr(st.seed_dev), k, r0, 1, gS.data_ptr(),
                                          gEl.data_ptr(),
                                          gW1[k].data_ptr(), gb1[k].data_ptr(), gW2[k].data_ptr(), gb2[k].data_ptr(),
                                          gM_scratch.data_ptr(), _lib.current_stream()), "dense_bwd")
            if peer:                                                  # L^T gS needs every rank's rows of gS
                mod._xchg.push(("gS", d_in), r0, nloc)
            elif sh is not None:
                gS_all = torch.empty(N_all, d_in, dtype=torch.float32, device=dev)
                all_gather_rows(gS_all, gS, mod._group)
            else:
                gS_all = gS
            vals = st.vals_b[k] if st.vals_b is not None else None
            last = (k == 0)
            gE_next = spmm(side, vals, gS_all, d_in, addend=gEl, slot=slot_loc if last else None,
                           gsum=gsum if last else None,
                           **st.dropout.args(k, transposed=True))              # gE_k = gEl + L^T gS (+ row grads)
            if mod._trace is not None:                                # debugging aid: per-layer backward tensors
                mod._trace.append(dict(k=k, gS=gS.clone(), gEl=gEl.clone(), gE=gE_next.clone()))
        if overlap:                                                   # join: the weight gradients are complete
            _lib.check(lib.ngcf_set_wgrad_stream(None), "set_wgrad_stream")
            if lib.ngcf_wgrad_stream_forked():                        # (FFMA layers never fork: nothing to wait for)
                torch.cuda.current_stream().wait_stream(mod._side_stream)
        rg.reset()
        if sh is not None:
            if mod._xchg is not None and dims[0] % 4 == 0:
                mod._xchg.push(("gE0", dims[0]), r0, nloc)             # tables are replicated: full gradient everywhere
                gE0 = gE0_all.clone()                                  # (the matrix is reused by the next step)
            else:
                gE0 = torch.empty(N_all, dims[0], dtype=torch.float32, device=dev)
                all_gather_rows(gE0, gE_next, mod._group)
            if wg_all is not None:                                    # W/b gradients: sum of the row blocks
                mod._xchg.push(("wgrad", wg_all.shape[1]), sh.rank, 1)
                total = wg_all.sum(0)[:n_flat]
                gW1, gW2, gb1, gb2, o = [], [], [], [], 0
                for k in range(K):
                    gW1.append(total[o:o + sizes[k]].view(dims[k + 1], dims[k])); o += sizes[k]
                    gW2.append(total[o:o + sizes[k]].view(dims[k + 1], dims[k])); o += sizes[k]
                    gb1.append(total[o:o + dims[k + 1]]); o += dims[k + 1]
                    gb2.append(total[o:o + dims[k + 1]]); o += dims[k + 1]
            else:
                dist.all_reduce(flat, group=mod._group)
        else:
            gE0 = gE_next
        gU, gI = gE0[:mod.n_user], gE0[mod.n_user:N]
        return (None, None, None, gU, gI, *gW1, *gb1, *gW2, *gb2)


def draw_seed(generator=None) -> int:
    """A per-forward device-RNG key from ``generator`` (default: torch's CPU generator, so ``torch.manual_seed``
    reproduces it)."""
    return int(torch.randint(0, 2 ** 62, (1,), generator=generator).item())


class _TableModel(nn.Module):
    """What NGCF and LightGCN share: E_0 of a forward is the live packed [N, d] table behind ``user_embedding`` and
    ``item_embedding`` (no copy), one execution plan per ``lap_list`` element, the row-gradient slot map, the rule
    that refuses to use a forward's E_0 once the table changed under it, and the forward's steps either side of the
    propagation: batch rows, feature mix, RNG key, and ``all_users_emb`` / ``all_items_emb`` built on first read.
    Subclasses set n_user, n_item, emb_size, n_layer, lap_list and rng, name themselves in _NAME and supply
    ``_readout``."""
    _STALE_ADVICE = "Run the forward again."

    def __init__(self):
        super().__init__()
        self._plans = {}
        self._table = None
        self._slot = None
        self._winner = None      # feature mix: per-user scratch of ngcf_feature_mix
        self._last = None        # _Ctx of the last forward
        self._all_E = None
        self._shard = None       # sharded.RowShards once NGCF.shard() was called
        self._snapshot = False
        self._mix_count = 0
        self._seed_dev = None    # device uint64 added to the RNG key (set by graph.GraphedStep)

    def _feature_tables(self, num_dict: dict):
        """The five feature tables in the reference's registration order (NGCF.py:39-45), which fixes the state_dict
        order; each nn.Embedding draws its initial values from the CPU generator.  The reference needs
        embed_size % 5 == 0 (its concat is 5*(emb//5) wide, NGCF.py:110-114); here the last table of the concat order
        (dow) absorbs the remainder, which is the same thing whenever emb % 5 == 0."""
        w = self.emb_size // 5
        self.feat_widths = [w, w, w, w, self.emb_size - 4 * w]          # age, sex, month, day, dow
        self.month_emb = nn.Embedding(int(num_dict['month']), w)
        self.day_emb = nn.Embedding(int(num_dict['day']), w)
        self.sex_emb = nn.Embedding(int(num_dict['sex']), w)
        self.age_emb = nn.Embedding(int(num_dict['age']), w)
        self.dow_emb = nn.Embedding(int(num_dict['dayofweek']), self.feat_widths[4])

    def _cuda_device(self) -> torch.device:
        dev = self.user_embedding.weight.device
        if dev.type != "cuda":
            raise RuntimeError(f"{self._NAME} (B200) runs on a CUDA device only; there is no CPU fallback. "
                               "Move the module with .to('cuda').")
        return dev

    def _batch(self, dev, u_id, pos_item, neg_item) -> _Ctx:
        """A forward's _Ctx with its row sets: users, positives and, unless ``neg_item`` is empty, negatives (st.rows,
        their offsets into the packed table in st.offsets).  With ``neg_item`` a HardNegatives the negatives are the
        buffer its device pass fills, and st.hneg holds that pass's operands."""
        st = _Ctx()
        u_id, pos_item = _index(u_id, dev), _index(pos_item, dev)
        hneg = neg_item if isinstance(neg_item, HardNegatives) else None
        if hneg is not None:
            if self._shard is not None:
                raise ValueError("HardNegatives: not available on a row-sharded model (the candidates' rows of the "
                                 "last layer are spread over the ranks)")
            if hneg.train.n_rows != self.n_user or hneg.train.n_items != self.n_item:
                raise ValueError(f"HardNegatives: train has {hneg.train.n_rows} rows over {hneg.train.n_items} items; "
                                 f"the model has {self.n_user} users and {self.n_item} items")
            neg_item = torch.empty(u_id.numel(), dtype=torch.int64, device=dev)   # written by the hard-negative pass
        else:
            neg_item = _index(neg_item, dev) if len(neg_item) > 0 else None   # NGCF.py:154
        st.rows = [u_id, pos_item] + ([neg_item] if neg_item is not None else [])
        st.offsets = [0, self.n_user] + ([self.n_user] if neg_item is not None else [])
        st.hneg = None
        if hneg is not None:
            M = hneg.n_candidates
            st.hneg = (hneg, hneg._on(dev), neg_item,
                       torch.empty(u_id.numel(), M, dtype=torch.int64, device=dev) if hneg.debug else None,
                       torch.empty(u_id.numel(), M, dtype=torch.float32, device=dev) if hneg.debug else None)
            hneg.chosen, hneg.cand, hneg.score = st.hneg[2:]
        return st

    def _feature_mix(self, table, u_id, feats):
        """The feature mix of the batch users' rows of ``table`` (NGCF.py:103-115) on the current stream; ``feats`` are
        the age, sex, month, day and dow indices."""
        dev = table.device
        if self._winner is None or self._winner.device != dev or self._winner.numel() != self.n_user:
            self._winner = torch.full((self.n_user,), -1, dtype=torch.int32, device=dev)
        tabs = [self.age_emb.weight, self.sex_emb.weight, self.month_emb.weight, self.day_emb.weight, self.dow_emb.weight]
        feats = [_index(t, dev) for t in feats]
        _lib.check(_lib.load().ngcf_feature_mix(table.data_ptr(), self.n_user, self.emb_size, _lib.ptr_array(tabs),
                                                _lib.int_array(self.feat_widths), _lib.ptr_array(feats),
                                                u_id.data_ptr(), u_id.numel(), float(self.emb_ratio),
                                                self._winner.data_ptr(), _lib.current_stream()), "feature_mix")
        self._mix_count += 1

    def _draw_seed(self, st: _Ctx, mess_dropout: bool = False, noise: bool = False):
        """The forward's RNG key from torch's CPU generator (reproducible under torch.manual_seed), drawn only when a
        device-RNG stream is live (dropout, hard negatives, XSimGCL's layer noise) and only after the rng="reference"
        mask draws, whose RNG stream it must not shift.  The hard-negative draws take the same key: with dropout on, a
        forward with HardNegatives and one without draw the same key from the generator and so the same dropout masks."""
        need = st.drop_p > 0 or mess_dropout or noise or st.hneg is not None
        if not need:
            st.seed = 0
        elif self.rng == "reference":
            if self._seed_gen is None:
                self._seed_gen = torch.Generator().manual_seed(torch.initial_seed() & (2 ** 63 - 1))
            st.seed = draw_seed(self._seed_gen)
        else:
            st.seed = draw_seed()
        # CUDA-graph mode (graph.GraphedStep): the launches are frozen, so the per-step key comes from a device counter
        st.seed_dev = self._seed_dev if need else None

    def _finish(self, st: _Ctx, outs):
        """Keeps the forward's state for the backward and all_users_emb; returns the (users, positives, negatives)
        rows, negatives ``torch.empty(0)`` when the batch has none (NGCF.py:153)."""
        self._last, self._all_E = st, None
        return outs[0], outs[1], (outs[2] if len(outs) > 2 else torch.empty(0))

    # ---- attributes the reference sets in forward (NGCF.py:147-149), materialised on first read ---------
    @_lib.on_device
    def _materialize(self):
        if self._last is None:
            raise AttributeError("all_users_emb / all_items_emb exist after the first forward")
        if self._all_E is None:
            self._check_fresh(self._last, "all_users_emb / all_items_emb")
            self._all_E = self._readout(self._last)
        return self._all_E

    @property
    def all_users_emb(self):
        return self._materialize()[:self.n_user, :]

    @property
    def all_items_emb(self):
        return self._materialize()[self.n_user:, :]

    def _packed_table(self) -> torch.Tensor:
        """[N, d] view over user_embedding.weight and item_embedding.weight laid out back to back, so that
        ``cat(user, item)`` (NGCF.py:120) costs nothing.  Re-packs (and rebinds both ``.data``) whenever the
        two parameters are not adjacent, e.g. after ``model.to(device)`` or ``load_state_dict``."""
        u, i = self.user_embedding.weight, self.item_embedding.weight
        d = self.emb_size
        adjacent = (u.is_contiguous() and i.is_contiguous() and u.dtype == torch.float32 and
                    u.data_ptr() + self.n_user * d * 4 == i.data_ptr() and
                    getattr(self, "_table", None) is not None and self._table.data_ptr() == u.data_ptr())
        if not adjacent:
            n_rows = self._shard.N_pad if self._shard is not None else self.n_user + self.n_item
            table = torch.zeros(n_rows, d, dtype=torch.float32, device=u.device)   # rows past N: shard padding
            table[:self.n_user].copy_(u.data)
            table[self.n_user:self.n_user + self.n_item].copy_(i.data)
            u.data = table[:self.n_user]
            i.data = table[self.n_user:self.n_user + self.n_item]
            self._table = table
        return self._table if self._shard is None else self._table   # [N_pad, d] when sharded (pad rows are zero)

    def _slot_map(self, N, dev):
        if self._slot is None or self._slot.device != dev or self._slot.numel() != N:
            self._slot = torch.full((N,), -1, dtype=torch.int32, device=dev)
        return self._slot

    def _plan(self, year_idx: int, dev) -> LaplacianPlan:
        L = self.lap_list[year_idx]
        p = self._plans.get(year_idx)
        if p is None or p.src is not L or p.coo_val.device != dev:
            p = LaplacianPlan(L, dev, shard=self._shard)
            self._plans[year_idx] = p
        N = self.n_user + self.n_item
        if p.N != N:
            raise ValueError(f"{self._NAME}: the Laplacian is {p.N}x{p.N} but n_user + n_item = {N}")
        return p

    def _fresh_key(self):
        return (self._mix_count, _lib.param_epoch(), self.user_embedding.weight._version,
                self.item_embedding.weight._version)

    def _check_fresh(self, st, what: str):
        """E_0 of a forward is the live table (see __init__): refuse to use it once something changed the table."""
        if self._snapshot or st.fresh_key == self._fresh_key():
            return
        why = "the step that produced it also ran the optimizer" if st.fresh_key is None else \
            "another forward (feature mix) or an optimizer step ran since"
        raise RuntimeError(f"{self._NAME} (B200): {what} needs the embedding table as the forward left it, but {why}. "
                           + self._STALE_ADVICE)


class NGCF(_TableModel):
    """Same surface as the reference ``NGCF`` (NGCF.py:8-17).  Extra keyword-only knobs:

    rng : "device" (default) draws node- and message-dropout decisions in-kernel from a counter-based hash stream keyed
          on a per-forward seed taken from torch's CPU generator;  "reference" reproduces the reference's host
          float64 ``nn.Dropout`` node mask bit for bit (NGCF.py:94) at its host cost.
    snapshot : False (default) keeps E_0 = the live parameter table (zero copy); a second forward or an optimizer step
          before ``backward()`` / before reading ``all_users_emb`` then raises.  True copies the table per forward, which
          is what the reference's ``torch.cat`` (NGCF.py:120) does, and lifts that restriction.

    ``forward(..., neg_item=HardNegatives(...), ...)`` chooses each row's negative on the device from that forward's
    own layer outputs (sampler.HardNegatives); the picks are then ``neg_item.chosen``.
    """
    _NAME = "NGCF"
    _STALE_ADVICE = ("Run the forward again, or construct the module with snapshot=True to keep a per-forward copy like "
                     "the reference's torch.cat (NGCF.py:120).")

    def __init__(self, embed_size: int, layer_size: list, node_dropout: float, mess_dropout: list,
                 emb_ratio: float, lap_list: list, num_dict: dict, batch_size: int, device, *, rng: str = "device",
                 snapshot: bool = False):
        super().__init__()
        if rng not in ("device", "reference"):
            raise ValueError("rng must be 'device' or 'reference'")
        self.n_user = int(num_dict['user'])
        self.n_item = int(num_dict['item'])
        self.emb_size = int(embed_size)
        self.weight_size = list(layer_size)
        self.n_layer = len(self.weight_size)
        self.batch_size = batch_size
        self.device = device
        self.node_dropout = node_dropout
        self.mess_dropout = mess_dropout
        self.emb_ratio = emb_ratio
        self.rng = rng
        if max([self.emb_size] + self.weight_size) > 128 or self.n_layer > 8:
            raise ValueError("embedding/layer widths up to 128 and up to 8 layers are supported")

        self._feature_tables(num_dict)
        self.item_embedding = nn.Embedding(self.n_item, self.emb_size)
        self.user_embedding = nn.Embedding(self.n_user, self.emb_size)
        self.lap_list = lap_list
        self.set_layers()
        self._mess_bits = os.environ.get("NGCF_B200_MESS_BITS", "0") == "1"   # precompute message-dropout bits per step
        self._node_mode = "compact"   # device-RNG node dropout: "compact" (survivors only), "bits", or "inkernel"
        # E_0 of a forward is the LIVE packed table, not a copy (the reference's torch.cat at NGCF.py:120 copies 2 x 18 MB
        # per step at Gowalla shape).  A later forward (its feature mix rewrites user rows) or an optimizer step changes it
        # under a pending backward / under all_users_emb: that is detected and refused (_check_fresh).  snapshot=True (or
        # NGCF_B200_SNAPSHOT=1) copies the table per forward instead and lifts the restriction.
        self._snapshot = bool(snapshot) or os.environ.get("NGCF_B200_SNAPSHOT", "0") == "1"
        self._seed_gen = None    # rng="reference": private generator for the device-RNG key (message dropout), so the
                                 # CPU generator is consumed by the node masks only, exactly like the reference's stream
        self._group = None
        self._xchg = None        # sharded.PeerExchange (peer-memory exchange) when available
        self._side_stream = None     # weight gradients beside the transposed product (_Propagate.backward)
        self._side_stream3 = None    # feature mix beside the node-dropout compaction (forward)
        self._trace = None       # debugging aid: set to a list to record the backward's per-layer tensors
        self._inject = None      # tests only: dict(edge_keep=[K x uint8[nnz]], mess_mult=[K x [N,d]])

    def set_layers(self):
        """Same initialisation calls in the same order as NGCF.py:56-91 (same RNG stream, same values)."""
        init = nn.init.kaiming_uniform_
        init(self.user_embedding.weight)
        init(self.item_embedding.weight)
        init(self.age_emb.weight)
        init(self.sex_emb.weight)
        init(self.month_emb.weight)
        init(self.dow_emb.weight)
        init(self.day_emb.weight)
        sizes = [self.emb_size] + self.weight_size
        w1, w2, nd, md = [], [], [], []
        for k in range(self.n_layer):
            w1.append(nn.Linear(sizes[k], sizes[k + 1], bias=True))
            w2.append(nn.Linear(sizes[k], sizes[k + 1], bias=True))
            if self.node_dropout is not None:
                nd.append(nn.Dropout(p=self.node_dropout))
            if self.mess_dropout is not None:
                md.append(nn.Dropout(p=self.mess_dropout[k]))
        self.w1_list = nn.Sequential(*w1)
        self.w2_list = nn.Sequential(*w2)
        self.node_dropout_list = nn.Sequential(*nd)
        self.mess_dropout_list = nn.Sequential(*md)

    # ---- multi-GPU ------------------------------------------------------------------------------------
    def shard(self, group=None, shards=None):
        """Row-partitions the propagation over the ranks of ``group`` (default process group): this rank then
        computes its contiguous block of rows of every layer (equal blocks, or ``shards`` = a sharded.BalancedShards
        cut by work).  Parameters stay replicated; every
        rank must call forward with the same batch and the same torch CPU RNG state (the per-step RNG key is drawn
        from it).  Explicit-mask node dropout (rng="reference") is not available in this mode."""
        if not dist.is_initialized():
            raise RuntimeError("NGCF.shard() needs an initialised torch.distributed process group")
        if self.rng != "device":
            raise ValueError("row-sharded runs need rng='device' (masks are keyed on global coordinates in-kernel)")
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        self._shard = shards if shards is not None else RowShards(self.n_user + self.n_item, world, rank)
        if self._shard.N != self.n_user + self.n_item or self._shard.world != world or self._shard.rank != rank:
            raise ValueError("the shard descriptor does not match this model / process group")
        self._group = group
        self._plans, self._table, self._slot = {}, None, None
        # per-layer exchange: peer-memory stores (sharded.PeerExchange) when symmetric memory is available on this box,
        # NCCL all-gathers otherwise (NGCF_B200_EXCHANGE=nccl forces them: A/B timing)
        self._xchg = None
        if world > 1 and os.environ.get("NGCF_B200_EXCHANGE", "peer") != "nccl":
            try:
                from .sharded import PeerExchange
                self._xchg = PeerExchange(group, self.user_embedding.weight.device)
            except Exception as e:                                     # no symmetric memory / no peer access
                self._xchg_error = f"{type(e).__name__}: {e}"
                ok = torch.tensor([0], device=self.user_embedding.weight.device)
            else:
                ok = torch.tensor([1], device=self.user_embedding.weight.device)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)    # all ranks or none
            if int(ok) == 0:
                self._xchg = None
        if self._xchg is None and world > 1 and not getattr(self._shard, "equal", True):
            raise RuntimeError("unequal row blocks (BalancedShards) need the peer-memory exchange, which is not available "
                               "here: " + getattr(self, "_xchg_error", "disabled by NGCF_B200_EXCHANGE=nccl"))
        return self

    def exchange_description(self) -> str:
        if self._shard is None:
            return "single GPU"
        if self._xchg is not None:
            how = "NVLS multicast stores (multimem.st)" if self._xchg.multicast() else "peer-memory stores"
            return (f"contiguous row blocks; per-layer exchange of E / gS / table-gradient rows by {how} over NVLink "
                    "(ngcf_push_rows on symmetric memory, no NCCL collective anywhere in the step; the last layer's "
                    "output travels for the batch rows only; W/b gradients: one more push + a rank-ordered sum)")
        return "equal row blocks, per-layer NCCL all-gather of E / gS, all-reduce of W/b grads"

    # ---- internal buffers ---------------------------------------------------------------------------
    def _reference_node_masks(self, nnz: int, dev):
        """Bit-exact reproduction of NGCF.sparse_dropout's host RNG stream (NGCF.py:94): float64 ones through a
        fresh (always-training) nn.Dropout on the CPU generator, over the surviving entries only."""
        alive = np.arange(nnz)
        out = []
        for _ in range(self.n_layer):
            m = nn.Dropout(self.node_dropout)(torch.tensor(np.ones(alive.size))).type(torch.bool).numpy()
            alive = alive[m]
            full = np.zeros(nnz, dtype=np.uint8)
            full[alive] = 1
            out.append(torch.from_numpy(full).to(dev))
        return out

    # ---- forward ---------------------------------------------------------------------------------------
    @_lib.on_device
    def forward(self, year, u_id, age, sex, month, day, dow, pos_item, neg_item, node_flag):
        dev = self._cuda_device()
        K = self.n_layer
        if (self._side_stream is None or self._side_stream.device != dev) and not _capturing():
            # second streams of the capture-time overlaps, handed out of torch's pool BEFORE any capture begins
            self._side_stream, self._side_stream3 = (torch.cuda.Stream(device=dev) for _ in range(2))
        st = self._batch(dev, u_id, pos_item, neg_item)
        year_idx = int(year.min()) % 18                                      # == year.unique()[0] % 18, NGCF.py:117

        table = self._packed_table()
        feats = (age, sex, month, day, dow)                                  # concat order, NGCF.py:110
        # the feature mix (two small launches that rewrite <= B user rows) on a second stream beside the node-dropout
        # compaction, which does not touch the table; joined before the first product (0.502 -> 0.499 ms per step)
        st.fm_stream = None
        if self._shard is None and _capturing() and bool(node_flag) and \
                (self.node_dropout or 0) > 0 and self.rng == "device":
            main = torch.cuda.current_stream()
            if self._side_stream3 is None:
                self._side_stream3 = torch.cuda.Stream(device=dev)
            self._side_stream3.wait_stream(main)
            with torch.cuda.stream(self._side_stream3):
                self._feature_mix(table, st.rows[0], feats)
            st.fm_stream = self._side_stream3
        else:
            self._feature_mix(table, st.rows[0], feats)

        st.fresh_key = self._fresh_key()
        st.plan = plan = self._plan(year_idx, dev)
        if self._shard is not None and "edge_keep" in (self._inject or {}):
            raise ValueError("explicit edge masks are not supported in row-sharded mode")
        st.dims = [self.emb_size] + self.weight_size
        inj = self._inject or {}
        # node dropout: active whenever node_flag is set, in eval mode too (NGCF.py:124-126)
        masked = bool(node_flag) and (self.node_dropout is not None) and (self.node_dropout > 0 or "edge_keep" in inj)
        st.vals_f = st.vals_b = None
        st.drop_p = 0.0
        masks = None
        if masked:
            if "edge_keep" in inj:
                masks = [m.to(device=dev, dtype=torch.uint8).contiguous() for m in inj["edge_keep"]]
            elif self.rng == "reference":
                masks = self._reference_node_masks(plan.nnz, dev)
            else:
                st.drop_p = float(self.node_dropout)               # decided in-kernel, no mask pass
        # message dropout: nn.Dropout semantics, only in training mode (NGCF.py:142)
        st.mess_mult = None
        st.mess_p = [0.0] * K
        if "mess_mult" in inj:
            st.mess_mult = [m.to(device=dev, dtype=torch.float32).contiguous() for m in inj["mess_mult"]]
        elif self.training and self.mess_dropout is not None:
            st.mess_p = [float(p) for p in self.mess_dropout[:K]]
        self._draw_seed(st, mess_dropout=any(p > 0 for p in st.mess_p))
        if masks is not None:
            st.vals_f = [plan.entries(plan.fwd, masks[k]) for k in range(K)]
            st.vals_b = [plan.entries(plan.bwd, masks[k]) for k in range(K)]

        wb = [l.weight for l in self.w1_list] + [l.bias for l in self.w1_list] + \
             [l.weight for l in self.w2_list] + [l.bias for l in self.w2_list]
        outs = _Propagate.apply(self, st, len(st.rows), self.user_embedding.weight, self.item_embedding.weight, *wb)
        return self._finish(st, outs)

    def _readout(self, st: _Ctx) -> torch.Tensor:
        """[N, sum(dims)]: the concatenated layer outputs of every row (NGCF.py:144-149)."""
        if st.last_partial is not None:                       # row-sharded: the last layer travelled for the batch
            sh = self._shard                                   # rows only; complete it now (COLLECTIVE: every rank
            self._xchg.push(st.last_partial, sh.r0, sh.rows)   # must read the attribute)
            st.last_partial = None
        N, D = self.n_user + self.n_item, sum(st.dims)
        out = torch.empty(N, D, dtype=torch.float32, device=st.E[0].device)
        _lib.check(_lib.load().ngcf_gather_concat(_lib.ptr_array(st.E), _lib.int_array(st.dims), self.n_layer + 1, None,
                                                  0, N, out.data_ptr(), D, _lib.current_stream()), "gather_concat")
        return out
