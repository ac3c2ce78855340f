"""``LightGCN`` (He et al., SIGIR 2020) over the B200 kernels: NGCF's propagation without its dense transforms,
nonlinearity and normalisation.

    E_{k+1} = L_k · E_k           (L_k: lap_list[year] with layer k's node-dropout survivors)
    final row = (E_0 + E_1 + ... + E_K) / (K + 1)

The products are ``ngcf_spmm`` (the kernel NGCF propagates with), the readout is ``ngcf_layer_mean``.  The backward reads
no activations: the model is linear in E_0, and the readout hands every layer the same row gradient G / (K + 1), so

    gE_K = G / (K + 1),    gE_k = L_k^T · gE_{k+1} + G / (K + 1)    (k = K-1 .. 0)

and gE_0 is the table gradient.  G is the batch's row gradients summed per distinct row (``ngcf_rowgrad_scatter``'s slot
map); ``ngcf_rowgrad_expand`` writes the dense G / (K + 1) and each transposed product adds the sparse rows through
``ngcf_spmm``'s slot/gsum addend.  Same ``forward`` signature and outputs as ``NGCF``, so ``BPR``, ``SoftmaxLoss``,
``HardNegatives``, ``GraphedStep``, ``Adam``, ``Experiment`` and ``full_rank_eval`` take either model."""
from __future__ import annotations

import torch
import torch.nn as nn

from . import _lib
from .NGCF import _Ctx, _RowGrads, _TableModel
from .plan import NodeDropout, node_dropout_mode, spmm

MAX_LAYERS = 8          # NGCF_MAX_LAYERS
MAX_WIDTH = 128         # NGCF_MAX_WIDTH


class _LightPropagate(torch.autograd.Function):
    """K products + layer-mean readout of the batch's row sets, and the activation-free backward (module docstring)."""

    @staticmethod
    def forward(ctx, mod, st: _Ctx, n_sets, user_w, item_w):
        lib = _lib.load()
        K, d = mod.n_layer, mod.emb_size
        side = st.plan.fwd
        st.E = [mod._packed_table()]                                   # E_0: the live table, no copy
        st.dropout = NodeDropout(st.plan, mod._node_mode, st.drop_p, st.seed, st.seed_dev, K, 0, [d])
        for k in range(K):
            st.E.append(spmm(side, None, st.E[k], d, **st.dropout.args(k)))
        layers = _lib.ptr_array(st.E)
        if st.hneg is not None:                                        # dynamic hard negatives: fills st.rows[2]
            hn, train, chosen, cand, score = st.hneg
            _lib.check(lib.ngcf_hard_negatives_mean(layers, d, K + 1, mod.n_user, st.rows[0].data_ptr(),
                                                    st.rows[0].numel(), train.ptr.data_ptr(), _lib.ptr(train.idx),
                                                    mod.n_item, hn.n_candidates, int(hn.signed), st.seed,
                                                    _lib.ptr(st.seed_dev), chosen.data_ptr(), _lib.ptr(cand),
                                                    _lib.ptr(score), _lib.current_stream()), "hard_negatives_mean")
        outs = [torch.empty(st.rows[j].numel(), d, dtype=torch.float32, device=user_w.device) for j in range(n_sets)]
        _lib.check(lib.ngcf_layer_mean_sets(layers, K + 1, d, _lib.ptr_array(st.rows[:n_sets]),
                                            _lib.i64_array(st.offsets[:n_sets]),
                                            _lib.i64_array([r.numel() for r in st.rows[:n_sets]]), _lib.ptr_array(outs),
                                            n_sets, d, _lib.current_stream()), "layer_mean_sets")
        ctx.st, ctx.mod, ctx.n_sets = st, mod, n_sets
        return tuple(outs)

    @staticmethod
    def backward(ctx, *gouts):
        lib = _lib.load()
        st, mod, n_sets = ctx.st, ctx.mod, ctx.n_sets
        K, d = mod.n_layer, mod.emb_size
        N = mod.n_user + mod.n_item
        dev = st.E[0].device
        rg = _RowGrads(mod, st, gouts, n_sets, d, N)
        gE = torch.empty(N, d, dtype=torch.float32, device=dev)       # gE_K = G / (K+1); gsum scaled with it
        _lib.check(lib.ngcf_rowgrad_expand(rg.slot.data_ptr(), N, rg.gsum.data_ptr(), d, d, 1.0 / (K + 1), gE.data_ptr(),
                                           d, _lib.current_stream()), "rowgrad_expand")
        side = st.plan.side(True, False)
        st.dropout.draw_transposed()
        for k in range(K - 1, -1, -1):                                 # gE_k = L_k^T gE_{k+1} + G / (K+1)
            gE = spmm(side, None, gE, d, slot=rg.slot, gsum=rg.gsum, **st.dropout.args(k, transposed=True))
        rg.reset()
        return None, None, None, gE[:mod.n_user], gE[mod.n_user:]


class LightGCN(_TableModel):
    """``LightGCN(embed_size, n_layers, lap_list, num_dict, node_dropout=0.0, emb_ratio=0.0)``.

    ``forward(year, u_id, age, sex, month, day, dow, pos_item, neg_item, node_flag)`` has NGCF's signature and returns
    the layer-mean rows of the batch's users, positives and negatives, each [B, embed_size] (negatives: ``torch.empty(0)``
    when ``neg_item`` is empty).  ``neg_item`` may be a ``HardNegatives``; ``year`` picks ``lap_list[year.min() % 18]``.
    ``all_users_emb`` / ``all_items_emb`` are the layer mean over all rows of the last forward, built on first read.

    node_dropout : with ``node_flag`` set, layer k propagates over the entries of L that survive layers 0..k of the
          device-RNG draws NGCF uses (entries deleted, values not rescaled).  There is no message dropout.
    emb_ratio : > 0 registers the five feature tables (age, sex, month, day, dow) and runs NGCF's feature mix on the
          batch users' rows before propagating, so the project's Seoul data and ``TourDataset`` batches work unchanged;
          0 (default) ignores those index arguments.

    Every table is initialised with normal_(std=0.1), as in LightGCN's reference code.  E_0 is the live table, as in
    NGCF: reading ``all_users_emb`` after an optimizer step or another forward raises."""
    _NAME = "LightGCN"
    rng = "device"

    def __init__(self, embed_size: int, n_layers: int, lap_list: list, num_dict: dict, *, node_dropout: float = 0.0,
                 emb_ratio: float = 0.0):
        super().__init__()
        self.emb_size, self.n_layer = int(embed_size), int(n_layers)
        if not 1 <= self.n_layer <= MAX_LAYERS:
            raise ValueError(f"LightGCN: n_layers {self.n_layer} not in [1, {MAX_LAYERS}]")
        if not 1 <= self.emb_size <= MAX_WIDTH:
            raise ValueError(f"LightGCN: embed_size {self.emb_size} not in [1, {MAX_WIDTH}]")
        self.node_dropout, self.emb_ratio = float(node_dropout), float(emb_ratio)
        if not 0.0 <= self.node_dropout < 1.0:
            raise ValueError(f"LightGCN: node_dropout {self.node_dropout} not in [0, 1)")
        if not 0.0 <= self.emb_ratio <= 1.0:
            raise ValueError(f"LightGCN: emb_ratio {self.emb_ratio} not in [0, 1]")
        self.n_user, self.n_item = int(num_dict["user"]), int(num_dict["item"])
        if self.n_user < 1 or self.n_item < 1:
            raise ValueError(f"LightGCN: {self.n_user} users and {self.n_item} items")
        N = self.n_user + self.n_item
        lap_list = list(lap_list)
        if not lap_list:
            raise ValueError("LightGCN: lap_list is empty")
        for j, L in enumerate(lap_list):
            if tuple(L.shape) != (N, N):
                raise ValueError(f"LightGCN: lap_list[{j}] is {tuple(L.shape)}, but n_user + n_item = {N}")
        self.lap_list = lap_list
        if self.emb_ratio > 0:                    # NGCF's feature tables, in its registration order and widths
            self._feature_tables(num_dict)
        self.user_embedding = nn.Embedding(self.n_user, self.emb_size)
        self.item_embedding = nn.Embedding(self.n_item, self.emb_size)
        for e in self.modules():
            if isinstance(e, nn.Embedding):
                nn.init.normal_(e.weight, std=0.1)
        self._node_mode = node_dropout_mode("compact", [self.emb_size])   # or "bits" / "inkernel" (plan.NodeDropout)

    def shard(self, group=None, shards=None):
        raise NotImplementedError("LightGCN: row-sharded runs are not supported; use NGCF.shard() for those")

    @_lib.on_device
    def forward(self, year, u_id, age, sex, month, day, dow, pos_item, neg_item, node_flag):
        dev = self._cuda_device()
        st = self._batch(dev, u_id, pos_item, neg_item)
        year_idx = int(year.min()) % 18
        table = self._packed_table()
        if self.emb_ratio > 0:                                         # NGCF's feature mix of the batch users' rows
            self._feature_mix(table, st.rows[0], (age, sex, month, day, dow))
        st.fresh_key = self._fresh_key()
        st.plan = self._plan(year_idx, dev)
        st.drop_p = self.node_dropout if bool(node_flag) and self.node_dropout > 0 else 0.0
        self._draw_seed(st)
        outs = _LightPropagate.apply(self, st, len(st.rows), self.user_embedding.weight, self.item_embedding.weight)
        return self._finish(st, outs)

    def _readout(self, st: _Ctx) -> torch.Tensor:
        """[N, embed_size]: the layer mean of every row."""
        N = self.n_user + self.n_item
        out = torch.empty(N, self.emb_size, dtype=torch.float32, device=st.E[0].device)
        _lib.check(_lib.load().ngcf_layer_mean(_lib.ptr_array(st.E), self.n_layer + 1, self.emb_size, None, 0, N,
                                               out.data_ptr(), self.emb_size, _lib.current_stream()), "layer_mean")
        return out
