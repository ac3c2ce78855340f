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
from .NGCF import _TableModel, draw_seed
from .plan import node_dropout_bits, node_dropout_compact, spmm
from .sampler import HardNegatives

MAX_LAYERS = 8          # NGCF_MAX_LAYERS
MAX_WIDTH = 128         # NGCF_MAX_WIDTH


def _stream() -> int:
    return _lib.current_stream()


class _Ctx:
    """Per-forward state shared by the autograd node and the module (what ``GraphedStep`` reads is rows, hneg,
    fresh_key)."""
    __slots__ = ("plan", "E", "seed", "seed_dev", "drop_p", "node_mode", "comp_f", "comp_b", "bits_f", "bits_b",
                 "rows", "offsets", "fresh_key", "hneg")


class _LightPropagate(torch.autograd.Function):
    """K products + layer-mean readout of the batch's row sets, and the activation-free backward (module docstring)."""

    @staticmethod
    def forward(ctx, mod, st: _Ctx, n_sets, user_w, item_w):
        lib = _lib.load()
        K, d = mod.n_layer, mod.emb_size
        side = st.plan.fwd
        st.E = [mod._packed_table()]                                   # E_0: the live table, no copy
        st.comp_f = st.comp_b = st.bits_f = st.bits_b = None
        if st.drop_p > 0:
            # this step's decisions for all K layers in one pass; a symmetric L serves L^T from the same pass
            shared = st.plan.side(True, False) is side
            if st.node_mode == "compact":
                st.comp_f, ct = node_dropout_compact(side, st.drop_p, st.seed, st.seed_dev, K, as_L=True, as_Lt=shared)
                st.comp_b = ct if shared else None
            else:
                st.bits_f, bt = node_dropout_bits(side, st.drop_p, st.seed, st.seed_dev, K, as_L=True, as_Lt=shared)
                st.bits_b = bt if shared else None
        for k in range(K):
            st.E.append(spmm(side, None, st.E[k], d, drop_p=st.drop_p, seed=st.seed, seed_dev=st.seed_dev, layer=k,
                             keep_bits=st.bits_f, compact=st.comp_f[k] if st.comp_f is not None else None))
        layers = _lib.ptr_array(st.E)
        if st.hneg is not None:                                        # dynamic hard negatives: fills st.rows[2]
            hn, train, chosen, cand, score = st.hneg
            _lib.check(lib.ngcf_hard_negatives_mean(layers, d, K + 1, mod.n_user, st.rows[0].data_ptr(),
                                                    st.rows[0].numel(), train.ptr.data_ptr(), _lib.ptr(train.idx),
                                                    mod.n_item, hn.n_candidates, int(hn.signed), st.seed,
                                                    _lib.ptr(st.seed_dev), chosen.data_ptr(), _lib.ptr(cand),
                                                    _lib.ptr(score), _stream()), "hard_negatives_mean")
        outs = [torch.empty(st.rows[j].numel(), d, dtype=torch.float32, device=user_w.device) for j in range(n_sets)]
        _lib.check(lib.ngcf_layer_mean_sets(layers, K + 1, d, _lib.ptr_array(st.rows[:n_sets]),
                                            _lib.i64_array(st.offsets[:n_sets]),
                                            _lib.i64_array([r.numel() for r in st.rows[:n_sets]]), _lib.ptr_array(outs),
                                            n_sets, d, _stream()), "layer_mean_sets")
        ctx.st, ctx.mod, ctx.n_sets = st, mod, n_sets
        return tuple(outs)

    @staticmethod
    def backward(ctx, *gouts):
        lib = _lib.load()
        st, mod, n_sets = ctx.st, ctx.mod, ctx.n_sets
        K, d = mod.n_layer, mod.emb_size
        N = mod.n_user + mod.n_item
        dev = st.E[0].device
        g = [(go.contiguous() if go is not None else torch.zeros(st.rows[j].numel(), d, device=dev))
             for j, go in enumerate(gouts)]
        batch = [r.numel() for r in st.rows[:n_sets]]
        rows_h, offs_h, batch_h = _lib.ptr_array(st.rows[:n_sets]), _lib.i64_array(st.offsets[:n_sets]), \
            _lib.i64_array(batch)
        slot = mod._slot_map(N, dev)
        gsum = torch.empty(max(sum(batch), 1), d, dtype=torch.float32, device=dev)
        _lib.check(lib.ngcf_rowgrad_scatter(rows_h, offs_h, _lib.ptr_array(g), batch_h, n_sets, d, slot.data_ptr(),
                                            gsum.data_ptr(), _stream()), "rowgrad_scatter")
        gE = torch.empty(N, d, dtype=torch.float32, device=dev)       # gE_K = G / (K+1); gsum scaled with it
        _lib.check(lib.ngcf_rowgrad_expand(slot.data_ptr(), N, gsum.data_ptr(), d, d, 1.0 / (K + 1), gE.data_ptr(), d,
                                           _stream()), "rowgrad_expand")
        side = st.plan.side(True, False)
        if st.drop_p > 0 and st.node_mode == "compact" and st.comp_b is None:
            _, st.comp_b = node_dropout_compact(side, st.drop_p, st.seed, st.seed_dev, K, as_L=False, as_Lt=True)
        if st.drop_p > 0 and st.node_mode == "bits" and st.bits_b is None:
            _, st.bits_b = node_dropout_bits(side, st.drop_p, st.seed, st.seed_dev, K, as_L=False, as_Lt=True)
        for k in range(K - 1, -1, -1):                                 # gE_k = L_k^T gE_{k+1} + G / (K+1)
            gE = spmm(side, None, gE, d, slot=slot, gsum=gsum, drop_p=st.drop_p, seed=st.seed, seed_dev=st.seed_dev,
                      layer=k, transposed=True, keep_bits=st.bits_b,
                      compact=st.comp_b[k] if st.comp_b is not None else None)
        _lib.check(lib.ngcf_rowgrad_reset(rows_h, offs_h, batch_h, n_sets, slot.data_ptr(), _stream()), "rowgrad_reset")
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
            w = self.emb_size // 5
            self.feat_widths = [w, w, w, w, self.emb_size - 4 * w]          # age, sex, month, day, dow
            self.month_emb = nn.Embedding(int(num_dict["month"]), w)
            self.day_emb = nn.Embedding(int(num_dict["day"]), w)
            self.sex_emb = nn.Embedding(int(num_dict["sex"]), w)
            self.age_emb = nn.Embedding(int(num_dict["age"]), w)
            self.dow_emb = nn.Embedding(int(num_dict["dayofweek"]), self.feat_widths[4])
        self.user_embedding = nn.Embedding(self.n_user, self.emb_size)
        self.item_embedding = nn.Embedding(self.n_item, self.emb_size)
        for e in self.modules():
            if isinstance(e, nn.Embedding):
                nn.init.normal_(e.weight, std=0.1)
        # survivor lists feed the streaming SpMM (widths that are multiples of 4); other widths take decision bytes
        self._node_mode = "compact" if self.emb_size % 4 == 0 else "bits"
        self._plans, self._table, self._slot, self._winner = {}, None, None, None
        self._shard = None
        self._snapshot = False
        self._mix_count = 0
        self._seed_dev = None    # device uint64 added to the RNG key (set by graph.GraphedStep)
        self._last = None
        self._all_E = None

    def shard(self, group=None, shards=None):
        raise NotImplementedError("LightGCN: row-sharded runs are not supported; use NGCF.shard() for those")

    @_lib.on_device
    def forward(self, year, u_id, age, sex, month, day, dow, pos_item, neg_item, node_flag):
        lib = _lib.load()
        dev = self.user_embedding.weight.device
        if dev.type != "cuda":
            raise RuntimeError("LightGCN (B200) runs on a CUDA device only; there is no CPU fallback. "
                               "Move the module with .to('cuda').")
        N = self.n_user + self.n_item

        def ix(t):
            return t.to(device=dev, dtype=torch.int64).contiguous()

        u_id, pos_item = ix(u_id), ix(pos_item)
        hneg = neg_item if isinstance(neg_item, HardNegatives) else None
        if hneg is not None:
            if hneg.train.n_rows != self.n_user or hneg.train.n_items != self.n_item:
                raise ValueError(f"HardNegatives: train has {hneg.train.n_rows} rows over {hneg.train.n_items} items; "
                                 f"the model has {self.n_user} users and {self.n_item} items")
            has_neg = True
            neg_item = torch.empty(u_id.numel(), dtype=torch.int64, device=dev)   # written by the kernel
        else:
            has_neg = len(neg_item) > 0
            neg_item = ix(neg_item) if has_neg else None
        year_idx = int(year.min()) % 18

        table = self._packed_table()
        if self.emb_ratio > 0:                                         # NGCF's feature mix of the batch users' rows
            if self._winner is None or self._winner.device != dev:
                self._winner = torch.full((self.n_user,), -1, dtype=torch.int32, device=dev)
            tabs = [self.age_emb.weight, self.sex_emb.weight, self.month_emb.weight, self.day_emb.weight,
                    self.dow_emb.weight]
            feats = [ix(age), ix(sex), ix(month), ix(day), ix(dow)]
            _lib.check(lib.ngcf_feature_mix(table.data_ptr(), self.n_user, self.emb_size, _lib.ptr_array(tabs),
                                            _lib.int_array(self.feat_widths), _lib.ptr_array(feats), u_id.data_ptr(),
                                            u_id.numel(), self.emb_ratio, self._winner.data_ptr(), _stream()),
                       "feature_mix")
            self._mix_count += 1

        st = _Ctx()
        st.fresh_key = self._fresh_key()
        st.plan = self._plan(year_idx, dev)
        if st.plan.N != N:
            raise ValueError(f"LightGCN: the Laplacian is {st.plan.N}x{st.plan.N} but n_user + n_item = {N}")
        st.drop_p = self.node_dropout if bool(node_flag) and self.node_dropout > 0 else 0.0
        st.node_mode = self._node_mode
        need_seed = st.drop_p > 0 or hneg is not None
        st.seed = draw_seed() if need_seed else 0
        st.seed_dev = self._seed_dev if need_seed else None
        st.rows = [u_id, pos_item] + ([neg_item] if has_neg else [])
        st.offsets = [0, self.n_user] + ([self.n_user] if has_neg else [])
        st.hneg = None
        if hneg is not None:
            M = hneg.n_candidates
            st.hneg = (hneg, hneg._on(dev), neg_item,
                       torch.empty(u_id.numel(), M, dtype=torch.int64, device=dev) if hneg.debug else None,
                       torch.empty(u_id.numel(), M, dtype=torch.float32, device=dev) if hneg.debug else None)
            hneg.chosen, hneg.cand, hneg.score = st.hneg[2:]
        outs = _LightPropagate.apply(self, st, len(st.rows), self.user_embedding.weight, self.item_embedding.weight)
        self._last, self._all_E = st, None
        return outs[0], outs[1], (outs[2] if has_neg else torch.empty(0))

    @_lib.on_device
    def _materialize(self):
        if self._last is None:
            raise AttributeError("all_users_emb / all_items_emb exist after the first forward")
        if self._all_E is None:
            self._check_fresh(self._last, "all_users_emb / all_items_emb")
            st, lib = self._last, _lib.load()
            N = self.n_user + self.n_item
            out = torch.empty(N, self.emb_size, dtype=torch.float32, device=st.E[0].device)
            _lib.check(lib.ngcf_layer_mean(_lib.ptr_array(st.E), self.n_layer + 1, self.emb_size, None, 0, N,
                                           out.data_ptr(), self.emb_size, _stream()), "layer_mean")
            self._all_E = out
        return self._all_E

    @property
    def all_users_emb(self):
        return self._materialize()[:self.n_user, :]

    @property
    def all_items_emb(self):
        return self._materialize()[self.n_user:, :]
