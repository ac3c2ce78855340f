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
``HardNegatives``, ``GraphedStep``, ``Adam``, ``Experiment`` and ``full_rank_eval`` take either model.

``XSimGCL`` (Yu et al., TKDE 2023) runs the same propagation with ``ngcf_perturb_rows``' noise after each product, reads
out mean(E_1 .. E_K) (E_0 left out) and adds a cosine InfoNCE between that readout and one intermediate layer
(``ngcf_infonce``); see its docstring for the backward."""
from __future__ import annotations

import ctypes as C

import torch
import torch.nn as nn

from . import _lib
from .NGCF import _Ctx, _RowGrads, _TableModel
from .plan import NodeDropout, node_dropout_mode, spmm

MAX_LAYERS = 8          # NGCF_MAX_LAYERS
MAX_WIDTH = 128         # NGCF_MAX_WIDTH
MAX_INFONCE_BATCH = 4096   # ngcf_infonce


class _LightPropagate(torch.autograd.Function):
    """K products + layer-mean readout of the batch's row sets, and the activation-free backward (module docstring).

    first : the readout's first layer, 0 (LightGCN: mean of E_0..E_K) or 1 (XSimGCL: mean of E_1..E_K).
    eps : > 0 adds ngcf_perturb_rows' noise to every E_{k+1} after its product (0: off).
    cl_layer : > 0 also returns the view-2 rows, E_{cl_layer} of the batch's users and positives (two more outputs)."""

    @staticmethod
    def forward(ctx, mod, st: _Ctx, n_sets, first, eps, cl_layer, user_w, item_w):
        lib = _lib.load()
        K, d = mod.n_layer, mod.emb_size
        N = mod.n_user + mod.n_item
        side = st.plan.fwd
        st.E = [mod._packed_table()]                                   # E_0: the live table, no copy
        st.dropout = NodeDropout(st.plan, mod._node_mode, st.drop_p, st.seed, st.seed_dev, K, 0, [d])
        for k in range(K):
            st.E.append(spmm(side, None, st.E[k], d, **st.dropout.args(k)))
            if eps > 0:
                _lib.check(lib.ngcf_perturb_rows(st.E[k + 1].data_ptr(), N, d, d, float(eps), st.seed,
                                                 _lib.ptr(st.seed_dev), k + 1, _lib.current_stream()), "perturb_rows")
        n_read = K + 1 - first
        layers = _lib.ptr_array(st.E[first:])
        if st.hneg is not None:                                        # dynamic hard negatives: fills st.rows[2]
            hn, train, chosen, cand, score = st.hneg
            _lib.check(lib.ngcf_hard_negatives_mean(layers, d, n_read, mod.n_user, st.rows[0].data_ptr(),
                                                    st.rows[0].numel(), train.ptr.data_ptr(), _lib.ptr(train.idx),
                                                    mod.n_item, hn.n_candidates, int(hn.signed), st.seed,
                                                    _lib.ptr(st.seed_dev), chosen.data_ptr(), _lib.ptr(cand),
                                                    _lib.ptr(score), _lib.current_stream()), "hard_negatives_mean")
        outs = [torch.empty(st.rows[j].numel(), d, dtype=torch.float32, device=user_w.device) for j in range(n_sets)]
        _lib.check(lib.ngcf_layer_mean_sets(layers, n_read, d, _lib.ptr_array(st.rows[:n_sets]),
                                            _lib.i64_array(st.offsets[:n_sets]),
                                            _lib.i64_array([r.numel() for r in st.rows[:n_sets]]), _lib.ptr_array(outs),
                                            n_sets, d, _lib.current_stream()), "layer_mean_sets")
        if cl_layer:                                                   # view 2: E_cl of the users and positives
            view2 = [torch.empty(st.rows[j].numel(), d, dtype=torch.float32, device=user_w.device) for j in range(2)]
            _lib.check(lib.ngcf_layer_mean_sets(_lib.ptr_array([st.E[cl_layer]]), 1, d, _lib.ptr_array(st.rows[:2]),
                                                _lib.i64_array(st.offsets[:2]),
                                                _lib.i64_array([r.numel() for r in st.rows[:2]]),
                                                _lib.ptr_array(view2), 2, d, _lib.current_stream()), "layer_mean_sets")
            outs += view2
        ctx.st, ctx.mod, ctx.n_sets, ctx.first, ctx.cl_layer = st, mod, n_sets, first, cl_layer
        return tuple(outs)

    @staticmethod
    def backward(ctx, *gouts):
        lib = _lib.load()
        st, mod, n_sets, first, cl = ctx.st, ctx.mod, ctx.n_sets, ctx.first, ctx.cl_layer
        K, d = mod.n_layer, mod.emb_size
        N = mod.n_user + mod.n_item
        dev = st.E[0].device
        rg = _RowGrads(mod, st, gouts[:n_sets], n_sets, d, N)
        gE = torch.empty(N, d, dtype=torch.float32, device=dev)       # gE_K = G / n_read; gsum scaled with it
        _lib.check(lib.ngcf_rowgrad_expand(rg.slot.data_ptr(), N, rg.gsum.data_ptr(), d, d, 1.0 / (K + 1 - first),
                                           gE.data_ptr(), d, _lib.current_stream()), "rowgrad_expand")
        gsum_cl = rg.gsum
        H = gouts[n_sets:]
        if cl and any(h is not None for h in H):                       # + H at layer cl: on gE_K, or through a second
            H = [(h.contiguous() if h is not None else torch.zeros(st.rows[j].numel(), d, device=dev))   # gsum on the
                 for j, h in enumerate(H)]                                                                # same slots
            if cl == K:
                dst, slot, ld = gE, None, d
            else:
                gsum_cl = rg.gsum.clone()
                dst, slot, ld = gsum_cl, rg.slot.data_ptr(), d
            _lib.check(lib.ngcf_rowgrad_add(_lib.ptr_array(st.rows[:2]), _lib.i64_array(st.offsets[:2]), _lib.ptr_array(H),
                                            _lib.i64_array([h.shape[0] for h in H]), 2, d, slot, dst.data_ptr(), ld,
                                            _lib.current_stream()), "rowgrad_add")
        side = st.plan.side(True, False)
        st.dropout.draw_transposed()
        for k in range(K - 1, -1, -1):                  # gE_k = L_k^T gE_{k+1} + G / n_read (k >= first) + H (k == cl)
            addend = dict(slot=rg.slot, gsum=gsum_cl if k == cl else rg.gsum) if k >= first else {}
            gE = spmm(side, None, gE, d, **addend, **st.dropout.args(k, transposed=True))
        rg.reset()
        return None, None, None, None, None, None, gE[:mod.n_user], gE[mod.n_user:]


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
    _first = 0                                    # readout: mean of E_0 .. E_K

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
        st, outs = self._propagate(year, u_id, age, sex, month, day, dow, pos_item, neg_item, node_flag, 0.0, 0)
        return self._finish(st, outs)

    def _propagate(self, year, u_id, age, sex, month, day, dow, pos_item, neg_item, node_flag, eps, cl_layer):
        """The forward up to the readout: its _Ctx and _LightPropagate's outputs (with noise eps and view 2 at
        cl_layer, _LightPropagate's arguments)."""
        dev = self._cuda_device()
        st = self._batch(dev, u_id, pos_item, neg_item)
        year_idx = int(year.min()) % 18
        table = self._packed_table()
        if self.emb_ratio > 0:                                         # NGCF's feature mix of the batch users' rows
            self._feature_mix(table, st.rows[0], (age, sex, month, day, dow))
        st.fresh_key = self._fresh_key()
        st.plan = self._plan(year_idx, dev)
        st.drop_p = self.node_dropout if bool(node_flag) and self.node_dropout > 0 else 0.0
        self._draw_seed(st, noise=eps > 0)
        return st, _LightPropagate.apply(self, st, len(st.rows), self._first, eps, cl_layer, self.user_embedding.weight,
                                         self.item_embedding.weight)

    def _readout(self, st: _Ctx) -> torch.Tensor:
        """[N, embed_size]: the layer mean of every row."""
        N = self.n_user + self.n_item
        out = torch.empty(N, self.emb_size, dtype=torch.float32, device=st.E[0].device)
        _lib.check(_lib.load().ngcf_layer_mean(_lib.ptr_array(st.E[self._first:]), self.n_layer + 1 - self._first,
                                               self.emb_size, None, 0, N, out.data_ptr(), self.emb_size,
                                               _lib.current_stream()), "layer_mean")
        return out


class _InfoNCEFn(torch.autograd.Function):
    """ngcf_infonce: the cosine InfoNCE of two views over the distinct ids of a batch, with both views' gradients."""

    @staticmethod
    def forward(ctx, x1, x2, ids, temperature):
        lib = _lib.load()
        B, D = x1.shape
        ws_bytes = C.c_size_t()
        _lib.check(lib.ngcf_infonce_workspace(B, D, C.byref(ws_bytes)), "infonce_workspace")
        ws = torch.empty(ws_bytes.value, dtype=torch.uint8, device=x1.device)
        loss = torch.empty((), dtype=torch.float32, device=x1.device)
        grad = any(ctx.needs_input_grad[:2])
        g1, g2 = (torch.empty_like(x1), torch.empty_like(x2)) if grad else (None, None)
        _lib.check(lib.ngcf_infonce(x1.data_ptr(), x2.data_ptr(), B, D, ids.data_ptr(), float(temperature),
                                    loss.data_ptr(), _lib.ptr(g1), _lib.ptr(g2), ws.data_ptr(), ws_bytes.value,
                                    _lib.current_stream()), "infonce")
        ctx.grads = (g1, g2)
        return loss

    @staticmethod
    def backward(ctx, gloss):
        g1, g2 = ctx.grads
        return g1 * gloss, g2 * gloss, None, None


class XSimGCL(LightGCN):
    """``XSimGCL(embed_size, n_layers, lap_list, num_dict, *, eps=0.2, cl_weight=0.2, cl_layer=1, temperature=0.2,
    emb_ratio=0.0)``: XSimGCL (Yu et al., "XSimGCL: Towards Extremely Simple Graph Contrastive Learning for
    Recommendation", TKDE 2023) on LightGCN's propagation, as in the authors' SELFRec code:

        E_{k+1} = L E_k + eps * sign(L E_k) * normalize(U_{k+1}),   U ~ Uniform[0, 1)^{N x d}   (training forward only)
        rows    = mean(E_1 .. E_K)                                   (E_0 is not in the readout)
        cl_loss = cl_weight * (InfoNCE(rows[users], E_cl[users]) + InfoNCE(rows[positives], E_cl[positives]))

    InfoNCE(a, b) = mean_i [-log softmax_j(cos(a_i, b_j) / temperature)_ii] over the batch's DISTINCT ids (the first
    occurrence of each).  ``forward`` has LightGCN's signature and outputs (rows of mean(E_1 .. E_K)).  ``node_flag``
    set is the training forward: it perturbs every layer and leaves the contrastive term, a 0-d tensor with autograd
    history already multiplied by cl_weight, in ``model.cl_loss``; add it to the recommendation loss
    (``loss = crit(u, p, n) + model.cl_loss``; ``GraphedStep`` and ``Experiment.train`` do).  ``node_flag`` unset, or
    cl_weight = 0, leaves ``cl_loss`` None; the evaluation forward adds no noise either.  There is no node dropout.
    The noise is keyed on the forward's RNG key (a CUDA-graph replay draws new noise); ``HardNegatives`` score on the
    same step's perturbed mean(E_1 .. E_K).  The state_dict is LightGCN's.

    Backward: the noise's derivative is zero almost everywhere, so the model stays linear in E_0.  With G the batch's
    row gradients of mean(E_1 .. E_K) and H those of the view-2 rows,
        gE_K = G/K (+ H if cl_layer == K),  gE_k = L^T gE_{k+1} + G/K + [k == cl_layer] H,  gE_0 = L^T gE_1."""
    _NAME = "XSimGCL"
    _first = 1                                    # readout: mean of E_1 .. E_K

    def __init__(self, embed_size: int, n_layers: int, lap_list: list, num_dict: dict, *, eps: float = 0.2,
                 cl_weight: float = 0.2, cl_layer: int = 1, temperature: float = 0.2, emb_ratio: float = 0.0):
        super().__init__(embed_size, n_layers, lap_list, num_dict, node_dropout=0.0, emb_ratio=emb_ratio)
        self.eps, self.cl_weight, self.temperature = float(eps), float(cl_weight), float(temperature)
        self.cl_layer = int(cl_layer)
        if not (self.eps >= 0.0 and self.eps < float("inf")):
            raise ValueError(f"XSimGCL: eps {eps} is not >= 0")
        if not (self.cl_weight >= 0.0 and self.cl_weight < float("inf")):
            raise ValueError(f"XSimGCL: cl_weight {cl_weight} is not >= 0")
        if not (self.temperature > 0.0 and self.temperature < float("inf")):
            raise ValueError(f"XSimGCL: temperature {temperature} is not > 0")
        if not 1 <= self.cl_layer <= self.n_layer:
            raise ValueError(f"XSimGCL: cl_layer {self.cl_layer} not in [1, n_layers = {self.n_layer}]")
        self.cl_loss = None

    def shard(self, group=None, shards=None):
        raise NotImplementedError("XSimGCL: row-sharded runs are not supported; use NGCF.shard() for those")

    @_lib.on_device
    def forward(self, year, u_id, age, sex, month, day, dow, pos_item, neg_item, node_flag):
        train = bool(node_flag)
        cl_layer = self.cl_layer if train and self.cl_weight > 0 else 0
        if cl_layer and not 1 <= len(u_id) <= MAX_INFONCE_BATCH:
            raise ValueError(f"XSimGCL: a training batch of {len(u_id)} rows; the contrastive loss takes 1 to "
                             f"{MAX_INFONCE_BATCH} (or set cl_weight=0)")
        self.cl_loss = None
        st, outs = self._propagate(year, u_id, age, sex, month, day, dow, pos_item, neg_item, node_flag,
                                   self.eps if train else 0.0, cl_layer)
        if cl_layer:
            outs, (v2u, v2p) = outs[:-2], outs[-2:]
            self.cl_loss = self.cl_weight * (_InfoNCEFn.apply(outs[0], v2u, st.rows[0], self.temperature) +
                                             _InfoNCEFn.apply(outs[1], v2p, st.rows[1], self.temperature))
        return self._finish(st, outs)
