"""Drop-in ``Experiment`` (reference: model/experiment.py:9-130): the training loop over the B200 modules and the
evaluation loop with its metric block fused into one kernel (SURVEY.md section 8(f) #4).

``eval()`` returns the reference's tuple ``(BPR, HR, NDCG, RMSE)`` (experiment.py:119).  Two modes:

* ``eval_mode="reference"`` (default) — one full-graph forward per test batch, in loader order, exactly as
  experiment.py:75-91 does (each forward overwrites its users' table rows, NGCF.py:114-115, so later batches see
  them); the per-batch metric arithmetic (experiment.py:92-116: an mm, two topk, a BPR call, an MSE and ~6 ``.item()``
  / ``.cpu()`` syncs per batch) is deferred to ONE ``ngcf_eval_groups`` launch over all batches and one 16-byte read.
* ``eval_mode="batched"`` — one propagation per distinct Laplacian (year bucket) for ALL test rows, then the same
  launch.  Equal to the reference whenever the feature mix of the test rows is idempotent on the table it meets
  (``emb_ratio == 0``, or ``emb_ratio == 1`` with every test user already mixed — e.g. any eval() after the first);
  otherwise it differs by the rows of users whose test batch comes later in the loader.
"""
from __future__ import annotations

import torch
import torch.nn as nn

from . import _lib
from .softmax_loss import SoftmaxLoss


@_lib.on_device
def eval_groups(u_embeds, item_embeds, item_ids, rating, *, group=None, group_ptr=None, ks, weight_decay, batch_size,
                k_hr=3, return_per_group=False):
    """The metric block of experiment.py:92-116 for every test batch at once.

    u_embeds / item_embeds: [rows, D] CUDA fp32 (what NGCF.forward returned, batches stacked in loader order);
    item_ids [rows] int64; rating [rows]; ``group`` = rows per batch (``test_batch``) or ``group_ptr`` int64 [G+1]
    offsets for ragged batches.  Returns a CUDA tensor [4] = (BPR, HR, NDCG, RMSE) (and the per-group arrays)."""
    if u_embeds.device.type != "cuda" or item_embeds.device.type != "cuda":
        raise RuntimeError("eval_groups (B200) runs on CUDA tensors only; there is no CPU fallback")
    lib = _lib.load()
    dev = u_embeds.device
    u = u_embeds.detach().to(torch.float32).contiguous()
    it = item_embeds.detach().to(torch.float32).contiguous()
    ids = item_ids.to(device=dev, dtype=torch.int64).contiguous()
    rt = rating.to(device=dev, dtype=torch.float32).contiguous()
    rows, D = u.shape
    if it.shape != u.shape or ids.numel() != rows or rt.numel() != rows:
        raise RuntimeError(f"eval_groups: u {tuple(u.shape)}, items {tuple(it.shape)}, ids {ids.numel()}, "
                           f"rating {rt.numel()} do not describe the same rows")
    if group_ptr is not None:
        gp_host = group_ptr.to("cpu", torch.int64)
        sizes = gp_host[1:] - gp_host[:-1]
        G = sizes.numel()
        if G and (int(gp_host[0]) != 0 or int(gp_host[-1]) != rows or int(sizes.min()) < 2 or int(sizes.max()) > 128):
            raise RuntimeError("eval_groups: group_ptr must cover the rows with groups of 2..128 rows")
        group = int(sizes.min()) if G else 2
        gp = gp_host.to(dev)
    else:
        if group is None or group < 2 or rows % group:
            raise RuntimeError(f"eval_groups: {rows} rows are not whole groups of {group}")
        G, gp = rows // group, None
    if ks > group or k_hr > group:
        raise RuntimeError("selected index k out of range")              # torch.topk, experiment.py:104,109
    per = torch.empty(4, max(G, 1), dtype=torch.float32, device=dev)
    totals = torch.zeros(4, dtype=torch.float32, device=dev)
    _lib.check(lib.ngcf_eval_groups(u.data_ptr(), it.data_ptr(), ids.data_ptr(), rt.data_ptr(), _lib.ptr(gp), G,
                                    int(group), D, int(k_hr), int(ks), float(weight_decay), float(batch_size),
                                    per[0].data_ptr(), per[1].data_ptr(), per[2].data_ptr(), per[3].data_ptr(), None,
                                    totals.data_ptr(), _lib.current_stream()), "eval_groups")
    if return_per_group:
        return totals, per[:, :G]
    return totals


class Experiment(nn.Module):
    """Same constructor and methods as the reference class (experiment.py:9-30); ``train()`` / ``eval()`` shadow
    ``nn.Module``'s like the reference's do."""

    def __init__(self, model, optimizer, criterion, test_criterion, train_dataloader, test_dataloader, epochs: int,
                 ks: int, device, eval_mode: str = "reference", verbose: bool = True, graphed: bool = False):
        super().__init__()
        if eval_mode not in ("reference", "batched"):
            raise ValueError("eval_mode is 'reference' or 'batched'")
        self.model = model
        self.optimizer = optimizer
        self.criterion = criterion
        self.test_criterion = test_criterion
        self.train_dataloader = train_dataloader
        self.test_dataloader = test_dataloader
        self.epochs = epochs
        self.ks = ks
        self.device = device
        self.eval_mode = eval_mode
        self.verbose = verbose
        # graphed=True: each training batch is one replay of graph.GraphedStep (forward + BPR + backward + optimizer
        # in one CUDA graph); needs ngcf_b200.Adam as the optimizer and a drop_last loader (main.py:39-42 has one)
        self.graphed = graphed
        self._gstep = None

    # experiment.py:32-64
    def train(self):
        history = []
        for epoch in range(self.epochs):
            total_loss = torch.zeros((), device=self.device)
            for year, u_id, age, sex, month, day, dow, pos_item, neg_item in self.train_dataloader:
                if self.graphed:
                    loss = self._graphed_step(dict(year=year, u_id=u_id, age=age, sex=sex, month=month, day=day,
                                                   dow=dow, pos_item=pos_item, neg_item=neg_item))
                else:
                    u, p, n = self.model(year=year, u_id=u_id, age=age, sex=sex, month=month, day=day, dow=dow,
                                         pos_item=pos_item, neg_item=neg_item, node_flag=True)
                    self.optimizer.zero_grad()
                    if isinstance(self.criterion, SoftmaxLoss):         # item ids mask the batch's false negatives
                        dev = u.device
                        neg_ids = neg_item.to(dev, torch.int64) if n.numel() else None
                        loss = self.criterion(u, p, n, pos_item.to(dev, torch.int64), neg_ids)
                    else:
                        loss = self.criterion(u, p, n)
                    if getattr(self.model, "cl_loss", None) is not None:    # XSimGCL's contrastive term
                        loss = loss + self.model.cl_loss
                    loss.backward()
                    self.optimizer.step()
                total_loss += loss.detach()
            BPR, HR, NDCG, RMSE = self.eval()
            train_bpr = float(total_loss) / len(self.train_dataloader)
            history.append((train_bpr, BPR, HR, NDCG, RMSE))
            if self.verbose:
                print(f"epoch {epoch + 1}, Train BPR: {train_bpr}, Test BPR: {BPR}, HR:{HR}, NDCG:{NDCG}, RMSE:{RMSE}")
        return history

    def _graphed_step(self, batch):
        from .graph import GraphedStep
        training = self.model.training
        if self._gstep is None or self._gstep[0] != training:      # train/eval mode is frozen into a capture
            self._gstep = (training, GraphedStep(self.model, self.criterion, batch["u_id"].numel(), node_flag=True,
                                                 optimizer=self.optimizer))
        batch["year"] = batch["year"].cpu()
        return self._gstep[1](batch)

    def _forward(self, b):
        u, p, _ = self.model(year=b[0], u_id=b[1], age=b[2], sex=b[3], month=b[4], day=b[5], dow=b[6],
                             pos_item=b[8], neg_item=torch.empty(0), node_flag=False)      # experiment.py:82-91
        return u, p

    # experiment.py:66-119
    def eval(self):
        wd, tb = self.test_criterion.weight_decay, self.test_criterion.batch_size
        us, ps, ids, rts, sizes = [], [], [], [], []
        with torch.no_grad():
            self.model.eval()                                  # never undone, like experiment.py:72
            batches = [tuple(torch.as_tensor(t) for t in b) for b in self.test_dataloader]
            if not batches:
                raise ZeroDivisionError("division by zero")     # len(self.test_dataloader) == 0, experiment.py:119
            if self.eval_mode == "reference":
                for b in batches:
                    u, p = self._forward(b)
                    us.append(u); ps.append(p)
            else:
                # one propagation per Laplacian: NGCF.py:117 picks it by the smallest year of the batch
                bucket = {}
                for j, b in enumerate(batches):
                    bucket.setdefault(int(b[0].min()) % 18, []).append(j)
                us, ps = [None] * len(batches), [None] * len(batches)
                for _, members in sorted(bucket.items()):
                    cat = [torch.cat([batches[j][c] for j in members]) for c in range(9)]
                    u, p = self._forward(cat)
                    o = 0
                    for j in members:
                        n = batches[j][1].numel()
                        us[j], ps[j] = u[o:o + n], p[o:o + n]
                        o += n
            for b in batches:
                ids.append(b[8]); rts.append(b[7]); sizes.append(b[1].numel())
            dev = us[0].device
            kw = dict(ks=self.ks, weight_decay=wd, batch_size=tb)
            if len(set(sizes)) == 1:
                kw["group"] = sizes[0]
            else:
                kw["group_ptr"] = torch.tensor([0] + sizes, dtype=torch.int64).cumsum(0)
            totals = eval_groups(torch.cat(us), torch.cat(ps), torch.cat(ids).to(dev), torch.cat(rts).to(dev), **kw)
            BPR, HR, NDCG, RMSE = totals.tolist()              # the one device->host read of the evaluation
        return BPR, HR, NDCG, RMSE
