"""Whole-step CUDA graph around the drop-in modules.

One reference training step (experiment.py:45-57: ``model(...)``, ``criterion(u, pos, neg)``, ``loss.backward()``)
is ~35 kernel launches of 5-70 us each; issued eagerly from Python the host is the bottleneck (and, row-sharded over
several GPUs, so are the NCCL launches).  ``GraphedStep`` captures exactly those three calls once — same modules,
same kernels, same collectives — and replays them: per step the host does one pinned H2D copy of the index batch
and one graph launch.  Gradients land in ``param.grad`` like after ``zero_grad(); loss.backward()``.

Dropout stays fresh on every replay: the RNG key of a step is ``seed + *seed_dev`` (include/ngcf_b200.h) and the
graph bumps the device counter ``seed_dev`` itself.
"""
from __future__ import annotations

import torch

from .softmax_loss import SoftmaxLoss

FIELDS = ("u_id", "age", "sex", "month", "day", "dow", "pos_item", "neg_item")


class GraphedStep:
    """``step = GraphedStep(model, criterion, batch_size); loss = step(batch)`` with ``batch`` a dict of int64
    tensors (host or device) holding ``year`` plus the eight index fields of ``TourDataset`` (utils.py:167-275).
    ``year`` must be a host tensor (it selects ``lap_list[year.min() % 18]`` on the host, NGCF.py:117); one graph is
    kept per selected Laplacian.  ``node_flag`` / train-vs-eval mode are frozen at capture time.

    ``negatives``: a ``HardNegatives``; each replay then chooses every row's negative on the device, from fresh
    candidates, and batches carry no ``neg_item``.  After each call ``negatives.chosen`` holds that step's picks."""

    def __init__(self, model, criterion, batch_size: int, node_flag: bool = True, warmup: int = 1, optimizer=None,
                 negatives=None):
        dev = model.user_embedding.weight.device
        if dev.type != "cuda":
            raise RuntimeError("GraphedStep needs the model on a CUDA device")
        self.model, self.criterion, self.node_flag, self.warmup = model, criterion, bool(node_flag), int(warmup)
        self.B = int(batch_size)
        self.negatives = negatives
        self.fields = FIELDS[:-1] if negatives is not None else FIELDS
        # optional ngcf_b200.Adam: its step (and the zeroing of the gradients for the next batch, experiment.py:55,58)
        # joins the graph, so a replay is the reference's whole training iteration
        self.optimizer = optimizer
        self.static_idx = torch.zeros(len(self.fields), self.B, dtype=torch.int64, device=dev)
        # pinned staging buffers for host batches, rotated: the H2D copy below is asynchronous, so a buffer may only be
        # rewritten once the copy that read it has run (its event); with one buffer a host running ahead of the GPU
        # would overwrite a batch that is still waiting to be copied
        self.stages = [torch.zeros(len(self.fields), self.B, dtype=torch.int64).pin_memory() for _ in range(3)]
        self.stage_events = [None] * len(self.stages)
        self._stage_i = 0
        self.seed_dev = torch.zeros(1, dtype=torch.int64, device=dev)
        self.graphs = {}
        self.launches_per_step = None

    def _run(self, year, with_optimizer: bool = True):
        m = self.model
        f = {k: self.static_idx[i] for i, k in enumerate(self.fields)}
        neg = self.negatives if self.negatives is not None else f["neg_item"]
        u, p, n = m(year=year, u_id=f["u_id"], age=f["age"], sex=f["sex"], month=f["month"], day=f["day"], dow=f["dow"],
                    pos_item=f["pos_item"], neg_item=neg, node_flag=self.node_flag)
        if isinstance(self.criterion, SoftmaxLoss):
            # the batch's item ids mask false negatives; under capture these are the static index rows (or the
            # HardNegatives picks), so every replay masks with its own batch's ids
            rows = m._last.rows
            loss = self.criterion(u, p, n, rows[1], rows[2] if len(rows) > 2 else None)
        else:
            loss = self.criterion(u, p, n)
        if getattr(m, "cl_loss", None) is not None:                   # XSimGCL's contrastive term
            loss = loss + m.cl_loss
        loss.backward()
        if self.optimizer is not None and with_optimizer:
            self.optimizer.step()         # (a replay overwrites every gradient buffer, so nothing needs zeroing)
        self.seed_dev.add_(0x9E3779B97F4A7C15 & (2 ** 62 - 1))        # next step: a different RNG key
        return loss

    def _capture(self, year):
        from . import _lib
        m = self.model
        m._seed_dev = self.seed_dev
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):                                    # warm-up outside the graph (plans, buffers)
            # the forward rewrites the batch users' rows in place (feature mix, NGCF.py:114-115: not idempotent unless
            # emb_ratio == 1), so the warm-up runs on a snapshot of the user table that is put back afterwards
            users_before = m.user_embedding.weight.detach().clone()
            for _ in range(self.warmup):
                m.zero_grad(set_to_none=True)
                self._run(year, with_optimizer=False)                 # no parameter changes before the capture
            if self.optimizer is not None:                            # optimizer state must exist before the capture
                self.optimizer.prepare([p for p in m.parameters() if p.grad is not None])
            m.user_embedding.weight.data.copy_(users_before)
        torch.cuda.current_stream().wait_stream(s)
        m.zero_grad(set_to_none=True)
        g = torch.cuda.CUDAGraph()
        n0 = _lib.load().ngcf_launch_count()
        with torch.cuda.graph(g):
            loss = self._run(year)
        self.launches_per_step = int(_lib.load().ngcf_launch_count() - n0)
        grads = {k: p.grad for k, p in m.named_parameters() if p.grad is not None}
        return g, loss, grads, m._last

    def __call__(self, batch):
        year = batch["year"]
        if year.device.type != "cpu":
            raise ValueError("GraphedStep: pass `year` as a host tensor (it is only used to pick lap_list[year % 18])")
        if self.negatives is not None and "neg_item" in batch:
            raise ValueError("GraphedStep: built with negatives=, so the batch must not carry neg_item")
        on_host = [batch[k].device.type == "cpu" for k in self.fields]
        stage = None
        if any(on_host):
            j = self._stage_i
            self._stage_i = (j + 1) % len(self.stages)
            if self.stage_events[j] is not None:
                self.stage_events[j].synchronize()                    # the copy that last read this buffer has run
            stage = self.stages[j]
        for i, k in enumerate(self.fields):
            t = batch[k]
            if t.numel() != self.B:
                raise ValueError(f"GraphedStep was built for batches of {self.B} rows, got {t.numel()} for {k}")
            if on_host[i]:
                stage[i].copy_(t)
        if all(on_host):
            self.static_idx.copy_(stage, non_blocking=True)           # one pinned H2D copy for the whole batch
        else:
            for i, k in enumerate(self.fields):
                self.static_idx[i].copy_(stage[i] if on_host[i] else batch[k], non_blocking=True)
        if stage is not None:
            if self.stage_events[j] is None:
                self.stage_events[j] = torch.cuda.Event()
            self.stage_events[j].record()
        key = int(year.min()) % 18
        entry = self.graphs.get(key)
        if entry is None:                                             # first batch of this Laplacian: `warmup` eager
            entry = self.graphs[key] = self._capture(year)            # steps on it (no parameter changes), then capture
        g, loss, grads, last = entry
        g.replay()
        self.model._last, self.model._all_E = last, None              # all_users_emb / all_items_emb: rebuild on read
        if last.hneg is not None:                                     # this graph's output buffers of the picks
            last.hneg[0].chosen, last.hneg[0].cand, last.hneg[0].score = last.hneg[2:]
        if self.optimizer is not None:
            from . import _lib
            _lib.bump_param_epoch()                                   # the replay stepped the parameters
            last.fresh_key = None                                     # ... so E_0 (the live table) no longer matches H_k
        else:
            self.model._mix_count += 1                                # the replay ran the feature mix
            last.fresh_key = self.model._fresh_key()
        for k, p in self.model.named_parameters():                    # survive an optimizer.zero_grad(set_to_none=True)
            if k in grads and p.grad is not grads[k]:
                p.grad = grads[k]
        return loss
