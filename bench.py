#!/usr/bin/env python
"""Benchmark of the NGCF embedding-propagation hot path (BASELINE.json metric:
"NGCF epoch time (fwd+bwd+BPR) at Gowalla shape; propagation SpMM HBM GB/s vs peak").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--shape gowalla] [--dump-outputs DIR]

A step is one reference training step (experiment.py:45-57): NGCF.forward over the full graph for one
1024-triple batch with node_flag=True in training mode, BPR loss, backward to every parameter gradient
(the optimizer step is not part of the metric).  One JSON line is printed by rank 0.

--dump-outputs DIR writes, after the timed steps, what the timed path returned in its last step (the loss and every
parameter gradient) as DIR/<name>.npy.  Inputs are seeded, so two builds run with the same arguments can be compared
output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

BATCH = 1024                     # parsers.py:5
WEIGHT_DECAY = 0.025             # main.py:75
NODE_P, MESS_P = 0.3, 0.1        # parsers.py:11-12
METRIC = "ngcf_epoch_time_fwd_bwd_bpr"
L2_FLUSH_BYTES = 512 << 20


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--shape", default="gowalla")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-epoch", action="store_true", help="skip the measured whole-epoch leg")
    ap.add_argument("--eager", action="store_true", help="time the eager drop-in path only (no CUDA graph)")
    ap.add_argument("--breakdown", action="store_true", help="print a per-entry-point time table to stderr")
    ap.add_argument("--no-extra", action="store_true", help="skip the extra legs (other named shapes at the same N)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss and parameter gradients of the last timed step as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return a


def log(*a):
    print(*a, file=sys.stderr, flush=True)


_json_out = None


def protect_stdout():
    """stdout carries exactly one JSON line: whatever libraries print there (NCCL's version banner under
    NCCL_DEBUG=VERSION, for one) is sent to stderr by pointing fd 1 at fd 2 and keeping the real stdout aside."""
    global _json_out
    if _json_out is None:
        sys.stdout.flush()
        _json_out = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(obj):
    f = _json_out or sys.stdout
    f.write(json.dumps(obj) + "\n")
    f.flush()


# ------------------------------------------------------------------------------------------------------------
# workload
# ------------------------------------------------------------------------------------------------------------
def make_workload(shape: str, n_batches: int = 8):
    from seoul_tourism_recommendation_ngcf_b200 import laplacian, synth
    n_user, n_item, n_edges, emb, K = synth.SHAPES[shape]
    t0 = time.time()
    u, i, r = synth.powerlaw_bipartite(n_user, n_item, n_edges, alpha=0.8, seed=0)
    L = laplacian.laplacian_coo(u, i, r, n_user, n_item)
    batches = [synth.random_batch(n_user, n_item, BATCH, seed=1 + j) for j in range(n_batches)]
    deg = np.bincount(np.concatenate([u, i + n_user]), minlength=n_user + n_item)
    info = dict(workload=f"{shape}-shaped synthetic power-law graph (Zipf 0.8), {n_user} users / {n_item} items / "
                         f"{n_edges} interactions, emb {emb}, {K} layers, batch {BATCH}, node_flag=True, training mode",
                shape=shape, n_user=n_user, n_item=n_item, interactions=n_edges, nnz=int(L._nnz()), emb=emb, layers=K,
                batch=BATCH, steps_per_epoch=n_edges // BATCH, max_degree=int(deg.max()),
                mean_degree=float(deg.mean()))
    log(f"[bench] workload built in {time.time() - t0:.1f}s: N={n_user + n_item} nnz={L._nnz()} max_deg={deg.max()}")
    return L, batches, info


def make_model(info, L, device, rng="device"):
    import seoul_tourism_recommendation_ngcf_b200 as pkg
    from seoul_tourism_recommendation_ngcf_b200 import synth
    torch.manual_seed(0)
    K = info["layers"]
    m = pkg.NGCF(info["emb"], [info["emb"]] * K, NODE_P, [MESS_P] * K, 1.0, [L, L],
                 synth.num_dict_for(info["n_user"], info["n_item"]), BATCH, device, rng=rng)
    return m


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, loss, model):
    """Writes what a caller of the timed step holds after it: the loss (float64) as loss.npy and every parameter
    gradient (float32) as grad.<parameter>.npy.  Past DUMP_BYTES in all, each gradient keeps a fixed, seeded sample of
    its rows: the same rows on every run of the same shape."""
    grads = {k: p.grad.detach() for k, p in model.named_parameters() if p.grad is not None}
    frac = min(1.0, DUMP_BYTES / (4 * sum(g.numel() for g in grads.values())))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), np.array([float(loss.detach())], dtype=np.float64))
    for k, g in grads.items():
        if frac < 1.0 and g.shape[0] > 1:
            rows = np.sort(np.random.default_rng(0).choice(g.shape[0], max(1, int(g.shape[0] * frac)), replace=False))
            g = g[torch.from_numpy(rows).to(g.device)]
        np.save(os.path.join(out_dir, f"grad.{k}.npy"), g.float().cpu().numpy())


# ------------------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,utilization.gpu")

    def __init__(self, index=0):
        self.samples, self.proc, self.thread = [], None, None
        self.index = index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.time(), line.strip()))

    def stop(self, windows):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        mhz, mx, reasons, n_in = [], None, set(), 0
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.samples:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            inside = any(a - 0.05 <= ts <= b + 0.15 for a, b in windows)
            try:
                util = float(f[6])
            except ValueError:
                util = 0.0
            if not inside and util < 5:
                continue
            n_in += 1
            try:
                mhz.append(float(f[0])); mx = float(f[1])
            except ValueError:
                continue
            for nm, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(mhz) if mhz else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": n_in}


# ------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------
class CallTimer:
    """Wraps the ctypes library so every C-ABI call is bracketed by CUDA events (breakdown pass only)."""

    def __init__(self, lib):
        self._lib, self.rec = lib, []

    def __getattr__(self, name):
        fn = getattr(self._lib, name)
        if not name.startswith("ngcf_") or name in ("ngcf_last_error", "ngcf_launch_count", "ngcf_abi_version",
                                                    "ngcf_spmm_split_threshold") or name.endswith("_workspace"):
            return fn

        def wrapped(*a):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            rc = fn(*a)
            e1.record()
            self.rec.append((name, e0, e1))
            return rc
        return wrapped

    def table(self):
        torch.cuda.synchronize()
        agg = {}
        for name, e0, e1 in self.rec:
            t, c = agg.get(name, (0.0, 0))
            agg[name] = (t + e0.elapsed_time(e1), c + 1)
        return agg


def time_shape(pkg, shape, dev, world, rank, steps=10, warmup=3):
    """ms per step (CUDA graph replay, device-resident batches, max over ranks) of another named shape at this N: the
    extra legs of the bench line (BASELINE.json configs 3 and 4)."""
    import torch.distributed as dist
    L, batches, info = make_workload(shape, n_batches=4)
    model = make_model(info, L, dev).to(dev)
    if world > 1:
        shards = None
        if os.environ.get("NGCF_B200_EXCHANGE", "peer") != "nccl" and os.environ.get("NGCF_B200_SHARDS", "balanced") == "balanced":
            from seoul_tourism_recommendation_ngcf_b200.sharded import BalancedShards
            row_nnz = np.bincount(L._indices()[0].numpy(), minlength=int(L.shape[0]))
            shards = BalancedShards(int(L.shape[0]), world, rank, BalancedShards.cut(row_nnz + 32.0, world))
        try:
            model.shard(shards=shards)
        except RuntimeError:
            model.shard()
    model.train()
    crit = pkg.BPR(WEIGHT_DECAY, BATCH)
    db = [{k: (torch.from_numpy(v) if k == "year" else torch.from_numpy(v).to(dev)) for k, v in b.items()} for b in batches]
    gstep = pkg.GraphedStep(model, crit, BATCH, node_flag=True)
    for j in range(warmup):
        gstep(db[j % len(db)])
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for j in range(steps):
        ev[j][0].record()
        gstep(db[j % len(db)])
        ev[j][1].record()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = sum(a.elapsed_time(b) for a, b in ev) / steps
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t)
    out = {"ms_per_step": round(ms, 4), "value": round(ms * info["steps_per_epoch"] / 1e3, 4), "unit": "s/epoch",
           "workload": info["workload"], "steps": steps, "gpu_launches_per_step": gstep.launches_per_step,
           "l2": "not flushed (back-to-back replays)"}
    del gstep, model, L
    torch.cuda.empty_cache()
    return out


def run_ours(args):
    import seoul_tourism_recommendation_ngcf_b200 as pkg
    from seoul_tourism_recommendation_ngcf_b200 import _lib
    from seoul_tourism_recommendation_ngcf_b200.plan import spmm

    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank, local = int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus != world:
        raise SystemExit(f"--gpus {args.gpus} needs {args.gpus} ranks: launch with python -m torch.distributed.run "
                         f"--nnodes=1 --nproc-per-node {args.gpus} --master-addr 127.0.0.1 bench.py --gpus {args.gpus} ...")
    assert torch.cuda.is_available(), "bench.py --impl ours needs a CUDA device (no CPU fallback)"
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl")
    lib = _lib.load()
    L, batches, info = make_workload(args.shape)
    model = make_model(info, L, dev).to(dev)
    shards = None
    if world > 1:
        # row partition (sharded.py); every rank steps the same batches.  With the peer-memory exchange the blocks are cut
        # by work (entries + 32 per row) instead of by row count: item rows are several times heavier than user rows
        if os.environ.get("NGCF_B200_EXCHANGE", "peer") != "nccl" and os.environ.get("NGCF_B200_SHARDS", "balanced") == "balanced":
            from seoul_tourism_recommendation_ngcf_b200.sharded import BalancedShards
            row_nnz = np.bincount(L._indices()[0].numpy(), minlength=int(L.shape[0]))
            shards = BalancedShards(int(L.shape[0]), world, rank, BalancedShards.cut(row_nnz + 32.0, world))
        try:
            model.shard(shards=shards)
        except RuntimeError as e:                                     # no peer-memory exchange here: equal blocks + NCCL
            log(f"[bench] {e}; falling back to equal blocks")
            shards = None
            model.shard()
    model.train()

    def max_over_ranks(ms: float) -> float:
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    def fence():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- N > 1: the sharded step must BE the 1-GPU step before any of its timings mean anything (VERDICT r1 #1) -------
    parity = None
    if world > 1:
        from seoul_tourism_recommendation_ngcf_b200 import synth
        from seoul_tourism_recommendation_ngcf_b200.sharded import parity_vs_unsharded
        pb = {k: torch.from_numpy(v) for k, v in batches[0].items()}
        res = parity_vs_unsharded(info["emb"], [info["emb"]] * info["layers"], L,
                                  synth.num_dict_for(info["n_user"], info["n_item"]), pb, BATCH, dev,
                                  node_p=NODE_P, mess_p=MESS_P, weight_decay=WEIGHT_DECAY, shards=shards)
        worst = torch.tensor([res["out"], res["loss"], res["all_E"], res["worst_grad"]], dtype=torch.float64, device=dev)
        dist.all_reduce(worst, op=dist.ReduceOp.MAX)                 # the worst rank's figures
        parity = {"out": float(worst[0]), "loss": float(worst[1]), "all_E": float(worst[2]),
                  "worst_grad": float(worst[3]), "tolerance": 1e-5,
                  "what": "one training step (node + message dropout ON, device RNG) row-sharded over all ranks vs the same "
                          "step unsharded on each rank's own GPU; max|a-b|/max|b| of the batch outputs, the loss, "
                          "all_users/items_emb and the worst parameter gradient; max over ranks"}
        log(f"[bench] parity_vs_1gpu: {parity}")
        if max(parity["out"], parity["loss"], parity["all_E"], parity["worst_grad"]) > 1e-5:
            if rank == 0:
                emit({"metric": METRIC, "error": "row-sharded step differs from the 1-GPU step", "n_gpus": world,
                      "parity_vs_1gpu": parity})
            sys.stdout.flush()
            sys.stderr.flush()
            os._exit(3)
        torch.cuda.empty_cache()

    crit = pkg.BPR(WEIGHT_DECAY, BATCH)
    dbatches = [{k: torch.from_numpy(v).to(dev) for k, v in b.items()} for b in batches]
    hbatches = [{k: torch.from_numpy(v).pin_memory() for k, v in b.items()} for b in batches]
    flush = torch.empty(L2_FLUSH_BYTES, dtype=torch.uint8, device=dev)

    def step(b):
        model.zero_grad(set_to_none=True)
        u, p, n = model(year=b["year"], u_id=b["u_id"], age=b["age"], sex=b["sex"], month=b["month"], day=b["day"],
                        dow=b["dow"], pos_item=b["pos_item"], neg_item=b["neg_item"], node_flag=True)
        loss = crit(u, p, n)
        loss.backward()
        return loss

    # year stays on the host for index selection (NGCF.py:117) so the step has no device sync
    for b in dbatches:
        b["year"] = b["year"].cpu()
    for j in range(max(args.warmup, 3)):
        step(dbatches[j % len(dbatches)])
    fence()

    sampler = ClockSampler(local)
    sampler.start()
    windows = []

    def timed_resident(fn, dump=False):
        """K steps on device-resident batches, per-step CUDA events, L2 flushed between steps; max over ranks.  With
        ``dump``, rank 0 writes the last step's outputs to --dump-outputs afterwards."""
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        fence()
        w0 = time.time()
        for j in range(args.steps):
            flush.zero_()
            ev[j][0].record()
            loss = fn(dbatches[j % len(dbatches)])
            ev[j][1].record()
        fence()
        windows.append((w0, time.time()))
        if dump and args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, loss, model)
        return max_over_ranks(sum(a.elapsed_time(b) for a, b in ev)) / args.steps

    def timed_e2e(fn, to_dev):
        """K steps from pinned host batches: H2D copy + step + loss read back inside the timed region."""
        for j in range(3):
            b = hbatches[j % len(hbatches)]
            float(fn({k: (v if (k == "year" or not to_dev) else v.to(dev, non_blocking=True)) for k, v in b.items()}).detach())
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        fence()
        w0 = time.time()
        e0.record()
        last = 0.0
        for j in range(args.steps):
            b = hbatches[j % len(hbatches)]
            db = {k: (v if (k == "year" or not to_dev) else v.to(dev, non_blocking=True)) for k, v in b.items()}
            last = float(fn(db).detach())                       # device -> host read of the step's result
        e1.record()
        fence()
        windows.append((w0, time.time()))
        return max_over_ranks(e0.elapsed_time(e1)) / args.steps, last

    # ---- the eager drop-in path first (before any graph capture touches the allocator) ---------------------------
    h2d = sum(v.numel() * v.element_size() for k, v in hbatches[0].items() if k != "year")
    launches0 = lib.ngcf_launch_count()
    ms_eager = timed_resident(step, dump=args.eager)
    launches_eager = (lib.ngcf_launch_count() - launches0) / args.steps
    ms_e2e_eager, loss_eager = timed_e2e(step, to_dev=True)

    # the same three calls captured once as a CUDA graph (graph.GraphedStep): the repo's fast public path
    gstep, api = None, "drop-in NGCF.forward + BPR + loss.backward(), eager"
    if not args.eager:
        try:
            gstep = pkg.GraphedStep(model, crit, BATCH, node_flag=True)
            for j in range(max(args.warmup, 3)):
                gstep(dbatches[j % len(dbatches)])
            fence()
            api = "GraphedStep = drop-in NGCF.forward + BPR + loss.backward() captured once as a CUDA graph, replayed per step"
        except Exception as e:                                   # e.g. a collective that cannot be captured
            log(f"[bench] CUDA-graph capture failed ({type(e).__name__}: {e}); measuring the eager path")
            gstep = None
            model._seed_dev = None
    run = gstep if gstep is not None else step

    # ---- value: device-resident inputs ------------------------------------------------------------------------
    # (a failed capture times the eager step again here: its first timed window's outputs are gone by now)
    ms_per_step = ms_eager if args.eager else timed_resident(run, dump=True)
    launches = gstep.launches_per_step if gstep is not None else launches_eager

    # ---- warm variant (no flush, back-to-back) — reported as context only -------------------------------------
    fence()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0 = time.time()
    e0.record()
    for j in range(args.steps):
        run(dbatches[j % len(dbatches)])
    e1.record()
    fence()
    windows.append((w0, time.time()))
    ms_warm = max_over_ranks(e0.elapsed_time(e1)) / args.steps

    # ---- e2e: host (pinned) inputs -> H2D inside the timed region -> step -> loss read back ---------------------
    if gstep is not None:
        ms_e2e, loss_val = timed_e2e(run, to_dev=False)          # GraphedStep copies the host batch itself (one H2D)
    else:
        ms_e2e, loss_val = ms_e2e_eager, loss_eager

    # ---- the reference's whole training iteration (experiment.py:45-58): the step above + Adam (main.py:74) -----------
    # reported beside the metric, not in it (BASELINE.json's metric is fwd + bwd + BPR)
    with_adam = None
    gstep_opt = None
    if gstep is not None and world == 1:
        try:
            gstep_opt = pkg.GraphedStep(model, crit, BATCH, node_flag=True, optimizer=pkg.Adam(model.parameters(), lr=5e-5))
            for j in range(max(args.warmup, 3)):
                gstep_opt(dbatches[j % len(dbatches)])
            fence()
            ms_opt = timed_resident(gstep_opt)
            with_adam = {"ms_per_step": round(ms_opt, 5), "adam_ms": round(ms_opt - ms_per_step, 5),
                         "api": "GraphedStep(optimizer=ngcf_b200.Adam(lr=5e-5)): fwd + BPR + bwd + ngcf_adam_step (one launch "
                                "over all parameters) in one replayed graph",
                         "adam_algorithmic_bytes": 28 * sum(p.numel() for p in model.parameters() if p.grad is not None)}
        except Exception as e:
            log(f"[bench] step + Adam graph failed ({type(e).__name__}: {e})")

    # ---- one WHOLE epoch, measured instead of extrapolated: the reference's Experiment.train loop for one epoch
    # (experiment.py:36-60) over triples drawn by the device sampler, host batches, Adam in the step ---------------------
    measured_epoch = None
    if gstep_opt is not None and with_adam is not None and not args.no_epoch:
        try:
            w0 = time.time()
            measured_epoch = run_epoch(pkg, gstep_opt, info, dev)
            windows.append((w0, time.time()))
        except Exception as e:
            log(f"[bench] measured epoch failed ({type(e).__name__}: {e})")

    # ---- roofline of the dominant kernel: the propagation SpMM of layer 0 exactly as the step runs it (this step's
    # node-dropout survivors, compacted), timed alone, cold L2 ----------------------------------------------------------
    from seoul_tourism_recommendation_ngcf_b200.plan import node_dropout_compact
    plan = model._last.plan                       # this rank's row shard when world > 1
    N, nnz, d = plan.fwd.n_rows, plan.fwd.nnz, info["emb"]
    X = model._packed_table()
    Y = torch.empty(N, d, device=dev)
    comp, _ = node_dropout_compact(plan.fwd, NODE_P, 1, None, info["layers"], model._shard.r0 if model._shard else 0,
                                   as_L=True, as_Lt=False)
    def kept_entries(side, cnt):
        return int(cnt.sum())

    nnz_kept = kept_entries(plan.fwd, comp[0][1])
    reps = 20

    def time_spmm(compact):
        kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
        for _ in range(3):
            spmm(plan.fwd, None, X, d, out=Y, compact=compact)
        torch.cuda.synchronize()
        for j in range(reps):
            flush.zero_()
            kev[j][0].record()
            spmm(plan.fwd, None, X, d, out=Y, compact=compact)
            kev[j][1].record()
        torch.cuda.synchronize()
        return statistics.mean(a.elapsed_time(b) for a, b in kev)

    w0 = time.time()
    k_ms = time_spmm(comp[0])
    k_ms_full = time_spmm(None)                                  # the same product without node dropout (eval / demo)
    windows.append((w0, time.time()))
    alg_bytes = 8 * nnz_kept + 4 * (N + 1) + 8 * N * d          # SURVEY.md section 8(d), SpMM-only per layer
    alg_bytes_full = 8 * nnz + 4 * (N + 1) + 8 * N * d
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    achieved = alg_bytes / (k_ms * 1e-3) / 1e9
    # dram__bytes of this kernel come from an ncu --set full capture (never from a timed run): the committed figure of the
    # same launch at N = 1; a row shard at N > 1 is a different launch and has no capture, so it reports null
    traffic, traffic_src = None, None
    tpath = os.path.join(ROOT, "profiles", "spmm_traffic.json")
    if os.path.exists(tpath) and world == 1:
        tj = json.load(open(tpath))
        traffic, traffic_src = tj.get(args.shape), tj.get("source")
    roofline = {"kernel": "spmm_stream_kernel<16> (hub-chunk tiles + row tiles in one launch) + hub_finish_kernel = one "
                          "ngcf_spmm call: layer 0 of the step, node-dropout survivors (p = 0.3) compacted"
                          + (f", row shard of rank 0 of {world}" if world > 1 else ""),
                "bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                "frac": round(achieved / peak, 4), "traffic": traffic, "traffic_source": traffic_src,
                "algorithmic_bytes": alg_bytes,
                "entries_gathered": nnz_kept, "kernel_ms": round(k_ms, 5), "peak_source": peak_src,
                "timing": "CUDA events around the call, cold L2 (flushed), mean of 20",
                "l2_gather_tb_s": round(nnz_kept * 4 * d / (k_ms * 1e-3) / 1e12, 2),
                "l2_gather_ceiling_tb_s": 19.6,
                "note": "every entry gathers one 4*d-byte embedding row through L2 (l2_gather_tb_s): that traffic, "
                        "not HBM, bounds the kernel.  l2_gather_ceiling_tb_s = what a kernel that ONLY gathers this "
                        "product's column stream reaches on a B200 (tools/l2_gather_bench.cu, profiles/r02_l2_gather_bench.txt); "
                        "see DESIGN.md section 4",
                "no_dropout": {"kernel_ms": round(k_ms_full, 5), "algorithmic_bytes": alg_bytes_full,
                               "achieved": round(alg_bytes_full / (k_ms_full * 1e-3) / 1e9, 1),
                               "frac": round(alg_bytes_full / (k_ms_full * 1e-3) / 1e9 / peak, 4),
                               "l2_gather_tb_s": round(nnz * 4 * d / (k_ms_full * 1e-3) / 1e12, 2)}}

    clocks = sampler.stop(windows)

    # ---- optional per-entry-point breakdown ------------------------------------------------------------------
    breakdown = None
    if args.breakdown:
        timer = CallTimer(lib)
        _lib._lib = timer
        for j in range(10):
            step(dbatches[j % len(dbatches)])
        agg = timer.table()
        _lib._lib = lib
        breakdown = {k: {"ms_per_step": round(t / 10, 4), "calls_per_step": c / 10} for k, (t, c) in sorted(agg.items())}
        for k, v in breakdown.items():
            log(f"[breakdown] {k:28s} {v['ms_per_step']:8.4f} ms/step  x{v['calls_per_step']:.0f}")

    # ---- extra legs: the other named single-node shapes at this N (BASELINE.json configs 3 / 4) -------------------------
    extra = None
    if not args.no_extra and args.shape == "gowalla":
        extra = {}
        try:
            del gstep_opt
        except NameError:
            pass
        torch.cuda.empty_cache()
        # BASELINE.json configs 4 and 3, and at N = 1 config 0: the reference's own shape (width 65 everywhere, main.py:63-64:
        # the exact-fp32 FFMA dense kernels and the row-per-warp SpMM) with the reference's CPU step beside it
        for shp in ("amazon-book", "yelp2018") + (("seoul",) if world == 1 else ()):
            try:
                extra[shp] = time_shape(pkg, shp, dev, world, rank, steps=args.steps)
                log(f"[bench] extra {shp}: {extra[shp]['ms_per_step']} ms/step")
            except Exception as e:
                extra[shp] = {"error": f"{type(e).__name__}: {e}"}
        if "seoul" in extra and "error" not in extra["seoul"] and not args.no_cpu_baseline:
            try:
                Ls, bs, infos = make_workload("seoul", n_batches=4)
                mods = load_reference_modules()
                if mods is not None:
                    s_cpu, n_cpu = time_reference_modules(mods, Ls, bs, infos, "cpu", 10, 1, 4.0, threads=os.cpu_count() or 1)
                    extra["seoul"]["reference_cpu"] = {"ms_per_step": round(s_cpu * 1e3, 2), "steps": n_cpu,
                                                       "cores": os.cpu_count() or 1, "kind": "reference"}
            except Exception as e:
                log(f"[bench] seoul CPU reference failed ({type(e).__name__}: {e})")

    # ---- CPU baseline beside it ------------------------------------------------------------------------------
    cpu, torch_cuda = None, None
    if not args.no_cpu_baseline and world == 1:
        try:
            torch_cuda = time_torch_cuda(L, batches, info, dev)
            torch_cuda["speedup_of_value"] = round(torch_cuda["ms_per_step"] / ms_per_step, 2)
        except Exception as e:
            log(f"[bench] torch-CUDA baseline failed ({type(e).__name__}: {e})")
        cpu = time_cpu_reference(L, batches, info, max_steps=40, warmup=1, budget_s=15.0)
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
        if rank != 0:
            # no destroy_process_group(): tearing the communicator down while captured CUDA graphs still hold NCCL
            # kernels blocks (observed: hangs until killed); the process simply exits after the final barrier
            sys.stdout.flush()
            os._exit(0)

    spe = info["steps_per_epoch"]
    out = {
        "metric": METRIC, "value": round(ms_per_step * spe / 1e3, 6), "unit": "s/epoch", "n_gpus": world,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": round(ms_per_step, 5),
        "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": info["workload"], "steps_per_epoch": spe},       # the same dict in both arms
        "run": {"nnz": int(L._nnz()), "N": int(L.shape[0]),
                "parallelism": "single GPU" if world == 1 else
                f"row-sharded x{world} ({model.exchange_description()})",
                "row_blocks": None if world == 1 else ("balanced by entries + 32 per row: " + str(shards.starts) if shards
                                                       is not None else "equal"),
                "rng": "device (counter-based hash); node-dropout survivors compacted once per step",
                "l2": f"flushed between timed steps ({L2_FLUSH_BYTES >> 20} MiB write)", "api": api},
        "parity_vs_1gpu": parity,
        "e2e": {"value": round(ms_e2e * spe / 1e3, 6), "unit": "s/epoch", "ms_per_step": round(ms_e2e, 5),
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "last_loss": loss_val},
        "warm_ms_per_step": round(ms_warm, 5),
        "eager": {"ms_per_step": round(ms_eager, 5), "e2e_ms_per_step": round(ms_e2e_eager, 5),
                  "api": "drop-in NGCF.forward + BPR + loss.backward() issued eagerly from Python"},
        "gpu_launches": int(round(launches * args.steps)), "gpu_launches_per_step": launches,
        "gpu_launches_note": "library kernels per step (captured once, replayed per step under GraphedStep)",
        "roofline": roofline, "cpu_baseline": cpu, "torch_cuda_baseline": torch_cuda, "clocks": clocks,
        "training_iteration_with_adam": with_adam,
        "measured_epoch": measured_epoch,
        "extra": extra,
    }
    if breakdown:
        out["breakdown"] = breakdown
    emit(out)
    if world > 1:
        sys.stderr.flush()
        os._exit(0)


# ------------------------------------------------------------------------------------------------------------
# BASELINE.json config 5 and its family: graphs generated on the device per row shard (no host copy exists)
# ------------------------------------------------------------------------------------------------------------
def run_pl(args):
    import torch.distributed as dist
    import seoul_tourism_recommendation_ngcf_b200 as pkg
    from seoul_tourism_recommendation_ngcf_b200 import _lib, plgraph, synth
    from seoul_tourism_recommendation_ngcf_b200.plan import node_dropout_bits, node_dropout_compact, spmm
    from seoul_tourism_recommendation_ngcf_b200.sharded import BalancedShards, RowShards, parity_vs_unsharded
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank, local = int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0"))
    if args.gpus != world:
        raise SystemExit(f"--gpus {args.gpus} needs {args.gpus} ranks (torchrun)")
    balanced = os.environ.get("NGCF_B200_EXCHANGE", "peer") != "nccl" and os.environ.get("NGCF_B200_SHARDS", "balanced") == "balanced"
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl")
    lib = _lib.load()
    n_user, n_item, n_edges, emb, K = synth.SHAPES[args.shape]
    N = n_user + n_item
    nd = synth.num_dict_for(n_user, n_item)
    steps = args.steps
    warm = max(min(args.warmup, 3), 3)

    def fence():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    # ---- N > 1: the sharded step on a device-built shard must be the 1-GPU step (checked on the 1/100-scale graph) -------
    parity = None
    if world > 1:
        pu, pi, pe, _, _ = synth.SHAPES["pl-10m"]
        shp = BalancedShards(pu + pi, world, rank, BalancedShards.cut_bipartite(pu, pi, pe, world)) if balanced \
            else RowShards(pu + pi, world, rank)
        L_full = plgraph.powerlaw_laplacian(pu, pi, pe, dev)
        L_part = plgraph.powerlaw_laplacian(pu, pi, pe, dev, shard=shp)
        pb = {k: torch.from_numpy(v) for k, v in synth.random_batch(pu, pi, BATCH, seed=1).items()}
        res = parity_vs_unsharded(emb, [emb] * K, L_full, synth.num_dict_for(pu, pi), pb, BATCH, dev, node_p=NODE_P,
                                  mess_p=MESS_P, weight_decay=WEIGHT_DECAY, L_shard=L_part, shards=shp)
        worst = torch.tensor([res["out"], res["loss"], res["all_E"], res["worst_grad"]], dtype=torch.float64, device=dev)
        dist.all_reduce(worst, op=dist.ReduceOp.MAX)
        parity = {"out": float(worst[0]), "loss": float(worst[1]), "all_E": float(worst[2]), "worst_grad": float(worst[3]),
                  "tolerance": 1e-5, "what": "pl-10m (the same generator at 1/100 scale): one training step on device-built "
                  "row shards vs the same step on the unsharded device-built graph on each rank's own GPU"}
        log(f"[bench] parity_vs_1gpu (pl-10m): {parity}")
        del L_full, L_part
        torch.cuda.empty_cache()
        if max(parity["out"], parity["loss"], parity["all_E"], parity["worst_grad"]) > 1e-5:
            if rank == 0:
                emit({"metric": METRIC, "error": "row-sharded step differs from the 1-GPU step", "n_gpus": world,
                      "parity_vs_1gpu": parity})
            os._exit(3)

    t0 = time.time()
    sh = None
    if world > 1:
        sh = BalancedShards(N, world, rank, BalancedShards.cut_bipartite(n_user, n_item, n_edges, world)) if balanced \
            else RowShards(N, world, rank)
    csr = plgraph.powerlaw_laplacian(n_user, n_item, n_edges, dev, shard=sh)
    torch.cuda.synchronize()
    t_graph = time.time() - t0
    nnz_tot = torch.tensor([csr.nnz], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(nnz_tot)
    nnz_tot = int(nnz_tot)
    log(f"[bench] rank {rank}: device-built Laplacian shard in {t_graph:.1f}s: rows {csr.n_rows}, nnz {csr.nnz} (all ranks {nnz_tot})")
    torch.manual_seed(0)
    t0 = time.time()
    model = pkg.NGCF(emb, [emb] * K, NODE_P, [MESS_P] * K, 1.0, [csr, csr], nd, BATCH, torch.device("cpu")).to(dev)
    if world > 1:
        model.shard(shards=sh)
    model.train()
    # survivor lists cost 8 B x nnz per layer and direction: past ~40 GB the step uses per-step decision bytes instead
    if csr.nnz * 8 * 2 * K > 40e9:
        model._node_mode = "bits"
    if os.environ.get("NGCF_B200_NODE_MODE"):
        model._node_mode = os.environ["NGCF_B200_NODE_MODE"]       # (A/B runs: the 1-GPU run only fits with "bits")
    crit = pkg.BPR(WEIGHT_DECAY, BATCH)
    batches = [synth.random_batch(n_user, n_item, BATCH, seed=1 + j) for j in range(4)]
    hb = [{k: torch.from_numpy(v).pin_memory() for k, v in b.items()} for b in batches]
    gstep = pkg.GraphedStep(model, crit, BATCH, node_flag=True)
    for j in range(warm):
        gstep(hb[j % len(hb)])
    fence()
    t_plan = time.time() - t0
    sampler = ClockSampler(local)
    sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    w0 = time.time()
    fence()
    db = [{k: (v if k == "year" else v.to(dev)) for k, v in b.items()} for b in hb]
    for j in range(steps):
        ev[j][0].record()
        loss = gstep(db[j % len(db)])
        ev[j][1].record()
    fence()
    windows = [(w0, time.time())]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, loss, model)
    ms = max_over_ranks(sum(a.elapsed_time(b) for a, b in ev)) / steps
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    fence()
    w0 = time.time()
    e0.record()
    last = 0.0
    for j in range(steps):
        last = float(gstep(hb[j % len(hb)]).detach())
    e1.record()
    fence()
    ms_e2e = max_over_ranks(e0.elapsed_time(e1)) / steps
    windows.append((w0, time.time()))
    # roofline: layer 0's product on this rank's shard, exactly as the step runs it
    plan = model._last.plan
    r0 = model._shard.r0 if model._shard else 0
    X = model._packed_table()
    Y = torch.empty(plan.fwd.n_rows, emb, device=dev)
    if model._node_mode == "compact":
        comp, _ = node_dropout_compact(plan.fwd, NODE_P, 1, None, K, r0, as_L=True, as_Lt=False)
        kept = int(comp[0][1].sum())
        run = lambda: spmm(plan.fwd, None, X, emb, out=Y, compact=comp[0])
    else:
        bits, _ = node_dropout_bits(plan.fwd, NODE_P, 1, None, K, r0, as_L=True, as_Lt=False)
        kept = plan.fwd.nnz
        run = lambda: spmm(plan.fwd, None, X, emb, out=Y, keep_bits=bits, layer=0)
    for _ in range(2):
        run()
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(5)]
    torch.cuda.synchronize()
    for a_, b_ in kev:
        a_.record(); run(); b_.record()
    torch.cuda.synchronize()
    k_ms = statistics.mean(a_.elapsed_time(b_) for a_, b_ in kev)
    alg = 8 * kept + 4 * (plan.fwd.n_rows + 1) + 4 * N * emb + 4 * plan.fwd.n_rows * emb
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak = float(json.load(open(peaks_path))["hbm_gbs"]) if os.path.exists(peaks_path) else 6650.0
    clocks = sampler.stop(windows)
    mem = torch.cuda.max_memory_allocated(dev) / 2 ** 30
    fence()
    if rank != 0:
        os._exit(0)
    spe = n_edges // BATCH
    out = {
        "metric": METRIC, "value": round(ms * spe / 1e3, 3), "unit": "s/epoch", "n_gpus": world, "steps": steps, "warmup": warm,
        "ms_per_step": round(ms, 4), "higher_is_better": False, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": f"{args.shape}-shaped synthetic power-law graph (Zipf 0.8) generated on the device per row "
                               f"shard, {n_user} users / {n_item} items / {n_edges} interactions, emb {emb}, {K} layers, "
                               f"batch {BATCH}, node_flag=True, training mode", "steps_per_epoch": spe},
        "run": {"nnz": nnz_tot, "N": N, "parallelism": "single GPU" if world == 1 else
                f"row-sharded x{world} ({model.exchange_description()})",
                "row_blocks": None if world == 1 else (f"balanced by entries + 32 per row: {sh.starts}" if balanced else "equal"),
                "node_dropout": model._node_mode,
                "graph_build_s": round(t_graph, 2), "plan_and_capture_s": round(t_plan, 2),
                "peak_device_memory_gib_rank0": round(mem, 2), "l2": "working set exceeds L2 (no flush needed)",
                "api": "GraphedStep over the drop-in modules; lap_list = device-built CSR row shards (plgraph.py)"},
        "parity_vs_1gpu": parity,
        "e2e": {"value": round(ms_e2e * spe / 1e3, 3), "unit": "s/epoch", "ms_per_step": round(ms_e2e, 4),
                "h2d_bytes_per_step": 8 * BATCH * 8, "d2h_bytes_per_step": 4, "last_loss": last},
        "gpu_launches": int(gstep.launches_per_step * steps), "gpu_launches_per_step": gstep.launches_per_step,
        "roofline": {"kernel": f"ngcf_spmm (streaming kernel), layer 0 of the step on rank 0's row shard, node dropout "
                               f"'{model._node_mode}'", "bound": "hbm", "achieved": round(alg / (k_ms * 1e-3) / 1e9, 1),
                     "peak": peak, "unit": "GB/s", "frac": round(alg / (k_ms * 1e-3) / 1e9 / peak, 4), "traffic": None,
                     "algorithmic_bytes": alg, "entries_gathered": kept, "kernel_ms": round(k_ms, 4),
                     "note": "E (3.8 GB at pl-1b) does not fit L2: every gathered 256-byte row is an HBM access; "
                             "gathered bytes = entries x 256"},
        "cpu_baseline": None, "torch_cuda_baseline": None, "clocks": clocks,
        "note": "the reference cannot build this graph at all (dense N x N Laplacian, matrix.py:55-62); no CPU baseline",
    }
    emit(out)
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)


# ------------------------------------------------------------------------------------------------------------
# a whole measured epoch through the drop-in sampler + GraphedStep(optimizer=Adam)
# ------------------------------------------------------------------------------------------------------------
def run_epoch(pkg, gstep_opt, info, dev):
    """main.py:34-42 + experiment.py:36-60 for ONE epoch: TourDataset(train=True) negatives (device sampler), a
    shuffled drop_last loader of 1024-row HOST batches, and per batch forward + BPR + backward + Adam; the epoch's
    loss sum is read back once at the end (experiment.py:59,62)."""
    from seoul_tourism_recommendation_ngcf_b200 import sampler as S, synth
    from seoul_tourism_recommendation_ngcf_b200.graph import FIELDS
    n_user, n_item, E = info["n_user"], info["n_item"], info["interactions"]
    u, i, _ = synth.powerlaw_bipartite(n_user, n_item, E, alpha=0.8, seed=0)          # the bench graph's edges
    nd = synth.num_dict_for(n_user, n_item)
    rng = np.random.default_rng(5)
    feat = {k: rng.integers(0, nd[c], n_user) for k, c in (("age", "age"), ("sex", "sex"), ("month", "month"),
                                                          ("day", "day"), ("dow", "dayofweek"))}   # id -> features
    cols = {"userid": u.astype(np.int64), "itemid": i.astype(np.int64), "rating": np.ones(E, dtype=np.float32)}
    t0 = time.time()
    ix = S.index_frame(cols, np.arange(n_item), "rating")
    t_index = time.time() - t0
    d = {k: torch.from_numpy(v).to(dev) for k, v in ix.items()}
    user_d, item_d = torch.from_numpy(cols["userid"]).to(dev), torch.from_numpy(cols["itemid"]).to(dev)
    feat_d = {k: torch.from_numpy(v).to(dev) for k, v in feat.items()}
    torch.cuda.synchronize()
    t0 = time.time()
    neg = pkg.sample_negatives(d["pos_ptr"], d["pos_idx"], d["row_user"], d["candidates"], 1, seed=1)[:, 0]
    perm = torch.randperm(E, device=dev)                                              # DataLoader(shuffle=True)
    rows = d["rows"][perm]
    uid = user_d[rows]
    by_field = {"u_id": uid, "pos_item": item_d[rows], "neg_item": neg[perm]}
    by_field.update({k: feat_d[k][uid] for k in feat_d})
    table = torch.stack([by_field[k] for k in FIELDS]).cpu().pin_memory()             # [8, E] host, like the loader's
    t_sample = time.time() - t0
    steps = E // BATCH                                                                # drop_last=True, main.py:39-42
    year = torch.full((BATCH,), 18, dtype=torch.int64)
    losses = torch.zeros(steps, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    t0 = time.time()
    e0.record()
    for s in range(steps):
        b = {k: table[j, s * BATCH:(s + 1) * BATCH] for j, k in enumerate(FIELDS)}
        b["year"] = year
        losses[s] = gstep_opt(b).detach()
    total = float(losses.sum())                                                       # the epoch's one read-back
    e1.record()
    torch.cuda.synchronize()
    wall = time.time() - t0
    ls = losses.cpu().numpy()
    return {"steps": steps, "seconds": round(e0.elapsed_time(e1) / 1e3, 4), "wall_seconds": round(wall, 4),
            "ms_per_step": round(e0.elapsed_time(e1) / steps, 5), "sampler_and_shuffle_seconds": round(t_sample, 4),
            "host_index_seconds": round(t_index, 3), "train_bpr": total / steps,
            "loss_first_50": float(ls[:50].mean()), "loss_last_50": float(ls[-50:].mean()),
            "h2d_bytes_per_step": 8 * BATCH * 8,
            "what": "one full epoch as experiment.py:36-60 runs it: device-sampled negatives (TourDataset), shuffled "
                    "drop_last batches of 1024 from pinned host memory, forward + BPR + backward + Adam(lr=5e-5) per "
                    "batch (GraphedStep), no L2 flush, CUDA events around the whole loop"}


# ------------------------------------------------------------------------------------------------------------
# reference arm / CPU baseline / torch-CUDA bar
# ------------------------------------------------------------------------------------------------------------
def load_reference_modules():
    """(NGCF, BPR) classes of the UNMODIFIED reference from baseline/_ref/model (installed by baseline/install_ref.py at
    build time; it ships to the GPU box), or None when that install is absent."""
    import importlib.util
    from baseline.install_ref import ref_dir
    d = ref_dir()
    if d is None:
        return None
    out = []
    for name, cls in (("NGCF", "NGCF"), ("bprloss", "BPR")):
        spec = importlib.util.spec_from_file_location("ngcf_reference_" + name, os.path.join(d, name + ".py"))
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        out.append(getattr(mod, cls))
    return tuple(out)


def time_reference_modules(mods, L, batches, info, device, max_steps, warmup, budget_s, threads=None):
    """The reference's own training step (experiment.py:45-57: model(...), criterion, zero_grad, backward) issued through
    its unmodified NGCF / BPR modules on ``device``.  emb % 5 != 0 crashes the stock module (NGCF.py:110-114), so — as for
    the golden vectors (SURVEY.md section 8(c)) — the dow table of the INSTANCE is widened to absorb the remainder; the
    reference's forward then runs unmodified."""
    import torch.nn as nn
    from seoul_tourism_recommendation_ngcf_b200 import synth
    RefNGCF, RefBPR = mods
    if threads:
        torch.set_num_threads(threads)
    emb, K = info["emb"], info["layers"]
    dev = torch.device(device)
    torch.manual_seed(0)
    Ld = L.to(dev)
    m = RefNGCF(emb, [emb] * K, NODE_P, [MESS_P] * K, 1.0, [Ld, Ld], synth.num_dict_for(info["n_user"], info["n_item"]),
                BATCH, dev)
    if emb % 5:
        m.dow_emb = nn.Embedding(synth.FEATURE_CARD["dayofweek"], emb - 4 * (emb // 5))
        nn.init.kaiming_uniform_(m.dow_emb.weight)
    m = m.to(dev).train()
    crit = RefBPR(WEIGHT_DECAY, BATCH).to(dev)

    def one(j):
        b = {k: torch.from_numpy(v).to(dev) for k, v in batches[j % len(batches)].items()}
        u, p, n = m(year=b["year"], u_id=b["u_id"], age=b["age"], sex=b["sex"], month=b["month"], day=b["day"],
                    dow=b["dow"], pos_item=b["pos_item"], neg_item=b["neg_item"], node_flag=True)
        m.zero_grad()
        loss = crit(u, p, n)
        loss.backward()
        if dev.type == "cuda":
            torch.cuda.synchronize(dev)
        return loss

    t_start = time.time()
    for j in range(warmup):
        one(j)
    ts = []
    for j in range(max_steps):
        t0 = time.time()
        one(warmup + j)
        ts.append(time.time() - t0)
        if time.time() - t_start > budget_s and len(ts) >= 1:
            break
    return statistics.mean(ts), len(ts)


def time_cpu_reference(L, batches, info, max_steps, warmup, budget_s):
    """CPU arm: the unmodified reference modules when installed (kind "reference"), else the oracle port ("port")."""
    mods = None
    try:
        mods = load_reference_modules()
    except Exception as e:
        log(f"[bench] reference modules not loadable ({type(e).__name__}: {e}); using the oracle port")
    if mods is None:
        return time_oracle(L, batches, info, max_steps, warmup, budget_s)
    cores = os.cpu_count() or 1
    s, n = time_reference_modules(mods, L, batches, info, "cpu", max_steps, warmup, budget_s, threads=cores)
    single = None
    if cores > 1:                    # the reference's COO SpMM does not scale with threads (SURVEY.md section 8(d))
        s1, _ = time_reference_modules(mods, L, batches, info, "cpu", 2, 0, 1e9, threads=1)
        torch.set_num_threads(cores)
        single = {"ms_per_step": round(s1 * 1e3, 2), "cores": 1, "sample": "mean of 2 steps"}
    return {"value": round(s * info["steps_per_epoch"], 3), "unit": "s/epoch", "ms_per_step": round(s * 1e3, 2),
            "cores": cores, "kind": "reference", "steps": n, "single_thread": single,
            "sample": f"{n} full training steps (of {info['steps_per_epoch']} per epoch) of the same workload, {warmup} "
                      f"warm-up; the reference's unmodified NGCF.py / bprloss.py (baseline/_ref) on device='cpu': "
                      f"torch.sparse COO mm + host float64 node-dropout mask + autograd"}


def time_torch_cuda(L, batches, info, dev, steps=20, warmup=3):
    """SURVEY.md section 8(d): "the reference on the same B200 (device='cuda', cuSPARSE path) - the bar the kernels must
    beat".  The unmodified reference modules on the GPU when installed and runnable there, else the oracle's restatement
    of the same torch calls with its tensors on the GPU."""
    try:
        mods = load_reference_modules()
        if mods is not None:
            s, n = time_reference_modules(mods, L, batches, info, dev, steps, warmup, 60.0)
            return {"ms_per_step": round(s * 1e3, 4), "value": round(s * info["steps_per_epoch"], 4), "unit": "s/epoch",
                    "kind": "reference", "steps": n,
                    "what": "the reference's unmodified NGCF.py / bprloss.py with device='cuda' (lap_list resident on the "
                            "GPU): host float64 node mask + index ops, coalesce + cusparse SpMM, cuBLAS Linear, autograd; "
                            "wall clock per step with a device sync, same batches and shapes as `value`"}
    except Exception as e:
        log(f"[bench] reference modules on cuda failed ({type(e).__name__}: {e}); timing the oracle restatement on cuda")
    from oracle import ngcf_oracle as O
    model = make_model(info, L, torch.device("cpu"))
    params = {k: v.detach().clone().to(dev) for k, v in model.state_dict().items()}
    K, N = info["layers"], info["n_user"] + info["n_item"]
    Ld = L.to(dev)
    ts = []
    for j in range(warmup + steps):
        b = {k: torch.from_numpy(v).to(dev) for k, v in batches[j % len(batches)].items()}
        t0 = time.time()
        keep, mult = O.reference_dropout_draws(L._nnz(), N, [info["emb"]] * K, NODE_P, [MESS_P] * K, True, True)
        keep = [k_.to(dev) for k_ in keep] if keep is not None else None
        mult = [m_.to(dev) for m_ in mult] if mult is not None else None
        O.train_step(params, Ld, b, emb_ratio=1.0, weight_decay=WEIGHT_DECAY, batch_size_ctor=BATCH, edge_keep=keep,
                     mess_mult=mult)
        torch.cuda.synchronize(dev)
        if j >= warmup:
            ts.append(time.time() - t0)
    s = statistics.mean(ts)
    return {"ms_per_step": round(s * 1e3, 4), "value": round(s * info["steps_per_epoch"], 4), "unit": "s/epoch",
            "kind": "port", "steps": len(ts),
            "what": "oracle/ngcf_oracle.py (the reference's torch calls, line by line) with its tensors on the GPU"}


def time_oracle(L, batches, info, max_steps, warmup, budget_s):
    from oracle import ngcf_oracle as O
    torch.set_num_threads(os.cpu_count() or 1)
    model = make_model(info, L, torch.device("cpu"))
    params = {k: v.detach().clone() for k, v in model.state_dict().items()}
    K, N = info["layers"], info["n_user"] + info["n_item"]
    dims = [info["emb"]] * K

    def one(j):
        b = {k: torch.from_numpy(v) for k, v in batches[j % len(batches)].items()}
        keep, mult = O.reference_dropout_draws(L._nnz(), N, dims, NODE_P, [MESS_P] * K, True, True)
        O.train_step(params, L, b, emb_ratio=1.0, weight_decay=WEIGHT_DECAY, batch_size_ctor=BATCH,
                     edge_keep=keep, mess_mult=mult)

    t_start = time.time()
    for j in range(warmup):
        one(j)
    ts = []
    for j in range(max_steps):
        t0 = time.time()
        one(warmup + j)
        ts.append(time.time() - t0)
        if time.time() - t_start > budget_s and len(ts) >= 1:
            break
    s = statistics.mean(ts)
    cores = torch.get_num_threads()
    # the reference's COO SpMM does not scale with threads (SURVEY.md section 8(d)): a short single-thread sample too
    single = None
    if cores > 1:
        torch.set_num_threads(1)
        t1 = []
        for j in range(2):
            t0 = time.time()
            one(warmup + len(ts) + j)
            t1.append(time.time() - t0)
        torch.set_num_threads(cores)
        single = {"ms_per_step": round(min(t1) * 1e3, 2), "cores": 1, "sample": "best of 2 steps"}
    return {"value": round(s * info["steps_per_epoch"], 3), "unit": "s/epoch", "ms_per_step": round(s * 1e3, 2),
            "cores": cores, "kind": "port", "steps": len(ts), "single_thread": single,
            "sample": f"{len(ts)} full training steps (of {info['steps_per_epoch']} per epoch) of the same workload, "
                      f"{warmup} warm-up; oracle/ngcf_oracle.py = the reference's torch.sparse CPU path incl. its host "
                      f"float64 node-dropout mask"}


def run_reference(args):
    if int(os.environ.get("RANK", "0")) != 0:
        return
    if args.shape.startswith("pl-"):
        emit({"impl": "reference", "unavailable": "the reference builds its Laplacian through dense N x N arrays "
              "(matrix.py:55-62) and cannot hold this graph; no CPU run exists for the device-generated pl-* shapes"})
        return
    L, batches, info = make_workload(args.shape)
    warmup = min(args.warmup, 2)
    res = time_cpu_reference(L, batches, info, max_steps=args.steps, warmup=warmup, budget_s=float("inf"))
    spe = info["steps_per_epoch"]
    out = {"impl": "reference", "metric": METRIC, "value": res["value"], "unit": "s/epoch", "n_gpus": args.gpus,
           "steps": res["steps"], "warmup": warmup, "ms_per_step": res["ms_per_step"], "higher_is_better": False,
           "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": info["workload"], "steps_per_epoch": spe},
           "run": {"device": "cpu", "kind": res["kind"], "cores": res["cores"]},
           "cpu_baseline": res,
           "e2e": {"value": res["value"], "unit": "s/epoch", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
           "gpu_launches": 0}
    emit(out)


if __name__ == "__main__":
    a = parse_args()
    protect_stdout()
    if a.impl == "reference":
        run_reference(a)
    elif a.shape.startswith("pl-"):
        run_pl(a)
    else:
        run_ours(a)
