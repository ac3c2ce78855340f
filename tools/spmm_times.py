"""SpMM-only timings (CUDA events, warm and cold L2) for A/B builds:  NGCF_B200_LIB=... python tools/spmm_times.py [shape]"""
import os, sys, statistics
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import bench
from seoul_tourism_recommendation_ngcf_b200 import _lib
from seoul_tourism_recommendation_ngcf_b200.plan import LaplacianPlan, node_dropout_compact, spmm

shape = sys.argv[1] if len(sys.argv) > 1 else "gowalla"
L, batches, info = bench.make_workload(shape)
dev = torch.device("cuda:0")
lib = _lib.load()
plan = LaplacianPlan(L, dev)
N, d = plan.N, info["emb"]
X = torch.randn(N, d, device=dev); Y = torch.empty(N, d, device=dev); S = torch.randn(N, d, device=dev)
flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)

def t(name, fn, reps=30):
    for _ in range(3): fn()
    out = {}
    for mode in ("warm", "cold"):
        ev = []
        for _ in range(reps):
            if mode == "cold": flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record(); ev.append((e0, e1))
        torch.cuda.synchronize()
        out[mode] = statistics.median(a.elapsed_time(b) for a, b in ev) * 1e3
    print(f"{name:44s} warm {out['warm']:8.1f} us   cold {out['cold']:8.1f} us", flush=True)

tag = os.environ.get("NGCF_B200_LIB", "default").split("libngcf_")[-1]
print(f"== {tag}: tiles {plan.fwd.tiles.shape[0]} + {0 if plan.fwd.chunk_tiles is None else plan.fwd.chunk_tiles.shape[0]} chunk tiles, "
      f"tile {lib.ngcf_spmm_tile_rows()} rows / {lib.ngcf_spmm_tile_entries()} entries")
t("spmm (no dropout)", lambda: spmm(plan.fwd, None, X, d, out=Y))
cl, ct = node_dropout_compact(plan.fwd, 0.3, 1, None, 3, as_L=True, as_Lt=True)
t("spmm (compacted survivors, layer 0)", lambda: spmm(plan.fwd, None, X, d, out=Y, compact=cl[0]))
t("spmm transposed + addend (compacted, layer 1)", lambda: spmm(plan.fwd, None, X, d, out=Y, addend=S, transposed=True, compact=ct[1]))
t("node_dropout_compact (L and L^T, 3 layers)", lambda: node_dropout_compact(plan.fwd, 0.3, 1, None, 3, as_L=True, as_Lt=True))
