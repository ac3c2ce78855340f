"""Per-entry-point device times at a named shape (CUDA events, warm L2 and cold L2), for DESIGN.md / profiles.
  python tools/kernel_times.py [shape]"""
import os, sys, statistics
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import bench
from seoul_tourism_recommendation_ngcf_b200 import _lib
from seoul_tourism_recommendation_ngcf_b200.plan import LaplacianPlan, node_dropout_bits, node_dropout_compact, spmm

shape = sys.argv[1] if len(sys.argv) > 1 else "gowalla"
L, batches, info = bench.make_workload(shape)
dev = torch.device("cuda:0")
lib = _lib.load()
plan = LaplacianPlan(L, dev)
N, d = plan.N, info["emb"]
st = torch.cuda.current_stream().cuda_stream
X = torch.randn(N, d, device=dev); Y = torch.empty(N, d, device=dev); S = torch.randn(N, d, device=dev)
E_out = torch.randn(N, d, device=dev); gE = torch.randn(N, d, device=dev)
W1 = torch.randn(d, d, device=dev) * 0.1; W2 = torch.randn(d, d, device=dev) * 0.1
b1 = torch.randn(d, device=dev); b2 = torch.randn(d, device=dev)
wcat = torch.empty(2 * d * d, device=dev); bias = torch.empty(d, device=dev)
lib.ngcf_pack_weights(W1.data_ptr(), b1.data_ptr(), W2.data_ptr(), b2.data_ptr(), d, d, wcat.data_ptr(), bias.data_ptr(), st)
gS = torch.empty(N, d, device=dev); gEl = torch.empty(N, d, device=dev); gM = torch.empty(N, d, device=dev)
gW1 = torch.zeros(d, d, device=dev); gW2 = torch.zeros(d, d, device=dev); gb1 = torch.zeros(d, device=dev); gb2 = torch.zeros(d, device=dev)
slot = torch.full((N,), -1, dtype=torch.int32, device=dev)
rows = torch.randperm(N, device=dev)[:3000]; slot[rows] = torch.arange(3000, dtype=torch.int32, device=dev)
gsum = torch.randn(3000, 4 * d, device=dev)
bl, bt = node_dropout_bits(plan.fwd, 0.3, 1, None, 3, as_L=True, as_Lt=True)
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

t("spmm (no dropout)", lambda: spmm(plan.fwd, None, X, d, out=Y))
t("spmm (in-kernel Philox dropout)", lambda: spmm(plan.fwd, None, X, d, out=Y, drop_p=0.3, seed=1, layer=1))
t("spmm (precomputed dropout bits)", lambda: spmm(plan.fwd, None, X, d, out=Y, layer=1, keep_bits=bl))
t("spmm transposed + addend (bits)", lambda: spmm(plan.fwd, None, X, d, out=Y, addend=S, layer=1, transposed=True, keep_bits=bt))
cl, ct = node_dropout_compact(plan.fwd, 0.3, 1, None, 3, as_L=True, as_Lt=True)
for k in range(3):
    t(f"spmm (compacted survivors, layer {k})", lambda: spmm(plan.fwd, None, X, d, out=Y, compact=cl[k]))
t("spmm transposed + addend (compacted, layer 1)", lambda: spmm(plan.fwd, None, X, d, out=Y, addend=S, transposed=True, compact=ct[1]))
t("node_dropout_compact (L and L^T, 3 layers)", lambda: node_dropout_compact(plan.fwd, 0.3, 1, None, 3, as_L=True, as_Lt=True))
t("node_dropout_bits (L and L^T)", lambda: node_dropout_bits(plan.fwd, 0.3, 1, None, 3, as_L=True, as_Lt=True))
t("dense_fwd (mess_p 0.1)", lambda: lib.ngcf_dense_fwd(S.data_ptr(), X.data_ptr(), N, d, d, wcat.data_ptr(), bias.data_ptr(), 0.2, None, None, 0.1, 1, None, 0, 0, Y.data_ptr(), st))
t("dense_fwd (no dropout)", lambda: lib.ngcf_dense_fwd(S.data_ptr(), X.data_ptr(), N, d, d, wcat.data_ptr(), bias.data_ptr(), 0.2, None, None, 0.0, 1, None, 0, 0, Y.data_ptr(), st))
t("dense_bwd + wgrad (mess_p 0.1)", lambda: lib.ngcf_dense_bwd(gE.data_ptr(), slot.data_ptr(), gsum.data_ptr(), 4 * d, d, E_out.data_ptr(), S.data_ptr(), X.data_ptr(), N, d, d, W1.data_ptr(), W2.data_ptr(), 0.2, None, None, 0.1, 1, None, 0, 0, 1, gS.data_ptr(), gEl.data_ptr(), gW1.data_ptr(), gb1.data_ptr(), gW2.data_ptr(), gb2.data_ptr(), gM.data_ptr(), st))
# the FFMA kernels: what runs at widths the tensor-core kernels do not take, such as the reference's own 65
w = 65
S6, X6, E6, gE6 = (torch.randn(N, w, device=dev) for _ in range(4))
Y6, gS6, gEl6, gM6 = (torch.empty(N, w, device=dev) for _ in range(4))
W1_6 = torch.randn(w, w, device=dev) * 0.1; W2_6 = torch.randn(w, w, device=dev) * 0.1
b1_6 = torch.randn(w, device=dev); b2_6 = torch.randn(w, device=dev)
wcat6 = torch.empty(2 * w * w, device=dev); bias6 = torch.empty(w, device=dev)
lib.ngcf_pack_weights(W1_6.data_ptr(), b1_6.data_ptr(), W2_6.data_ptr(), b2_6.data_ptr(), w, w, wcat6.data_ptr(), bias6.data_ptr(), st)
gW1_6 = torch.zeros(w, w, device=dev); gW2_6 = torch.zeros(w, w, device=dev); gb1_6 = torch.zeros(w, device=dev); gb2_6 = torch.zeros(w, device=dev)
gsum6 = torch.randn(3000, 4 * w, device=dev)
t("dense_fwd FFMA, width 65 (mess_p 0.1)", lambda: lib.ngcf_dense_fwd(S6.data_ptr(), X6.data_ptr(), N, w, w, wcat6.data_ptr(), bias6.data_ptr(), 0.2, None, None, 0.1, 1, None, 0, 0, Y6.data_ptr(), st))
t("dense_bwd FFMA, width 65 (mess_p 0.1)", lambda: lib.ngcf_dense_bwd(gE6.data_ptr(), slot.data_ptr(), gsum6.data_ptr(), 4 * w, w, E6.data_ptr(), S6.data_ptr(), X6.data_ptr(), N, w, w, W1_6.data_ptr(), W2_6.data_ptr(), 0.2, None, None, 0.1, 1, None, 0, 0, 1, gS6.data_ptr(), gEl6.data_ptr(), gW1_6.data_ptr(), gb1_6.data_ptr(), gW2_6.data_ptr(), gb2_6.data_ptr(), gM6.data_ptr(), st))
