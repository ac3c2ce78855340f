"""XSimGCL's captured training step against LightGCN's at the same batch and against a torch fp32 XSimGCL written the
SELFRec way, with the split of the XSimGCL step, all measured in one run, on the Gowalla-, Yelp2018- and
Amazon-Book-shaped synthetic graphs at embedding 64, 3 layers, batch 2048 (XSimGCL's usual batch), BPR loss, Adam:

  xsimgcl     GraphedStep(XSimGCL(eps=0.2, cl_weight=0.2, cl_layer=1, temperature=0.2), BPR, optimizer=ngcf_b200.Adam)
  lightgcn    GraphedStep(LightGCN without node dropout, BPR, optimizer=ngcf_b200.Adam)
  torch       XSimGCL in torch fp32 as SELFRec writes it: torch.sparse.mm, rand_like + F.normalize noise per layer,
              torch.unique for the contrastive rows, InfoNCE with F.normalize and log_softmax, BPR, autograd and
              torch.optim.Adam (eager)
  split       the pieces of one XSimGCL step, each captured in a CUDA graph of its own and replayed: the 2K = 6
              propagation products (K forward, K transposed; the transposed ones add the batch rows' gradients through a
              slot map of the batch, layer cl_layer's from the gsum copy that holds H), the K noise kernels, the two
              InfoNCE calls (users, positive items; forward + gradients), and the row-gradient plumbing of the backward
              (scatter, dense last-layer gradient, the view-2 add, reset); "rest" is the step minus these: the readouts,
              the loss, autograd's small kernels and Adam

CUDA events, medians of alternated calls after warm-up, no L2 flush (operands are read warm, as in a training loop).
Prints the card and its power limit read in the same run.
python tools/xsimgcl_time.py [--reps N] [--out PATH]"""
import argparse
import ctypes
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
import torch.nn.functional as F

import seoul_tourism_recommendation_ngcf_b200 as pkg
from seoul_tourism_recommendation_ngcf_b200 import _lib, laplacian, synth
from seoul_tourism_recommendation_ngcf_b200.NGCF import _RowGrads
from seoul_tourism_recommendation_ngcf_b200.plan import spmm

dev = torch.device("cuda:0")
EMB, K, B, EPS, CL_W, CL_LAYER, TAU, WD, LR = 64, 3, 2048, 0.2, 0.2, 1, 0.2, 1e-4, 1e-3


def timed(fns, reps):
    """medians (ms) of each fn in fns, called alternately"""
    for fn in fns:
        for _ in range(3):
            fn()
    ev = [[] for _ in fns]
    for _ in range(reps):
        for j, fn in enumerate(fns):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            ev[j].append((e0, e1))
    torch.cuda.synchronize()
    return [statistics.median(a.elapsed_time(b) for a, b in e) for e in ev]


def graphed(fn):
    """fn captured once in a CUDA graph (after a warm-up call); returns the replay, which keeps fn alive: the graph
    reads and writes the buffers fn's closure owns, and once they were freed a replay would write into memory the
    allocator has handed to other tensors"""
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fn()
    torch.cuda.current_stream().wait_stream(s)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        fn()

    def replay():
        g.replay()
    replay.fn = fn
    return replay


class TorchXSimGCL:
    """fp32 torch XSimGCL with torch.optim.Adam, after SELFRec's XSimGCL encoder and cal_cl_loss"""

    def __init__(self, L, n_user, n_item):
        Lc = L.coalesce().to(dev)
        self.L = torch.sparse_coo_tensor(Lc.indices(), Lc.values().float(), Lc.shape).to_sparse_csr()
        self.N, self.n_user = n_user + n_item, n_user
        g = torch.Generator(device="cpu").manual_seed(0)
        self.emb = (torch.randn(self.N, EMB, generator=g) * 0.1).to(dev).requires_grad_(True)
        self.opt = torch.optim.Adam([self.emb], lr=LR)

    @staticmethod
    def info_nce(a, b):
        a, b = F.normalize(a, dim=1), F.normalize(b, dim=1)
        return -torch.diag(F.log_softmax(a @ b.T / TAU, dim=1)).mean()

    def step(self, u, p, n):
        E, layers = self.emb, []
        for k in range(K):
            E = torch.sparse.mm(self.L, E)
            E = E + torch.sign(E) * F.normalize(torch.rand_like(E), dim=-1) * EPS
            layers.append(E)
        Fr = torch.stack(layers, 1).mean(1)
        V2 = layers[CL_LAYER - 1]
        ur, pr, nr = Fr[u], Fr[self.n_user + p], Fr[self.n_user + n]
        x = (ur * pr).sum(1) - (ur * nr).sum(1)
        rec = (-F.logsigmoid(x).sum() + WD * ((ur * ur).sum() + (pr * pr).sum() + (nr * nr).sum())) / B
        uu, ii = torch.unique(u), torch.unique(p) + self.n_user
        cl = CL_W * (self.info_nce(Fr[uu], V2[uu]) + self.info_nce(Fr[ii], V2[ii]))
        loss = rec + cl
        self.opt.zero_grad()
        loss.backward()
        self.opt.step()
        return loss


def pieces(m):
    """the split of m's last (eager) step: products, noise kernels, the two InfoNCE calls and the row-gradient plumbing,
    each as a function"""
    lib = _lib.load()
    st = m._last
    N = m.n_user + m.n_item
    fwd, bwd = st.plan.fwd, st.plan.side(True, False)
    grads = [torch.randn(r.numel(), EMB, device=dev) for r in st.rows]
    # the products' slot map of the batch rows, built once and kept (the step's own map is reset by its backward)
    slot = torch.full((N,), -1, dtype=torch.int32, device=dev)
    gsum = torch.empty(sum(r.numel() for r in st.rows), EMB, device=dev)
    _lib.check(lib.ngcf_rowgrad_scatter(_lib.ptr_array(st.rows), _lib.i64_array(st.offsets), _lib.ptr_array(grads),
                                        _lib.i64_array([r.numel() for r in st.rows]), len(st.rows), EMB,
                                        slot.data_ptr(), gsum.data_ptr(), _lib.current_stream()), "rowgrad_scatter")
    gsum_cl = gsum + 1.0
    layers = [e.clone() for e in st.E[1:]]

    def products():
        for k in range(K):
            spmm(fwd, None, st.E[k], EMB)
        for k in range(K - 1, -1, -1):
            addend = dict(slot=slot, gsum=gsum_cl if k == CL_LAYER else gsum) if k >= 1 else {}
            spmm(bwd, None, st.E[k + 1], EMB, **addend)

    def rowgrads():
        rg = _RowGrads(m, st, grads, len(st.rows), EMB, N)
        gE = torch.empty(N, EMB, device=dev)
        _lib.check(lib.ngcf_rowgrad_expand(rg.slot.data_ptr(), N, rg.gsum.data_ptr(), EMB, EMB, 1.0 / K, gE.data_ptr(),
                                           EMB, _lib.current_stream()), "rowgrad_expand")
        g_cl = rg.gsum.clone()
        _lib.check(lib.ngcf_rowgrad_add(_lib.ptr_array(st.rows[:2]), _lib.i64_array(st.offsets[:2]),
                                        _lib.ptr_array(grads[:2]), _lib.i64_array([B, B]), 2, EMB, rg.slot.data_ptr(),
                                        g_cl.data_ptr(), EMB, _lib.current_stream()), "rowgrad_add")
        rg.reset()

    def noise():
        for k in range(K):
            _lib.check(lib.ngcf_perturb_rows(layers[k].data_ptr(), N, EMB, EMB, EPS, st.seed, None, k + 1,
                                             _lib.current_stream()), "perturb_rows")

    x1 = [torch.randn(B, EMB, device=dev) for _ in range(2)]
    x2 = [x + 0.1 * torch.randn_like(x) for x in x1]
    ids = [st.rows[0], st.rows[1]]
    ws_bytes = ctypes.c_size_t()
    _lib.check(lib.ngcf_infonce_workspace(B, EMB, ctypes.byref(ws_bytes)), "infonce_workspace")
    ws = torch.empty(ws_bytes.value, dtype=torch.uint8, device=dev)
    loss = torch.empty((), device=dev)
    g1, g2 = torch.empty(B, EMB, device=dev), torch.empty(B, EMB, device=dev)

    def infonce():
        for j in range(2):
            _lib.check(lib.ngcf_infonce(x1[j].data_ptr(), x2[j].data_ptr(), B, EMB, ids[j].data_ptr(), TAU,
                                        loss.data_ptr(), g1.data_ptr(), g2.data_ptr(), ws.data_ptr(), ws_bytes.value,
                                        _lib.current_stream()), "infonce")
    return products, noise, infonce, rowgrads


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                                  "profiles", "r07_xsimgcl_time.txt"))
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    say(f"card: {torch.cuda.get_device_name(0)}; nvidia-smi (name, power limit, max SM clock): {q[0] if q else '?'}")
    say(f"emb {EMB}, {K} layers, batch {B}, XSimGCL eps {EPS} cl_weight {CL_W} cl_layer {CL_LAYER} temperature {TAU}, "
        f"LightGCN without node dropout, BPR, Adam; medians of {args.reps} alternated calls, times in us")
    for shape in ("gowalla", "yelp2018", "amazon-book"):
        n_user, n_item, n_inter, _, _ = synth.SHAPES[shape]
        ui, ii, ri = synth.powerlaw_bipartite(n_user, n_item, n_inter, alpha=0.8, seed=0)
        L = laplacian.laplacian_coo(ui, ii, ri, n_user, n_item)
        nd = synth.num_dict_for(n_user, n_item)
        batch = {k: torch.from_numpy(v) for k, v in synth.random_batch(n_user, n_item, B, seed=1).items()}
        torch.manual_seed(0)
        xs = pkg.XSimGCL(EMB, K, [L, L], nd, eps=EPS, cl_weight=CL_W, cl_layer=CL_LAYER, temperature=TAU).to(dev)
        s_xs = pkg.GraphedStep(xs, pkg.BPR(WD, B), B, optimizer=pkg.Adam(xs.parameters(), lr=LR))
        torch.manual_seed(0)
        lg = pkg.LightGCN(EMB, K, [L, L], nd).to(dev)
        s_lg = pkg.GraphedStep(lg, pkg.BPR(WD, B), B, optimizer=pkg.Adam(lg.parameters(), lr=LR))
        tx = TorchXSimGCL(L, n_user, n_item)
        u, p, n = (batch[k].to(dev) for k in ("u_id", "pos_item", "neg_item"))
        # one eager forward of a second XSimGCL leaves a step's plan, layers and batch rows for the split
        xs1 = pkg.XSimGCL(EMB, K, [L, L], nd, eps=EPS, cl_weight=CL_W, cl_layer=CL_LAYER, temperature=TAU).to(dev)
        d = {k: v.to(dev) for k, v in batch.items()}
        with torch.no_grad():
            xs1(d["year"], d["u_id"], d["age"], d["sex"], d["month"], d["day"], d["dow"], d["pos_item"], d["neg_item"],
                True)
        p_prod, p_noise, p_nce, p_rg = (graphed(f) for f in pieces(xs1))
        t_xs, t_lg, t_torch, t_prod, t_noise, t_nce, t_rg = timed(
            [lambda: s_xs(batch), lambda: s_lg(batch), lambda: tx.step(u, p, n), p_prod, p_noise, p_nce, p_rg],
            args.reps)
        t_rest = t_xs - t_prod - t_noise - t_nce - t_rg
        nnz = xs._last.plan.nnz
        say(f"{shape:11s} ({n_user} users, {n_item} items, nnz(L) {nnz}): XSimGCL step {t_xs * 1e3:7.1f} "
            f"({s_xs.launches_per_step} launches), LightGCN step {t_lg * 1e3:7.1f} ({s_lg.launches_per_step} launches), "
            f"torch fp32 XSimGCL {t_torch * 1e3:8.1f} ({t_torch / t_xs:.1f}x); split of the XSimGCL step: "
            f"{2 * K} products {t_prod * 1e3:6.1f} ({100 * t_prod / t_xs:.0f}%), {K} noise kernels {t_noise * 1e3:5.1f} "
            f"({100 * t_noise / t_xs:.0f}%), 2 InfoNCE calls {t_nce * 1e3:6.1f} ({100 * t_nce / t_xs:.0f}%), row-gradient "
            f"plumbing {t_rg * 1e3:5.1f} ({100 * t_rg / t_xs:.0f}%), rest {t_rest * 1e3:6.1f} ({100 * t_rest / t_xs:.0f}%)")
        del s_xs, s_lg, xs, xs1, lg, tx, p_prod, p_noise, p_nce, p_rg
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
