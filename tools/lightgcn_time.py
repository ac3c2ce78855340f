"""LightGCN's captured training step against NGCF's on the same graph and against a torch fp32 LightGCN, all measured in
one run, on the Gowalla-, Yelp2018- and Amazon-Book-shaped synthetic graphs at embedding 64, 3 layers, batch 1024, node
dropout 0.3 (bench.py's; NGCF also runs its message dropout 0.1), BPR loss, Adam:

  lightgcn    GraphedStep(LightGCN, BPR, optimizer=ngcf_b200.Adam)
  ngcf        GraphedStep(NGCF, BPR, optimizer=ngcf_b200.Adam)
  torch       the same LightGCN in torch fp32: per layer a CSR of L with this step's cumulative node-dropout mask on its
              values, torch.sparse.mm, the layer mean, the BPR loss, autograd and torch.optim.Adam (eager)
  products    the 2K = 6 propagation products of one LightGCN step alone (K forward products on a step's compacted L
              survivors, K transposed ones on its L^T survivors), to give their share of the step

CUDA events, medians of alternated calls after warm-up, no L2 flush (operands are read warm, as in a training loop).
Prints the card and its power limit read in the same run.
python tools/lightgcn_time.py [--reps N] [--out PATH]"""
import argparse
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import seoul_tourism_recommendation_ngcf_b200 as pkg
from seoul_tourism_recommendation_ngcf_b200 import laplacian, synth
from seoul_tourism_recommendation_ngcf_b200.plan import spmm

dev = torch.device("cuda:0")
EMB, K, B, NODE_P, MESS_P, WD, LR = 64, 3, 1024, 0.3, 0.1, 1e-4, 1e-3


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


class TorchLightGCN:
    """fp32 torch LightGCN with torch.optim.Adam: the comparison point a user without this library would write."""

    def __init__(self, L, n_user, n_item):
        Lc = L.coalesce().to(dev)
        csr = torch.sparse_coo_tensor(Lc.indices(), Lc.values().float(), Lc.shape).to_sparse_csr()
        self.crow, self.col, self.val = csr.crow_indices(), csr.col_indices(), csr.values()
        self.N, self.n_user = n_user + n_item, n_user
        g = torch.Generator(device="cpu").manual_seed(0)
        self.emb = (torch.randn(self.N, EMB, generator=g) * 0.1).to(dev).requires_grad_(True)
        self.opt = torch.optim.Adam([self.emb], lr=LR)

    def step(self, u, p, n):
        keep = torch.ones_like(self.val, dtype=torch.bool)
        E, acc = self.emb, self.emb
        for _ in range(K):
            keep = keep & (torch.rand_like(self.val) >= NODE_P)              # cumulative node dropout, unscaled
            Lk = torch.sparse_csr_tensor(self.crow, self.col, self.val * keep, (self.N, self.N))
            E = torch.sparse.mm(Lk, E)
            acc = acc + E
        F = acc / (K + 1)
        ur, pr, nr = F[u], F[self.n_user + p], F[self.n_user + n]
        x = (ur * pr).sum(1).abs() - (ur * nr).sum(1).abs()
        loss = (-torch.nn.functional.logsigmoid(x).sum() + WD * ((ur * ur).sum() + (pr * pr).sum() + (nr * nr).sum())) / B
        self.opt.zero_grad()
        loss.backward()
        self.opt.step()
        return loss


def products(m):
    """the 2K products of m's last step, on its own compacted survivors, outputs into fresh buffers"""
    st = m._last
    fwd, bwd = st.plan.fwd, st.plan.side(True, False)
    slot = m._slot_map(m.n_user + m.n_item, dev)
    gsum = torch.zeros(3 * B, EMB, device=dev)

    def run():
        for k in range(K):
            spmm(fwd, None, st.E[k], EMB, **st.dropout.args(k))
        for k in range(K - 1, -1, -1):
            spmm(bwd, None, st.E[k + 1], EMB, slot=slot, gsum=gsum, **st.dropout.args(k, transposed=True))
    return run


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                                  "profiles", "r06_lightgcn_time.txt"))
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    say(f"card: {torch.cuda.get_device_name(0)}; nvidia-smi (name, power limit, max SM clock): {q[0] if q else '?'}")
    say(f"emb {EMB}, {K} layers, batch {B}, node dropout {NODE_P} (NGCF: message dropout {MESS_P} too), BPR, Adam; "
        f"medians of {args.reps} alternated calls, times in us")
    for shape in ("gowalla", "yelp2018", "amazon-book"):
        n_user, n_item, n_inter, _, _ = synth.SHAPES[shape]
        ui, ii, ri = synth.powerlaw_bipartite(n_user, n_item, n_inter, alpha=0.8, seed=0)
        L = laplacian.laplacian_coo(ui, ii, ri, n_user, n_item)
        nd = synth.num_dict_for(n_user, n_item)
        batch = {k: torch.from_numpy(v) for k, v in synth.random_batch(n_user, n_item, B, seed=1).items()}
        torch.manual_seed(0)
        lg = pkg.LightGCN(EMB, K, [L, L], nd, node_dropout=NODE_P).to(dev).train()
        s_lg = pkg.GraphedStep(lg, pkg.BPR(WD, B), B, optimizer=pkg.Adam(lg.parameters(), lr=LR))
        torch.manual_seed(0)
        ng = pkg.NGCF(EMB, [EMB] * K, NODE_P, [MESS_P] * K, 1.0, [L, L], nd, B, dev).to(dev).train()
        s_ng = pkg.GraphedStep(ng, pkg.BPR(WD, B), B, optimizer=pkg.Adam(ng.parameters(), lr=LR))
        tl = TorchLightGCN(L, n_user, n_item)
        u, p, n = (batch[k].to(dev) for k in ("u_id", "pos_item", "neg_item"))
        # one forward of a second LightGCN leaves a step's survivors (L is symmetric: for L^T too) and layers in its
        # _last for the products alone
        lg1 = pkg.LightGCN(EMB, K, [L, L], nd, node_dropout=NODE_P).to(dev).train()
        d = {k: v.to(dev) for k, v in batch.items()}
        with torch.no_grad():
            lg1(d["year"], d["u_id"], d["age"], d["sex"], d["month"], d["day"], d["dow"], d["pos_item"], d["neg_item"],
                True)
        t_lg, t_ng, t_torch, t_prod = timed([lambda: s_lg(batch), lambda: s_ng(batch), lambda: tl.step(u, p, n),
                                             products(lg1)], args.reps)
        nnz = lg._last.plan.nnz
        say(f"{shape:11s} ({n_user} users, {n_item} items, nnz(L) {nnz}): LightGCN step {t_lg * 1e3:7.1f} "
            f"({s_lg.launches_per_step} launches), NGCF step {t_ng * 1e3:7.1f} ({s_ng.launches_per_step} launches), "
            f"torch fp32 LightGCN {t_torch * 1e3:8.1f} ({t_torch / t_lg:.1f}x); the 2K = {2 * K} products alone "
            f"{t_prod * 1e3:6.1f} ({100 * t_prod / t_lg:.0f}% of the LightGCN step)")
        del s_lg, s_ng, lg, lg1, ng, tl
        torch.cuda.empty_cache()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
