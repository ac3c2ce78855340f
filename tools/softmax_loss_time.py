"""Sampled-softmax loss (SoftmaxLoss, ngcf_softmax_loss) against BPR and against a torch fp32 composition of the same
loss, all measured in one run:

  loss        forward + backward (the gradients of u, p, n) at (B, D) = (1024, 256) and (4096, 640), with and without
              negatives, item ids given (masking on); BPR's kernel on the same rows (it always takes n); the torch
              composition: fp32 mm + masked logsumexp + autograd (torch.autograd.grad), default fp32 matmul precision
  step        the captured Gowalla training step (GraphedStep with Adam) with BPR and with SoftmaxLoss, alternated

CUDA events, medians, no L2 flush (the operands are read warm, as inside a training step).  Prints the card and its
power limit read in the same run.
python tools/softmax_loss_time.py [--reps N] [--out PATH]"""
import argparse
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

import seoul_tourism_recommendation_ngcf_b200 as pkg
from seoul_tourism_recommendation_ngcf_b200 import laplacian, synth

dev = torch.device("cuda:0")
TAU, WD = 0.2, 0.025


def timed(fns, reps):
    """medians (ms) of each fn in fns, called alternately"""
    for fn in fns:
        fn(); fn()
    ev = [[] for _ in fns]
    for _ in range(reps):
        for j, fn in enumerate(fns):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record()
            ev[j].append((e0, e1))
    torch.cuda.synchronize()
    return [statistics.median(a.elapsed_time(b) for a, b in e) for e in ev]


def torch_loss(u, p, n, pos, neg, bs):
    """the same loss composed of torch fp32 ops"""
    has_n = n.numel() > 0
    cols = torch.cat([p, n]) if has_n else p
    s = u @ cols.T / TAU
    col_ids = torch.cat([pos, neg]) if has_n else pos
    keep = col_ids[None, :] != pos[:, None]
    keep.fill_diagonal_(True)
    lse = torch.logsumexp(s.masked_fill(~keep, float("-inf")), dim=1)
    reg = (u * u).sum(1) + (p * p).sum(1) + ((n * n).sum(1) if has_n else 0.0)
    return (lse - s.diagonal() + WD * reg).sum() / bs


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))),
                                                  "profiles", "r05_softmax_loss_time.txt"))
    args = ap.parse_args()
    lines = []

    def say(s):
        print(s, flush=True)
        lines.append(s)

    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    say(f"card: {torch.cuda.get_device_name(0)}; nvidia-smi (name, power limit, max SM clock): {q[0] if q else '?'}")
    say(f"tau {TAU}, weight_decay {WD}; medians of {args.reps} alternated calls, times in us")

    for B, D in ((1024, 256), (4096, 640)):
        g = torch.Generator().manual_seed(B + D)
        u, p, n = (torch.randn(B, D, generator=g).div_(D ** 0.5).to(dev).requires_grad_(True) for _ in range(3))
        pos = torch.randint(0, 40981, (B,), generator=g).to(dev)
        neg = torch.randint(0, 40981, (B,), generator=g).to(dev)
        empty = torch.empty(0, device=dev)
        sm, bpr = pkg.SoftmaxLoss(WD, B, TAU), pkg.BPR(WD, B)
        res = {}
        for with_n in (False, True):
            nn_ = n if with_n else empty
            xs = [u, p, n] if with_n else [u, p]
            nid = neg if with_n else None

            def fused():
                torch.autograd.grad(sm(u, p, nn_, pos, nid), xs)

            def composed():
                torch.autograd.grad(torch_loss(u, p, nn_, pos, neg, B), xs)

            fns = [fused, composed]
            if with_n:
                fns.append(lambda: torch.autograd.grad(bpr(u, p, n), [u, p, n]))
            res[with_n] = timed(fns, args.reps)
            # outputs of the two paths at this shape
            lf, lc = float(sm(u, p, nn_, pos, nid)), float(torch_loss(u, p, nn_, pos, neg, B))
            res[with_n].append(abs(lf - lc) / abs(lc))
        n_cols = 2 * B
        flop = 3 * 2 * B * n_cols * D
        for with_n in (False, True):
            t = res[with_n]
            cols = 2 * B if with_n else B
            line = (f"loss B {B} D {D} {'with n   ' if with_n else 'without n'} ({cols} columns): fused fwd+bwd "
                    f"{t[0] * 1e3:8.1f}, torch fp32 composition {t[1] * 1e3:8.1f} ({t[1] / t[0]:.1f}x)")
            if with_n:
                line += f", BPR kernel fwd+bwd {t[2] * 1e3:6.1f}"
            line += f"; loss rel diff fused vs torch {t[-1]:.1e}"
            say(line)
        say(f"    (B {B} D {D}, 2B columns: three products of {flop / 3 / 1e9:.2f} GFLOP; 3xTF32 makes "
            f"{3 * flop / 1e12 * 1e3:.1f} GFLOP of tensor work, {3 * flop / 1125e12 * 1e6:.1f} us at 1,125 TFLOP/s; "
            f"fused achieved {flop / (res[True][0] * 1e-3) / 1e12:.1f} TFLOP/s of fp32-equivalent work)")

    # captured Gowalla step, BPR vs SoftmaxLoss, alternated
    n_user, n_item, n_inter, emb, K = synth.SHAPES["gowalla"]
    B = 1024
    ui, ii, ri = synth.powerlaw_bipartite(n_user, n_item, n_inter, alpha=0.8, seed=0)
    L = laplacian.laplacian_coo(ui, ii, ri, n_user, n_item)
    batch = {k: torch.from_numpy(v) for k, v in synth.random_batch(n_user, n_item, B, seed=1).items()}
    steps = []
    for crit in (pkg.BPR(WD, B), pkg.SoftmaxLoss(WD, B, TAU)):
        torch.manual_seed(0)
        m = pkg.NGCF(emb, [emb] * K, 0.3, [0.1] * K, 1.0, [L, L], synth.num_dict_for(n_user, n_item), B, dev).to(dev)
        m.train()
        steps.append(pkg.GraphedStep(m, crit, B, node_flag=True, optimizer=pkg.Adam(m.parameters(), lr=1e-3)))
    t_bpr, t_sm = timed([lambda: steps[0](batch), lambda: steps[1](batch)], args.reps)
    say(f"step  Gowalla (emb {emb} x {K}, D {emb * (K + 1)}, batch {B}) GraphedStep + Adam: BPR {t_bpr * 1e3:.1f}, "
        f"SoftmaxLoss {t_sm * 1e3:.1f} (+{(t_sm - t_bpr) * 1e3:.1f}); launches per step {steps[0].launches_per_step} "
        f"vs {steps[1].launches_per_step}")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
